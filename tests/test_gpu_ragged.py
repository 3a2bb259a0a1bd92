"""Variable-length batches on the B200: every lengths-aware kernel and model path against the existing, already verified
fixed-length path.  The reference for utterance b of length L is the `lengths=None` call on the batch cropped to T = L --
same B, so the host picks the same kernels (weight-stationary / wavefront / batched, gate group, sub-batching) -- and
the ragged run must be BIT-identical to it on frames < L and exactly 0 past it."""
import pytest
import torch

from oracle import rel_l2, templates
from oracle.autovc import autovc_forward
from oracle.lstmdv import lstmdv_forward
from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker
from tests.test_gpu_parity import TOL

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _lengths(B, T, multiple, seed):
    g = torch.Generator().manual_seed(seed)
    vals = (torch.randint(1, T // multiple + 1, (B,), generator=g) * multiple).tolist()
    vals[0] = T                                       # one full-length utterance
    return vals


def _dev_lengths(vals):
    return torch.tensor(vals, dtype=torch.int32, device=DEV)


# ------------------------------------------------------------------------------------------------ avc_zero_tail
@pytest.mark.parametrize("dtype,C", [(torch.float32, 336), (torch.bfloat16, 1024), (torch.float16, 512),
                                     (torch.float32, 80), (torch.float16, 80)])
@pytest.mark.parametrize("row0,extra", [(0, 0), (3, 5)])
def test_zero_tail(dtype, C, row0, extra):
    from autoformer_b200 import ops
    B, T = 7, 96
    lengths = _lengths(B, T, 1, 3)
    buf = torch.full((B, row0 + T + extra, C), float("nan"), dtype=dtype, device=DEV)
    ops.zero_tail(buf, row0, T, _dev_lengths(lengths))
    torch.cuda.synchronize()
    for b, n in enumerate(lengths):
        assert torch.isnan(buf[b, :row0 + n].float()).all() and torch.isnan(buf[b, row0 + T:].float()).all()
        assert (buf[b, row0 + n:row0 + T].view(torch.int16 if dtype != torch.float32 else torch.int32) == 0).all()


# ------------------------------------------------------------------------------------------------ avc_bilstm_small
# H = 32, B <= 128: bilstm32_kernel; H = 32, B > 128: bilstm_small_kernel<1, true>; H < 32: <1, false>; H > 32: <2, false>
@pytest.mark.parametrize("H,B", [(32, 6), (32, 160), (16, 10), (44, 6), (64, 9)])
@pytest.mark.parametrize("freq", [1, 22, 32])
@pytest.mark.parametrize("out_kind", ["fp32", "split", "bf16", "none"])
def test_bilstm_small_lengths(H, B, freq, out_kind):
    from autoformer_b200 import ops
    T = 4 * freq if freq > 1 else 70
    g = torch.Generator().manual_seed(H + B + freq)
    xproj = (torch.randn(B, T, 8 * H, generator=g) * 0.5).to(DEV)
    w_hh = (torch.randn(2, 4 * H, H, generator=g) * (1.0 / H ** 0.5)).to(DEV)
    lengths = _lengths(B, T, freq, freq)

    def run(xp, T_):
        width, dt = {"fp32": (2 * H, torch.float32), "split": (4 * H, torch.bfloat16), "bf16": (2 * H, torch.bfloat16),
                     "none": (None, None)}[out_kind]
        out = torch.full((B, T_, width), float("nan"), dtype=dt, device=DEV) if width else None
        codes = torch.full((B, T_ // freq, 2 * H), float("nan"), device=DEV)
        return out, codes, xp.reshape(B * T_, 8 * H).contiguous()

    out, codes, xp = run(xproj, T)
    ops.bilstm_small(xp, w_hh, B, T, H, out=out, codes=codes, freq=freq, split=out_kind == "split",
                     lengths=_dev_lengths(lengths))
    for L in sorted(set(lengths)):
        o_ref, c_ref, xp_ref = run(xproj[:, :L], L)
        ops.bilstm_small(xp_ref, w_hh, B, L, H, out=o_ref, codes=c_ref, freq=freq, split=out_kind == "split")
        for b in (b for b in range(B) if lengths[b] == L):
            assert torch.equal(codes[b, :L // freq], c_ref[b]) and not codes[b, L // freq:].any()
            if out is not None:
                assert torch.equal(out[b, :L], o_ref[b]) and not out[b, L:].any()


# ------------------------------------------------------------------------------------------------ h_last of the recurrences
@pytest.mark.parametrize("path", ["ws", "ws_f16", "stack", "seq_step16", "seq_persist32", "seq_fused"])
def test_h_last_lengths(path):
    from autoformer_b200 import layers, ops, packing
    g = torch.Generator().manual_seed(7)
    H, C, T = 768 if path.startswith(("ws", "stack")) else 512, 256, 40
    B = 12 if path.startswith(("ws", "stack")) else 96
    prec = "fp16x2" if path in ("ws_f16", "stack") else "fp32"
    lengths = _lengths(B, T, 1, 11)
    x = (torch.randn(B, T, C, generator=g)).to(DEV)
    mk = lambda *s: (torch.randn(*s, generator=g) * (1.0 / H ** 0.5)).to(DEV)

    if path == "stack":
        lay = [layers.LstmLayer(mk(4 * H, C if i == 0 else H), mk(4 * H, H), mk(4 * H), mk(4 * H), prec) for i in range(3)]
        st = layers.LstmStack(lay, prec, wavefront=True)
        assert st.eligible(B, True)

        def run(x_, T_, lens=None):
            h = torch.full((B, H), float("nan"), device=DEV)
            xa = ops.to_act(x_.contiguous(), prec)
            ih, _ = lay[0].packs(packing.WS_GROUP)
            xp = torch.empty(B * T_, 4 * H, device=DEV)
            ih(xa, B, T_, out2=xp)
            hs = ops.lstm_stack_ws(xp, st.packs(), B, T_, H, h_last=h, **({} if lens is None else {"lengths": lens}))
            return h, hs
        h, hs = run(x, T, _dev_lengths(lengths))
        for b, n in enumerate(lengths):                        # the fp16 sequence and the fp32 last state agree
            assert torch.equal(h[b].half(), hs[2, n, b])
    else:
        layer = layers.LstmLayer(mk(4 * H, C), mk(4 * H, H), mk(4 * H), mk(4 * H), prec,
                                 fused=path == "seq_fused")
        layer.ws = path.startswith("ws")
        persistent = path != "seq_step16"

        def run(x_, T_, lens=None):
            h = torch.full((B, H), float("nan"), device=DEV)
            layer(ops.to_act(x_.contiguous(), prec), B, T_, h_last=h, persistent=persistent,
                  **({} if lens is None else {"lengths": lens}))
            return h, None
        h, _ = run(x, T, _dev_lengths(lengths))
    for L in sorted(set(lengths)):
        ref, _ = run(x[:, :L], L)
        for b in (b for b in range(B) if lengths[b] == L):
            assert torch.equal(h[b], ref[b]), (path, b, L)


# ------------------------------------------------------------------------------------------------ models
def _autovc(args, precision, seed=0, persistent=True):
    from autoformer_b200.factory.AutoVC import AutoVC
    sd = seeded_state_dict(templates.autovc_template(*args), seed)
    m = AutoVC(*args).to(DEV)
    m.load_state_dict(sd)
    m.eval()
    m.precision = precision
    m.persistent_lstm = persistent
    return m, sd


def _check_autovc(m, x, c_org, c_trg, lengths):
    B, T = x.shape[:2]
    F = m.freq
    mel, post, codes = m(x, c_org, c_trg, lengths=lengths)
    codes = codes.view(B, T // F, -1)
    for L in sorted(set(lengths)):
        rm, rp, rc = m(x[:, :L].contiguous(), c_org, c_trg)
        rc = rc.view(B, L // F, -1)
        for b in (b for b in range(B) if lengths[b] == L):
            assert torch.equal(mel[b, :, :L], rm[b]) and torch.equal(post[b, :, :L], rp[b]), (b, L)
            assert torch.equal(codes[b, :L // F], rc[b]), (b, L)
            assert not mel[b, :, L:].any() and not post[b, :, L:].any() and not codes[b, L // F:].any()
    return mel, post, codes


@pytest.mark.parametrize("args", [(32, 256, 512, 32), (44, 256, 512, 22)])
@pytest.mark.parametrize("precision", ["fp32", "fp16x2"])
@pytest.mark.parametrize("B", [6, 96, 600])
def test_autovc_ragged_bit_identical(args, precision, B):
    F = args[3]
    T = 8 * F
    m, _ = _autovc(args, precision)
    x = synthetic_mel(B, T, 5).to(DEV)
    c_org, c_trg = synthetic_speaker(B, 5, "org").to(DEV), synthetic_speaker(B, 5, "trg").to(DEV)
    lengths = _lengths(B, T, F, B)
    _check_autovc(m, x, c_org, c_trg, lengths)


@pytest.mark.parametrize("precision,persistent", [("tf32", True), ("bf16", True), ("fp32", False)])
def test_autovc_ragged_other_paths(precision, persistent):
    args = (32, 256, 512, 32)
    B, T = 40, 192
    m, _ = _autovc(args, precision, persistent=persistent)
    x = synthetic_mel(B, T, 6).to(DEV)
    c = synthetic_speaker(B, 6, "org").to(DEV)
    _check_autovc(m, x, c, c, _lengths(B, T, 32, 2))


@pytest.mark.parametrize("precision", ["fp32", "fp16x2", "tf32", "bf16"])
def test_autovc_full_lengths_equal_fixed(precision):
    m, _ = _autovc((32, 256, 512, 32), precision)
    B, T = 20, 128
    x, c = synthetic_mel(B, T, 8).to(DEV), synthetic_speaker(B, 8, "org").to(DEV)
    for a, b in zip(m(x, c, c, lengths=[T] * B), m(x, c, c)):
        assert torch.equal(a, b)


def test_autovc_other_utterances_do_not_leak():
    m, _ = _autovc((32, 256, 512, 32), "fp16x2")
    B, T = 8, 256
    x, c = synthetic_mel(B, T, 9).to(DEV), synthetic_speaker(B, 9, "org").to(DEV)
    lengths = _lengths(B, T, 32, 4)
    a = m(x, c, c, lengths=lengths)
    x2 = x.clone()
    x2[1:] = synthetic_mel(B - 1, T, 77).to(DEV)
    x2[0, lengths[0]:] = 5.0
    b = m(x2, c, c, lengths=[lengths[0]] + _lengths(B - 1, T, 32, 99))
    assert torch.equal(a[1][0], b[1][0]) and torch.equal(a[2].view(B, -1)[0], b[2].view(B, -1)[0])


@pytest.mark.parametrize("args", [(32, 256, 512, 32), (44, 256, 512, 22)])
def test_autovc_ragged_vs_oracle(args):
    m, sd = _autovc(args, "fp32")
    F = args[3]
    B, T = 3, 6 * F
    lengths = [T, 2 * F, 4 * F]
    x = synthetic_mel(B, T, 3)
    c_org, c_trg = synthetic_speaker(B, 3, "org"), synthetic_speaker(B, 3, "trg")
    mel, post, codes = m(x.to(DEV), c_org.to(DEV), c_trg.to(DEV), lengths=lengths)
    codes = codes.view(B, T // F, -1).cpu()
    for b, n in enumerate(lengths):
        ref = autovc_forward(sd, x[b:b + 1, :n], c_org[b:b + 1], c_trg[b:b + 1], args[0], F, dtype=torch.float64)
        assert rel_l2(post[b:b + 1, :, :n].cpu(), ref[1]) < TOL["fp32"]
        assert rel_l2(codes[b:b + 1, :n // F].reshape(1, -1), ref[2]) < TOL["fp32"]


@pytest.mark.parametrize("path", ["wavefront", "layers", "batched"])
def test_lstmdv_ragged_bit_identical(path):
    from autoformer_b200.factory.LstmDV import LstmDV
    sd = seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5)
    m = LstmDV().to(DEV)
    m.load_state_dict(sd)
    m.precision = "fp16x2"
    m.wavefront = path == "wavefront"
    B = 96 if path == "batched" else 24
    T = 120
    x = synthetic_mel(B, T, 4).to(DEV)
    lengths = _lengths(B, T, 1, 5)
    e = m(x, lengths=lengths)
    for L in sorted(set(lengths)):
        ref = m(x[:, :L].contiguous())
        for b in (b for b in range(B) if lengths[b] == L):
            assert torch.equal(e[b], ref[b]), (path, b, L)
    assert torch.equal(m(x, lengths=[T] * B), m(x))


def test_lstmdv_ragged_vs_oracle():
    from autoformer_b200.factory.LstmDV import LstmDV
    sd = seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5)
    m = LstmDV().to(DEV)
    m.load_state_dict(sd)
    x = synthetic_mel(3, 50, 2)
    lengths = [50, 17, 33]
    e = m(x.to(DEV), lengths=lengths).cpu()
    for b, n in enumerate(lengths):
        assert rel_l2(e[b:b + 1], lstmdv_forward(sd, x[b:b + 1, :n], dtype=torch.float64)) < TOL["fp32"]
