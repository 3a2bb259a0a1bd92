"""CPU tests of variable-length batches (AutoVC / LstmDV ``forward(..., lengths=...)``, sharding.make_ragged_batches):
the batching plan, the host-side validation, and the ragged forwards on the CPU stand-ins of tests/emulate.py plus the
stand-ins below for the lengths-aware entry points, compared per utterance with the oracle on the cropped utterance."""
import warnings

import pytest
import torch

from oracle import rel_l2, templates
from oracle.autovc import autovc_forward
from oracle.lstmdv import lstmdv_forward
from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker
from tests import emulate

warnings.filterwarnings("ignore", category=FutureWarning)


# ------------------------------------------------------------------------------------------------ stand-ins for lengths
def _emu_zero_tail(buf, row0, T, lengths):
    for b, n in enumerate(lengths.tolist()):
        buf[b, row0 + n:row0 + T] = 0
    return buf


def _emu_bilstm_small(xproj, w_hh, B, T, H, out=None, codes=None, freq=1, round_tf32=True, split=False, lengths=None):
    if lengths is None:
        return emulate._emu_bilstm_small(xproj, w_hh, B, T, H, out, codes, freq, round_tf32, split)
    xp = xproj.view(B, T, 8 * H)
    for b, n in enumerate(lengths.tolist()):       # utterance b alone over its first n frames
        ob = torch.empty((1, n) + tuple(out.shape[2:]), dtype=out.dtype) if out is not None else None
        cb = torch.empty(1, n // freq, 2 * H) if codes is not None else None
        emulate._emu_bilstm_small(xp[b:b + 1, :n].reshape(n, 8 * H), w_hh, 1, n, H, ob, cb, freq, round_tf32, split)
        if out is not None:
            out[b].zero_()
            out[b, :n] = ob[0]
        if codes is not None:
            codes[b].zero_()
            codes[b, :n // freq] = cb[0]
    return out, codes


def _with_h_last_at_lengths(run, B, T, H, hseq_f32, h_last, lengths):
    """Run a stand-in with an exact fp32 sequence and take h_last[b] at frame lengths[b] - 1 from it."""
    f32 = hseq_f32 if hseq_f32 is not None else torch.empty(B, T, H)
    out = run(f32, None)
    if h_last is not None:
        for b, n in enumerate(lengths.tolist()):
            h_last[b] = f32[b, n - 1]
    return out


def _emu_lstm_seq(xproj, w_hh, B, T, H, precision, group, hseq=None, hseq_f32=None, h_last=None, persistent=False,
                  xin=None, w_ih=None, bias=None, c_in=None, lengths=None):
    def run(f32, hl):
        return emulate._emu_lstm_seq(xproj, w_hh, B, T, H, precision, group, hseq, f32, hl, persistent, xin, w_ih, bias,
                                     c_in)
    if lengths is None:
        return run(hseq_f32, h_last)
    return _with_h_last_at_lengths(run, B, T, H, hseq_f32, h_last, lengths)


def _emu_lstm_seq_ws(xproj, w_hh, B, T, H, hseq=None, hseq_f32=None, h_last=None, precision="fp32", lengths=None):
    def run(f32, hl):
        return emulate._emu_lstm_seq_ws(xproj, w_hh, B, T, H, hseq, f32, hl, precision)
    if lengths is None:
        return run(hseq_f32, h_last)
    return _with_h_last_at_lengths(run, B, T, H, hseq_f32, h_last, lengths)


def _emu_lstm_stack_ws(xproj0, packs, B, T, H, h_last=None, hs=None, debug_clk=None, lengths=None):
    hs = emulate._emu_lstm_stack_ws(xproj0, packs, B, T, H, None if lengths is not None else h_last, hs)
    if lengths is not None and h_last is not None:
        xp = xproj0.view(B, T, 4 * H)
        for b, n in enumerate(lengths.tolist()):      # the top layer's h at frame n - 1: the cropped run's h_last
            hl = torch.empty(1, H)
            emulate._emu_lstm_stack_ws(xp[b:b + 1, :n].reshape(n, 4 * H), packs, 1, n, H, hl)
            h_last[b] = hl[0]
    return hs


class _Recorder:
    """Wraps the stand-ins and records (name, keyword names) of every call."""

    def __init__(self):
        self.calls = []

    def wrap(self, name, fn):
        def rec(*a, **kw):
            self.calls.append((name, tuple(sorted(kw))))
            return fn(*a, **kw)
        return rec


@pytest.fixture
def rec(monkeypatch):
    from autoformer_b200 import ops
    emulate.install_cpu_kernels(monkeypatch)
    r = _Recorder()
    for name, fn in (("zero_tail", _emu_zero_tail), ("bilstm_small", _emu_bilstm_small), ("lstm_seq", _emu_lstm_seq),
                     ("lstm_seq_ws", _emu_lstm_seq_ws), ("lstm_stack_ws", _emu_lstm_stack_ws)):
        monkeypatch.setattr(ops, name, r.wrap(name, fn))
    return r


def _autovc(args, seed, precision="fp32"):
    from autoformer_b200.factory.AutoVC import AutoVC
    sd = seeded_state_dict(templates.autovc_template(*args), seed)
    m = AutoVC(*args)
    m.load_state_dict(sd)
    m.eval()
    m.precision = precision
    return m, sd


# ------------------------------------------------------------------------------------------------ batching plan
def test_make_ragged_batches():
    from autoformer_b200 import sharding
    g = torch.Generator().manual_seed(0)
    lengths = torch.randint(1, 300, (1000,), generator=g).tolist()
    batches = sharding.make_ragged_batches(lengths, 128, 32)
    assert batches == sharding.make_ragged_batches(lengths, 128, 32)
    ids = [i for _, run in batches for i in run]
    assert sorted(ids) == list(range(1000))
    padded = [(t + 31) // 32 * 32 for t in lengths]
    assert [padded[i] for i in ids] == sorted(padded, reverse=True)
    for T, run in batches:
        assert 1 <= len(run) <= 128 and T % 32 == 0 and T == max(padded[i] for i in run)
        assert run == sorted(run, key=lambda i: (-padded[i], i))
    assert all(len(run) == 128 for _, run in batches[:-1])
    plan = sharding.plan_ragged(lengths, 3, 128, 32)
    assert sorted(i for rank in plan for _, run in rank for i in run) == list(range(1000))


# ------------------------------------------------------------------------------------------------ host validation
@pytest.mark.parametrize("lengths,what", [([64, 64], "entries"), ([64, 0, 32], r"\[1, T"), ([64, 96, 32], r"\[1, T"),
                                          ([64, 40, 32], "multiples of freq")])
def test_autovc_lengths_validation(rec, lengths, what):
    m, _ = _autovc((32, 256, 512, 32), 0)
    x, c = synthetic_mel(3, 64, 1), synthetic_speaker(3, 1, "org")
    with pytest.raises(ValueError, match=what):
        m(x, c, c, lengths=lengths)
    assert not rec.calls


def test_autovc_lengths_with_batch_stats(rec):
    m, _ = _autovc((32, 256, 512, 32), 0)
    m.bn_stats = "batch"
    x, c = synthetic_mel(2, 64, 1), synthetic_speaker(2, 1, "org")
    with pytest.raises(ValueError, match="bn_stats"):
        m(x, c, c, lengths=[64, 32])


def test_lstmdv_lengths_validation(rec):
    from autoformer_b200.factory.LstmDV import LstmDV
    m = LstmDV()
    with pytest.raises(ValueError, match="entries"):
        m(synthetic_mel(2, 10, 1), lengths=torch.tensor([10]))
    with pytest.raises(ValueError, match=r"\[1, T"):
        m(synthetic_mel(2, 10, 1), lengths=torch.tensor([10, 11]))


# ------------------------------------------------------------------------------------------------ ragged forwards
@pytest.mark.parametrize("args,lengths,precision,tol", [((32, 256, 512, 32), [96, 32, 64], "fp32", 1e-4),
                                                        ((32, 256, 512, 32), [64, 96, 32], "fp16x2", 1e-3),
                                                        ((44, 256, 512, 22), [44, 66, 22], "fp32", 1e-4)])
def test_autovc_ragged_matches_cropped_oracle(rec, args, lengths, precision, tol):
    m, sd = _autovc(args, 2, precision)
    B, T, F = len(lengths), max(lengths), args[3]
    x, c_org, c_trg = synthetic_mel(B, T, 7), synthetic_speaker(B, 7, "org"), synthetic_speaker(B, 7, "trg")
    for b, n in enumerate(lengths):
        x[b, n:] = 1e3                                  # whatever the padded frames hold is ignored
    mel, post, codes = m(x, c_org, c_trg, lengths=lengths)
    assert sum(1 for name, _ in rec.calls if name == "zero_tail") == 13
    codes = codes.view(B, T // F, -1)
    for b, n in enumerate(lengths):
        ref = autovc_forward(sd, x[b:b + 1, :n], c_org[b:b + 1], c_trg[b:b + 1], args[0], F)
        assert rel_l2(mel[b:b + 1, :, :n], ref[0]) < tol and rel_l2(post[b:b + 1, :, :n], ref[1]) < tol
        assert rel_l2(codes[b:b + 1, :n // F].reshape(1, -1), ref[2]) < tol
        assert not mel[b, :, n:].any() and not post[b, :, n:].any() and not codes[b, n // F:].any()


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("fp16x2", 2e-3)])
def test_lstmdv_ragged_matches_cropped_oracle(rec, monkeypatch, precision, tol):
    from autoformer_b200 import ops
    from autoformer_b200.factory.LstmDV import LstmDV
    monkeypatch.setattr(ops, "linear_rows", lambda h, w, bias, want_raw=True, want_normed=False: (
        (h.double() @ w.double().t() + bias.double()).float(), emulate._emu_linear_l2norm(h, w, bias)))
    from autoformer_b200.make_data.factory.LstmDV import LstmDV as Twin
    sd = seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5)
    lengths = [20, 7, 13]
    x = synthetic_mel(3, 20, 5)
    m = LstmDV()
    m.load_state_dict(sd)
    m.precision = precision
    e = m(x, lengths=torch.tensor(lengths))
    for b, n in enumerate(lengths):
        assert rel_l2(e[b:b + 1], lstmdv_forward(sd, x[b:b + 1, :n])) < tol
    twin = Twin()
    twin.load_state_dict({**sd, **{k: v for k, v in twin.state_dict().items() if k.startswith("output.")}})
    twin.precision = precision
    assert torch.equal(twin(x, lengths=lengths)[1], e)


def test_fixed_length_calls_are_unchanged(rec):
    """lengths=None: no ops function gets a `lengths` keyword and nothing is zero-tailed -- the fixed-length forward
    launches exactly what it launched before variable-length batches existed."""
    from autoformer_b200.factory.LstmDV import LstmDV
    m, _ = _autovc((32, 256, 512, 32), 0)
    x, c = synthetic_mel(2, 64, 1), synthetic_speaker(2, 1, "org")
    m(x, c, c)
    dv = LstmDV()
    for precision in ("fp32", "fp16x2"):
        dv.precision = precision
        dv(synthetic_mel(2, 10, 1))
    names = {name for name, _ in rec.calls}
    assert {"bilstm_small", "lstm_seq_ws", "lstm_stack_ws"} <= names and "zero_tail" not in names
    assert all("lengths" not in kw for _, kw in rec.calls)


def test_sub_batched_lstm_slices_lengths(rec, monkeypatch):
    """Persistent sub-batching (B above the one-wave cap) hands each sub-batch its slice of the lengths."""
    from autoformer_b200 import layers, ops, packing
    monkeypatch.setattr(ops, "persistent_batch_cap", lambda H, n_sm=148: 2)
    g = torch.Generator().manual_seed(1)
    C, H, B, T = 64, 64, 5, 9
    layer = layers.LstmLayer(torch.randn(4 * H, C, generator=g) * 0.1, torch.randn(4 * H, H, generator=g) * 0.1,
                             torch.randn(4 * H, generator=g) * 0.1, torch.randn(4 * H, generator=g) * 0.1, "fp32")
    layer.ws = False
    x = packing.to_act(torch.randn(B, T, C, generator=g), "fp32")
    lengths = torch.tensor([9, 3, 5, 1, 7], dtype=torch.int32)
    h_last = torch.empty(B, H)
    layer(x, B, T, h_last=h_last, persistent=True, lengths=lengths)
    for b, n in enumerate(lengths.tolist()):
        ref = torch.empty(1, H)
        layer(x[b:b + 1, :n].contiguous(), 1, n, h_last=ref, persistent=True)
        assert torch.allclose(h_last[b], ref[0], atol=1e-6)


def test_convert_and_embed_utterances(rec):
    """pipeline.convert_utterances / embed_utterances: any lengths in, per-utterance results out in input order, each
    equal to the plain call on the utterance alone (padded to a multiple of freq and trimmed, as pipeline.convert)."""
    from autoformer_b200 import pipeline
    from autoformer_b200.factory.LstmDV import LstmDV
    m, _ = _autovc((32, 256, 512, 32), 4)
    lens = [40, 64, 17, 96, 64]
    mels = [synthetic_mel(1, n, 10 + i)[0] for i, n in enumerate(lens)]
    c_org, c_trg = synthetic_speaker(len(lens), 3, "org"), synthetic_speaker(len(lens), 3, "trg")
    outs = pipeline.convert_utterances(m, mels, c_org, c_trg, max_batch=2)
    for i, (mel, o) in enumerate(zip(mels, outs)):
        ref = pipeline.convert(m, mel[None], c_org[i:i + 1], c_trg[i:i + 1])[0]
        assert o.shape == (lens[i], 80) and rel_l2(o, ref) < 1e-5
    dv = LstmDV()
    dv.load_state_dict(seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5))
    e = pipeline.embed_utterances(dv, [m_[:n] for m_, n in zip(mels, [5, 9, 17, 3, 12])], max_batch=3)
    for i, n in enumerate([5, 9, 17, 3, 12]):
        assert rel_l2(e[i:i + 1], dv(mels[i][None, :n])) < 1e-5
