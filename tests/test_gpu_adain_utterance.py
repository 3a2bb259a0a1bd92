"""Per-utterance AdaIN statistics on the B200: avc_segment_stats and avc_adain_segmented element by element against
fp64 through the C ABI, their determinism contract, and AutoVC2 / MetaPool2 / MetaConv2 with adain_stats = "utterance"
against the per-utterance oracle, the fixed-length path (bit for bit) and the pipeline."""
import pytest
import torch

from oracle import rel_l2
from oracle.adain import autovc2_forward
from oracle.seeded import synthetic_mel, synthetic_speaker
from tests.test_adain_utterance import ARGS, adain2, check_against_cropped_oracle, golden_row_call, ragged_inputs
from tests.test_gpu_kernel_contract import check_bound, check_sentinel, nan_buf
from tests.test_gpu_meta_contract import FORMATS, bits, call, check_stored, decode, fp64_moments_bound, lib, \
    offset_rows, u

pytestmark = pytest.mark.gpu
DEV = "cuda"
B, T, C = 7, 96, 80
LENGTHS = [96, 32, 1, 64, 57, 96, 2]          # freq (32) and T among them


def _data(seed, B_=B, T_=T, lengths=LENGTHS):
    """offset_rows data (|mean| / std up to 1000) with NaN past every length."""
    g = torch.Generator().manual_seed(seed)
    x = offset_rows((B_, T_ * C), (0.0, 100.0, 1000.0), g).view(B_, T_, C)
    for b, n in enumerate(lengths):
        x[b, n:] = float("nan")
    return x.contiguous()


def _segment_stats(x, lengths):
    """avc_segment_stats through the C ABI on NaN stats / scratch buffers; the spare stats slot stays NaN."""
    Bx, Tx, Cx = x.shape
    chunks = -(-Tx * Cx // 4096)
    st = nan_buf((Bx + 1, 2), torch.float32)
    scratch = nan_buf((2 * Bx * chunks,), torch.float64)
    lens = torch.tensor(lengths, dtype=torch.int32, device=DEV) if lengths is not None else None
    call(lib().avc_segment_stats, x.to(DEV), Bx, Tx, Cx, lens, st, scratch)
    region = torch.zeros(st.shape, dtype=torch.bool)
    region[:Bx] = True
    check_sentinel(st, region, "segment_stats")
    return st[:Bx].cpu()


# ------------------------------------------------------------------------------------------------ avc_segment_stats
def test_segment_stats_against_fp64():
    x = _data(1)
    st = _segment_stats(x, LENGTHS)
    for b, n in enumerate(LENGTHS):
        # chains: 16 additions per thread, 5 shuffle and 8 shared levels, then at most 2 chunks
        mean, var, e_mean, e_var = fp64_moments_bound(x[b, :n].reshape(1, -1), 64, bessel=True)
        std = torch.sqrt(var)
        check_bound(st[b:b + 1, 0], mean, e_mean, f"segment_stats mean b={b}")
        check_bound(st[b:b + 1, 1], std, std * 2 * u + e_var / (2 * std), f"segment_stats std b={b}")
    assert torch.equal(bits(_segment_stats(x, LENGTHS)), bits(st)), "a repeated call differs"
    full = _data(2, lengths=[T] * B)
    assert torch.equal(bits(_segment_stats(full, None)), bits(_segment_stats(full, [T] * B)))


def test_segment_stats_bits_depend_only_on_the_utterance():
    x = _data(3)
    st = _segment_stats(x, LENGTHS)
    # other neighbours (other data, other lengths)
    lens2 = list(LENGTHS)
    y = _data(4, lengths=[T] * B)
    y[0], lens2[1:] = x[0], [5, 96, 17, 3, 80, 40]
    assert torch.equal(bits(_segment_stats(y, lens2)[0]), bits(st[0]))
    # a longer T (NaN padding) and a smaller B
    x_long = torch.cat((x, torch.full((B, 64, C), float("nan"))), 1)
    assert torch.equal(bits(_segment_stats(x_long, LENGTHS)), bits(st))
    assert torch.equal(bits(_segment_stats(x[2:5].contiguous(), LENGTHS[2:5])), bits(st[2:5]))
    assert torch.equal(bits(_segment_stats(x[:1].contiguous(), LENGTHS[:1])), bits(st[:1]))


# ------------------------------------------------------------------------------------------------ avc_adain_segmented
@pytest.mark.parametrize("per_utt_style", [False, True], ids=["broadcast", "per_utterance"])
def test_adain_segmented_against_fp64(per_utt_style):
    from autoformer_b200 import packing
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(B, T, C, generator=g) * 2.5 + 0.7)
    for b, n in enumerate(LENGTHS):
        x[b, n:] = float("nan")
    xs = torch.stack([torch.stack([x[b, :n].double().mean(), x[b, :n].double().std()])
                      for b, n in enumerate(LENGTHS)]).float()
    if per_utt_style:                              # target std up to 3e4: values beyond ~2.2 std saturate fp16
        ts = torch.stack([torch.linspace(-0.3, 0.5, B), torch.logspace(-1, 4.5, B)], 1).float().contiguous()
    else:
        ts = torch.tensor([-0.3, 3e4])
    tsb = ts.double().expand(B, 2)
    d = x.double() - xs[:, 0].double().view(B, 1, 1)
    k = (tsb[:, 1] / xs[:, 1].double()).view(B, 1, 1)
    y = d * k + tsb[:, 0].view(B, 1, 1)
    e = 6 * u * (d.abs() * k.abs() + tsb[:, 0].abs().view(B, 1, 1))
    valid = torch.zeros(B, T, dtype=torch.bool)
    for b, n in enumerate(LENGTHS):
        valid[b, :n] = True
    lens = torch.tensor(LENGTHS, dtype=torch.int32, device=DEV)
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(C, fmt)
        for want_f32, want_op in ((True, False), (False, True), (True, True)):
            f32 = nan_buf((B + 1, T, C), torch.float32) if want_f32 else None
            op = nan_buf((B + 1, T, ach), packing.TORCH_DTYPE[fmt]) if want_op else None
            call(lib().avc_adain_segmented, x.to(DEV), xs.to(DEV), ts.to(DEV), 2 if per_utt_style else 0, lens, f32, op,
                 dt, rnd, B, T, C)
            what = f"adain_segmented {fmt}/{dt}/{rnd} f32={want_f32} op={want_op}"
            for buf, name in ((f32, "out_f32"), (op, "out_op")):
                if buf is None:
                    continue
                region = torch.zeros(buf.shape, dtype=torch.bool)
                region[:B] = True
                check_sentinel(buf, region, f"{what} {name}")
                got = buf[:B].cpu()
                assert not bits(got[~valid]).any(), f"{what} {name}: rows past a length are not exactly 0"
                if name == "out_f32":
                    check_bound(got[valid], y[valid], e[valid], f"{what} {name}")
                else:
                    check_stored(decode(got, fmt)[valid], y[valid], e[valid], fmt, rnd, f"{what} {name}")


def test_adain_segmented_b1_is_avc_adain():
    from autoformer_b200 import packing
    g = torch.Generator().manual_seed(6)
    x = (torch.randn(1, T, C, generator=g) * 1.7 - 0.4).to(DEV)
    xs = torch.tensor([-0.41, 1.69], device=DEV)
    ts = torch.tensor([0.3, 2.2], device=DEV)
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(C, fmt)
        outs = []
        for seg in (False, True):
            f32 = nan_buf((T, C), torch.float32)
            op = nan_buf((T, ach), packing.TORCH_DTYPE[fmt])
            if seg:
                call(lib().avc_adain_segmented, x, xs, ts, 0, None, f32, op, dt, rnd, 1, T, C)
            else:
                call(lib().avc_adain, x, xs, ts, f32, op, dt, rnd, T, C)
            outs.append((bits(f32), bits(op)))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), fmt


def test_ops_wrappers_equal_the_direct_calls():
    from autoformer_b200 import ops
    x = _data(7, lengths=[T] * B).to(DEV)
    lens = torch.tensor(LENGTHS, dtype=torch.int32, device=DEV)
    st = nan_buf((B, 2), torch.float32)
    call(lib().avc_segment_stats, x, B, T, C, lens, st, torch.empty(2 * B * 2, dtype=torch.float64, device=DEV))
    assert torch.equal(bits(ops.segment_stats(x, lens)), bits(st))
    ts = torch.rand(B, 2, device=DEV) + 0.5
    af, ao = torch.empty_like(x), ops.alloc_act(B, T, C, "fp16x2", DEV)
    call(lib().avc_adain_segmented, x, st, ts, 2, lens, af, ao, 3, 1, B, T, C)
    wo, wf = ops.adain_segmented(x, st, ts, "fp16x2", lens, want_f32=True)
    assert torch.equal(bits(wo), bits(ao)) and torch.equal(bits(wf), bits(af))


# ------------------------------------------------------------------------------------------------ AutoVC2
def _model(precision, seed=3):
    m, sd = adain2(None, ARGS, seed, precision)
    return m.cuda(), sd


def _on_dev(*ts):
    return tuple(t.to(DEV) for t in ts)


# fp16x2 codes: 1.08e-3 measured on the B200 for a full-length utterance, as for the same utterance converted alone with
# the default batch statistics -- the pre-extract puts three more fp16 operand roundings ahead of the encoder (AutoVC's
# own fp16x2 codes are at ~5e-4), so the codes gate of this precision is 1.5e-3
@pytest.mark.parametrize("precision,tol,feat_tol,codes_tol", [("fp32", 3e-4, 1e-4, 3e-4), ("fp16x2", 1e-3, 5e-3, 1.5e-3)])
def test_autovc2_utterance_vs_oracle(precision, tol, feat_tol, codes_tol):
    m, sd = _model(precision)
    lengths = [96, 32, 64]
    check_against_cropped_oracle(m, sd, *_on_dev(*ragged_inputs(lengths, 8)), lengths, tol, feat_tol,
                                 codes_tol=codes_tol)
    x = (synthetic_mel(3, 96, 8) * torch.tensor([1.0, 0.5, 2.0]).view(3, 1, 1)).to(DEV)
    c = synthetic_speaker(3, 8, "org").to(DEV)
    check_against_cropped_oracle(m, sd, x, c, c, None, tol, feat_tol, codes_tol=codes_tol)


def test_autovc2_per_utterance_target_feature():
    m, sd = _model("fp32")
    lengths = [64, 96, 32]
    x, c_org, c_trg = _on_dev(*ragged_inputs(lengths, 9))
    _, fo = m(synthetic_mel(3, 96, 77).to(DEV), c_org, None)
    perm = [2, 0, 1]
    tf = [[mu[perm].clone(), s[perm].clone()] for mu, s in fo]
    ref_tf = lambda b: [[mu[b].cpu(), s[b].cpu()] for mu, s in tf]
    check_against_cropped_oracle(m, sd, x, c_org, c_trg, lengths, 3e-4, 1e-4, tf, ref_tf)


@pytest.mark.parametrize("precision", ["fp32", "fp16x2"])
@pytest.mark.parametrize("Bn", [6, 96])
def test_autovc2_ragged_bit_identical_to_cropped_batches(precision, Bn):
    m, _ = _model(precision)
    Tn = 8 * ARGS[3]
    g = torch.Generator().manual_seed(Bn)
    lengths = (torch.randint(1, 9, (Bn,), generator=g) * ARGS[3]).tolist()
    lengths[0] = Tn
    x, c_org, c_trg = _on_dev(synthetic_mel(Bn, Tn, 5), synthetic_speaker(Bn, 5, "org"), synthetic_speaker(Bn, 5, "trg"))
    mel, post, codes = m(x, c_org, c_trg, lengths=lengths)
    _, feats = m(x, c_org, None, lengths=lengths)
    codes = codes.view(Bn, Tn // ARGS[3], -1)
    for L in sorted(set(lengths)):
        rm, rp, rc = m(x[:, :L].contiguous(), c_org, c_trg)
        _, rf = m(x[:, :L].contiguous(), c_org, None)
        rc = rc.view(Bn, L // ARGS[3], -1)
        for b in (b for b in range(Bn) if lengths[b] == L):
            assert torch.equal(mel[b, :, :L], rm[b]) and torch.equal(post[b, :, :L], rp[b]), (b, L)
            assert torch.equal(codes[b, :L // ARGS[3]], rc[b]), (b, L)
            assert all(torch.equal(f[k][b], r[k][b]) for f, r in zip(feats, rf) for k in range(2)), (b, L)
            assert not mel[b, :, L:].any() and not post[b, :, L:].any() and not codes[b, L // ARGS[3]:].any()


def test_autovc2_other_utterances_do_not_leak():
    m, _ = _model("fp16x2")
    Bn, Tn = 8, 256
    x, c = synthetic_mel(Bn, Tn, 9).to(DEV), synthetic_speaker(Bn, 9, "org").to(DEV)
    lengths = [192, 256, 32, 64, 128, 224, 96, 160]
    a = m(x, c, c, lengths=lengths)
    x2 = x.clone()
    x2[1:] = synthetic_mel(Bn - 1, Tn, 77).to(DEV) * 3.0
    x2[0, lengths[0]:] = 5.0
    b = m(x2, c, c, lengths=[lengths[0]] + [256, 64, 32, 96, 256, 128, 32])
    assert torch.equal(a[1][0], b[1][0]) and torch.equal(a[2].view(Bn, -1)[0], b[2].view(Bn, -1)[0])
    x2[0] = x[0]                                   # and without lengths
    a, b = m(x, c, c), m(x2, c, c)
    assert torch.equal(a[1][0], b[1][0]) and torch.equal(a[2].view(Bn, -1)[0], b[2].view(Bn, -1)[0])


def test_autovc2_b1_utterance_equals_batch_within_rounding():
    m, _ = _model("fp32")
    x, c_org, c_trg = _on_dev(synthetic_mel(1, 128, 12), synthetic_speaker(1, 12, "org"), synthetic_speaker(1, 12, "trg"))
    m.adain_stats = "utterance"
    u_out, (_, u_feats) = m(x, c_org, c_trg), m(x, c_org, None)
    m.adain_stats = "batch"
    b_out, (_, b_feats) = m(x, c_org, c_trg), m(x, c_org, None)
    for p, q in zip(u_out, b_out):
        assert rel_l2(p, q) <= 1e-5
    for pf, qf in zip(u_feats, b_feats):
        for p, q in zip(pf, qf):
            assert p.shape == (1,) and q.dim() == 0 and abs(float(p[0]) - float(q)) <= 1e-5 * max(1.0, abs(float(q)))


# ------------------------------------------------------------------------------------------------ Meta2 golden rows
@pytest.mark.parametrize("name,kind", [("metapool2_b1_t176", "pool"), ("metaconv2_b1_t176", "conv")])
def test_meta2_golden_row_in_a_batch(name, kind):
    from tests.test_host_logic import _adain_model
    from tests.test_oracle_golden import adain_case, check_adain_outputs
    g, args, sd, i, _ = adain_case(name, kind)
    m = _adain_model(kind, args, sd).cuda()
    m.adain_stats = "utterance"
    check_adain_outputs(g, golden_row_call(m, i), 3e-4, 1e-4)
    m.adain_stats = "batch"
    assert rel_l2(golden_row_call(m, i)("x", True, None)[1], torch.from_numpy(g["own_mel_postnet"])) > 1e-2


# ------------------------------------------------------------------------------------------------ pipeline
def test_convert_utterances_adain_vs_oracle():
    from autoformer_b200 import pipeline
    m, sd = _model("fp32", seed=5)
    lens = [40, 64, 17, 96, 70]
    mels = [synthetic_mel(1, n, 20 + i)[0] for i, n in enumerate(lens)]
    c_org, c_trg = synthetic_speaker(len(lens), 6, "org"), synthetic_speaker(len(lens), 6, "trg")
    outs = pipeline.convert_utterances(m, [t.to(DEV) for t in mels], c_org.to(DEV), c_trg.to(DEV), max_batch=3)
    for i, (mel, o) in enumerate(zip(mels, outs)):
        x, _ = pipeline.pad_to_multiple(mel[None], ARGS[3])
        ref = autovc2_forward(sd, x, c_org[i:i + 1], c_trg[i:i + 1], ARGS[0], ARGS[3], dtype=torch.float64)
        assert o.shape == (lens[i], 80) and rel_l2(o, ref[1].squeeze(1)[0, :lens[i]]) < 3e-4, i


def test_convert_batches_pairs_adain_batches_bit_equal():
    from autoformer_b200 import ops, pipeline
    m, _ = _model("fp16x2")
    shapes = [(100, 64), (80, 96)]                  # two under-filled batches: they run side by side on two streams
    batches = [_on_dev(synthetic_mel(Bn, Tn, 7 + i), synthetic_speaker(Bn, i, "org"), synthetic_speaker(Bn, i, "trg"))
               for i, (Bn, Tn) in enumerate(shapes)]
    alone = [tuple(t.clone() for t in m(*b)) for b in batches]
    got = pipeline.convert_batches(m, batches)
    torch.cuda.synchronize()
    assert ops.LSTM_CTA_BUDGET is None
    for a, g in zip(alone, got):
        for p, q in zip(a, g):
            assert torch.equal(p, q)
