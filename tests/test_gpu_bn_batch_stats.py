"""Batch-statistics BatchNorm on the B200: the two kernels element by element against fp64 (avc_bn_batch_stats,
avc_bn_apply), the nine BatchNorm models in ``bn_stats = "batch"`` against the fp64 oracle in batch mode, and the
controls (batch vs running, batch coupling, reproducibility, mode switches, convert_batches, the single-value error)."""
import warnings

import pytest
import torch

from oracle import rel_l2, templates
from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker
from tests.bn_oracle import batch_statistics

warnings.filterwarnings("ignore", category=FutureWarning)
pytestmark = pytest.mark.gpu


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32).cpu()


# ------------------------------------------------------------------------------------------------ op level: statistics
def _stats_ref(v, gamma, beta, eps, momentum, rm, rv, nbt):
    vd = v.double().cpu()
    n = vd.shape[0]
    mean, var = vd.mean(0), vd.var(0, unbiased=False)
    scale = gamma.double().cpu() / torch.sqrt(var + eps)
    count = int(nbt) + 1
    m = 1.0 / count if momentum is None else momentum
    return (torch.stack([scale, beta.double().cpu() - mean * scale]), (1 - m) * rm.double().cpu() + m * mean,
            (1 - m) * rv.double().cpu() + m * var * n / (n - 1), count)


@pytest.mark.parametrize("C", [80, 176, 344, 512])
@pytest.mark.parametrize("rows", [2, 33, 1000 + 7, 2 * 176 + 5, 65536 + 3])
@pytest.mark.parametrize("momentum", [0.1, 1.0, None])
def test_bn_batch_stats_against_fp64(C, rows, momentum):
    from autoformer_b200 import ops
    g = torch.Generator().manual_seed(C * 7 + rows)
    v = torch.randn(rows, C + 4, generator=g) * torch.rand(C + 4, generator=g) * 3 + torch.randn(C + 4, generator=g)
    v[:, 1] = 1000.0 + 1.0 * torch.randn(rows, generator=g)       # |mean| ~ 1e3 std: cancellation in E[v^2] - mean^2
    v = v.cuda()[:, :C]                                            # row stride C + 4: a view, as the layers never pass
    gamma, beta = (torch.rand(C, generator=g) + 0.5).cuda(), (torch.randn(C, generator=g) * 0.2).cuda()
    rm, rv = (torch.randn(C, generator=g) * 0.5).cuda(), (torch.rand(C, generator=g) * 1.5 + 0.5).cuda()
    nbt = torch.tensor(4, dtype=torch.int64).cuda()
    want_ss, want_rm, want_rv, want_n = _stats_ref(v, gamma, beta, 1e-5, momentum, rm, rv, nbt)
    rm0, rv0, nbt0 = rm.clone(), rv.clone(), nbt.clone()
    ss = ops.bn_batch_stats(v, gamma, beta, 1e-5, momentum, rm, rv, nbt)
    # fp32 results of fp64 arithmetic: a few fp32 ulps
    assert torch.allclose(ss.cpu().double(), want_ss, rtol=2e-6, atol=1e-6), (ss.cpu().double() - want_ss).abs().max()
    assert torch.allclose(rm.cpu().double(), want_rm, rtol=2e-6, atol=1e-6)
    assert torch.allclose(rv.cpu().double(), want_rv, rtol=2e-6, atol=1e-6)
    assert int(nbt) == want_n
    # the same call again on the same inputs: the same bits (fixed reduction order)
    rm2, rv2, nbt2 = rm0.clone(), rv0.clone(), nbt0.clone()
    ss2 = ops.bn_batch_stats(v, gamma, beta, 1e-5, momentum, rm2, rv2, nbt2)
    assert torch.equal(_bits(ss), _bits(ss2)) and torch.equal(_bits(rm), _bits(rm2)) and torch.equal(_bits(rv), _bits(rv2))


def test_bn_batch_stats_without_buffers_and_errors():
    from autoformer_b200 import ops
    v = torch.randn(50, 16, device="cuda")
    g, b = torch.ones(16, device="cuda"), torch.zeros(16, device="cuda")
    ss = ops.bn_batch_stats(v, g, b)
    ref = torch.stack([1 / torch.sqrt(v.double().var(0, unbiased=False) + 1e-5), -v.double().mean(0) / torch.sqrt(v.double().var(0, unbiased=False) + 1e-5)])
    assert torch.allclose(ss.double(), ref, rtol=2e-6, atol=1e-6)
    with pytest.raises(ValueError, match="more than 1 value per channel"):
        ops.bn_batch_stats(v[:1], g, b)


# ------------------------------------------------------------------------------------------------ op level: apply
SPARE_ROWS, SPARE_CH = 3, 8
FMT = {0: "tf32", 1: "bf16", 2: "fp32", 3: "fp16x2", 4: "fp16s"}


@pytest.mark.parametrize("act", ["none", "relu", "tanh"])
@pytest.mark.parametrize("res", [None, "before", "after"])
@pytest.mark.parametrize("dtype", [0, 1, 2, 3, 4])
def test_bn_apply_every_path(act, res, dtype):
    from autoformer_b200 import ops, packing
    from autoformer_b200.packing import TORCH_DTYPE
    B, T, C = 3, 37, 176
    fmt = FMT[dtype]
    g = torch.Generator().manual_seed(dtype * 9 + (res is not None))
    v = (torch.randn(B * T, C, generator=g) * 3).cuda()
    ss = torch.stack([torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)]).cuda()
    resid = (torch.randn(B * T, C + SPARE_CH, generator=g)).cuda()[:, :C] if res else None
    Cp = packing.act_channels(C, fmt)
    out = torch.full((B, T + SPARE_ROWS, Cp + SPARE_CH), float("nan"), dtype=TORCH_DTYPE[fmt], device="cuda")
    out2 = torch.full((B * T + SPARE_ROWS, C + SPARE_CH), float("nan"), device="cuda")
    ops.bn_apply(v, ss, B, T, act, out=out, out2=out2[:B * T], residual=resid, res_after=res == "after", out_fmt=fmt)
    y = v.double() * ss[0].double() + ss[1].double()
    if res == "before":
        y = y + resid.double()
    y = {"none": lambda t: t, "relu": torch.relu, "tanh": torch.tanh}[act](y)
    if res == "after":
        y = y + resid.double()
    # out2: fp32 arithmetic (fma + one residual add) and the GEMM epilogue's tanh (~1e-7 absolute)
    got2 = out2[:B * T, :C]
    assert (got2.double() - y).abs().max() < 2e-6 * (1 + y.abs().max()), (got2.double() - y).abs().max()
    # writes exactly the region: spare rows / channels still NaN
    assert torch.isnan(out2[B * T:]).all() and torch.isnan(out2[:, C:]).all() and torch.isfinite(got2).all()
    assert torch.isnan(out[:, T:].float()).all() and torch.isnan(out[:, :, Cp:].float()).all()
    # out: bit for bit the host conversion of out2 (the GEMM epilogue's stores)
    assert torch.equal(_bits(out[:, :T, :Cp]), _bits(packing.to_act(got2.reshape(B, T, C).cpu(), fmt)))


# ------------------------------------------------------------------------------------------------ model level
AUTOVC_ARGS = (32, 256, 512, 32)
META_ARGS = (44, 256, 512, 22)
# Output gates.  Batch statistics make the forward far less well conditioned than the eval-mode one: every BatchNorm
# rescales its conv output to unit variance, so relative errors are re-amplified layer after layer.  On these seeded
# weights a 1e-6 relative change of the input moves the fp64 AutoVC mel_postnet by 5e-5 in batch mode against 1e-7 with
# running statistics (tests/test_bn_batch_stats.py notes the same on the CPU stand-ins, whose statistics are exact fp64).
# The Meta and Adjust families' fp32 runs still meet their eval-mode gates (1e-3, 3e-4); the gates below are the B200
# measurements (NVIDIA B200, 1000 W power limit) with ~1.5x headroom where a family's eval-mode gate is exceeded:
#   fp32:   AutoVC 2.9e-4 (eval gate 2e-4), AutoVC2 3.5e-4 (3e-4), AutoVC_Adjust < 3e-4, Meta* <= 8.5e-5
#   fp16x2: AutoVC-based 1.0e-2 .. 2.4e-2 (eval gate 1e-3: fp16 activations carry 4.9e-4 rounding into the amplification),
#           Meta-based 2.1e-3 .. 2.7e-3 (eval gate 1.5e-3)
# The kernels themselves are gated element by element above; these gates check the plumbing, not the arithmetic.
OUT_TOL = {"fp32": {"autovc": 4e-4, "adjust": 3e-4, "adain": 5e-4, "meta": 1e-3},
           "fp16x2": {"autovc": 3.5e-2, "meta": 4e-3}}
# BN buffers after the forward, relative L2 against the fp64 oracle's: the estimates this feature started from; the
# B200 run measured at most 1.9e-5 (fp32) and 2.8e-4 (fp16x2) on the cases it printed
BUF_TOL = {"fp32": 1e-4, "fp16x2": 2e-3}


def _out_tol(name, family, precision):
    if precision == "fp32":
        return OUT_TOL["fp32"][family]
    return OUT_TOL["fp16x2"]["meta" if name.startswith("Meta") else "autovc"]


def _build(name):
    from autoformer_b200.factory.AutoVC import AutoVC
    from autoformer_b200.factory.AutoVC2 import AutoVC2
    from autoformer_b200.factory.AutoVC_Adjust import AutoVC_Adjust
    from autoformer_b200.factory.MetaConv import MetaConv
    from autoformer_b200.factory.MetaConv2 import MetaConv2
    from autoformer_b200.factory.MetaConv_Adjust import MetaConv_Adjust
    from autoformer_b200.factory.MetaPool import MetaPool
    from autoformer_b200.factory.MetaPool2 import MetaPool2
    from autoformer_b200.factory.MetaPool_Adjust import MetaPool as MetaPool_Adjust
    from oracle.adain import autovc2_forward, meta2_forward
    from oracle.adjust import autovc_adjust_forward, meta_adjust_forward
    from oracle.autovc import autovc_forward
    from oracle.meta import meta_forward
    T = templates
    table = {
        "AutoVC": (AutoVC, AUTOVC_ARGS, T.autovc_template, "autovc",
                   lambda sd, x, xt, co, ct, taps: autovc_forward(sd, x, co, ct, 32, 32, torch.float64, taps)),
        "AutoVC_Adjust": (AutoVC_Adjust, AUTOVC_ARGS, T.autovc_adjust_template, "adjust",
                          lambda sd, x, xt, co, ct, taps: autovc_adjust_forward(sd, x, co, ct, 32, 32, True, xt,
                                                                                torch.float64)),
        "AutoVC2": (AutoVC2, AUTOVC_ARGS, T.autovc2_template, "adain",
                    lambda sd, x, xt, co, ct, taps: autovc2_forward(sd, x, co, ct, 32, 32, None, torch.float64)),
    }
    for kind, cls, cls2, clsa in (("pool", MetaPool, MetaPool2, MetaPool_Adjust), ("conv", MetaConv, MetaConv2, MetaConv_Adjust)):
        k = kind
        table["Meta" + kind.capitalize()] = (cls, META_ARGS, lambda *a, k=k: T.meta_template(k, *a), "meta",
                                             lambda sd, x, xt, co, ct, taps, k=k: meta_forward(sd, x, co, ct, 44, 22, k, torch.float64, taps))
        table["Meta" + kind.capitalize() + "2"] = (cls2, META_ARGS, lambda *a, k=k: T.meta2_template(k, *a), "adain",
                                                   lambda sd, x, xt, co, ct, taps, k=k: meta2_forward(sd, k, x, co, ct, 44, 22, None, torch.float64))
        table["Meta" + kind.capitalize() + "_Adjust"] = (clsa, META_ARGS, lambda *a, k=k: T.meta_adjust_template(k, *a), "adjust",
                                                         lambda sd, x, xt, co, ct, taps, k=k: meta_adjust_forward(sd, k, x, co, ct, 44, 22, True, xt, torch.float64))
    return table[name]


MODELS = ["AutoVC", "AutoVC_Adjust", "AutoVC2", "MetaPool", "MetaConv", "MetaPool2", "MetaConv2", "MetaPool_Adjust",
          "MetaConv_Adjust"]


def _case(name, B, pad):
    cls, args, tpl, family, oracle = _build(name)
    sd = seeded_state_dict(tpl(*args), 11)
    T = 128 if args == AUTOVC_ARGS else 176
    x, xt = synthetic_mel(B, T, 41), synthetic_mel(B, T, 42)
    if pad:
        x[-1, T - pad:] = 0.0                                     # the Evaluator's zero padding to len_crop
    co, ct = synthetic_speaker(B, 41, "org"), synthetic_speaker(B, 41, "trg")
    return cls, args, sd, family, oracle, (x, xt, co, ct)


def _run(m, name, x, xt, co, ct):
    if name.endswith("_Adjust"):
        return m(x, co, ct, True, xt)
    return m(x, co, ct)


@pytest.mark.parametrize("precision", ["fp32", "fp16x2"])
@pytest.mark.parametrize("name,B,pad", [(n, 2, 0) for n in MODELS] + [("MetaPool", 1, 0), ("MetaConv_Adjust", 1, 0),
                                                                     ("AutoVC", 2, 40), ("MetaConv", 2, 70)])
def test_batch_mode_model_against_oracle(name, B, pad, precision):
    cls, args, sd, family, oracle, (x, xt, co, ct) = _case(name, B, pad)
    m = cls(*args)
    m.load_state_dict(sd)
    m = m.cuda()
    m.precision, m.bn_stats, m.collect_taps = precision, "batch", True
    out = _run(m, name, x.cuda(), xt.cuda(), co.cuda(), ct.cuda())
    ref_sd, rt = dict(sd), {}
    with batch_statistics():
        ref = oracle(ref_sd, x, xt, co, ct, rt)
    tol = _out_tol(name, family, precision)
    errs = [rel_l2(a, b) for a, b in zip(out, ref)]
    print(name, B, pad, precision, "outputs rel-L2:", ["%.2e" % e for e in errs])
    worst_stage = 0.0
    for k, v in rt.items():                                       # staged taps (AutoVC and Meta forwards record them)
        if k in m.taps:
            got = m.taps[k]
            want = v if got.shape == v.shape else v.transpose(1, 2)
            worst_stage = max(worst_stage, rel_l2(got, want))
    worst_buf, counts = 0.0, {}
    for k, v in m.state_dict().items():
        if k.endswith("num_batches_tracked"):
            counts[k] = int(v)
        elif k.endswith(("running_mean", "running_var")):
            worst_buf = max(worst_buf, rel_l2(v, ref_sd[k]))
    print("   worst stage rel-L2 %.2e, worst BN buffer rel-L2 %.2e" % (worst_stage, worst_buf))
    assert all(e < tol for e in errs), errs
    assert worst_stage < 1.5 * tol
    assert worst_buf < BUF_TOL[precision]
    assert counts and all(n == int(ref_sd[k]) for k, n in counts.items())
    assert all(n == (2 if k.startswith("adjust.") and name != "MetaPool_Adjust" else 1) for k, n in counts.items()), counts


# ------------------------------------------------------------------------------------------------ controls
def _autovc(sd=None, precision="fp32"):
    from autoformer_b200.factory.AutoVC import AutoVC
    sd = sd or seeded_state_dict(templates.autovc_template(*AUTOVC_ARGS), 11)
    m = AutoVC(*AUTOVC_ARGS)
    m.load_state_dict(sd)
    m = m.cuda()
    m.precision = precision
    return m


def _inputs(B=2, T=128, seed=41):
    return (synthetic_mel(B, T, seed).cuda(), synthetic_speaker(B, seed, "org").cuda(),
            synthetic_speaker(B, seed, "trg").cuda())


def test_batch_and_running_differ_and_batch_couples_utterances():
    m = _autovc()
    x, co, ct = _inputs()
    run = m(x, co, ct)[1]
    m.bn_stats = "batch"
    bat = m(x, co, ct)[1]
    assert rel_l2(bat, run) > 0.1
    x2 = x.clone()
    x2[1] = synthetic_mel(1, 128, 99).cuda()[0]
    assert rel_l2(m(x2, co, ct)[1][0], bat[0]) > 1e-4           # utterance 0 depends on utterance 1


def test_batch_mode_is_reproducible_bit_for_bit():
    for precision in ("fp32", "fp16x2"):
        a, b = _autovc(precision=precision), _autovc(precision=precision)
        a.bn_stats = b.bn_stats = "batch"
        x, co, ct = _inputs()
        for u, v in zip(a(x, co, ct), b(x, co, ct)):
            assert torch.equal(u, v)
        for (k, u), v in zip(a.state_dict().items(), b.state_dict().values()):
            assert torch.equal(u, v), k


@pytest.mark.parametrize("frozen", [False, True])
def test_back_to_running_uses_the_updated_buffers(frozen):
    m = _autovc()
    x, co, ct = _inputs()
    if frozen:
        m.freeze_weights()
    m(x, co, ct)                                                  # running plan packed (and frozen)
    m.bn_stats = "batch"
    m(x, co, ct)
    m(x * 0.5, co, ct)
    m.bn_stats = "running"
    got = m(x, co, ct)
    fresh = _autovc({k: v.cpu() for k, v in m.state_dict().items()})
    for u, v in zip(got, fresh(x, co, ct)):
        assert torch.equal(u, v)


def test_convert_batches_in_batch_mode_equals_a_loop():
    from autoformer_b200 import pipeline
    a, b = _autovc(), _autovc()
    a.bn_stats = b.bn_stats = "batch"
    batches = [_inputs(100, 64, s) for s in (3, 4)] + [_inputs(70, 64, 5)]    # 64 < B <= 256: would be paired
    got = pipeline.convert_batches(a, batches)
    want = [b(*bt) for bt in batches]
    for u, v in zip(got, want):
        for s, t in zip(u, v):
            assert torch.equal(s, t)
    for (k, s), t in zip(a.state_dict().items(), b.state_dict().values()):
        assert torch.equal(s, t), k


def test_single_value_per_channel_raises_and_leaves_buffers():
    from autoformer_b200.factory.AutoVC import AutoVC
    m = AutoVC(32, 256, 512, 1)
    m.load_state_dict(seeded_state_dict(templates.autovc_template(32, 256, 512, 1), 11))
    m = m.cuda()
    m.bn_stats = "batch"
    before = {k: v.clone() for k, v in m.state_dict().items()}
    with pytest.raises(ValueError, match="more than 1 value per channel"):
        m(*_inputs(1, 1))
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k]), k
