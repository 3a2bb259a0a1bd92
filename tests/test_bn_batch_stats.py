"""Batch-statistics BatchNorm (``bn_stats = "batch"``) without a GPU: the oracle's ``batchnorm_train`` against torch's
own ``nn.BatchNorm1d`` in training mode, and the host logic of the models -- plan caching, buffer updates, mode
switches, ``convert_batches`` ordering, the single-value error -- through CPU stand-ins of the kernels."""
import warnings

import pytest
import torch

from oracle import rel_l2, templates
from oracle.autovc import autovc_forward
from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker
from tests.bn_oracle import batch_statistics, batchnorm_train
from tests.emulate import install_cpu_kernels

warnings.filterwarnings("ignore", category=FutureWarning)


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("momentum", [0.1, None])
@pytest.mark.parametrize("B,C,L", [(2, 5, 7), (1, 3, 2), (4, 16, 1)])
def test_batchnorm_train_matches_torch_over_three_calls(momentum, B, C, L):
    torch.manual_seed(0)
    bn = torch.nn.BatchNorm1d(C, momentum=momentum).double().train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.normal_(0.0, 0.2)
        bn.running_mean.normal_(0.0, 0.5)
        bn.running_var.uniform_(0.5, 2.0)
    sd = {f"bn.{k}": v.clone() for k, v in bn.state_dict().items()}
    for call in range(3):
        x = torch.randn(B, C, L, dtype=torch.float64) * (1 + call) + call
        want = bn(x)
        got = batchnorm_train(sd, "bn", x, eps=bn.eps, momentum=momentum)
        assert torch.allclose(got, want, rtol=1e-12, atol=1e-12), call
        assert torch.allclose(sd["bn.running_mean"], bn.running_mean, rtol=1e-12, atol=1e-14), call
        assert torch.allclose(sd["bn.running_var"], bn.running_var, rtol=1e-12, atol=1e-14), call
        assert int(sd["bn.num_batches_tracked"]) == int(bn.num_batches_tracked) == call + 1


def test_batchnorm_train_single_value_raises_and_leaves_buffers():
    bn = torch.nn.BatchNorm1d(4).train()
    sd = dict(("bn." + k, v.clone()) for k, v in bn.state_dict().items())
    before = {k: v.clone() for k, v in sd.items()}
    with pytest.raises(ValueError, match="more than 1 value per channel"):
        batchnorm_train(sd, "bn", torch.randn(1, 4, 1))
    for k, v in before.items():
        assert torch.equal(sd[k], v)
    with pytest.raises(ValueError, match="more than 1 value per channel"):
        bn(torch.randn(1, 4, 1))                                  # torch's own message
    assert torch.equal(bn.running_mean, before["bn.running_mean"]) and torch.equal(bn.running_var, before["bn.running_var"])


def test_batchnorm_train_never_writes_the_callers_tensors():
    """The oracle replaces buffers in its dict: a state_dict sharing storage with a live module stays untouched."""
    bn = torch.nn.BatchNorm1d(3)
    sd = {"bn." + k: v for k, v in bn.state_dict().items()}      # shares storage with bn's buffers
    batchnorm_train(sd, "bn", torch.randn(2, 3, 5))
    assert int(bn.num_batches_tracked) == 0 and torch.equal(bn.running_mean, torch.zeros(3))
    assert int(sd["bn.num_batches_tracked"]) == 1


def test_oracle_default_is_eval_and_batch_writes_buffers_back():
    args = (32, 256, 512, 32)
    sd = seeded_state_dict(templates.autovc_template(*args), 0)
    keep = {k: v.clone() for k, v in sd.items()}
    x, c_org, c_trg = synthetic_mel(2, 32, 5), synthetic_speaker(2, 5, "org"), synthetic_speaker(2, 5, "trg")
    autovc_forward(sd, x, c_org, c_trg, 32, 32, dtype=torch.float64)
    assert all(sd[k] is not None and torch.equal(sd[k], v) for k, v in keep.items())     # eval: nothing written back
    with batch_statistics():
        autovc_forward(sd, x, c_org, c_trg, 32, 32, dtype=torch.float64)
    n_bn = sum(k.endswith("num_batches_tracked") for k in sd)
    assert n_bn == 11 and all(int(sd[k]) == 1 for k in sd if k.endswith("num_batches_tracked"))
    assert all(sd[k].dtype == torch.float64 for k in sd if k.endswith("running_mean"))
    assert rel_l2(sd["postnet.convolutions.0.1.running_var"], keep["postnet.convolutions.0.1.running_var"]) > 1e-3
    import oracle.adain
    import oracle.layers
    import oracle.meta
    from oracle.layers import batchnorm_eval, cast_state_dict
    assert oracle.layers.batchnorm_eval is batchnorm_eval and oracle.meta.batchnorm_eval is batchnorm_eval
    assert oracle.adain.batchnorm_eval is batchnorm_eval and oracle.meta.cast_state_dict is cast_state_dict


def test_batch_statistics_reaches_through_nested_copies():
    """meta_adjust_forward copies the state_dict and meta_forward copies it again: the Adjust buffers (two calls) and
    the Meta buffers (one call) still come back to the caller."""
    from oracle.adjust import meta_adjust_forward
    args = (44, 256, 512, 22)
    sd = seeded_state_dict(templates.meta_adjust_template("conv", *args), 3)
    x, xt = synthetic_mel(1, 176, 7), synthetic_mel(1, 176, 8)
    with batch_statistics():
        meta_adjust_forward(sd, "conv", x, synthetic_speaker(1, 7, "org"), synthetic_speaker(1, 7, "trg"), 44, 22, True, xt)
    counts = {k: int(v) for k, v in sd.items() if k.endswith("num_batches_tracked")}
    assert counts and all(n == (2 if k.startswith("adjust.") else 1) for k, n in counts.items()), counts


# ------------------------------------------------------------------------------------------------ host logic (CPU stand-ins)
def _emu_bn_batch_stats(v, gamma, beta, eps=1e-5, momentum=0.1, running_mean=None, running_var=None,
                        num_batches_tracked=None, scale_shift=None):
    """avc_bn_batch_stats in fp64 torch: the kernel's contract (include/avc_b200.h)."""
    rows, C = v.shape
    if rows <= 1:
        raise ValueError(f"Expected more than 1 value per channel when training, got input size {(rows, C)}")
    vd = v.double()
    mean, var = vd.mean(0), vd.var(0, unbiased=False)
    scale = gamma.double() / torch.sqrt(var + eps)
    if running_mean is not None:
        num_batches_tracked += 1
        m = 1.0 / float(num_batches_tracked) if momentum is None else momentum
        running_mean.copy_((1 - m) * running_mean.double() + m * mean)
        running_var.copy_((1 - m) * running_var.double() + m * var * (rows / (rows - 1)))
    return torch.stack([scale, beta.double() - mean * scale]).float()


def _emu_bn_apply(v, scale_shift, B, T, act="none", out=None, out2=None, residual=None, res_after=False, out_fmt=None,
                  round_tf32=True):
    from autoformer_b200 import packing
    C = v.shape[1]
    y = v * scale_shift[0] + scale_shift[1]
    if residual is not None and not res_after:
        y = y + residual[:, :C]
    y = {"none": lambda t: t, "relu": torch.relu, "tanh": torch.tanh}[act](y)
    if residual is not None and res_after:
        y = y + residual[:, :C]
    if out2 is not None:
        out2[:, :C] = y
    if out is not None:
        o = packing.to_act(y.view(B, T, C), out_fmt)
        out[:, :T, :o.shape[2]] = o
    return out if out is not None else out2


@pytest.fixture
def cpu_kernels(monkeypatch):
    from autoformer_b200 import ops
    install_cpu_kernels(monkeypatch)
    monkeypatch.setattr(ops, "bn_batch_stats", _emu_bn_batch_stats)
    monkeypatch.setattr(ops, "bn_apply", _emu_bn_apply)


def _autovc(args=(32, 256, 512, 32), seed=0, cls=None):
    from autoformer_b200.factory.AutoVC import AutoVC
    sd = seeded_state_dict(templates.autovc_template(*args), seed)
    m = (cls or AutoVC)(*args)
    m.load_state_dict(sd)
    return m, sd


def _bn_buffers(sd):
    return {k: v for k, v in sd.items() if k.rsplit(".", 1)[-1] in ("running_mean", "running_var", "num_batches_tracked")}


def test_autovc_batch_mode_host_logic(cpu_kernels, monkeypatch):
    """Outputs and every BN buffer against the fp64 oracle in batch mode, the plan built once over three forwards
    (a counting builder), then back to "running" with the updated buffers, bit for bit a fresh model's output."""
    from autoformer_b200.factory import AutoVC as autovc_mod
    builds = []
    real = autovc_mod._Plan
    monkeypatch.setattr(autovc_mod, "_Plan", lambda *a, **k: builds.append(a[2:]) or real(*a, **k))
    m, sd = _autovc()
    m.bn_stats = "batch"
    x, c_org, c_trg = synthetic_mel(2, 64, 5), synthetic_speaker(2, 5, "org"), synthetic_speaker(2, 5, "trg")
    ref_sd = dict(sd)
    for call in range(3):
        out = m(x * (1 + 0.1 * call), c_org, c_trg)
        with batch_statistics():
            ref = autovc_forward(ref_sd, x * (1 + 0.1 * call), c_org, c_trg, 32, 32, dtype=torch.float64)
        for a, b in zip(out, ref):
            # batch statistics re-amplify every conv output to unit scale: on these seeded weights a 1e-6 relative
            # change of the input moves the fp64 mel_postnet by 5e-5 (1e-7 with running statistics), so the stand-ins'
            # fp32-grade GEMMs land at ~4e-4 instead of ~1e-5
            assert rel_l2(a, b) < 1e-3, call
    assert len(builds) == 1 and builds[0][0] is m                # one batch-mode plan, bound to the live module
    live = _bn_buffers(m.state_dict())
    assert len(live) == 33
    for k, v in live.items():
        if k.endswith("num_batches_tracked"):
            assert int(v) == 3, k
        else:
            assert rel_l2(v, ref_sd[k]) < 1e-4, k
    # back to running statistics: re-packed once, with the updated buffers
    m.bn_stats = "running"
    m.eval()
    got = m(x, c_org, c_trg)
    assert len(builds) == 2 and builds[1][0] is None
    fresh, _ = _autovc()
    fresh.load_state_dict(m.state_dict())
    fresh.eval()
    for a, b in zip(got, fresh(x, c_org, c_trg)):
        assert torch.equal(a, b)
    # frozen: a batch-mode forward between two running-mode forwards still re-packs the running plan
    m.freeze_weights()
    m.bn_stats = "batch"
    m(x, c_org, c_trg)
    m.bn_stats = "running"
    got = m(x, c_org, c_trg)
    fresh.load_state_dict(m.state_dict())
    for a, b in zip(got, fresh(x, c_org, c_trg)):
        assert torch.equal(a, b)


def test_plan_cache_key_excludes_bn_buffers_only_in_batch_mode():
    from autoformer_b200 import layers
    m, _ = _autovc()
    count = []
    builder = lambda: count.append(1) or object()
    cache = layers.PlanCache()
    for i in range(3):
        cache.get(m, ("fp32", "batch"), builder, skip_bn_stats=True)
        m.encoder.convolutions[0][1].running_mean.add_(1.0)      # what a batch-mode forward does
        m.encoder.convolutions[0][1].num_batches_tracked.add_(1)
    assert len(count) == 1
    with torch.no_grad():
        m.encoder.convolutions[0][1].weight.mul_(1.5)            # a real weight change still re-packs
    cache.get(m, ("fp32", "batch"), builder, skip_bn_stats=True)
    assert len(count) == 2
    cache.get(m, ("fp32", "running"), builder)                   # running mode keys on the buffers
    m.encoder.convolutions[0][1].running_var.add_(1.0)
    cache.get(m, ("fp32", "running"), builder)
    assert len(count) == 4


def test_adjust_runs_twice_and_governed_by_the_model(cpu_kernels):
    from autoformer_b200.factory.AutoVC_Adjust import AutoVC_Adjust
    from oracle.adjust import autovc_adjust_forward
    args = (32, 256, 512, 32)
    sd = seeded_state_dict(templates.autovc_adjust_template(*args), 3)
    m = AutoVC_Adjust(*args)
    m.load_state_dict(sd)
    m.bn_stats = "batch"
    x, xt = synthetic_mel(2, 32, 7), synthetic_mel(2, 32, 8)
    c_org, c_trg = synthetic_speaker(2, 7, "org"), synthetic_speaker(2, 7, "trg")
    out = m(x, c_org, c_trg, True, xt)
    ref_sd = dict(sd)
    with batch_statistics():
        ref = autovc_adjust_forward(ref_sd, x, c_org, c_trg, 32, 32, True, xt, dtype=torch.float64)
    for a, b in zip(out, ref):
        assert rel_l2(a, b) < 1e-3                               # see test_autovc_batch_mode_host_logic
    for k, v in _bn_buffers(m.state_dict()).items():
        if k.endswith("num_batches_tracked"):
            assert int(v) == (2 if k.startswith("adjust.") else 1), k
        else:
            assert rel_l2(v, ref_sd[k]) < 1e-4, k


def test_convert_batches_runs_batch_mode_in_order(cpu_kernels, monkeypatch):
    from autoformer_b200 import ops, pipeline
    monkeypatch.setattr(pipeline, "_side_streams", lambda dev: pytest.fail("batch mode must not use side streams"))
    a, _ = _autovc()
    b, _ = _autovc()
    a.bn_stats = b.bn_stats = "batch"
    batches = [(synthetic_mel(B, 32, s), synthetic_speaker(B, s, "org"), synthetic_speaker(B, s, "trg"))
               for s, B in ((1, 100), (2, 100), (3, 2))]
    got = pipeline.convert_batches(a, batches)
    want = [b(*bt) for bt in batches]
    assert ops.LSTM_CTA_BUDGET is None
    for u, v in zip(got, want):
        for s, t in zip(u, v):
            assert torch.equal(s, t)
    for (k, s), t in zip(a.state_dict().items(), b.state_dict().values()):
        assert torch.equal(s, t), k


def test_single_value_per_channel_raises_before_any_work(cpu_kernels):
    m, _ = _autovc(args=(32, 256, 512, 1))
    m.bn_stats = "batch"
    before = {k: v.clone() for k, v in m.state_dict().items()}
    with pytest.raises(ValueError, match="more than 1 value per channel"):
        m(synthetic_mel(1, 1, 3), synthetic_speaker(1, 3, "org"), synthetic_speaker(1, 3, "trg"))
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k]), k
    m.bn_stats = "running"
    m(synthetic_mel(1, 1, 3), synthetic_speaker(1, 3, "org"), synthetic_speaker(1, 3, "trg"))     # eval: fine


def test_bn_stats_rejects_unknown_modes(cpu_kernels):
    m, _ = _autovc()
    m.bn_stats = "train"
    with pytest.raises(ValueError, match="bn_stats"):
        m(synthetic_mel(1, 32, 3), synthetic_speaker(1, 3, "org"), synthetic_speaker(1, 3, "trg"))
