"""Op-level contract of the MetaPool / MetaConv / AdaIN glue kernels (csrc/avc_meta.cu), element by element.

The nine entry points are called through the C ABI so that every output is a NaN-filled buffer with a spare utterance
(and a spare stats slot): exactly the expected region may become finite.  Every operand format is stored: out_dtype 0
(TF32-rounded and raw), 1 bf16, 2 split bf16, 3 fp16.

The elementwise kernels are teacher-forced: they get fp32 statistics rounded from fp64, and each result is held to a
per-element worst-case bound of a few 2^-24 times the sum of the magnitudes of its terms (constant derived per
operation below), plus half an ulp of the stored format.  fp16 stores must saturate at +-65504 as packing.to_act does.
Data movement (patchify without statistics, the transposed copies, decoder input, code gathering) must be bit-exact.

LayerNorm statistics (avc_ln_transpose's scratch) are held to a bound linear in |mean| / std,
(ceil(n / G) + log2 G + 3) 2^-24 (max|x| rstd + 1) on the normalised value, G the number of partial Welford chains
(32 lanes per row, 8 row groups per column).  A single-pass E[x^2] - mean^2 misses it from |mean| / std = 10 on.
The CPU tests at the bottom check the checkers: correct stand-ins pass, faulty ones fail.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import emulate
from tests.test_gpu_kernel_contract import _special_values, check_bound, check_sentinel, half_ulp, nan_buf

u = 2.0 ** -24
FP16_MAX = 65504.0
# (packing format, out_dtype, out_round_tf32)
FORMATS = [("tf32", 0, 1), ("tf32", 0, 0), ("bf16", 1, 1), ("fp32", 2, 1), ("fp16x2", 3, 1)]
RATIOS = (0.0, 10.0, 100.0, 1000.0)


# ------------------------------------------------------------------------------------------------ references and checks
def decode(buf, fmt):
    from autoformer_b200 import packing
    return packing.act_to_float(buf.cpu(), fmt).double()


def stored(t, fmt, rnd):
    """packing.to_act of fp32 values, or the raw values for out_dtype 0 without TF32 rounding."""
    from autoformer_b200 import packing
    return packing.to_act(t.float(), fmt) if (fmt != "tf32" or rnd) else t.float()


def bits(t):
    t = t.contiguous().cpu()
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def check_stored(got, ref, e, fmt, rnd, what):
    """got (decoded) against the fp64 ref, |kernel fp32 value - ref| <= e, plus the rounding of the stored format.  fp16
    saturates: where even ref - e lies beyond +-65504 the stored value is exactly +-65504."""
    if fmt == "fp16x2":
        big = (ref.abs() - e) > FP16_MAX
        assert torch.equal(got[big], FP16_MAX * ref[big].sign()), f"{what}: fp16 store does not saturate"
        ref = ref.clamp(-FP16_MAX, FP16_MAX)
    check_bound(got, ref, e + half_ulp(ref.abs() + e, fmt, bool(rnd)), what)


def ln_stats_bound(x, G):
    """x [rows][n] fp32 -> fp64 (mean, rstd, bound on |(x - m) r - (x - mean) rstd| for every x of the row)."""
    xd = x.double()
    n = x.shape[1]
    mean = xd.mean(1)
    rstd = 1.0 / torch.sqrt(xd.var(1, unbiased=False) + 1e-5)
    K = -(-n // G) + int(math.log2(G)) + 3
    return mean, rstd, K * u * (xd.abs().amax(1) * rstd + 1.0)


def check_ln_stats(x, st, G, what):
    """st [rows][2] = the kernel's (mean, rstd) of each row of x [rows][n]: the normalised values they give are within
    ln_stats_bound of fp64 LayerNorm's."""
    mean, rstd, bound = ln_stats_bound(x, G)
    xd, st = x.double(), st.double().cpu()
    assert bool(torch.isfinite(st).all()), f"{what}: non-finite statistics"
    err = ((xd - st[:, :1]) * st[:, 1:] - (xd - mean[:, None]) * rstd[:, None]).abs().amax(1)
    bad = err > bound
    if bool(bad.any()):
        i = int(bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {err.numel()} rows beyond the bound; worst "
                             f"{float((err / bound).max()):.3g} x bound; row {i}: err {float(err[i]):.3g}, bound "
                             f"{float(bound[i]):.3g}, |mean|/std {float(mean[i].abs() * rstd[i]):.3g}")
    return float((err / bound).max())


def fp64_moments_bound(x, chain, bessel):
    """fp64 mean, rstd (GroupNorm) or std (bessel) of x [B][n] and the bounds of kernels that accumulate sum x and
    sum x^2 in fp64 along chains of `chain` additions and round the results to fp32."""
    xd = x.double()
    n = x.shape[1]
    mean = xd.mean(1)
    var = xd.var(1, unbiased=bessel)
    A, Q = xd.abs().mean(1), (xd * xd).mean(1)
    e_mean = u * mean.abs() + chain * 2.0 ** -53 * A
    # sum x^2 / n - mean^2: both terms carry chain * 2^-53 relative error (and the mean's error enters twice)
    e_var = 2 * chain * 2.0 ** -53 * (Q + 2 * mean.abs() * A) * (n / (n - 1) if bessel else 1.0)
    return mean, var, e_mean, e_var


def pool_ref(x, rstd, g):
    """gn_pool_residual in fp64 from the kernel's fp32 rstd and its bound: pool = (x[t-1] + x[t] + x[t+1]) / cnt with
    two additions, a rounded 1/cnt, a product; then pool - x, rstd * gamma, the product, + x: <= 10 u (|x| + |rstd
    gamma| (P + |x|)), P the sum of magnitudes of the pooled terms."""
    xd = x.double()
    B, L, C = x.shape
    pool = F.avg_pool1d(xd.transpose(1, 2), 3, stride=1, padding=1, count_include_pad=False).transpose(1, 2)
    P = F.avg_pool1d(xd.abs().transpose(1, 2), 3, stride=1, padding=1, count_include_pad=False).transpose(1, 2)
    cnt = torch.full((L,), 3.0, dtype=torch.float64)
    cnt[0] = cnt[-1] = 2.0
    cnt[:] = torch.minimum(cnt, torch.tensor(float(L)))
    P = P * cnt.view(1, L, 1)
    rg = rstd.double().view(B, 1, 1) * g.double().view(1, 1, C)
    y = xd + rg * (pool - xd)
    e = 10 * u * (xd.abs() + rg.abs() * (P + xd.abs()))
    if L >= 2:        # the end frames average two samples (count_include_pad=False), written out independently
        end = torch.stack([(xd[:, 0] + xd[:, 1]) / 2, (xd[:, -1] + xd[:, -2]) / 2], dim=1)
        assert torch.allclose(pool[:, [0, -1]], end, rtol=0, atol=1e-12)
    return y, e


def affine_ref(x, mean, rstd, g, be):
    """(x - mean) * rstd * g + be in fp64 from fp32 (mean, rstd) and its bound: a subtraction, two products and an
    addition, <= 5 u (|x - mean| |rstd g| + |be|).  mean / rstd / g / be broadcast against x."""
    d = x.double() - mean.double()
    rg = rstd.double() * g.double()
    y = d * rg + be.double()
    return y, 5 * u * (d.abs() * rg.abs() + be.double().abs())


def ln_apply_ref(x, mean, rstd, g, be):
    """ln_transpose's fmaf(x, rstd g, be - mean rstd g) in fp64 from fp32 (mean, rstd) and its bound:
    <= 5 u (|x rstd g| + |mean rstd g| + |be|)."""
    rg = rstd.double() * g.double()
    y = (x.double() - mean.double()) * rg + be.double()
    return y, 5 * u * ((x.double().abs() + mean.double().abs()) * rg.abs() + be.double().abs())


def patchify_perm(img, p):
    """image [B][S][S] (rows h, columns w) -> tokens [B][(S/p)^2][p*p], feature (h % p) * p + w % p."""
    B, S, _ = img.shape
    n = S // p
    return img.reshape(B, n, p, n, p).permute(0, 1, 3, 2, 4).reshape(B, n * n, p * p)


def transposed_padded(y, R8):
    """y [B][R][C] -> [B][C][R8], zero columns [R, R8)."""
    B, R, C = y.shape
    out = torch.zeros(B, C, R8, dtype=y.dtype)
    out[:, :, :R] = y.transpose(1, 2)
    return out


def check_pad_zero(buf, R, R8, fmt, what):
    """Columns [R, R8) of an ln_transpose output are exactly zero, in both halves of a split format."""
    from autoformer_b200 import packing
    buf = buf.cpu().float()
    halves = [buf[..., :R8], buf[..., R8:]] if fmt in packing.SPLIT_ACTS else [buf]
    for h in halves:
        assert bool((h[..., R:R8] == 0).all()), f"{what}: pad columns not zero"


def ln_rows_cols(x, axis):
    """The vectors LayerNorm normalises: [B * R][C] rows on axis 1, [B * C][R] columns on axis 2, and G."""
    B, R, C = x.shape
    if axis == 1:
        return x.reshape(B * R, C), 32
    return x.transpose(1, 2).reshape(B * C, R), 8


def check_ln_outputs(x, g, be, axis, st, out, fmt, rnd, what):
    """out (decoded [B][C][R8]): teacher-forced on the kernel's statistics st [rows][2], then end to end against fp64
    LayerNorm with the statistics bound carried through."""
    B, R, C = x.shape
    st = st.double().cpu()
    if axis == 1:
        m, r = st[:, 0].view(B, R, 1), st[:, 1].view(B, R, 1)
        gg, bb = g.view(1, 1, C), be.view(1, 1, C)
    else:
        m, r = st[:, 0].view(B, 1, C), st[:, 1].view(B, 1, C)
        gg, bb = g.view(1, R, 1), be.view(1, R, 1)
    y, e = ln_apply_ref(x, m, r, gg, bb)
    got = out[:, :, :R].transpose(1, 2)
    check_stored(got, y, e, fmt, rnd, what + " (teacher-forced)")
    v, G = ln_rows_cols(x, axis)
    mean, rstd, sb = ln_stats_bound(v, G)
    if axis == 1:
        mean, rstd, sb = mean.view(B, R, 1), rstd.view(B, R, 1), sb.view(B, R, 1)
    else:
        mean, rstd, sb = mean.view(B, 1, C), rstd.view(B, 1, C), sb.view(B, 1, C)
    y64 = (x.double() - mean) * rstd * gg.double() + bb.double()
    check_stored(got, y64, e + gg.double().abs() * sb, fmt, rnd, what + " (end to end)")


# ------------------------------------------------------------------------------------------------ inputs
def offset_rows(shape, ratios, g, dims=(-1,)):
    """randn with a std per vector spanning `dims` (log-normal) and a mean of +-ratio * std, ratios cycling over the
    vectors."""
    x = torch.randn(*shape, generator=g)
    vshape = list(shape)
    for d in dims:
        vshape[d] = 1
    nv = int(np.prod(vshape))
    sd = torch.exp(torch.randn(nv, generator=g)).view(vshape)
    r = torch.tensor([ratios[i % len(ratios)] for i in range(nv)], dtype=torch.float32).view(vshape)
    sign = torch.where(torch.rand(nv, generator=g) < 0.5, -1.0, 1.0).view(vshape)
    return (x * sd + sign * r * sd).float().contiguous()


def grid_cap_float4():
    """avc_meta.cu grid_for: at most 16 blocks of 256 threads per SM, one float4 per thread and pass."""
    return torch.cuda.get_device_properties(0).multi_processor_count * 16 * 256


def lib():
    from autoformer_b200 import _lib
    return _lib.load()


def call(fn, *args):
    """fn(*args, stream) with tensors passed as device pointers; the argument tuple keeps every tensor (also a
    temporary such as x.cuda()) alive until the launch has finished."""
    from autoformer_b200 import _lib, ops
    ptrs = [a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args]
    _lib.check(fn(*ptrs, ops._stream()), fn.__name__)
    torch.cuda.synchronize()


def fp64_stats(x, B):
    """fp32 (mean, rstd) rounded from fp64 (teacher forcing)."""
    xd = x.double().reshape(B, -1)
    return torch.stack([xd.mean(1), 1.0 / torch.sqrt(xd.var(1, unbiased=False) + 1e-5)], 1).float()


# ------------------------------------------------------------------------------------------------ GroupNorm statistics
@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 4 * 1001, 176 * 512, 344 * 512])
@pytest.mark.parametrize("B", [1, 3, 33])
def test_gn_stats(n, B):
    g = torch.Generator().manual_seed(n + B)
    for ratio in (0.0, 100.0, 1000.0):
        x = offset_rows((B, n), (ratio,), g)
        st = nan_buf((B + 1, 2), torch.float32)
        call(lib().avc_gn_stats, x.cuda(), st, B, n, 1e-5)
        region = torch.zeros(B + 1, 2, dtype=torch.bool)
        region[:B] = True
        check_sentinel(st, region, "gn_stats")
        got = st[:B].double().cpu()
        mean, var, e_mean, e_var = fp64_moments_bound(x, n // 512 + 32, bessel=False)
        rstd = 1.0 / torch.sqrt(var + 1e-5)
        check_bound(got[:, 0], mean, e_mean, f"gn_stats mean ratio {ratio}")
        check_bound(got[:, 1], rstd, rstd * (2 * u + e_var / (var + 1e-5)), f"gn_stats rstd ratio {ratio}")


# ------------------------------------------------------------------------------------------------ pooling mixer / GN apply
GN_SHAPES = [(3, L, C) for L in (1, 2, 3, 176, 344) for C in (4, 176, 512)] + [(33, 344, 512)]


def _gn_inputs(B, L, C, seed):
    g = torch.Generator().manual_seed(seed)
    x = offset_rows((B, L, C), (0.0, 3.0), g, dims=(1, 2))
    first = x[0].view(-1)            # fp16 saturation, in utterance 0 only (it dominates that utterance's statistics)
    first[torch.randint(0, first.numel(), (max(2, first.numel() // 500),), generator=g)] = 1.5e5
    first[torch.randint(0, first.numel(), (max(2, first.numel() // 500),), generator=g)] = -2e5
    gamma = torch.rand(C, generator=g) + 0.5
    beta = torch.randn(C, generator=g) * 0.2
    beta[::7] = 9e4                                                                   # saturates in gn_apply
    return x, fp64_stats(x, B), gamma, beta


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,C", GN_SHAPES, ids=[f"B{b}L{l}C{c}" for b, l, c in GN_SHAPES])
def test_gn_pool_residual(B, L, C):
    from autoformer_b200 import packing
    if B == 33:
        assert B * L * C // 4 > grid_cap_float4()          # the grid-stride loop runs more than one pass
    x, st, gamma, _ = _gn_inputs(B, L, C, B * 1000 + L * 10 + C)
    y, e = pool_ref(x, st[:, 1], gamma)
    xc, stc, gc = x.cuda(), st.cuda(), gamma.cuda()
    f32_region = torch.zeros(B + 1, L, C, dtype=torch.bool)
    f32_region[:B] = True
    f32_alone = None
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(C, fmt)
        op_region = torch.zeros(B + 1, L, ach, dtype=torch.bool)
        op_region[:B] = True
        for want_f32, want_op in ((True, False), (False, True), (True, True)):
            if want_f32 and not want_op and f32_alone is not None:
                continue
            f32 = nan_buf((B + 1, L, C), torch.float32) if want_f32 else None
            op = nan_buf((B + 1, L, ach), packing.TORCH_DTYPE[fmt]) if want_op else None
            call(lib().avc_gn_pool_residual, xc, stc, gc, f32, op, dt, rnd, B, L, C)
            what = f"gn_pool {fmt}/{dt}/{rnd} f32={want_f32} op={want_op}"
            if want_f32:
                check_sentinel(f32, f32_region, what + " out_f32")
                got = f32[:B].double().cpu()
                check_bound(got, y, e, what + " out_f32")
                check_bound(got[:, [0, -1]], y[:, [0, -1]], e[:, [0, -1]], what + " end frames")
                if L == 1:
                    assert torch.equal(f32[:B].cpu(), x), what + ": L = 1 must return x"
                if f32_alone is None:
                    f32_alone = f32[:B].cpu()
                else:
                    assert torch.equal(f32[:B].cpu(), f32_alone), what + ": out_f32 depends on out_op"
            if want_op:
                check_sentinel(op, op_region, what + " out_op")
                got = decode(op[:B], fmt)
                check_stored(got, y, e, fmt, rnd, what + " out_op")
                check_stored(got[:, [0, -1]], y[:, [0, -1]], e[:, [0, -1]], fmt, rnd, what + " end frames")


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,C", GN_SHAPES, ids=[f"B{b}L{l}C{c}" for b, l, c in GN_SHAPES])
def test_gn_apply(B, L, C):
    from autoformer_b200 import packing
    if B == 33:
        assert B * L * C // 4 > grid_cap_float4()
    x, st, gamma, beta = _gn_inputs(B, L, C, B * 2000 + L * 10 + C)
    y, e = affine_ref(x, st[:, 0].view(B, 1, 1), st[:, 1].view(B, 1, 1), gamma, beta)
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(C, fmt)
        op = nan_buf((B + 1, L, ach), packing.TORCH_DTYPE[fmt])
        call(lib().avc_gn_apply, x.cuda(), st.cuda(), gamma.cuda(), beta.cuda(), op, dt, rnd, B, L, C)
        region = torch.zeros(B + 1, L, ach, dtype=torch.bool)
        region[:B] = True
        what = f"gn_apply {fmt}/{dt}/{rnd}"
        check_sentinel(op, region, what)
        check_stored(decode(op[:B], fmt), y, e, fmt, rnd, what)


# ------------------------------------------------------------------------------------------------ patchify
PATCH = [(176, 8), (176, 16), (344, 8), (16, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("S,pp", PATCH, ids=[f"S{s}p{q}" for s, q in PATCH])
def test_patchify(S, pp):
    from autoformer_b200 import packing
    B = 3
    g = torch.Generator().manual_seed(S * pp)
    a = offset_rows((B, S, S), (0.0, 2.0), g, dims=(1, 2))
    a_sp = a.clone()                 # format edges (fp16 saturation, rounding ties, subnormals) for the plain copy
    pick = torch.rand(a.numel(), generator=g) < 0.05
    a_sp.view(-1)[pick] = _special_values(a.numel(), S)[pick]
    st = fp64_stats(a, B)
    gs, bs = torch.rand(S, generator=g) + 0.5, torch.randn(S, generator=g) * 0.2
    bs[::5] = -1e5
    img = a.double().transpose(1, 2)                           # image rows h = channel, columns w = length
    y, e = affine_ref(img, st[:, 0].view(B, 1, 1), st[:, 1].view(B, 1, 1), gs.view(1, S, 1), bs.view(1, S, 1))
    y, e = patchify_perm(y, pp), patchify_perm(e, pp)
    plain = patchify_perm(a_sp.transpose(1, 2), pp).contiguous()
    ntok, F_ = (S // pp) ** 2, pp * pp
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(F_, fmt)
        region = torch.zeros(B + 1, ntok, ach, dtype=torch.bool)
        region[:B] = True
        for with_stats in (False, True):
            op = nan_buf((B + 1, ntok, ach), packing.TORCH_DTYPE[fmt])
            sp = (st.cuda(), gs.cuda(), bs.cuda()) if with_stats else (None, None, None)
            call(lib().avc_patchify, (a if with_stats else a_sp).cuda(), *sp, op, dt, rnd, B, S,
                 pp)
            what = f"patchify {fmt}/{dt}/{rnd} stats={with_stats}"
            check_sentinel(op, region, what)
            if with_stats:
                check_stored(decode(op[:B], fmt), y, e, fmt, rnd, what)
            else:
                assert torch.equal(bits(op[:B]), bits(stored(plain, fmt, rnd))), what


# ------------------------------------------------------------------------------------------------ LayerNorm + transpose
LN_CASES = [  # (B, R, C, axis): the mixers' shapes, then edges
    (2, 484, 176, 1), (2, 121, 176, 1), (1, 1849, 344, 1), (2, 176, 488, 2), (2, 176, 128, 2), (1, 344, 1856, 2),
    (2, 344, 88, 0), (2, 88, 176, 0),
    (5, 37, 30, 1), (1, 37, 30, 2), (5, 70, 45, 2), (1, 70, 45, 1), (5, 13, 6, 0), (1, 3, 5, 1), (5, 9, 100, 2),
    (3, 100, 9, 1), (5, 130, 66, 2), (1, 66, 130, 1),
]


def _ln_inputs(B, R, C, axis, seed):
    g = torch.Generator().manual_seed(seed)
    x = offset_rows((B, R, C), RATIOS, g, dims=((2,) if axis == 1 else (1,)))
    n = C if axis == 1 else R
    gamma, beta = torch.rand(n, generator=g) + 0.5, torch.randn(n, generator=g) * 0.2
    if n > 2:
        gamma[1] = 4e4                                       # normalised values of a few sigma saturate fp16
        beta[2] = -9e4
    return x, gamma, beta


@pytest.mark.gpu
@pytest.mark.parametrize("B,R,C,axis", LN_CASES, ids=[f"B{b}R{r}C{c}ax{a}" for b, r, c, a in LN_CASES])
def test_ln_transpose(B, R, C, axis):
    from autoformer_b200 import packing
    x, gamma, beta = _ln_inputs(B, R, C, axis, B * 7 + R * 13 + C * 17 + axis)
    R8 = (R + 7) // 8 * 8
    xc = x.cuda()
    gc, bc = (gamma.cuda(), beta.cuda()) if axis else (None, None)
    xt = transposed_padded(x, R8)
    n_st = 2 * B * (R if axis == 1 else C) if axis else 0
    st_ref = None
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(R8, fmt)
        what = f"ln_transpose ax{axis} {fmt}/{dt}/{rnd}"
        op = nan_buf((B + 1, C, ach), packing.TORCH_DTYPE[fmt])
        f32 = nan_buf((B + 1, C, R8), torch.float32)
        scratch = nan_buf((2 * B * max(R, C) + 8,), torch.float32)
        call(lib().avc_ln_transpose, xc, gc, bc, axis, op, dt, rnd, f32, scratch, B, R, C)
        region = torch.zeros(B + 1, C, ach, dtype=torch.bool)
        region[:B] = True
        check_sentinel(op, region, what + " out_op")
        check_sentinel(f32, region[..., :R8], what + " out_f32")
        sreg = torch.zeros(scratch.numel(), dtype=torch.bool)
        sreg[:n_st] = True
        check_sentinel(scratch, sreg, what + " scratch")
        assert torch.equal(f32[:B].cpu(), xt), what + ": out_f32 is not the transposed copy"
        check_pad_zero(op[:B], R, R8, fmt, what)
        if axis == 0:
            assert torch.equal(bits(op[:B]), bits(stored(xt, fmt, rnd))), what
        else:
            st = scratch[:n_st].view(-1, 2).cpu()
            if st_ref is None:
                v, G = ln_rows_cols(x, axis)
                check_ln_stats(v, st, G, what + " statistics")
                st_ref = st
            assert torch.equal(st, st_ref), what + ": statistics differ between calls"
            check_ln_outputs(x, gamma, beta, axis, st, decode(op[:B], fmt), fmt, rnd, what)
        # each output alone gives the same bits
        op1 = nan_buf((B + 1, C, ach), packing.TORCH_DTYPE[fmt])
        call(lib().avc_ln_transpose, xc, gc, bc, axis, op1, dt, rnd, None, scratch, B, R, C)
        assert torch.equal(bits(op1), bits(op)), what + ": out_op alone"
        if fmt == "fp16x2":
            f1 = nan_buf((B + 1, C, R8), torch.float32)
            call(lib().avc_ln_transpose, xc, gc, bc, axis, None, dt, rnd, f1, scratch, B, R, C)
            assert torch.equal(bits(f1), bits(f32)), what + ": out_f32 alone"


# ------------------------------------------------------------------------------------------------ decoder input / codes
TF = [(T, fr) for T in (8, 176, 344) for fr in sorted({1, 22, T}) if T % fr == 0]


@pytest.mark.gpu
@pytest.mark.parametrize("T,freq", TF, ids=[f"T{t}f{f}" for t, f in TF])
def test_meta_decoder_input_and_gather_codes(T, freq):
    from autoformer_b200 import packing
    B, H, E = 3, 44, 256
    nc = T // freq
    codes = _special_values(B * nc * 2 * H, T + freq).view(B, nc, 2 * H)
    c_trg = _special_values(B * E, T * freq).view(B, E)
    full = torch.cat((codes.repeat_interleave(freq, dim=1), c_trg[:, None, :].expand(B, T, E)), -1).transpose(1, 2)
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(T, fmt)
        op = nan_buf((B + 1, 2 * H + E, ach), packing.TORCH_DTYPE[fmt])
        call(lib().avc_meta_decoder_input, codes.cuda(), c_trg.cuda(), op, dt, rnd, B, T, freq, 2 * H, E)
        region = torch.zeros(op.shape, dtype=torch.bool)
        region[:B] = True
        what = f"meta_decoder_input {fmt}/{dt}/{rnd}"
        check_sentinel(op, region, what)
        assert torch.equal(bits(op[:B]), bits(stored(full.contiguous(), fmt, rnd))), what
    out = torch.randn(B, T, 2 * H, generator=torch.Generator().manual_seed(T * freq))
    got = nan_buf((B + 1, nc, 2 * H), torch.float32)
    call(lib().avc_gather_codes, out.cuda(), got, B, T, H, freq)
    region = torch.zeros(got.shape, dtype=torch.bool)
    region[:B] = True
    check_sentinel(got, region, "gather_codes")
    assert torch.equal(got[:B].cpu(), gather_ref(out, H, freq)), "gather_codes"


def gather_ref(out, H, freq):
    """codes[b][j] = [out[b][j freq + freq - 1][:H] || out[b][j freq][H:]], indexed frame by frame."""
    B, T, _ = out.shape
    j = torch.arange(T // freq)
    return torch.cat((out[:, j * freq + freq - 1, :H], out[:, j * freq, H:]), -1)


# ------------------------------------------------------------------------------------------------ AdaIN "2"
@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 8, 1020, 4 * 256 * 256 + 4, 33 * 176 * 512])
def test_global_stats(n):
    g = torch.Generator().manual_seed(n)
    for ratio in (0.0, 100.0, 1000.0):
        x = offset_rows((1, n), (ratio,), g)
        st = nan_buf((3,), torch.float32)
        scratch = nan_buf((512,), torch.float64)
        call(lib().avc_global_stats, x.cuda(), n, st, scratch)
        region = torch.tensor([True, True, False])
        check_sentinel(st, region, "global_stats")
        first = st.cpu().clone()
        call(lib().avc_global_stats, x.cuda(), n, st, scratch)
        assert torch.equal(bits(st), bits(first)), "global_stats: a repeated call differs"
        # fixed-order partial sums: chains of n / 65536 + 13 additions per thread, then up to 256 partials
        mean, var, e_mean, e_var = fp64_moments_bound(x, n // 65536 + 16 + 256, bessel=True)
        std = torch.sqrt(var)
        got = first[:2].double()
        check_bound(got[:1], mean, e_mean, f"global_stats mean ratio {ratio}")
        check_bound(got[1:], std, std * 2 * u + e_var / (2 * std), f"global_stats std ratio {ratio}")


ADAIN = [(7 * 96, 80), (3, 4), (33 * 344, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("rows,C", ADAIN, ids=[f"r{r}C{c}" for r, c in ADAIN])
def test_adain(rows, C):
    from autoformer_b200 import packing
    if rows * C // 4 > 1e6:
        assert rows * C // 4 > grid_cap_float4()
    g = torch.Generator().manual_seed(rows + C)
    x = (torch.randn(rows, C, generator=g) * 2.5 + 0.7).contiguous()
    xd = x.double()
    xs = torch.stack([xd.mean(), xd.std()]).float()
    ts = torch.tensor([-0.3, 3e4])               # target std 3e4: values beyond ~2.2 std saturate fp16
    d = xd - xs[0].double()
    k = ts[1].double() / xs[1].double()
    y = d * k + ts[0].double()
    # 1 / std rounded, then a subtraction, two products and an addition
    e = 6 * u * (d.abs() * k.abs() + abs(float(ts[0])))
    for fmt, dt, rnd in FORMATS:
        ach = packing.act_channels(C, fmt)
        for want_f32, want_op in ((True, False), (False, True), (True, True)):
            f32 = nan_buf((rows + 3, C), torch.float32) if want_f32 else None
            op = nan_buf((rows + 3, ach), packing.TORCH_DTYPE[fmt]) if want_op else None
            call(lib().avc_adain, x.cuda(), xs.cuda(), ts.cuda(), f32, op, dt, rnd, rows, C)
            what = f"adain {fmt}/{dt}/{rnd} f32={want_f32} op={want_op}"
            if want_f32:
                region = torch.zeros(f32.shape, dtype=torch.bool)
                region[:rows] = True
                check_sentinel(f32, region, what + " out_f32")
                check_bound(f32[:rows], y, e, what + " out_f32")
            if want_op:
                region = torch.zeros(op.shape, dtype=torch.bool)
                region[:rows] = True
                check_sentinel(op, region, what + " out_op")
                check_stored(decode(op[:rows], fmt), y, e, fmt, rnd, what + " out_op")


# ------------------------------------------------------------------------------------------------ the ops wrappers
@pytest.mark.gpu
def test_ops_wrappers_equal_the_direct_calls():
    """Each ops wrapper passes its arguments through unchanged: its result has the bits of the direct call."""
    from autoformer_b200 import ops
    B, L, C, S, pp = 2, 176, 512, 176, 8
    g = torch.Generator().manual_seed(5)
    x = offset_rows((B, L, C), (0.0, 50.0), g).cuda()
    gamma, beta = (torch.rand(C, generator=g) + 0.5).cuda(), torch.randn(C, generator=g).cuda()
    fmt, dt = "fp16x2", 3
    st = nan_buf((B, 2), torch.float32)
    call(lib().avc_gn_stats, x, st, B, L * C, 1e-5)
    assert torch.equal(bits(ops.gn_stats(x, B)), bits(st))
    f32, op = torch.empty_like(x), ops.alloc_act(B, L, C, fmt, "cuda")
    call(lib().avc_gn_pool_residual, x, st, gamma, f32, op, dt, 1, B, L, C)
    wf, wo = ops.gn_pool_residual(x, st, gamma, fmt)
    assert torch.equal(bits(wf), bits(f32)) and torch.equal(bits(wo), bits(op))
    call(lib().avc_gn_apply, x, st, gamma, beta, op, dt, 1, B, L, C)
    assert torch.equal(bits(ops.gn_apply(x, st, gamma, beta, fmt)), bits(op))
    a = x[:, :, :S].contiguous()
    sa = ops.gn_stats(a, B)
    tk = ops.alloc_act(B, (S // pp) ** 2, pp * pp, fmt, "cuda")
    call(lib().avc_patchify, a, sa, gamma[:S], beta[:S], tk, dt, 1, B, S, pp)
    assert torch.equal(bits(ops.patchify(a, sa, gamma[:S], beta[:S], pp, fmt)), bits(tk))
    for axis in (0, 1, 2):
        R8 = (L + 7) // 8 * 8
        n = C if axis == 1 else L
        lo, lf = ops.alloc_act(B, C, R8, fmt, "cuda"), torch.empty(B, C, R8, device="cuda")
        scratch = torch.empty(2 * B * max(L, C), device="cuda")
        gb = (gamma[:n], beta[:n]) if axis else (None, None)
        call(lib().avc_ln_transpose, x, *gb, axis, lo, dt, 1, lf, scratch, B, L, C)
        wo, wf = ops.ln_transpose(x, *gb, axis, fmt, want_f32=True)
        assert torch.equal(bits(wo), bits(lo)) and torch.equal(bits(wf), bits(lf)), axis
    codes, c_trg = x[:, :8, :88].contiguous(), x[:, 0, :256].contiguous()
    di = ops.alloc_act(B, 88 + 256, 176, fmt, "cuda")
    call(lib().avc_meta_decoder_input, codes, c_trg, di, dt, 1, B, 176, 22, 88, 256)
    assert torch.equal(bits(ops.meta_decoder_input(codes, c_trg, 176, 22, fmt)), bits(di))
    out = x[:, :, :88].contiguous()
    gc = torch.empty(B, 8, 88, device="cuda")
    call(lib().avc_gather_codes, out, gc, B, 176, 44, 22)
    assert torch.equal(bits(ops.gather_codes(out, 44, 22)), bits(gc))
    gs, scratch = torch.empty(2, device="cuda"), torch.empty(512, dtype=torch.float64, device="cuda")
    call(lib().avc_global_stats, x, x.numel(), gs, scratch)
    assert torch.equal(bits(ops.global_stats(x)), bits(gs))
    ts = torch.tensor([0.4, 1.3], device="cuda")
    af, ao = torch.empty_like(x), ops.alloc_act(B, L, C, fmt, "cuda")
    call(lib().avc_adain, x, gs, ts, af, ao, dt, 1, B * L, C)
    wo, wf = ops.adain(x, gs, ts, fmt, want_f32=True)
    assert torch.equal(bits(wo), bits(ao)) and torch.equal(bits(wf), bits(af))


# ------------------------------------------------------------------------------------------------ model level
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pool", "conv"])
def test_meta_fp32_with_offset_mixer_embeddings(kind, monkeypatch):
    """A common offset on every mixer embedding bias (`*.mlp.1.bias`) leaves LayerNorm's output unchanged but puts the
    metablock mixers' LayerNorm inputs at |mean| / std of a few hundred: the "fp32" conversion must still meet the fp32
    gate of the full-size test against the fp64 oracle."""
    import oracle.meta as om
    from autoformer_b200.factory.MetaConv import MetaConv
    from autoformer_b200.factory.MetaPool import MetaPool
    from oracle import rel_l2, templates
    from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker
    args = (44, 256, 512, 22)
    sd = seeded_state_dict(templates.meta_template(kind, *args), 30 + (kind == "conv"))
    sd = {k: (v + 100.0 if k.endswith("mlp.1.bias") else v) for k, v in sd.items()}
    B = 2
    x, c_org, c_trg = synthetic_mel(B, 176, 43), synthetic_speaker(B, 43, "org"), synthetic_speaker(B, 43, "trg")
    ratios = {}
    ln = om.layer_norm

    def spy(sd_, prefix, z, eps=1e-5):
        ratios[prefix] = float((z.mean(-1).abs() / z.std(-1, unbiased=False)).median())
        return ln(sd_, prefix, z, eps)

    monkeypatch.setattr(om, "layer_norm", spy)
    ref = om.meta_forward(sd, x, c_org, c_trg, args[0], args[3], kind, dtype=torch.float64)
    block_ratios = [r for k, r in ratios.items() if "metablock" in k]
    assert len(block_ratios) == 8 and min(block_ratios) >= 100, ratios
    m = (MetaPool if kind == "pool" else MetaConv)(*args)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    m.precision = "fp32"
    out = m(x.cuda(), c_org.cuda(), c_trg.cuda())
    errs = [rel_l2(a, b) for a, b in zip(out, ref)]
    print(f"Meta{kind} fp32 with mixer embedding offset 100: rel-L2 (mel, mel_postnet, codes) {errs}")
    assert all(e < 2e-4 for e in errs), errs


# ------------------------------------------------------------------------------------------------ CPU: the checkers
def _moments_f32(x, G, welford):
    """float32 emulation of the LayerNorm statistics kernels on x [rows][n]: element j goes to chain j % G in order;
    the G partials merge in a halving tree (the warp's xor butterfly seen from lane 0, the column kernel's shared-memory
    tree).  welford=False is the single pass sum x, sum x^2 -> E[x^2] - mean^2 the kernels used before."""
    f = np.float32
    x = x.numpy().astype(f)
    rows, n = x.shape
    k = -(-n // G)
    xp = np.full((rows, k * G), np.nan, f)
    xp[:, :n] = x
    xp = xp.reshape(rows, k, G)
    if welford:
        cnt, m, M2 = (np.zeros((rows, G), f) for _ in range(3))
        for j in range(k):
            v = xp[:, j]
            ok = ~np.isnan(v)
            v = np.where(ok, v, f(0))
            c2 = cnt + f(1)
            d = v - m
            m2 = m + d * (f(1) / c2)
            M22 = M2 + d * (v - m2)
            cnt, m, M2 = np.where(ok, c2, cnt), np.where(ok, m2, m), np.where(ok, M22, M2)
        s = G // 2
        while s:
            na, ma, Ma, nb, mb, Mb = cnt[:, :s], m[:, :s], M2[:, :s], cnt[:, s:2 * s], m[:, s:2 * s], M2[:, s:2 * s]
            nn = na + nb
            d = mb - ma
            wb = nb / np.maximum(nn, f(1))
            m = np.where(nn > 0, ma + d * wb, ma)
            M2 = np.where(nn > 0, Ma + Mb + d * d * (na * wb), Ma)
            cnt = nn
            s //= 2
        mean, var = m[:, 0], M2[:, 0] / f(n)
    else:
        sv, ss = np.zeros((rows, G), f), np.zeros((rows, G), f)
        for j in range(k):
            v = np.nan_to_num(xp[:, j])
            sv, ss = sv + v, ss + v * v
        s = G // 2
        while s:
            sv, ss = sv[:, :s] + sv[:, s:2 * s], ss[:, :s] + ss[:, s:2 * s]
            s //= 2
        mean = sv[:, 0] / f(n)
        var = np.maximum(ss[:, 0] / f(n) - mean * mean, f(0))
    rstd = f(1) / np.sqrt(var + f(1e-5))
    return torch.from_numpy(np.stack([mean, rstd], 1).astype(f))


@pytest.mark.parametrize("G,n", [(32, 4), (32, 30), (32, 176), (32, 344), (8, 9), (8, 176), (8, 344)])
def test_ln_stats_bound_separates_welford_from_single_pass(G, n):
    """CPU: the float32 emulation of the fixed statistics meets the bound at every |mean| / std up to 1000; the
    single-pass algorithm fails it at every ratio from 10 on."""
    g = torch.Generator().manual_seed(G * n)
    for ratio in RATIOS:
        x = offset_rows((300, n), (ratio,), g)
        worst = check_ln_stats(x, _moments_f32(x, G, True), G, f"welford ratio {ratio}")
        assert worst < 0.5, worst
        if ratio >= 10:
            with pytest.raises(AssertionError, match="beyond the bound"):
                check_ln_stats(x, _moments_f32(x, G, False), G, f"single pass ratio {ratio}")


def test_elementwise_bounds_accept_the_stand_ins_and_reject_faults():
    """CPU: the fp64 stand-ins of tests/emulate.py (rounded to fp32 and stored) pass every elementwise check, and the
    faults the checks exist for fail them: divisor 3 at the pooling mixer's end frames, p1 and p2 swapped in patchify,
    the lo term of the split store dropped, pad columns left NaN, an off-by-one frame in gather_codes."""
    from autoformer_b200 import packing
    B, L, C = 2, 7, 12
    x, st, gamma, beta = _gn_inputs(B, L, C, 1)
    # pooling mixer
    y, e = pool_ref(x, st[:, 1], gamma)
    rf, ro = emulate._emu_gn_pool_residual(x, st, gamma, "fp32")
    check_bound(rf.double(), y, e, "gn_pool stand-in")
    check_stored(decode(ro, "fp32"), y, e, "fp32", 1, "gn_pool stand-in")
    ro16 = emulate._emu_gn_pool_residual(x, st, gamma, "fp16x2")[1]
    check_stored(decode(ro16, "fp16x2"), y, e, "fp16x2", 1, "gn_pool stand-in fp16")
    xd = x.double()
    bad = y.clone()
    bad[:, 0] = xd[:, 0] + st[:, 1].double().view(B, 1) * gamma.double() * ((xd[:, 0] + xd[:, 1]) / 3 - xd[:, 0])
    with pytest.raises(AssertionError):
        check_bound(bad.float().double(), y, e, "divisor 3")
    # dropped lo term of the split store
    hi = ro.clone()
    hi[..., C:] = 0
    with pytest.raises(AssertionError):
        check_stored(decode(hi, "fp32"), y, e, "fp32", 1, "lo dropped")
    # gn_apply
    ya, ea = affine_ref(x, st[:, 0].view(B, 1, 1), st[:, 1].view(B, 1, 1), gamma, beta)
    for fmt, _, rnd in FORMATS:
        check_stored(decode(stored(ya.float(), fmt, rnd), fmt), ya, ea, fmt, rnd, f"gn_apply stand-in {fmt}")
    check_stored(decode(emulate._emu_gn_apply(x, st, gamma, beta, "fp16x2"), "fp16x2"), ya, ea, "fp16x2", 1, "gn_apply")
    # patchify with GroupNorm
    S, pp = 16, 4
    g = torch.Generator().manual_seed(2)
    a = offset_rows((B, S, S), (0.0, 2.0), g, dims=(1, 2))
    sa = fp64_stats(a, B)
    gs, bs = torch.rand(S, generator=g) + 0.5, torch.randn(S, generator=g)
    img = a.double().transpose(1, 2)
    yp, ep = affine_ref(img, sa[:, 0].view(B, 1, 1), sa[:, 1].view(B, 1, 1), gs.view(1, S, 1), bs.view(1, S, 1))
    emu = decode(emulate._emu_patchify(a, sa, gs, bs, pp, "fp32"), "fp32")
    check_stored(emu, patchify_perm(yp, pp), patchify_perm(ep, pp), "fp32", 1, "patchify stand-in")
    n = S // pp
    swapped = yp.reshape(B, n, pp, n, pp).permute(0, 1, 3, 4, 2).reshape(B, n * n, pp * pp)  # (w % p) p + h % p
    with pytest.raises(AssertionError):
        check_stored(swapped.float().double(), patchify_perm(yp, pp), patchify_perm(ep, pp), "fp32", 1, "p1 <-> p2")
    # ln_transpose: the stand-in passes the output checks on its own fp32 statistics; NaN pad columns fail
    for axis, (Bl, R, Cl) in ((1, (2, 37, 30)), (2, (2, 37, 30))):
        xl, gl, bl = _ln_inputs(Bl, R, Cl, axis, 3)
        v, G = ln_rows_cols(xl, axis)
        stl = _moments_f32(v, G, True)
        R8 = (R + 7) // 8 * 8
        for fmt, _, rnd in FORMATS:
            if not rnd:
                continue                     # the stand-in always stores TF32-rounded
            opf, f32 = emulate._emu_ln_transpose(xl, gl, bl, axis, fmt, want_f32=True)
            check_pad_zero(opf, R, R8, fmt, "ln stand-in")
            check_ln_outputs(xl, gl, bl, axis, stl, decode(opf, fmt), fmt, rnd, f"ln stand-in ax{axis} {fmt}")
            assert torch.equal(f32, transposed_padded(xl, R8))
        opf = emulate._emu_ln_transpose(xl, gl, bl, axis, "fp32")[0]
        nanpad = opf.clone()
        nanpad[..., R8 + R:] = float("nan")          # the lo half's pad columns
        with pytest.raises(AssertionError):
            check_pad_zero(nanpad, R, R8, "fp32", "NaN pad")
    # gather_codes: the stand-in equals the frame-by-frame reference; an off-by-one frame does not
    out = torch.randn(2, 176, 88)
    assert torch.equal(emulate._emu_gather_codes(out, 44, 22), gather_ref(out, 44, 22))
    off = torch.cat((out[:, 20::22, :44], out[:, ::22, 44:]), -1)
    assert not torch.equal(off, gather_ref(out, 44, 22))
    # statistics: the stand-ins meet the fp64 bounds
    xs = offset_rows((3, 4004), (1000.0,), torch.Generator().manual_seed(4))
    mean, var, e_mean, e_var = fp64_moments_bound(xs, 4004 // 512 + 32, bessel=False)
    est = emulate._emu_gn_stats(xs, 3).double()
    check_bound(est[:, 0], mean, e_mean, "gn_stats stand-in")
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    check_bound(est[:, 1], rstd, rstd * (2 * u + e_var / (var + 1e-5)), "gn_stats stand-in rstd")
    gst = emulate._emu_global_stats(xs.view(1, -1)).double()
    mean, var, e_mean, e_var = fp64_moments_bound(xs.view(1, -1), 64, bessel=True)
    check_bound(gst[:1], mean, e_mean, "global_stats stand-in")
    check_bound(gst[1:], var.sqrt(), var.sqrt() * 2 * u + e_var / (2 * var.sqrt()), "global_stats stand-in std")
    # adain and fp16 saturation of every elementwise check
    xa = torch.randn(5, 8, generator=torch.Generator().manual_seed(6)) * 3
    xsa = torch.stack([xa.double().mean(), xa.double().std()]).float()
    ts = torch.tensor([-0.3, 6e4])
    ya = (xa.double() - xsa[0].double()) * (ts[1].double() / xsa[1].double()) + ts[0].double()
    ea = 6 * u * ((xa.double() - xsa[0].double()).abs() * abs(float(ts[1] / xsa[1])) + 0.3)
    ops_, f32_ = emulate._emu_adain(xa, xsa, ts, "fp16x2", want_f32=True)
    check_bound(f32_.double(), ya, ea, "adain stand-in")
    check_stored(decode(ops_, "fp16x2"), ya, ea, "fp16x2", 1, "adain stand-in fp16")
    big = (ya.abs() > 7e4).nonzero()
    assert len(big) and bool((decode(ops_, "fp16x2").abs()[ya.abs() > 7e4] == FP16_MAX).all())
    i = tuple(big[0].tolist())
    inf = ops_.clone()
    inf[i] = float("inf")
    with pytest.raises(AssertionError):
        check_stored(decode(inf, "fp16x2"), ya, ea, "fp16x2", 1, "fp16 overflow to inf")
    unsat = decode(ops_, "fp16x2")
    unsat[i] = 65472.0 * unsat[i].sign()
    with pytest.raises(AssertionError, match="saturate"):
        check_stored(unsat, ya, ea, "fp16x2", 1, "fp16 short of saturation")
