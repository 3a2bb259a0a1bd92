"""Op-level contract of avc_conv_gemm's epilogue paths and of the glue kernels, element by element.

Every conv-GEMM case is held to two independent checks:
  * a per-element worst-case bound against an fp64 reference computed from the operands the kernel actually reads (the
    packed weights and the stored activations, through tests/emulate.py's k-block walk): for v = sum a*w + bias,
    |err v| <= (K_phys + 2) 2^-23 (sum |a*w| + |bias|), carried through the activation's derivative, plus the activation's
    own approximation error and half an ulp of the output format.  Worst case, so never flaky; any indexing, masking,
    halo or phase error is of order |v| and fails it;
  * a global rel-L2 against torch's own op in fp64 on the unrounded inputs (the tolerances of
    test_gpu_parity.test_conv_gemm_matches_conv1d), which catches a dropped precision term that the worst-case bound is
    too loose to see.
Outputs are written into NaN-filled buffers with spare rows and channels: exactly the expected region must become finite.

The GPU cases are declared in CONV_CASES; a CPU test mirrors the kernel's tile split and path predicate and checks that
the cases reach every (epilogue path x tile geometry) cell.
"""
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

from oracle import rel_l2
from tests import emulate

U = 2.0 ** -23
ACT_NAMES = ("none", "relu", "tanh", "lrelu", "gelu", "log10_clamp")
# rel-L2 of a launch against torch in fp64 on the unrounded inputs (test_gpu_parity.test_conv_gemm_matches_conv1d);
# "fp16s" (three products of two-term fp16 values) is fp32-grade like "fp32"
LAYER_TOL = {"fp32": 5e-5, "tf32": 2e-3, "bf16": 1e-2, "fp16x2": 5e-4, "fp16s": 5e-5}
# what rounding the stored output to its format adds
FMT_TOL = {"fp32": 5e-5, "tf32": 2e-3, "bf16": 1e-2, "fp16x2": 5e-4, "f16": 5e-4, "fp16s": 5e-5}
MODE = {"tf32": 0, "bf16": 1, "fp32": 2, "fp16x2": 3, "f16": 3, "fp16s": 4}     # out_dtype codes (ops._dt)


# ------------------------------------------------------------------------------------------------ kernel mirrors
def tile_split(B, T):
    """Mirror of avc_gemm.cu:571-586: the power-of-two split of 128 rows into bb utterances x tb frames with the fewest
    tile rows (ties keep the larger tb).  Returns (tb_log2, m_tiles)."""
    best, tb_log2 = -1, 7
    for l in range(7, -1, -1):
        tb, bb = 1 << l, 128 >> l
        rows = -(-T // tb) * -(-B // bb)
        if best < 0 or rows < best:
            best, tb_log2 = rows, l
    tb, bb = 1 << tb_log2, 128 >> tb_log2
    return tb_log2, -(-T // tb) * -(-B // bb)


def tile_paths(N, bn, phases=1, phase0=0, phase_count=None, out=None, out2=False, raw=None, res=False,
               res_after=False, reflect=0, round_tf32=True, tb_log2=7):
    """Mirror of epilogue_tile's path choice (avc_gemm.cu:150-168 and :203-315) for every n-tile of a launch.
    `out` / `raw` are format names or None.  Returns the set of path names."""
    phase_count = phase_count or phases
    cs = N // phase_count
    out_mode = MODE[out] if out else (MODE[raw] if raw else 0)
    raw_mode = MODE[raw] if raw else out_mode
    paths = set()
    for n0 in range(0, N, bn):
        chunks = min(bn // 32, -(-(N - n0) // 32))
        split_rows = chunks == 1                                                    # :150-151
        simple = 0
        if not split_rows and reflect == 0 and ((phases == 1 and phase0 == 0) or cs % 32 == 0):   # :165
            if out and not out2 and not res and out_mode != 0 and (not raw or raw_mode != 0):     # :166
                simple = 1
            if not out and out2 and not (res and res_after) and phases == 1 and not raw:        # :167
                simple = 2
        fast = tb_log2 >= 5                                                         # :203
        if simple == 1:
            if not fast:
                paths.add("s1_row")
            elif not raw and out_mode == 3:
                paths.add("s1_fast_f16")                                            # :218
            elif not raw and out_mode == 4:
                paths.add("s1_fast_f16s")                                           # :228
            else:
                paths.add("s1_fast_store16_" + ("raw" if raw else {1: "bf16", 2: "bf16s"}.get(out_mode, str(out_mode))))
        elif simple == 2:
            paths.add(("s2_fast_res" if res else "s2_fast") if fast else "s2_row")
        elif split_rows:
            paths.add("gen_split_rows")
        else:
            if res and res_after:
                paths.add("gen_res_after")
            if out and reflect:
                paths.add("gen_reflect")
            if out == "tf32":
                paths.add("gen_fp32_round" if round_tf32 else "gen_fp32")
            if out and out2:
                paths.add("gen_out_out2")
            paths.add("gen")
    return paths


def geometry_classes(B, T):
    tb_log2, m_tiles = tile_split(B, T)
    cls = set()
    if m_tiles == 1:
        cls.add("single")                       # avc_gemm.cu:617-618: one m-tile runs the single-CTA kernel
    if tb_log2 >= 5:
        if m_tiles % 2 == 1 and m_tiles >= 3:
            cls.add("phantom")                  # CTA pairs: the last pair holds a masked phantom tile
        if T < (1 << tb_log2):
            cls.add("short")
    elif m_tiles >= 2:
        cls.add("row")
    return cls


# ------------------------------------------------------------------------------------------------ declared GPU cases
# path -> (layer precision and call arguments, the geometry classes the path must meet)
FAST_GEOS = ("phantom", "short", "single")
ROW_GEOS = ("row", "single")
GEN_GEOS = ("phantom", "row", "single")
PATHS = {
    "s1_fast_f16": (dict(prec="fp16x2", out="fp16x2"), FAST_GEOS),
    "s1_fast_f16s": (dict(prec="fp16s", out="fp16s"), FAST_GEOS),
    "s1_fast_store16_raw": (dict(prec="fp16s", out="f16", raw="fp16s"), FAST_GEOS),
    "s1_fast_store16_bf16": (dict(prec="bf16", out="bf16"), FAST_GEOS),
    "s1_fast_store16_bf16s": (dict(prec="fp32", out="fp32"), FAST_GEOS),
    "s1_row": (dict(prec="fp16s", out="f16", raw="fp16s"), ROW_GEOS),
    "s2_fast": (dict(prec="fp32", out2=True), FAST_GEOS),
    "s2_fast_res": (dict(prec="fp16x2", out2=True, res=True), FAST_GEOS),
    "s2_row": (dict(prec="fp16s", out2=True, res=True), ROW_GEOS),
    "gen_res_after": (dict(prec="fp16x2", out="fp16x2", out2=True, res=True, res_after=True), GEN_GEOS),
    "gen_reflect": (dict(prec="fp16s", out="fp16s", reflect=3), GEN_GEOS),
    "gen_fp32_round": (dict(prec="tf32", out="tf32", round_tf32=True), GEN_GEOS),
    "gen_fp32": (dict(prec="tf32", out="tf32", round_tf32=False), GEN_GEOS),
    "gen_out_out2": (dict(prec="fp32", out="fp32", out2=True), GEN_GEOS),
    "gen_split_rows": (dict(prec="fp16s", out="fp16s", raw="fp16s"), GEN_GEOS),
}
# shapes (B, T) of each geometry class; "single" differs for the fast-loop and row-loop paths
FAST_SHAPES = {"phantom": [(2, 176), (33, 24), (5, 96)], "short": [(3, 33), (33, 24), (2, 40)],
               "single": [(2, 17), (2, 40)]}
ROW_SHAPES = {"row": [(130, 16), (64, 3), (130, 1)], "single": [(7, 5)]}
GEN_SHAPES = {"phantom": [(2, 176), (5, 96)], "row": [(130, 16), (64, 3), (130, 1)], "single": [(7, 5), (2, 17)]}
# (N, block_n): 512 packed with each tile width; 36 = a second chunk with one live lane group; 80 = a ragged n-tile
WIDE_N = [(36, None), (80, None), (512, 64), (512, 128), (512, 256), (80, 64)]
SPLIT_N = [(16, None), (32, None)]


def _declare_cases():
    cases = []
    i = 0
    for path, (kw, geos) in PATHS.items():
        shapes = FAST_SHAPES if geos is FAST_GEOS else (ROW_SHAPES if geos is ROW_GEOS else GEN_SHAPES)
        for g in geos:
            fits = [(B, T) for B, T in shapes[g] if T > kw.get("reflect", 0)]     # a reflected halo needs T > reflect
            B, T = fits[i % len(fits)]
            ns = SPLIT_N if path == "gen_split_rows" else WIDE_N
            N, bn = ns[i % len(ns)]
            act = ACT_NAMES[i % len(ACT_NAMES)]
            if act == "log10_clamp" and kw["prec"] not in ("fp32", "tf32"):
                act = "gelu"            # inputs around 1e-5 are fp16 subnormals: log10 layers run in split bf16 / TF32
            cases.append(dict(kw, path=path, geo=g, B=B, T=T, N=N, bn=bn, act=act, c_in=24 + 8 * (i % 3), k=3))
            i += 1
    return cases


CONV_CASES = _declare_cases()


def _case_id(c):
    return f"{c['path']}-{c['geo']}-B{c['B']}T{c['T']}-N{c['N']}bn{c['bn']}-{c['act']}"


def _case_paths(c):
    from autoformer_b200 import packing
    bn = c["bn"] or packing.choose_block_n(c["N"])
    return tile_paths(c["N"], bn, out=c.get("out"), out2=c.get("out2", False), raw=c.get("raw"), res=c.get("res", False),
                      res_after=c.get("res_after", False), reflect=c.get("reflect", 0),
                      round_tf32=c.get("round_tf32", True), tb_log2=tile_split(c["B"], c["T"])[0])


def test_conv_case_matrix_covers_every_cell():
    """CPU: the declared cases reach every (path x geometry) cell through the mirrored predicate, every N class and
    block_n, and all six activations."""
    from autoformer_b200 import packing
    cells = set()
    for c in CONV_CASES:
        paths = _case_paths(c)
        assert c["path"] in paths, (_case_id(c), paths)
        for p in paths:
            for g in geometry_classes(c["B"], c["T"]):
                cells.add((p, g))
    need = {(p, g) for p, (_, geos) in PATHS.items() for g in geos}
    assert need <= cells, sorted(need - cells)
    ns = {(c["N"], c["bn"] or packing.choose_block_n(c["N"])) for c in CONV_CASES}
    assert {(16, 64), (32, 64), (36, 64), (80, 128), (512, 64), (512, 128), (512, 256)} <= ns, ns
    assert {c["act"] for c in CONV_CASES} == set(ACT_NAMES)
    # the special-geometry cases below: a partial-phase pair and r = 2 with cs % 32 != 0 (general loop)
    assert "s1_fast_f16s" in tile_paths(128, 128, phases=8, phase0=4, phase_count=4, out="fp16s", tb_log2=6)
    assert "s1_fast_store16_raw" in tile_paths(128, 128, phases=8, phase0=0, phase_count=4, out="f16", raw="fp16s",
                                               tb_log2=6)
    assert tile_paths(96, 128, phases=2, out="fp16s", tb_log2=6) == {"gen"}
    assert tile_paths(32, 64, phases=2, out="fp16s", tb_log2=6) == {"gen_split_rows"}
    # the shapes the geometry classes are named after
    assert tile_split(130, 16) == (4, 17) and tile_split(7, 5)[1] == 1 and tile_split(2, 17) == (6, 1)
    assert tile_split(2, 176) == (6, 3) and tile_split(130, 1) == (0, 2) and tile_split(64, 3) == (2, 2)


# ------------------------------------------------------------------------------------------------ reference helpers
def _phys(layer, srcs):
    """The physical operand list the kernel walks (ops.ConvGemm.__call__): split precision reads [hi|lo] against
    [w_hi|w_hi] and hi against w_lo; fp16x2 reads the buffer twice."""
    meta = layer.meta
    if meta.get("split"):
        out = []
        for a, c in zip(srcs, meta["logical_channels"]):
            out += [a, a[:, :, :c]]
        return out
    if meta.get("dup"):
        return [a for a in srcs for _ in range(2)]
    return list(srcs)


def exact_operand_ref(layer, srcs, B, T):
    """(v, S): fp64 v = sum a*w + bias over the stored operands, and S = sum |a*w| + |bias|."""
    phys = [a.cpu() for a in _phys(layer, srcs)]
    w, b = layer.w.cpu(), layer.bias.cpu()
    v = emulate.emulate_conv_gemm(w, b, layer.meta, phys, B, T, layer.tap_t0, layer.tap_dt)
    s = emulate.emulate_conv_gemm(w.float().abs(), b.abs(), layer.meta, [a.float().abs() for a in phys], B, T,
                                  layer.tap_t0, layer.tap_dt)
    return v, s


def v_bound(layer, S):
    return (layer.meta["k_pad"] + 2) * U * S


def act_ref_and_bound(act, v, e_v):
    """fp64 act(v) and the bound on |kernel act - act(v)| given |kernel v - v| <= e_v (apply_act, avc_gemm.cu:54-74)."""
    if act == "none":
        return v, e_v
    if act == "relu":
        return v.clamp(min=0), e_v
    if act == "lrelu":
        o = torch.where(v > 0, v, 0.2 * v)
        return o, e_v + 2 * U * o.abs()
    if act == "tanh":
        # tanh_fast: __expf and __fdividef (a few ulp each) around 1 - e / 1 + e: absolute error ~1e-7
        return torch.tanh(v), e_v + 2e-6
    if act == "gelu":
        o = 0.5 * v * (1.0 + torch.erf(v / 2 ** 0.5))
        x = v.abs() / 2 ** 0.5
        q = torch.erfc(x)
        # derivative <= 1.13; A&S 7.1.26 |erf error| <= 1.5e-7; the fp32 evaluation of erfc (exp of a rounded -x^2,
        # reciprocal, polynomial) is relatively accurate to a few ulp plus x^2 ulp; the final products round
        act_err = 0.5 * v.abs() * (1.5e-7 + q * (16 * U + x * x * 2 * U)) + 4 * U * (o.abs() + v.abs())
        return o, 1.13 * e_v + act_err
    if act == "log10_clamp":
        o = torch.log10(v.clamp(min=1e-5))
        d = 1.0 / ((v - e_v).clamp(min=1e-5) * math.log(10.0))
        return o, d * e_v + 4 * U * o.abs() + 1e-7            # log10f a few ulp; clamp at fp32(1e-5)
    raise ValueError(act)


def half_ulp(mag, fmt, round_tf32=True):
    """Half an ulp of the stored format at magnitude `mag` (>= |value|)."""
    if fmt == "bf16":
        return mag * 2.0 ** -8
    if fmt in ("fp16x2", "f16"):
        return mag * 2.0 ** -11 + 2.0 ** -25                   # fp16 subnormal floor: step 2^-24
    if fmt == "fp32":                                           # split bf16: lo = bf16(v - hi), |v - hi| <= 2^-8 |v|
        return mag * 2.0 ** -16
    if fmt == "fp16s":                                          # split fp16: lo = fp16(v - hi), |v - hi| <= 2^-11 |v|
        return mag * 2.0 ** -22 + 2.0 ** -25
    if fmt == "tf32":
        return mag * 2.0 ** -11 if round_tf32 else mag * 0.0
    raise ValueError(fmt)


def check_bound(got, ref, bound, what):
    got = got.double().cpu()
    ref, bound = ref.cpu(), bound.cpu()
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite values"
    err = (got - ref).abs()
    bad = err > bound
    if bool(bad.any()):
        idx = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} of {err.numel()} elements beyond the bound; first at {idx}: "
                             f"got {float(got[tuple(idx)])}, ref {float(ref[tuple(idx)])}, bound {float(bound[tuple(idx)])}")


def nan_buf(shape, dtype):
    return torch.full(shape, float("nan"), dtype=dtype, device="cuda")


def check_sentinel(buf, region, what):
    """Exactly `region` (a bool mask of buf's shape) is finite; everything else still NaN."""
    fin = torch.isfinite(buf.float()).cpu()
    assert bool(fin[region].all()), f"{what}: {int((~fin[region]).sum())} expected elements not written"
    assert not bool(fin[~region].any()), f"{what}: {int(fin[~region].sum())} elements written outside the output"


def torch_conv_src(x, w, t0, dt, T):
    """out[t] = sum_j x[t + t0 + j dt] w[:, :, j] (zero outside the utterance) with torch in fp64; x [B][rows][C]."""
    k = w.shape[2]
    xt = x.double().transpose(1, 2)
    left = max(0, -t0)
    right = max(0, t0 + (k - 1) * dt + T - x.shape[1])
    y = F.conv1d(F.pad(xt, (left, right)), w.double(), dilation=dt)
    return y[:, :, t0 + left:t0 + left + T].transpose(1, 2)


def torch_act(act, v):
    return act_ref_and_bound(act, v, torch.zeros_like(v))[0]


def make_inputs(act, B, T, c_in, N, k, seed):
    g = torch.Generator().manual_seed(seed)
    if act == "log10_clamp":     # mel-like: non-negative operands, pre-activations straddling the 1e-5 clamp
        w = torch.rand(N, c_in, k, generator=g) / (c_in * k)
        x = torch.rand(B, T, c_in, generator=g) * torch.exp(torch.randn(B, T, 1, generator=g) * 2.0) * 2e-5
        b = torch.zeros(N)
        return w, b, x
    w = torch.randn(N, c_in, k, generator=g) / (c_in * k) ** 0.5
    b = torch.randn(N, generator=g) * (4.0 if act == "gelu" else 1.0)      # GELU: far negative and around zero
    x = torch.randn(B, T, c_in, generator=g)
    return w, b, x


# ------------------------------------------------------------------------------------------------ the epilogue matrix
class Launch:
    """One avc_conv_gemm launch into sentinel buffers, with the reference and the checks of everything it writes."""

    SPARE_ROWS, SPARE_CH = 2, 8

    def __init__(self, layer, srcs, B, T, *, out=None, raw=None, out2=False, res=None, res_after=False, reflect=0,
                 round_tf32=True, phases=1, phase0=0, phase_count=None, bufs=None):
        from autoformer_b200 import packing
        self.layer, self.B, self.T = layer, B, T
        self.out_fmt, self.raw_fmt, self.reflect, self.round = out, raw, reflect, round_tf32
        self.phases, self.phase0 = phases, phase0
        self.phase_count = phase_count or phases
        N = layer.meta["N"]
        self.cs = N // self.phase_count
        t_out = T * phases
        self.row0 = reflect + 1
        bufs = bufs or {}
        if out:
            self.out = bufs.get("out")
            if self.out is None:
                self.out = nan_buf((B, self.row0 + t_out + reflect + self.SPARE_ROWS,
                                    packing.act_channels(self.cs, out) + self.SPARE_CH), packing.TORCH_DTYPE[out])
        if raw:
            self.raw_full = bufs.get("raw")
            if self.raw_full is None:
                self.raw_full = nan_buf((B * t_out + self.SPARE_ROWS, packing.act_channels(self.cs, raw) + self.SPARE_CH),
                                        packing.TORCH_DTYPE[raw])
        if out2:
            self.out2_full = nan_buf((B * t_out + self.SPARE_ROWS, self.cs + self.SPARE_CH), torch.float32)
        self.res = res
        layer(srcs, B, T, out=self.out if out else None, out_row0=self.row0, round_tf32=round_tf32, reflect=reflect,
              out2=self.out2_full[:B * t_out] if out2 else None, residual=res, res_after=res_after,
              out_raw=self.raw_full[:B * t_out] if raw else None, phases=phases, out_fmt=out, raw_fmt=raw,
              phase0=phase0, phase_count=phase_count)
        torch.cuda.synchronize()
        # reference over the stored operands, scattered into output time
        v, S = exact_operand_ref(layer, srcs, B, T)
        e = v_bound(layer, S)
        pc, cs = self.phase_count, self.cs
        v = v.view(B, T, pc, cs)
        e = e.view(B, T, pc, cs)
        self.times = (torch.arange(T)[:, None] * phases + phase0 + torch.arange(pc)[None, :]).reshape(-1)
        self.v = v.reshape(B, T * pc, cs)
        self.e = e.reshape(B, T * pc, cs)
        if res is not None:
            r = res.double().cpu().view(B, t_out, -1)[:, self.times, :cs]
            if not res_after:
                self.v = self.v + r
                self.e = self.e + 2 * U * self.v.abs()
            self.r_after = r if res_after else None
        else:
            self.r_after = None

    def act(self, act):
        o, eo = act_ref_and_bound(act, self.v, self.e)
        if self.r_after is not None:
            o = o + self.r_after
            eo = eo + 2 * U * o.abs()
        return o, eo

    def check(self, act, what):
        from autoformer_b200 import packing
        B, t_out = self.B, self.T * self.phases
        o, eo = self.act(act)
        if self.out_fmt:
            ach = packing.act_channels(self.cs, self.out_fmt)
            R = self.reflect
            rows = self.row0 + self.times
            region = torch.zeros(self.out.shape, dtype=torch.bool)
            region[:, rows, :ach] = True
            if R:
                region[:, self.row0 - R:self.row0, :ach] = True
                region[:, self.row0 + t_out:self.row0 + t_out + R, :ach] = True
            check_sentinel(self.out, region, what + " out")
            got = packing.act_to_float(self.out[:, :, :ach], self.out_fmt)
            bound = eo + half_ulp(o.abs() + eo, self.out_fmt, self.round)
            check_bound(got[:, rows], o, bound, what + " out")
            if R:
                idx = torch.arange(-R, t_out + R)
                src = idx.abs()
                src = torch.where(src >= t_out, 2 * (t_out - 1) - src, src)
                assert self.phase_count == self.phases
                check_bound(got[:, self.row0 - R:self.row0 + t_out + R], o[:, src], bound[:, src], what + " halo")
        if self.raw_fmt:
            ach = packing.act_channels(self.cs, self.raw_fmt)
            full = self.raw_full
            region = torch.zeros(full.shape, dtype=torch.bool)
            flat_rows = (torch.arange(B)[:, None] * t_out + self.times[None, :]).reshape(-1)
            region[flat_rows, :ach] = True
            check_sentinel(full, region, what + " out_raw")
            got = packing.act_to_float(full[:B * t_out, :ach], self.raw_fmt).view(B, t_out, -1)[:, self.times]
            check_bound(got, self.v, self.e + half_ulp(self.v.abs() + self.e, self.raw_fmt, self.round), what + " out_raw")
        if hasattr(self, "out2_full"):
            full = self.out2_full
            region = torch.zeros(full.shape, dtype=torch.bool)
            region[:B * t_out, :self.cs] = True
            check_sentinel(full, region, what + " out2")
            check_bound(full[:B * t_out, :self.cs].view(B, t_out, self.cs)[:, self.times], o, eo, what + " out2")
        return o


def _run_case(c, seed):
    from autoformer_b200 import ops, packing
    B, T, N, k, c_in, act, prec = c["B"], c["T"], c["N"], c["k"], c["c_in"], c["act"], c["prec"]
    w, b, x = make_inputs(act, B, T, c_in, N, k, seed)
    layer = ops.ConvGemm(*packing.pack_conv(w, b, prec, block_n=c["bn"]), act=act).to("cuda")
    res = None
    if c.get("res"):
        res = torch.randn(B * T, N + 4, generator=torch.Generator().manual_seed(seed + 1)).cuda()   # res_ld > N
    xs = packing.to_act(x, prec).cuda()
    L = Launch(layer, [xs], B, T, out=c.get("out"), raw=c.get("raw"), out2=c.get("out2", False), res=res,
               res_after=c.get("res_after", False), reflect=c.get("reflect", 0), round_tf32=c.get("round_tf32", True))
    L.check(act, _case_id(c))
    # independent: torch's conv on the unrounded inputs
    v = F.conv1d(x.double().transpose(1, 2), w.double(), b.double(), padding=k // 2).transpose(1, 2)
    if res is not None and not c.get("res_after"):
        v = v + res.double().cpu().view(B, T, -1)[..., :N]
    ref = torch_act(act, v)
    if res is not None and c.get("res_after"):
        ref = ref + res.double().cpu().view(B, T, -1)[..., :N]
    tol = LAYER_TOL[prec]
    if c.get("out2"):
        assert rel_l2(L.out2_full[:B * T, :N].view(B, T, N), ref) < tol
    if c.get("out"):
        got = packing.act_to_float(L.out[:, L.row0:L.row0 + T, :packing.act_channels(N, c["out"])], c["out"])
        fmt_tol = FMT_TOL[c["out"]] if (c["out"] != "tf32" or c.get("round_tf32", True)) else 5e-5
        assert rel_l2(got, ref) < 2 * max(tol, fmt_tol)
    if c.get("raw"):
        got = packing.act_to_float(L.raw_full[:B * T, :packing.act_channels(N, c["raw"])], c["raw"]).view(B, T, N)
        assert rel_l2(got, v) < 2 * max(tol, FMT_TOL[c["raw"]])


@pytest.mark.gpu
@pytest.mark.parametrize("case", CONV_CASES, ids=_case_id)
def test_conv_gemm_epilogue_path(case):
    _run_case(case, seed=zlib.crc32(_case_id(case).encode()) % 10007)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,c_out,act", [(2, 40, 48, "none"), (33, 24, 48, "lrelu"), (130, 1, 16, "none"),
                                           (3, 33, 32, "lrelu")])
def test_conv_transpose_r2(B, T, c_out, act):
    """r = 2 up-sampler as one 2-phase GEMM: C_out = 48 (cs % 32 != 0) keeps the general loop, C_out = 16 the split-rows
    loop, C_out = 32 takes the fast loop."""
    from autoformer_b200 import ops, packing
    torch.manual_seed(B + T)
    c_in, r = 40, 2
    wt = torch.randn(c_in, c_out, 2 * r) / (2 * c_in) ** 0.5
    bias = torch.randn(c_out)
    x = torch.randn(B, T, c_in)
    w3 = packing.conv_transpose_as_conv(wt, r, r // 2 + r % 2)
    layer = ops.ConvGemm(*packing.pack_conv(w3, bias.repeat(r), "fp16s"), tap_t0=[-1], act=act).to("cuda")
    L = Launch(layer, [packing.to_act(x, "fp16s").cuda()], B, T, out="fp16s", phases=r)
    o = L.check(act, "r2")
    ref = torch_act(act, F.conv_transpose1d(x.double().transpose(1, 2), wt.double(), bias.double(), stride=r,
                                            padding=r // 2 + r % 2, output_padding=r % 2).transpose(1, 2))
    assert ref.shape == (B, T * r, c_out)
    got = packing.act_to_float(L.out[:, L.row0:L.row0 + T * r, :2 * c_out], "fp16s")
    assert rel_l2(got, ref) < LAYER_TOL["fp16s"] and rel_l2(o, ref) < LAYER_TOL["fp16s"]


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(2, 40), (33, 24), (130, 16), (7, 5)])
@pytest.mark.parametrize("form", ["raw", "act"])
def test_conv_transpose_r8_two_half_launches(B, T, form):
    """MelGAN's r = 8 ConvTranspose1d as two GEMMs of two taps (phases [0, 4) and [4, 8), built like _PlanF16s) into one
    buffer: after the first launch the other phases' rows are still untouched."""
    from autoformer_b200 import ops, packing
    torch.manual_seed(T)
    c_in, c_out, r = 64, 32, 8
    wt = torch.randn(c_in, c_out, 2 * r) / (2 * c_in) ** 0.5
    bias = torch.randn(c_out)
    x = torch.randn(B, T, c_in)
    w3 = packing.conv_transpose_as_conv(wt, r, r // 2 + r % 2)
    half = r // 2 * c_out
    act = "none" if form == "raw" else "lrelu"
    parts = [(packing.pack_conv(w3[:half, :, 0:2].contiguous(), bias.repeat(r // 2), "fp16s"), -1, 0),
             (packing.pack_conv(w3[half:, :, 1:3].contiguous(), bias.repeat(r // 2), "fp16s"), 0, r // 2)]
    xs = packing.to_act(x, "fp16s").cuda()
    out_fmt, raw_fmt = ("fp16s", None) if form == "raw" else ("f16", "fp16s")
    bufs, launches = {}, []
    for pk, t0, p0 in parts:
        layer = ops.ConvGemm(*pk, tap_t0=[t0], act=act).to("cuda")
        L = Launch(layer, [xs], B, T, out=out_fmt, raw=raw_fmt, phases=r, phase0=p0, phase_count=r // 2, bufs=bufs)
        bufs = dict(out=L.out, raw=getattr(L, "raw_full", None))
        if not launches:
            L.check(act, f"r8 phases {p0}..{p0 + r // 2}")     # the second half's rows are still NaN
        launches.append(L)
    # both halves: every row of the up-sampled signal written
    full = Launch.__new__(Launch)
    full.__dict__.update(launches[1].__dict__)
    full.phase0, full.phase_count = 0, r
    full.times = torch.arange(T * r)
    vs = torch.stack([l.v.view(B, T, r // 2, c_out) for l in launches], dim=2).reshape(B, T * r, c_out)
    es = torch.stack([l.e.view(B, T, r // 2, c_out) for l in launches], dim=2).reshape(B, T * r, c_out)
    full.v, full.e = vs, es
    o = full.check(act, "r8 both halves")
    ref = F.conv_transpose1d(x.double().transpose(1, 2), wt.double(), bias.double(), stride=r,
                             padding=r // 2 + r % 2, output_padding=r % 2).transpose(1, 2)
    assert ref.shape == (B, T * r, c_out)
    assert rel_l2(vs, ref) < LAYER_TOL["fp16s"]
    assert rel_l2(o, torch_act(act, ref)) < LAYER_TOL["fp16s"]
    got = packing.act_to_float(full.out[:, full.row0:full.row0 + T * r, :packing.act_channels(c_out, out_fmt)], out_fmt)
    assert rel_l2(got, torch_act(act, ref)) < 2 * max(LAYER_TOL["fp16s"], FMT_TOL[out_fmt])


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,prec", [(2, 40, "fp16s"), (130, 16, "fp16s"), (33, 24, "fp32"), (7, 5, "fp16x2")])
def test_two_sources_with_different_tap_offsets(B, T, prec):
    """K-concatenated sources [h1, x] (MelGAN's block.4 + shortcut) with different tap_t0 and taps."""
    from autoformer_b200 import ops, packing
    torch.manual_seed(B * T)
    N, c1, c2 = 64, 48, 32
    w1, w2 = torch.randn(N, c1, 3) / (3 * c1) ** 0.5, torch.randn(N, c2, 2) / (2 * c2) ** 0.5
    b = torch.randn(N)
    x1, x2 = torch.randn(B, T, c1), torch.randn(B, T, c2)
    t0 = [-2, 1]
    layer = ops.ConvGemm(*packing.pack_conv_sources([w1, w2], b, prec), tap_t0=t0, act="lrelu").to("cuda")
    srcs = [packing.to_act(x1, prec).cuda(), packing.to_act(x2, prec).cuda()]
    L = Launch(layer, srcs, B, T, out=prec, out2=True)
    L.check("lrelu", "two sources")
    ref = F.leaky_relu(torch_conv_src(x1, w1, t0[0], 1, T) + torch_conv_src(x2, w2, t0[1], 1, T) + b.double(), 0.2)
    assert rel_l2(L.out2_full[:B * T, :N].view(B, T, N), ref) < LAYER_TOL[prec]


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,k,dt,t0", [(3, 5, 3, 9, -9), (2, 17, 3, 9, 0), (33, 2, 7, 1, -3), (130, 2, 7, 1, -3)])
def test_taps_mostly_in_the_zero_fill(B, T, k, dt, t0):
    """Dilation 9 with T smaller than the tap span, and k = 7 on two-frame utterances: most taps land in TMA's zero fill,
    so any read across an utterance boundary shows."""
    from autoformer_b200 import ops, packing
    torch.manual_seed(k * 100 + T)
    N, c_in = 64, 40
    w, b = torch.randn(N, c_in, k) / (k * c_in) ** 0.5, torch.randn(N)
    x = torch.randn(B, T, c_in) * 3
    for prec in ("fp16x2", "fp32"):
        layer = ops.ConvGemm(*packing.pack_conv(w, b, prec), tap_t0=[t0], tap_dt=[dt], act="none").to("cuda")
        L = Launch(layer, [packing.to_act(x, prec).cuda()], B, T, out=prec, out2=True)
        L.check("none", f"taps {prec}")
        ref = torch_conv_src(x, w, t0, dt, T) + b.double()
        assert rel_l2(L.out2_full[:B * T, :N].view(B, T, N), ref) < LAYER_TOL[prec]


# ------------------------------------------------------------------------------------------------ bit-exact invariances
def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32).cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,u", [(5, 96, 3), (33, 24, 32), (130, 16, 129), (64, 3, 0)])
def test_utterance_alone_equals_its_rows_in_the_batch(B, T, u):
    """The K loop runs (source, tap, chunk) in the same order whatever the tile split: converting one utterance alone
    gives the same bits as its rows of the batch."""
    from autoformer_b200 import ops, packing
    torch.manual_seed(B + u)
    N, c_in = 512, 72
    w, b = torch.randn(N, c_in, 3) / (3 * c_in) ** 0.5, torch.randn(N)
    x = torch.randn(B, T, c_in)
    for prec, act in (("fp16x2", "gelu"), ("fp16s", "lrelu")):
        layer = ops.ConvGemm(*packing.pack_conv(w, b, prec), act=act).to("cuda")
        xs = packing.to_act(x, prec).cuda()
        full = ops.alloc_act(B, T, N, prec, "cuda")
        layer(xs, B, T, out=full)
        one = ops.alloc_act(1, T, N, prec, "cuda")
        layer(xs[u:u + 1].contiguous(), 1, T, out=one)
        torch.cuda.synchronize()
        assert torch.equal(_bits(one[0]), _bits(full[u])), (prec, tile_split(B, T), tile_split(1, T))


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(33, 24), (2, 176), (130, 16)])
def test_tile_width_and_cta_group_do_not_change_bits(B, T):
    from autoformer_b200 import ops, packing
    torch.manual_seed(T)
    N, c_in = 512, 72
    w, b = torch.randn(N, c_in, 3) / (3 * c_in) ** 0.5, torch.randn(N)
    x = torch.randn(B, T, c_in)
    for prec in ("fp16x2", "fp32"):
        xs = packing.to_act(x, prec).cuda()
        outs = {}
        for bn in (64, 128, 256):
            for cta in (1, 2):
                layer = ops.ConvGemm(*packing.pack_conv(w, b, prec, block_n=bn), act="tanh").to("cuda")
                layer.cta_group = cta
                o = ops.alloc_act(B, T, N, prec, "cuda")
                o2 = torch.empty(B * T, N, device="cuda")
                layer(xs, B, T, out=o)
                layer(xs, B, T, out2=o2)
                torch.cuda.synchronize()
                outs[(bn, cta)] = (_bits(o), _bits(o2))
        ref = outs[(256, 2)]
        for key, (o, o2) in outs.items():
            assert torch.equal(o, ref[0]) and torch.equal(o2, ref[1]), (prec, key)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(33, 24), (130, 16), (2, 17)])
@pytest.mark.parametrize("act", ["none", "gelu", "tanh", "lrelu"])
def test_store_paths_agree_bit_for_bit(B, T, act):
    """packing.to_act of the fp32 out2 launch (simple 2) equals the bits of the out-only launch (simple 1: the fp16,
    split-fp16, bf16 and split-bf16 loops) and, with no activation, of out_raw beside an "f16" out."""
    from autoformer_b200 import ops, packing
    torch.manual_seed(B + T)
    N, c_in = 256, 40
    w, b = torch.randn(N, c_in, 3) / (3 * c_in) ** 0.5, torch.randn(N) * 2
    x = torch.randn(B, T, c_in)
    for prec in ("fp16x2", "fp16s", "bf16", "fp32"):
        layer = ops.ConvGemm(*packing.pack_conv(w, b, prec), act=act).to("cuda")
        xs = packing.to_act(x, prec).cuda()
        o2 = torch.empty(B * T, N, device="cuda")
        layer(xs, B, T, out2=o2)
        o = ops.alloc_act(B, T, N, prec, "cuda")
        layer(xs, B, T, out=o)
        torch.cuda.synchronize()
        assert torch.equal(_bits(o), _bits(packing.to_act(o2.view(B, T, N).cpu(), prec))), prec
        if act == "none" and prec == "fp16s":
            oa = ops.alloc_act(B, T, N, "f16", "cuda")
            raw = ops.alloc_act(B, T, N, "fp16s", "cuda")
            layer(xs, B, T, out=oa, out_raw=raw, out_fmt="f16", raw_fmt="fp16s")
            torch.cuda.synchronize()
            assert torch.equal(_bits(raw), _bits(packing.to_act(o2.view(B, T, N).cpu(), "fp16s")))
            assert torch.equal(_bits(oa), _bits(packing.to_act(o2.view(B, T, N).cpu(), "f16")))


# ------------------------------------------------------------------------------------------------ glue: data movement
def _special_values(n, seed):
    """fp32 values at the format edges: fp16 saturation, bf16 / fp16 rounding ties, fp16 subnormals, TF32 RNA ties."""
    g = torch.Generator().manual_seed(seed)
    sp = [65504.0, -65504.0, 65519.0, 65520.0, 70000.0, -1e6, 1e30, -1e30,
          1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8), 2.0 ** 100 * (1 + 2.0 ** -8),   # bf16 ties
          1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, -(1.0 + 2.0 ** -11), 2048.0 + 1.0, 2048.0 + 3.0,   # fp16 / tf32 ties
          2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -25, 2.0 ** -26, -(2.0 ** -24) * 5.5, 6.0e-5, 2.0 ** -14 * (1 - 2.0 ** -11),
          0.0, -0.0, 3.0e-8, -7.0e-6]
    v = torch.randn(n, generator=g) * torch.exp(torch.randn(n, generator=g) * 4)
    sp = torch.tensor(sp, dtype=torch.float32)
    v[:sp.numel() * (n // sp.numel())] = sp.repeat(n // sp.numel())
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("prec,round_tf32", [("tf32", True), ("tf32", False), ("bf16", True), ("fp32", True),
                                             ("fp16x2", True)])
def test_to_act_and_concat_bcast_stores(prec, round_tf32):
    from autoformer_b200 import ops, packing
    B, T, C1, C2, div = 3, 10, 36, 8, 2
    seq = _special_values(B * T // div * C1, 1).view(B, T // div, C1)
    vec = _special_values(B * C2, 2).view(B, C2)
    got = ops.to_act(seq.cuda(), prec, round_tf32=round_tf32).cpu()
    want = packing.to_act(seq, prec) if round_tf32 or prec != "tf32" else seq
    assert torch.equal(_bits(got), _bits(want)), prec
    got = ops.concat_bcast(seq.cuda(), vec.cuda(), T, div, prec, round_tf32=round_tf32).cpu()
    full = torch.cat([seq.repeat_interleave(div, dim=1), vec[:, None, :].expand(B, T, C2)], dim=-1)
    want = packing.to_act(full, prec) if round_tf32 or prec != "tf32" else full
    assert torch.equal(_bits(got), _bits(want)), prec
    if round_tf32:
        assert torch.equal(_bits(got), _bits(emulate._emu_concat_bcast(seq, vec, T, div, prec)))


def test_packing_to_act_saturates_fp16_like_the_kernels():
    """CPU: the host mirror of the operand formats saturates at +-65504 as the kernels' fp16 stores do
    (cvt.rn.satfinite), in one-term and two-term form, and keeps fp16's round-to-nearest-even and subnormals."""
    from autoformer_b200 import packing
    v = torch.tensor([[65504.0, 65519.0, 65520.0, 1e6, -70000.0, 1.0 + 2.0 ** -11, 2.0 ** -25, 3 * 2.0 ** -25]])
    one = packing.to_act(v, "fp16x2").float()
    assert one.tolist()[0] == [65504.0, 65504.0, 65504.0, 65504.0, -65504.0, 1.0, 0.0, 2.0 ** -23]
    two = packing.act_to_float(packing.to_act(v, "fp16s"), "fp16s")
    assert bool(torch.isfinite(two).all()) and two[0, 3] == 65504.0 and two[0, 4] == -65504.0


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["tf32", "bf16", "fp32", "fp16x2", "fp16s"])
@pytest.mark.parametrize("pad,L", [(0, 1), (3, 4), (3, 37), (0, 70)])
def test_transpose_pad(prec, pad, L):
    from autoformer_b200 import ops, packing
    B, C = 2, 44
    x = _special_values(B * C * L, L).view(B, C, L)
    got = ops.transpose_pad(x.cuda(), pad, prec).cpu()
    assert torch.equal(_bits(got), _bits(emulate._emu_transpose_pad(x, pad, prec)))
    y = F.pad(x, (pad, pad), mode="reflect") if pad else x
    assert torch.equal(_bits(got), _bits(packing.to_act(y.transpose(1, 2).contiguous(), prec)))
    if prec == "tf32":
        raw = ops.transpose_pad(x.cuda(), pad, prec, round_tf32=False).cpu()
        assert torch.equal(_bits(raw), _bits(y.transpose(1, 2).contiguous()))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,C", [(torch.float16, 8), (torch.bfloat16, 24), (torch.float32, 4), (torch.float32, 12)])
@pytest.mark.parametrize("reflect", [1, 2, 3, 5, 9])
def test_reflect_halo(dtype, C, reflect):
    from autoformer_b200 import ops
    B, L, row0, spare = 3, reflect + 1, reflect + 2, 3
    rows = row0 + L + reflect + spare
    torch.manual_seed(reflect)
    buf = torch.randn(B, rows, C).to(dtype)
    buf[:, :row0] = float("nan")                      # everything outside the interior is a sentinel ...
    buf[:, row0 + L:] = float("nan")
    got = ops.reflect_halo(buf.cuda(), row0, L, reflect).cpu()
    want = emulate._emu_reflect_halo(buf.clone(), row0, L, reflect)
    assert torch.equal(_bits(got), _bits(want))
    inner = buf[:, row0:row0 + L].float().transpose(1, 2)
    pad = F.pad(inner, (reflect, reflect), mode="reflect").transpose(1, 2).to(dtype)
    assert torch.equal(_bits(got[:, row0 - reflect:row0 + L + reflect]), _bits(pad))
    # ... and the rows beyond the halo stay untouched
    assert bool(torch.isnan(got[:, :row0 - reflect].float()).all()) and bool(torch.isnan(got[:, row0 + L + reflect:].float()).all())


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["tf32", "bf16", "fp32", "fp16x2"])
@pytest.mark.parametrize("L,pad,hop,rows", [(1000, 384, 256, 8), (385, 384, 256, 6), (77, 12, 16, 9), (13, 12, 8, 12)])
def test_audio_frames(prec, L, pad, hop, rows):
    """L not a multiple of hop, L just above pad, rows beyond the padded signal (zero-filled)."""
    from autoformer_b200 import ops, packing
    B = 3
    torch.manual_seed(L)
    audio = torch.randn(B, L)
    got = ops.audio_frames(audio.cuda(), pad, hop, rows, prec).cpu()
    assert torch.equal(_bits(got), _bits(emulate._emu_audio_frames(audio, pad, hop, rows, prec)))
    padded = F.pad(audio[:, None], (pad, pad), mode="reflect")[:, 0]
    sig = F.pad(padded, (0, max(0, rows * hop - padded.shape[1])))[:, :rows * hop]
    assert torch.equal(_bits(got), _bits(packing.to_act(sig.reshape(B, rows, hop), prec)))
    if rows * hop > L + 2 * pad:
        assert not packing.act_to_float(got, prec).view(B, -1)[:, L + 2 * pad:].any()


# ------------------------------------------------------------------------------------------------ glue: arithmetic
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["tf32", "bf16", "fp32", "fp16x2"])
@pytest.mark.parametrize("rows,bins,bins_pad", [(37, 513, 520), (5, 9, 16), (300, 64, 64)])
def test_complex_mag(prec, rows, bins, bins_pad):
    from autoformer_b200 import ops, packing
    torch.manual_seed(bins)
    spec = torch.randn(rows, 2 * bins) * torch.exp(torch.randn(rows, 1) * 2)
    got = packing.act_to_float(ops.complex_mag(spec.cuda(), bins, bins_pad, prec).cpu(), prec)[0]
    assert got.shape == (rows, bins_pad)
    ref = torch.zeros(rows, bins_pad, dtype=torch.float64)
    ref[:, :bins] = torch.hypot(spec[:, :bins].double(), spec[:, bins:].double())
    bound = 4 * U * ref + half_ulp(ref * (1 + 4 * U), prec)        # a*a + b*b (maybe fused) and sqrtf: a few ulp
    check_bound(got, ref, bound, "complex_mag")
    emu = packing.act_to_float(emulate._emu_complex_mag(spec, bins, bins_pad, prec), prec)[0]
    check_bound(got, emu.double(), 2 * bound, "complex_mag vs emulate")
    assert not got[:, bins:].any()


def _mono_ref(x, w, bias):
    K = w.shape[0]
    xp = F.pad(x.double().transpose(1, 2), (K // 2, K // 2), mode="reflect")
    v = F.conv1d(xp, w.double().t().unsqueeze(0)).squeeze(1) + bias
    s = F.conv1d(xp.abs(), w.double().abs().t().unsqueeze(0)).squeeze(1) + abs(bias)
    return v, s


@pytest.mark.gpu
@pytest.mark.parametrize("K", [3, 5, 7, 15])
@pytest.mark.parametrize("C", [4, 32, 64])
@pytest.mark.parametrize("Lsel", ["min", "tile", "long"])
def test_conv_to_mono_tanh(K, C, Lsel):
    from autoformer_b200 import ops
    L = {"min": K // 2 + 1, "tile": 128, "long": 1037}[Lsel]
    B = 3
    torch.manual_seed(K * C + L)
    x = torch.randn(B, L, C)
    w = torch.randn(K, C) / (K * C) ** 0.5
    bias = 0.3
    out = ops.conv_to_mono_tanh(x.cuda(), w.cuda(), bias).cpu()
    v, s = _mono_ref(x, w, bias)
    bound = (K * C + 2) * U * s + 2e-6
    check_bound(out, torch.tanh(v), bound, "mono")
    check_bound(out, emulate._emu_conv_to_mono_tanh(x, w, bias).double(), bound + 2 ** -23, "mono vs emulate")


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 300])
@pytest.mark.parametrize("K", [4, 36, 768])
@pytest.mark.parametrize("N", [4, 256, 1024])
def test_linear_l2norm_and_rows(B, K, N):
    from autoformer_b200 import ops
    torch.manual_seed(B + K + N)
    h, w, b = torch.randn(B, K), torch.randn(N, K) / K ** 0.5, torch.randn(N) * 0.1
    e = h.double() @ w.double().t() + b.double()
    s = h.double().abs() @ w.double().abs().t() + b.double().abs()
    E = (K + 2) * U * s                                          # fp32 fma chain over K
    nrm = e.norm(dim=-1, keepdim=True)
    n = e / nrm
    # ||e||: N squares summed in fp32 (+ error of e itself), rsqrtf (2 ulp)
    rel = 0.5 * (N + 2) * U + 2 * U + (E.norm(dim=-1, keepdim=True) / nrm) * 2
    En = E / nrm + n.abs() * rel + U * n.abs()
    raw, normed = ops.linear_rows(h.cuda(), w.cuda(), b.cuda(), want_raw=True, want_normed=True)
    check_bound(raw, e, E, "linear_rows raw")
    check_bound(normed, n, En, "linear_rows normed")
    only_raw, none = ops.linear_rows(h.cuda(), w.cuda(), b.cuda(), want_raw=True, want_normed=False)
    assert none is None and torch.equal(only_raw, raw)
    _, only_n = ops.linear_rows(h.cuda(), w.cuda(), b.cuda(), want_raw=False, want_normed=True)
    assert torch.equal(only_n, normed)
    l2 = ops.linear_l2norm(h.cuda(), w.cuda(), b.cuda())
    check_bound(l2, n, En, "linear_l2norm")
    check_bound(l2, emulate._emu_linear_l2norm(h, w, b).double(), En + U * n.abs(), "linear_l2norm vs emulate")
