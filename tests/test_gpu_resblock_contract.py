"""Op-level contract of the fused MelGAN ResnetBlock kernels, element by element against fp64:

  resblock_kernel<C>             avc_resblock, split bf16, C = 32 / 64 (MelGAN precision "fp32")
  resblock2_kernel<C, RAGGED>    avc_resblock2, "fp16s", C = 32 / 64, fixed length or per-utterance lengths
  resblock2_big_kernel<RAGGED>   avc_resblock2, "fp16s", C = 128 on CTA pairs

Every launch is held to two independent checks against references built from the RAW PyTorch-layout weights (split
with packing.split_bf16 / split_f16, never read back from the packed tiles, so a packing-layout error fails too):
  * a per-element worst-case bound.  The reference forms exactly the products the kernel forms (v1: a_hi w_hi +
    a_lo w_hi + a_hi w_lo; v2 k3: xa (w_hi + w_lo) with the one-fp16 operand xa emulated bit for bit; v2 k1 and
    shortcut: three products).  The bound chains (K + 4) U S of GEMM1, the LeakyReLU rounding and the two-term store of
    the intermediate (RN bf16 split for v1, avc_pipe.cuh's truncating fp16 split for v2) through |W1| into y, then adds
    what the output format costs.  Worst case, so never flaky.  It catches what moves single elements by O(|y|): a halo
    row off by one, a wrong tap at a tile seam, a swizzled chunk, a tile given to the wrong utterance, a wrong slope;
  * a global rel-L2 against torch fp64 with operands rounded only where the kernel rounds them (3e-5 for v1, 2e-5 for
    v2).  It catches a dropped precision term (the intermediate's lo term, a weight's lo term) whose error spreads
    thinly over every element and can hide inside the worst-case bound;
  * and every output goes into NaN-filled buffers with spare rows, spare channels and a spare utterance: exactly the
    expected region becomes finite (the sentinel check), which catches a missing or stray store.
What each input magnitude class is held to:
  * "normal" (|x| ~ 3): sentinel, bound and rel-L2;
  * "tiny" (x and biases ~ 2^-17, so the k3 operand, the intermediate and the outputs are fp16 subnormals): sentinel and
    bound.  No rel-L2: the two-term fp16 stores quantise to the subnormal step 2^-24, a few percent of these values,
    so a global relative norm measures that quantisation, not the kernel; the bound carries the 2^-24 floors instead;
  * "huge" (|x| ~ 2e4, some at 65504): sentinel, every output finite and the two-term outputs saturated at 65504.  No
    bound or rel-L2: the intermediate and the outputs saturate (cvt.rn.satfinite), which no fp64 reference follows; the
    contract there is finite, saturated values instead of inf / NaN.
The CPU tests below run the checker against the emulation of tests/emulate.py (it must pass) and against a stand-in
with injected faults (each must fail, in the check named for it).

The GPU cases are declared in CASES; a CPU test mirrors the launch grid and checks that they reach every cell of
kernel instantiation x output form x geometry class.
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import rel_l2
from tests import emulate
from tests.test_gpu_kernel_contract import U, check_bound, check_sentinel, half_ulp, nan_buf

F16_MAX = 65504.0
NAN = float("nan")
SPARE_ROWS, SPARE_CH = 3, 8
REL_TOL = {1: 3e-5, 2: 2e-5}


# ------------------------------------------------------------------------------------------------ the case matrix
INSTS = {  # kernel instantiation -> (version, C, ragged)
    "v1_c32": (1, 32, False), "v1_c64": (1, 64, False),
    "v2_c32": (2, 32, False), "v2_c64": (2, 64, False), "v2_c32_ragged": (2, 32, True), "v2_c64_ragged": (2, 64, True),
    "big": (2, 128, False), "big_ragged": (2, 128, True),
}
V1_FORMS = ("out", "out_reflect", "out_raw", "out2", "out+out_raw", "out_raw+out2")
V2_FORMS = ("y", "y_act", "out2", "wav3", "wav5", "wav7")
BIG_FORMS = ("y", "y_act")
GEOS = ("one_tile", "persist", "many_per_utt")
BIG_GEOS = GEOS + ("phantom", "pair_split", "b1_l128")
MAX_DIL = {32: 16, 64: 16, 128: 12}        # RbCfg / Rb2Cfg::kMaxDilation, big::kMaxDilation
DILS = ("max", 1, 3, 9)
REFLECTS = (9, 16, 0, 1)


def inst_forms(inst):
    version, C, _ = INSTS[inst]
    if version == 1:
        return V1_FORMS
    return BIG_FORMS if C == 128 else (V2_FORMS if C == 32 else V2_FORMS[:3])


def inst_geos(inst):
    return BIG_GEOS if INSTS[inst][1] == 128 else GEOS


def form_stride(form):
    """Rows per tile: 128, or 128 - (K - 1) for the fused output convolution (tiles overlap by K - 1)."""
    return 128 - (int(form[3:]) - 1) if form.startswith("wav") else 128


def launch_grid(inst, form, B, L, lengths, n_sms):
    """Mirror of launch / launch2 / launch_resblock2_big: (tiles per utterance, n_tiles, CTAs, tiles per CTA).
    For C = 128 the unit is a pair: CTAs = 2 x min(ceil(n_tiles / 2), SMs / 2), tiles per CTA = pair iterations."""
    version, C, ragged = INSTS[inst]
    S = form_stride(form)
    per_utt = [-(-n // S) for n in lengths] if ragged else [-(-L // S)] * B
    n_tiles = sum(per_utt)
    if C == 128:
        n_pairs = (n_tiles + 1) // 2
        pairs = min(n_pairs, n_sms // 2)
        return per_utt, n_tiles, 2 * pairs, -(-n_pairs // pairs)
    ctas = min(n_tiles, n_sms * (2 if C == 32 else 1))
    return per_utt, n_tiles, ctas, -(-n_tiles // ctas)


def persist_tiles(inst):
    """Tiles some CTA must run before every barrier of the kernel has completed in both parities and every buffer has
    been reloaded.  resblock2_kernel double-buffers its window (buffer it & 1, win_free[buf] waited with parity
    (use - 1) & 1, use = it >> 1): both buffers reloaded twice, hence both parities of both win_free barriers, need
    it = 0..5.  resblock_kernel and the C = 128 kernel load one window per tile: three iterations (phases 0, 1, 0)."""
    version, C, _ = INSTS[inst]
    return 6 if version == 2 and C < 128 else 3


def geometry_classes(inst, form, B, L, lengths, n_sms):
    per_utt, n_tiles, _, per_cta = launch_grid(inst, form, B, L, lengths, n_sms)
    cls = set()
    if n_tiles == 1:
        cls.add("one_tile")
    if per_cta >= persist_tiles(inst):
        cls.add("persist")
    if max(per_utt) >= 3:
        cls.add("many_per_utt")
    if INSTS[inst][1] == 128:
        if n_tiles % 2:
            cls.add("phantom")
        owner = [b for b, k in enumerate(per_utt) for _ in range(k)]
        if any(owner[2 * u] != owner[2 * u + 1] for u in range(n_tiles // 2)):
            cls.add("pair_split")
        if B == 1 and L == 128:
            cls.add("b1_l128")
    return cls


def class_exempt(inst, form, geo):
    """The one cell that cannot exist: a fixed-length waveform launch never has one tile (L is a multiple of 128 and a
    tile covers 128 - (K - 1) rows)."""
    return geo == "one_tile" and form.startswith("wav") and not INSTS[inst][2]


def case_shape(case, n_sms):
    """(B, L, lengths) of a case; `persist` is sized from the SM count so that some CTA runs persist_tiles tiles."""
    inst, geo = case["inst"], case["geo"]
    _, C, ragged = INSTS[inst]
    if "B" in case:
        B, L = case["B"], case["L"]
        return B, L, case.get("lengths") or [L] * B
    if geo == "persist":
        B = 3
        for k in range(2, 4096):
            L = 128 * k
            lengths = [L, L - 677, L // 2 + 11] if ragged else [L] * B
            if all("persist" in geometry_classes(inst, f, B, L, lengths, n_sms) for f in inst_forms(inst)):
                return B, L, lengths
        raise AssertionError("no persist shape")
    B, L, lengths = {
        "one_tile": (1, 128, [100]),
        "many_per_utt": (2, 640, [640, 300]),
        "phantom": (2, 384, [384, 130]) if ragged else (1, 384, None),
        "pair_split": (3, 128, [100, 128, 37]),
        "b1_l128": (1, 128, [128]),
    }[geo]
    return B, L, (lengths if ragged else [L] * B)


def _declare_cases():
    cases = []
    for j, inst in enumerate(INSTS):
        C = INSTS[inst][1]
        for i, geo in enumerate(inst_geos(inst)):
            k = i + j
            dil = DILS[k % 4]
            R = REFLECTS[(k + i // 4) % 4]
            cases.append(dict(inst=inst, geo=geo, d=MAX_DIL[C] if dil == "max" else dil, R=R,
                              row0=R + (2 if k % 2 else 0), mag="normal", seed=100 * j + i))
    # magnitude classes: operands in fp16's subnormal range (biases scaled with them), and near its limit
    for j, inst in enumerate(("v2_c32", "v2_c64_ragged", "big", "big_ragged")):
        for mag in ("tiny", "huge"):
            cases.append(dict(inst=inst, geo="many_per_utt", d=(3, 9, 1, 12)[j], R=(1, 16, 9, 0)[j], row0=(1, 16, 11, 2)[j],
                              mag=mag, seed=7000 + 10 * j + len(mag)))
    # the shapes of the op-level tests this file replaces (test_resblock2_matches_torch, test_fused_resblock_matches_torch)
    for version, shapes in ((2, LEGACY_V2), (1, LEGACY_V1)):
        for (C, d, B, L) in shapes:
            inst = f"v{version}_c{C}" if C < 128 else "big"
            cases.append(dict(inst=inst, geo="legacy", d=d, R=9, row0=9, mag="normal", seed=100 * C + d, B=B, L=L))
    return cases


# (C, d, B, L) of the removed tests: more tiles than CTAs (B = 150 / 700 / 301), many tiles per utterance (37 / 41 x 128)
LEGACY_V2 = [(64, 1, 2, 256), (64, 9, 1, 384), (32, 3, 3, 128), (32, 9, 2, 640), (64, 3, 150, 128), (32, 1, 700, 128),
             (64, 9, 2, 128 * 37), (32, 3, 2, 128 * 37), (128, 1, 2, 256), (128, 9, 1, 384), (128, 3, 3, 128),
             (128, 3, 301, 128), (128, 9, 2, 128 * 41)]
LEGACY_V1 = [(64, 1, 2, 256), (64, 9, 1, 384), (32, 3, 3, 128), (32, 9, 2, 640), (64, 3, 150, 128)]
CASES = _declare_cases()


def _case_id(c):
    return f"{c['inst']}-{c['geo']}-d{c['d']}-R{c['R']}-{c['mag']}" + (f"-B{c['B']}L{c['L']}" if "B" in c else "")


def test_resblock_case_matrix_covers_every_cell():
    """CPU: for several SM counts, the declared cases reach every (instantiation x form x geometry) cell through the
    mirrored launch grid, every dilation class and reflect width, row0 > reflect, both magnitude extremes, and every
    shape and form of the tests they replace."""
    for n_sms in (148, 132, 160):
        cells = set()
        for c in CASES:
            B, L, lengths = case_shape(c, n_sms)
            for f in inst_forms(c["inst"]):
                for g in geometry_classes(c["inst"], f, B, L, lengths, n_sms):
                    cells.add((c["inst"], f, g))
                if c["geo"] != "legacy":
                    assert c["geo"] in geometry_classes(c["inst"], f, B, L, lengths, n_sms) or \
                        class_exempt(c["inst"], f, c["geo"]), (_case_id(c), f)
        need = {(i, f, g) for i in INSTS for f in inst_forms(i) for g in inst_geos(i)}
        for c in CASES:          # the double-buffered window: some CTA runs six tiles, so both buffers go round twice
            if c["geo"] == "persist":
                for f in inst_forms(c["inst"]):
                    per_cta = launch_grid(c["inst"], f, *case_shape(c, n_sms), n_sms)[3]
                    assert per_cta >= (6 if c["inst"].startswith("v2") else 3), (_case_id(c), f, n_sms, per_cta)
        impossible = {(i, f, g) for i, f, g in need if class_exempt(i, f, g)}
        assert impossible == {("v2_c32", f, "one_tile") for f in ("wav3", "wav5", "wav7")}
        assert all(launch_grid(i, f, 1, 128, [128], n_sms)[1] == 2 for i, f, _ in impossible)
        assert need - impossible <= cells, (n_sms, sorted(need - impossible - cells))
    for C in (32, 64, 128):
        dils = {c["d"] for c in CASES if INSTS[c["inst"]][1] == C and c["geo"] != "legacy"}
        assert dils >= {1, 3, 9, MAX_DIL[C]}, (C, dils)
    assert {c["R"] for c in CASES} >= {0, 1, 9, 16} and any(c["row0"] > c["R"] for c in CASES)
    for inst in ("v2_c32", "v2_c64_ragged", "big", "big_ragged"):
        assert {c["mag"] for c in CASES if c["inst"] == inst} == {"normal", "tiny", "huge"}
    legacy = {(INSTS[c["inst"]][0], INSTS[c["inst"]][1], c["d"], c["B"], c["L"]) for c in CASES if c["geo"] == "legacy"}
    assert {(2,) + s for s in LEGACY_V2} | {(1,) + s for s in LEGACY_V1} <= legacy
    # the removed tests' forms: v1 out (reflect 9) + out_raw, out2, out alone; v2 y (reflect 9), y_act, out2, wav 3/5/7
    assert {"out+out_raw", "out2", "out"} <= set(V1_FORMS) and {"y", "y_act", "out2", "wav3", "wav5", "wav7"} <= set(V2_FORMS)


# ------------------------------------------------------------------------------------------------ roundings (CPU, fp32)
_SLOPE = {s: torch.tensor(s, dtype=torch.float32) for s in (0.2, 0.25)}


def lrelu32(v, slope=0.2):
    """fmaxf(v, 0.2f * v) in fp32: one IEEE multiply, exact on the CPU."""
    return torch.maximum(v, v * _SLOPE[slope])


def sat_f16(v):
    """cvt.rn.satfinite.f16.f32: round to nearest, out-of-range values to +-65504 (NaN stays NaN)."""
    return v.clamp(-F16_MAX, F16_MAX).half()


def xa_operand(hi, lo, slope=0.2):
    """The k3 operand of avc_resblock2, bit for bit: fp16_satfinite(max(v, 0.2f v)) with v = fl32(hi + lo)."""
    return sat_f16(lrelu32(hi.float() + lo.float(), slope))


def split_f16_trunc(v):
    """avc_pipe.cuh split_f16_pair_trunc: hi = v with its 13 low mantissa bits cleared, lo = v - hi, both packed with
    cvt.rn.satfinite."""
    v = v.float().contiguous()
    h = (v.view(torch.int32) & -8192).view(torch.float32)
    return sat_f16(h), sat_f16(v - h)


def split_two(v, fmt):
    """Two-term store of fp32 values: "bf16s" (v1: RN bf16 split) or "f16t" (v2: truncating fp16 split)."""
    from autoformer_b200 import packing
    return packing.split_bf16(v.float()) if fmt == "bf16s" else split_f16_trunc(v)


def store_err(mag, fmt):
    """|stored hi + lo - v| for |v| <= mag."""
    if fmt == "bf16s":
        return half_ulp(mag, "fp32")
    return 2 * half_ulp(mag, "fp16s")       # hi truncated: |lo| < 2^-10 |v|, then lo's RN and both subnormal floors


def lo_max(mag, fmt):
    """|lo| of the two-term store for |v| <= mag."""
    return mag * 2.0 ** -8 if fmt == "bf16s" else mag * 2.0 ** -10 + 2.0 ** -24


def lrelu64(v, slope=0.2):
    return torch.where(v > 0, v, slope * v)


def conv(a, w, d=1):
    """[B][rows][Cin] x (Cout, Cin, k), dilation d -> [B][rows - (k - 1) d][Cout] in fp64."""
    return F.conv1d(a.double().transpose(1, 2), w.double(), dilation=d).transpose(1, 2)


# ------------------------------------------------------------------------------------------------ the fp64 reference
def make_weights(C, seed, bias_scale=1.0):
    g = torch.Generator().manual_seed(seed)
    w3 = torch.randn(C, C, 3, generator=g) / (3 * C) ** 0.5
    w1, wsc = torch.randn(C, C, 1, generator=g) / C ** 0.5, torch.randn(C, C, 1, generator=g) / C ** 0.5
    b3, b1, bsc = (torch.randn(C, generator=g) * bias_scale for _ in range(3))
    return w3, b3, w1, b1, wsc, bsc


class Ref:
    """fp64 reference of one block over a batch: y, LeakyReLU(y) and their element bounds ([B][L][C]), and the rel-L2
    reference (y_l2, ya_l2).  Rows whose receptive field holds padding (NaN input) come out NaN and are never checked.
    The bound holds while nothing saturates: the "huge" magnitude class is checked for finite, saturated outputs
    instead, and the "tiny" class skips only the rel-L2 (see the module docstring)."""

    def __init__(self, version, raw, inp, d, L):
        from autoformer_b200 import packing
        w3, b3, w1, b1, wsc, bsc = raw
        C = w3.shape[0]
        split = packing.split_bf16 if version == 1 else packing.split_f16
        (w3h, w3l), (w1h, w1l), (wsh, wsl) = [tuple(t.double() for t in split(w)) for w in (w3, w1, wsc)]
        bias1 = (b1.float() + bsc.float()).double()        # the packed bias the kernel adds (b1 + bsc in fp32)
        if version == 1:
            xa_buf, x_buf = inp
            ah, al = xa_buf[..., :C].double(), xa_buf[..., C:2 * C].double()
            z = conv(ah + al, w3h, d) + conv(ah, w3l, d)
            s = conv(ah.abs() + al.abs(), w3h.abs(), d) + conv(ah.abs(), w3l.abs(), d)
            z_l2 = conv(ah + al, w3, d)
            xh, xl = x_buf[:, :L, :C].double(), x_buf[:, :L, C:2 * C].double()
            k1, self.fmt = 9 * C, "bf16s"
        else:
            x_buf = inp
            xa = xa_operand(x_buf[..., :C], x_buf[..., C:2 * C]).double()
            z = conv(xa, w3h + w3l, d)
            s = conv(xa.abs(), w3h.abs() + w3l.abs(), d)
            z_l2 = conv(xa, w3, d)
            xh, xl = x_buf[:, d:d + L, :C].double(), x_buf[:, d:d + L, C:2 * C].double()
            k1, self.fmt = 6 * C, "f16t"
        fmt = self.fmt
        b3d = b3.double()
        mid = lrelu64(z + b3d)
        e_mid = (k1 + 4) * U * (s + b3d.abs()) + 3 * U * mid.abs()   # GEMM1 + bias, 0.2f * v, the fp32 value itself
        mh, ml = (t.double() for t in split_two(mid, fmt))
        m = mid.abs() + e_mid
        dv = e_mid + 2 * store_err(m, fmt)                  # |(hi + lo) kernel - (hi + lo) reference|
        dh = dv + 2 * lo_max(m, fmt)                        # |hi kernel - hi reference|
        y = conv(mh + ml, w1h) + conv(mh, w1l) + conv(xh + xl, wsh) + conv(xh, wsl) + bias1
        S2 = (conv(mh.abs() + ml.abs(), w1h.abs()) + conv(mh.abs(), w1l.abs()) + conv(xh.abs() + xl.abs(), wsh.abs())
              + conv(xh.abs(), wsl.abs()) + bias1.abs())
        self.y = y
        self.e_y = (6 * C + 4) * U * S2 + conv(dv, w1h.abs()) + conv(dh, w1l.abs())
        self.ya = lrelu64(y)
        self.e_a = self.e_y + 2 * U * self.ya.abs()
        mid_l2 = sum(t.double() for t in split_two(lrelu64(z_l2 + b3d), fmt))
        self.y_l2 = conv(mid_l2, w1) + conv(xh + xl, wsc) + b1.double() + bsc.double()
        self.ya_l2 = lrelu64(self.y_l2)

    def values(self, act):
        return (self.ya, self.e_a, self.ya_l2) if act else (self.y, self.e_y, self.y_l2)


def wav_reference(ya, e_a, ya_l2, w_out, b_out, n):
    """The generator's output layer fused into the epilogue (tanh(Conv1d(C -> 1, K)) over ReflectionPad1d(K // 2) of
    LeakyReLU(y), mirrored at the utterance's own last sample n - 1) for one utterance: (value, bound, rel-L2 value).
    The bound carries the staged LeakyReLU(y)'s bound through |w_out|; tanh_fast costs ~1e-7 absolute."""
    K, C = w_out.shape
    pad = lambda t: F.pad(t[:n].double().t()[None], (K // 2, K // 2), mode="reflect")
    wk = w_out.double().t().unsqueeze(0)                                            # (1, C, K)
    v = F.conv1d(pad(ya), wk)[0, 0] + b_out
    s = F.conv1d(pad(ya.abs()), wk.abs())[0, 0] + abs(b_out)
    bound = F.conv1d(pad(e_a), wk.abs())[0, 0] + (K * C + 2) * U * s + 2e-6
    return torch.tanh(v), bound, torch.tanh(F.conv1d(pad(ya_l2), wk)[0, 0] + b_out)


# ------------------------------------------------------------------------------------------------ launch geometry
class Geo:
    """Buffers of one case: inputs with NaN spare channels, a NaN spare utterance and NaN padding past each utterance's
    reflected halo; outputs allocated per form (NaN, spare rows / channels / utterance)."""

    def __init__(self, case, B, L, lengths, device="cpu"):
        self.case, self.B, self.L, self.lengths = case, B, L, lengths
        self.version, self.C, self.ragged = INSTS[case["inst"]]
        self.d, self.R, self.row0, self.mag = case["d"], case["R"], case["row0"], case["mag"]
        self.device = device

    def make_inputs(self, seed):
        from autoformer_b200 import packing
        B, L, C, d = self.B, self.L, self.C, self.d
        g = torch.Generator().manual_seed(seed)
        scale = {"normal": 3.0, "tiny": 2.0 ** -17, "huge": 2.0e4}[self.mag]
        if self.version == 1:
            xa = torch.full((B + 1, L + 2 * d, 2 * C + SPARE_CH), NAN, dtype=torch.bfloat16)
            x = torch.full((B + 1, L, 2 * C + SPARE_CH), NAN, dtype=torch.bfloat16)
            v = torch.randn(B, L, C, generator=g)
            x[:B, :, :2 * C] = packing.to_act(v, "fp32")
            xs = packing.act_to_float(x[:B, :, :2 * C], "fp32").double()
            xp = F.pad(F.leaky_relu(xs, 0.2).transpose(1, 2), (d, d), mode="reflect").transpose(1, 2)
            xa[:B, :, :2 * C] = packing.to_act(xp.float(), "fp32")
            return xa, x
        x = torch.full((B + 1, L + 2 * d, 2 * C + SPARE_CH), NAN, dtype=torch.float16)
        for b, n in enumerate(self.lengths):
            v = torch.randn(n, C, generator=g) * scale
            if self.mag == "huge":           # a few at the limit itself
                v.view(-1)[::97] = F16_MAX * torch.sign(v.view(-1)[::97])
            xp = F.pad(v.t()[None], (d, d), mode="reflect")[0].t()        # the caller's reflected halo at 0 and n
            x[b, :n + 2 * d, :2 * C] = packing.to_act(xp[None].contiguous(), "fp16s")[0]
        return x

    def outputs(self, form):
        """Output descriptors of a form: (name, act, row0, reflect)."""
        R = self.R
        if self.version == 1:
            Rr = max(R, 1)
            halo_out = ("out", True, max(self.row0, Rr), Rr)
            return {"out": [("out", True, self.row0, 0)], "out_reflect": [halo_out], "out_raw": [("out_raw", False, 0, 0)],
                    "out2": [("out2", True, 0, 0)], "out+out_raw": [halo_out, ("out_raw", False, 0, 0)],
                    "out_raw+out2": [("out_raw", False, 0, 0), ("out2", True, 0, 0)]}[form]
        if form == "y":
            return [("y", False, self.row0, R)]
        if form == "y_act":
            return [("y", True, self.row0 - R, 0)]
        if form == "out2":
            return [("out2", True, 0, 0)]
        return [("wav", True, 0, 0)]

    def alloc(self, name, row0, reflect):
        B, L, C = self.B, self.L, self.C
        dt = torch.bfloat16 if self.version == 1 else torch.float16
        mk = lambda shape, dtype: torch.full(shape, NAN, dtype=dtype, device=self.device)
        if name in ("out", "y"):
            return mk((B + 1, row0 + L + reflect + SPARE_ROWS, 2 * C + SPARE_CH), dt)
        if name == "out_raw":
            return mk((B + 1, L, 2 * C + SPARE_CH), dt)
        if name == "out2":
            return mk((B * L + SPARE_ROWS, C + 4), torch.float32)
        return mk((B * L + L,), torch.float32)            # wav: a spare utterance behind the batch

    def ran_rows(self, b, S=128):
        """Rows of utterance b covered by the tiles that run (all of them at fixed length)."""
        n = self.lengths[b]
        return min(self.L, -(-n // S) * S) if self.ragged else self.L

    def mono(self, K):
        g = torch.Generator().manual_seed(K)
        return torch.randn(K, self.C, generator=g) / (K * self.C) ** 0.5, 0.05 * K


# ------------------------------------------------------------------------------------------------ the checker
def check_launch(geo, ref, form, bufs):
    """Every check of one launch; returns [(check, message)] of those that failed: "sentinel" (exactly the expected
    region written), "bound" (per element), "rel-l2" (global), "saturation" (near the fp16 limit)."""
    fails = []

    def run(kind, fn):
        try:
            fn()
        except AssertionError as e:
            fails.append((kind, str(e)))

    B, L, C = geo.B, geo.L, geo.C
    fmt = ref.fmt
    for (name, act, row0, R), buf in zip(geo.outputs(form), bufs):
        buf = buf.cpu()
        val, bnd, v_l2 = ref.values(act)
        must = torch.zeros(buf.shape, dtype=torch.bool)
        may = torch.zeros(buf.shape, dtype=torch.bool)
        got_all, ref_all, bnd_all, l2_all = [], [], [], []
        for b, n in enumerate(geo.lengths):
            S = form_stride(form) if name == "wav" else 128
            ran = geo.ran_rows(b, S)
            if name in ("out", "y"):
                two = buf[b, :, :2 * C].double()
                got = two[:, :C] + two[:, C:]
                halo = [(row0 - k, k) for k in range(1, R + 1)]
                if not geo.ragged or n == L:
                    halo += [(row0 + L - 1 + k, L - 1 - k) for k in range(1, R + 1)]
                r_idx = torch.tensor([row0 + t for t in range(n)] + [r for r, _ in halo], dtype=torch.long)
                t_idx = torch.tensor(list(range(n)) + [t for _, t in halo], dtype=torch.long)
                must[b, r_idx, :2 * C] = True
                may[b, r_idx, :2 * C] = True
                may[b, row0:row0 + ran, :2 * C] = True
                if ran >= L:
                    may[b, row0 + L:row0 + L + R, :2 * C] = True
                got_all.append(got[r_idx])
                ref_all.append(val[b, t_idx])
                bnd_all.append(bnd[b, t_idx] + store_err(val[b, t_idx].abs() + bnd[b, t_idx], fmt))
                l2_all.append(v_l2[b, t_idx])
            elif name == "out_raw":
                two = buf[b, :, :2 * C].double()
                must[b, :n, :2 * C] = True
                may[b, :ran, :2 * C] = True
                got_all.append((two[:, :C] + two[:, C:])[:n])
                ref_all.append(val[b, :n])
                bnd_all.append(bnd[b, :n] + store_err(val[b, :n].abs() + bnd[b, :n], fmt))
                l2_all.append(v_l2[b, :n])
            elif name == "out2":
                must[b * L:b * L + n, :C] = True
                may[b * L:b * L + ran, :C] = True
                got_all.append(buf[b * L:b * L + n, :C].double())
                ref_all.append(val[b, :n])
                bnd_all.append(bnd[b, :n])
                l2_all.append(v_l2[b, :n])
            else:
                K = int(form[3:])
                w_out, b_out = geo.mono(K)
                wv, wb, wl = wav_reference(val[b], bnd[b], v_l2[b], w_out, b_out, n)
                must[b * L:b * L + ran] = True
                may[b * L:b * L + ran] = True
                got_all.append(buf[b * L:b * L + n].double())
                ref_all.append(wv)
                bnd_all.append(wb)
                l2_all.append(wl)
                if ran > n:                                 # the last tile's samples past the utterance's end are 0
                    run("bound", lambda b=b, n=n, ran=ran: _assert_zero(buf[b * L + n:b * L + ran], f"{name}[{b}] tail"))
        got, want, bound, want_l2 = (torch.cat(t) for t in (got_all, ref_all, bnd_all, l2_all))
        what = f"{form}/{name}"
        if geo.ragged or name == "wav":
            run("sentinel", lambda: _check_written(buf, must, may, what))
        else:
            run("sentinel", lambda: check_sentinel(buf, must, "sentinel " + what))
        if geo.mag == "huge":
            run("saturation", lambda: _check_saturation(got, name, what))
            continue
        run("bound", lambda: check_bound(got, want, bound, "bound " + what))
        if geo.mag == "normal":
            run("rel-l2", lambda: _check_rel_l2(got, want_l2, REL_TOL[geo.version], what))
    return fails


def _assert_zero(t, what):
    assert bool((t == 0).all()), f"{what}: not zero"


def _check_written(buf, must, may, what):
    fin = torch.isfinite(buf.float())
    assert bool(fin[must].all()), f"sentinel {what}: {int((~fin[must]).sum())} expected elements not written / not finite"
    assert not bool(fin[~may].any()), f"sentinel {what}: {int(fin[~may].sum())} elements written outside the output"


def _check_rel_l2(got, want, tol, what):
    e = rel_l2(got, want)
    assert e < tol, f"rel-l2 {what}: {e:.3g} >= {tol}"


def _check_saturation(got, name, what):
    """Near the fp16 limit the contract is that every output stays finite (the satfinite packs) and the two-term outputs
    saturate instead of overflowing."""
    assert bool(torch.isfinite(got).all()), f"saturation {what}: non-finite output"
    if name in ("out", "y"):
        assert float(got.abs().max()) >= F16_MAX, f"saturation {what}: the case never reached the fp16 limit"


def assert_launch_ok(geo, ref, form, bufs):
    fails = check_launch(geo, ref, form, bufs)
    assert not fails, fails


# ------------------------------------------------------------------------------------------------ CPU stand-ins
def _ragged_rows(geo, device):
    from autoformer_b200 import ops
    return ops.ragged_rows(geo.lengths, (1,), (128, 126, 124, 122), device)[0]


def run_emulation(geo, blk, inp, form, bufs):
    """tests/emulate.py's _emu_resblock_call / _emu_resblock2_call writing into views of the launch buffers."""
    B, L, C = geo.B, geo.L, geo.C
    outs = geo.outputs(form)
    kw = {}
    for (name, act, row0, R), buf in zip(outs, bufs):
        if name == "out":
            kw.update(out=buf[:B, :, :2 * C], out_row0=row0, reflect=R)
        elif name == "out_raw":
            kw.update(out_raw=buf[:B, :, :2 * C])
        elif name == "out2":
            kw.update(out2=buf[:B * L, :C])
        elif name == "y":
            kw.update(y=buf[:B, :, :2 * C], y_row0=row0, y_reflect=R, y_act=act)
        else:
            w_out, b_out = geo.mono(int(form[3:]))
            kw.update(wav=buf[:B * L].view(B, L), mono=(w_out, b_out))
    if geo.version == 1:
        xa, x = inp
        emulate._emu_resblock_call(blk, xa[:B, :, :2 * C], x[:B, :, :2 * C], B, L, **kw)
    else:
        if geo.ragged:
            kw["lengths"] = _ragged_rows(geo, "cpu")
        emulate._emu_resblock2_call(blk, inp[:B, :, :2 * C], B, L, **kw)


FAULTS = ("halo_mirror", "halo_missing", "tap2_late", "swizzle", "mid_lo", "cta_swap", "pair_utt", "slope",
          "spare_row", "spare_channel")


def run_stand_in(geo, blk, inp, form, bufs, fault=None):
    """A tile-level CPU model of the kernels (packed weights decoded by emulate.resblock_terms, the products the kernel
    forms, its two-term stores, the tiles that run, the halo stores), with one fault injected where asked."""
    B, L, C, d = geo.B, geo.L, geo.C, geo.d
    slope = 0.25 if fault == "slope" else 0.2
    w = blk.w.clone()
    if fault == "cta_swap":                       # the two CTA halves of every packed C = 128 weight tile exchanged
        w = w.view(-1, 2, 128, 64).flip(1).reshape(w.shape)
    terms = emulate.resblock_terms(w, C, geo.version)
    t = torch.arange(L)
    if geo.version == 1:
        xa, x = inp
        ah, al = xa[:, :, :C].double(), xa[:, :, C:2 * C].double()
        src = lambda idx, h, l: (ah + al)[:, idx] @ h.t() + ah[:, idx] @ l.t()
        xh, xl = x[:, :L, :C].double(), x[:, :L, C:2 * C].double()
        fmt = "bf16s"
    else:
        xa = xa_operand(inp[..., :C], inp[..., C:2 * C], slope).double()
        src = lambda idx, h, l: xa[:, idx] @ (h + l).t()
        xh, xl = inp[:, d:d + L, :C].double(), inp[:, d:d + L, C:2 * C].double()
        fmt = "f16t"
    z = blk.bias3.double().clone()
    for tap in range(3):
        idx = t + tap * d
        if fault == "tap2_late" and tap == 2:     # the last row of each tile reads one row late
            idx = torch.clamp(idx + (t % 128 == 127).long(), max=L + 2 * d - 1)
        z = z + src(idx, *terms[tap])
    mid = lrelu64(z, slope).float()
    mh, ml = (v.double() for v in split_two(mid, fmt))
    if fault == "mid_lo":
        ml[..., :C // 2] = 0
    (w1h, w1l), (wsh, wsl) = terms[3], terms[4]
    y = (mh + ml) @ w1h.t() + mh @ w1l.t() + (xh + xl) @ wsh.t() + xh @ wsl.t() + blk.bias1.double()
    owner = [b for b, n in enumerate(geo.lengths) for _ in range(-(-n // 128))] if geo.ragged else None
    for (name, act, row0, R), buf in zip(geo.outputs(form), bufs):
        a = lrelu64(y, slope) if act else y.clone()
        if fault == "swizzle":                    # one 8-channel chunk exchanged with its neighbour on rows = 7 (mod 8)
            rows7 = t % 8 == 7
            a[:, rows7, 0:16] = torch.cat([a[:, rows7, 8:16], a[:, rows7, 0:8]], dim=-1)
        if fault == "pair_utt" and owner is not None:  # the second tile of a pair computed for its partner's utterance
            for u in range(len(owner) // 2):
                b0, b1 = owner[2 * u], owner[2 * u + 1]
                if b0 != b1:
                    j = 2 * u + 1 - owner.index(b1)
                    a[b1, 128 * j:128 * j + 128] = a[b0, 128 * j:128 * j + 128]
        if name == "out2":
            for b in range(B):
                buf[b * L:b * L + geo.ran_rows(b), :C] = a[b, :geo.ran_rows(b)].float()
        elif name == "wav":
            K = int(form[3:])
            w_out, b_out = geo.mono(K)
            S = form_stride(form)
            for b, n in enumerate(geo.lengths):
                v, _, _ = wav_reference(a[b].float().double(), torch.zeros(n, C), a[b], w_out, b_out, n)
                buf[b * L:b * L + n] = v.float()
                buf[b * L + n:b * L + geo.ran_rows(b, S)] = 0
        else:
            hi, lo = split_two(a.float(), fmt)
            two = torch.cat([hi, lo], dim=-1)
            for b in range(B):
                ran = geo.ran_rows(b)
                buf[b, row0:row0 + ran, :2 * C] = two[b, :ran]
                if fault == "halo_missing":
                    continue
                for k in range(1, R + 1):
                    buf[b, row0 - k, :2 * C] = two[b, k - 1 if (fault == "halo_mirror" and k == R) else k]
                    if ran >= L:
                        buf[b, row0 + L - 1 + k, :2 * C] = two[b, L - 1 - k]
        if fault == "spare_row":
            buf[0, row0 + L + R, :2 * C] = 0
        if fault == "spare_channel":
            buf[0, row0, 2 * C] = 0


def _cpu_block(geo, raw):
    from autoformer_b200 import ops, packing
    if geo.version == 1:
        return ops.Resblock(*packing.pack_resblock(*raw), dilation=geo.d)
    return ops.Resblock2(*packing.pack_resblock2(*raw), dilation=geo.d)


def _cpu_case(inst, B, L, lengths, d, R, row0, mag="normal", seed=1):
    geo = Geo(dict(inst=inst, d=d, R=R, row0=row0, mag=mag), B, L, lengths if INSTS[inst][2] else [L] * B)
    scale = 2.0 ** -17 if mag == "tiny" else 1.0
    raw = make_weights(geo.C, seed, scale)
    inp = geo.make_inputs(seed + 1)
    return geo, raw, inp, Ref(geo.version, raw, inp, d, L)


CPU_SHAPES = {   # instantiation -> (B, L, lengths, d, R, row0)
    "v1_c32": (2, 256, None, 3, 9, 11), "v1_c64": (1, 256, None, 16, 16, 16),
    "v2_c32": (2, 256, None, 3, 9, 9), "v2_c64": (1, 256, None, 16, 1, 3),
    "v2_c32_ragged": (3, 384, [384, 200, 37], 9, 16, 16), "v2_c64_ragged": (2, 256, [130, 256], 1, 9, 9),
    "big": (1, 384, None, 12, 9, 9), "big_ragged": (3, 128, [100, 128, 37], 3, 1, 2),
}


@pytest.mark.parametrize("inst", list(INSTS))
def test_checker_accepts_the_emulation(inst):
    """CPU: the checker passes tests/emulate.py's stand-ins (which round the intermediate to nearest, not by
    truncation) and the fault model with no fault, on every form."""
    B, L, lengths, d, R, row0 = CPU_SHAPES[inst]
    geo, raw, inp, ref = _cpu_case(inst, B, L, lengths, d, R, row0)
    blk = _cpu_block(geo, raw)
    for form in inst_forms(inst):
        for runner in (run_emulation, run_stand_in):
            bufs = [geo.alloc(n, r0, r) for n, _, r0, r in geo.outputs(form)]
            runner(geo, blk, inp, form, bufs)
            assert_launch_ok(geo, ref, form, bufs)


@pytest.mark.parametrize("mag", ["tiny", "huge"])
def test_checker_accepts_the_magnitude_extremes(mag):
    geo, raw, inp, ref = _cpu_case("v2_c32", 2, 256, None, 3, 9, 9, mag=mag, seed=5)
    blk = _cpu_block(geo, raw)
    for form in ("y", "y_act", "out2", "wav7"):
        bufs = [geo.alloc(n, r0, r) for n, _, r0, r in geo.outputs(form)]
        run_stand_in(geo, blk, inp, form, bufs)
        assert_launch_ok(geo, ref, form, bufs)


# fault -> (instantiation, form, the check that must reject it)
FAULT_CASES = [
    ("halo_mirror", "v2_c32", "y", "bound"), ("halo_mirror", "v1_c64", "out_reflect", "bound"),
    ("halo_missing", "v2_c64", "y", "sentinel"), ("halo_missing", "big", "y", "sentinel"),
    ("tap2_late", "v2_c32", "y_act", "bound"), ("tap2_late", "v1_c32", "out2", "bound"),
    ("tap2_late", "big", "y", "bound"),
    ("swizzle", "v2_c64", "out2", "bound"), ("swizzle", "v1_c64", "out+out_raw", "bound"),
    ("mid_lo", "v2_c32", "out2", "rel-l2"), ("mid_lo", "v1_c32", "out_raw", "rel-l2"), ("mid_lo", "big", "y", "rel-l2"),
    ("cta_swap", "big", "y", "bound"), ("cta_swap", "big_ragged", "y_act", "bound"),
    ("pair_utt", "big_ragged", "y", "bound"),
    ("slope", "big", "y_act", "bound"), ("slope", "v2_c32", "wav5", "bound"), ("slope", "v1_c32", "out", "bound"),
    ("spare_row", "v2_c32_ragged", "y", "sentinel"), ("spare_row", "v1_c32", "out", "sentinel"),
    ("spare_channel", "v2_c64_ragged", "y_act", "sentinel"), ("spare_channel", "big", "y", "sentinel"),
]


@pytest.mark.parametrize("fault,inst,form,check", FAULT_CASES)
def test_checker_rejects_injected_fault(fault, inst, form, check):
    """CPU: each injected fault fails the check the module docstring names for it."""
    B, L, lengths, d, R, row0 = CPU_SHAPES[inst]
    geo, raw, inp, ref = _cpu_case(inst, B, L, lengths, d, R, row0)
    blk = _cpu_block(geo, raw)
    bufs = [geo.alloc(n, r0, r) for n, _, r0, r in geo.outputs(form)]
    run_stand_in(geo, blk, inp, form, bufs, fault=fault)
    fails = check_launch(geo, ref, form, bufs)
    assert check in {k for k, _ in fails}, (fault, fails)


def test_fault_list_is_complete():
    assert {f for f, *_ in FAULT_CASES} == set(FAULTS)


def test_split_f16_trunc_matches_the_kernel_formula():
    """CPU: hi keeps 10 mantissa bits (exact in fp16 over its normal range), lo = v - hi; hi + lo = v to 2^-21 relative
    plus the subnormal floors; out-of-range values saturate."""
    g = torch.Generator().manual_seed(3)
    v = torch.cat([torch.randn(4096, generator=g) * s for s in (1.0, 1e3, 2.0 ** -16, 2.0 ** -20)]
                  + [torch.tensor([7e4, -7e4, 65504.0, 0.0])])
    hi, lo = split_f16_trunc(v)
    assert bool(torch.isfinite(hi).all() & torch.isfinite(lo).all())
    body = v.abs() <= F16_MAX
    err = (hi.double() + lo.double() - v.double()).abs()
    assert bool((err[body] <= store_err(v.double().abs(), "f16t")[body]).all())
    normal = (v.abs() >= 2.0 ** -14) & body
    assert bool((hi.float()[normal] == (v[normal].view(torch.int32) & -8192).view(torch.float32)).all())
    assert float(hi[-4]) == F16_MAX and float(hi[-3]) == -F16_MAX


# ------------------------------------------------------------------------------------------------ the GPU matrix
def _gpu_launch(geo, blk, xin, form, bufs, B=None, lengths=None):
    """One launch of `form` into `bufs` (device).  Through ops.Resblock / ops.Resblock2 where the wrapper can express the
    geometry, through the C ABI where an output's row stride exceeds the minimum (out_raw, out2)."""
    from autoformer_b200 import _lib, ops
    B = B or geo.B
    L, C = geo.L, geo.C
    outs = geo.outputs(form)
    names = [o[0] for o in outs]
    lib = _lib.load()
    if geo.version == 1:
        xa, x = xin
        if names in (["out"],):
            _, _, row0, R = outs[0]
            blk(xa[:B, :, :2 * C], x[:B, :, :2 * C], B, L, out=bufs[0][:B, :, :2 * C], out_row0=row0, reflect=R)
            return
        desc = _lib.ResblockDesc()
        desc.xa, desc.xa_ld, desc.x, desc.x_ld = xa.data_ptr(), xa.stride(1), x.data_ptr(), x.stride(1)
        desc.w, desc.bias3, desc.bias1 = blk.w.data_ptr(), blk.bias3.data_ptr(), blk.bias1.data_ptr()
        desc.B, desc.L, desc.C, desc.dilation = B, L, C, geo.d
        for (name, _, row0, R), buf in zip(outs, bufs):
            if name == "out":
                desc.out, desc.out_ld, desc.out_rows_per_utt = buf.data_ptr(), buf.stride(1), buf.shape[1]
                desc.out_row0, desc.out_reflect = row0, R
            elif name == "out_raw":
                desc.out_raw, desc.out_raw_ld = buf.data_ptr(), buf.stride(1)
            else:
                desc.out2, desc.out2_ld = buf.data_ptr(), buf.stride(0)
        _lib.check(lib.avc_resblock(ctypes.byref(desc), ops._stream()), "avc_resblock")
        return
    rows = None
    if geo.ragged:
        rows = ops.ragged_rows(lengths or geo.lengths, (1,), (128, 126, 124, 122), "cuda")[0]
    name, act, row0, R = outs[0]
    if name == "y":
        blk(xin[:B, :, :2 * C], B, L, y=bufs[0][:B, :, :2 * C], y_row0=row0, y_reflect=R, y_act=act, lengths=rows)
    elif name == "wav":
        w_out, b_out = geo.mono(int(form[3:]))
        blk(xin[:B, :, :2 * C], B, L, wav=bufs[0][:B * L].view(B, L), mono=(w_out.cuda(), b_out), lengths=rows)
    else:
        desc = _lib.Resblock2Desc()
        desc.x, desc.x_ld = xin.data_ptr(), xin.stride(1)
        desc.w, desc.bias3, desc.bias1 = blk.w.data_ptr(), blk.bias3.data_ptr(), blk.bias1.data_ptr()
        desc.B, desc.L, desc.C, desc.dilation = B, L, C, geo.d
        desc.out2, desc.out2_ld = bufs[0].data_ptr(), bufs[0].stride(0)
        if rows is not None:
            tile_start, n_tiles = rows.tiles[128]
            desc.lengths, desc.tile_start, desc.n_tiles = rows.rows.data_ptr(), tile_start.data_ptr(), n_tiles
        _lib.check(lib.avc_resblock2(ctypes.byref(desc), ops._stream()), "avc_resblock2")


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32).cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_resblock_contract(case):
    """One case of the matrix: every output form of its instantiation into NaN buffers, each launch held to the
    sentinel, the per-element bound and the rel-L2; for every form a repeated launch gives the same bits, and the
    batch's last utterance run alone (B = 1) gives the same bits as its rows in the batch (zero tails included)."""
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    B, L, lengths = case_shape(case, n_sms)
    geo = Geo(case, B, L, lengths, device="cuda")
    for form in inst_forms(case["inst"]):
        if case["geo"] != "legacy":
            assert case["geo"] in geometry_classes(case["inst"], form, B, L, lengths, n_sms) or \
                class_exempt(case["inst"], form, case["geo"]), form
    raw = make_weights(geo.C, case["seed"], 2.0 ** -17 if case["mag"] == "tiny" else 1.0)
    inp = geo.make_inputs(case["seed"] + 1)
    ref = Ref(geo.version, raw, inp, geo.d, L)
    blk = _cpu_block(geo, raw).to("cuda")
    xin = tuple(t.cuda() for t in inp) if geo.version == 1 else inp.cuda()
    u = B - 1
    one = Geo(case, 1, L, [lengths[u]], device="cuda")
    x1 = tuple(t[u:u + 1].contiguous() for t in xin) if geo.version == 1 else xin[u:u + 1].contiguous()
    for form in inst_forms(case["inst"]):
        bufs = [geo.alloc(n, r0, r) for n, _, r0, r in geo.outputs(form)]
        _gpu_launch(geo, blk, xin, form, bufs)
        torch.cuda.synchronize()
        assert_launch_ok(geo, ref, form, bufs)
        again = [geo.alloc(n, r0, r) for n, _, r0, r in geo.outputs(form)]
        _gpu_launch(geo, blk, xin, form, again)
        # the last utterance alone: the same tiles over the same rows, so the same arithmetic
        alone = [one.alloc(n, r0, r) for n, _, r0, r in one.outputs(form)]
        _gpu_launch(one, blk, x1, form, alone, B=1, lengths=[lengths[u]])
        torch.cuda.synchronize()
        for (name, *_), full, rep, a in zip(geo.outputs(form), bufs, again, alone):
            assert torch.equal(_bits(full), _bits(rep)), (form, name, "a repeated launch changed bits")
            got, want = (a[0], full[u]) if name in ("out", "y", "out_raw") else (a[:L], full[u * L:(u + 1) * L])
            assert torch.equal(_bits(got), _bits(want)), (form, name, "utterance alone differs from its rows in the batch")


# ------------------------------------------------------------------------------------------------ host refusals
def _refusals():
    """(name, C ABI, C, descriptor edits): each must be refused before anything is launched."""
    return [
        ("dilation 17", 2, 32, dict(dilation=17)), ("dilation 17 v1", 1, 64, dict(dilation=17)),
        ("dilation 13 at C = 128", 2, 128, dict(dilation=13)),
        ("out with out2", 1, 32, dict(out2=True)), ("y with out2", 2, 64, dict(out2=True)),
        ("C = 128 with out2", 2, 128, dict(y=False, out2=True)),
        ("wav with C = 64", 2, 64, dict(y=False, wav=7)), ("wav with 9 taps", 2, 32, dict(y=False, wav=9)),
        ("L % 128", 2, 32, dict(L=200)), ("L % 128 v1", 1, 32, dict(L=200)),
        ("row0 < reflect", 2, 64, dict(row0=3, reflect=4)), ("row0 < reflect v1", 1, 64, dict(row0=3, reflect=4)),
        ("reflect 17", 2, 32, dict(row0=17, reflect=17)), ("reflect 17 at C = 128", 2, 128, dict(row0=17, reflect=17)),
        ("too few rows_per_utt", 2, 32, dict(rows=-1)), ("too few rows_per_utt v1", 1, 32, dict(rows=-1)),
        ("n_tiles below B", 2, 32, dict(lengths=True, n_tiles=1)),
        ("n_tiles past the tile space", 2, 64, dict(lengths=True, n_tiles=7)),
        ("n_tiles past the tile space at C = 128", 2, 128, dict(lengths=True, n_tiles=7)),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("name,version,C,edit", _refusals(), ids=[r[0] for r in _refusals()])
def test_host_refuses_bad_geometry(name, version, C, edit):
    """avc_resblock / avc_resblock2 refuse what the kernels cannot run; the sentinel buffers stay untouched."""
    from autoformer_b200 import _lib, ops, packing
    lib = _lib.load()
    B, L, d = 2, edit.get("L", 256), min(edit.get("dilation", 3), 17)
    Lb = 384
    raw = make_weights(C, 1)
    blk = (ops.Resblock(*packing.pack_resblock(*raw), dilation=3) if version == 1 else
           ops.Resblock2(*packing.pack_resblock2(*raw), dilation=3)).to("cuda")
    dt = torch.bfloat16 if version == 1 else torch.float16
    x = torch.zeros(B, Lb + 2 * 17, 2 * C, dtype=dt, device="cuda")
    row0, reflect = edit.get("row0", 9), edit.get("reflect", 9)
    rows = row0 + L + reflect + edit.get("rows", 0)
    y = nan_buf((B, rows + 8, 2 * C), dt)
    out2 = nan_buf((B * Lb, C), torch.float32)
    wav = nan_buf((B, Lb), torch.float32)
    if version == 1:
        desc = _lib.ResblockDesc()
        desc.xa, desc.xa_ld, desc.x, desc.x_ld = x.data_ptr(), 2 * C, x.data_ptr(), 2 * C
        desc.w, desc.bias3, desc.bias1 = blk.w.data_ptr(), blk.bias3.data_ptr(), blk.bias1.data_ptr()
        desc.B, desc.L, desc.C, desc.dilation = B, L, C, d
        desc.out, desc.out_ld, desc.out_rows_per_utt, desc.out_row0, desc.out_reflect = y.data_ptr(), 2 * C, rows, row0, reflect
        if edit.get("out2"):
            desc.out2, desc.out2_ld = out2.data_ptr(), C
        call = lambda: _lib.check(lib.avc_resblock(ctypes.byref(desc), ops._stream()), "avc_resblock")
    else:
        desc = _lib.Resblock2Desc()
        desc.x, desc.x_ld = x.data_ptr(), 2 * C
        desc.w, desc.bias3, desc.bias1 = blk.w.data_ptr(), blk.bias3.data_ptr(), blk.bias1.data_ptr()
        desc.B, desc.L, desc.C, desc.dilation = B, L, C, d
        if edit.get("y", True):
            desc.y, desc.y_ld, desc.y_rows_per_utt, desc.y_row0, desc.y_reflect = y.data_ptr(), 2 * C, rows, row0, reflect
        if edit.get("out2"):
            desc.out2, desc.out2_ld = out2.data_ptr(), C
        if edit.get("wav"):
            K = edit["wav"]
            w_out = torch.zeros(K, C, device="cuda")
            desc.wav, desc.mono_w, desc.mono_bias, desc.mono_taps = wav.data_ptr(), w_out.data_ptr(), 0.0, K
        if edit.get("lengths"):
            rr = ops.ragged_rows([L, L], (1,), (128,), "cuda")[0]
            desc.lengths, desc.tile_start, desc.n_tiles = rr.rows.data_ptr(), rr.tiles[128][0].data_ptr(), edit["n_tiles"]
        call = lambda: _lib.check(lib.avc_resblock2(ctypes.byref(desc), ops._stream()), "avc_resblock2")
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError):
        call()
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0, name
    for buf in (y, out2, wav):
        assert bool(torch.isnan(buf.float()).all()), (name, "a refused call wrote")
