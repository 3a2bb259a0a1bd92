"""Op-level contract of the LSTM recurrence kernels, frame by frame and element by element.

Every kernel reads h_{t-1} back from a buffer the test can see (avc_lstm_seq and avc_lstm_seq_ws: the operand-format
hseq; avc_lstm_stack_ws: hs[l][t] and hs[l-1][t+1]; avc_bilstm_small: the exact fp32 h, visible when `out` is fp32 and
unrounded).  So the reference does not free-run: for every frame it recomputes the pre-activations in fp64 from the
kernel's own stored h_{t-1}, with exactly the products the kernel forms, from the RAW PyTorch-layout weights split with
packing.split_terms / sat_f16 (never from the packed tensors, so a gate-permutation packing error fails too):
    split bf16 ("fp32")  a_hi w_hi + a_lo w_hi + a_hi w_lo      (the kernel drops lo * lo)
    "fp16x2"             a w_hi + a w_lo
    "bf16", "tf32"       a w on the stored operands
    stack kernel         one fp16 term of W_hh and of W_ih
    BiLSTM               fp32 weights
The cell state is not exported: c is chained in fp64 from the teacher-forced gates.  Each launch is held to
  * a per-element worst-case bound on every stored fp32 h (and on every fp16 h of the stack kernel's hs, plus half an
    fp16 ulp): |dz| <= (K_phys + c) 2^-23 S with S = sum |products| + |x part| and c the extra fp32 adds, carried
    through the derivatives of the gates, plus the error of lstm_cell's __expf / __fdividef evaluation (derived from
    __expf's 2 + floor(1.173 |x|) ulp), accumulated through the c chain per (b, u).  Worst case, so never flaky; any
    indexing, masking, race or phase error is of order |h| and fails it;
  * a teacher-forced rel-L2 gate per kernel and precision (measured values in TF_GATE), which catches a dropped
    precision term the worst-case bound is too loose to see;
  * bit-exact stores (operand hseq = packing.to_act(hseq_f32), h_last = the last frame, stack frame 0 = 0, BiLSTM
    output formats and codes against the unrounded fp32 run);
  * NaN sentinels around every output (spare utterances, a spare layer, NaN channels past the input's logical ones);
  * bit identity of per-step and persistent launches and of a repeated launch.
The CPU tests check the declared cases against mirrors of the host dispatch, and check the checker itself on the
tests/emulate.py stand-ins, with and without injected faults.

Not covered, on purpose: AVC_LSTM_NO_COOP (a profiling aid that launches the same persistent kernels without the
cooperative attribute).  It is read once per process.
"""
import itertools
import zlib

import pytest
import torch

from oracle import rel_l2
from tests import emulate
from tests.test_gpu_kernel_contract import U, check_bound, check_sentinel, half_ulp, nan_buf

PRECS = ("tf32", "bf16", "fp32", "fp16x2")
MODE = {"tf32": 0, "bf16": 1, "fp32": 2, "fp16x2": 3}
NPROD = {"tf32": 1, "bf16": 1, "fp32": 3, "fp16x2": 2}     # products per logical multiply-add
# Teacher-forced rel-L2 of the stored h of a launch against the reference above, per kernel and precision: the largest
# value over the cases of this file, measured on an NVIDIA B200 at a 1000 W power limit.  The gates are 4x those.  Every
# entry is of fp32 h except "lstm_stack/hs", which is the stack kernel's fp16 record (fp16 rounding dominates it).
TF_MEASURED = {"lstm_seq/tf32": 5.2e-7, "lstm_seq/bf16": 2.8e-7, "lstm_seq/fp32": 2.1e-6, "lstm_seq/fp16x2": 1.9e-6,
               "lstm_ws/fp32": 9.0e-7, "lstm_ws/fp16x2": 3.5e-7, "lstm_stack/hs": 2.2e-4, "lstm_stack/h_last": 7.3e-7,
               "bilstm_small/fp32": 1.9e-7}
TF_GATE = {k: 4 * v for k, v in TF_MEASURED.items()}


def _nan(shape, dtype, dev):
    return nan_buf(shape, dtype) if dev == "cuda" else torch.full(shape, float("nan"), dtype=dtype)


# ------------------------------------------------------------------------------------------------ dispatch mirrors
def seq_cell(B, H, prec, group, fused):
    """Mirror of avc_lstm_seq's host dispatch (avc_lstm.cu:663-769): (kernel, MODE, BN, geometry, a_rows < 128)."""
    from autoformer_b200 import packing
    assert group in (16, 32)
    kc = packing.KC[prec]
    assert H % kc == 0 and H % 4 == 0 and H % group == 0
    m_tiles = -(-B // 128)
    a_rows = -(-B // 8) * 8 if m_tiles == 1 else 128
    geo = "single" if m_tiles == 1 else ("phantom" if m_tiles % 2 else "pair")
    return ("fused" if fused else "step", MODE[prec], 4 * group, geo, a_rows < 128)


def ws_cell(B, H, n_sm=148):
    """Mirror of avc_lstm_seq_ws's choice of accumulator rows AR and K-slices S (avc_lstm_ws.cu:410, :437-449)."""
    ar = 16 if B <= 16 else (32 if B <= 32 else 64)
    S = 8 if H % 512 == 0 and 4 * H // 128 * 8 <= n_sm else 4
    return ar, S


def bilstm_kernel(B, H):
    """Mirror of avc_bilstm_small's kernel choice (avc_misc.cu:465-479)."""
    if H == 32:
        return "bilstm32" if B <= 128 else "<1,true>"
    return "<1,false>" if H <= 32 else "<2,false>"


def sub_batches(B, H):
    """Mirror of LstmLayer.__call__'s split of a persistent batch above ops.persistent_batch_cap."""
    from autoformer_b200 import ops
    cap = ops.persistent_batch_cap(H)
    if not B > cap > 0:
        return [(0, B)]
    return [(b0, min(B, b0 + cap)) for b0 in range(0, B, cap)]


# ------------------------------------------------------------------------------------------------ declared cases
SEQ_B = {"single": 37, "pair": 200, "phantom": 300}      # 37: a_rows = 40 < 128


def _declare_seq():
    cases = []
    for i, (kern, prec, group, geo) in enumerate(itertools.product(("step", "fused"), PRECS, (16, 32),
                                                                   ("single", "pair", "phantom"))):
        cases.append(dict(kern=kern, prec=prec, group=group, B=SEQ_B[geo], H=128, T=(5, 1, 2, 7)[i % 4],
                          c_in=(72, 40, 104)[i % 3]))
    return cases


SEQ_CASES = _declare_seq()


def _seq_id(c):
    return f"{c['kern']}-{c['prec']}-G{c['group']}-B{c['B']}H{c['H']}T{c['T']}"


def _declare_ws():
    cases = []
    Bs = {16: (1, 16), 32: (17, 32), 64: (33, 64)}
    for i, (prec, H, ar) in enumerate(itertools.product(("fp32", "fp16x2"), (512, 768, 1024), (16, 32, 64))):
        if H == 768 and ar == 32:
            continue                    # S = 4 is met at H = 768 and 1024; keep the matrix short
        cases.append(dict(prec=prec, H=H, B=Bs[ar][i % 2], T=(1, 9, 4)[i % 3]))
    return cases


WS_CASES = _declare_ws()


def _declare_stack():
    from autoformer_b200 import ops
    cases = []
    Bs = {16: (1, 13), 32: (17, 32), 64: (33, 64)}
    for i, (L, ar) in enumerate(itertools.product((2, 3, 4), (16, 32, 64))):
        Hs = [H for H in (128, 384, 640, 768) if ops.stack_supported(Bs[ar][0], H, L, "fp16x2")]
        cases.append(dict(L=L, H=Hs[i % len(Hs)], B=Bs[ar][i % 2], T=(1, 2, 3, 300)[i % 4]))
    return cases


STACK_CASES = _declare_stack()
BILSTM_CASES = [dict(H=32, B=6, T=64, freq=32), dict(H=32, B=130, T=22, freq=22), dict(H=16, B=5, T=32, freq=1),
                dict(H=24, B=7, T=44, freq=22), dict(H=44, B=9, T=32, freq=32), dict(H=64, B=3, T=24, freq=24)]


def test_lstm_case_matrix_covers_every_cell():
    """CPU: the declared cases reach every cell of the host dispatch of the four recurrence entry points."""
    from autoformer_b200 import ops, packing
    cells = {seq_cell(c["B"], c["H"], c["prec"], c["group"], c["kern"] == "fused") for c in SEQ_CASES}
    need = {(k, MODE[p], bn, g) for k in ("step", "fused") for p in PRECS for bn in (64, 128)
            for g in ("single", "pair", "phantom")}
    assert need <= {c[:4] for c in cells}, sorted(need - {c[:4] for c in cells})
    assert all(c[4] == (c[3] == "single") for c in cells)                  # one m-tile loads only its rows
    assert {1, 2} <= {c["T"] for c in SEQ_CASES}
    for p in PRECS:                   # an input width that is not a whole number of k-blocks, in every precision
        assert any(c["c_in"] % packing.KC[p] for c in SEQ_CASES if c["prec"] == p and c["kern"] == "fused")
    # every seq case runs per-step and persistent; persistent grids fit one wave
    for c in SEQ_CASES:
        m = -(-c["B"] // 128)
        assert (m + m % 2 if m >= 2 else 1) * -(-c["H"] // c["group"]) <= 148, _seq_id(c)
    # sub-batches of a persistent batch above the cap: 512 + 88 at H = 1024, the second a single m-tile
    assert sub_batches(600, 1024) == [(0, 512), (512, 600)]
    assert seq_cell(88, 1024, "fp16x2", 32, True)[3] == "single"
    # avc_lstm_seq_ws: AR x S x precision, ragged B, T = 1
    ws = {(ws_cell(c["B"], c["H"]), c["prec"]) for c in WS_CASES}
    assert {((ar, s), p) for ar in (16, 32, 64) for s in (8, 4) for p in ("fp32", "fp16x2")} <= ws, ws
    assert all(ops.ws_supported(c["B"], c["H"], c["prec"]) for c in WS_CASES)
    assert {1, 17, 33, 64} <= {c["B"] for c in WS_CASES} and 1 in {c["T"] for c in WS_CASES}
    # avc_lstm_stack_ws: L x AR, the widths with an odd chunk count per K half (384, 640), T in {1, 2, 3, 300}
    assert all(ops.stack_supported(c["B"], c["H"], c["L"], "fp16x2") for c in STACK_CASES)
    assert {(c["L"], ws_cell(c["B"], c["H"])[0]) for c in STACK_CASES} == set(itertools.product((2, 3, 4), (16, 32, 64)))
    assert {c["H"] for c in STACK_CASES} == {128, 384, 640, 768} and {c["T"] for c in STACK_CASES} == {1, 2, 3, 300}
    assert not ops.stack_supported(8, 640, 4, "fp16x2") and ops.stack_supported(8, 384, 4, "fp16x2")
    # avc_bilstm_small: every kernel, a partial last CTA of 4 utterances, freq in {1, 22, 32, T}
    assert {bilstm_kernel(c["B"], c["H"]) for c in BILSTM_CASES} == {"bilstm32", "<1,true>", "<1,false>", "<2,false>"}
    assert {c["H"] for c in BILSTM_CASES if bilstm_kernel(c["B"], c["H"]) == "<1,false>"} == {16, 24}
    assert {c["H"] for c in BILSTM_CASES if bilstm_kernel(c["B"], c["H"]) == "<2,false>"} == {44, 64}
    assert any(c["B"] % 4 for c in BILSTM_CASES if bilstm_kernel(c["B"], c["H"]) != "bilstm32")
    assert {1, 22, 32} <= {c["freq"] for c in BILSTM_CASES} and any(c["freq"] == c["T"] for c in BILSTM_CASES)
    # production shapes reach the kernels the tests below launch them on
    for B in (512, 300):
        for H in (512, 1024):
            assert ops.choose_gate_group(B, H, True) == {512: 16, 1024: 32}[H]
    assert seq_cell(512, 1024, "fp16x2", 32, True)[3] == "pair" and seq_cell(300, 1024, "fp16x2", 32, True)[3] == "phantom"
    assert ops.persistent_batch_cap(512) >= 512 and ops.persistent_batch_cap(1024) >= 512
    assert ops.stack_supported(32, 768, 3, "fp16x2") and ops.stack_supported(8, 768, 3, "fp16x2")


# ------------------------------------------------------------------------------------------------ the reference
def _eta(x):
    """Relative error bound of __expf(x): 2 + floor(1.173 |x|) ulp (CUDA C Programming Guide, intrinsic functions)."""
    return (2.0 + torch.floor(1.173 * x.abs())) * U


def _sig_err(z, s):
    """|sigmoid as lstm_cell evaluates it - sigmoid(z)| for the exact input z: the error of e = __expf(-z) moves
    1 / (1 + e) by s (1 - s) eta; __fdividef (2 ulp) and the ~10 roundings of the shared-reciprocal products
    (avc_pipe.cuh:lstm_cell) are 2^-20 relative; the clamp at +-25 costs sigmoid(-25) < 2e-11."""
    return s * (1 - s) * _eta(z.clamp(-25, 25)) + s * 2.0 ** -20 + 2e-11


def _tanh_err(z, t):
    """The same for tanh = (1 - e) / (1 + e), e = __expf(-2 |z|): de / e = eta moves it by (1 - t^2) eta."""
    return (1 - t * t) * _eta(2 * z) + t.abs() * 2.0 ** -20 + 1e-30


def _lin(z, e, d, dmax, dd):
    """Worst-case move of a function with derivative d(z) <= dmax and |d'| <= dd under an input error e."""
    return torch.clamp(d + dd * e, max=dmax) * e


def tf_chain(z, ez, reverse=False):
    """fp64 LSTM cell over teacher-forced pre-activations z [B][T][4H] (PyTorch gate order) with input error bounds ez;
    c chained from c_{-1} = 0.  Returns (h, bound on |kernel h - h|) [B][T][H]."""
    B, T, H4 = z.shape
    H = H4 // 4
    h = torch.empty(B, T, H, dtype=torch.float64, device=z.device)
    bound = torch.empty_like(h)
    c = torch.zeros(B, H, dtype=torch.float64, device=z.device)
    dc = torch.zeros_like(c)
    for s in range(T):
        t = T - 1 - s if reverse else s
        zi, zf, zg, zo = z[:, t].split(H, dim=1)
        ei, ef, eg, eo = ez[:, t].split(H, dim=1)
        i, f, g, o = torch.sigmoid(zi), torch.sigmoid(zf), torch.tanh(zg), torch.sigmoid(zo)
        di = _lin(zi, ei, i * (1 - i), 0.25, 0.1) + _sig_err(zi, i)
        df = _lin(zf, ef, f * (1 - f), 0.25, 0.1) + _sig_err(zf, f)
        do = _lin(zo, eo, o * (1 - o), 0.25, 0.1) + _sig_err(zo, o)
        dg = _lin(zg, eg, 1 - g * g, 1.0, 0.77) + _tanh_err(zg, g)
        cn = f * c + i * g
        # c~ - c = f~ (c~p - cp) + cp (f~ - f) + i~ (g~ - g) + g (i~ - i), plus the fp32 rounding of f c + i g
        dc = (f + df) * dc + c.abs() * df + (i + di) * dg + g.abs() * di + 4 * 2.0 ** -24 * ((f * c).abs() + (i * g).abs())
        c = cn
        tc = torch.tanh(c)
        hn = o * tc
        h[:, t] = hn
        bound[:, t] = tc.abs() * do + (o + do) * (_lin(c, dc, 1 - tc * tc, 1.0, 0.77) + _tanh_err(c, tc)) \
            + 2 * 2.0 ** -24 * hn.abs()
    return h, bound


def tf_reference(base, pairs, nadd, reverse=False):
    """h and its bound from z = base + sum_k A_k @ W_k^T, with A_k [B][T][K] the stored operands of each product (already
    placed at the frame that consumes them) and W_k [4H][K] the weight terms, both fp64, PyTorch gate order;
    base [B][T][4H] (xproj) or [4H] (bias).  |dz| <= nadd 2^-23 S, S = |base| + sum |A_k| @ |W_k|^T."""
    B, T = pairs[0][0].shape[:2]
    z = torch.empty(B, T, pairs[0][1].shape[0], dtype=torch.float64, device=pairs[0][0].device)
    S = torch.empty_like(z)
    step = max(1, (1 << 26) // (B * z.shape[2]))
    for t0 in range(0, T, step):
        t1 = min(T, t0 + step)
        b = base[:, t0:t1] if base.dim() == 3 else base
        zz = b.expand(B, t1 - t0, -1).clone()
        ss = b.abs().expand(B, t1 - t0, -1).clone()
        for A, W in pairs:
            zz += A[:, t0:t1] @ W.t()
            ss += A[:, t0:t1].abs() @ W.abs().t()
        z[:, t0:t1], S[:, t0:t1] = zz, ss
    return tf_chain(z, nadd * U * S, reverse)


def weight_terms(w, prec):
    """The weight terms the kernels multiply, from a raw PyTorch-layout matrix: [(term, operand slot)] where slot "hi"
    multiplies the hi (or only) activation term and "lo" the lo activation term of split precision."""
    from autoformer_b200 import packing
    if prec in packing.TWO_TERM_WEIGHTS:
        hi, lo = packing.split_terms(w.float(), prec)
        return hi.double(), lo.double()
    if prec == "f16":
        return packing.sat_f16(w).to(torch.float16).double(), None
    return packing.to_operand(w.float(), prec).double(), None


def op_pairs(a_op, w, prec, C):
    """(A, W) products of an operand-format activation sequence a_op [B][T][>= act_channels(C)] with raw weights
    w [4H][C]: split bf16 = a_hi (w_hi + w_lo) + a_lo w_hi; fp16x2 = a (w_hi + w_lo), both exact in fp64."""
    w_hi, w_lo = weight_terms(w, prec)
    if prec == "fp32":
        return [(a_op[..., :C].double(), w_hi + w_lo), (a_op[..., C:2 * C].double(), w_hi)]
    return [(a_op[..., :C].double(), w_hi + w_lo if w_lo is not None else w_hi)]


def shift(a, reverse=False):
    """a[:, t - 1] at frame t (a[:, t + 1] when reverse), zero at the first frame."""
    out = torch.zeros_like(a)
    if reverse:
        out[:, :-1] = a[:, 1:]
    else:
        out[:, 1:] = a[:, :-1]
    return out


def nprod_k(prec, H, kx=0):
    return NPROD.get(prec, 1) * (H + kx)


def check_h(got, ref, bound, what):
    """check_bound, screened on the device first: only a failing launch is copied to the host."""
    if got.is_cuda and bool(torch.isfinite(got).all()) and bool(((got.double() - ref).abs() <= bound).all()):
        return
    check_bound(got, ref, bound, what)


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32).cpu()


def _gate(key, got, ref):
    """The teacher-forced rel-L2 gate of the kernels.  The CPU stand-ins keep the lo * lo product and evaluate the cell
    exactly, so it does not apply to them."""
    if got.is_cuda:
        v = rel_l2(got, ref)
        assert v < TF_GATE[key], f"{key}: teacher-forced rel-L2 {v:.3e} >= gate {TF_GATE[key]:.3e}"


# ------------------------------------------------------------------------------------------------ inputs
def make_layer(H, c_in, seed, dev):
    g = torch.Generator().manual_seed(seed)
    w_ih = torch.randn(4 * H, c_in, generator=g) * 1.5 / c_in ** 0.5
    w_hh = torch.randn(4 * H, H, generator=g) * 2.0 / H ** 0.5
    b_ih, b_hh = torch.randn(4 * H, generator=g) * 0.5, torch.randn(4 * H, generator=g) * 0.5
    return tuple(t.to(dev) for t in (w_ih, w_hh, b_ih, b_hh))


def make_xproj(B, T, H4, seed, dev, scale=1.5):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, T, H4, generator=g) * scale).to(dev)


# ------------------------------------------------------------------------------------------------ avc_lstm_seq
class SeqRun:
    """One avc_lstm_seq (or avc_lstm_seq_ws, or LstmLayer) launch into sentinel buffers with its reference checks."""
    SPARE = 2

    def __init__(self, B, T, H, prec, dev):
        from autoformer_b200 import packing
        self.B, self.T, self.H, self.prec, self.dev = B, T, H, prec, dev
        self.ach = packing.act_channels(H, prec)
        self.hseq_big = _nan((B + 2 * self.SPARE, T, self.ach), packing.TORCH_DTYPE[prec], dev)
        self.f32_big = _nan((B + 2 * self.SPARE, T, H), torch.float32, dev)
        self.last_big = _nan((B + 2 * self.SPARE, H), torch.float32, dev)
        sl = slice(self.SPARE, self.SPARE + B)
        self.hseq, self.hseq_f32, self.h_last = self.hseq_big[sl], self.f32_big[sl], self.last_big[sl]

    def check(self, base, x_pairs, w_hh, nadd, what, key):
        from autoformer_b200 import packing
        B, T, H, prec = self.B, self.T, self.H, self.prec
        region = torch.zeros(self.hseq_big.shape[0], dtype=torch.bool)
        region[self.SPARE:self.SPARE + B] = True
        for big in (self.hseq_big, self.f32_big, self.last_big):
            check_sentinel(big, region.view(-1, *[1] * (big.dim() - 1)).expand(big.shape).cpu(), what)
        # bit-exact stores
        assert torch.equal(_bits(self.hseq), _bits(packing.to_act(self.hseq_f32, prec))), what + ": hseq != to_act(hseq_f32)"
        assert torch.equal(_bits(self.h_last), _bits(self.hseq_f32[:, -1])), what + ": h_last != hseq_f32[:, -1]"
        # teacher-forced reference from the stored operands
        pairs = list(x_pairs) + [(shift(A), W) for A, W in op_pairs(self.hseq, w_hh, prec, H)]
        h, bound = tf_reference(base, pairs, nadd)
        check_h(self.hseq_f32, h, bound, what + " hseq_f32")
        check_h(self.h_last, h[:, -1], bound[:, -1], what + " h_last")
        _gate(key, self.hseq_f32, h)
        return h, bound


def xin_buffer(x, prec, dev, spare_ch=8):
    """The input sequence in the operand format, with NaN channels past act_channels(c_in) (xin_ld > logical)."""
    from autoformer_b200 import packing
    a = packing.to_act(x.float().cpu(), prec)
    buf = torch.full((*a.shape[:2], a.shape[2] + spare_ch), float("nan"), dtype=a.dtype)
    buf[..., :a.shape[2]] = a
    return buf.to(dev)


def fused_base_and_pairs(xin, w_ih, b_ih, b_hh, prec, c_in):
    bias = (b_ih.float() + b_hh.float()).double()            # packing.pack_lstm_ih_fused sums the biases in fp32
    return bias, op_pairs(xin, w_ih, prec, c_in)


def seq_nadd(prec, H, kx, extra=3):
    """K_phys + the extra fp32 adds: the two accumulator blocks of split precision and acc + xproj / bias."""
    return nprod_k(prec, H, kx) + extra


def run_seq_case(c, dev, lstm_seq=None, seed=None):
    """Launch one declared avc_lstm_seq case per-step and persistent (plus a repeat) and check every launch.  Returns
    the persistent SeqRun."""
    from autoformer_b200 import _lib, ops, packing
    lstm_seq = lstm_seq or ops.lstm_seq
    seed = zlib.crc32(_seq_id(c).encode()) % 10007 if seed is None else seed
    B, T, H, prec, G, c_in = c["B"], c["T"], c["H"], c["prec"], c["group"], c["c_in"]
    fused = c["kern"] == "fused"
    w_ih, w_hh, b_ih, b_hh = make_layer(H, c_in, seed, "cpu")
    kc = packing.KC[prec]
    if fused:
        x = make_xproj(B, T, c_in, seed + 1, "cpu", 1.0)
        xin = xin_buffer(x, prec, dev)
    else:
        xproj = make_xproj(B, T, 4 * H, seed + 1, "cpu")
    runs = {}
    perm = packing.gate_permutation(H, G)
    hh = packing.pack_lstm_hh(w_hh, prec, G).to(dev)
    for persistent in (False, True, True):
        r = SeqRun(B, T, H, prec, dev)
        kw = dict(hseq=r.hseq, hseq_f32=r.hseq_f32, h_last=r.h_last, persistent=persistent)
        n0 = _lib.launch_count() if dev == "cuda" else 0
        if fused:
            wih, bias = packing.pack_lstm_ih_fused(w_ih, b_ih, b_hh, prec, G)
            lstm_seq(None, hh, B, T, H, prec, G, xin=xin, w_ih=wih.to(dev), bias=bias.to(dev), c_in=c_in, **kw)
        else:
            lstm_seq(xproj[..., perm].contiguous().view(B * T, 4 * H).to(dev), hh, B, T, H, prec, G, **kw)
        if dev == "cuda":
            torch.cuda.synchronize()
            assert _lib.launch_count() - n0 == (1 if persistent else T), "persistent grid fell back to per-step"
        runs.setdefault(persistent, []).append(r)
    what = _seq_id(c)
    if fused:
        base, x_pairs = fused_base_and_pairs(xin, w_ih.to(dev), b_ih.to(dev), b_hh.to(dev), prec, c_in)
        nadd = seq_nadd(prec, H, -(-c_in // kc) * kc)
    else:
        base, x_pairs, nadd = xproj.double().to(dev), [], seq_nadd(prec, H, 0)
    key = f"lstm_seq/{prec}"
    main = runs[True][0]
    main.check(base, x_pairs, w_hh.to(dev), nadd, what + " persistent", key)
    runs[False][0].check(base, x_pairs, w_hh.to(dev), nadd, what + " per-step", key)
    ref_bits = _bits(main.hseq_f32)
    for persistent, rs in runs.items():
        for r in rs:
            assert torch.equal(_bits(r.hseq_f32), ref_bits), f"{what}: persistent={persistent} differs in bits"
            assert torch.equal(_bits(r.hseq), _bits(main.hseq))
    return main


@pytest.mark.gpu
@pytest.mark.parametrize("case", SEQ_CASES, ids=_seq_id)
def test_lstm_seq_contract(case):
    run_seq_case(case, "cuda")


# ------------------------------------------------------------------------------------------------ avc_lstm_seq_ws
def _ws_id(c):
    return f"{c['prec']}-B{c['B']}H{c['H']}T{c['T']}"


def run_ws_case(c, dev, lstm_seq_ws=None):
    from autoformer_b200 import ops, packing
    lstm_seq_ws = lstm_seq_ws or ops.lstm_seq_ws
    seed = zlib.crc32(_ws_id(c).encode()) % 10007
    B, T, H, prec = c["B"], c["T"], c["H"], c["prec"]
    _, w_hh, _, _ = make_layer(H, 8, seed, "cpu")
    xproj = make_xproj(B, T, 4 * H, seed + 1, "cpu")
    perm = packing.gate_permutation(H, packing.WS_GROUP)
    hh = packing.pack_lstm_hh(w_hh, prec, packing.WS_GROUP).to(dev)
    xp = xproj[..., perm].contiguous().view(B * T, 4 * H).to(dev)
    runs = []
    for _ in range(2):
        r = SeqRun(B, T, H, prec, dev)
        out = lstm_seq_ws(xp, hh, B, T, H, hseq=r.hseq, hseq_f32=r.hseq_f32, h_last=r.h_last, precision=prec)
        assert out is not None, "avc_lstm_seq_ws: the grid is not co-resident"
        runs.append(r)
    if dev == "cuda":
        torch.cuda.synchronize()
    S = ws_cell(B, H)[1]
    runs[0].check(xproj.double().to(dev), [], w_hh.to(dev), nprod_k(prec, H) + S + 2, "ws " + _ws_id(c), f"lstm_ws/{prec}")
    assert torch.equal(_bits(runs[1].hseq_f32), _bits(runs[0].hseq_f32)), "second launch differs"
    return runs[0]


@pytest.mark.gpu
@pytest.mark.parametrize("case", WS_CASES, ids=_ws_id)
def test_lstm_ws_contract(case):
    run_ws_case(case, "cuda")


# ------------------------------------------------------------------------------------------------ avc_lstm_stack_ws
def _stack_id(c):
    return f"L{c['L']}-B{c['B']}H{c['H']}T{c['T']}"


def check_stack(hs_big, h_last_big, L, B, T, H, xproj0, raws, what, spare=1):
    """hs_big [L + spare][T + 1][B][H] fp16 (hs = its first L layers), h_last_big [B + 2 spare][H] fp32."""
    from autoformer_b200 import packing
    dev = hs_big.device
    region = torch.zeros(hs_big.shape, dtype=torch.bool)
    region[:L] = True
    check_sentinel(hs_big, region, what + " hs")
    lreg = torch.zeros(h_last_big.shape, dtype=torch.bool)
    lreg[spare:spare + B] = True
    check_sentinel(h_last_big, lreg, what + " h_last")
    hs = hs_big[:L]
    h_last = h_last_big[spare:spare + B]
    assert not bool(hs[:, 0].float().any()), what + ": frame 0 of hs is not zero"
    assert torch.equal(_bits(h_last.to(torch.float16)), _bits(hs[L - 1, T])), what + ": fp16(h_last) != hs[L-1][T]"
    seq = hs.permute(0, 2, 1, 3)                              # [L][B][T + 1][H]
    for l in range(L):
        w_ih, w_hh, b_ih, b_hh = raws[l]
        Whh = weight_terms(w_hh.to(dev), "f16")[0]
        pairs = [(seq[l, :, :T].double(), Whh)]                  # frame t reads hs[l][t] = h^l_{t-1}
        if l == 0:
            base, kx = xproj0.double(), 0
        else:
            base = (b_ih.float() + b_hh.float()).double().to(dev)
            pairs.append((seq[l - 1, :, 1:].double(), weight_terms(w_ih.to(dev), "f16")[0]))   # hs[l-1][t+1]
            kx = H
        h, bound = tf_reference(base, pairs, H + kx + 3)
        got = seq[l, :, 1:].double()
        check_h(got, h, bound + half_ulp(h.abs() + bound, "f16"), f"{what} hs[{l}]")
        if l == L - 1:
            check_h(h_last, h[:, -1], bound[:, -1], what + " h_last")
            _gate("lstm_stack/h_last", h_last, h[:, -1])
        _gate("lstm_stack/hs", got, h)


def run_stack_case(c, dev, lstm_stack_ws=None):
    from autoformer_b200 import ops, packing
    lstm_stack_ws = lstm_stack_ws or ops.lstm_stack_ws
    L, B, T, H = c["L"], c["B"], c["T"], c["H"]
    seed = zlib.crc32(_stack_id(c).encode()) % 10007
    raws = [make_layer(H, H, seed + l, "cpu") for l in range(L)]
    packs = [tuple(None if t is None else t.to(dev) for t in packing.pack_lstm_stack(*r, first=l == 0))
             for l, r in enumerate(raws)]
    xproj0 = make_xproj(B, T, 4 * H, seed + 99, "cpu")
    perm = packing.gate_permutation(H, packing.WS_GROUP)
    xp = xproj0[..., perm].contiguous().view(B * T, 4 * H).to(dev)
    outs = []
    for _ in range(2):
        hs_big = _nan((L + 1, T + 1, B, H), torch.float16, dev)
        last_big = _nan((B + 2, H), torch.float32, dev)
        out = lstm_stack_ws(xp, packs, B, T, H, h_last=last_big[1:1 + B], hs=hs_big[:L])
        assert out is not None, "avc_lstm_stack_ws: the grid is not co-resident"
        outs.append((hs_big, last_big))
    check_stack(*outs[0], L, B, T, H, xproj0.to(dev), raws, "stack " + _stack_id(c))
    assert torch.equal(_bits(outs[1][0]), _bits(outs[0][0])) and torch.equal(_bits(outs[1][1]), _bits(outs[0][1]))
    return outs[0]


@pytest.mark.gpu
@pytest.mark.parametrize("case", STACK_CASES, ids=_stack_id)
def test_lstm_stack_contract(case):
    run_stack_case(case, "cuda")


# ------------------------------------------------------------------------------------------------ avc_bilstm_small
def _bi_id(c):
    return f"{bilstm_kernel(c['B'], c['H'])}-B{c['B']}H{c['H']}T{c['T']}f{c['freq']}"


def gather_codes(out, H, freq):
    return torch.cat((out[:, freq - 1::freq, :H], out[:, ::freq, H:]), dim=-1)


def check_bilstm(out_big, codes_big, B, T, H, freq, xproj, w_hh, what, spare=1):
    """out_big [B + 2 spare][T][2H] fp32 (unrounded), codes_big [B + 2 spare][T / freq][2H]."""
    for big in (out_big, codes_big):
        region = torch.zeros(big.shape, dtype=torch.bool)
        region[spare:spare + B] = True
        check_sentinel(big, region, what)
    out, codes = out_big[spare:spare + B], codes_big[spare:spare + B]
    assert torch.equal(_bits(codes), _bits(gather_codes(out, H, freq))), what + ": codes are not the gathered frames"
    x = xproj.double().view(B, T, 8 * H)
    for d in range(2):
        seq = out[..., d * H:(d + 1) * H].double()
        h, bound = tf_reference(x[..., d * 4 * H:(d + 1) * 4 * H], [(shift(seq, reverse=d == 1), w_hh[d].double())],
                                H + 3, reverse=d == 1)
        check_h(out[..., d * H:(d + 1) * H], h, bound, f"{what} dir {d}")
        _gate("bilstm_small/fp32", seq, h)


def run_bilstm_case(c, dev, bilstm_small=None):
    from autoformer_b200 import ops, packing
    bilstm_small = bilstm_small or ops.bilstm_small
    B, T, H, freq = c["B"], c["T"], c["H"], c["freq"]
    seed = zlib.crc32(_bi_id(c).encode()) % 10007
    g = torch.Generator().manual_seed(seed)
    w_hh = (torch.randn(2, 4 * H, H, generator=g) * 2.0 / H ** 0.5).to(dev)
    xproj = make_xproj(B, T, 8 * H, seed + 1, "cpu").view(B * T, 8 * H).to(dev)
    out_big = _nan((B + 2, T, 2 * H), torch.float32, dev)
    codes_big = _nan((B + 2, T // freq, 2 * H), torch.float32, dev)
    bilstm_small(xproj, w_hh, B, T, H, out=out_big[1:1 + B], codes=codes_big[1:1 + B], freq=freq, round_tf32=False)
    what = "bilstm " + _bi_id(c)
    check_bilstm(out_big, codes_big, B, T, H, freq, xproj, w_hh, what)
    out = out_big[1:1 + B].cpu()
    # every output format equals the host conversion of the unrounded run
    fmts = [("tf32", dict(round_tf32=True), torch.float32, 2 * H, packing.round_tf32),
            ("bf16", dict(), torch.bfloat16, 2 * H, lambda v: v.to(torch.bfloat16)),
            ("split", dict(split=True), torch.bfloat16, 4 * H, lambda v: packing.to_act(v, "fp32")),
            ("fp16", dict(), torch.float16, 2 * H, lambda v: packing.to_act(v, "fp16x2"))]
    for name, kw, dtype, C, conv in fmts:
        big = _nan((B + 2, T, C), dtype, dev)
        bilstm_small(xproj, w_hh, B, T, H, out=big[1:1 + B], **kw)
        region = torch.zeros(big.shape, dtype=torch.bool)
        region[1:1 + B] = True
        check_sentinel(big, region, f"{what} {name}")
        assert torch.equal(_bits(big[1:1 + B]), _bits(conv(out))), f"{what}: {name} out != host conversion"


@pytest.mark.gpu
@pytest.mark.parametrize("case", BILSTM_CASES, ids=_bi_id)
def test_bilstm_small_contract(case):
    run_bilstm_case(case, "cuda")


# ------------------------------------------------------------------------------------------------ LstmLayer / production
def _layer_run(layer, xin, B, T, persistent, dev):
    r = SeqRun(B, T, layer.H, layer.precision, dev)
    layer(xin, B, T, hseq_f32=r.hseq_f32, h_last=r.h_last, persistent=persistent, hseq=r.hseq)
    torch.cuda.synchronize()
    return r


def check_layer(layer, r, xin, what):
    from autoformer_b200 import packing
    prec, H = layer.precision, layer.H
    dev = xin.device
    base, x_pairs = fused_base_and_pairs(xin, layer.w_ih.to(dev), layer.b_ih.to(dev), layer.b_hh.to(dev), prec,
                                         layer.C_in)
    kx = -(-layer.C_in // packing.KC[prec]) * packing.KC[prec]
    return r.check(base, x_pairs, layer.w_hh.to(dev), seq_nadd(prec, H, kx), what, f"lstm_seq/{prec}")


@pytest.mark.gpu
def test_lstm_layer_sub_batches_above_the_persistent_cap():
    """B = 600 at H = 1024: LstmLayer runs 512 + 88 utterances as two persistent launches into slices of one buffer."""
    from autoformer_b200 import layers
    B, T, H, c_in = 600, 3, 1024, 320
    w_ih, w_hh, b_ih, b_hh = make_layer(H, c_in, 600, "cuda")
    layer = layers.LstmLayer(w_ih, w_hh, b_ih, b_hh, "fp16x2", fused=True)
    xin = xin_buffer(make_xproj(B, T, c_in, 601, "cpu", 1.0), "fp16x2", "cuda")
    r = _layer_run(layer, xin, B, T, True, "cuda")
    check_layer(layer, r, xin, "LstmLayer B600")


@pytest.mark.gpu
@pytest.mark.parametrize("B", [512, 300])
def test_autovc_decoder_lstms_production_shape(B):
    """The headline's three recurrences: decoder lstm1 (320 -> 512) and lstm2 (512 -> 1024 -> 1024), T = 128, fp16x2,
    persistent, fused input projection, each layer reading the one below."""
    from autoformer_b200 import layers, packing
    T = 128
    x = xin_buffer(make_xproj(B, T, 320, B, "cpu", 1.0), "fp16x2", "cuda")
    for i, (c_in, H) in enumerate([(320, 512), (512, 1024), (1024, 1024)]):
        layer = layers.LstmLayer(*make_layer(H, c_in, 7 * B + i, "cuda"), "fp16x2", fused=True)
        r = _layer_run(layer, x, B, T, True, "cuda")
        check_layer(layer, r, x, f"decoder layer {i} B{B}")
        x = r.hseq


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,c_in", [(32, 1000, 80), (8, 64, 512)], ids=["LstmDV", "Adjust"])
def test_lstm_stack_production_shape(B, T, c_in):
    """LstmDV's stack (80 -> 768 x 3) and Adjust's (512 -> 768 x 3) as one wavefront launch, layer 0's projection
    through its ConvGemm as LstmStack does."""
    from autoformer_b200 import layers, ops, packing
    H, L = 768, 3
    raws = [make_layer(H, c_in if l == 0 else H, 31 * B + l, "cuda") for l in range(L)]
    stack = layers.LstmStack([layers.LstmLayer(*r, "fp16x2") for r in raws], "fp16x2", wavefront=True)
    assert stack.eligible(B, True)
    ih, _ = stack.layers[0].packs(packing.WS_GROUP)
    x = packing.to_act(make_xproj(B, T, c_in, B, "cpu", 1.0), "fp16x2").cuda()
    xp = torch.empty(B * T, 4 * H, device="cuda")
    ih(x, B, T, out2=xp)
    hs_big = nan_buf((L + 1, T + 1, B, H), torch.float16)
    last_big = nan_buf((B + 2, H), torch.float32)
    assert ops.lstm_stack_ws(xp, stack.packs(), B, T, H, h_last=last_big[1:1 + B], hs=hs_big[:L]) is not None
    torch.cuda.synchronize()
    perm = packing.gate_permutation(H, packing.WS_GROUP)
    xproj0 = torch.empty_like(xp.view(B, T, 4 * H))
    xproj0[..., perm] = xp.view(B, T, 4 * H)                    # back to PyTorch gate order, read exactly
    check_stack(hs_big, last_big, L, B, T, H, xproj0, raws, f"stack B{B}T{T}")


# ------------------------------------------------------------------------------------------------ the checker, on CPU
def _expect_fail(fn, *needles):
    with pytest.raises(AssertionError) as e:
        fn()
    assert any(n in str(e.value) for n in needles), str(e.value)


SELF_SEQ = [dict(kern="step", prec="fp32", group=16, B=5, H=64, T=4, c_in=40),
            dict(kern="fused", prec="fp16x2", group=32, B=130, H=128, T=3, c_in=40),
            dict(kern="fused", prec="bf16", group=32, B=3, H=64, T=3, c_in=24),
            dict(kern="step", prec="tf32", group=16, B=4, H=32, T=2, c_in=40)]


@pytest.mark.parametrize("case", SELF_SEQ, ids=_seq_id)
def test_checker_passes_emulated_lstm_seq(case):
    """CPU: tests/emulate.py's avc_lstm_seq stand-in (fp64 math, lo * lo products kept) passes every check."""
    run_seq_case(case, "cpu", lstm_seq=emulate._emu_lstm_seq)


def _seq_fixture():
    c = SELF_SEQ[0]
    from autoformer_b200 import packing
    B, T, H, prec = c["B"], c["T"], c["H"], c["prec"]
    w_ih, w_hh, b_ih, b_hh = make_layer(H, c["c_in"], 5, "cpu")
    xproj = make_xproj(B, T, 4 * H, 6, "cpu")
    perm = packing.gate_permutation(H, c["group"])
    r = SeqRun(B, T, H, prec, "cpu")
    emulate._emu_lstm_seq(xproj[..., perm].contiguous().view(B * T, 4 * H), packing.pack_lstm_hh(w_hh, prec, c["group"]),
                          B, T, H, prec, c["group"], hseq=r.hseq, hseq_f32=r.hseq_f32, h_last=r.h_last)
    check = lambda: r.check(xproj.double(), [], w_hh, seq_nadd(prec, H, 0), "self", "lstm_seq/fp32")
    return r, check


def test_checker_catches_injected_faults():
    """CPU: each injected fault alone is reported by the check meant to catch it."""
    r, check = _seq_fixture()
    h, bound = check()
    B, T, H = r.B, r.T, r.H
    from autoformer_b200 import packing

    def fault(apply, *needles):
        r2, check2 = _seq_fixture()
        apply(r2)
        _expect_fail(check2, *needles)

    def swap_units(x):                      # two hidden units exchanged in one frame, in every store
        x.hseq_f32[1, 2, [3, 7]] = x.hseq_f32[1, 2, [7, 3]].clone()
        x.hseq.copy_(packing.to_act(x.hseq_f32, "fp32"))
    fault(swap_units, "beyond the bound")

    def shift_utt(x):                        # one utterance one frame late
        x.hseq_f32[2, 1:] = x.hseq_f32[2, :-1].clone()
        x.hseq.copy_(packing.to_act(x.hseq_f32, "fp32"))
        x.h_last.copy_(x.hseq_f32[:, -1])
    fault(shift_utt, "beyond the bound")

    fault(lambda x: x.hseq[0, 1, H:].zero_(), "to_act")          # lo half of one operand row lost

    def perturb(x):                           # one element off by twice its bound
        x.hseq_f32[3, 2, 5] += 2 * float(bound[3, 2, 5])
        x.hseq.copy_(packing.to_act(x.hseq_f32, "fp32"))
    fault(perturb, "beyond the bound")

    fault(lambda x: x.hseq_big.__setitem__((B + SeqRun.SPARE, 0, 0), 0.5), "outside the output")   # past the slice
    fault(lambda x: x.f32_big.__setitem__((SeqRun.SPARE - 1, T - 1, H - 1), 0.5), "outside the output")


def test_checker_passes_emulated_ws_stack_bilstm():
    """CPU: the avc_lstm_seq_ws, avc_lstm_stack_ws and avc_bilstm_small stand-ins pass every check; codes taken from the
    wrong frame fail, as does one stack element off by twice its bound."""
    run_ws_case(dict(prec="fp32", H=256, B=3, T=3), "cpu", lstm_seq_ws=emulate._emu_lstm_seq_ws)
    run_ws_case(dict(prec="fp16x2", H=256, B=2, T=2), "cpu", lstm_seq_ws=emulate._emu_lstm_seq_ws)
    hs_big, last_big = run_stack_case(dict(L=2, H=128, B=3, T=4), "cpu", lstm_stack_ws=emulate._emu_lstm_stack_ws)
    # bilstm: the stand-in writes fp32 output and codes exactly as the kernel's formats are defined
    B, T, H, freq = 3, 8, 16, 4
    g = torch.Generator().manual_seed(3)
    w_hh = torch.randn(2, 4 * H, H, generator=g) * 2.0 / H ** 0.5
    xproj = torch.randn(B * T, 8 * H, generator=g) * 1.5
    out_big = torch.full((B + 2, T, 2 * H), float("nan"))
    codes_big = torch.full((B + 2, T // freq, 2 * H), float("nan"))
    emulate._emu_bilstm_small(xproj, w_hh, B, T, H, out=out_big[1:1 + B], codes=codes_big[1:1 + B], freq=freq,
                              round_tf32=False)
    check_bilstm(out_big, codes_big, B, T, H, freq, xproj, w_hh, "bilstm emu")
    bad = codes_big.clone()
    bad[1:1 + B] = torch.cat((out_big[1:1 + B, ::freq, :H], out_big[1:1 + B, ::freq, H:]), dim=-1)   # r == 0 both ways
    _expect_fail(lambda: check_bilstm(out_big, bad, B, T, H, freq, xproj, w_hh, "bilstm codes"), "gathered")
    wrong = out_big.clone()
    wrong[2, 3, 5] += 0.01
    _expect_fail(lambda: check_bilstm(wrong, codes_big, B, T, H, freq, xproj, w_hh, "bilstm out"), "beyond the bound",
                 "gathered")


def test_checker_stack_faults():
    """CPU: a stack hs element off by twice its bound, and h_last of the wrong frame, are reported."""
    c = dict(L=2, H=128, B=3, T=4)
    hs_big, last_big = run_stack_case(c, "cpu", lstm_stack_ws=emulate._emu_lstm_stack_ws)
    L, B, T, H = c["L"], c["B"], c["T"], c["H"]
    seed = zlib.crc32(_stack_id(c).encode()) % 10007
    raws = [make_layer(H, H, seed + l, "cpu") for l in range(L)]
    xproj0 = make_xproj(B, T, 4 * H, seed + 99, "cpu")
    bad = hs_big.clone()
    bad[0, 2, 1, 4] = float(bad[0, 2, 1, 4]) + 0.01
    _expect_fail(lambda: check_stack(bad, last_big, L, B, T, H, xproj0, raws, "hs"), "beyond the bound")
    lbad = last_big.clone()
    lbad[1:1 + B] = hs_big[L - 1, T - 1].float()
    _expect_fail(lambda: check_stack(hs_big, lbad, L, B, T, H, xproj0, raws, "h_last"), "h_last")
