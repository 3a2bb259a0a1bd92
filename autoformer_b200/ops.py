"""Thin Python wrappers over the C ABI (include/avc_b200.h).  torch is used only for device memory and the
current stream; every arithmetic operation runs in libavc_b200.so.  Nothing here falls back to torch math."""
import ctypes
import warnings

import torch

from . import _lib
from . import packing
from .packing import KC, TORCH_DTYPE


def _stream():
    """The current stream of the CURRENT device.  Every op checks (``_require_cuda``) that its tensors live on that
    device; the model classes enter ``torch.cuda.device(x.device)`` around their forward (``on_device_of_input``), so
    a model on cuda:1 launches on cuda:1 whatever the caller's current device is."""
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def on_device_of_input(forward):
    """Decorator for a drop-in model's ``forward``: run it with the first tensor argument's device current (kernel
    launches, tensor maps and function attributes are per device; the C ABI launches on the current device)."""
    import functools

    @functools.wraps(forward)
    def wrapped(self, x, *args, **kwargs):
        if isinstance(x, torch.Tensor) and x.is_cuda and x.device.index != torch.cuda.current_device():
            with torch.cuda.device(x.device):
                return forward(self, x, *args, **kwargs)
        return forward(self, x, *args, **kwargs)
    return wrapped


class Profiler:
    """Optional per-op CUDA-event timing on the launching stream (bench.py's roofline numbers).
    Disabled by default: the hot path then records nothing."""

    def __init__(self):
        self.enabled = False
        self.records = []          # (family, start_event, end_event, work dict)

    class _Span:
        def __init__(self, prof, family, work):
            self.prof, self.family, self.work = prof, family, work

        def __enter__(self):
            if self.prof.enabled:
                self.start = torch.cuda.Event(enable_timing=True)
                self.end = torch.cuda.Event(enable_timing=True)
                self.start.record()
            return self

        def __exit__(self, *exc):
            if self.prof.enabled:
                self.end.record()
                self.prof.records.append((self.family, self.start, self.end, self.work))
            return False

    def span(self, family, **work):
        return Profiler._Span(self, family, work)

    def summary(self):
        """family -> dict(ms=total, launches=n, flops=sum, bytes=sum); call after a synchronize."""
        out = {}
        for family, s, e, work in self.records:
            d = out.setdefault(family, dict(ms=0.0, calls=0, launches=0, flops=0.0, bytes=0.0))
            d["ms"] += s.elapsed_time(e)
            d["calls"] += 1
            d["launches"] += work.get("launches", 1)
            d["flops"] += work.get("flops", 0.0)
            d["bytes"] += work.get("bytes", 0.0)
        return out

    def reset(self):
        self.records = []


PROFILER = Profiler()
_warned_not_resident = False


def _require_cuda(*tensors):
    """Every tensor of a launch must be a CUDA tensor on the current device (the one the launch goes to)."""
    cur = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("autoformer_b200 kernels need CUDA tensors (there is no CPU fallback)")
        if cur is None:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            raise RuntimeError(f"tensor on {t.device} but the current CUDA device is cuda:{cur}: call the op under "
                               "`with torch.cuda.device(t.device)` (the model classes do this themselves) and keep "
                               "all tensors of a call on one device")


def _dt(precision):
    """Operand-format code of an activation buffer (include/avc_b200.h out_dtype): 0 fp32/TF32, 1 bf16, 2 split bf16,
    3 fp16, 4 split fp16."""
    return {"tf32": _lib.DTYPE_TF32, "bf16": _lib.DTYPE_BF16, "fp32": 2, "fp16x2": 3, "f16": 3, "fp16s": 4}[precision]


def alloc_act(B, rows, C, precision, device):
    """Activation buffer carrying C logical channels in the storage format of `precision`."""
    return torch.empty(B, rows, packing.act_channels(C, precision), dtype=TORCH_DTYPE[precision], device=device)


def _out_dtype(t, split):
    """C-ABI out_dtype code of an operand-format output buffer: 0 fp32, 1 bf16, 2 split bf16, 3 fp16, 4 split fp16."""
    assert t.dtype in (torch.float32, torch.bfloat16, torch.float16)
    if t.dtype == torch.float16:
        return 4 if split else 3
    return (2 if split else 1) if t.dtype == torch.bfloat16 else 0


class ConvGemm:
    """A packed conv / linear layer bound to avc_conv_gemm.

    ``w``/``bias``/``meta`` come from ``packing.pack_conv*``; ``tap_t0``/``tap_dt`` per source give the buffer row
    read by tap 0 for output frame 0 (``-pad`` for an unpadded input buffer) and the dilation."""

    def __init__(self, w, bias, meta, tap_t0=None, tap_dt=None, act="none", tag="gemm"):
        self.w, self.bias, self.meta = w, bias, meta
        self.tag = tag
        # algorithmic MACs per output row: real channels x taps x real output channels
        if meta.get("split") or meta.get("dup"):
            self.macs_per_row = sum(c * k for c, k in zip(meta["logical_channels"], meta["logical_taps"])) * meta["N"]
        else:
            self.macs_per_row = sum(c * k for c, k in zip(meta["channels"], meta["taps"])) * meta["N"]
        n_src = len(meta["taps"])
        # tap geometry is given per LOGICAL source; split precision duplicates it for the two physical sources
        rep = 2 if (meta.get("split") or meta.get("dup")) else 1
        if tap_t0 is not None:
            self.tap_t0 = [v for v in tap_t0 for _ in range(rep)]
        else:
            self.tap_t0 = [-(k // 2) for k in meta["taps"]]
        self.tap_dt = [v for v in tap_dt for _ in range(rep)] if tap_dt is not None else [1] * n_src
        assert len(self.tap_t0) == n_src and len(self.tap_dt) == n_src
        self.act = _lib.ACTS[act]
        self.precision = meta["precision"]

    def to(self, device):
        self.w = self.w.to(device)
        self.bias = self.bias.to(device)
        return self

    def __call__(self, srcs, B, T, out=None, out_row0=0, round_tf32=True, reflect=0, out2=None, residual=None,
                 out_raw=None, phases=1, res_after=False, out_fmt=None, raw_fmt=None, halo_after=False, phase0=0,
                 phase_count=None):
        """srcs: channels-last activation tensors [B][rows][C_s], one per logical source.
        out: act(v) [B][rows_out][Cs'] (operand format) at rows out_row0 + time (+ `reflect` mirrored halo rows);
        out_raw: v before the activation [B][phases*T][Cs'] (operand format); out2: act(v) as exact fp32
        [B*phases*T][Cs]; residual fp32 [B*phases*T][Cs] is added before the activation.  Cs = N / phases.
        out_fmt / raw_fmt: operand format (a precision name) of out / out_raw when it differs from this layer's own
        input precision -- e.g. a "fp16s" layer writing LeakyReLU(y) as "f16" and y as "fp16s".
        halo_after: write the `reflect` halo rows with a separate avc_reflect_halo launch instead of in the GEMM's
        epilogue, which keeps the GEMM on its branch-free store path.
        phase0 / phase_count: this layer produces only phases [phase0, phase0 + phase_count) of the `phases` (its N is
        phase_count * Cs); the halo launch, if any, is then the caller's business."""
        lib = _lib.load()
        meta = self.meta
        if not isinstance(srcs, (list, tuple)):
            srcs = [srcs]
        _require_cuda(self.w, *srcs)
        split = bool(meta.get("split"))
        if split:      # one buffer [hi | lo] per logical source: all 2C channels, then the hi half
            assert len(srcs) == len(meta["logical_channels"])
            phys = []
            for a, c in zip(srcs, meta["logical_channels"]):
                assert a.shape[2] == 2 * c, (a.shape, c)
                phys += [a, a[:, :, :c]]
            srcs = phys
        elif meta.get("dup"):     # fp16x2: the same buffer against w_hi and against w_lo
            assert len(srcs) == len(meta["logical_channels"])
            srcs = [a for a in srcs for _ in range(2)]
        assert len(srcs) == len(meta["taps"])
        d = _lib.GemmDesc()
        want = TORCH_DTYPE[self.precision]
        for s, a in enumerate(srcs):
            assert a.dim() == 3 and a.shape[0] == B and a.dtype == want and a.stride(2) == 1, (a.shape, a.dtype)
            assert a.shape[2] == meta["channels"][s], (a.shape, meta["channels"])
            assert a.stride(0) == a.shape[1] * a.stride(1)
            d.a_ptr[s] = a.data_ptr()
            d.a_channels[s] = a.shape[2]
            d.a_ld[s] = a.stride(1)
            d.a_rows_per_utt[s] = a.shape[1]
            d.a_taps[s] = meta["taps"][s]
            d.a_tap_t0[s] = self.tap_t0[s]
            d.a_tap_dt[s] = self.tap_dt[s]
        d.w_ptr = self.w.data_ptr()
        d.n_pad, d.k_pad = meta["n_pad"], meta["k_pad"]
        d.dtype = {"tf32": _lib.DTYPE_TF32, "fp16x2": _lib.DTYPE_F16, "fp16s": _lib.DTYPE_F16,
                   "f16": _lib.DTYPE_F16}.get(self.precision, _lib.DTYPE_BF16)
        d.B, d.T, d.N = B, T, meta["N"]
        d.bias = self.bias.data_ptr()
        d.act = self.act
        d.out_phases = phases
        if phase_count is None:
            phase_count = phases
        d.out_phase0, d.out_phase_count = phase0, phase_count
        cs = meta["N"] // phase_count
        out_fmt = out_fmt or self.precision
        raw_fmt = raw_fmt or out_fmt
        if out is not None:
            assert out.is_cuda and out.dim() == 3 and out.shape[0] == B and out.stride(2) == 1
            assert out.dtype == TORCH_DTYPE[out_fmt] and out.shape[2] >= packing.act_channels(cs, out_fmt)
            assert out.stride(0) == out.shape[1] * out.stride(1)
            d.out = out.data_ptr()
            d.out_ld = out.stride(1)
            d.out_rows_per_utt = out.shape[1]
            d.out_row0 = out_row0
            d.out_dtype = _dt(out_fmt)
            d.out_round_tf32 = 1 if (round_tf32 and out.dtype == torch.float32) else 0
            d.out_reflect = 0 if halo_after else reflect
            assert not halo_after or out.is_contiguous()
        if out_raw is not None:
            assert out_raw.is_cuda and out_raw.dtype == TORCH_DTYPE[raw_fmt] and out_raw.stride(-1) == 1
            assert out_raw.shape[-1] >= packing.act_channels(cs, raw_fmt)
            d.out_raw = out_raw.data_ptr()
            d.out_raw_ld = out_raw.stride(-2)
            d.out_raw_dtype = _dt(raw_fmt)
            if out is None:
                d.out_dtype = _dt(raw_fmt)
            d.out_round_tf32 = 1 if (round_tf32 and out_raw.dtype == torch.float32) else 0
        if out2 is not None:
            assert out2.is_cuda and out2.dtype == torch.float32 and out2.stride(-1) == 1
            d.out2 = out2.data_ptr()
            d.out2_ld = out2.stride(-2)
        if residual is not None:
            assert residual.is_cuda and residual.dtype == torch.float32 and residual.stride(-1) == 1
            d.residual = residual.data_ptr()
            d.res_ld = residual.stride(-2)
            d.res_after_act = 1 if res_after else 0
        d.block_n = meta["block_n"]
        d.cta_group = getattr(self, "cta_group", 0)
        dbg = getattr(self, "debug_clk", None)
        if dbg is not None:
            d.debug_clk = dbg.data_ptr()
        with PROFILER.span(self.tag, flops=2.0 * self.macs_per_row * B * T):
            _lib.check(lib.avc_conv_gemm(ctypes.byref(d), _stream()), "avc_conv_gemm")
        if halo_after and reflect and out is not None and phase_count == phases:
            reflect_halo(out, out_row0, T * phases, reflect)
        return out if out is not None else (out2 if out2 is not None else out_raw)


def reflect_halo(buf, row0, L, reflect, lengths=None):
    """Fill the `reflect` mirrored rows each side of rows [row0, row0 + L) of a channels-last buffer [B][rows][C'].
    lengths (device int32 [B], reflect < lengths[b] <= L): utterance b of a padded batch ends at row row0 + lengths[b]
    - 1, and its right halo mirrors about that row."""
    lib = _lib.load()
    _require_cuda(buf)
    assert buf.dim() == 3 and buf.is_contiguous()
    B, rows, _ = buf.shape
    lens = _check_lengths(lengths, B) if lengths is not None else None
    with PROFILER.span("halo", bytes=float(2 * B * 2 * reflect * buf.shape[2] * buf.element_size())):
        _lib.check(lib.avc_reflect_halo(buf.data_ptr(), B, rows, buf.shape[2] * buf.element_size(), row0, L, reflect,
                                        _stream(), lens), "avc_reflect_halo")
    return buf


def _check_lengths(lengths, B):
    """Per-utterance lengths of a padded batch: a device int32 [B] tensor (values are validated by the caller, on the
    host, before the upload -- the kernels trust them)."""
    assert lengths.dtype == torch.int32 and lengths.is_contiguous() and lengths.shape == (B,), (lengths.shape, B)
    _require_cuda(lengths)
    return lengths.data_ptr()


def zero_tail(buf, row0, T, lengths):
    """Zero rows row0 + lengths[b] .. row0 + T - 1 of utterance b of a channels-last buffer [B][rows][C'] (any operand
    format): the padded frames of a variable-length batch then read as the zero padding of the next convolution."""
    lib = _lib.load()
    _require_cuda(buf)
    assert buf.dim() == 3 and buf.is_contiguous()
    B, rows, _ = buf.shape
    row_bytes = buf.shape[2] * buf.element_size()
    with PROFILER.span("zero_tail", bytes=float(B * T * row_bytes)):
        _lib.check(lib.avc_zero_tail(buf.data_ptr(), B, rows, row_bytes, row0, T, _check_lengths(lengths, B), _stream()),
                   "avc_zero_tail")
    return buf


class RaggedRows:
    """Valid rows per utterance of one buffer geometry (one generator stage) of a padded batch.  ``host``: list of B
    ints; ``rows``: the same as a device int32 [B] tensor (the ``lengths`` of reflect_halo / zero_tail /
    conv_to_mono_tanh); ``tiles[S]``: (device int32 [B + 1] prefix table of ceil(host[b] / S), its total) -- the
    compacted tile space avc_resblock2 runs over with tiles of stride S."""

    def __init__(self, host, rows, tiles):
        self.host, self.rows, self.tiles = host, rows, tiles


def ragged_rows(lengths, scales, strides, device):
    """RaggedRows of rows = s * lengths[b] for every scale s, with tile tables for every stride.  `lengths` is a host
    list already validated by the caller; all rows and tables go to the device in ONE int32 copy."""
    B = len(lengths)
    flat, layout = [], []
    for s in scales:
        host = [s * n for n in lengths]
        off = len(flat)
        flat += host
        tables = {}
        for S in strides:
            start = [0]
            for r in host:
                start.append(start[-1] + (r + S - 1) // S)
            tables[S] = (len(flat), start[-1])
            flat += start
        layout.append((host, off, tables))
    dev = torch.tensor(flat, dtype=torch.int32).to(device)
    return [RaggedRows(host, dev[off:off + B], {S: (dev[o:o + B + 1], n) for S, (o, n) in tables.items()})
            for host, off, tables in layout]


# Cap on the CTAs one persistent LSTM launch may take (None: the whole device).  pipeline.convert_pairs sets it to half
# the SMs while it runs two under-filled batches on two streams, so that both cooperative grids are resident together.
LSTM_CTA_BUDGET = None


def persistent_batch_cap(H, n_sm=148):
    """Largest batch whose persistent LSTM grid (m-tiles x H/G n-tiles, one CTA each) fits one wave of the SMs."""
    best = 0
    for g in (32, 16):
        if H % g:
            continue
        m_tiles = n_sm // (H // g)
        if m_tiles >= 2:
            m_tiles -= m_tiles % 2                 # CTA pairs
        best = max(best, m_tiles * 128)
    return best


def choose_gate_group(B, H, persistent=False, n_sm=148):
    """Hidden units per accumulator tile (tile width 4G): fill the SMs without exceeding one wave when persistent."""
    if LSTM_CTA_BUDGET is not None:                # two batches side by side on two streams: each takes half the SMs
        n_sm = min(n_sm, LSTM_CTA_BUDGET)
    m_tiles = (B + 127) // 128
    if m_tiles >= 2:
        m_tiles = (m_tiles + 1) // 2 * 2          # CTA pairs: an odd tile count is rounded up with a masked tile
    choice = None
    for g in (32, 16):
        if H % g:
            continue
        ctas = m_tiles * (H // g)
        if ctas >= 96 and (not persistent or ctas <= n_sm):
            choice = g
            break
    if choice is None:
        for g in (16, 32):
            if H % g == 0 and (not persistent or m_tiles * (H // g) <= n_sm):
                choice = g
                break
    if choice is not None:
        return choice
    raise RuntimeError(f"no gate group fits B={B} H={H} persistent={persistent}")


def _lstm_desc(xproj, w_hh, B, T, H, precision, group, hseq, hseq_f32, h_last, persistent, debug_clk, xin, w_ih, bias,
               c_in, lengths, c_state):
    """Checked avc_lstm_desc of one layer; returns (desc, hseq, tensors the descriptor points to)."""
    fused = xin is not None
    _require_cuda(xin if fused else xproj, w_hh)
    dev = w_hh.device
    if fused:
        assert xproj is None and w_ih is not None and bias is not None and c_in is not None
        kp = (c_in + KC[precision] - 1) // KC[precision] * KC[precision]
        assert xin.dim() == 3 and xin.shape[0] == B and xin.shape[1] == T and xin.dtype == TORCH_DTYPE[precision]
        assert xin.shape[2] >= packing.act_channels(c_in, precision) and xin.stride(2) == 1
        assert xin.stride(0) == T * xin.stride(1) and c_in % 8 == 0
        assert w_ih.dtype == TORCH_DTYPE[precision] and w_ih.is_contiguous()
        assert w_ih.shape == (4 * H, 2 * kp if precision in packing.TWO_TERM_WEIGHTS else kp), (w_ih.shape, kp)
        assert bias.dtype == torch.float32 and bias.is_contiguous() and bias.numel() == 4 * H
        _require_cuda(w_ih, bias)
    else:
        assert xproj.dtype == torch.float32 and xproj.is_contiguous() and xproj.numel() == B * T * 4 * H
    wk = 2 * H if precision in packing.TWO_TERM_WEIGHTS else H
    assert w_hh.dtype == TORCH_DTYPE[precision] and w_hh.is_contiguous()
    assert w_hh.shape == (4 * H, wk), (w_hh.shape, H, group)
    if hseq is None:
        hseq = alloc_act(B, T, H, precision, dev)
    assert hseq.is_contiguous() and hseq.shape == (B, T, packing.act_channels(H, precision))
    assert hseq.dtype == TORCH_DTYPE[precision]
    if c_state is None:
        c_state = torch.empty(B, H, dtype=torch.float32, device=dev)
    assert c_state.is_contiguous() and c_state.shape == (B, H) and c_state.dtype == torch.float32
    d = _lib.LstmDesc()
    if fused:
        d.xin, d.xin_channels, d.xin_ld = xin.data_ptr(), c_in, xin.stride(1)
        d.w_ih, d.bias = w_ih.data_ptr(), bias.data_ptr()
    else:
        d.xproj = xproj.data_ptr()
    d.w_hh = w_hh.data_ptr()
    d.hseq = hseq.data_ptr()
    if lengths is not None:
        d.lengths = _check_lengths(lengths, B)
        if h_last is not None and hseq_f32 is None:
            hseq_f32 = torch.empty(B, T, H, dtype=torch.float32, device=dev)
    if hseq_f32 is not None:
        assert hseq_f32.is_contiguous() and hseq_f32.shape == (B, T, H) and hseq_f32.dtype == torch.float32
        d.hseq_f32 = hseq_f32.data_ptr()
    if h_last is not None:
        assert h_last.is_contiguous() and h_last.shape == (B, H) and h_last.dtype == torch.float32
        d.h_last = h_last.data_ptr()
    d.c_state = c_state.data_ptr()
    d.B, d.T, d.H = B, T, H
    d.dtype = _dt(precision)
    d.gate_group = group
    d.persistent = 1 if persistent else 0
    bar = None
    if persistent:
        bar = torch.empty(64 * 32, dtype=torch.int32, device=dev)     # zeroed by the library
        d.grid_barrier = bar.data_ptr()
    if debug_clk is not None:
        d.debug_clk = debug_clk.data_ptr()
    return d, hseq, (c_state, bar, hseq_f32)


def lstm_seq(xproj, w_hh, B, T, H, precision, group, hseq=None, hseq_f32=None, h_last=None, persistent=False,
             debug_clk=None, xin=None, w_ih=None, bias=None, c_in=None, lengths=None, c_state=None):
    """Run the recurrence of one uni-directional layer.  Either xproj [B*T][4H] fp32 (packed gate order, bias
    included), or -- fused input projection -- the layer input xin [B][T][C'] in the operand format of `precision`
    with w_ih / bias from packing.pack_lstm_ih_fused and c_in logical input channels.
    lengths: optional device int32 [B] of a padded batch -- h_last[b] is then h at frame lengths[b] - 1 (taken from the
    exact fp32 sequence, allocated here when hseq_f32 is not given).  c_state: optional [B][H] fp32 that receives the
    final cell state (scratch allocated here otherwise)."""
    lib = _lib.load()
    fused = xin is not None
    d, hseq, keep = _lstm_desc(xproj, w_hh, B, T, H, precision, group, hseq, hseq_f32, h_last, persistent, debug_clk,
                               xin, w_ih, bias, c_in, lengths, c_state)
    with PROFILER.span("lstm_step", flops=2.0 * 4 * H * (H + (c_in if fused else 0)) * B * T,
                       launches=1 if persistent else T):
        rc = lib.avc_lstm_seq(ctypes.byref(d), _stream())
        if rc == _lib.ERR_NOT_RESIDENT and persistent:
            # the one-wave persistent grid does not fit this device (fewer SMs available than planned): same kernel,
            # one launch per frame
            global _warned_not_resident
            if not _warned_not_resident:
                warnings.warn("persistent LSTM grid is not co-resident on this device; using per-frame launches: "
                              + lib.avc_last_error().decode("utf-8", "replace"))
                _warned_not_resident = True
            d.persistent = 0
            rc = lib.avc_lstm_seq(ctypes.byref(d), _stream())
        _lib.check(rc, "avc_lstm_seq")
    return hseq


def lstm_seq2(w_hh, B, T, H, precision, group, xin, w_ih, bias, c_in, hseq=(None, None), hseq_f32=(None, None),
              c_state=(None, None), debug_clk=None):
    """Two stacked layers with fused input projections as ONE persistent launch (avc_lstm_seq2), layer 1 two frames
    behind layer 0: bit-identical to two persistent lstm_seq calls.  w_hh / w_ih / bias / hseq / hseq_f32 / c_state are
    (layer 0, layer 1) pairs; xin is layer 0's input with c_in channels, layer 1 reads layer 0's hseq.  Returns the two
    hseq tensors, or None when the device cannot hold the grid (nothing was launched; run the layers one by one)."""
    lib = _lib.load()
    d0, h0, keep0 = _lstm_desc(None, w_hh[0], B, T, H, precision, group, hseq[0], hseq_f32[0], None, True, debug_clk,
                               xin, w_ih[0], bias[0], c_in, None, c_state[0])
    d1, h1, keep1 = _lstm_desc(None, w_hh[1], B, T, H, precision, group, hseq[1], hseq_f32[1], None, True, None,
                               h0, w_ih[1], bias[1], H, None, c_state[1])
    with PROFILER.span("lstm_step", flops=2.0 * 4 * H * ((H + c_in) + 2 * H) * B * T, launches=1):
        rc = lib.avc_lstm_seq2(ctypes.byref(d0), ctypes.byref(d1), _stream())
    if rc == _lib.ERR_NOT_RESIDENT:
        return None
    _lib.check(rc, "avc_lstm_seq2")
    return h0, h1


WS_MAX_BATCH = 64


def ws_supported(B, H, precision, n_sm=148):
    """Shapes the weight-stationary recurrence (avc_lstm_seq_ws) takes: split precision, B <= 64, the 4H/128 row
    blocks x 4 K-slices within one wave (8 slices are used when the device can hold them); the W slice lives in
    tensor memory (<= 256 of the 512 columns, beside the accumulator), the h slice and the reduction buffer in
    shared memory."""
    if precision not in packing.TWO_TERM_WEIGHTS or B < 1 or B > WS_MAX_BATCH or H % 256 or 4 * H // 128 * 4 > n_sm:
        return False
    ar = 16 if B <= 16 else (32 if B <= 32 else 64)
    chunks = H // 4 // 64
    red = (128 * ar * 4 + 1023) // 1024 * 1024
    stage = (ar * 8 * 4 + 1023) // 1024 * 1024
    return chunks * 2 * ar * 128 + red + stage + 1152 <= 227 * 1024 and 2 * ar + 64 * chunks <= 512


def lstm_seq_ws(xproj, w_hh, B, T, H, hseq=None, hseq_f32=None, h_last=None, debug_clk=None, precision="fp32",
                lengths=None):
    """Small-batch recurrence with W_hh resident in tensor memory (split precision).  xproj [B*T][4H] fp32 and w_hh
    [4H][2H] bf16 in the packing.WS_GROUP gate order.  Returns hseq, or None when the device cannot hold the grid
    (nothing was launched; the caller uses lstm_seq).  lengths: optional device int32 [B], h_last[b] = h at frame
    lengths[b] - 1."""
    lib = _lib.load()
    _require_cuda(xproj, w_hh)
    dev = w_hh.device
    assert xproj.dtype == torch.float32 and xproj.is_contiguous() and xproj.numel() == B * T * 4 * H
    assert precision in packing.TWO_TERM_WEIGHTS
    assert w_hh.dtype == TORCH_DTYPE[precision] and w_hh.shape == (4 * H, 2 * H) and w_hh.is_contiguous()
    if hseq is None:
        hseq = alloc_act(B, T, H, precision, dev)
    assert hseq.is_contiguous() and hseq.shape == (B, T, packing.act_channels(H, precision))
    assert hseq.dtype == TORCH_DTYPE[precision]
    d = _lib.LstmWsDesc()
    d.dtype = _dt(precision)
    d.xproj, d.w_hh, d.hseq = xproj.data_ptr(), w_hh.data_ptr(), hseq.data_ptr()
    if hseq_f32 is not None:
        assert hseq_f32.is_contiguous() and hseq_f32.shape == (B, T, H) and hseq_f32.dtype == torch.float32
        d.hseq_f32 = hseq_f32.data_ptr()
    if h_last is not None:
        assert h_last.is_contiguous() and h_last.shape == (B, H) and h_last.dtype == torch.float32
        d.h_last = h_last.data_ptr()
    if lengths is not None:
        d.lengths = _check_lengths(lengths, B)
    bar = torch.empty(256, dtype=torch.int32, device=dev)             # zeroed by the library
    d.grid_barrier = bar.data_ptr()
    d.B, d.T, d.H = B, T, H
    if debug_clk is not None:
        d.debug_clk = debug_clk.data_ptr()
    with PROFILER.span("lstm_ws", flops=2.0 * 4 * H * H * B * T, launches=1):
        rc = lib.avc_lstm_seq_ws(ctypes.byref(d), _stream())
    if rc == _lib.ERR_NOT_RESIDENT:
        return None
    _lib.check(rc, "avc_lstm_seq_ws")
    return hseq


def stack_supported(B, H, L, precision, n_sm=148):
    """Shapes the wavefront stack kernel (avc_lstm_stack_ws) takes: fp16 operands ("fp16x2"), 2 <= L <= 4 layers of the
    same width, B <= 64, H a multiple of 128 whose H/2 tensor-memory columns of weights fit beside the two accumulators,
    and L x 4H/128 x 2 CTAs within one wave."""
    if precision != "fp16x2" or not 1 <= B <= WS_MAX_BATCH or not 2 <= L <= _lib.STACK_MAX_LAYERS:
        return False
    if H % 128 or H // 2 + 128 > 512 or L * (4 * H // 128) * 2 > n_sm:
        return False
    ar = 16 if B <= 16 else (32 if B <= 32 else 64)
    nc = H // 128
    tiles = 2 * ((nc + 1) // 2) + nc                  # h^l_{t-1} half in whole load groups + h^{l-1}_{t+1} half
    return tiles * ar * 128 + 2 * ar * 64 * 4 + 4096 + 1152 <= 227 * 1024


def lstm_stack_ws(xproj0, packs, B, T, H, h_last=None, hs=None, debug_clk=None, lengths=None):
    """All layers of a small-batch LSTM stack as one wavefront launch.  xproj0 [B*T][4H] fp32 (layer 0's dense input
    projection, biases included), `packs` = [(w_ih, w_hh, bias)] per layer (packing.pack_lstm_stack; w_ih and bias are
    None for layer 0); all in the packing.WS_GROUP gate order.  Returns the scratch sequences hs [L][T+1][B][H] fp16
    (frame t+1 of layer l = h^l_t), or None when the device cannot hold the grid (nothing was launched).
    lengths: optional device int32 [B], h_last[b] = the top layer's h at frame lengths[b] - 1."""
    lib = _lib.load()
    _require_cuda(xproj0, packs[0][1])
    dev = packs[0][1].device
    L = len(packs)
    assert xproj0.dtype == torch.float32 and xproj0.is_contiguous() and xproj0.numel() == B * T * 4 * H
    if hs is None:
        hs = torch.empty(L, T + 1, B, H, dtype=torch.float16, device=dev)
    assert hs.is_contiguous() and hs.shape == (L, T + 1, B, H) and hs.dtype == torch.float16
    d = _lib.LstmStackDesc()
    d.xproj0, d.hs = xproj0.data_ptr(), hs.data_ptr()
    for l, (w_ih, w_hh, bias) in enumerate(packs):
        for w in (w_hh,) if l == 0 else (w_ih, w_hh):
            assert w.dtype == torch.float16 and w.shape == (4 * H, H) and w.is_contiguous() and w.device == dev
        d.w_hh[l] = w_hh.data_ptr()
        if l > 0:
            assert bias.dtype == torch.float32 and bias.shape == (4 * H,) and bias.is_contiguous() and bias.device == dev
            d.w_ih[l], d.bias[l] = w_ih.data_ptr(), bias.data_ptr()
    if h_last is not None:
        assert h_last.is_contiguous() and h_last.shape == (B, H) and h_last.dtype == torch.float32
        d.h_last = h_last.data_ptr()
    if lengths is not None:
        d.lengths = _check_lengths(lengths, B)
    bar = torch.empty(256, dtype=torch.int32, device=dev)             # zeroed by the library
    d.grid_barrier = bar.data_ptr()
    d.B, d.T, d.H, d.L = B, T, H, L
    if debug_clk is not None:
        d.debug_clk = debug_clk.data_ptr()
    flops = 2.0 * 4 * H * H * B * T * (2 * L - 1)      # W_hh of every layer + W_ih of the layers above the first
    with PROFILER.span("lstm_stack", flops=flops, launches=1):
        rc = lib.avc_lstm_stack_ws(ctypes.byref(d), _stream())
    if rc == _lib.ERR_NOT_RESIDENT:
        return None
    _lib.check(rc, "avc_lstm_stack_ws")
    return hs


def bilstm_small(xproj, w_hh, B, T, H, out=None, codes=None, freq=1, round_tf32=True, split=False, lengths=None):
    """xproj [B*T][8H] fp32; w_hh [2][4H][H] fp32; out [B][T][2H] (fp32/bf16; split: [B][T][4H] bf16) and/or
    codes [B][T/freq][2H] fp32.  lengths: optional device int32 [B] of a padded batch (each a multiple of freq, checked
    by the caller): utterance b runs over its first lengths[b] frames only, later out rows and codes are 0."""
    lib = _lib.load()
    _require_cuda(xproj, w_hh)
    assert xproj.dtype == torch.float32 and xproj.is_contiguous() and xproj.numel() == B * T * 8 * H
    assert w_hh.dtype == torch.float32 and w_hh.is_contiguous() and w_hh.shape == (2, 4 * H, H)
    out_ptr, out_dtype = None, 0
    if out is not None:
        assert out.is_contiguous() and out.shape == (B, T, (4 if split else 2) * H)
        out_ptr, out_dtype = out.data_ptr(), _out_dtype(out, split)
    codes_ptr = None
    if codes is not None:
        assert codes.is_contiguous() and codes.dtype == torch.float32 and codes.shape == (B, T // freq, 2 * H)
        codes_ptr = codes.data_ptr()
    len_ptr = _check_lengths(lengths, B) if lengths is not None else None
    with PROFILER.span("bilstm_small", flops=2.0 * 2 * 4 * H * H * B * T, bytes=4.0 * B * T * 8 * H):
        _lib.check(lib.avc_bilstm_small(xproj.data_ptr(), w_hh.data_ptr(), out_ptr, out_dtype, 1 if round_tf32 else 0,
                                        codes_ptr, B, T, H, freq, _stream(), len_ptr), "avc_bilstm_small")
    return out, codes


def concat_bcast(seq, vec, T, div, precision, round_tf32=True):
    """[seq[b, t // div, :] || vec[b, :]] -> [B][T][C1+C2] in the operand dtype of `precision`."""
    lib = _lib.load()
    _require_cuda(seq, vec)
    assert seq.dtype == torch.float32 and seq.is_contiguous()
    B, Tin, C1 = seq.shape
    C2 = 0
    if vec is not None:
        assert vec.dtype == torch.float32 and vec.is_contiguous() and vec.shape[0] == B
        C2 = vec.shape[1]
    assert Tin * div == T
    out = alloc_act(B, T, C1 + C2, precision, seq.device)
    vec_ptr = vec.data_ptr() if vec is not None else None
    with PROFILER.span("concat", bytes=float(seq.numel() * 4 + out.numel() * out.element_size())):
        _lib.check(lib.avc_concat_bcast(seq.data_ptr(), vec_ptr, out.data_ptr(), B, T, C1, C2, div,
                                        _dt(precision), 1 if round_tf32 else 0, _stream()),
                   "avc_concat_bcast")
    return out


def linear_l2norm(h, w, bias):
    lib = _lib.load()
    _require_cuda(h, w, bias)
    assert h.dtype == torch.float32 and h.is_contiguous() and w.is_contiguous() and bias.is_contiguous()
    B, K = h.shape
    N = w.shape[0]
    out = torch.empty(B, N, dtype=torch.float32, device=h.device)
    _lib.check(lib.avc_linear_l2norm(h.data_ptr(), w.data_ptr(), bias.data_ptr(), out.data_ptr(), B, K, N, _stream()),
               "avc_linear_l2norm")
    return out


def linear_rows(h, w, bias, want_raw=True, want_normed=False):
    """Small fp32 Linear on [B][K] rows: returns (W h + b, (W h + b) / ||.||_2), None for the one not requested."""
    lib = _lib.load()
    _require_cuda(h, w, bias)
    assert h.dtype == torch.float32 and h.is_contiguous() and w.is_contiguous() and bias.is_contiguous()
    assert want_raw or want_normed
    B, K = h.shape
    N = w.shape[0]
    raw = torch.empty(B, N, dtype=torch.float32, device=h.device) if want_raw else None
    normed = torch.empty(B, N, dtype=torch.float32, device=h.device) if want_normed else None
    _lib.check(lib.avc_linear_rows(h.data_ptr(), w.data_ptr(), bias.data_ptr(), raw.data_ptr() if want_raw else None,
                                   normed.data_ptr() if want_normed else None, B, K, N, _stream()), "avc_linear_rows")
    return raw, normed


def to_act(x, precision, round_tf32=True):
    """fp32 [B][T][C] -> operand format of `precision` (a concat_bcast launch with no broadcast part)."""
    return concat_bcast(x, None, x.shape[1], 1, precision, round_tf32)


def transpose_pad(x, pad, precision, round_tf32=True):
    """(B, C, L) fp32 -> channels-last [B][L + 2 pad][C'] operand format with reflected halo rows."""
    lib = _lib.load()
    _require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 3
    B, C, L = x.shape
    out = alloc_act(B, L + 2 * pad, C, precision, x.device)
    with PROFILER.span("transpose_pad", bytes=float(x.numel() * 4 + out.numel() * out.element_size())):
        _lib.check(lib.avc_transpose_pad(x.data_ptr(), out.data_ptr(), B, C, L, pad, _dt(precision),
                                         1 if round_tf32 else 0, _stream()), "avc_transpose_pad")
    return out


def conv_to_mono_tanh(x, w, bias, lengths=None):
    """x [B][L][C] fp32, w [K][C] fp32 -> tanh(conv) [B][L] with reflect padding K//2.  lengths (device int32 [B],
    K // 2 < lengths[b] <= L): utterance b reflects at its own last sample, its samples past it are 0."""
    lib = _lib.load()
    _require_cuda(x, w)
    assert x.dtype == torch.float32 and x.is_contiguous() and w.dtype == torch.float32 and w.is_contiguous()
    B, L, C = x.shape
    K = w.shape[0]
    lens = _check_lengths(lengths, B) if lengths is not None else None
    out = torch.empty(B, L, dtype=torch.float32, device=x.device)
    with PROFILER.span("mono_conv", bytes=float(x.numel() * 4 + out.numel() * 4), flops=2.0 * K * C * B * L):
        _lib.check(lib.avc_conv_to_mono_tanh(x.data_ptr(), w.data_ptr(), float(bias), out.data_ptr(), B, L, C, K,
                                             _stream(), lens), "avc_conv_to_mono_tanh")
    return out


class Resblock:
    """One MelGAN ResnetBlock bound to the fused kernel avc_resblock (split-bf16 precision, C = 32 / 64).

    ``w``/``bias3``/``bias1`` come from ``packing.pack_resblock``."""

    def __init__(self, w, bias3, bias1, dilation, tag="melgan_res"):
        self.w, self.bias3, self.bias1 = w, bias3, bias1
        self.C = w.shape[1] // 2
        self.dilation = dilation
        self.tag = tag

    @staticmethod
    def eligible(C, L, precision):
        return precision == "fp32" and C in packing.RESBLOCK_CHANNELS and L % 128 == 0

    def to(self, device):
        self.w, self.bias3, self.bias1 = self.w.to(device), self.bias3.to(device), self.bias1.to(device)
        return self

    def __call__(self, xa, x, B, L, out=None, out_row0=0, reflect=0, out_raw=None, out2=None):
        """xa [B][L + 2d][2C] LeakyReLU(x) with reflected halo rows, x [B][L][2C] (split bf16).
        out: LeakyReLU(y) [B][rows][2C] at rows out_row0 + t (+ `reflect` mirrored halo rows); out_raw: y [B][L][2C];
        out2: LeakyReLU(y) as exact fp32 [B*L][C]."""
        lib = _lib.load()
        C, d = self.C, self.dilation
        _require_cuda(self.w, xa, x)
        for a, rows in ((xa, L + 2 * d), (x, L)):
            assert a.dtype == torch.bfloat16 and a.dim() == 3 and a.shape == (B, rows, 2 * C), (a.shape, (B, rows, 2 * C))
            assert a.stride(2) == 1 and a.stride(0) == rows * a.stride(1)
        desc = _lib.ResblockDesc()
        desc.xa, desc.xa_ld = xa.data_ptr(), xa.stride(1)
        desc.x, desc.x_ld = x.data_ptr(), x.stride(1)
        desc.w, desc.bias3, desc.bias1 = self.w.data_ptr(), self.bias3.data_ptr(), self.bias1.data_ptr()
        desc.B, desc.L, desc.C, desc.dilation = B, L, C, d
        if out is not None:
            assert out.is_cuda and out.dtype == torch.bfloat16 and out.dim() == 3 and out.shape[0] == B
            assert out.shape[2] == 2 * C and out.stride(2) == 1 and out.stride(0) == out.shape[1] * out.stride(1)
            desc.out, desc.out_ld = out.data_ptr(), out.stride(1)
            desc.out_rows_per_utt, desc.out_row0, desc.out_reflect = out.shape[1], out_row0, reflect
        if out_raw is not None:
            assert out_raw.is_cuda and out_raw.dtype == torch.bfloat16 and out_raw.shape == (B, L, 2 * C)
            assert out_raw.is_contiguous()
            desc.out_raw, desc.out_raw_ld = out_raw.data_ptr(), out_raw.stride(1)
        if out2 is not None:
            assert out2.is_cuda and out2.dtype == torch.float32 and out2.shape == (B * L, C) and out2.is_contiguous()
            desc.out2, desc.out2_ld = out2.data_ptr(), out2.stride(0)
        with PROFILER.span(self.tag, flops=2.0 * 5 * C * C * B * L):
            _lib.check(lib.avc_resblock(ctypes.byref(desc), _stream()), "avc_resblock")
        return out if out is not None else (out2 if out2 is not None else out_raw)


class Resblock2:
    """One MelGAN ResnetBlock bound to avc_resblock2 ("fp16s" precision, C = 32 / 64): reads only the raw residual
    stream (two fp16 terms, halo rows included) and writes one tensor.  ``w``/``bias3``/``bias1`` from
    ``packing.pack_resblock2``."""

    def __init__(self, w, bias3, bias1, dilation, tag="melgan_res"):
        self.w, self.bias3, self.bias1 = w, bias3, bias1
        self.C = bias3.numel()
        self.dilation = dilation
        self.tag = tag

    @staticmethod
    def eligible(C, L):
        return C in packing.RESBLOCK2_CHANNELS and L % 128 == 0

    def to(self, device):
        self.w, self.bias3, self.bias1 = self.w.to(device), self.bias3.to(device), self.bias1.to(device)
        return self

    def __call__(self, x, B, L, y=None, y_row0=0, y_reflect=0, y_act=False, out2=None, wav=None, mono=None,
                 lengths=None):
        """x [B][L + 2d][2C] fp16 two-term residual stream with reflected halo rows (time t at row t + d).
        y: raw output (y_act False) or LeakyReLU(output) (True) as two fp16 terms [B][rows][2C] at rows y_row0 + t
        (+ `y_reflect` mirrored halo rows); out2: LeakyReLU(output) as exact fp32 [B*L][C]; wav [B][L] fp32 with
        mono = (w [K][C] fp32, bias): the generator's output layer applied in the block's epilogue (C = 32).
        Exactly one of y / out2 / wav.
        lengths (RaggedRows of this stage): a padded batch -- only the tiles holding a valid row run, wav reflects at
        each utterance's end and is 0 past it in its last tile; the right halo of y at each utterance's end is the
        caller's (reflect_halo with lengths), and so is zero-filling wav."""
        lib = _lib.load()
        C, d = self.C, self.dilation
        _require_cuda(self.w, x)
        assert x.dtype == torch.float16 and x.dim() == 3 and x.shape == (B, L + 2 * d, 2 * C), (x.shape, (B, L + 2 * d, 2 * C))
        assert x.stride(2) == 1 and x.stride(0) == x.shape[1] * x.stride(1)
        assert (y is not None) + (out2 is not None) + (wav is not None) == 1
        desc = _lib.Resblock2Desc()
        desc.x, desc.x_ld = x.data_ptr(), x.stride(1)
        desc.w, desc.bias3, desc.bias1 = self.w.data_ptr(), self.bias3.data_ptr(), self.bias1.data_ptr()
        desc.B, desc.L, desc.C, desc.dilation = B, L, C, d
        if y is not None:
            assert y.is_cuda and y.dtype == torch.float16 and y.dim() == 3 and y.shape[0] == B and y.shape[2] == 2 * C
            assert y.stride(2) == 1 and y.stride(0) == y.shape[1] * y.stride(1)
            desc.y, desc.y_ld = y.data_ptr(), y.stride(1)
            desc.y_rows_per_utt, desc.y_row0, desc.y_reflect, desc.y_act = y.shape[1], y_row0, y_reflect, 1 if y_act else 0
        elif out2 is not None:
            assert out2.is_cuda and out2.dtype == torch.float32 and out2.shape == (B * L, C) and out2.is_contiguous()
            desc.out2, desc.out2_ld = out2.data_ptr(), out2.stride(0)
        else:
            w_out, b_out = mono
            _require_cuda(wav, w_out)
            assert wav.dtype == torch.float32 and wav.shape == (B, L) and wav.is_contiguous()
            assert w_out.dtype == torch.float32 and w_out.is_contiguous() and w_out.shape[1] == C and w_out.shape[0] in (3, 5, 7)
            desc.wav, desc.mono_w, desc.mono_bias, desc.mono_taps = wav.data_ptr(), w_out.data_ptr(), float(b_out), w_out.shape[0]
        rows = B * L
        if lengths is not None:
            assert isinstance(lengths, RaggedRows) and len(lengths.host) == B and max(lengths.host) <= L
            stride = 128 - (mono[0].shape[0] - 1) if wav is not None else 128
            tile_start, n_tiles = lengths.tiles[stride]
            desc.lengths, desc.tile_start, desc.n_tiles = _check_lengths(lengths.rows, B), tile_start.data_ptr(), n_tiles
            rows = sum(lengths.host)
        dbg = getattr(self, "debug_clk", None)
        if dbg is not None:
            desc.debug_clk = dbg.data_ptr()
        extra = 2.0 * mono[0].numel() * rows if wav is not None else 0.0
        with PROFILER.span(self.tag, flops=2.0 * 5 * C * C * rows + extra,
                           bytes=float(x.numel() * 2 * rows / (B * L) + (rows * 4 if wav is not None else rows * C * 4))):
            _lib.check(lib.avc_resblock2(ctypes.byref(desc), _stream()), "avc_resblock2")
        return y if y is not None else (out2 if out2 is not None else wav)


# ------------------------------------------------------------------------------------------------ Meta glue
def _ptr(t):
    return t.data_ptr() if t is not None else None


def gn_stats(x, B, eps=1e-5):
    """x fp32, B samples of equal size -> [B][2] (mean, rstd) of GroupNorm(1, C)."""
    lib = _lib.load()
    _require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    n = x.numel() // B
    stats = torch.empty(B, 2, dtype=torch.float32, device=x.device)
    with PROFILER.span("gn_stats", bytes=4.0 * x.numel()):
        _lib.check(lib.avc_gn_stats(x.data_ptr(), stats.data_ptr(), B, n, eps, _stream()), "avc_gn_stats")
    return stats


def gn_pool_residual(x, stats, gamma, precision, want_f32=True, want_op=True):
    """x [B][L][C] fp32 -> (x1 fp32, x1 operand format), x1 = x + pool3(GN(x)) - GN(x)."""
    lib = _lib.load()
    _require_cuda(x)
    B, L, C = x.shape
    out_f32 = torch.empty_like(x) if want_f32 else None
    out_op = alloc_act(B, L, C, precision, x.device) if want_op else None
    with PROFILER.span("gn_pool", bytes=4.0 * x.numel() * 2):
        _lib.check(lib.avc_gn_pool_residual(x.data_ptr(), stats.data_ptr(), gamma.data_ptr(), _ptr(out_f32),
                                            _ptr(out_op), _dt(precision), 1, B, L, C, _stream()),
                   "avc_gn_pool_residual")
    return out_f32, out_op


def gn_apply(x, stats, gamma, beta, precision):
    lib = _lib.load()
    _require_cuda(x)
    B, L, C = x.shape
    out = alloc_act(B, L, C, precision, x.device)
    with PROFILER.span("gn_apply", bytes=4.0 * x.numel() * 2):
        _lib.check(lib.avc_gn_apply(x.data_ptr(), stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(),
                                    _dt(precision), 1, B, L, C, _stream()), "avc_gn_apply")
    return out


def patchify(a, stats, gamma, beta, p, precision):
    """a [B][S][S] fp32 channels-last -> tokens [B][(S/p)^2][p*p] operand format (after GroupNorm if stats given)."""
    lib = _lib.load()
    _require_cuda(a)
    B, S, S2 = a.shape
    assert S == S2 and a.is_contiguous() and a.dtype == torch.float32
    out = alloc_act(B, (S // p) ** 2, p * p, precision, a.device)
    with PROFILER.span("patchify", bytes=4.0 * a.numel() * 2):
        _lib.check(lib.avc_patchify(a.data_ptr(), _ptr(stats), _ptr(gamma), _ptr(beta), out.data_ptr(), _dt(precision),
                                    1, B, S, p, _stream()), "avc_patchify")
    return out


def ln_transpose(x, gamma, beta, ln_axis, precision, want_op=True, want_f32=False):
    """x [B][R][C] fp32 -> (out_op [B][C][R8] operand format, out_f32 [B][C][R8] raw), R8 = R rounded up to 8
    (pad columns are zero).  ln_axis 0 none / 1 per row over C / 2 per column over R."""
    lib = _lib.load()
    _require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    B, R, C = x.shape
    r8 = (R + 7) // 8 * 8
    out_op = alloc_act(B, C, r8, precision, x.device) if want_op else None
    out_f32 = torch.empty(B, C, r8, dtype=torch.float32, device=x.device) if want_f32 else None
    scratch = torch.empty(2 * B * max(R, C), dtype=torch.float32, device=x.device) if ln_axis else None
    with PROFILER.span("ln_transpose", bytes=4.0 * x.numel() * 2):
        _lib.check(lib.avc_ln_transpose(x.data_ptr(), _ptr(gamma), _ptr(beta), ln_axis, _ptr(out_op), _dt(precision), 1,
                                        _ptr(out_f32), _ptr(scratch), B, R, C, _stream()), "avc_ln_transpose")
    return out_op, out_f32


def meta_decoder_input(codes, c_trg, T, freq, precision):
    """codes [B][T/freq][2H] fp32, c_trg [B][E] -> [B][2H+E][T] operand format (channels = time)."""
    lib = _lib.load()
    _require_cuda(codes, c_trg)
    B, _, H2 = codes.shape
    E = c_trg.shape[1]
    out = alloc_act(B, H2 + E, T, precision, codes.device)
    with PROFILER.span("concat", bytes=float(out.numel() * out.element_size())):
        _lib.check(lib.avc_meta_decoder_input(codes.data_ptr(), c_trg.data_ptr(), out.data_ptr(), _dt(precision), 1, B,
                                              T, freq, H2, E, _stream()), "avc_meta_decoder_input")
    return out


def gather_codes(out, H, freq):
    """out [B][T][2H] fp32 -> codes [B][T/freq][2H]: [out[jF+F-1, :H] || out[jF, H:]]."""
    lib = _lib.load()
    _require_cuda(out)
    B, T, _ = out.shape
    codes = torch.empty(B, T // freq, 2 * H, dtype=torch.float32, device=out.device)
    _lib.check(lib.avc_gather_codes(out.data_ptr(), codes.data_ptr(), B, T, H, freq, _stream()), "avc_gather_codes")
    return codes


# ------------------------------------------------------------------------------------------------ AdaIN "2" variants
def global_stats(x, out=None):
    """x fp32 (any shape) -> out [2] = (x.mean(), x.std()) over ALL elements, torch defaults (Bessel-corrected std)."""
    lib = _lib.load()
    _require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.numel() % 4 == 0
    if out is None:
        out = torch.empty(2, dtype=torch.float32, device=x.device)
    scratch = torch.empty(512, dtype=torch.float64, device=x.device)
    with PROFILER.span("global_stats", bytes=4.0 * x.numel(), launches=2):
        _lib.check(lib.avc_global_stats(x.data_ptr(), x.numel(), out.data_ptr(), scratch.data_ptr(), _stream()),
                   "avc_global_stats")
    return out


def adain(x, x_stats, t_stats, precision, want_f32=False):
    """x [B][T][C] fp32 -> ((x - x_stats[0]) / x_stats[1] * t_stats[1] + t_stats[0]) in operand format (+ fp32 copy)."""
    lib = _lib.load()
    _require_cuda(x, x_stats, t_stats)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 3
    assert x_stats.dtype == torch.float32 and t_stats.dtype == torch.float32 and x_stats.numel() == 2 and t_stats.numel() == 2
    B, T, C = x.shape
    out_op = alloc_act(B, T, C, precision, x.device)
    out_f32 = torch.empty_like(x) if want_f32 else None
    with PROFILER.span("adain", bytes=4.0 * x.numel() * 2):
        _lib.check(lib.avc_adain(x.data_ptr(), x_stats.data_ptr(), t_stats.data_ptr(), _ptr(out_f32), out_op.data_ptr(),
                                 _dt(precision), 1, B * T, C, _stream()), "avc_adain")
    return out_op, out_f32


def segment_stats(x, lengths=None, out=None):
    """x [B][T][C] fp32 -> out [B][2] = (mean, std) of each utterance over its rows 0 .. lengths[b]-1 (all T rows
    without lengths), torch defaults (Bessel-corrected std); the bits of row b depend only on utterance b's valid rows."""
    lib = _lib.load()
    _require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 3
    B, T, C = x.shape
    lens = _check_lengths(lengths, B) if lengths is not None else None
    if out is None:
        out = torch.empty(B, 2, dtype=torch.float32, device=x.device)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == 2 * B
    # per call from the stream-ordered caching allocator: two batches on two streams never share it
    chunks = -(-T * C // _lib.SEGMENT_CHUNK)
    scratch = torch.empty(2 * B * chunks, dtype=torch.float64, device=x.device)
    with PROFILER.span("segment_stats", bytes=4.0 * x.numel(), launches=2):
        _lib.check(lib.avc_segment_stats(x.data_ptr(), B, T, C, lens, out.data_ptr(), scratch.data_ptr(), _stream()),
                   "avc_segment_stats")
    return out


def adain_segmented(x, x_stats, t_stats, precision, lengths=None, want_f32=False):
    """x [B][T][C] fp32 -> AdaIN with utterance b's statistics x_stats[b] (x_stats [B][2]) and the style t_stats ([2]:
    one for every utterance, or [B][2]: one per utterance), in operand format (+ fp32 copy); with lengths, the rows past
    each utterance's end are 0 in both outputs."""
    lib = _lib.load()
    _require_cuda(x, x_stats, t_stats)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 3
    B, T, C = x.shape
    assert x_stats.dtype == torch.float32 and x_stats.is_contiguous() and x_stats.numel() == 2 * B
    assert t_stats.dtype == torch.float32 and t_stats.is_contiguous() and t_stats.numel() in (2, 2 * B)
    t_stride = 0 if t_stats.dim() == 1 else 2
    assert t_stats.shape == ((2,) if t_stride == 0 else (B, 2)), t_stats.shape
    lens = _check_lengths(lengths, B) if lengths is not None else None
    out_op = alloc_act(B, T, C, precision, x.device)
    out_f32 = torch.empty_like(x) if want_f32 else None
    with PROFILER.span("adain", bytes=4.0 * x.numel() * 2):
        _lib.check(lib.avc_adain_segmented(x.data_ptr(), x_stats.data_ptr(), t_stats.data_ptr(), t_stride, lens,
                                           _ptr(out_f32), out_op.data_ptr(), _dt(precision), 1, B, T, C, _stream()),
                   "avc_adain_segmented")
    return out_op, out_f32


# ------------------------------------------------------------------------------------------------ batch-statistics BatchNorm
def bn_batch_stats(v, gamma, beta, eps=1e-5, momentum=0.1, running_mean=None, running_var=None,
                   num_batches_tracked=None, scale_shift=None):
    """v [rows][C] fp32 (row stride >= C) -> scale_shift [2][C] fp32 = (gamma / sqrt(var + eps), beta - mean * scale)
    with the statistics of all rows, as nn.BatchNorm1d in training mode; updates the running buffers in place on the
    device (momentum None: cumulative average).  Raises ValueError, as torch does, for a single row."""
    lib = _lib.load()
    _require_cuda(v, gamma, beta, running_mean, running_var, num_batches_tracked)
    assert v.dtype == torch.float32 and v.dim() == 2 and v.stride(1) == 1
    rows, C = v.shape
    if rows <= 1:
        raise ValueError(f"Expected more than 1 value per channel when training, got input size {(rows, C)}")
    for t in (gamma, beta, running_mean, running_var):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == C)
    assert (running_mean is None) == (running_var is None)
    if num_batches_tracked is not None:
        assert num_batches_tracked.dtype == torch.int64 and num_batches_tracked.numel() == 1
    if momentum is None and (num_batches_tracked is None or running_mean is None):
        raise ValueError("momentum=None (cumulative average) needs the running buffers and num_batches_tracked")
    if scale_shift is None:
        scale_shift = torch.empty(2, C, dtype=torch.float32, device=v.device)
    assert scale_shift.dtype == torch.float32 and scale_shift.is_contiguous() and scale_shift.shape == (2, C)
    # from the stream-ordered caching allocator, so layers run on two streams never share it
    scratch = torch.empty(2 + 2 * _lib.BN_MAX_PARTS * C, dtype=torch.float64, device=v.device)
    with PROFILER.span("bn_stats", bytes=4.0 * rows * C, launches=2):
        _lib.check(lib.avc_bn_batch_stats(v.data_ptr(), rows, C, v.stride(0), gamma.data_ptr(), beta.data_ptr(),
                                          float(eps), 0.0 if momentum is None else float(momentum),
                                          1 if momentum is None else 0, _ptr(running_mean), _ptr(running_var),
                                          _ptr(num_batches_tracked), scale_shift.data_ptr(), scratch.data_ptr(),
                                          _stream()), "avc_bn_batch_stats")
    return scale_shift


def bn_apply(v, scale_shift, B, T, act="none", out=None, out2=None, residual=None, res_after=False, out_fmt=None,
             round_tf32=True):
    """act(scale * v + shift) (+ residual before or after the activation) for v [B*T][C] fp32 -> out [B][rows][C']
    (operand format `out_fmt`, written at rows 0..T-1) and / or out2 [B*T][C] exact fp32."""
    lib = _lib.load()
    _require_cuda(v, scale_shift, out, out2, residual)
    assert v.dtype == torch.float32 and v.dim() == 2 and v.stride(1) == 1 and v.shape[0] == B * T
    C = v.shape[1]
    assert scale_shift.dtype == torch.float32 and scale_shift.is_contiguous() and scale_shift.shape == (2, C)
    assert out is not None or out2 is not None
    d = _lib.BnApplyDesc()
    d.v, d.v_ld, d.scale_shift = v.data_ptr(), v.stride(0), scale_shift.data_ptr()
    d.B, d.T, d.C = B, T, C
    d.act = _lib.ACTS[act]
    nbytes = 4.0 * B * T * C
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.stride(-1) == 1 and residual.shape[-1] >= C
        d.residual, d.res_ld, d.res_after_act = residual.data_ptr(), residual.stride(-2), 1 if res_after else 0
        nbytes += 4.0 * B * T * C
    if out is not None:
        fmt = out_fmt
        assert fmt is not None, "bn_apply: out needs its operand format (a precision name)"
        assert out.dim() == 3 and out.shape[0] == B and out.shape[1] >= T and out.stride(2) == 1
        assert out.dtype == TORCH_DTYPE[fmt] and out.shape[2] >= packing.act_channels(C, fmt)
        assert out.stride(0) == out.shape[1] * out.stride(1)
        d.out, d.out_ld, d.out_rows_per_utt, d.out_row0 = out.data_ptr(), out.stride(1), out.shape[1], 0
        d.out_dtype = _dt(fmt)
        d.out_round_tf32 = 1 if (round_tf32 and out.dtype == torch.float32) else 0
        nbytes += B * T * packing.act_channels(C, fmt) * out.element_size()
    if out2 is not None:
        assert out2.dtype == torch.float32 and out2.dim() == 2 and out2.stride(1) == 1 and out2.shape[0] == B * T
        assert out2.shape[1] >= C
        d.out2, d.out2_ld = out2.data_ptr(), out2.stride(0)
        nbytes += 4.0 * B * T * C
    with PROFILER.span("bn_apply", bytes=nbytes):
        _lib.check(lib.avc_bn_apply(ctypes.byref(d), _stream()), "avc_bn_apply")
    return out if out is not None else out2


# ------------------------------------------------------------------------------------------------ Audio2Mel front end
def audio_frames(audio, pad, hop, rows, precision):
    """audio [B][L] fp32 -> reflect-padded signal as rows of `hop` samples [B][rows][hop] in operand format."""
    lib = _lib.load()
    _require_cuda(audio)
    assert audio.dtype == torch.float32 and audio.is_contiguous() and audio.dim() == 2
    B, L = audio.shape
    out = alloc_act(B, rows, hop, precision, audio.device)
    with PROFILER.span("audio_frames", bytes=float(audio.numel() * 4 + out.numel() * out.element_size())):
        _lib.check(lib.avc_audio_frames(audio.data_ptr(), out.data_ptr(), B, L, pad, hop, rows, _dt(precision), 1,
                                        _stream()), "avc_audio_frames")
    return out


def complex_mag(spec, bins, bins_pad, precision):
    """spec [rows][2*bins] fp32 (re | im) -> |spec| [rows][bins_pad] in operand format (zero padding channels)."""
    lib = _lib.load()
    _require_cuda(spec)
    assert spec.dtype == torch.float32 and spec.is_contiguous() and spec.dim() == 2 and spec.shape[1] == 2 * bins
    rows = spec.shape[0]
    out = alloc_act(1, rows, bins_pad, precision, spec.device)
    with PROFILER.span("complex_mag", bytes=float(spec.numel() * 4 + out.numel() * out.element_size())):
        _lib.check(lib.avc_complex_mag(spec.data_ptr(), out.data_ptr(), rows, bins, bins_pad, _dt(precision), 1,
                                       _stream()), "avc_complex_mag")
    return out
