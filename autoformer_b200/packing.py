"""Host-side weight folding / re-packing for the sm_100a kernels.  Pure tensor code: runs on CPU or GPU.

Everything here happens once per ``load_state_dict`` (not per forward):
  * BatchNorm (eval) folded into the preceding conv: scale into the weights, shift into the bias
    (factory/AutoVC.py:26-39 + nn.BatchNorm1d running statistics, SURVEY.md Appendix D)
  * conv weights (C_out, C_in, K) -> K-major GEMM operand [n_pad][taps * chunks * kc], tap-major, each tap's
    channels zero-padded to a whole number of 128-byte k-blocks (kc = 32 TF32 / 64 bf16 channels)
  * LSTM gate rows interleaved in groups of G hidden units so one accumulator tile holds i,f,g,o of G units
  * weight norm folded (melgan/modules.py:18-23)
  * fp32 operands rounded to TF32 (round-to-nearest, ties away) so the tensor core's truncation is exact
"""
import torch

# precision modes: "tf32" (fp32 storage, one TF32 pass), "bf16" (one bf16 pass),
# "fp32" (split bf16: hi + lo channels, three bf16 products per fp32 product -- fp32-grade accuracy),
# "fp16x2" (fp16 activations, every weight as two fp16 terms w_hi + w_lo: two fp16 products per fp32 product; the
# only rounding is the 2^-12 of the activations -- ~3e-4 end to end on AutoVC, scripts/precision_study.py)
# "fp16s" (MelGAN, round 2): the split format with fp16 terms -- activations AND weights as two fp16 values hi + lo
# (~2^-22), three products per fp32 product like "fp32" -- used for the tensors whose rounding the vocoder's output is
# sensitive to (the residual stream, the ConvTranspose operands, the ResnetBlock intermediate), while the dilated k3
# convolutions read ONE fp16 value per activation ("fp16x2" products).  scripts/melgan_precision_study.py.
KC = {"tf32": 32, "bf16": 64, "fp32": 64, "fp16x2": 64, "f16": 64, "fp16s": 64}      # "f16": single fp16 operand (internal)
TORCH_DTYPE = {"tf32": torch.float32, "bf16": torch.bfloat16, "fp32": torch.bfloat16, "fp16x2": torch.float16,
               "f16": torch.float16, "fp16s": torch.float16}
TWO_TERM_WEIGHTS = ("fp32", "fp16x2")     # precisions whose packed LSTM weights are [w_hi | w_lo]
PRECISIONS = ("tf32", "bf16", "fp32", "fp16x2")
SPLIT_ACTS = ("fp32", "fp16s")            # activation buffers hold [hi | lo] halves (2C channels)
FP16_MAX = 65504.0


def act_channels(c: int, precision: str) -> int:
    """Channels of the activation buffer that carries c logical channels."""
    return 2 * c if precision in SPLIT_ACTS else c


def split_bf16(t: torch.Tensor):
    """v -> (hi, lo) with hi = bf16(v), lo = bf16(v - hi): v ~ hi + lo to ~2^-17 relative."""
    t = t.float()
    hi = t.to(torch.bfloat16)
    lo = (t - hi.float()).to(torch.bfloat16)
    return hi, lo


def split_f16(t: torch.Tensor):
    """v -> (hi, lo) fp16 with v ~ hi + lo to ~2^-22 relative (|v| well inside the fp16 range: weights)."""
    t = t.float()
    hi = t.to(torch.float16)
    lo = (t - hi.float()).to(torch.float16)
    return hi, lo


def split_terms(t: torch.Tensor, precision: str):
    return split_bf16(t) if precision == "fp32" else split_f16(t)


def sat_f16(t: torch.Tensor) -> torch.Tensor:
    return t.float().clamp(-FP16_MAX, FP16_MAX)


def to_act(t: torch.Tensor, precision: str) -> torch.Tensor:
    """fp32 channels-last activation -> the buffer format of `precision` (tests / host-side staging)."""
    if precision == "tf32":
        return round_tf32(t.float())
    if precision == "bf16":
        return t.to(torch.bfloat16)
    if precision in ("fp16x2", "f16"):
        return sat_f16(t).to(torch.float16)       # saturating like the kernels' fp16 stores (cvt.rn.satfinite)
    hi, lo = split_f16(sat_f16(t)) if precision == "fp16s" else split_bf16(t)
    return torch.cat([hi, lo], dim=-1).contiguous()


def act_to_float(buf: torch.Tensor, precision: str) -> torch.Tensor:
    if precision in SPLIT_ACTS:
        c = buf.shape[-1] // 2
        return buf[..., :c].float() + buf[..., c:].float()
    return buf.float()


def fp16_overflow_margin(taps) -> float:
    """fp16 range / largest |activation| over a model's stage taps (``model.collect_taps = True``).  The kernels'
    fp16 stores SATURATE at +-65504 (csrc/avc_ptx.cuh: sat_f16) so an out-of-range activation costs accuracy instead
    of poisoning the utterance with inf / NaN -- which also makes it silent.  A margin <= 1 means some activation
    reached the limit: the "fp16x2" precision is not valid for that checkpoint, use "fp32" (split bf16, fp32 range).
    Trained checkpoints should be probed once with this before serving in fp16x2."""
    peak = 0.0
    for v in taps.values():
        if torch.is_tensor(v) and v.numel():
            peak = max(peak, float(v.detach().abs().max()))
    return float("inf") if peak == 0.0 else FP16_MAX / peak


def round_tf32(t: torch.Tensor) -> torch.Tensor:
    """cvt.rna.tf32.f32 on the host: keep 10 mantissa bits, round to nearest, ties away from zero."""
    assert t.dtype == torch.float32
    i = t.contiguous().view(torch.int32)
    i = (i + 0x1000) & ~0x1FFF
    return i.view(torch.float32)


def to_operand(t: torch.Tensor, precision: str) -> torch.Tensor:
    """Weights / activations as the tensor core reads them (for "fp32" use split_bf16 / to_act instead)."""
    if precision == "tf32":
        return round_tf32(t.float())
    if precision == "bf16":
        return t.to(torch.bfloat16)
    if precision == "f16":
        return t.to(torch.float16)
    raise ValueError("two-term precisions have no single-tensor operand form")


def _ceil_to(x, m):
    return (x + m - 1) // m * m


def choose_block_n(n: int) -> int:
    """Output-channel tile: 256 when the layer is wide enough, otherwise the smallest tile that covers n."""
    if n >= 256:
        return 256
    if n > 64:
        return 128
    return 64


def fold_bn(weight, bias, bn_weight, bn_bias, running_mean, running_var, eps=1e-5):
    """conv + BatchNorm(eval) -> conv:  w' = s w,  b' = beta + s (b - mean),  s = gamma / sqrt(var + eps)."""
    s = bn_weight.double() / torch.sqrt(running_var.double() + eps)
    w = weight.double() * s.view(-1, *([1] * (weight.dim() - 1)))
    b = bn_bias.double() + s * (bias.double() - running_mean.double())
    return w.float(), b.float()


def pack_conv_sources(weights, bias, precision, block_n=None):
    """weights: list of (C_out, C_in_s, K_s) tensors, one per K-concatenated activation source.

    Returns (W [n_pad][k_pad] operand dtype, bias [n_pad] fp32, meta dict)."""
    kc = KC[precision]
    n = weights[0].shape[0]
    if precision in SPLIT_ACTS:
        # a*w ~ a_hi*w_hi + a_lo*w_hi + a_hi*w_lo: each logical source becomes two physical ones over the same
        # buffer: [a_hi|a_lo] x [w_hi|w_hi] (2C channels) and a_hi x w_lo (the first C channels)
        assert len(weights) <= 2, "at most two logical sources in split precision (four physical sources)"
        phys = []
        for w in weights:
            hi, lo = split_terms(w, precision)
            phys += [torch.cat([hi, hi], dim=1).float(), lo.float()]
        w_p, b_p, meta = pack_conv_sources(phys, bias, "bf16" if precision == "fp32" else "f16", block_n)
        meta.update(precision=precision, split=True, logical_channels=[w.shape[1] for w in weights],
                    logical_taps=[w.shape[2] for w in weights])
        return w_p, b_p, meta
    if precision == "fp16x2":
        # a*w = a*w_hi + a*w_lo: each logical source becomes two physical ones over the SAME channels
        assert len(weights) <= 2, "at most two logical sources (four physical sources)"
        phys = []
        for w in weights:
            hi, lo = split_f16(w)
            phys += [hi.float(), lo.float()]
        w_p, b_p, meta = pack_conv_sources(phys, bias, "f16", block_n)
        meta.update(precision="fp16x2", dup=True, logical_channels=[w.shape[1] for w in weights],
                    logical_taps=[w.shape[2] for w in weights])
        return w_p, b_p, meta
    bn_tile = block_n or choose_block_n(n)
    n_pad = _ceil_to(n, bn_tile)
    cols = []
    taps, chans = [], []
    for w in weights:
        assert w.dim() == 3 and w.shape[0] == n
        c_in, k = w.shape[1], w.shape[2]
        chunks = (c_in + kc - 1) // kc
        wp = torch.zeros(n, k, chunks * kc, dtype=torch.float32, device=w.device)
        wp[:, :, :c_in] = w.float().permute(0, 2, 1)
        cols.append(wp.reshape(n, k * chunks * kc))
        taps.append(k)
        chans.append(c_in)
    wk = torch.cat(cols, dim=1)
    k_pad = wk.shape[1]
    wfull = torch.zeros(n_pad, k_pad, dtype=torch.float32, device=wk.device)
    wfull[:n] = wk
    bfull = torch.zeros(n_pad, dtype=torch.float32, device=wk.device)
    bfull[:n] = bias.float()
    meta = dict(N=n, n_pad=n_pad, k_pad=k_pad, block_n=bn_tile, taps=taps, channels=chans, precision=precision)
    return to_operand(wfull, precision).contiguous(), bfull.contiguous(), meta


def pack_conv(weight, bias, precision, block_n=None):
    return pack_conv_sources([weight], bias, precision, block_n)


def pack_linear(weight, bias, precision, block_n=None):
    """nn.Linear (N, K) as a 1-tap convolution."""
    return pack_conv_sources([weight.unsqueeze(-1)], bias, precision, block_n)


RESBLOCK_CHANNELS = (32, 64)      # widths the fused ResnetBlock kernel (avc_resblock) is built for
RESBLOCK2_CHANNELS = (32, 64, 128)   # ... and its "fp16s" successor avc_resblock2 (128: CTA pairs, streamed weights)


def pack_resblock(w3, b3, w1, b1, wsc, bsc):
    """Weights of one MelGAN ResnetBlock (melgan/modules.py:72-85, weight norm already folded) for avc_resblock.

    w3 (C, C, 3) dilated conv, w1 / wsc (C, C, 1) block.4 / shortcut.  Returns (W [5][2C][64] bf16, bias3 [C], bias1 [C])
    with tiles W3 tap 0..2, W1, Wsc in the split-bf16 tile layouts of include/avc_b200.h:
      C = 64: rows [w_hi (64) ; w_lo (64)];   C = 32: rows [[w_hi | w_hi] (32) ; [w_lo | 0] (32)]."""
    c = w3.shape[0]
    assert c in RESBLOCK_CHANNELS and w3.shape == (c, c, 3) and w1.shape == (c, c, 1) and wsc.shape == (c, c, 1)
    mats = [w3[:, :, 0], w3[:, :, 1], w3[:, :, 2], w1[:, :, 0], wsc[:, :, 0]]
    tiles = []
    for m in mats:
        hi, lo = split_bf16(m)
        if c == 64:
            tiles.append(torch.cat([hi, lo], dim=0))
        else:
            tiles.append(torch.cat([torch.cat([hi, hi], dim=1), torch.cat([lo, torch.zeros_like(lo)], dim=1)], dim=0))
    w = torch.stack(tiles).contiguous()
    assert w.shape == (5, 2 * c, 64) and w.dtype == torch.bfloat16
    return w, b3.float().contiguous(), (b1.float() + bsc.float()).contiguous()


def pack_resblock2(w3, b3, w1, b1, wsc, bsc):
    """Weights of one MelGAN ResnetBlock for avc_resblock2 ("fp16s" precision: every weight as two fp16 terms).

    Returns (W [rows][64] fp16, bias3 [C], bias1 [C]); tiles in order W3 tap 0..2, W1 (block.4), Wsc (shortcut):
      C = 64: every tile rows [w_hi (64) ; w_lo (64)]
      C = 32: W3 tiles rows [w_hi | w_lo] (32 rows: the k3 operand rows are [xa | xa]);
              W1 / Wsc tiles rows [[w_hi | w_hi] (32) ; [w_lo | 0] (32)] (operand rows [a_hi | a_lo])."""
    c = w3.shape[0]
    assert c in RESBLOCK2_CHANNELS and w3.shape == (c, c, 3) and w1.shape == (c, c, 1) and wsc.shape == (c, c, 1)
    if c == 128:
        # CTA pairs, weights streamed: [matrix (W3 tap 0..2, W1, Wsc)][64-channel k-chunk][256 rows][64]; the 256 rows of a
        # tile are CTA 0's half then CTA 1's half, each [w_hi[64 r .. 64 r + 64) ; w_lo[64 r .. 64 r + 64)]
        tiles = []
        for m in (w3[:, :, 0], w3[:, :, 1], w3[:, :, 2], w1[:, :, 0], wsc[:, :, 0]):
            hi, lo = split_f16(m)
            for kc in range(c // 64):
                ks = slice(kc * 64, kc * 64 + 64)
                tiles.append(torch.cat([hi[0:64, ks], lo[0:64, ks], hi[64:128, ks], lo[64:128, ks]], dim=0))
        w = torch.cat(tiles, dim=0).contiguous()
        assert w.shape == (10 * 256, 64) and w.dtype == torch.float16
        return w, b3.float().contiguous(), (b1.float() + bsc.float()).contiguous()
    tiles = []
    for k in range(3):
        hi, lo = split_f16(w3[:, :, k])
        tiles.append(torch.cat([hi, lo], dim=0) if c == 64 else torch.cat([hi, lo], dim=1))
    for m in (w1[:, :, 0], wsc[:, :, 0]):
        hi, lo = split_f16(m)
        if c == 64:
            tiles.append(torch.cat([hi, lo], dim=0))
        else:
            tiles.append(torch.cat([torch.cat([hi, hi], dim=1), torch.cat([lo, torch.zeros_like(lo)], dim=1)], dim=0))
    w = torch.cat(tiles, dim=0).contiguous()
    assert w.shape == ((640 if c == 64 else 224), 64) and w.dtype == torch.float16
    return w, b3.float().contiguous(), (b1.float() + bsc.float()).contiguous()


WS_GROUP = "ws"     # gate packing of the weight-stationary small-batch recurrence (avc_lstm_seq_ws)


def gate_permutation(hidden: int, group, device=None) -> torch.Tensor:
    """index[p] = PyTorch gate row (g*H + u) stored at packed position p = (u//G)*4G + g*G + u%G; for
    group == WS_GROUP the four gates of a unit are adjacent: p = 128 (u//32) + 4 (u%32) + g."""
    p = torch.arange(4 * hidden, device=device)
    if group == WS_GROUP:
        assert hidden % 32 == 0
        return (p % 4) * hidden + (p // 128) * 32 + (p % 128) // 4
    assert hidden % group == 0
    blk = p // (4 * group)
    g = (p % (4 * group)) // group
    return g * hidden + blk * group + p % group


def pack_lstm_ih(w_ih, b_ih, b_hh, precision, group):
    """Input projection of one uni-directional layer with gate-interleaved output columns."""
    h = w_ih.shape[0] // 4
    perm = gate_permutation(h, group, w_ih.device)
    return pack_linear(w_ih[perm], (b_ih + b_hh)[perm], precision)


def pack_lstm_ih_fused(w_ih, b_ih, b_hh, precision, group):
    """W_ih for the recurrence kernel's fused input projection: gate-interleaved rows like W_hh, K zero-padded to whole
    k-blocks, [w_hi | w_lo] halves in split precision.  Returns (W [4H][Kp or 2Kp], bias [4H] fp32 = b_ih + b_hh)."""
    h, c_in = w_ih.shape[0] // 4, w_ih.shape[1]
    perm = gate_permutation(h, group, w_ih.device)
    kpad = _ceil_to(c_in, KC[precision])
    w = torch.zeros(perm.numel(), kpad, dtype=torch.float32, device=w_ih.device)
    w[:, :c_in] = w_ih.float()[perm]
    bias = (b_ih.float() + b_hh.float())[perm].contiguous()
    if precision in TWO_TERM_WEIGHTS:
        hi, lo = split_terms(w, precision)
        return torch.cat([hi, lo], dim=1).contiguous(), bias
    return to_operand(w, precision).contiguous(), bias


def pack_lstm_hh(w_hh, precision, group):
    h = w_hh.shape[1]
    perm = gate_permutation(h, group, w_hh.device)
    w = w_hh.float()[perm]
    if precision in TWO_TERM_WEIGHTS:
        hi, lo = split_terms(w, precision)
        # [w_hi | w_lo]; "fp32": the kernel forms a_hi*w_hi + a_lo*w_hi + a_hi*w_lo, "fp16x2": a*w_hi + a*w_lo
        return torch.cat([hi, lo], dim=1).contiguous()
    return to_operand(w, precision).contiguous()


def pack_lstm_stack(w_ih, w_hh, b_ih, b_hh, first):
    """One layer for the wavefront stack kernel (avc_lstm_stack_ws): W_hh (and, above the first layer, W_ih) as ONE fp16
    term, rows in the WS_GROUP gate order, plus the fp32 bias b_ih + b_hh in the same order.  The first layer's W_ih and
    bias go through the dense projection in front (pack_lstm_ih) and are None here."""
    h = w_hh.shape[1]
    perm = gate_permutation(h, WS_GROUP, w_hh.device)
    one = lambda w: sat_f16(w.float()[perm]).to(torch.float16).contiguous()
    if first:
        return None, one(w_hh), None
    assert w_ih.shape == (4 * h, h), "the layers above the first take the hidden sequence of the layer below"
    return one(w_ih), one(w_hh), (b_ih.float() + b_hh.float())[perm].contiguous()


def pack_bilstm_ih(w_ih_f, b_ih_f, b_hh_f, w_ih_r, b_ih_r, b_hh_r, precision):
    """Both directions of a bidirectional layer in one projection: columns dir*4H + gate*H + u."""
    w = torch.cat([w_ih_f, w_ih_r], dim=0)
    b = torch.cat([b_ih_f + b_hh_f, b_ih_r + b_hh_r], dim=0)
    return pack_linear(w, b, precision)


def fold_weight_norm(weight_g, weight_v):
    """Old-style torch.nn.utils.weight_norm, dim=0: W = g * v / ||v|| (norm over all axes but 0)."""
    v = weight_v.double()
    norm = v.reshape(v.shape[0], -1).norm(dim=1).reshape([-1] + [1] * (v.dim() - 1))
    return (weight_g.double() * v / norm).float()


def conv_transpose_as_conv(weight, stride, padding):
    """ConvTranspose1d(C_in, C_out, K=2r, stride=r, padding=p) as a 3-tap convolution producing r phases.

    weight (C_in, C_out, K).  Output sample n = r*q + phi of the transposed conv equals
        sum_i sum_{d in -1,0,1} x[i, q + d] * w[i, o, phi + p - r*d]        (terms with k outside [0,K) vanish)
    so with output channel index (phi*C_out + o) and taps d = -1,0,1 (tap_t0 = -1) it is an ordinary conv whose
    channels-last output [B][L][r*C_out] IS the up-sampled signal [B][r*L][C_out] (melgan/modules.py:101-112).
    Returns (C_out*r, C_in, 3)."""
    c_in, c_out, k = weight.shape
    r = stride
    w = torch.zeros(r, c_out, c_in, 3, dtype=weight.dtype, device=weight.device)
    for phi in range(r):
        for di, d in enumerate((-1, 0, 1)):
            kk = phi + padding - r * d
            if 0 <= kk < k:
                w[phi, :, :, di] = weight[:, :, kk].t()
    return w.reshape(r * c_out, c_in, 3)
