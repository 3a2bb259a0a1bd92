"""CPU emulation of the kernels' INDEXING (k-block schedule, gate interleave) on packed weights, in fp64.
Used by CPU tests to validate autoformer_b200.packing against torch's own conv/LSTM ops before any GPU run."""
import torch

from autoformer_b200.packing import KC


def emulate_conv_gemm(w, bias, meta, srcs, B, T, tap_t0, tap_dt):
    """Mirror of avc_conv_gemm's k-block walk: srcs are channels-last [B][rows][C] tensors."""
    kc = KC[meta["precision"]]
    n = meta["N"]
    W = w.double()[:n]
    out = bias.double()[:n].view(1, 1, n).expand(B, T, n).clone()
    col = 0
    for s, a in enumerate(srcs):
        a = a.double()
        C = meta["channels"][s]
        chunks = (C + kc - 1) // kc
        rows_avail = a.shape[1]
        for tap in range(meta["taps"][s]):
            rows = tap_t0[s] + torch.arange(T) + tap * tap_dt[s]
            ok = (rows >= 0) & (rows < rows_avail)
            A = torch.zeros(B, T, chunks * kc, dtype=torch.float64)
            A[:, ok, :C] = a[:, rows[ok], :]
            out += A @ W[:, col:col + chunks * kc].t()
            col += chunks * kc
    assert col == meta["k_pad"]
    return out


def emulate_lstm_seq(xproj, w_hh_packed, B, T, H, G):
    """Mirror of lstm_step_kernel: packed gate order, tile width 4G."""
    xp = xproj.double().view(B, T, 4 * H)
    W = w_hh_packed.double()
    h = torch.zeros(B, H, dtype=torch.float64)
    c = torch.zeros(B, H, dtype=torch.float64)
    out = torch.zeros(B, T, H, dtype=torch.float64)
    u = torch.arange(H)
    base = (u // G) * 4 * G + u % G
    for t in range(T):
        z = xp[:, t] + h @ W.t()
        zi, zf, zg, zo = (z[:, base + g * G] for g in range(4))
        c = torch.sigmoid(zf) * c + torch.sigmoid(zi) * torch.tanh(zg)
        h = torch.sigmoid(zo) * torch.tanh(c)
        out[:, t] = h
    return out


# ---------------------------------------------------------------------------------------------------------
# CPU stand-ins for the C-ABI entry points, so the drop-in models' HOST logic (weight packing, halo buffers,
# poly-phase outputs, gate interleave, buffer formats) can be exercised without a GPU.  Test-only: installed by
# the `cpu_kernels` fixture through monkeypatching; the product package never imports this file.
# ---------------------------------------------------------------------------------------------------------
import torch.nn.functional as F  # noqa: E402

from autoformer_b200 import ops, packing  # noqa: E402

_ACT = {0: lambda v: v, 1: torch.relu, 2: torch.tanh, 3: lambda v: F.leaky_relu(v, 0.2),
        4: lambda v: 0.5 * v * (1.0 + torch.erf(v / 2 ** 0.5)), 5: lambda v: torch.log10(torch.clamp(v, min=1e-5))}


def _emu_convgemm_call(self, srcs, B, T, out=None, out_row0=0, round_tf32=True, reflect=0, out2=None, residual=None,
                       out_raw=None, phases=1, res_after=False, out_fmt=None, raw_fmt=None, halo_after=False, phase0=0,
                       phase_count=None):
    meta = self.meta
    prec = self.precision
    out_fmt = out_fmt or prec
    raw_fmt = raw_fmt or out_fmt
    if not isinstance(srcs, (list, tuple)):
        srcs = [srcs]
    if meta.get("split"):
        phys = []
        for a, c in zip(srcs, meta["logical_channels"]):
            assert a.shape[2] == 2 * c
            phys += [a, a[:, :, :c]]
        srcs = phys
    elif meta.get("dup"):      # fp16x2: the same buffer against w_hi and against w_lo
        srcs = [a for a in srcs for _ in range(2)]
    for a, c in zip(srcs, meta["channels"]):
        assert a.shape[2] == c and a.dtype == packing.TORCH_DTYPE[prec]
    v = emulate_conv_gemm(self.w, self.bias, meta, srcs, B, T, self.tap_t0, self.tap_dt)
    n = meta["N"]
    if phase_count is not None and phase_count != phases:
        # a launch that produces only some of the phases: scatter its rows into the interleaved output
        assert residual is None and out2 is None and not reflect
        cs = n // phase_count
        v = v.reshape(B, T, phase_count, cs)
        a = _ACT[self.act](v)
        rows = (torch.arange(T)[:, None] * phases + phase0 + torch.arange(phase_count)[None, :]).reshape(-1)
        if out_raw is not None:
            out_raw.view(B, T * phases, -1)[:, rows, :packing.act_channels(cs, raw_fmt)] = \
                packing.to_act(v.reshape(B, -1, cs).float(), raw_fmt)
        if out is not None:
            out[:, out_row0 + rows, :packing.act_channels(cs, out_fmt)] = packing.to_act(a.reshape(B, -1, cs).float(), out_fmt)
        return out if out is not None else out_raw
    cs = n // phases
    tl = T * phases
    v = v.reshape(B, tl, cs)
    res = residual.reshape(B, tl, -1)[..., :cs].double() if residual is not None else 0.0
    if not res_after:
        v = v + res
    if out_raw is not None:
        assert out_raw.dtype == packing.TORCH_DTYPE[raw_fmt]
        out_raw.view(B, tl, -1)[..., :packing.act_channels(cs, raw_fmt)] = packing.to_act(v.float(), raw_fmt)
    a = _ACT[self.act](v)
    if res_after:
        a = a + res
    if out is not None:
        assert out.shape[1] >= out_row0 + tl + reflect and out_row0 >= reflect and out.dtype == packing.TORCH_DTYPE[out_fmt]
        full = a
        if reflect:
            full = F.pad(a.transpose(1, 2), (reflect, reflect), mode="reflect").transpose(1, 2)
        out[:, out_row0 - reflect:out_row0 + tl + reflect, :packing.act_channels(cs, out_fmt)] = \
            packing.to_act(full.float(), out_fmt)
    if out2 is not None:
        out2.view(B, tl, -1)[..., :cs] = a.float()
    return out if out is not None else (out2 if out2 is not None else out_raw)


def _emu_lstm_seq(xproj, w_hh, B, T, H, precision, group, hseq=None, hseq_f32=None, h_last=None, persistent=False,
                  xin=None, w_ih=None, bias=None, c_in=None):
    two = precision in packing.TWO_TERM_WEIGHTS
    if two:
        w = w_hh[:, :H].double() + w_hh[:, H:].double()
    else:
        w = w_hh.double()
    if xin is not None:      # fused input projection: K zero-padded to whole k-blocks, [hi | lo] halves when split
        assert xproj is None
        kc = KC[precision]
        kp = (c_in + kc - 1) // kc * kc
        assert w_ih.shape == (4 * H, 2 * kp if two else kp) and bias.shape == (4 * H,) and w_hh.shape[0] == 4 * H
        wi = (w_ih[:, :kp].double() + w_ih[:, kp:].double()) if two else w_ih.double()
        assert float(wi[:, c_in:].abs().max()) == 0.0 if kp > c_in else True
        assert xin.shape[:2] == (B, T) and xin.dtype == packing.TORCH_DTYPE[precision]
        xa = packing.act_to_float(xin[..., :packing.act_channels(c_in, precision)], precision).double()
        xproj = xa @ wi[:, :c_in].t() + bias.double()
    xp = xproj.double().reshape(B, T, -1)
    h = torch.zeros(B, H, dtype=torch.float64)
    c = torch.zeros(B, H, dtype=torch.float64)
    outs = torch.zeros(B, T, H, dtype=torch.float64)
    u = torch.arange(H)
    base = (u // group) * 4 * group + u % group
    for t in range(T):
        hq = packing.act_to_float(packing.to_act(h.float(), precision), precision).double()   # operand rounding of h
        z = xp[:, t] + hq @ w.t()
        zi, zf, zg, zo = (z[:, base + g * group] for g in range(4))
        c = torch.sigmoid(zf) * c + torch.sigmoid(zi) * torch.tanh(zg)
        h = torch.sigmoid(zo) * torch.tanh(c)
        outs[:, t] = h
    if hseq is None:
        hseq = torch.empty(B, T, packing.act_channels(H, precision), dtype=packing.TORCH_DTYPE[precision])
    hseq.copy_(packing.to_act(outs.float(), precision))
    if hseq_f32 is not None:
        hseq_f32.copy_(outs.float())
    if h_last is not None:
        h_last.copy_(outs[:, -1].float())
    return hseq


def _emu_lstm_seq_ws(xproj, w_hh, B, T, H, hseq=None, hseq_f32=None, h_last=None, precision="fp32"):
    """Mirror of lstm_ws_kernel: gate rows packed p = 128 (u//32) + 4 (u%32) + gate; split-bf16 or fp16x2 operands."""
    assert ops.ws_supported(B, H, precision)
    w = w_hh[:, :H].double() + w_hh[:, H:].double()
    xp = xproj.double().reshape(B, T, 4 * H)
    h = torch.zeros(B, H, dtype=torch.float64)
    c = torch.zeros(B, H, dtype=torch.float64)
    outs = torch.zeros(B, T, H, dtype=torch.float64)
    u = torch.arange(H)
    base = 128 * (u // 32) + 4 * (u % 32)
    for t in range(T):
        hq = packing.act_to_float(packing.to_act(h.float(), precision), precision).double()
        z = xp[:, t] + hq @ w.t()
        zi, zf, zg, zo = (z[:, base + g] for g in range(4))
        c = torch.sigmoid(zf) * c + torch.sigmoid(zi) * torch.tanh(zg)
        h = torch.sigmoid(zo) * torch.tanh(c)
        outs[:, t] = h
    if hseq is None:
        hseq = torch.empty(B, T, packing.act_channels(H, precision), dtype=packing.TORCH_DTYPE[precision])
    hseq.copy_(packing.to_act(outs.float(), precision))
    if hseq_f32 is not None:
        hseq_f32.copy_(outs.float())
    if h_last is not None:
        h_last.copy_(outs[:, -1].float())
    return hseq


def _emu_lstm_stack_ws(xproj0, packs, B, T, H, h_last=None, hs=None, debug_clk=None):
    """Mirror of lstm_stack_kernel: tick k finishes frame k - 2 l of layer l; hs[l][t + 1] = fp16(h^l_t), frame 0 zero;
    layer 0 adds xproj0, the layers above add the bias and ONE fp16 term of W_ih times the rows of the layer below at frame
    t + 1; every layer multiplies ONE fp16 term of W_hh with its own rows at frame t; gate rows packed
    p = 128 (u//32) + 4 (u%32) + gate."""
    L = len(packs)
    assert ops.stack_supported(B, H, L, "fp16x2")
    if hs is None:
        hs = torch.full((L, T + 1, B, H), float("nan"), dtype=torch.float16)
    hs[:, 0] = 0                                      # the library zeroes frame 0 of every layer
    xp = xproj0.double().reshape(B, T, 4 * H)
    u = torch.arange(H)
    base = 128 * (u // 32) + 4 * (u % 32)
    c = torch.zeros(L, B, H, dtype=torch.float64)
    for k in range(T + 2 * (L - 1)):
        new = {}
        for l in range(L):
            t = k - 2 * l
            if not 0 <= t < T:
                continue
            w_ih, w_hh, bias = packs[l]
            assert w_hh.dtype == torch.float16
            z = hs[l, t].double() @ w_hh.double().t()
            if l == 0:
                z = z + xp[:, t]
            else:
                assert w_ih.dtype == torch.float16 and not torch.isnan(hs[l - 1, t + 1].float()).any()
                z = z + bias.double() + hs[l - 1, t + 1].double() @ w_ih.double().t()
            zi, zf, zg, zo = (z[:, base + g] for g in range(4))
            c[l] = torch.sigmoid(zf) * c[l] + torch.sigmoid(zi) * torch.tanh(zg)
            new[l] = torch.sigmoid(zo) * torch.tanh(c[l])
        for l, h in new.items():                      # stores of a tick become visible at the grid barrier
            hs[l, k - 2 * l + 1] = h.to(torch.float16)
            if l == L - 1 and k - 2 * l == T - 1 and h_last is not None:
                h_last.copy_(h.float())
    return hs


def _emu_bilstm_small(xproj, w_hh, B, T, H, out=None, codes=None, freq=1, round_tf32=True, split=False):
    xp = xproj.double().view(B, T, 8 * H)
    res = torch.zeros(B, T, 2 * H, dtype=torch.float64)
    for d in range(2):
        w = w_hh[d].double()
        h = torch.zeros(B, H, dtype=torch.float64)
        c = torch.zeros(B, H, dtype=torch.float64)
        steps = range(T - 1, -1, -1) if d else range(T)
        for t in steps:
            z = xp[:, t, d * 4 * H:(d + 1) * 4 * H] + h @ w.t()
            zi, zf, zg, zo = z.split(H, dim=1)
            c = torch.sigmoid(zf) * c + torch.sigmoid(zi) * torch.tanh(zg)
            h = torch.sigmoid(zo) * torch.tanh(c)
            res[:, t, d * H:(d + 1) * H] = h
    if out is not None:
        if split:
            out.copy_(packing.to_act(res.float(), "fp32"))
        elif out.dtype == torch.bfloat16:
            out.copy_(res.to(torch.bfloat16))
        else:
            out.copy_(packing.round_tf32(res.float()) if round_tf32 else res.float())
    if codes is not None:
        codes.copy_(torch.cat((res[:, freq - 1::freq, :H], res[:, ::freq, H:]), dim=-1).float())
    return out, codes


def _emu_concat_bcast(seq, vec, T, div, precision, round_tf32=True):
    parts = [seq.repeat_interleave(div, dim=1)]
    if vec is not None:
        parts.append(vec.unsqueeze(1).expand(-1, T, -1))
    return packing.to_act(torch.cat(parts, dim=-1), precision)


def _emu_linear_l2norm(h, w, bias):
    e = h.double() @ w.double().t() + bias.double()
    return (e / e.norm(dim=-1, keepdim=True)).float()


def _emu_transpose_pad(x, pad, precision, round_tf32=True):
    y = F.pad(x, (pad, pad), mode="reflect") if pad else x
    return packing.to_act(y.transpose(1, 2).contiguous(), precision)


def _emu_conv_to_mono_tanh(x, w, bias):
    K = w.shape[0]
    xp = F.pad(x.double().transpose(1, 2), (K // 2, K // 2), mode="reflect")
    y = F.conv1d(xp, w.double().t().unsqueeze(0)) + bias
    return torch.tanh(y).squeeze(1).float()


def _emu_gn_stats(x, B, eps=1e-5):
    v = x.double().reshape(B, -1)
    mean = v.mean(dim=1)
    var = v.var(dim=1, unbiased=False)
    return torch.stack([mean, 1.0 / torch.sqrt(var + eps)], dim=1).float()


def _emu_gn_pool_residual(x, stats, gamma, precision, want_f32=True, want_op=True):
    xd = x.double()
    pool = F.avg_pool1d(xd.transpose(1, 2), 3, stride=1, padding=1, count_include_pad=False).transpose(1, 2)
    y = xd + stats[:, 1].double().view(-1, 1, 1) * gamma.double().view(1, 1, -1) * (pool - xd)
    return (y.float() if want_f32 else None), (packing.to_act(y.float(), precision) if want_op else None)


def _emu_gn_apply(x, stats, gamma, beta, precision):
    y = (x.double() - stats[:, 0].double().view(-1, 1, 1)) * stats[:, 1].double().view(-1, 1, 1) \
        * gamma.double().view(1, 1, -1) + beta.double().view(1, 1, -1)
    return packing.to_act(y.float(), precision)


def _emu_patchify(a, stats, gamma, beta, p, precision):
    B, S, _ = a.shape
    img = a.double().transpose(1, 2)                       # [B][h = channel][w = length]
    if stats is not None:
        img = (img - stats[:, 0].double().view(-1, 1, 1)) * stats[:, 1].double().view(-1, 1, 1) \
            * gamma.double().view(1, -1, 1) + beta.double().view(1, -1, 1)
    n = S // p
    tok = img.reshape(B, n, p, n, p).permute(0, 1, 3, 2, 4).reshape(B, n * n, p * p)
    return packing.to_act(tok.float(), precision)


def _emu_ln_transpose(x, gamma, beta, ln_axis, precision, want_op=True, want_f32=False):
    B, R, C = x.shape
    xd = x.double()
    y = xd
    if ln_axis == 1:
        y = (xd - xd.mean(-1, keepdim=True)) / torch.sqrt(xd.var(-1, unbiased=False, keepdim=True) + 1e-5) \
            * gamma.double() + beta.double()
    elif ln_axis == 2:
        y = (xd - xd.mean(1, keepdim=True)) / torch.sqrt(xd.var(1, unbiased=False, keepdim=True) + 1e-5) \
            * gamma.double().view(1, -1, 1) + beta.double().view(1, -1, 1)
    r8 = (R + 7) // 8 * 8
    yt = torch.zeros(B, C, r8, dtype=torch.float64)
    yt[:, :, :R] = y.transpose(1, 2)
    xt = torch.zeros(B, C, r8, dtype=torch.float64)
    xt[:, :, :R] = xd.transpose(1, 2)
    return (packing.to_act(yt.float(), precision) if want_op else None), (xt.float() if want_f32 else None)


def _emu_meta_decoder_input(codes, c_trg, T, freq, precision):
    up = codes.repeat_interleave(freq, dim=1)                                       # [B][T][2H]
    full = torch.cat((up, c_trg.unsqueeze(1).expand(-1, T, -1)), dim=-1)            # [B][T][2H+E]
    return packing.to_act(full.transpose(1, 2).contiguous(), precision)


def _emu_gather_codes(out, H, freq):
    return torch.cat((out[:, freq - 1::freq, :H], out[:, ::freq, H:]), dim=-1).contiguous()


def _emu_global_stats(x, out=None):
    v = x.double().reshape(-1)
    r = torch.stack([v.mean(), v.std()]).float()
    if out is not None:
        out.copy_(r)
        return out
    return r


def _emu_adain(x, x_stats, t_stats, precision, want_f32=False):
    xs, ts = x_stats.double(), t_stats.double()
    y = ((x.double() - xs[0]) / xs[1] * ts[1] + ts[0]).float()
    return packing.to_act(y, precision), (y if want_f32 else None)


def _emu_audio_frames(audio, pad, hop, rows, precision):
    B, L = audio.shape
    padded = F.pad(audio.unsqueeze(1), (pad, pad), mode="reflect").squeeze(1)
    buf = torch.zeros(B, rows * hop, dtype=torch.float32)
    n = min(rows * hop, padded.shape[1])
    buf[:, :n] = padded[:, :n]
    return packing.to_act(buf.view(B, rows, hop), precision)


def _emu_complex_mag(spec, bins, bins_pad, precision):
    mag = torch.zeros(spec.shape[0], bins_pad, dtype=torch.float64)
    mag[:, :bins] = torch.sqrt(spec[:, :bins].double() ** 2 + spec[:, bins:].double() ** 2)
    return packing.to_act(mag.float().unsqueeze(0), precision)


def resblock_terms(w, C, version):
    """(hi, lo) fp64 (C_out, C_in) terms of W3 tap 0..2, W1, Wsc decoded from the PACKED tiles of
    packing.pack_resblock (version 1) / pack_resblock2 (version 2), layouts as the kernels read them."""
    w = w.double()
    if version == 1:
        if C == 64:
            return [(w[i, :64], w[i, 64:]) for i in range(5)]
        assert torch.equal(w[:, :32, :32], w[:, :32, 32:]) and not w[:, 32:, 32:].any()
        return [(w[i, :32, :32], w[i, 32:, :32]) for i in range(5)]
    if C == 128:      # [matrix][k-chunk][CTA 0: w_hi[0:64]; w_lo[0:64] | CTA 1: w_hi[64:128]; w_lo[64:128]][64]
        terms = []
        for m in range(5):
            hi = torch.zeros(128, 128, dtype=torch.float64)
            lo = torch.zeros(128, 128, dtype=torch.float64)
            for kc in range(2):
                t = w[(m * 2 + kc) * 256:(m * 2 + kc + 1) * 256]
                ks = slice(kc * 64, kc * 64 + 64)
                hi[0:64, ks], lo[0:64, ks], hi[64:128, ks], lo[64:128, ks] = t[0:64], t[64:128], t[128:192], t[192:256]
            terms.append((hi, lo))
        return terms
    if C == 64:
        return [(w[128 * i:128 * i + 64], w[128 * i + 64:128 * (i + 1)]) for i in range(5)]
    k3 = [w[32 * i:32 * (i + 1)] for i in range(3)]
    k1 = [w[96 + 64 * i:96 + 64 * (i + 1)] for i in range(2)]
    for t in k1:
        assert torch.equal(t[:32, :32], t[:32, 32:]) and not t[32:, 32:].any()
    return [(t[:, :32], t[:, 32:]) for t in k3] + [(t[:32, :32], t[32:, :32]) for t in k1]


def _emu_resblock_call(self, xa, x, B, L, out=None, out_row0=0, reflect=0, out_raw=None, out2=None):
    """Mirror of avc_resblock: reads the PACKED tiles (so packing.pack_resblock is what gets validated), the halo
    window of LeakyReLU(x) with row-shifted taps, the split intermediate, and the three output forms."""
    C, d = self.C, self.dilation
    assert xa.shape == (B, L + 2 * d, 2 * C) and x.shape == (B, L, 2 * C) and L % 128 == 0
    mats = [hi + lo for hi, lo in resblock_terms(self.w, C, 1)]
    a = packing.act_to_float(xa, "fp32").double()
    mid = self.bias3.double().view(1, 1, C).expand(B, L, C).clone()
    for tap in range(3):
        mid = mid + a[:, tap * d:tap * d + L] @ mats[tap].t()
    mid = packing.act_to_float(packing.to_act(F.leaky_relu(mid, 0.2).float(), "fp32"), "fp32").double()
    y = mid @ mats[3].t() + packing.act_to_float(x, "fp32").double() @ mats[4].t() + self.bias1.double()
    if out_raw is not None:
        out_raw[:] = packing.to_act(y.float(), "fp32")
    ya = F.leaky_relu(y, 0.2)
    if out is not None:
        assert out2 is None and out.shape[1] >= out_row0 + L + reflect and out_row0 >= reflect
        full = F.pad(ya.transpose(1, 2), (reflect, reflect), mode="reflect").transpose(1, 2) if reflect else ya
        out[:, out_row0 - reflect:out_row0 + L + reflect] = packing.to_act(full.float(), "fp32")
    if out2 is not None:
        out2[:] = ya.float().reshape(B * L, C)
    return out if out is not None else (out2 if out2 is not None else out_raw)


def _emu_resblock2_call(self, x, B, L, y=None, y_row0=0, y_reflect=0, y_act=False, out2=None, wav=None, mono=None,
                        lengths=None):
    """Mirror of avc_resblock2: reads the PACKED tiles (packing.pack_resblock2 is what gets validated), forms the k3
    operand as ONE fp16 value from the two-term window, keeps the intermediate as two fp16 terms, reads the shortcut
    operand from the centre rows of the same window.  lengths (ops.RaggedRows): a padded batch -- only the tiles that
    hold a valid row are written, wav reflects at each utterance's own end and is 0 past it in its last tile."""
    if lengths is not None:
        return _emu_resblock2_ragged(self, x, B, L, lengths.host, y, y_row0, y_reflect, y_act, out2, wav, mono)
    C, d = self.C, self.dilation
    assert x.shape == (B, L + 2 * d, 2 * C) and x.dtype == torch.float16 and L % 128 == 0
    mats = [hi + lo for hi, lo in resblock_terms(self.w, C, 2)]
    xs = packing.act_to_float(x, "fp16s").double()                                   # the stored stream (hi + lo)
    xa = F.leaky_relu(xs, 0.2).float().half().double()                                # one fp16 value
    mid = self.bias3.double().view(1, 1, C).expand(B, L, C).clone()
    for tap in range(3):
        mid = mid + xa[:, tap * d:tap * d + L] @ mats[tap].t()
    mid = packing.act_to_float(packing.to_act(F.leaky_relu(mid, 0.2).float(), "fp16s"), "fp16s").double()
    v = mid @ mats[3].t() + xs[:, d:d + L] @ mats[4].t() + self.bias1.double()
    if y is not None:
        a = F.leaky_relu(v, 0.2) if y_act else v
        assert y.shape[1] >= y_row0 + L + y_reflect and y_row0 >= y_reflect
        full = F.pad(a.transpose(1, 2), (y_reflect, y_reflect), mode="reflect").transpose(1, 2) if y_reflect else a
        y[:, y_row0 - y_reflect:y_row0 + L + y_reflect] = packing.to_act(full.float(), "fp16s")
        return y
    if wav is not None:
        # the fused output layer, tile by tile like the kernel: tiles of 128 staged rows overlap by K - 1, output r of a
        # tile reads rows r .. r + K - 1, mirrored at the ends of the utterance
        w_out, b_out = mono
        K, lead = w_out.shape[0], w_out.shape[0] // 2
        assert C == 32 and wav.shape == (B, L) and w_out.shape == (K, C)
        a = F.leaky_relu(v, 0.2).float()                                              # staged as exact fp32
        stride = 128 - (K - 1)
        for j in range((L + stride - 1) // stride):
            t0 = j * stride - lead
            for r in range(stride):
                t = t0 + lead + r
                if t >= L:
                    break
                acc = torch.zeros(B, dtype=torch.float64)
                for k in range(K):
                    tau = t + k - lead
                    tau = -tau if tau < 0 else (2 * (L - 1) - tau if tau >= L else tau)
                    assert 0 <= tau - t0 < 128
                    acc += a[:, tau].double() @ w_out[k].double()
                wav[:, t] = torch.tanh(acc + b_out).float()
        return wav
    out2[:] = F.leaky_relu(v, 0.2).float().reshape(B * L, C)
    return out2


def _emu_resblock2_ragged(self, x, B, L, rows, y, y_row0, y_reflect, y_act, out2, wav, mono):
    """_emu_resblock2_call over a padded batch: the dense result, stored only where avc_resblock2's compacted tile
    space reaches (tiles of 128 rows, or of 128 - (K - 1) rows for wav); the right halo of y at an utterance's own end is
    the caller's, the kernel writes the one at L only when the utterance's last tile runs."""
    if wav is not None:
        w_out, b_out = mono
        K, lead = w_out.shape[0], w_out.shape[0] // 2
        stride = 128 - (K - 1)
        full = torch.empty(B * L, self.C)
        _emu_resblock2_call(self, x, B, L, out2=full)
        a = full.view(B, L, self.C).double()
        for b, n in enumerate(rows):
            tau = torch.arange(n)[:, None] + torch.arange(K)[None, :] - lead
            tau = torch.where(tau < 0, -tau, tau)
            tau = torch.where(tau >= n, 2 * (n - 1) - tau, tau)
            acc = (a[b][tau] * w_out.double()[None]).sum(dim=(1, 2)) + b_out
            wav[b, :n] = torch.tanh(acc).float()
            wav[b, n:min(L, -(-n // stride) * stride)] = 0
        return wav
    full = y.clone() if y is not None else out2.clone()
    _emu_resblock2_call(self, x, B, L, full if y is not None else None, y_row0, y_reflect, y_act,
                        full if out2 is not None else None)
    for b, n in enumerate(rows):
        end = -(-n // 128) * 128                                                # rows of the tiles that run
        if y is not None:
            y[b, y_row0 - y_reflect:y_row0 + end] = full[b, y_row0 - y_reflect:y_row0 + end]
            if end >= L:
                y[b, y_row0 + L:y_row0 + L + y_reflect] = full[b, y_row0 + L:y_row0 + L + y_reflect]
        else:
            out2[b * L:b * L + end] = full[b * L:b * L + end]
    return y if y is not None else out2


def _emu_reflect_halo(buf, row0, L, reflect):
    for k in range(1, reflect + 1):
        buf[:, row0 - k] = buf[:, row0 + k]
        buf[:, row0 + L - 1 + k] = buf[:, row0 + L - 1 - k]
    return buf


def install_cpu_kernels(monkeypatch):
    monkeypatch.setattr(ops, "reflect_halo", _emu_reflect_halo)
    monkeypatch.setattr(ops.Resblock, "__call__", _emu_resblock_call)
    monkeypatch.setattr(ops.Resblock2, "__call__", _emu_resblock2_call)
    monkeypatch.setattr(ops, "audio_frames", _emu_audio_frames)
    monkeypatch.setattr(ops, "complex_mag", _emu_complex_mag)
    monkeypatch.setattr(ops, "global_stats", _emu_global_stats)
    monkeypatch.setattr(ops, "adain", _emu_adain)
    monkeypatch.setattr(ops, "gn_stats", _emu_gn_stats)
    monkeypatch.setattr(ops, "gn_pool_residual", _emu_gn_pool_residual)
    monkeypatch.setattr(ops, "gn_apply", _emu_gn_apply)
    monkeypatch.setattr(ops, "patchify", _emu_patchify)
    monkeypatch.setattr(ops, "ln_transpose", _emu_ln_transpose)
    monkeypatch.setattr(ops, "meta_decoder_input", _emu_meta_decoder_input)
    monkeypatch.setattr(ops, "gather_codes", _emu_gather_codes)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops.ConvGemm, "__call__", _emu_convgemm_call)
    monkeypatch.setattr(ops, "lstm_seq", _emu_lstm_seq)
    monkeypatch.setattr(ops, "lstm_seq_ws", _emu_lstm_seq_ws)
    monkeypatch.setattr(ops, "lstm_stack_ws", _emu_lstm_stack_ws)
    monkeypatch.setattr(ops, "bilstm_small", _emu_bilstm_small)
    monkeypatch.setattr(ops, "concat_bcast", _emu_concat_bcast)
    monkeypatch.setattr(ops, "to_act", lambda x, precision, round_tf32=True: _emu_concat_bcast(x, None, x.shape[1], 1, precision))
    monkeypatch.setattr(ops, "linear_l2norm", _emu_linear_l2norm)
    monkeypatch.setattr(ops, "transpose_pad", _emu_transpose_pad)
    monkeypatch.setattr(ops, "conv_to_mono_tanh", _emu_conv_to_mono_tanh)
