"""Drop-in MelGAN ``Generator(input_size, ngf, n_residual_layers)`` on libavc_b200.so (melgan/modules.py:72-130).

The module tree only HOLDS parameters under the reference's state_dict names (``model.{i}.weight_g`` ...);
``forward`` folds weight norm once and runs every layer as a tcgen05 implicit GEMM on channels-last buffers:

  ReflectionPad1d(3) + transpose    -> avc_transpose_pad (halo rows written once)
  WNConv1d k7                       -> 7-tap conv, LeakyReLU fused (its only consumer applies it)
  LeakyReLU + WNConvTranspose1d(r)  -> 3-tap conv producing r output phases per input frame (poly-phase), whose
                                       epilogue writes both x (for the shortcut) and LeakyReLU(x) with the reflected
                                       halo rows the next dilated conv needs
  ResnetBlock                       -> [k3 dilated conv + LeakyReLU] then ONE GEMM over the K-concatenated pair
                                       (block output, shortcut input) x [W_k1 | W_shortcut]; the narrow, long stages
                                       (C = 64 / 32) run each block as ONE fused kernel (avc_resblock) with the
                                       intermediate in shared memory and the weights resident
  LeakyReLU + ReflectionPad1d(3) + WNConv1d(32 -> 1, k7) + Tanh -> avc_conv_to_mono_tanh
"""

import numpy as np
import torch
import torch.nn as nn
from torch.nn.utils import weight_norm

from .. import layers, ops, packing


def WNConv1d(*args, **kwargs):
    return weight_norm(nn.Conv1d(*args, **kwargs))


def WNConvTranspose1d(*args, **kwargs):
    return weight_norm(nn.ConvTranspose1d(*args, **kwargs))


class ResnetBlock(nn.Module):
    """Parameter container (melgan/modules.py:72-85)."""

    def __init__(self, dim, dilation=1):
        super().__init__()
        self.block = nn.Sequential(nn.LeakyReLU(0.2), nn.ReflectionPad1d(dilation),
                                   WNConv1d(dim, dim, kernel_size=3, dilation=dilation), nn.LeakyReLU(0.2),
                                   WNConv1d(dim, dim, kernel_size=1))
        self.shortcut = WNConv1d(dim, dim, kernel_size=1)
        self.dilation = dilation


class _Plan:
    def __init__(self, gen, precision):
        sd = layers.state_for_packing(gen)
        W = lambda p: packing.fold_weight_norm(sd[p + ".weight_g"], sd[p + ".weight_v"])
        b = lambda p: sd[p + ".bias"].float()
        self.precision = precision
        self.stem = ops.ConvGemm(*packing.pack_conv(W("model.1"), b("model.1"), precision), tap_t0=[0], act="lrelu",
                                 tag="melgan_conv")
        self.stages = []
        idx = 2
        for r in gen.ratios:
            wt = W(f"model.{idx + 1}")                                   # (C_in, C_out, 2r)
            c_out = wt.shape[1]
            w3 = packing.conv_transpose_as_conv(wt, r, r // 2 + r % 2)
            up = ops.ConvGemm(*packing.pack_conv(w3, b(f"model.{idx + 1}").repeat(r), precision), tap_t0=[-1],
                              act="lrelu", tag="melgan_up")
            blocks = []
            for j in range(gen.n_residual_layers):
                p = f"model.{idx + 2 + j}"
                d = 3 ** j
                c3 = ops.ConvGemm(*packing.pack_conv(W(p + ".block.2"), b(p + ".block.2"), precision), tap_t0=[0],
                                  tap_dt=[d], act="lrelu", tag="melgan_conv")
                k1 = ops.ConvGemm(*packing.pack_conv_sources([W(p + ".block.4"), W(p + ".shortcut")],
                                                             b(p + ".block.4") + b(p + ".shortcut"), precision),
                                  tap_t0=[0, 0], act="lrelu", tag="melgan_conv")
                fused = None
                if precision == "fp32" and c_out in packing.RESBLOCK_CHANNELS:
                    fused = ops.Resblock(*packing.pack_resblock(W(p + ".block.2"), b(p + ".block.2"), W(p + ".block.4"),
                                                                b(p + ".block.4"), W(p + ".shortcut"),
                                                                b(p + ".shortcut")), dilation=d)
                blocks.append((d, c3, k1, fused))
            self.stages.append((r, c_out, up, blocks))
            idx += 2 + gen.n_residual_layers
        wf = W(f"model.{idx + 2}")                                        # (1, ngf, 7)
        self.w_out = wf[0].t().contiguous().float()                      # [K][C]
        self.b_out = float(b(f"model.{idx + 2}")[0])


class _PlanF16s:
    """Packed layers of the "fp16s" precision (round 2).  Tensor formats, chosen per role from
    scripts/melgan_precision_study.py (waveform rel-L2 <= 5.3e-4 over six weight seeds, against 1.2e-3 when every
    activation is ONE fp16 value):
      two fp16 terms (hi | lo)  the residual stream x, the ConvTranspose operands, the ResnetBlock intermediate
      one fp16 value            LeakyReLU(x), the operand of the dilated k3 convolutions (60 % of a block's MMAs)
    Weights are two fp16 terms everywhere.  Stages of 32 / 64 channels run each ResnetBlock as ONE kernel
    (avc_resblock2) that reads the raw stream and writes its output, nothing else."""

    def __init__(self, gen):
        sd = layers.state_for_packing(gen)
        W = lambda p: packing.fold_weight_norm(sd[p + ".weight_g"], sd[p + ".weight_v"])
        b = lambda p: sd[p + ".bias"].float()
        self.precision = "fp16s"
        self.stem = ops.ConvGemm(*packing.pack_conv(W("model.1"), b("model.1"), "fp16s"), tap_t0=[0], act="lrelu",
                                 tag="melgan_conv")
        self.stages = []
        idx = 2
        for r in gen.ratios:
            wt = W(f"model.{idx + 1}")                                   # (C_in, C_out, 2r)
            c_out = wt.shape[1]
            w3 = packing.conv_transpose_as_conv(wt, r, r // 2 + r % 2)
            bias_up = b(f"model.{idx + 1}")
            # a fused stage wants the raw stream only; a layer-wise stage wants LeakyReLU(x) (one fp16) plus the raw x.
            # Each output phase of the transposed convolution uses two of the three input taps -- (t-1, t) for phases
            # < r/2, (t, t+1) for the rest -- so a wide up-sampler (r = 8) runs as two GEMMs of two taps each: a third
            # less MMA work and operand traffic than one GEMM whose weights are one third zeros.  (r = 2 stays one GEMM:
            # its halves would be N = C_out <= 64 wide, below the tile width at which the tensor pipe is fed.)
            if r >= 4:
                half = r // 2 * c_out
                assert not w3[:half, :, 2].any() and not w3[half:, :, 0].any()
                parts = [(packing.pack_conv(w3[:half, :, 0:2].contiguous(), bias_up.repeat(r // 2), "fp16s"), -1, 0),
                         (packing.pack_conv(w3[half:, :, 1:3].contiguous(), bias_up.repeat(r // 2), "fp16s"), 0, r // 2)]
            else:
                parts = [(packing.pack_conv(w3, bias_up.repeat(r), "fp16s"), -1, 0)]
            up_raw = [(ops.ConvGemm(*pk, tap_t0=[t0], act="none", tag="melgan_up"), p0) for pk, t0, p0 in parts]
            up_act = [(ops.ConvGemm(*pk, tap_t0=[t0], act="lrelu", tag="melgan_up"), p0) for pk, t0, p0 in parts]
            blocks = []
            for j in range(gen.n_residual_layers):
                p = f"model.{idx + 2 + j}"
                d = 3 ** j
                c3 = ops.ConvGemm(*packing.pack_conv(W(p + ".block.2"), b(p + ".block.2"), "fp16x2"), tap_t0=[0],
                                  tap_dt=[d], act="lrelu", tag="melgan_conv")
                k1 = ops.ConvGemm(*packing.pack_conv_sources([W(p + ".block.4"), W(p + ".shortcut")],
                                                             b(p + ".block.4") + b(p + ".shortcut"), "fp16s"),
                                  tap_t0=[0, 0], act="lrelu", tag="melgan_conv")
                fused = None
                if c_out in packing.RESBLOCK2_CHANNELS:
                    fused = ops.Resblock2(*packing.pack_resblock2(W(p + ".block.2"), b(p + ".block.2"), W(p + ".block.4"),
                                                                  b(p + ".block.4"), W(p + ".shortcut"),
                                                                  b(p + ".shortcut")), dilation=d)
                blocks.append((d, c3, k1, fused))
            self.stages.append((r, c_out, up_raw, up_act, blocks))
            idx += 2 + gen.n_residual_layers
        wf = W(f"model.{idx + 2}")                                        # (1, ngf, 7)
        self.w_out = wf[0].t().contiguous().float()                      # [K][C]
        self.b_out = float(b(f"model.{idx + 2}")[0])


def _inv_lrelu(a):
    """y from LeakyReLU(y) (slope 0.2): exact up to one fp32 rounding.  Used only for the parity taps."""
    return torch.where(a >= 0, a, a / 0.2)


class Audio2Mel(layers.PlanOwner, nn.Module):
    """Drop-in ``Audio2Mel`` (melgan/modules.py:26-69): audio (B, 1, L) -> log10-mel (B, n_mel, L // hop).

    The STFT is an implicit-GEMM convolution on the tensor cores: the reflect-padded signal is viewed as rows of
    ``hop`` samples, a frame is n_fft / hop consecutive rows, and the hann-windowed DFT basis is a (2 * bins, hop,
    n_fft / hop) convolution weight; magnitude, mel projection (``mel_basis`` buffer, same name as the reference's) and
    ``log10(clamp(., 1e-5))`` follow as one small kernel and one GEMM with the log in its epilogue."""

    def __init__(self, n_fft=1024, hop_length=256, win_length=1024, sampling_rate=22050, n_mel_channels=80,
                 mel_fmin=0.0, mel_fmax=None):
        super().__init__()
        from .filters import mel_filterbank
        assert n_fft % hop_length == 0 and hop_length % 8 == 0 and win_length <= n_fft
        self.register_buffer("mel_basis", torch.from_numpy(mel_filterbank(sampling_rate, n_fft, n_mel_channels,
                                                                          mel_fmin, mel_fmax)).float())
        self.register_buffer("window", torch.hann_window(win_length).float())
        self.n_fft, self.hop_length, self.win_length = n_fft, hop_length, win_length
        self.sampling_rate, self.n_mel_channels = sampling_rate, n_mel_channels
        self.precision = "fp32"
        self._cache = layers.PlanCache()

    def _plan(self):
        def build():
            N, hop, bins = self.n_fft, self.hop_length, self.n_fft // 2 + 1
            dev = self.mel_basis.device
            win = torch.zeros(N, dtype=torch.float64, device=dev)
            lo = (N - self.win_length) // 2                     # torch.stft centres a short window in the frame
            win[lo:lo + self.win_length] = self.window.double()
            j = torch.arange(N, dtype=torch.float64, device=dev)
            k = torch.arange(bins, dtype=torch.float64, device=dev)
            ang = 2.0 * torch.pi * k[:, None] * j[None, :] / N
            bins_pad = (bins + 7) // 8 * 8                      # 513 -> 520: channel counts must be multiples of 8
            basis = torch.zeros(2 * bins_pad, N, dtype=torch.float64, device=dev)           # re | im halves
            basis[:bins] = torch.cos(ang) * win
            basis[bins_pad:bins_pad + bins] = -torch.sin(ang) * win
            w = basis.view(2 * bins_pad, N // hop, hop).permute(0, 2, 1).contiguous().float()   # (C_out, C_in = hop, taps)
            stft = ops.ConvGemm(*packing.pack_conv(w, torch.zeros(2 * bins_pad, device=dev), self.precision),
                                tap_t0=[0], tag="stft")
            mb = torch.zeros(self.n_mel_channels, bins_pad, dtype=torch.float32, device=dev)
            mb[:, :bins] = self.mel_basis.float()
            mel = ops.ConvGemm(*packing.pack_linear(mb, torch.zeros(self.n_mel_channels, device=dev), self.precision),
                               act="log10_clamp", tag="mel")
            return dict(stft=stft, mel=mel, bins=bins, bins_pad=bins_pad)
        return self._cache.get(self, (self.precision,), build)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, audio):
        ops._require_cuda(audio)
        if audio.dim() == 3:
            audio = audio.squeeze(1)                            # (B, 1, L), modules.py:56-57
        audio = audio.contiguous().float()
        B, L = audio.shape
        plan = self._plan()
        hop, taps = self.hop_length, self.n_fft // self.hop_length
        pad = (self.n_fft - hop) // 2                           # modules.py:55
        if L <= pad:
            raise RuntimeError(f"reflect padding of {pad} samples needs more than {pad} input samples (got {L})")
        frames = (L + 2 * pad - self.n_fft) // hop + 1
        rows = frames + taps - 1
        x = ops.audio_frames(audio, pad, hop, rows, self.precision)
        spec = torch.empty(B * frames, 2 * plan["bins_pad"], dtype=torch.float32, device=audio.device)
        plan["stft"](x, B, frames, out2=spec)                   # torch.stft(center=False), modules.py:58-65
        mag = ops.complex_mag(spec, plan["bins_pad"], plan["bins_pad"], self.precision)      # :66 (pad bins are 0)
        out = torch.empty(B * frames, self.n_mel_channels, dtype=torch.float32, device=audio.device)
        plan["mel"](mag.view(B, frames, -1), B, frames, out2=out)                          # :67-68
        return out.view(B, frames, self.n_mel_channels).transpose(1, 2).contiguous()


class Generator(layers.PlanOwner, nn.Module):
    def __init__(self, input_size, ngf, n_residual_layers):
        super().__init__()
        ratios = [8, 8, 2, 2]
        self.ratios, self.n_residual_layers = ratios, n_residual_layers
        self.hop_length = int(np.prod(ratios))
        mult = int(2 ** len(ratios))
        model = [nn.ReflectionPad1d(3), WNConv1d(input_size, mult * ngf, kernel_size=7, padding=0)]
        for r in ratios:
            model += [nn.LeakyReLU(0.2),
                      WNConvTranspose1d(mult * ngf, mult * ngf // 2, kernel_size=r * 2, stride=r,
                                        padding=r // 2 + r % 2, output_padding=r % 2)]
            for j in range(n_residual_layers):
                model += [ResnetBlock(mult * ngf // 2, dilation=3 ** j)]
            mult //= 2
        model += [nn.LeakyReLU(0.2), nn.ReflectionPad1d(3), WNConv1d(ngf, 1, kernel_size=7, padding=0), nn.Tanh()]
        self.model = nn.Sequential(*model)
        self.precision = "fp32"
        self.collect_taps = False
        self.taps = {}
        # False: every ResnetBlock as two avc_conv_gemm launches (the unfused reference path)
        self.fuse_resblocks = True
        self._cache = layers.PlanCache()

    def _plan(self):
        build = (lambda: _PlanF16s(self)) if self.precision == "fp16s" else (lambda: _Plan(self, self.precision))
        return self._cache.get(self, (self.precision,), build)

    def _ragged_rows(self, plan, lengths, B, T, device):
        """Validated lengths of a padded batch -> RaggedRows of the stem (index 0) and of every stage (index si + 1),
        one upload.  The reference's own ReflectionPad1d(3) needs at least 4 frames."""
        vals = layers.check_lengths(lengths, B, T)
        if min(vals) < 4:
            raise ValueError(f"lengths must be at least 4 frames (ReflectionPad1d(3) of the first layer); got {min(vals)}")
        if self.collect_taps:
            raise NotImplementedError("stage taps (collect_taps) of a variable-length batch")
        scales = [1]
        for r in self.ratios:
            scales.append(scales[-1] * r)
        return ops.ragged_rows(vals, scales, (128, 128 - (plan.w_out.shape[0] - 1)), device)

    def _forward_f16s(self, plan, x, rows=None):
        """The "fp16s" data flow (see _PlanF16s): raw residual stream as two fp16 terms, one tensor between kernels.
        rows: RaggedRows per level of a padded batch (see forward)."""
        B, _, T = x.shape
        dev = x.device
        P = "fp16s"
        taps = self.taps if self.collect_taps else None
        m0 = ops.transpose_pad(x, 3, P)                                   # model.0 + layout change
        if rows is not None:
            ops.reflect_halo(m0, 3, T, 3, lengths=rows[0].rows)           # ReflectionPad1d(3) at each utterance's end
        cur = ops.alloc_act(B, T, plan.stem.meta["N"], P, dev)
        plan.stem(m0, B, T, out=cur)                                      # model.1 (+ model.2's LeakyReLU)
        L = T
        final = wav = None
        n_stage = len(plan.stages)
        for si, (r, C, up_raw, up_act, blocks) in enumerate(plan.stages):
            Lr = r * L
            last_stage = si + 1 == n_stage
            d0 = blocks[0][0]
            rs = rows[si + 1] if rows is not None else None
            halo_kw = layers._lengths_kw(rs.rows if rs is not None else None)
            block_kw = layers._lengths_kw(rs)
            if rows is not None:
                ops.zero_tail(cur, 0, L, rows[si].rows)    # the ConvTranspose reads frame m + 1 = lengths[b] as zero
            if self.fuse_resblocks and ops.Resblock2.eligible(C, Lr):
                xs = ops.alloc_act(B, Lr + 2 * d0, C, P, dev)
                for up, p0 in up_raw:                                                   # ConvTranspose1d: raw stream
                    up(cur, B, L, out=xs, out_row0=d0, phases=r, phase0=p0, phase_count=r // len(up_raw))
                ops.reflect_halo(xs, d0, Lr, d0, **halo_kw)                             # + the first block's halo rows
                if taps is not None:
                    taps[f"up{si}"] = packing.act_to_float(xs[:, d0:d0 + Lr], P)
                for j, (d, _, _, fused) in enumerate(blocks):
                    if j + 1 < len(blocks):
                        dn = blocks[j + 1][0]
                        ys = ops.alloc_act(B, Lr + 2 * dn, C, P, dev)
                        fused(xs, B, Lr, y=ys, y_row0=dn, y_reflect=dn, **block_kw)
                        if rs is not None:
                            # the right halo at each utterance's end: its rows lie inside the last tile, which the
                            # block TMA-stores whole, so they are written after the block, not by it
                            ops.reflect_halo(ys, dn, Lr, dn, lengths=rs.rows)
                        xs = ys
                    elif not last_stage:
                        cur = ops.alloc_act(B, Lr, C, P, dev)
                        fused(xs, B, Lr, y=cur, y_act=True, **block_kw)                  # + the next model.{i} LeakyReLU
                        if taps is not None:
                            taps[f"stage{si}"] = _inv_lrelu(packing.act_to_float(cur, P))
                    elif taps is None and C == 32:
                        # model.22-25 (LeakyReLU, ReflectionPad1d(3), Conv1d(32 -> 1, k7), tanh) in the block's epilogue:
                        # the block's output (1 GB at B = 32) is neither written nor re-read.  A padded batch skips the
                        # tiles past each utterance's end, so their samples come from the zero fill.
                        wav = (torch.zeros if rs is not None else torch.empty)(B, Lr, dtype=torch.float32, device=dev)
                        fused(xs, B, Lr, wav=wav, mono=(plan.w_out, plan.b_out), **block_kw)
                    else:
                        final = torch.empty(B * Lr, C, dtype=torch.float32, device=dev)
                        fused(xs, B, Lr, out2=final, **block_kw)
                        if taps is not None:
                            taps[f"stage{si}"] = _inv_lrelu(final.view(B, Lr, C))
            else:
                x_raw = ops.alloc_act(B, Lr, C, P, dev)
                xa = ops.alloc_act(B, Lr + 2 * d0, C, "f16", dev)
                for up, p0 in up_act:
                    up(cur, B, L, out=xa, out_row0=d0, out_raw=x_raw, phases=r, out_fmt="f16", raw_fmt=P, phase0=p0,
                       phase_count=r // len(up_act))
                ops.reflect_halo(xa, d0, Lr, d0, **halo_kw)
                if taps is not None:
                    taps[f"up{si}"] = packing.act_to_float(x_raw, P)
                for j, (d, c3, k1, _) in enumerate(blocks):
                    h1 = ops.alloc_act(B, Lr, C, P, dev)
                    c3(xa, B, Lr, out=h1, out_fmt=P)                                     # block.0-3 (one fp16 operand in)
                    if j + 1 < len(blocks):
                        dn = blocks[j + 1][0]
                        y_raw = ops.alloc_act(B, Lr, C, P, dev)
                        ya = ops.alloc_act(B, Lr + 2 * dn, C, "f16", dev)
                        k1([h1, x_raw], B, Lr, out=ya, out_row0=dn, reflect=dn if rs is None else 0, out_raw=y_raw,
                           out_fmt="f16", raw_fmt=P, halo_after=True)
                        if rs is not None:
                            ops.reflect_halo(ya, dn, Lr, dn, lengths=rs.rows)
                        x_raw, xa = y_raw, ya
                    elif not last_stage:
                        cur = ops.alloc_act(B, Lr, C, P, dev)
                        k1([h1, x_raw], B, Lr, out=cur)                                  # block.4 + shortcut + next LeakyReLU
                        if taps is not None:
                            taps[f"stage{si}"] = _inv_lrelu(packing.act_to_float(cur, P))
                    else:
                        final = torch.empty(B * Lr, C, dtype=torch.float32, device=dev)
                        k1([h1, x_raw], B, Lr, out2=final)
                        if taps is not None:
                            taps[f"stage{si}"] = _inv_lrelu(final.view(B, Lr, C))
            L = Lr
        if wav is None:
            last_kw = layers._lengths_kw(rows[-1].rows if rows is not None else None)
            wav = ops.conv_to_mono_tanh(final.view(B, L, -1), plan.w_out, plan.b_out, **last_kw)  # model.22-25
        return wav.unsqueeze(1)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, lengths=None):
        """x (B, input_size, T) log-mel -> waveform (B, 1, hop_length * T)   (melgan/modules.py:129-130).

        lengths (list, CPU or CUDA tensor of B ints, 4 <= lengths[b] <= T): a zero-padded batch of utterances of
        different lengths.  Samples < hop_length * lengths[b] of utterance b are what the generator gives for
        x[b:b+1, :, :lengths[b]] alone, the samples past them are 0, and whatever x holds past lengths[b] is ignored."""
        ops._require_cuda(x)
        plan = self._plan()
        prec = plan.precision
        rows = None
        if lengths is not None:
            rows = self._ragged_rows(plan, lengths, x.shape[0], x.shape[2], x.device)
        if prec == "fp16s":
            if self.collect_taps:
                self.taps.clear()
            return self._forward_f16s(plan, x.contiguous().float(), rows)
        x = x.contiguous().float()
        B, _, T = x.shape
        dev = x.device
        taps = self.taps if self.collect_taps else None
        if taps is not None:
            taps.clear()
        m0 = ops.transpose_pad(x, 3, prec)                                # model.0 + layout change
        if rows is not None:
            ops.reflect_halo(m0, 3, T, 3, lengths=rows[0].rows)           # ReflectionPad1d(3) at each utterance's end
        cur = ops.alloc_act(B, T, plan.stem.meta["N"], prec, dev)
        plan.stem(m0, B, T, out=cur)                                      # model.1 (+ model.2's LeakyReLU)
        L = T
        final = None
        n_stage = len(plan.stages)
        for si, (r, C, up, blocks) in enumerate(plan.stages):
            Lr = r * L
            d0 = blocks[0][0]
            rs = rows[si + 1] if rows is not None else None
            if rows is not None:
                ops.zero_tail(cur, 0, L, rows[si].rows)    # the ConvTranspose reads frame m + 1 = lengths[b] as zero
            x_raw = ops.alloc_act(B, Lr, C, prec, dev)
            xa = ops.alloc_act(B, Lr + 2 * d0, C, prec, dev)
            up(cur, B, L, out=xa, out_row0=d0, reflect=d0, out_raw=x_raw, phases=r)     # ConvTranspose1d
            if rs is not None:
                ops.reflect_halo(xa, d0, Lr, d0, lengths=rs.rows)          # the right halo at each utterance's end
            if taps is not None:
                taps[f"up{si}"] = packing.act_to_float(x_raw, prec)
            fuse = self.fuse_resblocks and ops.Resblock.eligible(C, Lr, prec)
            for j, (d, c3, k1, fused) in enumerate(blocks):
                if fuse and fused is not None:
                    # block.0-4 + shortcut in one kernel (intermediate in shared memory)
                    run = lambda _f=fused, _xa=xa, _x=x_raw, **kw: _f(_xa, _x, B, Lr, **kw)
                else:
                    h1 = ops.alloc_act(B, Lr, C, prec, dev)
                    c3(xa, B, Lr, out=h1)                                 # block.0-3
                    run = lambda _k1=k1, _h1=h1, _x=x_raw, **kw: _k1([_h1, _x], B, Lr, **kw)   # block.4 + shortcut
                if j + 1 < len(blocks):
                    dn = blocks[j + 1][0]
                    y_raw = ops.alloc_act(B, Lr, C, prec, dev)
                    ya = ops.alloc_act(B, Lr + 2 * dn, C, prec, dev)
                    run(out=ya, out_row0=dn, reflect=dn, out_raw=y_raw)
                    if rs is not None:
                        ops.reflect_halo(ya, dn, Lr, dn, lengths=rs.rows)
                    x_raw, xa = y_raw, ya
                elif si + 1 < n_stage:
                    cur = ops.alloc_act(B, Lr, C, prec, dev)
                    raw = ops.alloc_act(B, Lr, C, prec, dev) if taps is not None else None
                    run(out=cur, out_raw=raw)
                    if taps is not None:
                        taps[f"stage{si}"] = packing.act_to_float(raw, prec)
                else:
                    final = torch.empty(B * Lr, C, dtype=torch.float32, device=dev)
                    raw = ops.alloc_act(B, Lr, C, prec, dev) if taps is not None else None
                    run(out2=final, out_raw=raw)
                    if taps is not None:
                        taps[f"stage{si}"] = packing.act_to_float(raw, prec)
            L = Lr
        last_kw = layers._lengths_kw(rows[-1].rows if rows is not None else None)
        wav = ops.conv_to_mono_tanh(final.view(B, L, -1), plan.w_out, plan.b_out, **last_kw)      # model.22-25
        return wav.unsqueeze(1)
