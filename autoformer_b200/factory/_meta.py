"""Shared implementation of the drop-in MetaPool / MetaConv generators (factory/MetaPool.py, factory/MetaConv.py).

The module tree only holds parameters under the reference's state_dict names; ``forward`` runs on libavc_b200.so:
every Conv1d / Linear / Conv1d(k=1) of the MLP-Mixer is a tcgen05 GEMM (``avc_conv_gemm``), with BatchNorm folded,
ReLU / exact-erf GELU / residual adds in the epilogue; GroupNorm, the pooling token mixer, patchify, LayerNorm and
the layout transposes the mixer needs are fused HBM passes (``csrc/avc_meta.cu``).

Layout note (SURVEY.md Appendix D): the token-mixing MLP contracts over the TOKEN axis, so it runs on Z^T
[dim][tokens]; the channel-mixing MLP contracts over dim and runs on Z [tokens][dim]; ``avc_ln_transpose`` does the
LayerNorm and the transposition in one pass.  Token counts (484, 121, 1849) are zero-padded to multiples of 8 so every
row pitch is a multiple of 16 bytes (TMA) -- the padded weights are zero, so the padding never contributes.
"""
import warnings

import torch
import torch.nn as nn

from .. import layers, ops, packing
from .AutoVC import Postnet
from .Norm import ConvNorm, LinearNorm


def _ceil8(n):
    return (n + 7) // 8 * 8


# ------------------------------------------------------------------------------------------------ parameter containers
class PatchEmbed(nn.Module):
    """factory/Norm.py:63-82: a Conv1d under ``.proj``."""

    def __init__(self, patch_size=5, stride=1, padding=2, in_chans=336, embed_dim=512):
        super().__init__()
        self.proj = nn.Conv1d(in_chans, embed_dim, kernel_size=patch_size, stride=stride, padding=padding)
        self.norm = nn.Identity()


class PreNormResidual(nn.Module):
    """factory/MLPMixer.py:26-33."""

    def __init__(self, dim, fn):
        super().__init__()
        self.fn = fn
        self.norm = nn.LayerNorm(dim)


def _feed_forward(dim, dense):
    return nn.Sequential(dense(dim, dim * 4), nn.GELU(), nn.Dropout(0.0), dense(dim * 4, dim), nn.Dropout(0.0))


def mixer_container(image_size, patch_size, dim, out_dim):
    """Same module indices / parameter names as ``MLPMixer(...)`` (factory/MLPMixer.py:58-92), channels=1, depth=1."""
    num_patches = (image_size // patch_size) ** 2
    conv1 = lambda i, o: nn.Conv1d(i, o, kernel_size=1)
    return nn.Sequential(
        nn.Identity(),                                             # Rearrange (no parameters)
        nn.Linear(patch_size ** 2, dim),
        nn.Sequential(PreNormResidual(dim, _feed_forward(num_patches, conv1)),
                      PreNormResidual(dim, _feed_forward(dim, nn.Linear))),
        nn.Conv1d(num_patches, out_dim, kernel_size=5, padding=2))


def _conv_bn_relu(c_in, c_out):
    return nn.Sequential(ConvNorm(c_in, c_out, kernel_size=5, padding=2, w_init_gain="relu"), nn.BatchNorm1d(c_out),
                         nn.ReLU())


class MetaBlock(nn.Module):
    """factory/MetaPool.py:18-64 (kind="pool") / factory/MetaConv.py:8-63 (kind="conv")."""

    def __init__(self, kind, dim, source_emb=512, crop_len=176, out_dim_neck=88, patch_size=8):
        super().__init__()
        self.norm1 = nn.GroupNorm(1, dim)
        if kind == "conv":
            self.token_mixer = _conv_bn_relu(source_emb, source_emb)
        self.norm2 = nn.GroupNorm(1, crop_len)
        self.conv_1 = _conv_bn_relu(source_emb, crop_len)
        self.mlp = mixer_container(crop_len, patch_size, crop_len, out_dim_neck)
        self.conv_2 = _conv_bn_relu(out_dim_neck, source_emb)


class Encoder(nn.Module):
    def __init__(self, kind, dim_neck, freq, dim, num_layers=3):
        super().__init__()
        self.freq, self.dim_neck = freq, dim_neck
        self.embding = PatchEmbed()
        self.metablock = nn.Sequential(*[MetaBlock(kind, dim) for _ in range(num_layers)])
        self.output_conv = _conv_bn_relu(512, 176)
        self.mlp = mixer_container(176, 16, 176, 2 * dim_neck)


class Decoder(nn.Module):
    def __init__(self, kind, dim, num_layers=1):
        super().__init__()
        self.embding = PatchEmbed(in_chans=176)
        self.metablock = nn.Sequential(*[MetaBlock(kind, dim, crop_len=344, patch_size=8, out_dim_neck=88)
                                         for _ in range(num_layers)])
        self.output_conv_1 = _conv_bn_relu(512, 344)
        self.mlp = mixer_container(344, 8, 344, 88)
        self.output_conv_2 = _conv_bn_relu(344, 176)
        self.linear_projection = LinearNorm(88, 80)


# ------------------------------------------------------------------------------------------------ packed plans
def _pad2(w, rows, cols):
    out = torch.zeros(rows, cols, dtype=torch.float32, device=w.device)
    out[:w.shape[0], :w.shape[1]] = w
    return out


def _pad1(b, n):
    out = torch.zeros(n, dtype=torch.float32, device=b.device)
    out[:b.shape[0]] = b
    return out


class MixerPlan:
    def __init__(self, sd, prefix, image, patch, out_dim, precision):
        f = lambda k: sd[f"{prefix}.{k}"].float()
        self.precision = precision
        self.S, self.p, self.dim, self.out_dim = image, patch, image, out_dim
        self.np = (image // patch) ** 2
        self.np8 = _ceil8(self.np)
        self.h8 = _ceil8(4 * self.np)
        pl = lambda w, b, act="none": ops.ConvGemm(*packing.pack_linear(w, b, precision), act=act, tag="mixer")
        self.embed = pl(f("1.weight"), f("1.bias"))
        self.ln1 = (f("2.0.norm.weight").contiguous(), f("2.0.norm.bias").contiguous())
        self.tok1 = pl(_pad2(f("2.0.fn.0.weight")[:, :, 0], self.h8, self.np8), _pad1(f("2.0.fn.0.bias"), self.h8), "gelu")
        self.tok2 = pl(_pad2(f("2.0.fn.3.weight")[:, :, 0], self.np8, self.h8), _pad1(f("2.0.fn.3.bias"), self.np8))
        self.ln2 = (f("2.1.norm.weight").contiguous(), f("2.1.norm.bias").contiguous())
        self.ch1 = pl(f("2.1.fn.0.weight"), f("2.1.fn.0.bias"), "gelu")
        self.ch2 = pl(f("2.1.fn.3.weight"), f("2.1.fn.3.bias"))
        wc = f("3.weight")                                              # (out, np, 5)
        wcp = torch.zeros(wc.shape[0], self.np8, 5, dtype=torch.float32, device=wc.device)
        wcp[:, :self.np] = wc
        self.conv = ops.ConvGemm(*packing.pack_conv(wcp, f("3.bias"), precision), tag="mixer")

    def __call__(self, a, B, stats=None, gn=None, want_op=True, want_f32=False):
        """a [B][S][S] fp32 channels-last (rows = length, columns = channels) -> mixer output [B][S][out_dim]."""
        prec, dev = self.precision, a.device
        S, dim, np_, np8, h8 = self.S, self.dim, self.np, self.np8, self.h8
        tk = ops.patchify(a, stats, gn[0] if gn else None, gn[1] if gn else None, self.p, prec)
        z = torch.empty(B * np_, dim, dtype=torch.float32, device=dev)
        self.embed(tk, B, np_, out2=z)                                           # Linear(p^2 -> dim)
        y1t, zt = ops.ln_transpose(z.view(B, np_, dim), self.ln1[0], self.ln1[1], 1, prec, want_f32=True)
        g = ops.alloc_act(B, dim, h8, prec, dev)
        self.tok1(y1t, B, dim, out=g)                                            # tokens -> 4*tokens, GELU
        z2t = torch.empty(B * dim, np8, dtype=torch.float32, device=dev)
        self.tok2(g, B, dim, out2=z2t, residual=zt.view(B * dim, np8))           # back to tokens, + Z
        y2, z2 = ops.ln_transpose(z2t.view(B, dim, np8), self.ln2[0], self.ln2[1], 2, prec, want_f32=True)
        v = ops.alloc_act(B, np8, 4 * dim, prec, dev)
        self.ch1(y2, B, np8, out=v)                                              # dim -> 4*dim, GELU
        z3 = torch.empty(B * np8, dim, dtype=torch.float32, device=dev)
        self.ch2(v, B, np8, out2=z3, residual=z2.view(B * np8, dim))             # back to dim, + Z
        z3t, _ = ops.ln_transpose(z3.view(B, np8, dim), None, None, 0, prec)
        out_op = ops.alloc_act(B, dim, self.out_dim, prec, dev) if want_op else None
        out_f32 = torch.empty(B * dim, self.out_dim, dtype=torch.float32, device=dev) if want_f32 else None
        self.conv(z3t, B, dim, out=out_op, out2=out_f32)                         # Conv1d(tokens -> out, k5) over dim
        return out_op, out_f32


class BlockPlan:
    def __init__(self, sd, prefix, kind, crop, precision, bn_owner=None):
        f = lambda k: sd[f"{prefix}.{k}"].float().contiguous()
        self.kind, self.crop, self.precision = kind, crop, precision
        self.gn1 = (f("norm1.weight"), f("norm1.bias"))
        self.gn2 = (f("norm2.weight"), f("norm2.bias"))
        if kind == "conv":
            self.token_mixer = layers.conv_bn_layer(sd, f"{prefix}.token_mixer", precision, "relu", bn_owner)
        self.conv_1 = layers.conv_bn_layer(sd, f"{prefix}.conv_1", precision, "relu", bn_owner)
        self.mlp = MixerPlan(sd, f"{prefix}.mlp", crop, 8, 88, precision)
        self.conv_2 = layers.conv_bn_layer(sd, f"{prefix}.conv_2", precision, "relu", bn_owner)

    def __call__(self, x, B, L, want_op):
        """x fp32 [B][L][512] -> (x' fp32, x' operand format or None)   (MetaBlock.forward, MetaPool.py:66-77)."""
        prec, dev = self.precision, x.device
        assert L == self.crop, f"MetaBlock(crop_len={self.crop}) needs length {self.crop}, got {L}"
        st1 = ops.gn_stats(x, B)
        if self.kind == "pool":
            x1, x1_op = ops.gn_pool_residual(x, st1, self.gn1[0], prec)
        else:
            n1 = ops.gn_apply(x, st1, self.gn1[0], self.gn1[1], prec)
            x1 = torch.empty_like(x)
            x1_op = ops.alloc_act(B, L, 512, prec, dev)
            self.token_mixer(n1, B, L, out=x1_op, out2=x1.view(B * L, 512), residual=x.view(B * L, 512), res_after=True)
        a = torch.empty(B, L, self.crop, dtype=torch.float32, device=dev)
        self.conv_1(x1_op, B, L, out2=a.view(B * L, self.crop))
        st2 = ops.gn_stats(a, B)
        m_op, _ = self.mlp(a, B, stats=st2, gn=self.gn2)
        x2 = torch.empty_like(x)
        x2_op = ops.alloc_act(B, L, 512, prec, dev) if want_op else None
        self.conv_2(m_op, B, L, out=x2_op, out2=x2.view(B * L, 512), residual=x1.view(B * L, 512), res_after=True)
        return x2, x2_op


class _Plan:
    def __init__(self, model, kind, precision, bn_owner=None):
        sd = layers.state_for_packing(model)
        self.precision = precision
        emb = lambda p: ops.ConvGemm(*packing.pack_conv(sd[p + ".weight"].float(), sd[p + ".bias"].float(), precision),
                                     tag="conv")
        self.enc_embed = emb("encoder.embding.proj")
        self.enc_blocks = [BlockPlan(sd, f"encoder.metablock.{i}", kind, 176, precision, bn_owner) for i in range(3)]
        self.enc_out_conv = layers.conv_bn_layer(sd, "encoder.output_conv", precision, "relu", bn_owner)
        self.enc_mlp = MixerPlan(sd, "encoder.mlp", 176, 16, 2 * model.dim_neck, precision)
        self.dec_embed = emb("decoder.embding.proj")
        self.dec_block = BlockPlan(sd, "decoder.metablock.0", kind, 344, precision, bn_owner)
        self.dec_out_conv_1 = layers.conv_bn_layer(sd, "decoder.output_conv_1", precision, "relu", bn_owner)
        self.dec_mlp = MixerPlan(sd, "decoder.mlp", 344, 8, 88, precision)
        self.dec_out_conv_2 = layers.conv_bn_layer(sd, "decoder.output_conv_2", precision, "relu", bn_owner)
        self.linear = ops.ConvGemm(*packing.pack_linear(sd["decoder.linear_projection.linear_layer.weight"],
                                                        sd["decoder.linear_projection.linear_layer.bias"], precision),
                                   tag="linear")
        self.postnet = layers.Postnet(sd, "postnet", precision, bn_owner)


class MetaBase(layers.PlanOwner, nn.Module):
    KIND = None

    def __init__(self, dim_neck, dim, dim_pre, freq):
        super().__init__()
        self.encoder = Encoder(self.KIND, dim_neck, freq, dim_pre)
        self.decoder = Decoder(self.KIND, dim_pre)
        self.postnet = Postnet()
        self.dim_neck, self.freq = dim_neck, freq
        self.precision = "fp32"
        self.collect_taps = False
        self.taps = {}
        self.bn_stats = "running"       # "batch": train-mode BatchNorm statistics (see autoformer_b200.AutoVC)
        self._cache = layers.PlanCache()
        self._warned_train = False

    def _plan(self):
        batch = layers.check_bn_stats(self.bn_stats) == "batch"
        return self._cache.get(self, (self.precision, self.bn_stats),
                               lambda: _Plan(self, self.KIND, self.precision, self if batch else None),
                               skip_bn_stats=batch)

    # hooks of the AdaIN "2" variants (factory/_adain.py)
    def _encoder_features(self, x, plan, B, T):
        return x

    def _run_postnet(self, plan, mel_op, mel, B, T, taps):
        return plan.postnet(mel_op, mel, B, T, taps)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, c_org, c_trg):
        if self.training and not self._warned_train and self.bn_stats != "batch":
            warnings.warn("autoformer_b200 Meta models run the eval-mode forward (BatchNorm running statistics); "
                          "bn_stats='batch' selects train-mode BatchNorm statistics")
            self._warned_train = True
        if x.dim() == 4:
            x = x.squeeze(1)
        ops._require_cuda(x)
        x = x.contiguous().float()
        c_org = c_org.contiguous().float()
        B, T, _ = x.shape
        F, H = self.freq, self.dim_neck
        E = c_org.shape[1]
        # the reference hard-wires these shapes (PatchEmbed(in_chans=336 / 176), crop_len 176 / 344; SURVEY.md 0.2)
        if T != 176 or 80 + E != 336 or 2 * H + E != 344:
            raise RuntimeError(f"Meta models need T=176, dim_emb=256, dim_neck=44 (got T={T}, dim_emb={E}, dim_neck={H}): "
                               "channel mismatch in PatchEmbed, as in the reference")
        if T % F != 0:
            raise IndexError(f"T={T} is not a multiple of freq={F}")
        layers.check_bn_stats(self.bn_stats)
        plan = self._plan()
        prec, dev = plan.precision, x.device
        taps = self.taps if self.collect_taps else None
        if taps is not None:
            taps.clear()

        # ---- encoder (MetaPool.py:109-133)
        x = self._encoder_features(x, plan, B, T)
        h = ops.concat_bcast(x, c_org, T, 1, prec)
        xe = torch.empty(B, T, 512, dtype=torch.float32, device=dev)
        plan.enc_embed(h, B, T, out2=xe.view(B * T, 512))
        if taps is not None:
            taps["enc_embed"] = xe.clone()
        x_op = None
        for i, blk in enumerate(plan.enc_blocks):
            xe, x_op = blk(xe, B, T, want_op=i == len(plan.enc_blocks) - 1)
            if taps is not None:
                taps[f"encoder.metablock.{i}"] = xe
        a = torch.empty(B, T, 176, dtype=torch.float32, device=dev)
        plan.enc_out_conv(x_op, B, T, out2=a.view(B * T, 176))
        _, enc_out = plan.enc_mlp(a, B, want_op=False, want_f32=True)              # [B*176][2H]
        enc_out = enc_out.view(B, T, 2 * H)
        if taps is not None:
            taps["enc_out"] = enc_out
        codes = ops.gather_codes(enc_out, H, F)
        flat_codes = codes.reshape(B, -1)
        if taps is not None:
            taps["codes"] = flat_codes
        if c_trg is None:
            return flat_codes

        # ---- decoder (MetaPool.py:160-182): the (B, T, 2H+E) tensor is read as channels = T, length = 2H+E
        c_trg = c_trg.contiguous().float()
        Ld = 2 * H + E
        di = ops.meta_decoder_input(codes, c_trg, T, F, prec)                       # [B][344][176]
        xd = torch.empty(B, Ld, 512, dtype=torch.float32, device=dev)
        plan.dec_embed(di, B, Ld, out2=xd.view(B * Ld, 512))
        xd, xd_op = plan.dec_block(xd, B, Ld, want_op=True)
        if taps is not None:
            taps["decoder.metablock.0"] = xd
        a = torch.empty(B, Ld, 344, dtype=torch.float32, device=dev)
        plan.dec_out_conv_1(xd_op, B, Ld, out2=a.view(B * Ld, 344))
        _, m = plan.dec_mlp(a, B, want_op=False, want_f32=True)                     # [B*344][88]
        mt, _ = ops.ln_transpose(m.view(B, Ld, 88), None, None, 0, prec)           # x.transpose(2, 1): [B][88][344]
        c2 = torch.empty(B, 88, 176, dtype=torch.float32, device=dev)
        plan.dec_out_conv_2(mt, B, 88, out2=c2.view(B * 88, 176))
        if taps is not None:
            taps["dec_conv2"] = c2
        c2t, _ = ops.ln_transpose(c2, None, None, 0, prec)                          # [B][176][88]
        mel = torch.empty(B, T, 80, dtype=torch.float32, device=dev)
        mel_op = ops.alloc_act(B, T, 80, prec, dev)
        plan.linear(c2t, B, T, out=mel_op, out2=mel.view(B * T, 80))               # Linear(88 -> 80)

        post = self._run_postnet(plan, mel_op, mel, B, T, taps)
        if taps is not None:
            taps["mel"] = mel
            taps["mel_postnet"] = post
        return mel.unsqueeze(1), post.unsqueeze(1), flat_codes
