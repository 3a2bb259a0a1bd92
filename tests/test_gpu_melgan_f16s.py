"""GPU parity of the round-2 MelGAN precision "fp16s" (residual stream / ConvTranspose operands / ResnetBlock intermediate
as two fp16 terms, the k3 operand as one fp16 value) and of its fused ResnetBlock kernel avc_resblock2."""
import os
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import rel_l2, templates
from oracle.melgan import melgan_forward
from oracle.seeded import seeded_state_dict, synthetic_mel

pytestmark = pytest.mark.gpu
warnings.filterwarnings("ignore", category=FutureWarning)
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("C,d,B,L", [(64, 1, 2, 256), (64, 9, 1, 384), (32, 3, 3, 128), (32, 9, 2, 640), (64, 3, 150, 128),
                                     (32, 1, 700, 128), (64, 9, 2, 128 * 37), (32, 3, 2, 128 * 37),
                                     (128, 1, 2, 256), (128, 9, 1, 384), (128, 3, 3, 128), (128, 3, 301, 128),
                                     (128, 9, 2, 128 * 41)])
def test_resblock2_matches_torch(C, d, B, L):
    """avc_resblock2 (melgan/modules.py:72-85 in one kernel, reading only the raw stream) against torch fp64 with the
    operands rounded where the kernel rounds them: the raw output with the next block's reflected halo, the activated
    two-term output, the fp32 output; more tiles than CTAs (B = 150 / 700), many tiles per utterance (L = 37 x 128:
    both window buffers of every CTA are recycled)."""
    from autoformer_b200 import ops, packing
    torch.manual_seed(100 * C + d)
    w3, w1, wsc = torch.randn(C, C, 3) / (3 * C) ** 0.5, torch.randn(C, C, 1) / C ** 0.5, torch.randn(C, C, 1) / C ** 0.5
    b3, b1, bsc = torch.randn(C), torch.randn(C), torch.randn(C)
    x = torch.randn(B, L, C) * 3.0
    xpad = F.pad(x.transpose(1, 2), (d, d), mode="reflect").transpose(1, 2).contiguous()
    x_op = packing.to_act(xpad, "fp16s")                                     # [B][L + 2d][2C], halo rows included
    xs = packing.act_to_float(x_op, "fp16s").double()                        # what the kernel actually reads
    xa = F.leaky_relu(xs, 0.2).float().half().double()                       # its k3 operand: ONE fp16 value
    mid = F.leaky_relu(F.conv1d(xa.transpose(1, 2), w3.double(), b3.double(), dilation=d), 0.2)
    mid = packing.act_to_float(packing.to_act(mid.transpose(1, 2).float(), "fp16s"), "fp16s").double().transpose(1, 2)
    y = (F.conv1d(mid, w1.double(), b1.double())
         + F.conv1d(xs[:, d:d + L].transpose(1, 2), wsc.double(), bsc.double())).transpose(1, 2)
    ya = F.leaky_relu(y, 0.2)
    blk = ops.Resblock2(*packing.pack_resblock2(w3, b3, w1, b1, wsc, bsc), dilation=d).to("cuda")
    R = 9
    xd = x_op.cuda()
    raw = torch.zeros(B, L + 2 * R, 2 * C, dtype=torch.float16, device="cuda")
    blk(xd, B, L, y=raw, y_row0=R, y_reflect=R)
    act = torch.zeros(B, L, 2 * C, dtype=torch.float16, device="cuda")
    blk(xd, B, L, y=act, y_act=True)
    torch.cuda.synchronize()
    padded = F.pad(y.transpose(1, 2), (R, R), mode="reflect").transpose(1, 2)
    assert rel_l2(packing.act_to_float(raw, "fp16s"), padded) < 2e-5, rel_l2(packing.act_to_float(raw, "fp16s"), padded)
    assert rel_l2(packing.act_to_float(act, "fp16s"), ya) < 2e-5
    # determinism: a second run is bit-identical
    again = torch.zeros_like(act)
    blk(xd, B, L, y=again, y_act=True)
    assert torch.equal(again, act)
    if C == 128:                      # the wide kernel writes the two-term forms only (never the last stage)
        return
    out2 = torch.zeros(B * L, C, device="cuda")
    blk(xd, B, L, out2=out2)
    assert rel_l2(out2.view(B, L, C), ya) < 2e-5
    if C == 32:
        _check_wav_epilogue(blk, xd, B, L, d, xa, xs, mid, ya, w3, b3, w1, wsc)


def _check_wav_epilogue(blk, xd, B, L, d, xa, xs, mid, ya, w3, b3, w1, wsc):
    """The generator's output layer fused into the block's epilogue (wav=, mono=): tanh(Conv1d(C -> 1, K)) over
    ReflectionPad1d(K // 2) of LeakyReLU(y), run over 128-row tiles that overlap by K - 1.  Every sample is held to a
    worst-case bound -- the first and last K // 2 of each utterance (mirrored rows) and both sides of every tile seam
    included -- so an error confined to the seams or the ends shows, which the waveform's rel-L2 cannot see."""
    U = 2.0 ** -23
    C = ya.shape[2]
    # per-element bound on the staged LeakyReLU(y): the k3 sums (one fp16 operand x two fp16 weight terms), the two-term
    # rounding of the intermediate (which may round the other way), then block.4 + shortcut over the stored operands
    s3 = F.conv1d(xa.abs().transpose(1, 2), w3.double().abs(), b3.double().abs(), dilation=d)
    # LeakyReLU of a negative operand is 0.2f * x in fp32 on the device, 0.2 * x in fp64 here: the one-fp16 operand may
    # round to the neighbouring value (one fp16 ulp, 2^-11 relative)
    neg = F.conv1d((xa.abs() * (xs < 0)).transpose(1, 2), w3.double().abs(), dilation=d)
    e_mid = (3 * 2 * C + 2) * U * s3 + 2.0 ** -11 * neg
    e_mid = e_mid + 2 * (2.0 ** -22 * (mid.abs() + e_mid) + 2.0 ** -25)
    s1 = F.conv1d(mid.abs(), w1.double().abs()) + F.conv1d(xs[:, d:d + L].abs().transpose(1, 2), wsc.double().abs())
    s1 = s1 + blk.bias1.double().abs().cpu().view(1, C, 1)
    e_y = (F.conv1d(e_mid, w1.double().abs()) + (4 * 2 * C + 2) * U * s1).transpose(1, 2)
    e_a = e_y + 2 * U * ya.abs()
    for K in (3, 5, 7):
        g = torch.Generator().manual_seed(K)
        w_out = torch.randn(K, C, generator=g) / (K * C) ** 0.5
        b_out = 0.05 * K
        wav = torch.full((B, L), float("nan"), device="cuda")
        blk(xd, B, L, wav=wav, mono=(w_out.cuda(), b_out))
        torch.cuda.synchronize()
        pad = lambda t: F.pad(t.transpose(1, 2), (K // 2, K // 2), mode="reflect")
        wk = w_out.double().t().unsqueeze(0)                                  # (1, C, K)
        v = F.conv1d(pad(ya), wk).squeeze(1) + b_out
        s = F.conv1d(pad(ya).abs(), wk.abs()).squeeze(1) + abs(b_out)
        bound = F.conv1d(pad(e_a), wk.abs()).squeeze(1) + (K * C + 2) * U * s + 2e-6    # tanh_fast: ~1e-7 absolute
        got = wav.cpu().double()
        assert bool(torch.isfinite(got).all()), K
        err = (got - torch.tanh(v)).abs()
        stride = 128 - (K - 1)
        edges = sorted({*range(K // 2), *range(L - K // 2, L)} | {t for j in range(1, L // stride + 1)
                                                                  for t in (j * stride - 1, j * stride) if t < L})
        assert bool((err[:, edges] <= bound[:, edges]).all()), (K, "utterance ends / tile seams", float(err[:, edges].max()))
        bad = err > bound
        assert not bool(bad.any()), (K, bad.nonzero()[:5].tolist(), float((err - bound).max()))


@pytest.mark.parametrize("name", ["melgan_b1_t40", "melgan_b2_t17"])
def test_melgan_f16s_parity_and_golden(name):
    from autoformer_b200.melgan.modules import Generator
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    B, T = int(g["B"]), int(g["T"])
    sd = seeded_state_dict(templates.melgan_template(), int(g["wseed"]))
    mel = synthetic_mel(B, T, int(g["xseed"])).transpose(1, 2).contiguous()
    rt = {}
    ref = melgan_forward(sd, mel, taps=rt)
    gen = Generator(80, 32, 3)
    gen.load_state_dict(sd)
    gen = gen.cuda().eval()
    gen.precision = "fp16s"
    gen.collect_taps = True
    wav = gen(mel.cuda())
    assert wav.shape == (B, 1, 256 * T)
    errs = {k: rel_l2(gen.taps[k], rt[k].transpose(1, 2)) for k in ("up0", "stage0", "up1", "stage1", "up2", "stage2", "up3", "stage3")}
    errs["wav"] = rel_l2(wav, ref)
    print("fp16s", name, errs)
    assert all(e < 1e-3 for e in errs.values()), errs
    assert rel_l2(wav, torch.from_numpy(g["wav"])) < 1e-3                # the unmodified reference's waveform
    # fused and layer-wise paths are the same arithmetic up to summation order and the fp16 rounding of the operand
    gen.collect_taps = False
    gen.fuse_resblocks = False
    assert rel_l2(gen(mel.cuda()), wav) < 5e-4
    gen.fuse_resblocks = True
    assert rel_l2(gen(mel.flip(2).contiguous().cuda()), ref) > 1e-2       # negative control


@pytest.mark.parametrize("seed", [5, 9])
def test_melgan_f16s_margin_on_the_hard_seeds(seed):
    """The weight seeds on which ONE fp16 value per activation ("fp16x2") misses the 1e-3 gate
    (scripts/melgan_precision_study.py: 1.16e-3 / 1.22e-3): "fp16s" must keep a margin there."""
    from autoformer_b200.melgan.modules import Generator
    sd = seeded_state_dict(templates.melgan_template(), seed)
    mel = synthetic_mel(2, 48, 100 + seed).transpose(1, 2).contiguous()
    ref = melgan_forward(sd, mel, dtype=torch.float64)
    gen = Generator(80, 32, 3)
    gen.load_state_dict(sd)
    gen = gen.cuda().eval()
    gen.precision = "fp16s"
    err = rel_l2(gen(mel.cuda()), ref)
    print("fp16s seed", seed, "waveform rel-L2", err)
    assert err < 7e-4, err


def test_melgan_f16s_full_size_b32_t1000():
    from autoformer_b200.melgan.modules import Generator
    sd = seeded_state_dict(templates.melgan_template(), 4)
    B, T = 32, 1000
    mel = synthetic_mel(B, T, 51).transpose(1, 2).contiguous()
    gen = Generator(80, 32, 3)
    gen.load_state_dict(sd)
    gen = gen.cuda().eval()
    gen.precision = "fp16s"
    wav = gen(mel.cuda())
    assert wav.shape == (B, 1, 256 * T) and bool(torch.isfinite(wav).all())
    idx = [0, 31]
    ref = melgan_forward(sd, mel[idx])
    err = rel_l2(wav[idx], ref)
    print("MelGAN fp16s waveform rel-L2 at B=32, T=1000:", err)
    assert err < 1e-3, err
    alone = gen(mel[idx].cuda())
    assert rel_l2(alone, wav[idx]) < 5e-4
    assert rel_l2(gen(mel[idx].flip(2).contiguous().cuda()), ref) > 1e-2
