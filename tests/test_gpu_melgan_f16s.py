"""GPU parity of the round-2 MelGAN precision "fp16s" (residual stream / ConvTranspose operands / ResnetBlock intermediate
as two fp16 terms, the k3 operand as one fp16 value).  The fused ResnetBlock kernel avc_resblock2 itself is held to an
element-wise contract in test_gpu_resblock_contract.py."""
import os
import warnings

import numpy as np
import pytest
import torch

from oracle import rel_l2, templates
from oracle.melgan import melgan_forward
from oracle.seeded import seeded_state_dict, synthetic_mel

pytestmark = pytest.mark.gpu
warnings.filterwarnings("ignore", category=FutureWarning)
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


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
