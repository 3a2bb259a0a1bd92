"""Variable-length MelGAN batches on the B200: the lengths-aware glue kernels, the compacted-tile instantiations of the
fused ResnetBlock kernels and the Generator / pipeline paths.  Where the batch cropped to an utterance's length takes the
same kernels, the ragged run must be BIT-identical to the existing fixed-length call on it; otherwise it is held to the
bound the fixed-length kernel is held to against fp64.  Padded input frames hold NaN throughout: none may reach a valid
output."""
import warnings

import pytest
import torch
import torch.nn.functional as F

from oracle import rel_l2, templates
from oracle.melgan import melgan_forward
from oracle.seeded import seeded_state_dict, synthetic_mel

pytestmark = pytest.mark.gpu
warnings.filterwarnings("ignore", category=FutureWarning)

DEV = "cuda"
NAN = float("nan")
# waveform gates of the MelGAN parity tests (tests/test_gpu_parity.py, tests/test_gpu_melgan_f16s.py)
GATE = {"fp32": 1e-3, "tf32": 5e-3, "bf16": 5e-2, "fp16x2": 2e-3, "fp16s": 1e-3}


def _dev_lengths(vals):
    return torch.tensor(vals, dtype=torch.int32, device=DEV)


def _bits(t):
    """Bit pattern of a tensor (NaN == NaN)."""
    return t.view({2: torch.int16, 4: torch.int32}[t.element_size()])


def _generator(precision, seed=4):
    from autoformer_b200.melgan.modules import Generator
    sd = seeded_state_dict(templates.melgan_template(), seed)
    g = Generator(80, 32, 3)
    g.load_state_dict(sd)
    g = g.to(DEV).eval()
    g.precision = precision
    return g, sd


# ------------------------------------------------------------------------------------------------ avc_reflect_halo
@pytest.mark.parametrize("dtype,width", [(torch.float16, 64), (torch.float16, 256), (torch.bfloat16, 128),
                                         (torch.float32, 80)])
@pytest.mark.parametrize("reflect", [1, 3, 9])
def test_reflect_halo_lengths(dtype, width, reflect):
    from autoformer_b200 import ops
    B, L, row0 = 5, 200, reflect + 2
    lengths = [200, reflect + 1, 77, 128, 199]
    buf = torch.full((B, row0 + L + reflect + 3, width), NAN, dtype=dtype, device=DEV)
    for b, n in enumerate(lengths):
        buf[b, row0:row0 + n] = torch.randn(n, width, device=DEV).to(dtype)
    before = buf.clone()
    ops.reflect_halo(buf, row0, L, reflect, lengths=_dev_lengths(lengths))
    torch.cuda.synchronize()
    expect = before.clone()
    for b, n in enumerate(lengths):
        for k in range(1, reflect + 1):
            expect[b, row0 - k] = before[b, row0 + k]
            expect[b, row0 + n - 1 + k] = before[b, row0 + n - 1 - k]
    assert torch.equal(_bits(buf), _bits(expect))          # mirrored rows exact, every other row untouched (NaN stays)
    # lengths all L: the call without lengths, bit for bit
    full = before.clone()
    full[:, row0:row0 + L] = torch.randn(B, L, width, device=DEV).to(dtype)
    a, c = full.clone(), full.clone()
    ops.reflect_halo(a, row0, L, reflect)
    ops.reflect_halo(c, row0, L, reflect, lengths=_dev_lengths([L] * B))
    torch.cuda.synchronize()
    assert torch.equal(_bits(a), _bits(c))


# ------------------------------------------------------------------------------------------------ avc_conv_to_mono_tanh
@pytest.mark.parametrize("C,K", [(32, 7), (32, 3), (64, 5)])
def test_conv_to_mono_tanh_lengths(C, K):
    from autoformer_b200 import ops
    torch.manual_seed(C + K)
    B, L = 5, 700
    lengths = [700, 4, 256, 513, 255]
    x = torch.randn(B, L, C, device=DEV) * 0.5
    for b, n in enumerate(lengths):
        x[b, n:] = NAN
    w, bias = torch.randn(K, C, device=DEV) / C ** 0.5, 0.1
    out = ops.conv_to_mono_tanh(x, w, bias, lengths=_dev_lengths(lengths))
    torch.cuda.synchronize()
    for b, n in enumerate(lengths):
        alone = ops.conv_to_mono_tanh(x[b:b + 1, :n].contiguous(), w, bias)
        torch.cuda.synchronize()
        assert torch.equal(out[b, :n], alone[0]), b           # reflected at the utterance's own end
        assert torch.equal(out[b, n:], torch.zeros(L - n, device=DEV))


# ------------------------------------------------------------------------------------------------ avc_resblock2
def _block(C, d, seed):
    from autoformer_b200 import ops, packing
    g = torch.Generator().manual_seed(seed)
    w3 = torch.randn(C, C, 3, generator=g) / (3 * C) ** 0.5
    w1, wsc = torch.randn(C, C, 1, generator=g) / C ** 0.5, torch.randn(C, C, 1, generator=g) / C ** 0.5
    b3, b1, bsc = torch.randn(C, generator=g), torch.randn(C, generator=g), torch.randn(C, generator=g)
    blk = ops.Resblock2(*packing.pack_resblock2(w3, b3, w1, b1, wsc, bsc), dilation=d).to(DEV)
    return blk, (w3, b3, w1, b1, wsc, bsc)


def _ref_block(x_op, n, d, weights):
    """fp64 reference of one utterance (operands rounded where the kernel rounds them, as test_resblock2_matches_torch):
    y and LeakyReLU(y), (n, C)."""
    from autoformer_b200 import packing
    w3, b3, w1, b1, wsc, bsc = (t.double() for t in weights)
    xs = packing.act_to_float(x_op.cpu(), "fp16s").double()[:n + 2 * d]
    xa = F.leaky_relu(xs, 0.2).float().half().double()
    mid = F.leaky_relu(F.conv1d(xa.t()[None], w3, b3, dilation=d), 0.2)
    mid = packing.act_to_float(packing.to_act(mid[0].t().float(), "fp16s"), "fp16s").double().t()[None]
    y = (F.conv1d(mid, w1, b1) + F.conv1d(xs[d:d + n].t()[None], wsc, bsc))[0].t()
    return y, F.leaky_relu(y, 0.2)


@pytest.mark.parametrize("C", [32, 64, 128])
@pytest.mark.parametrize("d", [1, 3, 9])
def test_resblock2_ragged(C, d):
    """Compacted tiles: rows < L_b bit-identical to the fixed-length kernel on the utterance cropped to L_b where that
    crop is a multiple of 128, within the fp64 bound otherwise; output rows of tiles at or past L_b never written (the
    NaN sentinel survives); input rows past L_b + d are NaN."""
    from autoformer_b200 import ops, packing
    B, L, R = 4, 384, 9
    lengths = [384, 256, 200, 37]
    blk, weights = _block(C, d, 10 * C + d)
    g = torch.Generator().manual_seed(C * d)
    x = torch.full((B, L + 2 * d, 2 * C), NAN, dtype=torch.float16)
    crops = []
    for b, n in enumerate(lengths):
        v = torch.randn(n, C, generator=g) * 3.0
        xp = F.pad(v.t()[None], (d, d), mode="reflect")[0].t()
        x[b, :n + 2 * d] = packing.to_act(xp[None].contiguous(), "fp16s")[0]
        crops.append(x[b, :n + 2 * d].clone()[None])          # (a fresh [1][n + 2d][2C] buffer, dense strides)
    xd = x.to(DEV)
    rows = ops.ragged_rows(lengths, (1,), (128, 122), DEV)[0]
    kinds = ["y", "y_act"] + (["out2"] if C < 128 else []) + (["wav"] if C == 32 else [])
    w_out = torch.randn(7, C, generator=g) / (7 * C) ** 0.5
    mono = (w_out.to(DEV), 0.05)
    for kind in kinds:
        if kind.startswith("y"):
            out = torch.full((B, L + 2 * R, 2 * C), NAN, dtype=torch.float16, device=DEV)
            kw = dict(y=out, y_row0=R, y_reflect=R) if kind == "y" else dict(y=out, y_act=True)
            row0 = R if kind == "y" else 0
        elif kind == "out2":
            out = torch.full((B * L, C), NAN, device=DEV)
            kw = dict(out2=out)
        else:
            out = torch.full((B, L), NAN, device=DEV)
            kw = dict(wav=out, mono=mono)
        blk(xd, B, L, lengths=rows, **kw)
        torch.cuda.synchronize()
        for b, n in enumerate(lengths):
            if kind == "wav":
                stride = 122
                ran = min(L, -(-n // stride) * stride)
                got = out[b, :n].cpu()
                assert torch.equal(out[b, n:ran].cpu(), torch.zeros(ran - n)), (kind, b)
                assert torch.isnan(out[b, ran:]).all(), (kind, b)
            else:
                ran = -(-n // 128) * 128
                if kind == "out2":
                    v = out.view(B, L, C)[b]
                    got, skipped = v[:n].cpu().double(), v[ran:]
                else:
                    v = out[b]
                    got = packing.act_to_float(v[row0:row0 + n].cpu(), "fp16s").double()
                    skipped = v[row0 + ran:row0 + L]
                assert torch.isnan(skipped.float()).all(), (kind, b)       # tiles past the end never ran
            if n % 128 == 0:
                # the fixed-length kernel on the utterance alone: same tiles, same arithmetic
                if kind.startswith("y"):
                    ref = torch.full((1, n + 2 * R, 2 * C), NAN, dtype=torch.float16, device=DEV)
                    blk(crops[b].to(DEV), 1, n, **{**kw, "y": ref})
                    torch.cuda.synchronize()
                    assert torch.equal(_bits(out[b, row0:row0 + n]), _bits(ref[0, row0:row0 + n])), (kind, b)
                elif kind == "out2":
                    ref = torch.full((n, C), NAN, device=DEV)
                    blk(crops[b].to(DEV), 1, n, out2=ref)
                    torch.cuda.synchronize()
                    assert torch.equal(out.view(B, L, C)[b, :n], ref), (kind, b)
                else:
                    ref = torch.full((1, n), NAN, device=DEV)
                    blk(crops[b].to(DEV), 1, n, wav=ref, mono=mono)
                    torch.cuda.synchronize()
                    assert torch.equal(out[b, :n], ref[0]), (kind, b)
            else:
                y, ya = _ref_block(x[b], n, d, weights)
                if kind == "wav":
                    tau = torch.arange(n)[:, None] + torch.arange(7)[None, :] - 3
                    tau = torch.where(tau < 0, -tau, tau)
                    tau = torch.where(tau >= n, 2 * (n - 1) - tau, tau)
                    want = torch.tanh((ya[tau] * w_out.double()[None]).sum(dim=(1, 2)) + 0.05)
                    assert rel_l2(got, want) < 5e-5 and (got.double() - want).abs().max() < 1e-4, (kind, b)
                else:
                    want = y if kind == "y" else ya
                    assert rel_l2(got, want) < 2e-5, (kind, b, rel_l2(got, want))


# ------------------------------------------------------------------------------------------------ Generator
@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16", "fp16x2", "fp16s"])
def test_generator_ragged(precision):
    g, sd = _generator(precision)
    lengths = [48, 4, 31, 20, 47, 10, 33]
    B, T = len(lengths), max(lengths)
    clean = synthetic_mel(B, T, 12).transpose(1, 2).contiguous()
    mel = clean.clone()
    for b, n in enumerate(lengths):
        mel[b, :, n:] = NAN
    wav = g(mel.to(DEV), lengths=lengths)
    torch.cuda.synchronize()
    assert wav.shape == (B, 1, 256 * T) and torch.isfinite(wav).all()
    for b, n in enumerate(lengths):
        assert torch.equal(wav[b, :, 256 * n:], torch.zeros(1, 256 * (T - n), device=DEV)), b
        if n % 2 == 0:
            # the batch cropped to n takes the same kernels (every fused stage eligible): bit-identical
            crop = g(clean[:, :, :n].contiguous().to(DEV))
            torch.cuda.synchronize()
            assert torch.equal(wav[b, :, :256 * n], crop[b]), (precision, b, n)
        else:
            ref = melgan_forward(sd, clean[b:b + 1, :, :n])
            assert rel_l2(wav[b:b + 1, :, :256 * n], ref) < GATE[precision], (precision, b, n)
    # negative control: the padded batch without lengths, trimmed, misses the gate on the last frames of a short one
    padded = clean.clone()
    for b, n in enumerate(lengths):
        padded[b, :, n:] = 0
    plain = g(padded.to(DEV))
    b, n = 2, lengths[2]
    ref = melgan_forward(sd, clean[b:b + 1, :, :n])
    tail = slice(256 * (n - 2), 256 * n)
    assert rel_l2(plain[b:b + 1, :, tail], ref[:, :, tail]) > GATE[precision]
    assert rel_l2(wav[b:b + 1, :, tail], ref[:, :, tail]) < 5 * GATE[precision]
    if precision == "fp32":
        from autoformer_b200.melgan.interface import MelVocoder
        voc = MelVocoder(device=DEV, state_dict=sd)
        assert torch.equal(voc.inverse(mel, lengths=torch.tensor(lengths)), wav.squeeze(1))


def test_generator_ragged_full_size():
    """fp16s at B = 32, T_max = 1000, lengths 200 ... 1000: sampled utterances against the oracle on the utterance alone,
    the whole waveform finite; a flipped input as negative control of the comparison."""
    g, sd = _generator("fp16s")
    B, T = 32, 1000
    gen = torch.Generator().manual_seed(5)
    lengths = torch.randint(200, 1001, (B,), generator=gen).tolist()
    lengths[0], lengths[1] = 1000, 200
    mel = synthetic_mel(B, T, 71).transpose(1, 2).contiguous()
    for b, n in enumerate(lengths):
        mel[b, :, n:] = NAN
    wav = g(mel.to(DEV), lengths=lengths).squeeze(1)
    torch.cuda.synchronize()
    assert torch.isfinite(wav).all()
    for b in (0, 1, 17):
        n = lengths[b]
        ref = melgan_forward(sd, mel[b:b + 1, :, :n]).view(-1)
        got = wav[b, :256 * n].cpu()
        assert rel_l2(got, ref) < 1e-3, (b, n, rel_l2(got, ref))
        assert not wav[b, 256 * n:].any()
        assert rel_l2(got, melgan_forward(sd, mel[b:b + 1, :, :n].flip(2)).view(-1)) > 1e-2


# ------------------------------------------------------------------------------------------------ pipeline
def test_convert_and_vocode_utterances():
    """The config-4 recipe on utterances of mixed lengths against per-utterance convert_and_vocode (B = 1), in input
    order, within the config-4 waveform gate."""
    from autoformer_b200 import pipeline
    from autoformer_b200.factory.AutoVC import AutoVC
    from autoformer_b200.factory.LstmDV import LstmDV
    args = (32, 256, 512, 32)
    dv = LstmDV()
    dv.load_state_dict(seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5))
    dv = dv.to(DEV).eval()
    vc = AutoVC(*args)
    vc.load_state_dict(seeded_state_dict(templates.autovc_template(*args), 0))
    vc = vc.to(DEV).eval()
    g, _ = _generator("fp16s")
    lens = [64, 37, 100, 5, 128, 64, 71, 12, 90, 33, 128, 47]
    src = [synthetic_mel(1, n, 80 + i)[0].to(DEV) for i, n in enumerate(lens)]
    trg = [synthetic_mel(1, n, 120 + i)[0].to(DEV) for i, n in enumerate(lens)]
    mels, wavs, eo, et = pipeline.convert_and_vocode_utterances(dv, vc, g, src, trg)
    assert len(mels) == len(wavs) == len(lens) and eo.shape == et.shape == (len(lens), 256)
    for i, n in enumerate(lens):
        mel1, wav1, eo1, et1 = pipeline.convert_and_vocode(dv, vc, g, src[i][None], trg[i][None])
        assert mels[i].shape == (n, 80) and wavs[i].shape == (256 * n,)
        assert rel_l2(eo[i:i + 1], eo1) < 1e-3 and rel_l2(mels[i][None], mel1) < 1e-3, i
        assert rel_l2(wavs[i][None], wav1) < 1e-3, (i, rel_l2(wavs[i][None], wav1))
