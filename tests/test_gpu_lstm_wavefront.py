"""The two-layer LSTM launch (ops.lstm_seq2 / avc_lstm_seq2, layer 1 two frames behind layer 0 in one persistent
launch) against two one-layer persistent launches (ops.lstm_seq) on the same inputs, bit for bit: hseq and hseq_f32 of
both layers and the final c_state.  Every accumulator receives the same MMAs in the same order in both forms, so any
difference is a schedule error -- most likely an in-group overwriting an accumulator the cell warps have not read yet.

Op-level cases cover every precision, gate groups 16 and 32, the single-CTA (B = 37), CTA-pair (200) and phantom-tile
(300: three 128-row tiles in two pairs) geometries and T = 1, 2, 3, 7 (the ticks whose groups are partly out of range).
Each output sits between NaN sentinel rows, and a repeated launch must reproduce the same bits.  The production cases
run AutoVC's lstm2 shapes (512 -> 1024 -> 1024, T = 128) through layers.lstm_pair, including the sub-batch split of
B = 600, against the two LstmLayer calls."""
import pytest
import torch

from autoformer_b200 import _lib, layers, ops, packing

PRECS = ("tf32", "bf16", "fp32", "fp16x2")


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _sentinel(shape, dtype):
    """NaN buffer with one spare row on each side; returns (whole buffer, the inner rows)."""
    buf = torch.full((shape[0] + 2,) + tuple(shape[1:]), float("nan"), dtype=dtype, device="cuda")
    return buf, buf[1:-1]


def _layers(prec, c_in, H, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for k in (c_in, H):
        s = k ** -0.5
        w_ih, w_hh = (torch.rand(4 * H, k, generator=g) * 2 - 1) * s, (torch.rand(4 * H, H, generator=g) * 2 - 1) * s
        b_ih, b_hh = (torch.rand(4 * H, generator=g) * 2 - 1) * s, (torch.rand(4 * H, generator=g) * 2 - 1) * s
        out.append(layers.LstmLayer(w_ih.cuda(), w_hh.cuda(), b_ih.cuda(), b_hh.cuda(), prec))
    return out


def _pair_outputs(prec, group, pair, x, B, T, H, c_in):
    """lstm_seq2 into sentinel buffers: (whole buffers, inner views) of hseq0, hseq1, f32_0, f32_1, c0, c1."""
    (wih0, bias0, hh0), (wih1, bias1, hh1) = (l.fused_packs(group) for l in pair)
    C = packing.act_channels(H, prec)
    bufs = [_sentinel((B, T, C), packing.TORCH_DTYPE[prec]) for _ in range(2)]
    bufs += [_sentinel((B, T, H), torch.float32) for _ in range(2)]
    bufs += [_sentinel((B, H), torch.float32) for _ in range(2)]
    inner = [b[1] for b in bufs]
    out = ops.lstm_seq2((hh0, hh1), B, T, H, prec, group, x, (wih0, wih1), (bias0, bias1), c_in,
                        hseq=(inner[0], inner[1]), hseq_f32=(inner[2], inner[3]), c_state=(inner[4], inner[5]))
    assert out is not None, "the two-layer grid is not co-resident"
    return [b[0] for b in bufs], inner


def _reference(prec, group, pair, x, B, T, H, c_in):
    (wih0, bias0, hh0), (wih1, bias1, hh1) = (l.fused_packs(group) for l in pair)
    f0, f1 = (torch.empty(B, T, H, device="cuda") for _ in range(2))
    c0, c1 = (torch.empty(B, H, device="cuda") for _ in range(2))
    h0 = ops.lstm_seq(None, hh0, B, T, H, prec, group, hseq_f32=f0, persistent=True, xin=x, w_ih=wih0, bias=bias0,
                      c_in=c_in, c_state=c0)
    h1 = ops.lstm_seq(None, hh1, B, T, H, prec, group, hseq_f32=f1, persistent=True, xin=h0, w_ih=wih1, bias=bias1,
                      c_in=H, c_state=c1)
    return [h0, h1, f0, f1, c0, c1]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("group", (16, 32))
@pytest.mark.parametrize("B", (37, 200, 300))
def test_seq2_matches_two_launches(prec, group, B):
    H, c_in = 128, 72
    pair = _layers(prec, c_in, H, seed=B * 7 + group)
    for T in (1, 2, 3, 7):
        g = torch.Generator().manual_seed(T)
        x = packing.to_act(torch.randn(B, T, c_in, generator=g), prec).cuda()
        ref = _reference(prec, group, pair, x, B, T, H, c_in)
        whole, got = _pair_outputs(prec, group, pair, x, B, T, H, c_in)
        again = _pair_outputs(prec, group, pair, x, B, T, H, c_in)[1]
        torch.cuda.synchronize()
        names = ("hseq0", "hseq1", "hseq_f32_0", "hseq_f32_1", "c_state0", "c_state1")
        for name, r, o, a, w in zip(names, ref, got, again, whole):
            assert torch.equal(_bits(o), _bits(r)), f"{prec} G={group} B={B} T={T}: {name} differs"
            assert torch.equal(_bits(a), _bits(o)), f"{prec} G={group} B={B} T={T}: {name} differs on a repeat"
            assert torch.isnan(w[0].float()).all() and torch.isnan(w[-1].float()).all(), f"{name}: sentinel written"


@pytest.mark.gpu
@pytest.mark.parametrize("B", (512, 300, 600))
def test_lstm_pair_production_shapes(B):
    prec, T, H, c_in = "fp16x2", 128, 1024, 512
    pair = _layers(prec, c_in, H, seed=B)
    x = packing.to_act(torch.randn(B, T, c_in, generator=torch.Generator().manual_seed(1)), prec).cuda()
    f_ref = torch.empty(B, T, H, device="cuda")
    h_ref = pair[1](pair[0](x, B, T, persistent=True), B, T, hseq_f32=f_ref, persistent=True)
    f_new = torch.full((B, T, H), float("nan"), device="cuda")
    n0 = _lib.launch_count()
    h_new = layers.lstm_pair(pair, x, B, T, hseq_f32=f_new, persistent=True)
    torch.cuda.synchronize()
    if B <= ops.persistent_batch_cap(H):
        assert layers.wavefront_eligible(pair, B, True)
        assert _lib.launch_count() - n0 == 1, "the batch did not take the two-layer launch"
    assert torch.equal(_bits(h_new), _bits(h_ref))
    assert torch.equal(_bits(f_new), _bits(f_ref))
