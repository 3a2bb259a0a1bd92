"""CPU check of which lstm2 batches take the two-layer LSTM launch (layers.wavefront_eligible), for the batch sizes the
benchmark runs: the headline and full cfg5 batches (512) and large cfg5 tails do; cfg4 (B = 32 and 1) and small tails
do not, nor does a per-frame (non-persistent) forward."""
import pytest
import torch

from autoformer_b200 import layers


def _lstm2(precision):
    def layer(c_in, H=1024):
        return layers.LstmLayer(torch.zeros(4 * H, c_in), torch.zeros(4 * H, H), torch.zeros(4 * H), torch.zeros(4 * H),
                                precision)
    return [layer(512), layer(1024)]


@pytest.mark.parametrize("precision", ("fp16x2", "fp32", "bf16", "tf32"))
def test_wavefront_rule(precision):
    pair = _lstm2(precision)
    for B in (512, 300, 192):
        assert layers.wavefront_eligible(pair, B, True), B
        assert not layers.wavefront_eligible(pair, B, False), B
    for B in (191, 88, 32, 1):      # cfg4 batches and small tails: layer by layer, as before
        assert not layers.wavefront_eligible(pair, B, True), B
    assert not layers.wavefront_eligible(pair, 600, True)    # above one wave: lstm_pair splits it into 512 + 88 first


def test_lstm_pair_host_logic(monkeypatch):
    """layers.lstm_pair on the CPU stand-ins of tests/emulate.py, with ops.lstm_seq2 mirrored here as the two layers one
    after the other (what the kernel's outputs are bit-identical to): B = 600 runs as a 512-utterance sub-batch through
    the two-layer launch and an 88-utterance tail layer by layer, and matches two LstmLayer calls on the whole batch."""
    from autoformer_b200 import ops, packing
    from tests.emulate import install_cpu_kernels
    install_cpu_kernels(monkeypatch)
    calls = []

    def lstm_seq2(w_hh, B, T, H, precision, group, xin, w_ih, bias, c_in, hseq=(None, None), hseq_f32=(None, None),
                  c_state=(None, None), debug_clk=None):
        calls.append(B)
        h0 = ops.lstm_seq(None, w_hh[0], B, T, H, precision, group, hseq=hseq[0], hseq_f32=hseq_f32[0],
                          persistent=True, xin=xin, w_ih=w_ih[0], bias=bias[0], c_in=c_in)
        h1 = ops.lstm_seq(None, w_hh[1], B, T, H, precision, group, hseq=hseq[1], hseq_f32=hseq_f32[1],
                          persistent=True, xin=h0, w_ih=w_ih[1], bias=bias[1], c_in=H)
        return h0, h1

    monkeypatch.setattr(ops, "lstm_seq2", lstm_seq2)
    g = torch.Generator().manual_seed(0)
    pair = []
    for c_in in (512, 1024):
        w = lambda *s: (torch.rand(*s, generator=g) * 2 - 1) * 0.03
        pair.append(layers.LstmLayer(w(4096, c_in), w(4096, 1024), w(4096), w(4096), "fp16x2"))
    B, T = 600, 2
    x = packing.to_act(torch.randn(B, T, 512, generator=g), "fp16x2")
    f_ref, f_new = torch.empty(B, T, 1024), torch.full((B, T, 1024), float("nan"))
    h_ref = pair[1](pair[0](x, B, T, persistent=True), B, T, hseq_f32=f_ref, persistent=True)
    h_new = layers.lstm_pair(pair, x, B, T, hseq_f32=f_new, persistent=True)
    assert calls == [512]
    assert torch.equal(h_new, h_ref) and torch.equal(f_new, f_ref)
