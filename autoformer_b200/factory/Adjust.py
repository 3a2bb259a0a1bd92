"""Drop-in ``factory.Adjust.Adjust(dim_emb, dim_cell=768)`` on libavc_b200.so (factory/Adjust.py:7-43).

Re-estimates a speaker embedding from (mel, embedding): speaker-code concat, 3 x [Conv1d k5 + BatchNorm + ReLU],
3 x LSTM(512 -> 768), last time step, Linear(768 -> 256), L2 normalisation.  Every piece re-uses a kernel of the
conversion path: ``avc_concat_bcast``, ``avc_conv_gemm`` (BN folded, ReLU in the epilogue), ``avc_lstm_seq`` (only
h_T of the top layer leaves the kernel) and ``avc_linear_l2norm``.  Eval-mode semantics by default; ``bn_stats =
"batch"`` selects train-mode BatchNorm statistics (see autoformer_b200.AutoVC).  Inference only.
"""
import torch
import torch.nn as nn

from .. import layers, ops
from .Norm import ConvNorm, LinearNorm


class AdjustPlan:
    """Packed weights of one ``Adjust`` block taken from a (possibly enclosing) state_dict under ``prefix``."""

    def __init__(self, sd, prefix, precision, wavefront=None, bn_owner=None):
        p = prefix + "." if prefix else ""
        self.precision = precision
        self.convs = [layers.conv_bn_layer(sd, f"{p}convolutions.{i}", precision, "relu", bn_owner) for i in range(3)]
        self.lstm = layers.LstmStack(layers.lstm_layers(sd, f"{p}lstm", 3, precision), precision, wavefront)
        self.w = sd[f"{p}embedding.linear_layer.weight"].float().contiguous()
        self.b = sd[f"{p}embedding.linear_layer.bias"].float().contiguous()
        self.dim_cell = self.w.shape[1]

    def __call__(self, x, emb, persistent=False):
        """x (B,T,80) fp32 CUDA, emb (B,E) -> (B,256) unit-norm embedding."""
        B, T, _ = x.shape
        prec = self.precision
        h = ops.concat_bcast(x, emb, T, 1, prec)                        # Adjust.py:29-32
        for conv in self.convs:                                         # :36-37
            o = ops.alloc_act(B, T, 512, prec, x.device)
            conv(h, B, T, out=o)
            h = o
        h_last = torch.empty(B, self.dim_cell, dtype=torch.float32, device=x.device)
        self.lstm.last_hidden(h, B, T, h_last, persistent=persistent)   # :38-39 (only the last step is used)
        return ops.linear_l2norm(h_last, self.w, self.b)               # :40-42


class Adjust(layers.PlanOwner, nn.Module):
    def __init__(self, dim_emb, dim_cell=768):
        super().__init__()
        self.convolutions = nn.ModuleList([
            nn.Sequential(ConvNorm(80 + dim_emb if i == 0 else 512, 512, kernel_size=5, stride=1, padding=2,
                                   dilation=1, w_init_gain="relu"), nn.BatchNorm1d(512)) for i in range(3)])
        self.lstm = nn.LSTM(512, hidden_size=dim_cell, num_layers=3, batch_first=True)
        self.embedding = LinearNorm(dim_cell, 256)
        self.precision = "fp32"
        self.persistent_lstm = True
        self.wavefront = None           # None: the library default (layers.LstmStack)
        self.bn_stats = "running"
        self._cache = layers.PlanCache()

    def _plan(self):
        batch = layers.check_bn_stats(self.bn_stats) == "batch"

        def build():
            sd = layers.state_for_packing(self)
            return AdjustPlan(sd, "", self.precision, self.wavefront, self if batch else None)
        return self._cache.get(self, (self.precision, self.wavefront, self.bn_stats), build, skip_bn_stats=batch)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, emb):
        if x.dim() == 4:
            x = x.squeeze(1)                                            # Adjust.py:30
        ops._require_cuda(x, emb)
        if layers.check_bn_stats(self.bn_stats) == "batch" and x.shape[0] * x.shape[1] == 1:
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {(1, 512, 1)}")
        return self._plan()(x.contiguous().float(), emb.contiguous().float(), self.persistent_lstm)
