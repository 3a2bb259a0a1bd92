"""Drop-in ``factory.LstmDV.LstmDV`` (the d-vector speaker embedder) on libavc_b200.so.

Same constructor defaults, ``forward(x)`` contract and state_dict keys as the reference
(factory/LstmDV.py:4-24): 3 x LSTM(80 -> 768), last time step, Linear(768 -> 256), L2 normalisation.
Each LSTM layer is one dense input-projection GEMM plus the tensor-core recurrence; only h_T of the top
layer leaves the recurrence kernel (``h_last``), and the Linear + normalisation is one fused kernel.
Small batches in "fp16x2" run the three layers as one wavefront launch (``layers.LstmStack``, ``avc_lstm_stack_ws``);
``model.wavefront = False`` keeps them layer by layer (two-term weights everywhere, half the rounding error, ~3x the time).
"""
import torch
import torch.nn as nn

from .. import layers, ops


class LstmDV(layers.PlanOwner, nn.Module):
    def __init__(self, num_layers=3, dim_input=80, dim_cell=768, dim_emb=256):
        super().__init__()
        # the kernels cover a subset of what nn.LSTM / nn.Linear accept: say so here, not as an error code in the C ABI
        if dim_cell % 64 != 0 or dim_input % 8 != 0 or not 1 <= dim_emb <= 1024:
            raise ValueError(f"autoformer_b200.LstmDV supports dim_cell % 64 == 0, dim_input % 8 == 0, dim_emb <= 1024; "
                             f"got dim_cell={dim_cell}, dim_input={dim_input}, dim_emb={dim_emb}")
        self.lstm = nn.LSTM(input_size=dim_input, hidden_size=dim_cell, num_layers=num_layers, batch_first=True)
        self.embedding = nn.Linear(dim_cell, dim_emb)
        self.num_layers, self.dim_cell = num_layers, dim_cell
        self.precision = "fp32"
        self.persistent_lstm = True
        self.wavefront = None           # None: the library default (on, layers.LstmStack)
        self._cache = layers.PlanCache()

    def _build_plan(self):
        sd = layers.state_for_packing(self)
        return dict(lstm=layers.LstmStack(layers.lstm_layers(sd, "lstm", self.num_layers, self.precision), self.precision,
                                          self.wavefront),
                    w=sd["embedding.weight"].float().contiguous(), b=sd["embedding.bias"].float().contiguous())

    def _plan(self):
        return self._cache.get(self, (self.precision, self.wavefront), self._build_plan)

    def _last_hidden(self, plan, x, lengths=None):
        """h_T of the top LSTM layer, fp32 (B, dim_cell)   (LstmDV.py:20-21: ``lstm_out[:, -1, :]``); with lengths, h at
        frame lengths[b] - 1 of utterance b."""
        ops._require_cuda(x)
        x = x.contiguous().float()
        B, T, _ = x.shape
        h = ops.to_act(x, self.precision)
        h_last = torch.empty(B, self.dim_cell, dtype=torch.float32, device=x.device)
        if lengths is None:
            return plan["lstm"].last_hidden(h, B, T, h_last, persistent=self.persistent_lstm)
        return plan["lstm"].last_hidden(h, B, T, h_last, persistent=self.persistent_lstm,
                                        lengths=layers.upload_lengths(lengths, B, T, x.device))

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, *, lengths=None):
        """lengths: optional per-utterance valid frames of a padded batch (list or tensor); the d-vector of utterance b
        is then that of ``x[b:b+1, :lengths[b]]`` alone."""
        plan = self._plan()
        return ops.linear_l2norm(self._last_hidden(plan, x, lengths), plan["w"], plan["b"])        # LstmDV.py:21-24
