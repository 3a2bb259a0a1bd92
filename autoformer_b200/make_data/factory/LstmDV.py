"""Drop-in ``make_data.factory.LstmDV.LstmDV`` -- the speaker embedder WITH its classifier head
(make_data/factory/LstmDV.py:4-25).

This is the twin the reference's Evaluator actually calls: it indexes ``embedder(mel)[1]``
(util/evaluate.py:104,132,200), i.e. the ``d_vec`` of the ``(predictions, d_vec)`` pair.  Same constructor
``LstmDV(num_classes=256, num_layers=3, dim_input=80, dim_cell=768, dim_emb=256)`` and state_dict keys
(``lstm.*``, ``embedding.*``, ``output.*``), so checkpoints of the twin load with ``strict=True``.

The recurrence is the embedder's (factory/LstmDV.py on avc_lstm_seq, only h_T of the top layer leaves the kernel);
the tail runs as two launches of ``avc_linear_rows``: ``embeds = embedding(h_T)`` with both its raw and its
L2-normalised form (:21-23), then ``predictions = output(embeds)`` on the UN-normalised embedding (:24)."""
import torch
import torch.nn as nn

from ... import layers, ops
from ...factory.LstmDV import LstmDV as _Embedder


class LstmDV(_Embedder):
    def __init__(self, num_classes=256, num_layers=3, dim_input=80, dim_cell=768, dim_emb=256):
        super().__init__(num_layers=num_layers, dim_input=dim_input, dim_cell=dim_cell, dim_emb=dim_emb)
        self.output = nn.Linear(dim_emb, num_classes)
        self.num_classes = num_classes

    def _plan(self):
        def build():
            plan = self._build_plan()
            sd = layers.state_for_packing(self)
            plan["w_out"] = sd["output.weight"].float().contiguous()
            plan["b_out"] = sd["output.bias"].float().contiguous()
            return plan
        return self._cache.get(self, (self.precision, self.wavefront), build)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, *, lengths=None):
        """lengths: as the embedder's (factory/LstmDV.py): per-utterance valid frames of a padded batch."""
        plan = self._plan()
        h_last = self._last_hidden(plan, x, lengths)
        embeds, d_vec = ops.linear_rows(h_last, plan["w"], plan["b"], want_raw=True, want_normed=True)   # :21-23
        predictions, _ = ops.linear_rows(embeds, plan["w_out"], plan["b_out"], want_raw=True)            # :24
        return predictions, d_vec                                                                         # :25
