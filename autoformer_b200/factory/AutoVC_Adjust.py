"""Drop-in ``factory.AutoVC_Adjust.AutoVC_Adjust(dim_neck, dim_emb, dim_pre, freq)`` (factory/AutoVC_Adjust.py:169-205).

AutoVC whose speaker codes first pass through ``Adjust``: ``forward(x, c_org, c_trg, isConvert=False, x_target=None)``
returns ``(c_org_adjusted, mel, mel_postnet, codes)`` (or the codes alone when ``c_trg is None``).  The target code is
adjusted with ``x_target`` when ``isConvert`` is true, else with ``x`` itself (the training-time call)."""
import torch

from .. import ops
from .Adjust import Adjust
from .AutoVC import AutoVC


class AutoVC_Adjust(AutoVC):
    def __init__(self, dim_neck, dim_emb, dim_pre, freq):
        super().__init__(dim_neck, dim_emb, dim_pre, freq)
        self.adjust = Adjust(dim_emb)

    def _adjust(self, x, emb):
        self.adjust.precision = self.precision
        self.adjust.bn_stats = self.bn_stats                                    # governs the Adjust BatchNorms too
        self.adjust.persistent_lstm = self.persistent_lstm
        return self.adjust(x, emb)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, c_org, c_trg, isConvert=False, x_target=None):
        c_org = self._adjust(x, c_org)                                          # AutoVC_Adjust.py:179
        if c_trg is None:
            return super().forward(x, c_org, None)                              # :182-183
        c_trg = self._adjust(x_target if isConvert else x, c_trg)               # :184-189
        mel, post, codes = super().forward(x, c_org, c_trg)
        return c_org, mel, post, codes                                          # :205
