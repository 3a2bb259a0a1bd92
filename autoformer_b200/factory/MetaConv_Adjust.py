"""Drop-in ``factory.MetaConv_Adjust.MetaConv_Adjust`` (factory/MetaConv_Adjust.py:247-280): MetaConv whose source and
target speaker codes both pass through ``Adjust``; returns ``(c_org_adjusted, mel, mel_postnet, codes)``."""
import torch

from .. import ops
from .Adjust import Adjust
from ._meta import MetaBase


class MetaConv_Adjust(MetaBase):
    KIND = "conv"
    ADJUST_SOURCE = True

    def __init__(self, dim_neck, dim_emb, dim_pre, freq):
        super().__init__(dim_neck, dim_emb, dim_pre, freq)
        self.adjust = Adjust(dim_emb)

    def _adjust(self, x, emb):
        self.adjust.precision = self.precision
        self.adjust.bn_stats = self.bn_stats                                    # governs the Adjust BatchNorms too
        return self.adjust(x, emb)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, c_org, c_trg, isConvert=False, x_target=None):
        if self.ADJUST_SOURCE:
            c_org = self._adjust(x, c_org)                                      # MetaConv_Adjust.py:256
        if c_trg is None:
            return super().forward(x, c_org, None)
        c_trg = self._adjust(x_target if isConvert else x, c_trg)               # :260-263
        mel, post, codes = super().forward(x, c_org, c_trg)
        return c_org, mel, post, codes
