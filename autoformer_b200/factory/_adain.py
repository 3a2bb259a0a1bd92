"""The AdaIN "2" variants (factory/AutoVC2.py, MetaPool2.py, MetaConv2.py; SURVEY.md 8f.3) as a mixin over the drop-in
models.

Encoder side (AutoVC2.py:54-60): three [Conv1d(80 -> 80, k5) + BatchNorm] layers run on the mel BEFORE the speaker
concat; after each one the scalar ``x.mean()`` and ``x.std()`` over the whole (B, 80, T) tensor are recorded as the
utterance batch's "features", and the encoder continues from the third layer's output.  Postnet side
(AutoVC2.py:192-203): after the five postnet convolutions, three times ``x = combine_i(AdaIN(x, mu_i, std_i))`` with
``AdaIN(x, mu, std) = (x - x.mean()) / x.std() * std + mu`` (factory/Norm.py:86-94) and combine_i = Conv1d(80 -> 80, k5).
``forward(x, c_org, c_trg, target_feature=None)`` returns ``(codes, features)`` when both c_trg and target_feature are
None, else the usual 3-tuple, styled with ``target_feature`` if given (util/evaluate.py:81-82) or with the source's own
features.

``adain_stats`` selects what the six statistics are taken over:

- ``"batch"`` (default): batch-global scalars, exactly as in the reference: a call's result depends on which utterances
  share the batch, so in this mode these variants are NOT utterance-shardable (SURVEY.md 8e); per call they match the
  reference.  Kernels: ``avc_conv_gemm`` (the six small convolutions), ``avc_global_stats``, ``avc_adain``.
- ``"utterance"``: every statistic is taken over one utterance's own frames, so utterance b of a batch gets what the
  reference returns for ``x[b:b+1]`` alone -- the Evaluator's one call per utterance (util/evaluate.py:69-71) -- and a
  batch is shardable by utterance.  ``features()`` then holds ``(B,)`` tensors, ``target_feature`` takes per entry a
  0-dim value (one style for all) or a ``(B,)`` tensor (one style per utterance), and AutoVC2 takes ``lengths`` as
  AutoVC does (utterance b then gets the reference's result for ``x[b:b+1, :lengths[b]]``).  Needs
  ``bn_stats="running"``.  Kernels: ``avc_segment_stats``, ``avc_adain_segmented``.
"""
import torch
import torch.nn as nn

from .. import layers, ops, packing
from .AutoVC import AutoVC
from .Norm import ConvNorm

ADAIN_STATS = ("batch", "utterance")


class AdaIN(nn.Module):
    """Parameter-free placeholder so the module tree matches the reference (factory/Norm.py:86-94)."""


class AdaINPlan:
    def __init__(self, sd, precision, bn_owner=None):
        self.pre = [layers.conv_bn_layer(sd, f"encoder.feature_pre_extract.{i}", precision, "none", bn_owner)
                    for i in range(3)]
        self.combine = [ops.ConvGemm(*packing.pack_conv(sd[f"postnet.feature_last_combine.{i}.0.conv.weight"],
                                                        sd[f"postnet.feature_last_combine.{i}.0.conv.bias"], precision),
                                     act="none", tag="conv") for i in range(3)]


class AdaINMixin:
    """Mix in BEFORE the base model class: ``class AutoVC2(AdaINMixin, AutoVC)``."""

    def _init_adain(self):
        self.encoder.feature_pre_extract = nn.ModuleList([
            nn.Sequential(ConvNorm(80, 80, kernel_size=5, stride=1, padding=2, dilation=1, w_init_gain="linear"),
                          nn.BatchNorm1d(80)) for _ in range(3)])
        self.postnet.adain = AdaIN()
        self.postnet.feature_last_combine = nn.ModuleList([
            nn.Sequential(ConvNorm(80, 80, kernel_size=5, stride=1, padding=2, dilation=1, w_init_gain="linear"))
            for _ in range(3)])
        self._adain_cache = layers.PlanCache()
        self.adain_stats = "batch"
        self._features = None
        self._target_stats = None

    def _per_utterance(self):
        if self.adain_stats not in ADAIN_STATS:
            raise ValueError(f"adain_stats must be one of {ADAIN_STATS}, got {self.adain_stats!r}")
        if self.adain_stats == "utterance" and layers.check_bn_stats(self.bn_stats) == "batch":
            raise ValueError("adain_stats='utterance' with bn_stats='batch': batch BatchNorm statistics couple the "
                             "utterances again; use bn_stats='running'")
        return self.adain_stats == "utterance"

    def _adain_plan(self):
        batch = layers.check_bn_stats(self.bn_stats) == "batch"

        def build():
            sd = layers.state_for_packing(self)
            return AdaINPlan(sd, self.precision, self if batch else None)
        return self._adain_cache.get(self, (self.precision, self.bn_stats), build, skip_bn_stats=batch)

    # ---- hooks called by the base forward
    def _encoder_features(self, x, plan, B, T, lengths=None):
        ap = self._adain_plan()
        prec = self.precision
        per_utt = self.adain_stats == "utterance"
        stats = torch.empty((3, B, 2) if per_utt else (3, 2), dtype=torch.float32, device=x.device)
        h = ops.to_act(x, prec)
        if lengths is not None:        # the zero padding of each utterance alone for the k = 5 convolutions that read h
            ops.zero_tail(h, 0, T, lengths)
        for i, conv in enumerate(ap.pre):                                  # AutoVC2.py:57-60
            f32 = torch.empty(B, T, 80, dtype=torch.float32, device=x.device)
            o = ops.alloc_act(B, T, 80, prec, x.device)
            conv(h, B, T, out=o, out2=f32.view(B * T, 80))
            if lengths is not None and i < 2:      # the last operand is not read again: the encoder goes on from f32
                ops.zero_tail(o, 0, T, lengths)
            if per_utt:
                ops.segment_stats(f32, **layers._lengths_kw(lengths), out=stats[i])
            else:
                ops.global_stats(f32, out=stats[i])
            h, x = o, f32
        self._features = stats
        return x                                                           # the encoder continues from the features

    def _run_postnet(self, plan, mel_op, mel, B, T, taps, lengths=None):
        ap = self._adain_plan()
        prec = self.precision
        per_utt = self.adain_stats == "utterance"
        style = self._target_stats if self._target_stats is not None else self._features
        h = plan.postnet.hidden(mel_op, B, T, taps, **layers._lengths_kw(lengths))   # AutoVC2.py:193-194
        cur = torch.empty(B, T, 80, dtype=torch.float32, device=mel.device)
        plan.postnet.convs[4](h, B, T, out2=cur.view(B * T, 80))           # :196
        for i, comb in enumerate(ap.combine):                              # :197-199
            if per_utt:        # rows past an utterance's end: not counted, written as the combine's zero padding
                kw = layers._lengths_kw(lengths)
                a_op, _ = ops.adain_segmented(cur, ops.segment_stats(cur, **kw), style[i], prec, **kw)
            else:
                a_op, _ = ops.adain(cur, ops.global_stats(cur), style[i], prec)
            nxt = torch.empty(B, T, 80, dtype=torch.float32, device=mel.device)
            last = i == len(ap.combine) - 1                                # the residual mel + postnet rides on the last
            comb(a_op, B, T, out2=nxt.view(B * T, 80), residual=mel.view(B * T, 80) if last else None)
            cur = nxt
        return cur

    # ---- public surface
    def features(self):
        """[[mean, std]] x 3, the structure Encoder.forward returns (AutoVC2.py:60): 0-dim tensors, or with
        ``adain_stats = "utterance"`` (B,) tensors (entry b: utterance b's statistics)."""
        st = self._features
        return [[st[i, ..., 0], st[i, ..., 1]] for i in range(3)]

    @staticmethod
    def _as_stats(target_feature, device):
        rows = [torch.stack([torch.as_tensor(m, dtype=torch.float32, device=device).reshape(()),
                             torch.as_tensor(s, dtype=torch.float32, device=device).reshape(())])
                for m, s in target_feature]
        return torch.stack(rows).contiguous()

    @staticmethod
    def _as_utterance_stats(target_feature, device, B):
        """Per entry [2] (one style for every utterance) or [B][2] (one per utterance)."""
        out = []
        for m, s in target_feature:
            m, s = (torch.as_tensor(v, dtype=torch.float32, device=device) for v in (m, s))
            if any(v.shape not in ((), (B,)) for v in (m, s)):
                raise ValueError(f"target_feature entries must be 0-dim or of shape ({B},) with adain_stats="
                                 f"'utterance'; got {tuple(m.shape)} and {tuple(s.shape)}")
            out.append(torch.stack(torch.broadcast_tensors(m, s), -1).contiguous())
        return out

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, c_org, c_trg, target_feature=None, *, lengths=None):
        ops._require_cuda(x)
        per_utt = self._per_utterance()
        if lengths is not None:
            if not isinstance(self, AutoVC):
                raise ValueError(f"{type(self).__name__} runs at the reference's fixed T = 176 and takes no lengths")
            if not per_utt:
                raise ValueError("lengths with adain_stats='batch': batch-global statistics over padded frames match "
                                 "no per-utterance conversion; set adain_stats='utterance'")
        if target_feature is None:
            self._target_stats = None
        elif per_utt:
            self._target_stats = self._as_utterance_stats(target_feature, x.device, x.shape[0])
        else:
            self._target_stats = self._as_stats(target_feature, x.device)
        kw = layers._lengths_kw(lengths)
        try:
            if c_trg is None:
                if target_feature is not None:
                    raise AttributeError("'NoneType' object has no attribute 'unsqueeze' (c_trg is required when a "
                                         "target_feature is given, as in the reference)")
                codes = super().forward(x, c_org, None, **kw)
                return codes, self.features()                              # AutoVC2.py:219-220
            return super().forward(x, c_org, c_trg, **kw)
        finally:
            self._target_stats = None
