"""Packed layer objects shared by the drop-in models: they own folded/re-packed weights and call ``ops``."""
import torch
import torch.nn as nn

from . import ops, packing
from .packing import TORCH_DTYPE


# Where the one-off weight folding / re-packing of a model runs.  False (default): on the model's own device -- a few
# hundred tiny torch kernels per model, microseconds each.  True: on the host, the packed tensors then move to the device
# with plain copies -- no torch kernel is launched at all, which keeps a profiler's launch list of a short run (smoke())
# to this library's own kernels.  Same arithmetic either way (torch CPU vs CUDA elementwise ops, fp64 folding).
PACK_ON_CPU = False


def state_for_packing(module):
    """The module's state_dict as detached tensors, on the host when PACK_ON_CPU."""
    sd = {k: v.detach() for k, v in module.state_dict().items()}
    if PACK_ON_CPU:
        sd = {k: v.cpu() for k, v in sd.items()}
    return sd


def plan_to(obj, device, _seen=None):
    """Move every tensor reachable from a packed plan (objects of this package, lists, tuples, dicts) to `device`."""
    if _seen is None:
        _seen = set()
    if torch.is_tensor(obj):
        return obj.to(device)
    if isinstance(obj, (list, tuple)):
        moved = [plan_to(o, device, _seen) for o in obj]
        return type(obj)(moved) if isinstance(obj, tuple) else moved
    if isinstance(obj, dict):
        return {k: plan_to(v, device, _seen) for k, v in obj.items()}
    if hasattr(obj, "__dict__") and type(obj).__module__.startswith("autoformer_b200") and id(obj) not in _seen:
        _seen.add(id(obj))
        for k, v in list(vars(obj).items()):
            if torch.is_tensor(v) or isinstance(v, (list, tuple, dict)) or hasattr(v, "__dict__"):
                setattr(obj, k, plan_to(v, device, _seen))
    return obj


def bn_stat_buffer_ids(module):
    """ids of the running_mean / running_var / num_batches_tracked buffers of every BatchNorm under `module`."""
    ids = set()
    for m in module.modules():
        if isinstance(m, nn.modules.batchnorm._BatchNorm):
            ids.update(id(t) for t in (m.running_mean, m.running_var, m.num_batches_tracked) if t is not None)
    return ids


BN_STATS = ("running", "batch")


def check_bn_stats(mode):
    if mode not in BN_STATS:
        raise ValueError(f"bn_stats={mode!r}: 'running' (BatchNorm folded with its running statistics) or 'batch' "
                         "(statistics of each call's batch, updating the running buffers: nn.BatchNorm1d in train mode)")
    return mode


class PlanCache:
    """Re-pack weights only when a parameter/buffer was replaced, moved or modified.

    The key holds, per tensor, (data_ptr, _version, device, shape, dtype) AND a content digest: in-place writes
    through ``.data`` (``p.data.normal_()``, ``p.data.copy_(w)`` -- what the reference's MelGAN ``weights_init`` does,
    melgan/modules.py:9-15) do not bump ``_version``, so the version counter alone would leave a stale plan and the
    forward would silently run with old weights.  The digest is the 1- and 2-norm of every floating-point tensor,
    computed on the tensors' device with multi-tensor launches (``torch._foreach_norm``: a handful of kernels for all
    tensors of one dtype) and fetched with one small copy per forward.  ``frozen = True`` (set by the models' ``freeze_weights()``) skips the digest for serving loops
    that promise not to touch the weights; ``invalidate()`` forces a re-pack."""

    def __init__(self):
        self.key = None
        self.plan = None
        self.frozen = False

    @staticmethod
    def fingerprint(module, extra=(), contents=True, skip_bn_stats=False):
        items = []
        by_dev = {}
        skip = bn_stat_buffer_ids(module) if skip_bn_stats else ()
        for t in list(module.parameters()) + list(module.buffers()):
            if id(t) in skip:
                continue
            items.append((t.data_ptr(), t._version, str(t.device), tuple(t.shape), str(t.dtype)))
            if contents and t.numel() and t.is_floating_point():
                by_dev.setdefault(t.device, []).append(t.detach())
        digest = []
        for ts in by_dev.values():
            n1 = torch._foreach_norm(ts, 1)
            n2 = torch._foreach_norm(ts, 2)
            digest.append(tuple(torch.stack(list(n1) + list(n2)).tolist()))      # one stack, one copy
        return (tuple(items), tuple(extra), tuple(digest))

    def invalidate(self):
        """Forget the packed plan: the next forward re-folds and re-packs from the module's current weights."""
        self.key = None
        self.plan = None

    def get(self, module, extra, builder, skip_bn_stats=False):
        """``skip_bn_stats``: leave the BatchNorm running buffers out of the key -- a batch-statistics plan does not
        read them at packing time, and every one of its forwards updates them, which would otherwise re-pack the plan
        on the next call."""
        if self.frozen and self.plan is not None and self.key is not None and self.key[1] == tuple(extra):
            return self.plan
        key = self.fingerprint(module, extra, True, skip_bn_stats)
        if key != self.key:
            plan = builder()
            if PACK_ON_CPU:
                first = next(iter(module.parameters()), None)
                if first is not None and first.is_cuda:
                    plan = plan_to(plan, first.device)
            self.plan = plan
            self.key = key
        return self.plan


class PlanOwner:
    """Mixin of the drop-in models: public control over the packed-weight cache (``self._cache``)."""

    def invalidate(self):
        """Drop the packed weights; call after editing parameters in a way torch cannot see (the content digest catches
        ``.data`` writes by itself -- this is the explicit form, and the only one that works while frozen)."""
        for m in self.modules():
            c = getattr(m, "_cache", None)
            if isinstance(c, PlanCache):
                c.invalidate()

    repack = invalidate

    def freeze_weights(self, frozen=True):
        """Serving mode: skip the per-forward weight digest (two small launches and one host sync).  The weights must
        not change while frozen; ``invalidate()`` or ``freeze_weights(False)`` re-arms the check."""
        for m in self.modules():
            c = getattr(m, "_cache", None)
            if isinstance(c, PlanCache):
                c.frozen = frozen
                if not frozen:
                    c.invalidate()
        return self


class BatchStatsConvBn:
    """nn.Sequential(ConvNorm(k5,p2), BatchNorm1d) (+act) with the BatchNorm in training mode: each call normalises with
    the statistics of its own B x T rows and updates the module's running buffers, as the reference's notebooks run
    every such layer (they never call .eval(), SURVEY.md fact 1).

    Three launches after the conv's own: the conv (its bias, nothing folded) writes v as exact fp32; avc_bn_batch_stats
    reduces v per channel and updates running_mean / running_var / num_batches_tracked on the device;
    avc_bn_apply writes act(scale v + shift) (+ residual) where the folded layer's epilogue would have.  The buffers
    are read from the live nn.BatchNorm1d at every call (not from the packing-time state_dict), so ``state_dict()``
    shows the updates and momentum / eps are the module's own."""

    def __init__(self, sd, prefix, precision, act, bn):
        self.conv = ops.ConvGemm(*packing.pack_conv(sd[f"{prefix}.0.conv.weight"], sd[f"{prefix}.0.conv.bias"],
                                                    precision), act="none", tag="conv")
        self.gamma = sd[f"{prefix}.1.weight"].detach().float().contiguous()
        self.beta = sd[f"{prefix}.1.bias"].detach().float().contiguous()
        self.bn = bn
        self.act = act
        self.precision = precision
        self.C = self.gamma.numel()
        if bn.running_mean is None:
            raise ValueError(f"{prefix}.1: batch statistics need the running buffers (track_running_stats=True)")

    def __call__(self, srcs, B, T, out=None, out2=None, residual=None, res_after=False):
        """Same outputs as ConvGemm.__call__ with the BatchNorm folded: out (operand format) and / or out2 (fp32),
        residual fp32 added before the activation, or after it with res_after."""
        if B * T <= 1:
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {(B, self.C, T)}")
        bn = self.bn
        v = torch.empty(B * T, self.C, dtype=torch.float32, device=self.gamma.device)
        self.conv(srcs, B, T, out2=v)
        ss = ops.bn_batch_stats(v, self.gamma, self.beta, bn.eps, bn.momentum, bn.running_mean, bn.running_var,
                                bn.num_batches_tracked)
        return ops.bn_apply(v, ss, B, T, self.act, out=out, out2=out2, residual=residual, res_after=res_after,
                            out_fmt=self.precision)


def conv_bn_layer(sd, prefix, precision, act, bn_owner=None):
    """nn.Sequential(ConvNorm(k5,p2), BatchNorm1d) (+act) -> one packed conv (factory/AutoVC.py:26-39).

    bn_owner None: the BatchNorm folded into the conv with its running statistics (eval semantics).  bn_owner = the
    module `prefix` is relative to: batch statistics (``BatchStatsConvBn``) on that module's live BatchNorm."""
    if bn_owner is not None:
        return BatchStatsConvBn(sd, prefix, precision, act, bn_owner.get_submodule(f"{prefix}.1"))
    w, b = packing.fold_bn(sd[f"{prefix}.0.conv.weight"], sd[f"{prefix}.0.conv.bias"], sd[f"{prefix}.1.weight"],
                           sd[f"{prefix}.1.bias"], sd[f"{prefix}.1.running_mean"], sd[f"{prefix}.1.running_var"])
    return ops.ConvGemm(*packing.pack_conv(w, b, precision), act=act, tag="conv")


def check_lengths(lengths, B, T, multiple=1):
    """Per-utterance lengths of a padded batch (a list, a CPU tensor or a CUDA tensor, read back once), validated on the
    host -- B entries, 1 <= lengths[b] <= T, multiples of `multiple` -- as a list of ints."""
    if torch.is_tensor(lengths):
        lengths = lengths.detach().cpu().reshape(-1).tolist()
    vals = [int(v) for v in lengths]
    if len(vals) != B:
        raise ValueError(f"lengths has {len(vals)} entries for a batch of {B} utterances")
    bad = [v for v in vals if not 1 <= v <= T]
    if bad:
        raise ValueError(f"lengths must lie in [1, T={T}]; got {bad[:4]}")
    bad = [v for v in vals if v % multiple]
    if bad:
        raise ValueError(f"lengths must be multiples of freq={multiple} (pad each utterance as pipeline.convert does); "
                         f"got {bad[:4]}")
    return vals


def upload_lengths(lengths, B, T, device, multiple=1):
    """``check_lengths``, then uploaded once as a device int32 [B] tensor.  The kernels trust these values, so nothing
    unchecked reaches them."""
    return torch.tensor(check_lengths(lengths, B, T, multiple), dtype=torch.int32).to(device)


def _lengths_kw(lengths):
    """``lengths=`` for an ops call of a variable-length batch; nothing at all for a fixed-length one, so the ops of a
    fixed-length forward are called exactly as they were before variable-length batches existed."""
    return {} if lengths is None else {"lengths": lengths}


def lstm_fused_default():
    """LstmLayer's default for `fused`.  Kept as a function because bench.py imports it to name the roofline kernel."""
    return True


class LstmLayer:
    """One uni-directional nn.LSTM layer on the tensor-core recurrence kernel.  By default the input projection is
    fused into that kernel (its MMAs fill the tensor pipe while the cell update and the grid barrier of the previous
    frame are in flight); `fused=False` runs it as one dense GEMM per layer in front of the recurrence."""

    def __init__(self, w_ih, w_hh, b_ih, b_hh, precision, fused=True):
        self.w_ih, self.w_hh, self.b_ih, self.b_hh = w_ih.detach(), w_hh.detach(), b_ih.detach(), b_hh.detach()
        self.precision = precision
        self.H = w_hh.shape[1]
        self.C_in = w_ih.shape[1]
        self.fused = fused
        self.ws = True
        self._packs = {}
        self._fused_packs = {}

    def _raw(self):
        """The layer's raw weights where the (lazy, per gate group) packing runs: the host when PACK_ON_CPU."""
        ws = (self.w_ih, self.w_hh, self.b_ih, self.b_hh)
        return tuple(w.cpu() for w in ws) if PACK_ON_CPU else ws

    def fused_packs(self, group):
        if group not in self._fused_packs:
            w_ih, w_hh, b_ih, b_hh = self._raw()
            wih, bias = packing.pack_lstm_ih_fused(w_ih, b_ih, b_hh, self.precision, group)
            packs = (wih, bias, packing.pack_lstm_hh(w_hh, self.precision, group))
            self._fused_packs[group] = tuple(t.to(self.w_hh.device) for t in packs)
        return self._fused_packs[group]

    def packs(self, group):
        if group not in self._packs:
            w_ih, w_hh, b_ih, b_hh = self._raw()
            ih = ops.ConvGemm(*packing.pack_lstm_ih(w_ih, b_ih, b_hh, self.precision, group), tag="inproj")
            hh = packing.pack_lstm_hh(w_hh, self.precision, group)
            self._packs[group] = (ih.to(self.w_hh.device), hh.to(self.w_hh.device))
        return self._packs[group]

    def use_fused(self, B):
        """Fusing pays when the input part hides behind the cell update + grid barrier of the previous frame (about 7
        k-blocks' worth of MMAs), or when the batch fills the 128-row tiles so the in-kernel products are as
        efficient as the stand-alone GEMM; a small batch with a wide input (LstmDV layers 1-2 at B = 32: 12 k-blocks
        on a quarter-filled tile) is faster with the dense projection in front (measured: 37 ms vs 32 ms)."""
        kx = (self.C_in + packing.KC[self.precision] - 1) // packing.KC[self.precision]
        return self.fused and (kx <= 6 or B >= 192)

    def __call__(self, x, B, T, hseq_f32=None, h_last=None, persistent=False, hseq=None, lengths=None):
        """lengths: optional device int32 [B] of a padded batch; h_last[b] is then h at frame lengths[b] - 1 (hseq
        keeps all T frames: the recurrence is causal, so the frames past a length never reach a valid one)."""
        cap = ops.persistent_batch_cap(self.H) if persistent else 0
        if persistent and B > cap > 0:
            # utterances are independent: a batch too large for one wave of the persistent grid runs as sub-batches
            # (slices along the utterance axis are contiguous views, so nothing is copied)
            out = ops.alloc_act(B, T, self.H, self.precision, x.device) if hseq is None else hseq
            for b0 in range(0, B, cap):
                b1 = min(B, b0 + cap)
                self(x[b0:b1], b1 - b0, T, hseq_f32=hseq_f32[b0:b1] if hseq_f32 is not None else None,
                     h_last=h_last[b0:b1] if h_last is not None else None, persistent=True, hseq=out[b0:b1],
                     **_lengths_kw(lengths[b0:b1] if lengths is not None else None))
            return out
        if persistent and self.ws and ops.ws_supported(B, self.H, self.precision):
            # small batch: dense input projection, then the recurrence with W_hh resident in tensor memory
            ih, hh = self.packs(packing.WS_GROUP)
            xp = torch.empty(B * T, 4 * self.H, dtype=torch.float32, device=x.device)
            ih(x, B, T, out2=xp)
            out = ops.lstm_seq_ws(xp, hh, B, T, self.H, hseq=hseq, hseq_f32=hseq_f32, h_last=h_last,
                                  precision=self.precision, **_lengths_kw(lengths))
            if out is not None:
                return out
            self.ws = False             # the device cannot hold the grid: batched kernel from now on
        fused = self.use_fused(B)
        group = ops.choose_gate_group(B, self.H, persistent)
        if fused:
            wih, bias, hh = self.fused_packs(group)
            return ops.lstm_seq(None, hh, B, T, self.H, self.precision, group, hseq=hseq, hseq_f32=hseq_f32,
                                h_last=h_last, persistent=persistent, xin=x, w_ih=wih, bias=bias, c_in=self.C_in,
                                **_lengths_kw(lengths))
        ih, hh = self.packs(group)
        xp = torch.empty(B * T, 4 * self.H, dtype=torch.float32, device=x.device)
        ih(x, B, T, out2=xp)
        return ops.lstm_seq(xp, hh, B, T, self.H, self.precision, group, hseq=hseq, hseq_f32=hseq_f32, h_last=h_last,
                            persistent=persistent, **_lengths_kw(lengths))


def wavefront_eligible(pair, B, persistent):
    """Whether lstm_pair runs the two layers as one launch (ops.lstm_seq2) for a batch of B: persistent, not the
    small-batch weight-stationary path, the fused input projection for both layers, equal hidden sizes.  The benchmark
    has workloads on both sides: the 512-utterance batches take it, the smaller ones and the sub-batch tails do not."""
    l0, l1 = pair
    return (persistent and l0.H == l1.H and B <= ops.persistent_batch_cap(l0.H) and
            not any(l.ws and ops.ws_supported(B, l.H, l.precision) for l in pair) and
            l0.use_fused(B) and l1.use_fused(B))


def lstm_pair(pair, x, B, T, hseq_f32=None, persistent=False, hseq=None):
    """Two stacked LstmLayers (nn.LSTM(num_layers = 2)): layer 1's output sequence, with its exact fp32 copy in
    hseq_f32 when given.  Eligible batches (wavefront_eligible) run both layers as one persistent launch, layer 1 two
    frames behind layer 0, which hides each layer's cell update and barrier behind the other's MMAs; the results are
    bit-identical to calling the layers one after the other, which is what every other batch does."""
    l0, l1 = pair
    cap = ops.persistent_batch_cap(l0.H) if persistent else 0
    if persistent and B > cap > 0:
        # independent utterances: one wave of the persistent grid at a time, as LstmLayer splits its batch
        out = ops.alloc_act(B, T, l1.H, l1.precision, x.device) if hseq is None else hseq
        for b0 in range(0, B, cap):
            b1 = min(B, b0 + cap)
            lstm_pair(pair, x[b0:b1], b1 - b0, T, hseq_f32=hseq_f32[b0:b1] if hseq_f32 is not None else None,
                      persistent=True, hseq=out[b0:b1])
        return out
    if wavefront_eligible(pair, B, persistent):
        group = ops.choose_gate_group(B, l0.H, True)
        (wih0, bias0, hh0), (wih1, bias1, hh1) = l0.fused_packs(group), l1.fused_packs(group)
        out = ops.lstm_seq2((hh0, hh1), B, T, l0.H, l0.precision, group, x, (wih0, wih1), (bias0, bias1), l0.C_in,
                            hseq=(None, hseq), hseq_f32=(None, hseq_f32))
        if out is not None:
            return out[1]
    h = l0(x, B, T, persistent=persistent)      # the device cannot hold the grid, or an ineligible batch
    return l1(h, B, T, hseq_f32=hseq_f32, persistent=persistent, hseq=hseq)


def lstm_layers(sd, prefix, num_layers, precision):
    return [LstmLayer(sd[f"{prefix}.weight_ih_l{l}"], sd[f"{prefix}.weight_hh_l{l}"], sd[f"{prefix}.bias_ih_l{l}"],
                      sd[f"{prefix}.bias_hh_l{l}"], precision) for l in range(num_layers)]


class LstmStack:
    """nn.LSTM(num_layers = L) of which only the top layer's last frame is used (LstmDV.py:20-21, Adjust.py:40-41).

    Small batches in "fp16x2" run all layers as ONE wavefront launch (avc_lstm_stack_ws: layer l two ticks behind layer
    l - 1, T + 2 (L - 1) frame times instead of L x T).  On that path the recurrent and inter-layer weights are one fp16
    term instead of two -- what fits on chip -- which roughly doubles the rounding error of the embedding (2.8e-4
    instead of 1.6e-4 on the test weights, scripts/lstm_stack_precision.py; gate 1e-3); `wavefront=False` keeps the
    two-term layer-by-layer kernels."""

    def __init__(self, layers_, precision, wavefront=None):
        self.layers = layers_
        self.precision = precision
        self.H = layers_[0].H
        self.wavefront = True if wavefront is None else wavefront
        self._packs = None

    def packs(self):
        if self._packs is None:
            packs = []
            for i, layer in enumerate(self.layers):
                pk = packing.pack_lstm_stack(*layer._raw(), first=i == 0)
                packs.append(tuple(None if t is None else t.to(layer.w_hh.device) for t in pk))
            self._packs = packs
        return self._packs

    def eligible(self, B, persistent):
        first = self.layers[0]
        return (self.wavefront and persistent and first.ws and
                all(l.H == self.H and l.C_in == self.H for l in self.layers[1:]) and
                ops.stack_supported(B, self.H, len(self.layers), self.precision))

    def last_hidden(self, x, B, T, h_last, persistent=False, lengths=None):
        """x: the first layer's input in the operand format; fills h_last [B][H] fp32 with h_{T-1} of the top layer
        (with lengths, a device int32 [B]: h at frame lengths[b] - 1 of utterance b)."""
        if self.eligible(B, persistent):
            first = self.layers[0]
            ih, _ = first.packs(packing.WS_GROUP)
            xp = torch.empty(B * T, 4 * self.H, dtype=torch.float32, device=x.device)
            ih(x, B, T, out2=xp)
            if ops.lstm_stack_ws(xp, self.packs(), B, T, self.H, h_last=h_last, **_lengths_kw(lengths)) is not None:
                return h_last
            self.wavefront = False      # the device cannot hold the grid: layer by layer from now on
        h = x
        for i, layer in enumerate(self.layers):
            top = i == len(self.layers) - 1
            h = layer(h, B, T, h_last=h_last if top else None, persistent=persistent,
                      **_lengths_kw(lengths if top else None))
        return h_last


class BiLstmSmall:
    """Bidirectional nn.LSTM with a small hidden size (the AutoVC content encoder, factory/AutoVC.py:43)."""

    def __init__(self, sd, prefix, num_layers, precision):
        self.precision = precision
        self.layers = []
        for l in range(num_layers):
            g = lambda n, d="": sd[f"{prefix}.{n}_l{l}{d}"].detach()
            ih = ops.ConvGemm(*packing.pack_bilstm_ih(g("weight_ih"), g("bias_ih"), g("bias_hh"),
                                                      g("weight_ih", "_reverse"), g("bias_ih", "_reverse"),
                                                      g("bias_hh", "_reverse"), precision), tag="inproj")
            hh = torch.stack([g("weight_hh"), g("weight_hh", "_reverse")]).float().contiguous()
            self.layers.append((ih, hh))
        self.H = self.layers[0][1].shape[2]

    def __call__(self, x, B, T, freq=None, want_out=False, lengths=None):
        """Returns (out [B][T][2H] of the last layer or None, codes [B][T/freq][2H] fp32 or None).  lengths: optional
        device int32 [B] of a padded batch (multiples of freq): out rows / codes past an utterance's end are 0."""
        H = self.H
        out = None
        codes = None
        for i, (ih, hh) in enumerate(self.layers):
            last = i == len(self.layers) - 1
            xp = torch.empty(B * T, 8 * H, dtype=torch.float32, device=x.device)
            ih(x, B, T, out2=xp)
            if not last:
                out = ops.alloc_act(B, T, 2 * H, self.precision, x.device)
                ops.bilstm_small(xp, hh, B, T, H, out=out, split=self.precision == "fp32", **_lengths_kw(lengths))
                x = out
            else:
                out = torch.empty(B, T, 2 * H, dtype=torch.float32, device=x.device) if (want_out or freq is None) else None
                if freq is not None:
                    codes = torch.empty(B, T // freq, 2 * H, dtype=torch.float32, device=x.device)
                ops.bilstm_small(xp, hh, B, T, H, out=out, codes=codes, freq=freq or 1, round_tf32=False,
                                 **_lengths_kw(lengths))
        return out, codes


class Postnet:
    """Five conv+BN layers, tanh on the first four, residual add fused into the last (factory/AutoVC.py:117-179,206-209)."""

    def __init__(self, sd, prefix, precision, bn_owner=None):
        self.precision = precision
        self.convs = [conv_bn_layer(sd, f"{prefix}.convolutions.{i}", precision, "tanh" if i < 4 else "none", bn_owner)
                      for i in range(5)]

    def hidden(self, mel_op, B, T, taps=None, lengths=None):
        """The four conv+BN+tanh layers: [B][T][80] -> [B][T][512], operand format.  lengths (device int32 [B]): the
        rows past each utterance's end are zeroed after every layer, as the next k = 5 convolution's zero padding."""
        h = mel_op
        for i in range(4):
            o = ops.alloc_act(B, T, 512, self.precision, h.device)
            self.convs[i](h, B, T, out=o)
            if lengths is not None:
                ops.zero_tail(o, 0, T, lengths)
            h = o
            if taps is not None:
                taps[f"post_conv{i}"] = packing.act_to_float(h, self.precision)
        return h

    def __call__(self, mel_op, mel_f32, B, T, taps=None, lengths=None):
        """mel_op: [B][T][80] operand dtype; mel_f32: exact fp32 [B][T][80].  Returns mel + postnet(mel), fp32."""
        h = self.hidden(mel_op, B, T, taps) if lengths is None else self.hidden(mel_op, B, T, taps, lengths=lengths)
        out = torch.empty(B, T, 80, dtype=torch.float32, device=h.device)
        self.convs[4](h, B, T, out2=out.view(B * T, 80), residual=mel_f32.view(B * T, 80))
        return out
