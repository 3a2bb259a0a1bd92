"""Drop-in ``factory.AutoVC.AutoVC`` whose forward runs on libavc_b200.so (sm_100a).

Same constructor ``AutoVC(dim_neck, dim_emb, dim_pre, freq)``, same ``forward(x, c_org, c_trg)`` contract and the
same ``state_dict`` key names as the reference (factory/AutoVC.py:182-211), so reference checkpoints load
unchanged.  By default the semantics are the reference's *eval-mode* forward (BatchNorm uses running statistics,
SURVEY.md 0.1); ``bn_stats = "batch"`` selects its train-mode BatchNorm instead (batch statistics, running buffers
updated).  Inference only (outputs carry no autograd graph).  There is no CPU / eager fallback.
"""
import warnings

import torch
import torch.nn as nn

from .. import layers, ops, packing
from .Norm import ConvNorm, LinearNorm


class Encoder(nn.Module):
    """Parameter container for the content encoder (factory/AutoVC.py:18-43)."""

    def __init__(self, dim_neck, dim_emb, freq):
        super().__init__()
        self.dim_neck, self.freq = dim_neck, freq
        self.convolutions = nn.ModuleList([
            nn.Sequential(ConvNorm(80 + dim_emb if i == 0 else 512, 512, kernel_size=5, stride=1, padding=2,
                                   dilation=1, w_init_gain="relu"), nn.BatchNorm1d(512)) for i in range(3)])
        self.lstm = nn.LSTM(512, dim_neck, 2, batch_first=True, bidirectional=True)


class Decoder(nn.Module):
    """Parameter container for the decoder (factory/AutoVC.py:71-98)."""

    def __init__(self, dim_neck, dim_emb, dim_pre):
        super().__init__()
        self.lstm1 = nn.LSTM(dim_neck * 2 + dim_emb, dim_pre, 1, batch_first=True)
        self.convolutions = nn.ModuleList([
            nn.Sequential(ConvNorm(dim_pre, dim_pre, kernel_size=5, stride=1, padding=2, dilation=1,
                                   w_init_gain="relu"), nn.BatchNorm1d(dim_pre)) for _ in range(3)])
        self.lstm2 = nn.LSTM(dim_pre, 1024, 2, batch_first=True)
        self.linear_projection = LinearNorm(1024, 80)


class Postnet(nn.Module):
    """Parameter container for the postnet (factory/AutoVC.py:117-171)."""

    def __init__(self):
        super().__init__()
        chans = [(80, 512, "tanh"), (512, 512, "tanh"), (512, 512, "tanh"), (512, 512, "tanh"), (512, 80, "linear")]
        self.convolutions = nn.ModuleList([
            nn.Sequential(ConvNorm(ci, co, kernel_size=5, stride=1, padding=2, dilation=1, w_init_gain=g),
                          nn.BatchNorm1d(co)) for ci, co, g in chans])


def check_hyper_parameters(dim_neck, dim_emb, dim_pre, freq):
    """The kernels cover a subset of the shapes the reference's nn.Modules accept (they accept any); reject the rest
    at construction with the reason, not as an error code deep in the C ABI.  The reference's own configurations --
    (32, 256, 512, 32) of the paper and (44, 256, 512, 22) of train.py:142-148 -- are inside."""
    problems = []
    if not 1 <= dim_neck <= 64:
        problems.append(f"dim_neck={dim_neck}: the encoder BiLSTM kernel keeps W_hh in registers for 1..64 hidden units")
    if dim_pre % 64 != 0 or dim_pre < 64:
        problems.append(f"dim_pre={dim_pre}: the tensor-core LSTM kernel needs a multiple of 64 hidden units")
    if (80 + dim_emb) % 8 != 0:
        problems.append(f"dim_emb={dim_emb}: 80 + dim_emb input channels must be a multiple of 8 (16-byte TMA rows)")
    if (2 * dim_neck + dim_emb) % 8 != 0:
        problems.append(f"2*dim_neck + dim_emb = {2 * dim_neck + dim_emb}: the decoder input must be a multiple of 8 "
                        "channels (16-byte TMA rows)")
    if freq < 1:
        problems.append(f"freq={freq}")
    if problems:
        raise ValueError("autoformer_b200.AutoVC supports dim_neck <= 64, dim_pre % 64 == 0, (80 + dim_emb) % 8 == 0, "
                         "(2 dim_neck + dim_emb) % 8 == 0; got " + "; ".join(problems))


class _Plan:
    def __init__(self, model, precision, bn_owner=None):
        sd = layers.state_for_packing(model)
        self.precision = precision
        self.enc_convs = [layers.conv_bn_layer(sd, f"encoder.convolutions.{i}", precision, "relu", bn_owner)
                          for i in range(3)]
        self.enc_lstm = layers.BiLstmSmall(sd, "encoder.lstm", 2, precision)
        self.lstm1 = layers.lstm_layers(sd, "decoder.lstm1", 1, precision)
        self.dec_convs = [layers.conv_bn_layer(sd, f"decoder.convolutions.{i}", precision, "relu", bn_owner)
                          for i in range(3)]
        self.lstm2 = layers.lstm_layers(sd, "decoder.lstm2", 2, precision)
        self.linear = ops.ConvGemm(*packing.pack_linear(sd["decoder.linear_projection.linear_layer.weight"],
                                                        sd["decoder.linear_projection.linear_layer.bias"], precision),
                                   tag="linear")
        self.postnet = layers.Postnet(sd, "postnet", precision, bn_owner)


class AutoVC(layers.PlanOwner, nn.Module):
    """AutoVC generator (Qian et al. 2019) -- B200 kernels behind the reference API (factory/AutoVC.py:182-211).

    Extra, optional attributes (not in the reference): ``precision`` ("fp32" default: split-bf16
    three-product tensor-core arithmetic, ~3e-5 from the fp32 reference | "fp16x2": fp16 activations x two-term
    fp16 weights, two products, ~4e-4, 1.45x faster | "tf32": one TF32 pass, ~1e-3 | "bf16": one bf16 pass, ~1e-2),
    ``persistent_lstm`` (one cooperative launch per LSTM layer instead of one launch per frame),
    ``collect_taps`` (keep fp32 copies of every stage in ``self.taps`` for parity tests),
    ``bn_stats`` ("running" default: every BatchNorm folded with its running statistics, eval semantics | "batch":
    every BatchNorm normalises with the statistics of the call's B x T frames and updates running_mean, running_var
    and num_batches_tracked on the device, as nn.BatchNorm1d in train mode -- how the reference's notebooks convert).

    ``forward(x, c_org, c_trg, lengths=...)`` converts a padded batch of utterances of different lengths
    (nn.utils.rnn.pack_padded_sequence semantics): utterance b has ``lengths[b]`` valid frames (a multiple of freq) and
    gets exactly the mel, mel_postnet and codes of converting ``x[b:b+1, :lengths[b]]`` alone; frames and codes past its
    end are 0, and what the input holds there is ignored."""

    def __init__(self, dim_neck, dim_emb, dim_pre, freq):
        super().__init__()
        check_hyper_parameters(dim_neck, dim_emb, dim_pre, freq)
        self.encoder = Encoder(dim_neck, dim_emb, freq)
        self.decoder = Decoder(dim_neck, dim_emb, dim_pre)
        self.postnet = Postnet()
        self.dim_neck, self.dim_emb, self.dim_pre, self.freq = dim_neck, dim_emb, dim_pre, freq
        self.precision = "fp32"
        self.persistent_lstm = True
        self.collect_taps = False
        self.taps = {}
        self.bn_stats = "running"
        self._cache = layers.PlanCache()
        self._warned_train = False

    def _plan(self):
        batch = layers.check_bn_stats(self.bn_stats) == "batch"
        return self._cache.get(self, (self.precision, self.bn_stats),
                               lambda: _Plan(self, self.precision, self if batch else None), skip_bn_stats=batch)

    # hooks of the AdaIN "2" variants (factory/_adain.py); the plain model uses the mel as is and the plain postnet
    def _encoder_features(self, x, plan, B, T):
        return x

    def _run_postnet(self, plan, mel_op, mel, B, T, taps):
        return plan.postnet(mel_op, mel, B, T, taps)

    @ops.on_device_of_input
    @torch.no_grad()
    def forward(self, x, c_org, c_trg, *, lengths=None):
        if self.training and not self._warned_train and self.bn_stats != "batch":
            warnings.warn("autoformer_b200.AutoVC runs the eval-mode forward (BatchNorm running statistics) "
                          "even in train() mode; it is an inference path (bn_stats='batch' selects train-mode "
                          "BatchNorm statistics)")
            self._warned_train = True
        if x.dim() == 4:
            x = x.squeeze(1)                                    # AutoVC.py:46
        ops._require_cuda(x)
        x = x.contiguous().float()
        c_org = c_org.contiguous().float()
        B, T, n_mel = x.shape
        F, H = self.freq, self.dim_neck
        if T % F != 0:
            raise IndexError(f"T={T} is not a multiple of freq={F} (reference indexes i+freq-1, AutoVC.py:60-66)")
        if layers.check_bn_stats(self.bn_stats) == "batch" and B * T == 1:
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {(B, 512, T)}")
        if lengths is not None:
            if self.bn_stats == "batch":
                raise ValueError("lengths with bn_stats='batch': batch statistics over padded frames match no "
                                 "per-utterance conversion; convert each length separately")
            lengths = layers.upload_lengths(lengths, B, T, x.device, F)
        plan = self._plan()
        prec = plan.precision
        dev = x.device
        taps = self.taps if self.collect_taps else None
        if taps is not None:
            taps.clear()

        # ---- encoder: concat speaker code, 3x conv+BN+ReLU, BiLSTM, code down-sampling (AutoVC.py:45-68)
        x = self._encoder_features(x, plan, B, T)
        h = ops.concat_bcast(x, c_org, T, 1, prec)
        # a padded batch: every buffer a k = 5 convolution reads gets its rows past each utterance's end zeroed (the
        # zero padding of converting it alone); conv 2's output feeds a 1x1 projection and the length-aware BiLSTM
        if lengths is not None:
            ops.zero_tail(h, 0, T, lengths)
        for i, conv in enumerate(plan.enc_convs):
            o = ops.alloc_act(B, T, 512, prec, dev)
            conv(h, B, T, out=o)
            h = o
            if lengths is not None and i < 2:
                ops.zero_tail(h, 0, T, lengths)
            if taps is not None:
                taps[f"enc_conv{i}"] = packing.act_to_float(h, prec)
        enc_out, codes = plan.enc_lstm(h, B, T, freq=F, want_out=taps is not None, **layers._lengths_kw(lengths))
        if taps is not None:
            taps["enc_lstm"] = enc_out
        flat_codes = codes.reshape(B, -1)                        # cat(codes, dim=-1), AutoVC.py:195,211
        if taps is not None:
            taps["codes"] = flat_codes
        if c_trg is None:
            return flat_codes

        # ---- decoder (AutoVC.py:197-204, 100-114)
        c_trg = c_trg.contiguous().float()
        h = ops.concat_bcast(codes, c_trg, T, F, prec)          # up-sample codes + target speaker
        f32 = torch.empty(B, T, self.dim_pre, dtype=torch.float32, device=dev) if taps is not None else None
        h = plan.lstm1[0](h, B, T, hseq_f32=f32, persistent=self.persistent_lstm)
        if taps is not None:
            taps["dec_lstm1"] = f32
        if lengths is not None:
            ops.zero_tail(h, 0, T, lengths)
        for i, conv in enumerate(plan.dec_convs):
            o = ops.alloc_act(B, T, self.dim_pre, prec, dev)
            conv(h, B, T, out=o)
            h = o
            if lengths is not None and i < 2:        # conv 2 feeds the causal lstm2
                ops.zero_tail(h, 0, T, lengths)
            if taps is not None:
                taps[f"dec_conv{i}"] = packing.act_to_float(h, prec)
        f32 = torch.empty(B, T, 1024, dtype=torch.float32, device=dev) if taps is not None else None
        h = layers.lstm_pair(plan.lstm2, h, B, T, hseq_f32=f32, persistent=self.persistent_lstm)
        if taps is not None:
            taps["dec_lstm2"] = f32
        mel = torch.empty(B, T, 80, dtype=torch.float32, device=dev)
        mel_op = ops.alloc_act(B, T, 80, prec, dev)
        plan.linear(h, B, T, out=mel_op, out2=mel.view(B * T, 80))

        # ---- postnet + residual (AutoVC.py:173-179, 206-209)
        if lengths is None:
            post = self._run_postnet(plan, mel_op, mel, B, T, taps)
        else:
            ops.zero_tail(mel_op, 0, T, lengths)
            post = plan.postnet(mel_op, mel, B, T, taps, lengths=lengths)
            ops.zero_tail(mel, 0, T, lengths)
            ops.zero_tail(post, 0, T, lengths)
        if taps is not None:
            taps["mel"] = mel
            taps["mel_postnet"] = post
        return mel.unsqueeze(1), post.unsqueeze(1), flat_codes
