"""Batched conversion pipeline: speaker embedding -> AutoVC conversion -> MelGAN vocoding (BASELINE config 4).

Follows the reference's own recipe for utterances whose length is not a multiple of ``freq``: zero-pad the mel at
the end, convert, trim the padding off again (util/evaluate.py:36-43 ``crop_mel`` pads with constant 0;
:85-92 trims ``mel_trans`` back), then vocode ``mel_trans.transpose(2, 1)`` (conversion.ipynb cell 14,
util/evaluate.py:96-98).  ``convert`` and ``convert_batches`` take batches whose utterances share one T (plain zero
padding changes the result, SURVEY.md 5); ``convert_utterances``, ``embed_utterances``, ``vocode_utterances`` and
``convert_and_vocode_utterances`` take utterances of any length and batch them with per-utterance lengths, which gives
each one exactly its result computed alone."""
import os

import numpy as np
import torch


def crop_mel(mel, len_crop, rng=None):
    """The Evaluator's ``crop_mel`` (util/evaluate.py:36-50): numpy (T, 80) -> (tensor (1, len_crop, 80), pad_size).

    T < len_crop: zero-pad at the END up to ``len_crop`` (pad_size = len_crop - T); T == len_crop: as is; T > len_crop:
    a window of len_crop frames at a random offset in [0, T - len_crop) drawn from ``rng`` (default: numpy's global
    generator, like the reference) and pad_size = 0."""
    mel = np.asarray(mel)
    T = mel.shape[0]
    pad = 0
    if T < len_crop:
        pad = int(len_crop - T)
        mel = np.pad(mel, [(0, pad)] + [(0, 0)] * (mel.ndim - 1), mode="constant", constant_values=0)
    elif T > len_crop:
        left = (rng or np.random).randint(0, T - len_crop)
        mel = mel[left:left + len_crop]
    return torch.from_numpy(np.ascontiguousarray(mel)).unsqueeze(0), pad


@torch.no_grad()
def convert_cropped(model, mel_np, emb_org, emb_trg, len_crop, trim=True, device="cuda"):
    """One utterance through the Evaluator's recipe: ``crop_mel`` to ``len_crop`` -> ``model(x, c_org, c_trg)`` ->
    trim the padded frames (util/evaluate.py:63-64, 83-92 with ``isPlay``).  Returns (1, T', 80)."""
    x, pad = crop_mel(mel_np, len_crop)
    _, mel_trans, _ = model(x.to(device).float(), emb_org, emb_trg)
    mel_trans = mel_trans.squeeze(1)
    return mel_trans[:, :len_crop - pad, :] if (trim and pad > 0) else mel_trans


def pad_to_multiple(mel, multiple):
    """(B, T, 80) -> ((B, T', 80) zero-padded at the end, pad_size)   (util/evaluate.py:36-43)."""
    T = mel.shape[1]
    pad = (-T) % multiple
    if pad:
        mel = torch.nn.functional.pad(mel, (0, 0, 0, pad))
    return mel, pad


@torch.no_grad()
def convert(model, mel_src, emb_org, emb_trg, mel_target=None):
    """Conversion with pad -> convert -> trim.  Returns the converted mel (B, T, 80).

    ``mel_target`` (B, T2, 80) selects the ``*_Adjust`` call of the reference's Evaluator (util/evaluate.py:79-80:
    ``model(mel_source, emb_org, emb_trg, True, mel_target)``, 4-tuple return); otherwise the plain 3-argument call."""
    T = mel_src.shape[1]
    x, pad = pad_to_multiple(mel_src, model.freq)
    if mel_target is not None:
        xt, _ = pad_to_multiple(mel_target, model.freq)
        _, _, mel_trans, _ = model(x, emb_org, emb_trg, True, xt)   # util/evaluate.py:79-80
    else:
        _, mel_trans, _ = model(x, emb_org, emb_trg)             # util/evaluate.py:83
    mel_trans = mel_trans.squeeze(1)                             # :85
    return mel_trans[:, :T, :] if pad else mel_trans             # :87-90


@torch.no_grad()
def convert_and_vocode(embedder, model, generator, mel_src, mel_trg_ref):
    """mel_src (B, T, 80): utterances to convert; mel_trg_ref (B, T2, 80): utterances of the target speakers.

    Returns (converted mel (B, T, 80), waveform (B, 256 T), emb_org, emb_trg)."""
    if mel_src.shape == mel_trg_ref.shape:
        # utterances are independent in the embedder, so both sets share one launch sequence: at B = 32 the LSTM
        # recurrences are latency-bound and twice the rows per frame cost almost nothing extra
        emb = embedder(torch.cat((mel_src, mel_trg_ref), dim=0))     # LstmDV d-vectors (factory/LstmDV.py:19-24)
        emb_org, emb_trg = emb[:mel_src.shape[0]], emb[mel_src.shape[0]:]
    else:
        emb_org = embedder(mel_src)
        emb_trg = embedder(mel_trg_ref)
    mel_trans = convert(model, mel_src, emb_org, emb_trg)
    wav = generator(mel_trans.transpose(2, 1).contiguous()).squeeze(1)   # MelVocoder.inverse (interface.py:43-53)
    return mel_trans, wav, emb_org, emb_trg


class StreamingConverter:
    """Batched conversion from HOST tensors to HOST tensors with the PCIe copies overlapped with compute.

    ``submit(x, c_org, c_trg)`` (pinned or pageable CPU tensors) enqueues: H2D on a copy stream -> ``model`` on the
    compute stream -> D2H of ``(mel, mel_postnet, codes)`` into pinned buffers on a second copy stream, and returns
    the result of the PREVIOUS submission (or None): while batch i computes, batch i+1 uploads and batch i-1
    downloads.  ``flush()`` returns the last result.  Results are pinned host tensors owned by the converter and are
    overwritten two submissions later (double buffering) -- copy them if they must live longer.
    The model runs in submission order on the one compute stream, so a model with ``bn_stats = "batch"`` updates its
    BatchNorm running buffers in that order too.
    """

    def __init__(self, model, device=None):
        self.model = model
        self.device = torch.device(device or next(model.parameters()).device)
        self.h2d = torch.cuda.Stream(self.device)
        self.d2h = torch.cuda.Stream(self.device)
        self.slot = 0
        self.dev_in = [None, None]
        self.host_out = [None, None]
        self.done = [None, None]
        self.pending = None

    def _pinned_like(self, outs, slot):
        bufs = self.host_out[slot]
        if bufs is None or any(b.shape != o.shape for b, o in zip(bufs, outs)):
            bufs = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs]
            self.host_out[slot] = bufs
        return bufs

    @torch.no_grad()
    def submit(self, x, c_org, c_trg):
        s = self.slot
        compute = torch.cuda.current_stream(self.device)
        if self.done[s] is not None:
            self.done[s].synchronize()              # the slot's previous download has finished: buffers are free
        with torch.cuda.stream(self.h2d):
            dev = [t.to(self.device, non_blocking=True) for t in (x, c_org, c_trg)]
            up = torch.cuda.Event()
            up.record(self.h2d)
        self.dev_in[s] = dev                        # keep alive until the compute stream has consumed them
        compute.wait_event(up)
        outs = self.model(*dev)
        for t in dev:
            t.record_stream(compute)
        ready = torch.cuda.Event()
        ready.record(compute)
        bufs = self._pinned_like(outs, s)
        with torch.cuda.stream(self.d2h):
            self.d2h.wait_event(ready)
            for b, o in zip(bufs, outs):
                b.copy_(o, non_blocking=True)
                o.record_stream(self.d2h)
            ev = torch.cuda.Event()
            ev.record(self.d2h)
        self.done[s] = ev
        prev, self.pending = self.pending, (s, ev)
        self.slot ^= 1
        if prev is None:
            return None
        prev[1].synchronize()
        return tuple(self.host_out[prev[0]])

    def flush(self):
        if self.pending is None:
            return None
        s, ev = self.pending
        self.pending = None
        ev.synchronize()
        return tuple(self.host_out[s])


def _ragged_batches(mels, max_batch, multiple):
    """(T_batch, ids, padded input [n][T_batch][80], lengths) per variable-length batch (sharding.make_ragged_batches);
    utterance i padded with zeros to a multiple of `multiple` frames (util/evaluate.py:36-43), then to T_batch."""
    from . import sharding
    for T_batch, ids in sharding.make_ragged_batches([m.shape[0] for m in mels], max_batch, multiple):
        lens = [(mels[i].shape[0] + multiple - 1) // multiple * multiple for i in ids]
        x = mels[ids[0]].new_zeros(len(ids), T_batch, mels[ids[0]].shape[1])
        for k, i in enumerate(ids):
            x[k, :mels[i].shape[0]] = mels[i]
        yield T_batch, ids, x, lens


@torch.no_grad()
def convert_utterances(model, mels, c_org, c_trg, max_batch=512):
    """Convert utterances of any lengths: mels is a list of (T_i, 80) device tensors, c_org / c_trg (N, dim_emb).
    Each is zero-padded to a multiple of ``model.freq`` (the reference's recipe, as ``convert``), the utterances are
    batched by ``sharding.make_ragged_batches`` and every batch runs once with per-utterance lengths.  Returns the
    list of converted mels (mel_postnet, (T_i, 80)) in input order, each trimmed to T_i.  An AdaIN "2" model must have
    ``adain_stats = "utterance"`` (its forward refuses lengths otherwise); each utterance is then styled with its own
    features, the Evaluator's ``isAdain`` recipe (util/evaluate.py:69-71, 81-82)."""
    out = [None] * len(mels)
    for _, ids, x, lens in _ragged_batches(mels, max_batch, model.freq):
        idx = torch.as_tensor(ids, device=c_org.device)
        _, post, _ = model(x, c_org[idx], c_trg[idx], lengths=lens)
        post = post.squeeze(1)
        for k, i in enumerate(ids):
            out[i] = post[k, :mels[i].shape[0]]
    return out


@torch.no_grad()
def embed_utterances(embedder, mels, max_batch=64):
    """LstmDV d-vectors of utterances of any lengths (list of (T_i, 80) device tensors) with variable-length batches:
    row i of the (N, dim_emb) result is the embedder's output for mels[i] alone.  The default batch of 64 keeps the
    small-batch recurrence kernels (their cost per frame does not grow up to 64 utterances)."""
    out = [None] * len(mels)
    for _, ids, x, lens in _ragged_batches(mels, max_batch, 1):
        e = embedder(x, lengths=lens)
        e = e[1] if isinstance(e, tuple) else e                  # the classifier twin returns (predictions, d_vec)
        for k, i in enumerate(ids):
            out[i] = e[k]
    return torch.stack(out)


@torch.no_grad()
def vocode_utterances(generator, mels, max_batch=32):
    """MelGAN waveforms of utterances of any lengths: mels is a list of (T_i, 80) device tensors, T_i >= 4.  The
    utterances are batched by ``sharding.make_ragged_batches`` on their exact lengths and each batch is vocoded once
    with per-utterance lengths.  A batch is padded to an even number of frames, so that every stage of 32 / 64 / 128
    channels takes the fused ResnetBlock kernels (their stage length 64 T must be a multiple of 128).  Returns the list
    of waveforms (hop_length * T_i,) in input order, each what the generator gives for the utterance alone."""
    from . import sharding
    out = [None] * len(mels)
    hop = generator.hop_length
    for T_batch, ids in sharding.make_ragged_batches([m.shape[0] for m in mels], max_batch, 1):
        T_pad = T_batch + T_batch % 2
        x = mels[ids[0]].new_zeros(len(ids), mels[ids[0]].shape[1], T_pad)
        lens = [mels[i].shape[0] for i in ids]
        for k, i in enumerate(ids):
            x[k, :, :lens[k]] = mels[i].t()
        wav = generator(x, lengths=lens).squeeze(1)
        for k, i in enumerate(ids):
            out[i] = wav[k, :hop * lens[k]]
    return out


@torch.no_grad()
def convert_and_vocode_utterances(embedder, model, generator, mels_src, mels_trg_ref):
    """``convert_and_vocode`` on utterances of any lengths (lists of (T_i, 80) and (T2_i, 80) device tensors):
    ``embed_utterances`` -> ``convert_utterances`` -> ``vocode_utterances``, each with variable-length batches.
    Returns (converted mels [(T_i, 80)], waveforms [(256 T_i,)], emb_org, emb_trg), in input order."""
    n = len(mels_src)
    emb = embed_utterances(embedder, list(mels_src) + list(mels_trg_ref))
    emb_org, emb_trg = emb[:n], emb[n:]
    mels = convert_utterances(model, mels_src, emb_org, emb_trg)
    return mels, vocode_utterances(generator, mels), emb_org, emb_trg


# ------------------------------------------------------------------------------------------------ side-by-side batches
PAIR_BELOW = 256        # a batch of at most this many utterances takes one batch group of the persistent LSTM grid
_SIDE_STREAMS = {}


def _side_streams(device):
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = (torch.cuda.Stream(device=key), torch.cuda.Stream(device=key))
    return _SIDE_STREAMS[key]


@torch.no_grad()
def convert_batches(model, batches, reduce=None, pair_below=PAIR_BELOW):
    """Run ``model(x, c_org, c_trg)`` over a list of batches (each one exact length, as the sweep of BASELINE configs[4]
    buckets them) and return ``reduce(outputs)`` per batch in the order given (``reduce`` defaults to the 3-tuple itself).

    The recurrences are latency-bound: a batch of 200 utterances costs the LSTM kernels as much per frame as one of 512,
    and takes half of the SMs doing it.  Batches of at most ``pair_below`` utterances (the under-filled last batch of
    every length bucket) therefore run TWO AT A TIME on two streams, with each persistent LSTM grid capped at half of the
    device (``ops.LSTM_CTA_BUDGET``) so that both cooperative launches are resident together -- measured
    (scripts/two_stream_probe.py): 212 x 1024 + 180 x 992 frames 71.6 -> 52.3 ms, outputs bit-equal to the one-stream
    run.  Utterances stay independent and every batch keeps its exact length; only the schedule changes.

    A model with ``bn_stats = "batch"`` updates its BatchNorm running buffers on every call, so the order of the calls
    matters: its batches run in the order given on the current stream, exactly as a plain loop of ``model(*b)``."""
    from . import ops
    reduce = reduce or (lambda out: out)
    if getattr(model, "bn_stats", "running") == "batch":
        return [reduce(model(*b)) for b in batches]
    results = [None] * len(batches)
    small = [i for i, b in enumerate(batches) if 64 < b[0].shape[0] <= pair_below]
    # (batches of <= 64 utterances take the weight-stationary kernels, whose grids fill the device: no pairing)
    if os.environ.get("AVC_LSTM_NO_COOP") is not None or not getattr(model, "persistent_lstm", True):
        small = []      # without the cooperative attribute two grids could each be half resident and wait on one another
    small.sort(key=lambda i: -batches[i][0].shape[1])           # neighbours in length: the two streams finish together
    paired = set(small[:len(small) // 2 * 2])
    for i, b in enumerate(batches):
        if i not in paired:
            results[i] = reduce(model(*b))
    if paired:
        dev = batches[small[0]][0].device
        cur = torch.cuda.current_stream(dev)
        streams = _side_streams(dev)
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        saved = ops.LSTM_CTA_BUDGET
        ops.LSTM_CTA_BUDGET = n_sm // 2
        try:
            for k in range(0, len(paired), 2):
                for s in streams:
                    s.wait_stream(cur)
                for s, i in zip(streams, small[k:k + 2]):
                    with torch.cuda.stream(s):
                        results[i] = reduce(model(*batches[i]))
                        for t in (results[i] if isinstance(results[i], (tuple, list)) else (results[i],)):
                            if torch.is_tensor(t):
                                t.record_stream(cur)
                for s in streams:
                    cur.wait_stream(s)
        finally:
            ops.LSTM_CTA_BUDGET = saved
    return results
