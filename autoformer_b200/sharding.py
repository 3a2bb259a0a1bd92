"""Utterance-sharded data parallelism for the conversion path (SURVEY.md 8e, BASELINE config 5).

In eval mode every utterance is independent, so the path shards by utterance with NO data-path collective:
weights are replicated, each rank converts its own batches, and ``torch.distributed`` (NCCL over NVLink on the GPU
box, gloo in the CPU tests) is used only to gather fixed-size per-rank records (frames, time, checksum) and, on
request, the outputs.  Two ways to batch utterances of different lengths:

- ``plan``: bucketed by EXACT length, one launch sequence per distinct length (plain zero padding would change the
  result: the backward LSTM and LstmDV's last step would see the padding, SURVEY.md 5);
- ``plan_ragged``: sorted by length and cut into full batches, each padded to its longest utterance and run with
  per-utterance ``lengths`` (AutoVC / LstmDV ``forward(..., lengths=...)``), which gives every utterance exactly the
  result of converting it alone.  The recurrences cost per frame whatever the batch size, so a few full batches are
  cheaper than one under-filled batch per length.
"""
from collections import defaultdict

import torch
import torch.distributed as dist


def bucket_by_length(lengths):
    """lengths[i] = frames of utterance i -> {T: [utterance ids]} (ids ascending)."""
    buckets = defaultdict(list)
    for i, t in enumerate(lengths):
        buckets[int(t)].append(i)
    return dict(sorted(buckets.items()))


def make_batches(buckets, max_batch=512):
    """Split every bucket into batches of at most ``max_batch`` utterances: [(T, [ids])]."""
    batches = []
    for t, ids in buckets.items():
        for s in range(0, len(ids), max_batch):
            batches.append((t, ids[s:s + max_batch]))
    return batches


def frames_cost(T, n):
    """Cost of a batch of n utterances x T frames when only the frame count matters."""
    return float(T * n)


# per precision: (microseconds per frame of the LSTM layers, microseconds per utterance-frame of everything else)
_AUTOVC_COST = {"fp32": (47.5, 0.0596), "fp16x2": (29.8, 0.0421)}


PAIRED_LSTM_SHARE = 0.6      # of the per-frame term, for a batch that runs beside another one (pipeline.convert_batches)


def autovc_cost(T, n, precision="fp32", pair_below=256):
    """Measured cost model of one AutoVC conversion batch on a B200, in microseconds: the LSTM layers run one tile row
    per frame whatever the batch size up to 512 (split format: 47.5 us per frame, profiles/r01_bench_final_1gpu:
    6.08 ms / 128 frames; fp16x2: 29.8 us, profiles/r01_bench_fp16x2_1gpu: 3.82 ms / 128), everything else scales with
    utterances x frames (3.9 ms resp. 2.76 ms / 65,536).  A 212-utterance tail batch therefore costs 77 % of a full
    one for 41 % of its frames, which a frames-only balance does not see; run beside another tail batch
    (``pair_below``; 0 = the batches run one after the other) it costs about 0.6 of its frame time."""
    per_frame, per_utt_frame = _AUTOVC_COST.get(precision, _AUTOVC_COST["fp32"])
    if 64 < n <= pair_below:
        # pipeline.convert_batches runs such batches two at a time on two streams: the pair shares the frame time of the
        # recurrences (measured: 212 x 1024 + 180 x 992 frames 71.6 ms one after the other, 52.3 ms side by side)
        per_frame *= PAIRED_LSTM_SHARE
    return float(T) * (per_frame + per_utt_frame * n)


def autovc_cost_for(precision):
    return lambda T, n: autovc_cost(T, n, precision)


def assign_batches(batches, world_size, cost=frames_cost):
    """Greedy longest-processing-time assignment by ``cost(T, n)``.  Deterministic, identical on every rank.

    Returns a list (one entry per rank) of batch lists."""
    c = [cost(t, len(ids)) for t, ids in batches]
    order = sorted(range(len(batches)), key=lambda i: (-c[i], i))
    load = [0.0] * world_size
    out = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda k: (load[k], k))
        out[r].append(batches[i])
        load[r] += c[i]
    return out


def plan(lengths, world_size, max_batch=512, cost=frames_cost):
    return assign_batches(make_batches(bucket_by_length(lengths), max_batch), world_size, cost)


def make_ragged_batches(lengths, max_batch=512, multiple=1):
    """Variable-length batches: each length is padded up to `multiple` (AutoVC's freq), utterances are sorted by padded
    length (descending, ties by id) and consecutive runs of ``max_batch`` form the batches.  Returns [(T_batch, ids)]
    with T_batch the longest padded length of the run."""
    padded = [(int(t) + multiple - 1) // multiple * multiple for t in lengths]
    order = sorted(range(len(padded)), key=lambda i: (-padded[i], i))
    return [(padded[order[s]], order[s:s + max_batch]) for s in range(0, len(order), max_batch)]


def plan_ragged(lengths, world_size, max_batch=512, multiple=1, cost=frames_cost):
    return assign_batches(make_ragged_batches(lengths, max_batch, multiple), world_size, cost)


def gather_records(record, device=None):
    """All-gather one fixed-size float64 record per rank; returns a (world, len) tensor on every rank."""
    rec = torch.as_tensor(record, dtype=torch.float64, device=device)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return rec.unsqueeze(0)
    out = [torch.zeros_like(rec) for _ in range(dist.get_world_size())]
    dist.all_gather(out, rec)
    return torch.stack(out)


def gather_outputs(local, total_count, ids, dst=0, chunk=4096):
    """Gather per-utterance outputs of equal shape to rank ``dst``: local (n_local, ...) with global ids ``ids``.

    Point-to-destination: only ``dst`` allocates the (total_count, ...) result and a receive block of at most ``chunk``
    utterances; the other ranks send their rows in chunks and allocate nothing (an all_gather would hold
    world x max_count x shape on EVERY rank -- 65,536 waveforms at 8 ranks do not fit).  Returns the full tensor on
    ``dst`` and None elsewhere.  Outside any timed region in bench.py."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        full = local.new_zeros((total_count,) + tuple(local.shape[1:]))
        full[torch.as_tensor(ids, device=local.device, dtype=torch.long)] = local
        return full
    world, rank = dist.get_world_size(), dist.get_rank()
    counts = [int(c) for c in gather_records([float(len(ids))], device=local.device).flatten().tolist()]
    ids_t = torch.as_tensor(ids, dtype=torch.long, device=local.device)
    tail = tuple(local.shape[1:])
    if rank != dst:
        for s in range(0, counts[rank], chunk):
            dist.send(ids_t[s:s + chunk].contiguous(), dst)
            dist.send(local[s:s + chunk].contiguous(), dst)
        return None
    full = local.new_zeros((total_count,) + tail)
    full[ids_t] = local
    for src in range(world):
        if src == dst:
            continue
        for s in range(0, counts[src], chunk):
            n = min(chunk, counts[src] - s)
            rid = torch.empty(n, dtype=torch.long, device=local.device)
            rv = local.new_empty((n,) + tail)
            dist.recv(rid, src)
            dist.recv(rv, src)
            full[rid] = rv
    return full
