"""Variable-length batches vs length buckets, fp16x2, one GPU (DESIGN.md "Variable-length batches").

(a) 2,048 utterances, T uniform over {128, 160, ..., 1024} (seeded): sharding.plan + pipeline.convert_batches (one
    batch per exact length, under-filled tails paired on two streams) vs pipeline.convert_utterances (sorted, 4 batches
    of 512 padded to their longest utterance, per-utterance lengths); outputs compared per utterance.
(b) the config-5 distribution (bench.py sub_cfg5: random.Random(1234)) at 16,384 utterances, both ways.
(c) the headline 512 x 128 batch: lengths=None vs lengths=[128] * 512 -- the cost of the 13 zero-tail launches.
(d) LstmDV enrolment of 256 utterances over the same lengths: one call per exact length vs embed_utterances.

Each timed window is one pass after an untimed warm-up pass of the same schedule, between CUDA events, after a device
synchronise; the card's name and power limit are read (nvidia-smi --query-gpu, read-only) in the same run.  Inputs of
(a), (b), (d) are hundreds of MB to GB, larger than the 126 MB L2.

    python scripts/ragged_timing.py --out /tmp/ragged_timing
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def timed(fn, reps=1):
    fn()                                    # warm-up: same shapes, same schedule
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return best, out


def utterances(lengths, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    mels = [torch.rand(t, 80, generator=g, device=dev) * 6 - 5 for t in lengths]
    c = torch.nn.functional.normalize(torch.randn(2, len(lengths), 256, generator=g, device=dev), dim=-1)
    return mels, c[0].contiguous(), c[1].contiguous()


def autovc_both_ways(model, lengths, seed, dev, check):
    from autoformer_b200 import pipeline, sharding
    mels, c_org, c_trg = utterances(lengths, seed, dev)
    plan = sharding.plan(lengths, 1, 512, cost=sharding.autovc_cost_for("fp16x2"))[0]

    def bucketed():
        batches = []
        for T, ids in plan:
            idx = torch.as_tensor(ids, device=dev)
            batches.append((torch.stack([mels[i] for i in ids]), c_org[idx], c_trg[idx]))
        return plan, pipeline.convert_batches(model, batches, reduce=lambda out: out[1])

    def ragged():
        return pipeline.convert_utterances(model, mels, c_org, c_trg, max_batch=512)

    ms_b, (pl, outs_b) = timed(bucketed)
    ms_r, outs_r = timed(ragged)
    rec = dict(utterances=len(lengths), frames=int(sum(lengths)), bucketed_batches=len(plan),
               ragged_batches=len(sharding.make_ragged_batches(lengths, 512, model.freq)),
               bucketed_ms=round(ms_b, 2), ragged_ms=round(ms_r, 2), speedup=round(ms_b / ms_r, 3))
    if check:
        worst = 0.0
        for (T, ids), post in zip(pl, outs_b):
            for k, i in enumerate(ids):
                a, b = post[k, 0].double(), outs_r[i].double()
                worst = max(worst, float((a - b).norm() / b.norm()))
        rec["max_rel_l2_bucketed_vs_ragged"] = worst
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for ragged_timing.json")
    ap.add_argument("--cfg5-utterances", type=int, default=16384)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_timing.py needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    from oracle import templates
    from oracle.seeded import seeded_state_dict
    from autoformer_b200.factory.AutoVC import AutoVC
    from autoformer_b200.factory.LstmDV import LstmDV
    from autoformer_b200 import pipeline
    dev = torch.device("cuda:0")
    res = dict(device=device_info(), precision="fp16x2", torch=torch.__version__, when=time.strftime("%Y-%m-%d %H:%M"))

    args_vc = (32, 256, 512, 32)
    model = AutoVC(*args_vc).to(dev).eval()
    model.load_state_dict(seeded_state_dict(templates.autovc_template(*args_vc), 0))
    model.precision = "fp16x2"
    model(torch.zeros(2, 128, 80, device=dev), torch.zeros(2, 256, device=dev), torch.zeros(2, 256, device=dev))
    model.freeze_weights()

    rng = random.Random(7)
    res["a_2048_uniform"] = autovc_both_ways(model, [rng.choice(range(128, 1025, 32)) for _ in range(2048)], 1, dev, True)
    print(json.dumps(res["a_2048_uniform"]), flush=True)
    rng = random.Random(1234)                        # bench.py sub_cfg5's generator
    res["b_cfg5"] = autovc_both_ways(model, [rng.choice(range(128, 1025, 32)) for _ in range(args.cfg5_utterances)], 2,
                                     dev, False)
    print(json.dumps(res["b_cfg5"]), flush=True)

    g = torch.Generator(device=dev).manual_seed(3)
    x = torch.rand(512, 128, 80, generator=g, device=dev) * 6 - 5
    c = torch.nn.functional.normalize(torch.randn(512, 256, generator=g, device=dev), dim=-1)
    fixed, full = [], []
    for _ in range(5):                               # alternate the two forms, best of 5 each
        fixed.append(timed(lambda: model(x, c, c))[0])
        full.append(timed(lambda: model(x, c, c, lengths=[128] * 512))[0])
    res["c_headline_512x128"] = dict(lengths_none_ms=round(min(fixed), 3), lengths_full_ms=round(min(full), 3),
                                     mask_overhead_ms=round(min(full) - min(fixed), 3),
                                     bit_identical=all(torch.equal(a, b) for a, b in
                                                       zip(model(x, c, c), model(x, c, c, lengths=[128] * 512))))
    print(json.dumps(res["c_headline_512x128"]), flush=True)

    dv = LstmDV().to(dev)
    dv.load_state_dict(seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5))
    dv.precision = "fp16x2"
    dv.freeze_weights()
    rng = random.Random(11)
    lens = [rng.choice(range(128, 1025, 32)) for _ in range(256)]
    mels, _, _ = utterances(lens, 4, dev)

    def dv_bucketed():
        from autoformer_b200 import sharding
        out = torch.empty(len(mels), 256, device=dev)
        for T, ids in sharding.make_batches(sharding.bucket_by_length(lens), 64):
            out[torch.as_tensor(ids, device=dev)] = dv(torch.stack([mels[i] for i in ids]))
        return out

    ms_b, e_b = timed(dv_bucketed)
    ms_r, e_r = timed(lambda: pipeline.embed_utterances(dv, mels, max_batch=64))
    res["d_lstmdv_256"] = dict(utterances=256, bucketed_ms=round(ms_b, 2), ragged_ms=round(ms_r, 2),
                               speedup=round(ms_b / ms_r, 3),
                               max_rel_l2_bucketed_vs_ragged=float(((e_b - e_r).norm(dim=1) / e_r.norm(dim=1)).max()))
    print(json.dumps(res["d_lstmdv_256"]), flush=True)
    with open(os.path.join(args.out, "ragged_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
