"""Variable-length MelGAN batches vs length buckets, one GPU (DESIGN.md "Variable-length batches").

(a) B = 32, T = 1000, "fp16s": lengths=[1000] * 32 against lengths=None -- the cost of the halo and zero-tail launches a
    padded batch adds when every utterance has the full length (outputs compared bit for bit).
(b) 256 utterances, T uniform in 128 ... 1000 (seeded), "fp16s":
      ragged    the batches of pipeline.vocode_utterances (sorted, 32 per batch, padded to their even longest) with
                per-utterance lengths;
      bucketed  one generator call per distinct length (all utterances of that length in one batch);
      padded    the same padded batches WITHOUT lengths -- wrong at every shorter utterance's end, shown only for what
                the skipped tiles save;
    the three on batches assembled beforehand, plus pipeline.vocode_utterances end to end (its batch assembly included).
(b2) one unsorted batch, B = 32, T = 1000, lengths uniform in 200 ... 1000: lengths against None (what the skipped tiles
    save when the batch is far from one length).
(c) the config-4 pipeline on the same lengths (LstmDV and AutoVC "fp16x2", MelGAN "fp16s"):
    pipeline.convert_and_vocode_utterances against one pipeline.convert_and_vocode call per distinct length.

Each form is warmed up once on its own schedule, then timed between CUDA events after a device synchronise; the forms
are alternated and the best of the repetitions is kept.  The card's name and power limit are read (nvidia-smi
--query-gpu, read-only) in the same run.

    python scripts/ragged_vocode_timing.py --out /tmp/ragged_vocode_timing
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


def once(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def best_of(fns, reps):
    """{name: best ms} with the forms alternated, each warmed up first; also the last outputs."""
    outs = {k: fn() for k, fn in fns.items()}           # warm-up of every shape the timed windows use
    torch.cuda.synchronize()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            t, outs[k] = once(fn)
            ms[k].append(t)
    return {k: round(min(v), 3) for k, v in ms.items()}, outs


def by_length(lengths):
    groups = {}
    for i, n in enumerate(lengths):
        groups.setdefault(n, []).append(i)
    return groups


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for ragged_vocode_timing.json")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_vocode_timing.py needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    from oracle import templates
    from oracle.seeded import seeded_state_dict
    from autoformer_b200 import pipeline, sharding
    from autoformer_b200.factory.AutoVC import AutoVC
    from autoformer_b200.factory.LstmDV import LstmDV
    from autoformer_b200.melgan.modules import Generator
    dev = torch.device("cuda:0")
    res = dict(device=device_info(), torch=torch.__version__, when=time.strftime("%Y-%m-%d %H:%M"))

    gen = Generator(80, 32, 3)
    gen.load_state_dict(seeded_state_dict(templates.melgan_template(), 4))
    gen = gen.to(dev).eval()
    gen.precision = "fp16s"
    gen.freeze_weights()
    g = torch.Generator(device=dev).manual_seed(3)

    # (a) one length: what the extra launches cost
    x = torch.rand(32, 80, 1000, generator=g, device=dev) * 6 - 5
    ms, outs = best_of({"lengths_none": lambda: gen(x), "lengths_full": lambda: gen(x, lengths=[1000] * 32)}, args.reps)
    res["a_b32_t1000_fp16s"] = dict(lengths_none_ms=ms["lengths_none"], lengths_full_ms=ms["lengths_full"],
                                    overhead_ms=round(ms["lengths_full"] - ms["lengths_none"], 3),
                                    bit_identical=torch.equal(outs["lengths_none"], outs["lengths_full"]))
    print(json.dumps(res["a_b32_t1000_fp16s"]), flush=True)

    # (b) 256 utterances of mixed lengths
    rng = random.Random(7)
    lens = [rng.randint(128, 1000) for _ in range(256)]
    mels = [torch.rand(n, 80, generator=g, device=dev) * 6 - 5 for n in lens]
    groups = by_length(lens)
    batches = []
    for T, ids in sharding.make_ragged_batches(lens, 32, 1):
        T_pad = T + T % 2
        xb = torch.zeros(len(ids), 80, T_pad, device=dev)
        for k, i in enumerate(ids):
            xb[k, :, :lens[i]] = mels[i].t()
        batches.append(xb)

    batch_lens = [[lens[i] for i in ids] for _, ids in sharding.make_ragged_batches(lens, 32, 1)]
    buckets = [(ids, torch.stack([mels[i] for i in ids]).transpose(1, 2).contiguous()) for ids in groups.values()]

    def bucketed():
        out = [None] * len(mels)
        for ids, xb in buckets:
            w = gen(xb).squeeze(1)
            for k, i in enumerate(ids):
                out[i] = w[k]
        return out

    ms, outs = best_of({"ragged": lambda: [gen(xb, lengths=bl) for xb, bl in zip(batches, batch_lens)],
                        "bucketed": bucketed,
                        "padded_no_lengths": lambda: [gen(xb) for xb in batches],
                        "vocode_utterances": lambda: pipeline.vocode_utterances(gen, mels, max_batch=32)}, args.reps)
    worst = max(float((a.double() - b.double()).norm() / b.double().norm())
                for a, b in zip(outs["vocode_utterances"], outs["bucketed"]))
    padded_frames = sum(xb.shape[0] * xb.shape[2] for xb in batches)
    res["b_256_uniform_128_1000_fp16s"] = dict(
        utterances=256, frames=sum(lens), distinct_lengths=len(groups), ragged_batches=len(batches),
        padded_frames=padded_frames, valid_share=round(sum(lens) / padded_frames, 3),
        ragged_ms=ms["ragged"], bucketed_ms=ms["bucketed"], padded_no_lengths_ms=ms["padded_no_lengths"],
        vocode_utterances_ms=ms["vocode_utterances"], speedup_vs_bucketed=round(ms["bucketed"] / ms["ragged"], 3),
        max_rel_l2_ragged_vs_bucketed=worst)
    print(json.dumps(res["b_256_uniform_128_1000_fp16s"]), flush=True)

    rng = random.Random(5)
    lens32 = [rng.randint(200, 1000) for _ in range(32)]
    lens32[0] = 1000
    ms, outs = best_of({"lengths_none": lambda: gen(x), "lengths": lambda: gen(x, lengths=lens32)}, args.reps)
    res["b2_b32_t1000_uniform_200_1000_fp16s"] = dict(
        valid_share=round(sum(lens32) / 32000, 3), lengths_none_ms=ms["lengths_none"], lengths_ms=ms["lengths"],
        saved_ms=round(ms["lengths_none"] - ms["lengths"], 3))
    print(json.dumps(res["b2_b32_t1000_uniform_200_1000_fp16s"]), flush=True)

    # (c) config 4 end to end on the same lengths
    args_vc = (32, 256, 512, 32)
    vc = AutoVC(*args_vc).to(dev).eval()
    vc.load_state_dict(seeded_state_dict(templates.autovc_template(*args_vc), 0))
    vc.precision = "fp16x2"
    dv = LstmDV().to(dev).eval()
    dv.load_state_dict(seeded_state_dict(templates.lstmdv_template(), 3, lstm_gain=1.5))
    dv.precision = "fp16x2"
    vc.freeze_weights()
    dv.freeze_weights()
    trg = [torch.rand(n, 80, generator=g, device=dev) * 6 - 5 for n in lens]

    def c4_bucketed():
        out = [None] * len(mels)
        for n, ids in groups.items():
            _, w, _, _ = pipeline.convert_and_vocode(dv, vc, gen, torch.stack([mels[i] for i in ids]),
                                                     torch.stack([trg[i] for i in ids]))
            for k, i in enumerate(ids):
                out[i] = w[k]
        return out

    ms, outs = best_of({"ragged": lambda: pipeline.convert_and_vocode_utterances(dv, vc, gen, mels, trg)[1],
                        "bucketed": c4_bucketed}, max(2, args.reps // 2))
    worst = max(float((a.double() - b.double()).norm() / b.double().norm()) for a, b in zip(outs["ragged"], outs["bucketed"]))
    res["c_config4_256_uniform_128_1000"] = dict(
        precision="LstmDV / AutoVC fp16x2, MelGAN fp16s", ragged_ms=ms["ragged"], bucketed_ms=ms["bucketed"],
        speedup=round(ms["bucketed"] / ms["ragged"], 3), max_rel_l2_wav_ragged_vs_bucketed=worst)
    print(json.dumps(res["c_config4_256_uniform_128_1000"]), flush=True)
    with open(os.path.join(args.out, "ragged_vocode_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
