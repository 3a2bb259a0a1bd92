"""Per-utterance AdaIN statistics (adain_stats = "utterance") on one GPU (DESIGN.md "Per-utterance AdaIN statistics").

(a) 512 Evaluator-style utterances of 176 frames (util/evaluate.py:69-71: one self-styled conversion per utterance), on
    AutoVC2(44, 256, 512, 22) and MetaPool2, fp32 and fp16x2: one B = 1 call per utterance (the default "batch"
    statistics, which at B = 1 are the utterance's own) against "utterance" batches of 64 and of 512.  The B = 1 outputs
    are compared with the batched ones utterance by utterance (max rel-L2 of mel_postnet).
(b) one ragged batch of 512 utterances (lengths 22 .. 176, multiples of 22, seeded) through AutoVC2 in "utterance" mode
    and through AutoVC: the difference is what the AdaIN variant adds (three pre-extract and three combine convolutions,
    six statistics, three AdaIN passes); ops.PROFILER in a separate pass gives the statistics and AdaIN kernels' share.
(c) avc_segment_stats alone on [512][128][80] fp32 (21 MB): time per call and bytes read per second, rotating over 8
    inputs (168 MB, more than the 126 MB L2) so that every call reads from HBM; 320 calls captured in one CUDA graph.

Each timed window follows an untimed warm-up of the same shapes and lies between CUDA events after a device synchronise;
the card's name and power limit are read (nvidia-smi --query-gpu, read-only) in the same run.

    python scripts/adain_batch_timing.py --out profiles/r03_adain_batch_timing.json
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


def timed(fn, reps=3):
    fn()                                    # warm-up: same shapes, same schedule
    torch.cuda.synchronize()
    best, out = None, None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return best, out


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm())


def make(cls_name, args, precision, dev):
    from oracle import templates
    from oracle.seeded import seeded_state_dict
    from autoformer_b200.factory.AutoVC import AutoVC
    from autoformer_b200.factory.AutoVC2 import AutoVC2
    from autoformer_b200.factory.MetaPool2 import MetaPool2
    cls, tpl = {"AutoVC2": (AutoVC2, templates.autovc2_template(*args)),
                "MetaPool2": (MetaPool2, templates.meta2_template("pool", *args)),
                "AutoVC": (AutoVC, templates.autovc_template(*args))}[cls_name]
    m = cls(*args)
    m.load_state_dict(seeded_state_dict(tpl, 0))
    m = m.to(dev).eval()
    m.precision = precision
    return m


def evaluator_style(cls_name, precision, x, c_org, c_trg, dev):
    """(a): 512 B = 1 calls against "utterance" batches of 64 and 512."""
    m = make(cls_name, (44, 256, 512, 22), precision, dev)
    N = x.shape[0]

    def one_by_one():
        m.adain_stats = "batch"
        return [m(x[i:i + 1], c_org[i:i + 1], c_trg[i:i + 1])[1] for i in range(N)]

    def batched(size):
        def run():
            m.adain_stats = "utterance"
            return [m(x[i:i + size], c_org[i:i + size], c_trg[i:i + size])[1] for i in range(0, N, size)]
        return run

    ms1, outs1 = timed(one_by_one, reps=1)
    rec = dict(model=cls_name, precision=precision, utterances=N, frames=x.shape[1], b1_calls_ms=round(ms1, 2))
    for size in (64, 512):
        ms, outs = timed(batched(size))
        post = torch.cat(outs)
        rec[f"utterance_b{size}_ms"] = round(ms, 2)
        rec[f"speedup_b{size}"] = round(ms1 / ms, 1)
        rec[f"max_rel_l2_b1_vs_b{size}"] = max(rel_l2(post[i], outs1[i][0]) for i in range(N))
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("adain_batch_timing.py needs a CUDA device")
    from autoformer_b200 import _lib, ops
    dev = torch.device("cuda:0")
    res = dict(device=device_info(), torch=torch.__version__, when=time.strftime("%Y-%m-%d %H:%M"),
               note="(a) times one self-styled conversion per utterance; the Evaluator's isAdain recipe adds a "
                    "features-only call per utterance before it")

    g = torch.Generator(device=dev).manual_seed(1)
    N, T = 512, 176
    x = torch.rand(N, T, 80, generator=g, device=dev) * 6 - 5
    c = torch.nn.functional.normalize(torch.randn(2, N, 256, generator=g, device=dev), dim=-1)
    c_org, c_trg = c[0].contiguous(), c[1].contiguous()
    res["a_evaluator_512x176"] = []
    for cls_name in ("AutoVC2", "MetaPool2"):
        for precision in ("fp32", "fp16x2"):
            rec = evaluator_style(cls_name, precision, x, c_org, c_trg, dev)
            res["a_evaluator_512x176"].append(rec)
            print(json.dumps(rec), flush=True)

    rng = random.Random(5)
    lengths = [22 * rng.randint(1, 8) for _ in range(N)]
    res["b_ragged_512x176"] = []
    for precision in ("fp32", "fp16x2"):
        vc2 = make("AutoVC2", (44, 256, 512, 22), precision, dev)
        vc2.adain_stats = "utterance"
        vc = make("AutoVC", (44, 256, 512, 22), precision, dev)
        ms2, _ = timed(lambda: vc2(x, c_org, c_trg, lengths=lengths))
        ms1, _ = timed(lambda: vc(x, c_org, c_trg, lengths=lengths))
        ops.PROFILER.reset()
        ops.PROFILER.enabled = True
        vc2(x, c_org, c_trg, lengths=lengths)
        torch.cuda.synchronize()
        ops.PROFILER.enabled = False
        fam = ops.PROFILER.summary()
        ops.PROFILER.reset()
        rec = dict(precision=precision, utterances=N, T=T, frames=sum(lengths), autovc2_utterance_ms=round(ms2, 3),
                   autovc_ms=round(ms1, 3), adain_variant_extra_ms=round(ms2 - ms1, 3),
                   profiled_segment_stats_ms=round(fam["segment_stats"]["ms"], 3),
                   profiled_segment_stats_calls=fam["segment_stats"]["calls"],
                   profiled_adain_segmented_ms=round(fam["adain"]["ms"], 3),
                   profiled_adain_segmented_calls=fam["adain"]["calls"])
        res["b_ragged_512x176"].append(rec)
        print(json.dumps(rec), flush=True)

    K = 8
    xs = [torch.randn(512, 128, 80, generator=g, device=dev) for _ in range(K)]
    out = torch.empty(512, 2, device=dev)
    lib = _lib.load()
    scratch = torch.empty(2 * 512 * -(-128 * 80 // _lib.SEGMENT_CHUNK), dtype=torch.float64, device=dev)
    launch = lambda t: _lib.check(lib.avc_segment_stats(t.data_ptr(), 512, 128, 80, None, out.data_ptr(),
                                                        scratch.data_ptr(), ops._stream()), "avc_segment_stats")
    reps = 40 * K
    launch(xs[0])                            # warm-up outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()           # replayed, so that host launch overhead is not what is timed
    with torch.cuda.graph(graph):
        for i in range(reps):
            launch(xs[i % K])
    ms, _ = timed(graph.replay)
    nbytes = 4.0 * 512 * 128 * 80
    res["c_segment_stats_512x128x80"] = dict(us_per_call=round(1e3 * ms / reps, 2),
                                             bytes_per_call=int(nbytes), GB_per_s=round(nbytes * reps / ms / 1e6, 1),
                                             inputs_rotated=K, note="two launches per call, 320 calls replayed as one "
                                                                    "CUDA graph; input beyond L2")
    print(json.dumps(res["c_segment_stats_512x128x80"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
