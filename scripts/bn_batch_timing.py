"""What batch-statistics BatchNorm (``bn_stats = "batch"``) costs: step time of each model in both modes, and the two
new kernels alone on the shape of one 512-channel conv layer at the headline size.

Running and batch modes alternate in the same process (one warm-up round each first); every time is from CUDA events
around `--iters` forwards, median of `--rounds` rounds.  Kernel bandwidth is computed from bytes implied by the shapes:
avc_bn_batch_stats reads v once; avc_bn_apply reads v and writes the operand-format output.

    python scripts/bn_batch_timing.py [--iters 10] [--rounds 5] [--json out.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.filterwarnings("ignore")

from oracle import templates                                     # noqa: E402
from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker   # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception:                                            # no nvidia-smi: the name alone
        return torch.cuda.get_device_name(), "unknown"


def timed(fn, iters):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / iters


def model_case(name, B, T, precision):
    from autoformer_b200.factory.AutoVC import AutoVC
    from autoformer_b200.factory.MetaConv import MetaConv
    from autoformer_b200.factory.MetaPool import MetaPool
    cls, args, tpl = {"AutoVC(32,256,512,32)": (AutoVC, (32, 256, 512, 32), templates.autovc_template),
                      "AutoVC(44,256,512,22)": (AutoVC, (44, 256, 512, 22), templates.autovc_template),
                      "MetaPool": (MetaPool, (44, 256, 512, 22), lambda *a: templates.meta_template("pool", *a)),
                      "MetaConv": (MetaConv, (44, 256, 512, 22), lambda *a: templates.meta_template("conv", *a))}[name]
    m = cls(*args)
    m.load_state_dict(seeded_state_dict(tpl(*args), 0))
    m = m.cuda().eval()
    m.precision = precision
    x, co, ct = synthetic_mel(B, T, 1).cuda(), synthetic_speaker(B, 1, "org").cuda(), synthetic_speaker(B, 1, "trg").cuda()
    return m, (x, co, ct)


def measure_models(iters, rounds):
    rows = []
    for name, B, T, prec in (("AutoVC(32,256,512,32)", 512, 128, "fp16x2"), ("AutoVC(32,256,512,32)", 512, 128, "fp32"),
                             ("MetaPool", 512, 176, "fp16x2"), ("AutoVC(44,256,512,22)", 2, 176, "fp32"),
                             ("MetaConv", 2, 176, "fp32")):
        m, inp = model_case(name, B, T, prec)
        times = {"running": [], "batch": []}
        for r in range(rounds + 1):                              # round 0: warm-up (plan packing, first launches)
            for mode in ("running", "batch"):
                m.bn_stats = mode
                t = timed(lambda: m(*inp), iters)
                if r:
                    times[mode].append(t)
        run, bat = statistics.median(times["running"]), statistics.median(times["batch"])
        rows.append(dict(model=name, B=B, T=T, precision=prec, running_ms=round(run, 3), batch_ms=round(bat, 3),
                         extra_ms=round(bat - run, 3), extra_pct=round(100 * (bat - run) / run, 1)))
        print(json.dumps(rows[-1]), flush=True)
        del m
        torch.cuda.empty_cache()
    return rows


def measure_kernels(iters, rounds):
    from autoformer_b200 import ops
    out = []
    for rows_, C, fmt in ((512 * 128, 512, "fp16x2"), (512 * 128, 512, "fp32"), (512 * 128, 80, "fp16x2"),
                          (512 * 176, 176, "fp16x2"), (2 * 176, 512, "fp32")):
        v = torch.randn(rows_, C, device="cuda")
        gamma, beta = torch.ones(C, device="cuda"), torch.zeros(C, device="cuda")
        rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
        nbt = torch.zeros((), dtype=torch.int64, device="cuda")
        ss = ops.bn_batch_stats(v, gamma, beta, 1e-5, 0.1, rm, rv, nbt)
        o = ops.alloc_act(1, rows_, C, fmt, "cuda")
        stats_ms, apply_ms = [], []
        for r in range(rounds + 1):
            a = timed(lambda: ops.bn_batch_stats(v, gamma, beta, 1e-5, 0.1, rm, rv, nbt, scale_shift=ss), iters)
            b = timed(lambda: ops.bn_apply(v, ss, 1, rows_, "relu", out=o, out_fmt=fmt), iters)
            if r:
                stats_ms.append(a)
                apply_ms.append(b)
        sm, am = statistics.median(stats_ms), statistics.median(apply_ms)
        sb = 4.0 * rows_ * C
        ab = sb + o.numel() * o.element_size()
        out.append(dict(rows=rows_, C=C, out_format=fmt, stats_us=round(1e3 * sm, 2), stats_GBps=round(sb / sm / 1e6, 1),
                        apply_us=round(1e3 * am, 2), apply_GBps=round(ab / am / 1e6, 1)))
        print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    name, power = card()
    print(json.dumps(dict(card=name, power_limit=power)), flush=True)
    res = dict(card=name, power_limit=power, kernels=measure_kernels(a.iters * 10, a.rounds),
               models=measure_models(a.iters, a.rounds))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
