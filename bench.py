#!/usr/bin/env python
"""Benchmark of the batched voice-conversion forward path (BASELINE.json metric: converted mel-frames/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a kernels
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU PyTorch classes (baseline/_ref)

Headline workload (BASELINE.json configs[1]): AutoVC(32,256,512,32) conversion forward, batch 512 utterances x 128
frames x 80 mel bins per GPU (weak scaling: every rank converts its own batch), random-init weights, synthetic inputs.
One "step" = one forward over the batch.  `value` times K steps with inputs resident in HBM; `e2e` times the same K
steps through the public host-to-host API starting from pinned HOST buffers (H2D of x/c_org/c_trg and D2H of the three
outputs inside the timed region, which ends only after the last download has landed).

The same JSON line carries `configs`: sub-records for the other BASELINE configs, each measured in this very run with
CUDA events and checked on sampled utterances against the UNMODIFIED reference classes on the CPU (baseline/_ref):
  cfg3_metapool / cfg3_metaconv  MetaPool / MetaConv (44,256,512,22), 512 x 176 frames                 (N = 1 only)
  cfg4_b32 / cfg4_b1             LstmDV x2 -> AutoVC (pad 1000 -> 1024, trim) -> MelGAN, 1000-frame utt. (N = 1 only)
  cfg5_sweep                     65,536 utterances x 128..1024 frames, bucketed by exact length, LPT-sharded over the
                                 N ranks (STRONG scaling: the same utterances at every N)
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODEL_ARGS = (32, 256, 512, 32)            # AutoVC "original" hyper-parameters (SURVEY.md 8, config A)
META_ARGS = (44, 256, 512, 22)             # the only shape the reference's Meta models accept (SURVEY.md 0.2)
# SURVEY.md 8(d) algorithmic work
FLOP_PER_FRAME = 56_770_560                # AutoVC-A: conv 23,511,040 + in-proj/Linear 14,352,384 + recurrent 18,907,136
FLOP_LSTMDV_FRAME = 24_084_480
FLOP_MELGAN_FRAME = 90_341_376
FLOP_META_UTT = {"pool": 53.441e9, "conv": 55.727e9}
METRIC = "converted mel-frames/sec"
UNIT = "frames/s"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default="fp16x2", choices=["fp32", "fp16x2", "tf32", "bf16"],
                    help="fp16x2 (default): fp16 activations x two-term fp16 weights, 2 MMA passes, ~3e-4 from the "
                         "reference (the fastest mode inside the 1e-3 tolerance); fp32: split-bf16, 3 passes, ~3e-5; "
                         "tf32: ~1e-3; bf16: ~8e-3")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--frames", type=int, default=128)
    ap.add_argument("--lstm", default="persistent", choices=["persistent", "per-step"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-batch", type=int, default=32, help="utterances in the bounded CPU-baseline sample")
    ap.add_argument("--configs", default="all",
                    help="sub-records to measure after the headline: all | none | comma list of cfg3,cfg4,cfg5")
    ap.add_argument("--utterances", type=int, default=65536, help="utterances of the cfg5 sweep (whole job)")
    ap.add_argument("--workload", default="batch", choices=["batch", "sweep"],
                    help="batch: the default line; sweep: print the cfg5 sweep alone as the JSON line")
    ap.add_argument("--keep-digest", action="store_true",
                    help="keep the per-forward weight digest of the plan cache inside the timed region "
                         "(default: weights frozen after warm-up, as a serving loop would)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's outputs of the last timed headline step (mel, mel_postnet, codes) as "
                         "DIR/<name>.npy in float32, at most 64 MB in all (beyond that a fixed seeded sample of the "
                         "utterances); the inputs depend on the arguments only, so two builds compare output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "native" or args.workload != "batch"):
        ap.error("--dump-outputs writes the headline batch of the native arm (--impl native --workload batch)")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tflops_burst=p["bf16_tflops"], tflops_sustained=p["bf16_tflops_sustained"],
                    source="MEASURED_PEAKS.json")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def workload_config(args, world):
    """The `config` object: identical in both arms (--impl native / reference) for the same command line."""
    B, T = args.batch, args.frames
    act_gb = B * T * (336 + 512 * 10 + 4096 * 2 + 2048 + 1024 * 2 + 320 + 80 * 3) * 4 / 1e9
    return {"workload": "AutoVC(32,256,512,32) conversion forward (encoder+decoder+postnet), "
                        f"{B} utterances x {T} frames x 80 mel per GPU (BASELINE.json configs[1])",
            "batch_per_gpu": B, "frames": T,
            "parallelism": f"utterance-sharded x{world}, no data-path collective",
            "l2": f"no explicit flush: each step streams ~{act_gb:.1f} GB of activations, far beyond the 126 MB L2"}


class stdout_to_stderr:
    """stdout carries exactly ONE JSON line.  NCCL prints its version banner to the process's file descriptor 1 when the
    first communicator is created (NCCL_DEBUG=VERSION from the environment or from /etc/nccl.conf), so the descriptor
    itself is pointed at stderr while the process group comes up."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def init_nccl(dev):
    import torch
    import torch.distributed as dist
    with stdout_to_stderr():
        dist.init_process_group("nccl", device_id=dev)
        t = torch.zeros(1, device=dev)
        dist.all_reduce(t)                     # forces communicator creation (and the banner) inside the redirect
        torch.cuda.synchronize()


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5),
                          ("sw_power_cap", 6)):
            if any(s[col].lower().startswith("active") for s in self.samples):
                reasons.append(name)
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=float(self.samples[0][1]), samples=len(sm),
                    power_w_max=max(float(s[2]) for s in self.samples), reasons=reasons)


# --------------------------------------------------------------------------------------------------------------
# The reference on the CPU: the UNMODIFIED classes pip-installed into baseline/_ref (baseline/install_reference.py)
# --------------------------------------------------------------------------------------------------------------
def cpu_model_name():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


class Reference:
    """The reference's classes from baseline/_ref (kind "reference"); when that directory is missing, the oracle port of
    the same arithmetic (kind "port").  CPU, eval(), no_grad, fp32.  Never on the product path."""

    def __init__(self):
        import types
        import warnings
        warnings.filterwarnings("ignore", category=FutureWarning)
        self.kind = "reference" if os.path.isfile(os.path.join(REF_DIR, "factory", "AutoVC.py")) else "port"
        if self.kind == "reference":
            if "librosa" not in sys.modules:       # melgan/modules.py:4 imports it; only Audio2Mel would call it
                lib, filt = types.ModuleType("librosa"), types.ModuleType("librosa.filters")
                filt.mel = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("librosa is stubbed"))
                lib.filters = filt
                sys.modules["librosa"], sys.modules["librosa.filters"] = lib, filt
            if REF_DIR not in sys.path:
                sys.path.insert(0, REF_DIR)

    def describe(self):
        import torch
        return (f"unmodified reference classes (baseline/_ref, torch {torch.__version__} CPU fp32, eval, no_grad)"
                if self.kind == "reference" else
                f"oracle port of the reference arithmetic (torch {torch.__version__} CPU fp32): baseline/_ref is absent")

    def _module(self, mod, cls, args, sd):
        import importlib
        m = getattr(importlib.import_module(mod), cls)(*args)
        m.load_state_dict(sd)
        return m.eval()

    def autovc(self, sd, args=MODEL_ARGS):
        import torch
        if self.kind == "reference":
            m = self._module("factory.AutoVC", "AutoVC", args, sd)

            def run(x, c_org, c_trg):
                with torch.no_grad():
                    return m(x, c_org, c_trg)
            return run
        from oracle.autovc import autovc_forward
        return lambda x, c_org, c_trg: autovc_forward(sd, x, c_org, c_trg, args[0], args[3])

    def meta(self, kind, sd):
        import torch
        if self.kind == "reference":
            name = "MetaPool" if kind == "pool" else "MetaConv"
            m = self._module(f"factory.{name}", name, META_ARGS, sd)

            def run(x, c_org, c_trg):
                with torch.no_grad():
                    return m(x, c_org, c_trg)
            return run
        from oracle.meta import meta_forward
        return lambda x, c_org, c_trg: meta_forward(sd, x, c_org, c_trg, META_ARGS[0], META_ARGS[3], kind)

    def lstmdv(self, sd):
        import torch
        if self.kind == "reference":
            m = self._module("factory.LstmDV", "LstmDV", (), sd)

            def run(x):
                with torch.no_grad():
                    return m(x)
            return run
        from oracle.lstmdv import lstmdv_forward
        return lambda x: lstmdv_forward(sd, x)

    def melgan(self, sd):
        import torch
        if self.kind == "reference":
            m = self._module("melgan.modules", "Generator", (80, 32, 3), sd)

            def run(mel):
                with torch.no_grad():
                    return m(mel)
            return run
        from oracle.melgan import melgan_forward
        return lambda mel: melgan_forward(sd, mel)


def rel_l2(a, b):
    import torch
    a, b = a.detach().to("cpu", torch.float64).reshape(-1), b.detach().to("cpu", torch.float64).reshape(-1)
    return float((a - b).norm() / b.norm())


def bench_state_dict(cls=None):
    """Weights of the headline model: the class's own default init (xavier convs, torch LSTM init) with non-trivial
    BatchNorm statistics so the folding is exercised.  `cls`: the model class to instantiate (default: the drop-in
    AutoVC; the reference arm passes the reference's class so that nothing of this repo is on its path)."""
    import torch
    if cls is None:
        from autoformer_b200.factory.AutoVC import AutoVC as cls
    torch.manual_seed(1234)
    model = cls(*MODEL_ARGS)
    with torch.no_grad():
        g = torch.Generator().manual_seed(7)
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.5)
                m.running_var.copy_(torch.rand(m.num_features, generator=g) * 1.5 + 0.5)
                m.weight.copy_(torch.rand(m.num_features, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.num_features, generator=g) * 0.2)
    return model, {k: v.clone() for k, v in model.state_dict().items()}


def bench_inputs(B, T, rank):
    import torch
    gen = torch.Generator().manual_seed(1234 + rank)
    x = torch.rand(B, T, 80, generator=gen) * 6 - 5
    spk = lambda: torch.nn.functional.normalize(torch.randn(B, 256, generator=gen), dim=-1)
    return x, spk(), spk()


DUMP_LIMIT = 64_000_000         # bytes --dump-outputs may write, .npy headers included


def dump_outputs(dirname, outs):
    """Write {name: CPU tensor with the utterances on dim 0} as dirname/<name>.npy in float32.  When the whole batch
    exceeds DUMP_LIMIT, every array keeps the same utterances: a seeded sample that depends on the batch size only,
    in batch order."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    B = next(iter(outs.values())).shape[0]
    per_utt = sum(t[0].numel() * 4 for t in outs.values())
    keep = min(B, (DUMP_LIMIT - 4096 * len(outs)) // per_utt)        # 4 KB for every .npy header
    rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    for name, t in outs.items():
        np.save(os.path.join(dirname, name + ".npy"), t[rows].float().numpy())


def time_cpu(run, frames, min_seconds, max_seconds, min_runs=3):
    """Median wall time of `run()` after one warm-up: at least `min_runs` runs and `min_seconds`, at most `max_seconds`."""
    run()
    times = []
    t_start = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
        el = time.perf_counter() - t_start
        if (el >= min_seconds and len(times) >= min_runs) or el >= max_seconds:
            break
    times.sort()
    med = times[len(times) // 2]
    return frames / med, med, len(times)


def cpu_baseline(ref, state_dict, args):
    """The reference's CPU forward on the GPU box's host cores: a bounded sample of the headline workload (the first
    `--cpu-batch` utterances of rank 0's batch) on all threads, and the B = 2 configuration (BASELINE configs[0]) on all
    threads and on ONE thread (per-core figure, BASELINE.md 3)."""
    import torch
    cores = os.cpu_count() or 1
    sd = {k: v.detach().float().cpu() for k, v in state_dict.items()}
    fwd = ref.autovc(sd)
    x, c_org, c_trg = bench_inputs(args.batch, args.frames, 0)
    n = min(args.cpu_batch, args.batch)
    xs, cs, ct = x[:n].contiguous(), c_org[:n].contiguous(), c_trg[:n].contiguous()
    torch.set_num_threads(cores)
    v_all, med, runs = time_cpu(lambda: fwd(xs, cs, ct), n * args.frames, 8.0, 20.0)
    v_b2, med_b2, _ = time_cpu(lambda: fwd(xs[:2], cs[:2], ct[:2]), 2 * args.frames, 2.0, 6.0)
    torch.set_num_threads(1)
    v_1t, med_1t, _ = time_cpu(lambda: fwd(xs[:2], cs[:2], ct[:2]), 2 * args.frames, 2.0, 8.0)
    torch.set_num_threads(cores)
    return dict(value=v_all, unit=UNIT, cores=cores, kind=ref.kind, cpu_model=cpu_model_name(),
                sample=f"{ref.describe()}: AutoVC(32,256,512,32) forward on the first {n} of the {args.batch} utterances "
                       f"x {args.frames} frames of rank 0's batch, {cores} threads, median of {runs} runs "
                       f"({med * 1e3:.0f} ms each)",
                config1_b2=dict(value=v_b2, unit=UNIT, threads=cores, ms=med_b2 * 1e3,
                                workload="BASELINE configs[0]: batch 2 x 128 frames"),
                one_thread=dict(value=v_1t, unit=UNIT, threads=1, ms=med_1t * 1e3, workload="batch 2 x 128 frames"))


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the unmodified classes from baseline/_ref)
    on this arm's config, all host threads.  Each step is a bounded sample of the workload: the whole 512-utterance
    batch when K + W steps of it fit in ~2.5 minutes on this host, else the largest power-of-two slice that does."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    import torch
    ref = Reference()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if ref.kind == "reference":
        import importlib
        _, sd = bench_state_dict(importlib.import_module("factory.AutoVC").AutoVC)
    else:
        _, sd = bench_state_dict()
    fwd = ref.autovc(sd)
    x, c_org, c_trg = bench_inputs(args.batch, args.frames, 0)
    probe = min(16, args.batch)
    fwd(x[:probe], c_org[:probe], c_trg[:probe])
    t0 = time.perf_counter()
    fwd(x[:probe], c_org[:probe], c_trg[:probe])
    per_utt = (time.perf_counter() - t0) / probe
    B = args.batch
    budget = 150.0
    while B > probe and per_utt * B * (args.steps + args.warmup) > budget:
        B //= 2
    xs, cs, ct = x[:B].contiguous(), c_org[:B].contiguous(), c_trg[:B].contiguous()
    step = lambda: fwd(xs, cs, ct)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = B * args.frames * args.steps / dt
    sample = (f"{ref.describe()}: each step converts {B} of the {args.batch} utterances x {args.frames} frames of the "
              f"workload on {cores} threads ({cpu_model_name()})")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": ref.kind, "sample": sample,
                         "sample_batch": B, "cpu_model": cpu_model_name()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------------------
# helpers of the native arm
# --------------------------------------------------------------------------------------------------------------
class Ctx:
    """Device / process-group context of one rank."""

    def __init__(self):
        import torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback on the product path)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            init_nccl(self.dev)

    def sync_all(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms


def timed_steps(ctx, step_fn, steps, sampler=None, finish=None):
    """K steps bracketed by barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks.
    `finish()` (optional) runs after the last step and before the closing event: work that belongs to the timed region
    but completes on another stream (the e2e arm's last download)."""
    import torch
    from autoformer_b200 import _lib
    ctx.sync_all()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = _lib.launch_count()
    e0.record()
    for _ in range(steps):
        step_fn()
    if finish is not None:
        finish()
    e1.record()
    ctx.sync_all()
    if sampler:
        sampler.stop_flag.set()
    return ctx.max_over_ranks(e0.elapsed_time(e1)), _lib.launch_count() - n0


def family_summary(prof_steps, pk, passes):
    """Per kernel family (ops.PROFILER, CUDA events around every launch): ms, launches, algorithmic TFLOP/s or GB/s and
    the fractions of the measured peaks.  `issued_mma_frac_of_burst` multiplies by the MMA passes per algorithmic FLOP
    and divides by the BURST bf16 peak (sub-second regions run at full clock); ncu's own tensor-pipe counter for each
    kernel is in profiles/."""
    from autoformer_b200 import ops
    out = {}
    for name, d in ops.PROFILER.summary().items():
        ms = d["ms"] / prof_steps
        ent = dict(ms_per_step=ms, launches_per_step=d["launches"] // prof_steps)
        if d["flops"] > 0:
            tf = d["flops"] / prof_steps / (ms * 1e-3) / 1e12
            ent.update(tflops=tf, frac_of_bf16_burst=tf / pk["tflops_burst"],
                       frac_of_bf16_sustained=tf / pk["tflops_sustained"])
            if passes:
                ent["issued_mma_frac_of_burst"] = tf * passes / pk["tflops_burst"]
        if d["bytes"] > 0:
            gbs = d["bytes"] / prof_steps / (ms * 1e-3) / 1e9
            ent.update(gbs=gbs, frac_of_hbm=gbs / pk["hbm_gbs"])
        out[name] = ent
    return out


def profile_families(fn, steps, pk, passes):
    import torch
    from autoformer_b200 import ops
    ops.PROFILER.reset()
    ops.PROFILER.enabled = True
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    ops.PROFILER.enabled = False
    return family_summary(steps, pk, passes)


PASSES = {"fp32": 3, "fp16x2": 2, "tf32": 2, "bf16": 1, "fp16s": 3}      # bf16-MMA-equivalent passes per algorithmic FLOP


def dram_traffic(kernel, key):
    """DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum) of `kernel` in configuration `key`, read
    at run time from the committed summary of the `ncu --set full` capture (profiles/r02_dram_traffic.json, written by
    scripts/ncu_traffic.py from the .ncu-rep); None when no capture of this configuration is committed."""
    path = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    try:
        with open(path) as f:
            table = json.load(f)
    except (OSError, ValueError):
        return None, None
    ent = table.get(key, {}).get(kernel)
    if not ent:
        return None, None
    return ent["bytes_per_launch"], ent.get("source")


# --------------------------------------------------------------------------------------------------------------
# sub-records (BASELINE configs 3, 4, 5)
# --------------------------------------------------------------------------------------------------------------
def seeded(template_fn, seed, **kw):
    """Signal-preserving seeded weights shared with the parity tests (oracle/seeded.py: a 28 M-parameter state_dict is
    regenerated from its seed on both sides).  Weight generation only -- no oracle arithmetic."""
    from oracle.seeded import seeded_state_dict
    return seeded_state_dict(template_fn, seed, **kw)


def events_ms(fn, steps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def sub_cfg3(ctx, ref, kind, pk, precision="fp16x2", B=512, T=176):
    import torch
    from oracle import templates
    from autoformer_b200 import _lib
    from autoformer_b200.factory.MetaConv import MetaConv
    from autoformer_b200.factory.MetaPool import MetaPool
    cls = MetaPool if kind == "pool" else MetaConv
    sd = seeded(templates.meta_template(kind, *META_ARGS), 6 if kind == "pool" else 7)
    m = cls(*META_ARGS)
    m.load_state_dict(sd)
    m = m.to(ctx.dev).eval()
    m.precision = precision
    x, c_org, c_trg = bench_inputs(B, T, 100)
    xd, cod, ctd = x.to(ctx.dev), c_org.to(ctx.dev), c_trg.to(ctx.dev)
    out = m(xd, cod, ctd)
    m.freeze_weights()
    n0 = _lib.launch_count()
    ms = events_ms(lambda: m(xd, cod, ctd), steps=3, warmup=1)
    launches = (_lib.launch_count() - n0) // 4
    fam = profile_families(lambda: m(xd, cod, ctd), 1, pk, PASSES[precision])
    # parity on sampled utterances of the big batch against the reference on the CPU
    pick = [0, B // 2 + 61, B - 1]
    fwd = ref.meta(kind, sd)
    r_mel, r_post, r_codes = fwd(x[pick], c_org[pick], c_trg[pick])
    par = dict(mel=rel_l2(out[0][pick], r_mel), mel_postnet=rel_l2(out[1][pick], r_post),
               codes=rel_l2(out[2][pick], r_codes), utterances=pick, against=ref.kind)
    tf = FLOP_META_UTT[kind] * B / (ms * 1e-3) / 1e12
    del m
    torch.cuda.empty_cache()
    return dict(workload=f"{'MetaPool' if kind == 'pool' else 'MetaConv'}(44,256,512,22) forward, {B} x {T} frames "
                         "(BASELINE configs[2]; the reference's Meta models only accept T = 176)",
                precision=precision, ms=ms, frames_per_s=B * T / (ms * 1e-3), launches=launches, tflops=tf,
                frac_of_bf16_burst=tf / pk["tflops_burst"], frac_of_bf16_sustained=tf / pk["tflops_sustained"],
                rel_l2=par, families=fam)


def sub_cfg4(ctx, ref, pk, B, T=1000):
    import torch
    from oracle import templates
    from autoformer_b200 import _lib, pipeline
    from autoformer_b200.factory.AutoVC import AutoVC
    from autoformer_b200.factory.LstmDV import LstmDV
    from autoformer_b200.melgan.modules import Generator
    sd_dv = seeded(templates.lstmdv_template(), 3, lstm_gain=1.5)
    sd_vc = seeded(templates.autovc_template(*MODEL_ARGS), 0)
    sd_g = seeded(templates.melgan_template(), 4)
    dv, vc, gen = LstmDV(), AutoVC(*MODEL_ARGS), Generator(80, 32, 3)
    dv.load_state_dict(sd_dv), vc.load_state_dict(sd_vc), gen.load_state_dict(sd_g)
    dv, vc, gen = dv.to(ctx.dev).eval(), vc.to(ctx.dev).eval(), gen.to(ctx.dev).eval()
    dv.precision = vc.precision = "fp16x2"
    gen.precision = MELGAN_PRECISION
    src, _, _ = bench_inputs(B, T, 200)
    trg, _, _ = bench_inputs(B, T, 201)
    sd_, td_ = src.to(ctx.dev), trg.to(ctx.dev)
    mel, wav, eo, et = pipeline.convert_and_vocode(dv, vc, gen, sd_, td_)
    for m in (dv, vc, gen):
        m.freeze_weights()
    n0 = _lib.launch_count()
    ms = events_ms(lambda: pipeline.convert_and_vocode(dv, vc, gen, sd_, td_), steps=3, warmup=1)
    launches = (_lib.launch_count() - n0) // 4
    both = torch.cat((sd_, td_), 0)
    ms_dv = events_ms(lambda: dv(both), steps=2, warmup=1)
    ms_vc = events_ms(lambda: pipeline.convert(vc, sd_, eo, et), steps=2, warmup=1)
    melT = mel.transpose(2, 1).contiguous()
    ms_gen = events_ms(lambda: gen(melT), steps=2, warmup=1)
    fam_gen = profile_families(lambda: gen(melT), 1, pk, None)      # (mixed two- and three-product layers)
    fam_dv = profile_families(lambda: dv(both), 1, pk, PASSES["fp16x2"])
    # parity of one utterance end to end against the reference pipeline on the CPU (same recipe: embed both, zero-pad
    # to a multiple of freq, convert, trim, vocode), and of the vocoder alone on the reference's own converted mel
    i = B - 1
    r_dv, r_vc, r_gen = ref.lstmdv(sd_dv), ref.autovc(sd_vc), ref.melgan(sd_g)
    r_eo, r_et = r_dv(src[i:i + 1]), r_dv(trg[i:i + 1])
    pad = (-T) % MODEL_ARGS[3]
    r_mel = r_vc(torch.nn.functional.pad(src[i:i + 1], (0, 0, 0, pad)), r_eo, r_et)[1].squeeze(1)[:, :T]
    r_wav = r_gen(r_mel.transpose(1, 2)).squeeze(1)
    wav_alone = gen(r_mel.transpose(1, 2).contiguous().to(ctx.dev)).squeeze(1)
    par = dict(emb_org=rel_l2(eo[i:i + 1], r_eo), emb_trg=rel_l2(et[i:i + 1], r_et), mel=rel_l2(mel[i:i + 1], r_mel),
               waveform_end_to_end=rel_l2(wav[i:i + 1], r_wav), waveform_vocoder_alone=rel_l2(wav_alone, r_wav),
               utterance=i, against=ref.kind)
    tf_gen = FLOP_MELGAN_FRAME * B * T / (ms_gen * 1e-3) / 1e12
    tf_dv = FLOP_LSTMDV_FRAME * 2 * B * T / (ms_dv * 1e-3) / 1e12
    tf_vc = FLOP_PER_FRAME * B * (T + pad) / (ms_vc * 1e-3) / 1e12
    total_flop = FLOP_MELGAN_FRAME * B * T + FLOP_LSTMDV_FRAME * 2 * B * T + FLOP_PER_FRAME * B * (T + pad)
    tf = total_flop / (ms * 1e-3) / 1e12
    del dv, vc, gen
    torch.cuda.empty_cache()
    frac = lambda v: dict(tflops=v, frac_of_bf16_burst=v / pk["tflops_burst"], frac_of_bf16_sustained=v / pk["tflops_sustained"])
    return dict(workload=f"LstmDV(src) + LstmDV(trg) -> AutoVC(32,256,512,32) (pad {T} -> {T + pad}, trim) -> MelGAN, "
                         f"{B} utterances x {T} frames -> {256 * T} samples each (BASELINE configs[3])",
                precision=f"embedder / AutoVC fp16x2, MelGAN {MELGAN_PRECISION}", ms=ms, frames_per_s=B * T / (ms * 1e-3),
                launches=launches, **frac(tf),
                stages=dict(lstmdv_2B=dict(ms=ms_dv, **frac(tf_dv)), autovc=dict(ms=ms_vc, **frac(tf_vc)),
                            melgan=dict(ms=ms_gen, **frac(tf_gen))),
                rel_l2=par, families=dict(melgan=fam_gen, lstmdv=fam_dv))


# "fp16s" (round 2): residual stream / ConvTranspose operands / ResnetBlock intermediate as two fp16 terms, the k3 operand
# as one; waveform rel-L2 <= 5.3e-4 over six weight seeds (scripts/melgan_precision_study.py); "fp32" = split bf16
MELGAN_PRECISION = os.environ.get("AVC_BENCH_MELGAN_PRECISION", "fp16s")


def sub_cfg5(ctx, ref, pk, args, precision):
    """BASELINE configs[4]: `--utterances` utterances with T uniform in {128,160,...,1024}, bucketed by exact T, batches
    of <= 512, LPT-assigned to the ranks by the measured cost model; no data-path collective; strong scaling."""
    import random
    import torch
    from autoformer_b200 import _lib, pipeline, sharding
    from autoformer_b200.factory.AutoVC import AutoVC
    model, sd = bench_state_dict()
    model = model.to(ctx.dev).eval()
    model.precision = precision
    model.persistent_lstm = args.lstm != "per-step"
    rng = random.Random(1234)
    lengths = [rng.choice(range(128, 1025, 32)) for _ in range(args.utterances)]
    plan = sharding.plan(lengths, ctx.world, args.batch, cost=sharding.autovc_cost_for(precision))
    mine = plan[ctx.rank]
    pool = {}                 # the same synthetic pool on every rank: the job's checksum is comparable across N

    def inputs(T, n):
        if T not in pool:      # synthetic data: one resident batch per length, reused for every batch of that length
            g = torch.Generator(device=ctx.dev).manual_seed(4321 + T)
            x = torch.rand(args.batch, T, 80, generator=g, device=ctx.dev) * 6 - 5
            c = torch.nn.functional.normalize(torch.randn(2, args.batch, 256, generator=g, device=ctx.dev), dim=-1)
            pool[T] = (x, c[0].contiguous(), c[1].contiguous())
        x, co, ct = pool[T]
        return x[:n], co[:n], ct[:n]

    def one_pass():
        # pipeline.convert_batches: full batches one after the other, the under-filled last batch of every length bucket
        # two at a time on two streams (AVC_BENCH_PAIR=0: everything one after the other, for A/B timing)
        batches = [inputs(T, len(ids)) for T, ids in mine]
        sums = pipeline.convert_batches(model, batches, reduce=lambda out: out[1].double().sum(),
                                        pair_below=pipeline.PAIR_BELOW if os.environ.get("AVC_BENCH_PAIR", "1") != "0" else 0)
        return torch.stack(sums).sum() if sums else torch.zeros((), device=ctx.dev, dtype=torch.float64)

    for T, ids in mine:                                  # allocate every resident input before timing
        inputs(T, len(ids))
    # warm-up: one untimed pass over this rank's batches, through the same schedule as the timed one (weights packed for
    # every gate-group size, kernels loaded, and the caching allocator has seen every buffer size on every stream -- a
    # first-time cudaMalloc inside the timed pass costs milliseconds and synchronises; with N ranks each rank meets the
    # same ~29 lengths in 1/N of the work, which showed up as a 15 % strong-scaling loss at N = 2 that had nothing to do
    # with the GPUs)
    model(*inputs(*[(T, len(ids)) for T, ids in mine][0])) if mine else None
    model.freeze_weights()
    one_pass()
    model.freeze_weights()
    ctx.sync_all()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    chk = one_pass()
    e1.record()
    ctx.sync_all()
    ms = e0.elapsed_time(e1)
    frames = float(sum(t * len(i) for t, i in mine))
    recs = sharding.gather_records([frames, ms, float(chk), float(_lib.launch_count() - n0)], device=ctx.dev)
    # parity of two sampled utterances (shortest and longest bucket of this rank) against the reference on the CPU
    par = None
    if ctx.rank == 0 and mine:
        fwd = ref.autovc({k: v.cpu() for k, v in sd.items()})
        par = dict(against=ref.kind)
        for T in sorted({t for t, _ in mine})[::max(1, len({t for t, _ in mine}) - 1)][:2]:
            x, co, ct = inputs(T, 3)
            got = model(x, co, ct)[1][2:3]
            want = fwd(x[2:3].cpu(), co[2:3].cpu(), ct[2:3].cpu())[1]
            par[f"mel_postnet_T{T}"] = rel_l2(got, want)
    del model
    pool.clear()
    torch.cuda.empty_cache()
    if ctx.rank != 0:
        return None
    total = float(recs[:, 0].sum())
    ms_max = float(recs[:, 1].max())
    tf = total * FLOP_PER_FRAME / (ms_max * 1e-3) / 1e12 / ctx.world
    return dict(workload=f"AutoVC(32,256,512,32) conversion of {args.utterances} utterances x 128..1024 frames "
                         f"(BASELINE configs[4]), bucketed by exact length, batches <= {args.batch}, LPT-sharded over "
                         f"{ctx.world} rank(s) by a measured per-batch cost model; under-filled batches (<= 256 utterances) two at a "
                         f"time on two streams (pipeline.convert_batches); strong scaling",
                precision=precision, scaling="strong", n_gpus=ctx.world, utterances=args.utterances, frames_total=total,
                ms=ms_max, frames_per_s=total / (ms_max * 1e-3), tflops_per_gpu=tf,
                frac_of_bf16_burst=tf / pk["tflops_burst"], frac_of_bf16_sustained=tf / pk["tflops_sustained"],
                batches=sum(len(r) for r in plan), launches=int(recs[:, 3].sum()),
                rank_ms=[round(float(v), 2) for v in recs[:, 1].tolist()],
                rank_spread=float(recs[:, 1].max() / recs[:, 1].mean()), rel_l2=par,
                checksum=float(recs[:, 2].sum()))


# --------------------------------------------------------------------------------------------------------------
def run_native(args):
    import torch
    import torch.distributed as dist
    from autoformer_b200 import _lib
    from autoformer_b200.layers import lstm_fused_default
    from autoformer_b200.pipeline import StreamingConverter

    ctx = Ctx()
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    _lib.load()
    pk = peaks()
    B, T = args.batch, args.frames
    model, state_dict = bench_state_dict()
    model = model.to(dev).eval()
    model.precision = args.precision
    model.persistent_lstm = args.lstm == "persistent"

    x_c, co_c, ct_c = bench_inputs(B, T, rank)
    x_h, c_org_h, c_trg_h = x_c.pin_memory(), co_c.pin_memory(), ct_c.pin_memory()
    x_d, c_org_d, c_trg_d = x_h.to(dev), c_org_h.to(dev), c_trg_h.to(dev)
    out_h = [None, None, None]
    out_d = [None, None, None]

    def device_step():
        out_d[:] = model(x_d, c_org_d, c_trg_d)

    streamer = StreamingConverter(model, dev)      # public host-to-host API: copies overlap neighbouring batches

    def e2e_step():
        # every step uploads its inputs from pinned host memory and downloads all three outputs to pinned host memory
        res = streamer.submit(x_h, c_org_h, c_trg_h)
        if res is not None:
            out_h[:] = res

    def e2e_finish():
        # the timed region ends only when the LAST step's outputs are in host memory: wait for its download, then make
        # the closing event (recorded on the compute stream) follow the download stream
        res = streamer.flush()
        if res is not None:
            out_h[:] = res
        torch.cuda.current_stream(dev).wait_stream(streamer.d2h)

    for _ in range(max(args.warmup, 3)):
        device_step()
    if not args.keep_digest:
        model.freeze_weights()                     # serving loop: weights do not change between steps
    sampler = ClockSampler(ctx.local_rank) if rank == 0 else None
    ms_total, launches = timed_steps(ctx, device_step, args.steps, sampler)
    # copied before the e2e and profiling passes run the model again; written to disk after the last measurement
    dumped = dict(zip(("mel", "mel_postnet", "codes"), (t.cpu() for t in out_d))) if args.dump_outputs and rank == 0 else None
    frames_per_step = B * T * world
    value = frames_per_step * args.steps / (ms_total * 1e-3)

    for _ in range(3):
        e2e_step()
    streamer.flush()
    # the same nvidia-smi sampling runs beside the e2e region: every sample forks this process, which costs the launching
    # thread time -- with it on one region only, e2e read ~1 % FASTER than the device-resident number
    sampler_e2e = ClockSampler(ctx.local_rank) if rank == 0 else None
    ms_e2e, _ = timed_steps(ctx, e2e_step, args.steps, sampler_e2e, finish=e2e_finish)
    e2e_value = frames_per_step * args.steps / (ms_e2e * 1e-3)
    h2d = (x_h.numel() + c_org_h.numel() + c_trg_h.numel()) * 4
    d2h = sum(h.numel() * 4 for h in out_h)

    # per-kernel-family device times (CUDA events on the launching stream) for the roofline entry
    passes = PASSES[args.precision]
    kernels = profile_families(device_step, min(args.steps, 3), pk, passes)
    tensor_fams = {k: v for k, v in kernels.items() if "tflops" in v and k != "bilstm_small"}
    dom = max(tensor_fams, key=lambda k: tensor_fams[k]["ms_per_step"])
    dom_e = tensor_fams[dom]
    fused = lstm_fused_default()
    kernel_name = {"lstm_step": "lstm_fused_kernel" if fused else "lstm_step_kernel", "conv": "conv_gemm_kernel",
                   "inproj": "conv_gemm_kernel", "linear": "conv_gemm_kernel",
                   # weight-stationary LSTM kernels: the recurrence at small batches (ops.lstm_seq_ws / lstm_stack_ws)
                   "lstm_ws": "lstm_ws_kernel", "lstm_stack": "lstm_stack_kernel"}[dom]
    # the timed region is sub-second and runs at the full SM clock (see `clocks`): the burst bf16 figure is the peak a
    # kernel timed like this can reach; the sustained (power-capped, seconds-long) figure is kept beside it
    short = ms_total < 1000.0
    peak = pk["tflops_burst"] if short else pk["tflops_sustained"]
    traffic, traffic_src = dram_traffic(kernel_name, f"cfg2_{args.precision}_B{B}_T{T}_{args.lstm}")
    total_ms = sum(v["ms_per_step"] for v in kernels.values())
    roofline = {
        "kernel": f"{kernel_name} ({dom})", "bound": "tensor", "achieved": dom_e["tflops"], "peak": peak,
        "unit": "TFLOP/s", "frac": dom_e["tflops"] / peak, "traffic": traffic,
        "traffic_unit": "bytes per launch (mean over the launches of one step), ncu dram__bytes_read.sum + dram__bytes_write.sum",
        "traffic_source": traffic_src,
        "peak_source": pk["source"] + (" bf16_tflops (burst: timed region < 1 s at full clock)" if short
                                       else " bf16_tflops_sustained"),
        "frac_vs_sustained": dom_e["tflops"] / pk["tflops_sustained"],
        "share_of_step": dom_e["ms_per_step"] / total_ms,
        "avg_launch_us": dom_e["ms_per_step"] * 1e3 / max(1, dom_e["launches_per_step"]),
        "algorithmic_flops_per_launch": dom_e["tflops"] * 1e12 * dom_e["ms_per_step"] * 1e-3 / max(1, dom_e["launches_per_step"]),
        "mma_passes_per_flop": passes,
        "issued_mma_frac_of_peak": dom_e["tflops"] * passes / peak,
        "whole_step": {"tflops": FLOP_PER_FRAME * B * T / (ms_total / args.steps * 1e-3) / 1e12,
                       "frac": FLOP_PER_FRAME * B * T / (ms_total / args.steps * 1e-3) / 1e12 / peak},
        "note": "achieved = algorithmic FLOPs (recurrence 2*4H*H per frame per layer"
                + (" + its fused input projection 2*4H*C_in" if fused else "") + ") / CUDA-event time of the launches; "
                "fp16x2 issues 2 (split-bf16 'fp32': 3) 16-bit MMA FLOPs per algorithmic FLOP, so frac <= 1/2 (1/3) "
                "there; ncu's sm__pipe_tensor_cycles_active for every kernel is under profiles/",
    }

    # NCCL is used only to gather per-rank records (frames, time, output checksum) -- no data-path collective
    rec = torch.tensor([float(B * T), ms_total, float(out_h[1].double().sum())], device=dev, dtype=torch.float64)
    if world > 1:
        allrec = [torch.zeros_like(rec) for _ in range(world)]
        dist.all_gather(allrec, rec)
        ranks = [r.tolist() for r in allrec]
    else:
        ranks = [rec.tolist()]
    del streamer
    model_cpu_sd = state_dict
    del model
    torch.cuda.empty_cache()

    # ---- sub-records: the other BASELINE configs, measured in this run
    want = set(("cfg3", "cfg4", "cfg5") if args.configs == "all" else
               ([] if args.configs == "none" else args.configs.split(",")))
    ref = Reference()
    configs = {}

    def guarded(name, fn):
        try:
            r = fn()
            if r is not None:
                configs[name] = r
        except Exception as e:      # a failing sub-record must not take the headline line with it
            import traceback
            traceback.print_exc(file=sys.stderr)
            configs[name] = {"error": f"{type(e).__name__}: {e}"}

    if "cfg5" in want:
        if world > 1:
            r = sub_cfg5(ctx, ref, pk, args, args.precision)     # collective: every rank takes part
            if r is not None:
                configs["cfg5_sweep"] = r
        else:
            guarded("cfg5_sweep", lambda: sub_cfg5(ctx, ref, pk, args, args.precision))
    if world == 1 and "cfg3" in want:
        guarded("cfg3_metapool", lambda: sub_cfg3(ctx, ref, "pool", pk))
        guarded("cfg3_metaconv", lambda: sub_cfg3(ctx, ref, "conv", pk))
    if world == 1 and "cfg4" in want:
        guarded("cfg4_b32", lambda: sub_cfg4(ctx, ref, pk, 32))
        guarded("cfg4_b1", lambda: sub_cfg4(ctx, ref, pk, 1))

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(ref, model_cpu_sd, args)
        cfg = workload_config(args, world)
        cfg.update(precision=args.precision, lstm_launch=args.lstm,
                   lstm_input_projection="fused into the recurrence kernel" if fused else "separate GEMM",
                   plan_cache="weight digest kept in the timed region" if args.keep_digest else
                              "weights frozen after warm-up (model.freeze_weights(): no per-forward digest)")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "bf16x3 (split-bf16 three-product MMA, fp32 accumulate; fp32-grade)",
                      "fp16x2": "f16x2 (fp16 activations x two-term fp16 weights, two MMA passes, fp32 accumulate)",
                      "tf32": "tf32 (fp32 accumulate)", "bf16": "bf16 (fp32 accumulate)"}[args.precision],
            "data": "synthetic",
            "config": cfg,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "timed_region": "K x submit(pinned host inputs) ... flush(): ends after the last D2H has landed",
                    "clocks": sampler_e2e.summary() if sampler_e2e else None},
            "gpu_launches": launches,
            "clocks": sampler.summary() if sampler else None,
            "frac_of_model_roofline": value / world / (peak * 1e12 / FLOP_PER_FRAME),
            "kernels": kernels,
            "configs": configs,
            "ranks": [{"frames_per_step": r[0], "ms": r[1], "checksum": r[2]} for r in ranks],
        }
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_sweep(args):
    """--workload sweep: the cfg5 sub-record alone, printed as the JSON line (strong scaling)."""
    import torch.distributed as dist
    ctx = Ctx()
    pk = peaks()
    r = sub_cfg5(ctx, Reference(), pk, args, args.precision)
    if ctx.rank == 0:
        line = {"metric": METRIC, "value": r["frames_per_s"], "unit": UNIT, "n_gpus": ctx.world, "steps": 1, "warmup": 3,
                "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic", "config": {"workload": r["workload"]},
                "gpu_launches": r["launches"], "sweep": r}
        print(json.dumps(line))
    if ctx.world > 1:
        dist.destroy_process_group()
    return 0


def main():
    # stdout carries exactly ONE JSON line: keep NCCL's version banner (NCCL_DEBUG=VERSION prints to stdout) out of it
    if os.environ.get("NCCL_DEBUG", "WARN").upper() in ("VERSION", "WARN"):
        os.environ["NCCL_DEBUG"] = "WARN"      # an explicit value also overrides /etc/nccl.conf
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "sweep":
        return run_sweep(args)
    return run_native(args)


if __name__ == "__main__":
    sys.exit(main())
