"""bench.py's reference arm (the reference's CPU path on the host cores: the unmodified classes from baseline/_ref when
that install exists, else the oracle port) runs without a GPU; its JSON line must carry the keys the driver reads, alone
and under torchrun (rank 0 prints, the other ranks exit 0).  `--dump-outputs` of the native arm: the sampling of
outputs above its size limit (CPU) and the files of a small run (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e")


def _check(line, n_gpus, steps):
    d = json.loads(line)
    assert all(k in d for k in KEYS), [k for k in KEYS if k not in d]
    assert d["impl"] == "reference" and d["n_gpus"] == n_gpus and d["steps"] == steps and d["higher_is_better"] is True
    assert d["value"] > 0 and d["unit"] == "frames/s" and d["vs_baseline"] is None and "workload" in d["config"]
    cb = d["cpu_baseline"]
    have_ref = os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "factory", "AutoVC.py"))
    assert cb["kind"] == ("reference" if have_ref else "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert cb["sample"] and cb["sample_batch"] >= 16 and cb["cpu_model"]
    # both arms print the same `config` object for the same command line (the driver compares them)
    assert set(d["config"]) == {"workload", "batch_per_gpu", "frames", "parallelism", "l2"}
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_single_process():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--batch", "32"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    _check(lines[0], 1, 2)


def test_reference_arm_under_torchrun():
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29561", os.path.join(ROOT, "bench.py"),
                          "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--batch", "32"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                      # rank 0 alone prints
    _check(lines[0], 2, 1)


def test_dump_outputs_samples_the_same_utterances_under_the_limit(tmp_path):
    """--dump-outputs above 64 MB: every array keeps the same utterances, in batch order, the same on every run."""
    import bench
    B, T = 128, 1024                                     # 2 x 42 MB of mel: over the limit
    row = torch.arange(B, dtype=torch.float32)
    outs = dict(mel=row.view(B, 1, 1, 1).expand(B, 1, T, 80).contiguous(),
                mel_postnet=-row.view(B, 1, 1, 1).expand(B, 1, T, 80).contiguous(),
                codes=row.view(B, 1).expand(B, 256).contiguous())
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["codes.npy", "mel.npy", "mel_postnet.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_LIMIT
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    kept = got["codes"][:, 0]
    assert 0 < len(kept) < B and (np.diff(kept) > 0).all()
    assert (got["mel"] == kept[:, None, None, None]).all() and (got["mel_postnet"] == -kept[:, None, None, None]).all()
    assert all(v.dtype == np.float32 for v in got.values())
    assert all(np.array_equal(got[f[:-4]], np.load(tmp_path / "b" / f)) for f in files)


@pytest.mark.gpu
def test_native_arm_dumps_last_step_outputs(tmp_path):
    """--steps sets the timed steps; --dump-outputs writes the headline batch whole when it fits, finite float32."""
    B, T = 8, 64
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                          "--batch", str(B), "--frames", str(T), "--configs", "none", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    shapes = dict(mel=(B, 1, T, 80), mel_postnet=(B, 1, T, 80), codes=(B, 2 * 32 * T // 32))
    for name, shape in shapes.items():
        a = np.load(tmp_path / f"{name}.npy")
        assert a.shape == shape and a.dtype == np.float32 and np.isfinite(a).all(), name
