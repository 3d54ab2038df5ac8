"""bench.py's multi-rank control flow on two CPU ranks (see tests/bench_dryrun.py): every rank reaches every collective (no
hang), only rank 0 prints, and the JSON line carries the contract's keys.  Both the graph-replay and the eager variants."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches",
        "clocks", "roofline", "cpu_baseline"}  # fmt: skip


def _run(nproc, port, *flags, timeout=900, env=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "bench_dryrun.py"), ROOT, "--gpus", str(nproc), "--steps", "2", "--warmup", "1", "--batch", "2", "--skip-cpu-baseline", *flags]  # fmt: skip
    return subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=dict(os.environ, OMP_NUM_THREADS="4", **(env or {})))


@pytest.mark.parametrize("flags", [(), ("--no-graph",)], ids=["graph", "eager"])
def test_bench_two_rank_control_flow(flags):
    out = _run(2, 29541 if flags else 29542, *flags)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert out.stderr.count("finished") == 2, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]  # rank 0 alone reports
    line = json.loads(lines[0])
    assert KEYS <= set(line), KEYS - set(line)
    assert line["n_gpus"] == 2 and line["config"]["global_batch"] == 4 and line["config"]["parallelism"] == "dp2"
    assert line["config"]["cuda_graph"] == (not flags)
    assert line["value"] > 0 and line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] > 0
    assert line["roofline"]["conv_ms_per_step"] > 0 and line["gpu_launches"] == 0  # the stand-ins launch nothing


def test_bench_single_rank_control_flow():
    out = _run(1, 29543)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert KEYS <= set(line) and line["n_gpus"] == 1 and line["config"]["cuda_graph"] is True and line["value"] > 0


def test_bench_remeasures_a_throttled_region_on_every_rank():
    """Rank 0 alone sees hw_slowdown in the first timed region: its verdict is broadcast, BOTH ranks run the region again (it contains
    the gradient all-reduce), and the line records why."""
    out = _run(2, 29544, "--no-graph", env={"SGB_DRYRUN_THROTTLE": "1"})
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert out.stderr.count("finished") == 2
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert line["clocks"]["reasons"] == [] and line["clocks"]["remeasured_after"]["reasons"] == ["hw_slowdown"]


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs writes the last timed step's loss, its items and a sample of the trained parameters and of their EMA as float32 /
    float64 .npy files within 64 MB.  The same arguments give the same inputs and the same arrays; another --steps trains further."""
    import numpy as np

    runs = {"a": (), "b": (), "c": ("--steps", "3")}
    for port, (name, flags) in zip((29545, 29546, 29547), runs.items()):
        out = _run(1, port, "--dump-outputs", str(tmp_path / name), *flags)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["ema_params_sample.npy", "loss.npy", "loss_items.npy", "params_sample.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 << 20
    for n in names:
        a, b, c = (np.load(tmp_path / r / n) for r in runs)
        assert a.dtype in (np.float32, np.float64) and a.size and np.isfinite(a).all(), n
        assert np.array_equal(a, b), n
    assert not np.array_equal(np.load(tmp_path / "a" / "params_sample.npy"), np.load(tmp_path / "c" / "params_sample.npy"))
