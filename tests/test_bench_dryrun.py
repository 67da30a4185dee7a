"""bench.py code paths on CPU tensors with shrunken shapes (`--cpu-dryrun`): the JSON contract of both arms — same
metric/unit/config on the engine arm and on the unmodified-reference arm, `value` == `e2e.value`, required keys —
without a GPU box.  Never a measurement."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HAVE_REF = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "torchsnapshot"))


def _run(*extra):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--cpu-dryrun", "--steps", "2", "--warmup", "1", *extra],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, res.stdout[-2000:]
    return json.loads(lines[0])


def test_c3_line_contract_engine_arm():
    d = _run("--skip-cpu-baseline")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "e2e", "drain", "take_blocking_ms", "restore", "roofline", "e2e_roofline", "gpu_launches", "clocks"):
        assert k in d, k
    assert d["metric"] == "checkpoint_save_GBps" and d["unit"] == "GB/s" and d["steps"] == 2 and d["warmup"] == 1
    assert len(d["steps_ms"]) == 2
    assert d["value"] == d["e2e"]["value"] > 0 and d["restore"]["verified_all_tensors_all_ranks"] is True
    assert d["config"]["workload"].startswith("C3") and "impl" not in d


@pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref not staged")
def test_c3_reference_arm_is_the_unmodified_reference_on_the_same_config():
    ours = _run("--skip-cpu-baseline")
    ref = _run("--impl", "reference")
    assert ref["impl"] == "reference" and "unmodified" in ref["implementation"]
    assert ref["config"] == ours["config"], "both arms must describe the same workload"
    for k in ("metric", "unit", "higher_is_better", "scaling", "steps", "warmup", "n_gpus"):
        assert ref[k] == ours[k], k
    assert ref["cpu_baseline"]["kind"] == "reference" and ref["e2e"]["value"] == ref["value"] > 0
    assert ref["restore"]["verified_all_tensors_all_ranks"] is True


@pytest.mark.parametrize("cfg", ["c1", "c2", "c5"])
def test_other_configs_run(cfg):
    d = _run("--config", cfg)
    assert d["value"] > 0 and d["config"]["workload"].startswith(cfg.upper())
    assert d["steps"] == 2
    if cfg == "c5":  # the headline is the restore: --steps of them are timed
        assert d["e2e"]["timed_restores"] == 2


def test_dump_outputs_writes_the_last_steps_snapshot(tmp_path):
    """--dump-outputs: one float32 array per tensor of the last timed step's snapshot, equal to the seeded inputs (the
    dry run's snapshot is small enough to be written whole), identical from run to run."""
    import numpy as np
    import torch

    from benchmarks import workloads as W

    for run in ("a", "b"):
        _run("--skip-cpu-baseline", "--dump-outputs", str(tmp_path / run))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and len(names) == len(W.llama3_8b_shapes())
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    shapes = [(n, tuple(max(1, d // 32) for d in s)) for n, s in W.llama3_8b_shapes()]
    for name, (t, _, _) in W.build_llama_local(0, 1, torch.device("cpu"), shapes=shapes).items():
        a, b = np.load(tmp_path / "a" / f"0.model.{name}.npy"), np.load(tmp_path / "b" / f"0.model.{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, t.float().reshape(-1).numpy()) and np.array_equal(a, b), name
