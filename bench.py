#!/usr/bin/env python3
"""Headline benchmark: checkpoint GB/s and Snapshot.take() blocking ms (BASELINE.json), one process per GPU.

    python bench.py --gpus 1 --steps K --warmup W                       # this repo's engine, config C3
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    # ... and write what the last timed step computed
    python bench.py --impl reference --gpus 1 --steps K --warmup W      # the UNMODIFIED reference (oracle/_ref)
    torchrun ... bench.py --gpus N ... [--config c2|c3|c4|c5]

Both arms run the same code below on the same seeded app_state and differ only in the module they call:
``torchsnapshot_b200`` (this repo) or ``torchsnapshot`` staged from /root/reference by oracle/make_ref.sh.

One "step" of the default config (C3) = one ``Snapshot.take`` of an FSDP-layout Llama-3-8B bf16 sharded state dict
(16.06 GB total, dim-0 sharded over the ranks) into a fresh directory of the local filesystem, timed like
T:benchmarks/ddp/main.py:62-70 (barrier + synchronize on both sides), max over ranks.

  value / e2e.value : sum of payload bytes / take wall time  ("checkpoint GB/s": D2H copies, file writes and the
                      metadata commit are inside the timed region; reference semantics = returned, not fsynced)
  drain             : the device side alone, in situ: pack-kernel ms and the D2H span of the same takes
  take_blocking_ms  : time inside async_take() (the training loop is blocked), and inside take()
  restore           : the mirror: Snapshot.restore GB/s
  roofline          : the dominant kernel (bulk pack) against the measured HBM copy peak
  e2e_roofline      : the whole take against min(sum of the ranks' D2H link, host write sink), both measured in this
                      run with the engine's own ring and workers
  cpu_baseline      : the unmodified reference on a bounded sample (rank 0, N=1)

--dump-outputs DIR writes, after the timed steps, the tensors in the snapshot of the last timed step (read back from
its payload files; the restored table too for C5, whose headline is the restore) as DIR/<name>.npy, float32 or float64,
so that two builds can be compared output for output: the inputs are seeded, and a snapshot larger than 64 MB is
sampled at the same seeded element indices in every run.
"""
from __future__ import annotations

import argparse
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: nothing is written into it

import numpy as np  # noqa: E402

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from benchmarks import workloads as W  # noqa: E402

# kept for callers of the round-1 names
llama3_8b_shapes = W.llama3_8b_shapes
local_rows = W.local_rows
build_local_tensors = W.build_llama_local
wrap_sharded = W.wrap_sharded
wrap_dtensor = W.wrap_dtensor

REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def load_impl(impl: str):
    """The snapshot module of an arm.  'reference' is the unmodified pytorch/torchsnapshot package staged by
    oracle/make_ref.sh (pure Python; nothing of this repo is on its path of execution)."""
    if impl == "ours":
        import torchsnapshot_b200 as T

        return T, "torchsnapshot_b200"
    if not os.path.isdir(os.path.join(REF_DIR, "torchsnapshot")):
        return None, f"{REF_DIR}/torchsnapshot missing: run oracle/make_ref.sh where /root/reference exists"
    sys.path.insert(0, REF_DIR)
    import torchsnapshot as T  # noqa: E402

    assert os.path.abspath(T.__file__).startswith(REF_DIR), T.__file__
    commit = ""
    try:
        commit = open(os.path.join(REF_DIR, "REF_COMMIT")).read().strip()
    except OSError:
        pass
    return T, f"pytorch/torchsnapshot (unmodified, oracle/_ref, commit {commit or 'unknown'})"


# ---- clocks sampling (B200_PROFILING.md recipe) ---------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int) -> None:
        self.index = index
        self.proc = None
        self.lines = []

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self) -> None:
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---- helpers -------------------------------------------------------------------------------------------
def _sync(device) -> None:
    if device.type == "cuda":
        torch.cuda.synchronize(device)


def _engine(T, device):
    return T.get_engine(device.index if device.type == "cuda" else -1)


class Ctx:
    def __init__(self, args, rank, world, local_rank, device, base_dir):
        self.args, self.rank, self.world, self.local_rank, self.device, self.base = args, rank, world, local_rank, device, base_dir

    def path(self, tag: str) -> str:
        return os.path.join(self.base, tag)

    def barrier(self) -> None:
        if dist.is_initialized() and dist.get_world_size() > 1:
            if dist.get_backend() == "nccl":
                dist.barrier(device_ids=[self.device.index])
            else:
                dist.barrier()

    def _reduce(self, x: float, op) -> float:
        if not dist.is_initialized() or dist.get_world_size() == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=self.device if dist.get_backend() == "nccl" else "cpu")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x: float) -> float:
        return self._reduce(x, dist.ReduceOp.MAX)

    def sum(self, x: float) -> float:
        return self._reduce(x, dist.ReduceOp.SUM)

    def min(self, x: float) -> float:
        return self._reduce(x, dist.ReduceOp.MIN)

    def cleanup(self, tag: str) -> None:
        self.barrier()
        if self.rank == 0:
            shutil.rmtree(self.path(tag), ignore_errors=True)
        self.barrier()

    def timed(self, fn) -> float:
        """ms of fn(), bracketed like T:benchmarks/ddp/main.py:62-70, max over ranks."""
        self.barrier()
        _sync(self.device)
        t0 = time.perf_counter()
        out = fn()
        _sync(self.device)
        dt = (time.perf_counter() - t0) * 1e3
        return self.max(dt), out


def device_job(stats_list):
    """The engine job that touched the GPU (mixed CPU/GPU states also have a host-only job for the CPU tensors)."""
    jobs = stats_list or [{}]
    return max(jobs, key=lambda j: (j.get("n_kernel_launches", 0), j.get("direct_bytes", 0), j.get("payload_bytes", 0)))


class CpuMeter:
    """Host cores actually used by this process while a timed call runs: (user + system CPU time) / wall, and the
    largest thread count seen — measured, per rank."""

    def __init__(self) -> None:
        self.cpu_s = 0.0
        self.wall_s = 0.0
        self.max_threads = 0
        self._stop = None

    def start(self) -> None:
        import psutil

        self._t0 = time.perf_counter()
        t = os.times()
        self._c0 = t.user + t.system
        proc = psutil.Process()
        self._stop = threading.Event()

        def watch():
            while not self._stop.wait(0.02):
                try:
                    self.max_threads = max(self.max_threads, proc.num_threads())
                except Exception:
                    return

        self._th = threading.Thread(target=watch, daemon=True)
        self._th.start()

    def stop(self) -> None:
        t = os.times()
        self.cpu_s += t.user + t.system - self._c0
        self.wall_s += time.perf_counter() - self._t0
        self._stop.set()
        self._th.join()

    def report(self) -> dict:
        return {"cores_busy_avg": round(self.cpu_s / self.wall_s, 2) if self.wall_s else None, "threads_max": self.max_threads}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def mean(xs):
    xs = list(xs)
    return sum(xs) / len(xs) if xs else 0.0


def host_info(world: int) -> dict:
    return {"cpu_count": os.cpu_count(), "ranks_on_host": world, "cores_per_rank": (os.cpu_count() or 0) // max(1, world)}


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The single JSON line goes to the process's original stdout; everything else (NCCL banners, warnings
    printed by libraries) was re-routed to stderr in main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def ours_engine_extras(ctx: Ctx, eng, payload_local: int, want_write_probe: bool = True) -> dict:
    """Link and sink ceilings measured with the engine's own ring/workers, all ranks at once (they share the host)."""
    from torchsnapshot_b200 import _native as N

    out = {}
    nb = min(max(payload_local, 1 << 30), 4 << 30)
    ctx.barrier()
    d2h = eng.probe(N.PROBE_D2H, nb)
    ctx.barrier()
    h2d = eng.probe(N.PROBE_H2D, nb)
    out["link_d2h_gbs_sum"] = ctx.sum(d2h)
    out["link_h2d_gbs_sum"] = ctx.sum(h2d)
    out["link_d2h_gbs_min_rank"] = ctx.min(d2h)
    if want_write_probe:
        pdir = ctx.path(f"probe_r{ctx.rank}")
        os.makedirs(pdir, exist_ok=True)
        # best of 3 passes (fresh files each), every rank at once; the engine times only the I/O
        best_w = 0.0
        for _ in range(3):
            ctx.barrier()
            best_w = max(best_w, ctx.sum(eng.probe(N.PROBE_WRITE, nb, pdir)))
        ctx.barrier()
        rd = ctx.sum(eng.probe(N.PROBE_READ, nb, pdir))
        out["sink_write_gbs"] = best_w
        out["source_read_gbs"] = rd
        shutil.rmtree(pdir, ignore_errors=True)
    out["probe_bytes_per_rank"] = nb
    return out


def dump_trace(ctx: Ctx, tag: str, traces, out_dir: str) -> dict:
    """Writes the timeline of rank 0's job (Chrome trace + summary) and returns the summary."""
    from torchsnapshot_b200 import timeline as TL

    if not traces or not traces[0]:
        return {}
    summary = TL.summarize(traces[0])
    if ctx.rank == 0 and out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, f"{tag}_trace.json"), "w") as f:
            f.write(TL.to_chrome_trace(traces[0], tag))
        with open(os.path.join(out_dir, f"{tag}_summary.json"), "w") as f:
            json.dump(summary, f, indent=1)
    return summary


# ---- --dump-outputs -------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64_000_000


def _tensor_pieces(snap_dir: str):
    """(name, tensor entry) of every stored piece of every tensor in the snapshot's manifest, in manifest order."""
    with open(os.path.join(snap_dir, ".snapshot_metadata")) as f:
        manifest = json.load(f)["manifest"]
    for path, e in manifest.items():
        if e.get("type") == "Tensor":
            pieces = [e]
        elif e.get("type") == "ChunkedTensor":
            pieces = [c["tensor"] for c in e["chunks"]]
        elif e.get("type") in ("ShardedTensor", "DTensor"):
            pieces = [s["tensor"] for s in e["shards"]]
        else:
            continue
        for i, te in enumerate(pieces):
            yield path.replace("/", ".") + (f".piece{i}" if len(pieces) > 1 else ""), te


def _out_dtype(dtype: torch.dtype):
    return np.float64 if dtype in (torch.float64, torch.int32, torch.int64) else np.float32


def _sample(name: str, flat, numel: int, keep: int):
    """All of flat (1-D, indexable) or `keep` of its elements at indices seeded by the name: the same in every run."""
    if keep >= numel:
        return flat[:numel]
    idx = np.unique(np.random.default_rng(zlib.crc32(name.encode())).integers(0, numel, keep))
    return flat[torch.from_numpy(idx).to(flat.device)] if isinstance(flat, torch.Tensor) else flat[idx]


def _read_piece(snap_dir: str, te: dict, name: str, keep: int) -> np.ndarray:
    dtype = getattr(torch, te["dtype"].split(".")[-1])
    numel = 1
    for d in te["shape"]:
        numel *= d
    path = os.path.join(snap_dir, te["location"])
    lo = te["byte_range"][0] if te.get("byte_range") else 0
    if te["serializer"] == "buffer_protocol":
        esz = torch.empty(0, dtype=dtype).element_size()
        raw = np.memmap(path, dtype={1: np.int8, 2: np.int16, 4: np.int32, 8: np.int64}[esz], mode="r", offset=lo, shape=(numel,))
        vals = torch.from_numpy(np.array(_sample(name, raw, numel, keep))).view(dtype)
    else:  # torch_save
        with open(path, "rb") as f:
            f.seek(lo)
            blob = f.read(te["byte_range"][1] - lo) if te.get("byte_range") else f.read()
        t = torch.load(io.BytesIO(blob), map_location="cpu", weights_only=True)
        vals = _sample(name, t.reshape(-1), numel, keep)
    return vals.to(torch.float64 if _out_dtype(dtype) is np.float64 else torch.float32).numpy()


def dump_outputs(ctx: Ctx, snap_dir: str, extra=None) -> None:
    """--dump-outputs: every tensor piece of the snapshot at snap_dir (+ `extra` {name: tensor}) as DIR/<name>.npy,
    each sampled in proportion to its size when all of them would exceed DUMP_LIMIT_BYTES."""
    out_dir = ctx.args.dump_outputs
    if not out_dir or ctx.rank != 0:
        return
    items = [(n, te, 1) for n, te in _tensor_pieces(snap_dir)]
    items += [(n, t, 0) for n, t in (extra or {}).items()]
    sizes = []
    for n, x, from_file in items:
        dtype = getattr(torch, x["dtype"].split(".")[-1]) if from_file else x.dtype
        numel = int(np.prod(x["shape"])) if from_file else x.numel()
        sizes.append((numel, np.dtype(_out_dtype(dtype)).itemsize))
    total = sum(n * b for n, b in sizes)
    budget = DUMP_LIMIT_BYTES - 256 * len(items)  # .npy headers
    os.makedirs(out_dir, exist_ok=True)
    for (name, x, from_file), (numel, b) in zip(items, sizes):
        keep = numel if total <= budget else max(1, numel * budget // total)
        if from_file:
            arr = _read_piece(snap_dir, x, name, keep)
        else:
            arr = _sample(name, x.detach().reshape(-1), numel, keep).to(torch.float64 if b == 8 else torch.float32).cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)


# ---- C3: FSDP-layout Llama-3-8B ---------------------------------------------------------------------------------
C3_WORKLOAD = "C3: FSDP-layout Llama-3-8B bf16 sharded state_dict (291 tensors, 16.06 GB total, dim-0 sharded over n_gpus), Snapshot.take to local fs"


def common_line(ctx: Ctx, impl_desc: str, metric: str, value: float, unit: str, ms: float, config: dict, higher=True, scaling="strong") -> dict:
    a = ctx.args
    line = {
        "metric": metric,
        "value": value,
        "unit": unit,
        "n_gpus": ctx.world,
        "steps": a.steps,
        "warmup": a.warmup,
        "ms_per_step": ms,
        "higher_is_better": higher,
        "scaling": scaling,
        "vs_baseline": None,
        "dtype": config.pop("_dtype", "bf16 (byte copy)"),
        "data": "synthetic",
        "config": config,
        "implementation": impl_desc,
        "host": host_info(ctx.world),
    }
    if a.impl == "reference":
        line["impl"] = "reference"
    return line


def run_c3(ctx: Ctx, T, impl_desc: str) -> None:
    a, rank, world, device = ctx.args, ctx.rank, ctx.world, ctx.device
    ours = a.impl == "ours"
    shapes = [(n, tuple(max(1, d // 32) for d in s)) for n, s in W.llama3_8b_shapes()] if a.cpu_dryrun else None
    local = W.build_llama_local(rank, world, device, shapes=shapes)
    payload_local = sum(t.numel() * t.element_size() for t, _, _ in local.values())
    payload_total = ctx.sum(float(payload_local))
    if a.layout == "dtensor":
        state = W.wrap_dtensor(local, world, device)
    elif a.layout == "plain":
        state = {k: t for k, (t, _, _) in local.items()}
    else:
        state = W.wrap_sharded(local, rank, device)
    app_state = {"model": T.StateDict(**state)}
    eng = S = None
    if ours:
        from torchsnapshot_b200 import scheduler as S

        eng = _engine(T, device)

    for w in range(a.warmup):
        T.Snapshot.take(ctx.path(f"warm{w}"), app_state)
        ctx.cleanup(f"warm{w}")

    # -- timed steps: Snapshot.take through the public API --
    launches0 = eng.stats()["kernels_launched"] if ours else 0
    sampler = ClockSampler(device.index)
    if rank == 0:
        sampler.start()
    step_ms, per_step = [], []
    cpu = CpuMeter()
    for k in range(a.steps):
        cpu.start()
        ms, _ = ctx.timed(lambda: T.Snapshot.take(ctx.path(f"step{k}"), app_state))
        cpu.stop()
        step_ms.append(ms)
        if ours:
            per_step.append(device_job(S.LAST_STATS.get("save")))
        if k + 1 < a.steps:
            ctx.cleanup(f"step{k}")
    clocks = sampler.stop() if rank == 0 else {}
    launches = eng.stats()["kernels_launched"] - launches0 if ours else 0
    take_ms = mean(step_ms)
    take_gbs = payload_total / 1e9 / (take_ms / 1e3)
    keep_tag = f"step{a.steps - 1}"
    take_phases = dict(S.LAST_STATS.get("take_phases_ms") or {}) if ours else {}
    write_phases = dict(S.LAST_STATS.get("write_phases_ms") or {}) if ours else {}

    # -- restore (the snapshot of the last step) --
    restore_ms = []
    for _ in range(min(a.steps, 3)):
        for t, _, _ in local.values():
            t.zero_()
        ms, _ = ctx.timed(lambda: T.Snapshot(ctx.path(keep_tag)).restore(app_state))
        restore_ms.append(ms)
    load_stats = device_job(S.LAST_STATS.get("load")) if ours else {}
    regen = W.build_llama_local(rank, world, device, shapes=shapes)
    ok = all(torch.equal(local[n][0], regen[n][0]) for n in local)
    del regen
    ok = bool(ctx.min(1.0 if ok else 0.0))
    dump_outputs(ctx, ctx.path(keep_tag))
    ctx.cleanup(keep_tag)

    # -- async_take: how long the caller is blocked --
    block_ms, async_total_ms = [], []
    for k in range(min(a.steps, 3 if ours else 2)):
        ctx.barrier()
        _sync(device)
        t0 = time.perf_counter()
        pending = T.Snapshot.async_take(ctx.path(f"async{k}"), app_state)
        t1 = time.perf_counter()
        pending.wait()
        t2 = time.perf_counter()
        block_ms.append(ctx.max((t1 - t0) * 1e3))
        async_total_ms.append(ctx.max((t2 - t0) * 1e3))
        ctx.cleanup(f"async{k}")
    blocking_stats = device_job(S.LAST_STATS.get("save")) if ours else {}

    config = {
        "workload": C3_WORKLOAD,
        "layout": a.layout,
        "world_size": world,
        "payload_bytes_total": int(payload_total),
        "target_fs": a.target_fs,
        "semantics": "returned (no fsync), like the reference's fs plugin (T:storage_plugins/fs.py:36-38)",
        "l2": "inputs (>=2 GB per rank) exceed the 126 MB L2; every step writes a fresh directory",
    }
    line = common_line(ctx, impl_desc, "checkpoint_save_GBps", take_gbs, "GB/s", take_ms, config)
    line["e2e"] = {
        "value": take_gbs,
        "unit": "GB/s",
        "ms_per_step": take_ms,
        "h2d_bytes_per_step": int(mean(st.get("table_h2d_bytes", 0) for st in per_step)) if ours else 0,
        "d2h_bytes_per_step": int(payload_local),
        "definition": "Snapshot.take(path, app_state) wall clock through the public API: planning collectives, device->host copies of this rank's payload, file writes, metadata commit; max over ranks.  value is this same quantity.",
    }
    line["steps_ms"] = [round(x, 2) for x in step_ms]
    line["take_blocking_ms"] = {"async_take_returns_ms": mean(block_ms), "async_total_ms": mean(async_total_ms), "timed_async_takes": len(block_ms), "sync_take_ms": take_ms,
                                "engine_device_done_ms": blocking_stats.get("device_done_ms"), "async_take_returns_ms_each": [round(x, 2) for x in block_ms],
                                "phases_of_last_async_take_ms": {k: round(v, 2) for k, v in ((S.LAST_STATS.get("take_phases_ms") or {}) if ours else {}).items()},
                                "write_phases_of_last_async_take_ms": {k: round(v, 2) for k, v in ((S.LAST_STATS.get("write_phases_ms") or {}) if ours else {}).items()}}
    line["restore"] = {"value": payload_total / 1e9 / (mean(restore_ms) / 1e3), "unit": "GB/s", "ms": mean(restore_ms), "timed_restores": len(restore_ms), "verified_all_tensors_all_ranks": ok,
                       "scatter_kernel_ms": load_stats.get("kernel_ms")}
    line["clocks"] = clocks
    host_cpu = cpu.report()
    line["host_cpu_during_take"] = {"cores_busy_avg_max_over_ranks": ctx.max(host_cpu["cores_busy_avg"] or 0.0), "threads_max_rank0": host_cpu["threads_max"],
                                    "definition": "(user+system CPU seconds of the rank's process) / wall seconds over the timed takes; threads = peak thread count of the process"}
    line["payload_bytes_per_rank"] = int(payload_local)
    line["gpu_launches"] = int(launches)

    if ours:
        from torchsnapshot_b200 import _native as N

        kernel_ms = ctx.max(mean(st.get("kernel_ms", 0.0) for st in per_step))
        bulk_ms = mean(st.get("kernel_bulk_ms", 0.0) for st in per_step)
        copy_ms = ctx.max(mean(st.get("copy_ms", 0.0) for st in per_step))
        last = per_step[-1] if per_step else {}
        line["drain"] = {
            "pack_kernel_ms": kernel_ms,
            "d2h_span_ms": copy_ms,
            "gbs": payload_total / 1e9 / ((kernel_ms + copy_ms) / 1e3) if kernel_ms + copy_ms > 0 else None,
            "link_starved_ms": ctx.max(mean(st.get("link_starved_ms", 0.0) for st in per_step)),
            "definition": "device side of the same timed takes: CUDA-event time of the pack kernels + first-to-last D2H span on the copy stream (includes waits for free pinned slots, i.e. back-pressure from the writers); link_starved_ms = time the link idled for want of a pinned slot (no copy queued); max over ranks",
        }
        line["engine_step"] = {k: last.get(k) for k in ("plan_ms", "kernel_ms", "copy_ms", "device_done_ms", "total_ms", "n_files", "n_members", "n_tiles_bulk", "n_tiles_lsu",
                                                           "n_kernel_launches", "arena_bytes", "n_waves", "direct_bytes", "n_memcpy", "slot_wait_ms", "link_starved_ms", "io_busy_ms", "io_queue_ms")}
        line["take_phases_ms"] = {k: round(v, 2) for k, v in take_phases.items()}
        line["write_phases_ms"] = {k: round(v, 2) for k, v in write_phases.items()}
        line["host"]["engine_io_threads_per_rank"] = eng.io_threads
        line["host"]["pinned_ring"] = f"{eng.pinned_slots} x {eng.pinned_slot_bytes >> 20} MiB"
        # roofline of the dominant kernel: per launch it moves this rank's payload twice (read + write)
        peaks, peaks_src = measured_peaks()
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        bulk_bytes = 2.0 * float(last.get("bytes_bulk", payload_local))
        achieved = bulk_bytes / 1e9 / (bulk_ms / 1e3) if bulk_ms > 0 else 0.0
        traffic, traffic_src = a.ncu_traffic_bytes, "command line"
        if traffic is None:
            try:
                with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                    cap = json.load(f)
                # DRAM traffic per algorithmic byte of the same kernel from the committed `ncu --set full` capture (N=1)
                traffic = cap["traffic_bytes"] * (bulk_bytes / cap["algorithmic_bytes"])
                traffic_src = f"profiles/ncu_traffic.json ({cap.get('capture')}): measured ratio {cap['traffic_bytes'] / cap['algorithmic_bytes']:.4f} x this launch's algorithmic bytes"
            except Exception:
                traffic, traffic_src = None, "no capture"
        line["roofline"] = {"bound": "hbm", "kernel": "tsnap_bulk_copy_kernel (pack)", "achieved": achieved, "peak": hbm_peak,
                            "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks_src})", "unit": "GB/s", "frac": achieved / hbm_peak if hbm_peak else None,
                            "algorithmic_bytes_per_launch": bulk_bytes, "launch_ms": bulk_ms, "traffic": traffic, "traffic_source": traffic_src,
                            "share_of_step": bulk_ms / take_ms if take_ms else None}
        probes = ours_engine_extras(ctx, eng, payload_local) if device.type == "cuda" else {"link_d2h_gbs_sum": 1.0, "link_h2d_gbs_sum": 1.0}
        sink = probes.get("sink_write_gbs")
        peak = min(probes["link_d2h_gbs_sum"], sink) if sink else probes["link_d2h_gbs_sum"]
        line["e2e_roofline"] = {"bound": "host link / host write sink", "achieved": take_gbs, "peak": peak, "unit": "GB/s", "frac": take_gbs / peak if peak else None,
                                "link_d2h_gbs_all_ranks": probes["link_d2h_gbs_sum"], "host_write_peak_gbs": sink,
                                "restore_peak": min(probes["link_h2d_gbs_sum"], probes.get("source_read_gbs") or 1e9),
                                "restore_frac": line["restore"]["value"] / min(probes["link_h2d_gbs_sum"], probes.get("source_read_gbs") or 1e9),
                                "how": "tsnap_engine_probe: ring-slot-sized cudaMemcpyAsync chunks HBM<->pinned ring (link) and the engine's I/O workers writing/reading fresh files from the ring (sink/source), every rank at once, right after the timed steps",
                                "probes": probes}
        # -- one traced take + restore (untimed): pack || D2H || pwrite overlap evidence --
        if a.trace_dir:
            N.reset_engines()
            os.environ["TSNAP_B200_ENGINE_FLAGS"] = str(int(os.environ.get("TSNAP_B200_ENGINE_FLAGS", "0")) | N.ENGINE_TRACE)
            for t in ("tracewarm", "trace"):
                T.Snapshot.take(ctx.path(t), app_state)
            ts = dump_trace(ctx, f"{a.trace_tag}_take_n{world}", S.LAST_STATS.get("save_trace"), a.trace_dir)
            T.Snapshot(ctx.path("trace")).restore(app_state)
            tr = dump_trace(ctx, f"{a.trace_tag}_restore_n{world}", S.LAST_STATS.get("load_trace"), a.trace_dir)
            line["timeline"] = {"take": {k: ts.get(k) for k in ("overlap", "job_span_ms")}, "restore": {k: tr.get(k) for k in ("overlap", "job_span_ms")}}
            ctx.cleanup("tracewarm")
            ctx.cleanup("trace")
        # -- cpu baseline: the unmodified reference on a bounded sample (rank 0, N=1) --
        if rank == 0 and world == 1 and not a.skip_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_c3(ctx, local)
    else:
        line["cpu_baseline"] = {"value": take_gbs, "unit": "GB/s", "kind": "reference", "cores": round(line["host_cpu_during_take"]["cores_busy_avg_max_over_ranks"], 2),
                                "cores_definition": "measured: CPU seconds / wall seconds of one rank's process during the timed takes (max over ranks); the pipeline's thread budget is 1 + 4 + 16 per rank (T:scheduler.py:32, T:knobs.py:38)",
                                "threads_max_rank0": host_cpu["threads_max"], "host_cores_available": os.cpu_count(),
                                "sample": "the whole workload on every rank (no sampling): same app_state, same ranks, same target directory as the other arm"}
    if rank == 0:
        emit(line)


def reference_threads() -> int:
    """Host threads the reference's pipeline uses per rank: asyncio loop + 4 staging threads (T:scheduler.py:32) + the
    loop's default executor running aiofiles calls for <=16 concurrent I/Os (T:knobs.py:38; ThreadPoolExecutor default
    min(32, cpu+4) workers)."""
    return 1 + 4 + 16


def cpu_baseline_c3(ctx: Ctx, local) -> dict:
    Tref, desc = load_impl("reference")
    if Tref is None:
        return {"unavailable": desc}
    sample, total = {}, 0
    limit = ctx.args.ref_sample_gib << 30
    for name, (t, shape, lo) in local.items():
        nb = t.numel() * t.element_size()
        if total + nb > limit and sample:
            continue
        sample[name] = (t, shape, lo)
        total += nb
    app = {"model": Tref.StateDict(**W.wrap_sharded(sample, 0, ctx.device))}
    times = []
    for rep in range(3):
        d = ctx.path(f"cpu{rep}")
        _sync(ctx.device)
        t0 = time.perf_counter()
        Tref.Snapshot.take(d, app)
        _sync(ctx.device)
        if rep:
            times.append(time.perf_counter() - t0)
        shutil.rmtree(d, ignore_errors=True)
    return {"value": total / 1e9 / mean(times), "unit": "GB/s", "cores": reference_threads(), "host_cores_available": os.cpu_count(), "kind": "reference",
            "sample": f"unmodified torchsnapshot.Snapshot.take on {len(sample)} of {len(local)} ShardedTensors ({total / 1e9:.2f} GB), 2 timed passes after 1 warm-up"}


# ---- C2: DDP ResNet-50 + Adam ------------------------------------------------------------------------------------
def run_c2(ctx: Ctx, T, impl_desc: str) -> None:
    a, rank, world, device = ctx.args, ctx.rank, ctx.world, ctx.device
    ours = a.impl == "ours"
    app_state, kw, payload = W.build_c2(T, rank, world, device, ctx.local_rank)
    S = eng = None
    if ours:
        from torchsnapshot_b200 import scheduler as S

        eng = _engine(T, device)
    for w in range(a.warmup):
        T.Snapshot.take(ctx.path(f"warm{w}"), app_state, **kw)
        ctx.cleanup(f"warm{w}")
    launches0 = eng.stats()["kernels_launched"] if ours else 0
    step_ms, per_step, phases = [], [], []
    coll_per_take = None
    for k in range(a.steps):
        if ours:
            from torchsnapshot_b200 import pg_wrapper as PGW

            c0 = PGW.COLLECTIVE_COUNT["total"]
        ms, _ = ctx.timed(lambda: T.Snapshot.take(ctx.path(f"step{k}"), app_state, **kw))
        if ours:
            coll_per_take = PGW.COLLECTIVE_COUNT["total"] - c0
        step_ms.append(ms)
        if ours:
            per_step.append(device_job(S.LAST_STATS.get("save")))
            phases.append(dict(S.LAST_STATS.get("take_phases_ms") or {}))
        if k + 1 < a.steps:
            ctx.cleanup(f"step{k}")
    launches = eng.stats()["kernels_launched"] - launches0 if ours else 0
    keep = f"step{a.steps - 1}"
    # restore into perturbed copies
    sd = app_state["model"].state_dict()
    saved = {k: v.clone() for k, v in sd.items()}
    opt = app_state["optim"]
    saved_opt = [{k: v.clone() for k, v in st.items()} for st in opt.state.values()]
    restore_ms = []
    for _ in range(min(a.steps, 3)):
        with torch.no_grad():
            for v in sd.values():
                v.zero_()
            for st in opt.state.values():
                for v in st.values():
                    v.zero_()
        ms, _ = ctx.timed(lambda: T.Snapshot(ctx.path(keep)).restore(app_state))
        restore_ms.append(ms)
    sd2 = app_state["model"].state_dict()
    ok = all(torch.equal(saved[k], sd2[k]) for k in saved)
    for st, ref in zip(opt.state.values(), saved_opt):
        ok = ok and all(torch.equal(st[k], ref[k]) for k in ref)
    ok = bool(ctx.min(1.0 if ok else 0.0))
    # manifest facts
    man = T.Snapshot(ctx.path(keep)).get_manifest()
    n_entries = len(man)
    dump_outputs(ctx, ctx.path(keep))
    ctx.cleanup(keep)
    take_ms = mean(step_ms)
    config = {"workload": "C2: DDP ResNet-50 (320 state_dict tensors) + Adam (exp_avg, exp_avg_sq, 0-d fp32 CPU step per parameter), replicated=['**'], partitioned write to local fs",
              "world_size": world, "payload_bytes_total": int(payload), "target_fs": a.target_fs, "_dtype": "fp32/int64 (byte copy)",
              "semantics": "returned (no fsync)", "l2": "payload (0.31 GB) exceeds the 126 MB L2 at N<=2; fresh directory every step"}
    line = common_line(ctx, impl_desc, "checkpoint_save_GBps", payload / 1e9 / (take_ms / 1e3), "GB/s", take_ms, config)
    line["e2e"] = {"value": line["value"], "unit": "GB/s", "ms_per_step": take_ms, "h2d_bytes_per_step": int(mean(st.get("table_h2d_bytes", 0) for st in per_step)) if ours else 0,
                   "d2h_bytes_per_step": int(payload // max(1, world)), "definition": "Snapshot.take wall clock, max over ranks; replicated payload counted once"}
    line["steps_ms"] = [round(x, 2) for x in step_ms]
    line["restore"] = {"ms": mean(restore_ms), "value": payload * world / 1e9 / (mean(restore_ms) / 1e3), "unit": "GB/s (every rank restores the full replicated state)", "timed_restores": len(restore_ms), "verified": ok}
    line["manifest_entries"] = n_entries
    line["gpu_launches"] = int(launches)
    if ours:
        last = per_step[-1]
        ph = {k: mean(p.get(k, 0.0) for p in phases) for k in phases[-1]} if phases else {}
        data_plane = mean(st.get("total_ms", 0.0) for st in per_step)
        line["take_phases_ms"] = {k: round(v, 2) for k, v in ph.items()}
        line["control_vs_data_ms"] = {"take_ms": take_ms, "engine_job_total_ms": data_plane, "control_plane_ms": take_ms - data_plane,
                                      "collectives_per_take": coll_per_take}
        line["engine_step"] = {k: last.get(k) for k in ("plan_ms", "kernel_ms", "kernel_bulk_ms", "kernel_lsu_ms", "copy_ms", "device_done_ms", "total_ms", "n_files", "n_members",
                                                           "n_tiles_bulk", "n_tiles_lsu", "bytes_bulk", "bytes_lsu", "n_kernel_launches", "arena_bytes", "n_memcpy")}
        peaks, peaks_src = measured_peaks()
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        lsu_ms = mean(st.get("kernel_lsu_ms", 0.0) for st in per_step)
        lsu_bytes = 2.0 * float(last.get("bytes_lsu", 0))
        bulk_ms = mean(st.get("kernel_bulk_ms", 0.0) for st in per_step)
        bulk_bytes = 2.0 * float(last.get("bytes_bulk", 0))
        line["roofline"] = {"bound": "hbm", "kernel": "tsnap_lsu_copy_kernel (unaligned slab members) + tsnap_bulk_copy_kernel", "unit": "GB/s", "peak": hbm_peak,
                            "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks_src})",
                            "achieved": (lsu_bytes + bulk_bytes) / 1e9 / ((lsu_ms + bulk_ms) / 1e3) if lsu_ms + bulk_ms > 0 else None,
                            "frac": ((lsu_bytes + bulk_bytes) / 1e9 / ((lsu_ms + bulk_ms) / 1e3)) / hbm_peak if lsu_ms + bulk_ms > 0 else None,
                            "lsu": {"ms": lsu_ms, "algorithmic_bytes": lsu_bytes, "gbs": lsu_bytes / 1e9 / (lsu_ms / 1e3) if lsu_ms else None},
                            "bulk": {"ms": bulk_ms, "algorithmic_bytes": bulk_bytes, "gbs": bulk_bytes / 1e9 / (bulk_ms / 1e3) if bulk_ms else None},
                            "traffic": None,
                            "note": "per-rank launches move ~payload/world bytes: a few MB per kernel at N=8, far below the size where HBM bandwidth (not launch latency) bounds a kernel"}
    else:
        line["cpu_baseline"] = {"value": line["value"], "unit": "GB/s", "kind": "reference", "cores": reference_threads(), "host_cores_available": os.cpu_count(), "sample": "whole workload, every rank"}
    if rank == 0:
        emit(line)


# ---- C4: async_take under a DDP training loop -----------------------------------------------------------------
def run_c4(ctx: Ctx, T, impl_desc: str) -> None:
    from torch.nn.parallel import DistributedDataParallel as DDP

    a, rank, world, device = ctx.args, ctx.rank, ctx.world, ctx.device
    torch.manual_seed(0)
    model = (W.GPT2Medium(vocab=1000, d=64, layers=2, ctx=512) if a.cpu_dryrun else W.GPT2Medium()).to(device)
    nccl = dist.is_initialized() and dist.get_backend() == "nccl" and world > 1
    ddp = DDP(model, device_ids=[ctx.local_rank]) if nccl else model
    opt = torch.optim.AdamW(ddp.parameters(), lr=1e-4)
    ctxlen, batch = 512, 4

    def step():
        x = torch.randint(0, model.vocab, (batch, ctxlen), device=device)
        with torch.autocast(device.type, dtype=torch.bfloat16):
            loss = torch.nn.functional.cross_entropy(ddp(x).float().view(-1, model.vocab), x.view(-1))
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)

    def timed_steps(n):
        _sync(device)
        t0 = time.perf_counter()
        for _ in range(n):
            step()
        _sync(device)
        return (time.perf_counter() - t0) / n * 1e3

    for _ in range(3):
        step()
    app = {"model": ddp, "optim": opt}
    kw = {"replicated": ["**"]} if world > 1 else {}
    nparams = sum(p.numel() for p in model.parameters())
    payload = nparams * 4 * 3
    for w in range(max(1, min(a.warmup, 2))):
        T.Snapshot.take(ctx.path(f"warm{w}"), app, **kw)
        ctx.cleanup(f"warm{w}")
    base_ms = ctx.max(timed_steps(10))
    res = []
    # fixed number of steps on every rank while the snapshot drains (DDP collectives must stay in lock step)
    during = a.c4_steps_during
    for k in range(a.steps):
        ctx.barrier()
        _sync(device)
        t0 = time.perf_counter()
        pending = T.Snapshot.async_take(ctx.path(f"s{k}"), app, **kw)
        t1 = time.perf_counter()
        for _ in range(during):
            step()
        _sync(device)
        t2 = time.perf_counter()
        still = not pending.done()
        pending.wait()
        t3 = time.perf_counter()
        res.append({"blocked_ms": ctx.max((t1 - t0) * 1e3), "steps_ms_total": ctx.max((t2 - t1) * 1e3), "wait_after_steps_ms": ctx.max((t3 - t2) * 1e3),
                    "still_draining_after_steps": ctx.max(float(still))})
        if k + 1 == a.steps:
            dump_outputs(ctx, ctx.path(f"s{k}"))
        ctx.cleanup(f"s{k}")
    # a synchronous take for comparison: the loop is blocked for all of it
    sync_ms, _ = ctx.timed(lambda: T.Snapshot.take(ctx.path("sync"), app, **kw))
    ctx.cleanup("sync")
    blocked = mean(r["blocked_ms"] for r in res)
    extra = mean(max(0.0, r["steps_ms_total"] - during * base_ms) for r in res)
    drain = mean(r["steps_ms_total"] + r["wait_after_steps_ms"] for r in res)
    # overlap: share of the snapshot's background time during which training made progress at full speed
    overlap = 1.0 - extra / drain if drain > 0 else None
    config = {"workload": "C4: GPT-2-medium (354.8 M fp32 params + AdamW = 4.26 GB of state) DDP training loop, bf16 autocast, batch 4 x 512 tokens per rank; async_take between steps, replicated=['**']",
              "world_size": world, "payload_bytes_total": int(payload), "steps_during_drain": during, "target_fs": a.target_fs, "_dtype": "fp32 state (byte copy); bf16 autocast training",
              "l2": "state (4.26 GB) exceeds the 126 MB L2"}
    line = common_line(ctx, impl_desc, "async_take_blocking_ms", blocked, "ms", blocked, config, higher=False, scaling="strong")
    line["e2e"] = {"value": blocked, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": int(payload // max(1, world)),
                   "definition": "time inside Snapshot.async_take() with the training loop stopped, max over ranks; the D2H of this rank's partition happens before it returns (reference) or right after it, from the HBM staging copy (engine)"}
    line["train_step_ms"] = base_ms
    line["step_ms_during_drain"] = mean(r["steps_ms_total"] for r in res) / during
    line["overlap_pct"] = round(100 * overlap, 1) if overlap is not None else None
    line["training_time_lost_per_snapshot_ms"] = blocked + extra  # blocked inside async_take + slow-down of the steps that overlap the drain
    line["overlap_definition"] = "1 - (extra time the training steps took while the snapshot drained) / (time from async_take returning until the snapshot was complete)"
    line["background_ms"] = drain
    line["sync_take_ms"] = sync_ms
    line["async_take"] = [{k: round(v, 2) for k, v in r.items()} for r in res]
    line["gpu_launches"] = None
    if a.impl == "ours":
        eng = _engine(T, device)
        line["gpu_launches"] = int(eng.stats()["kernels_launched"])
    else:
        line["cpu_baseline"] = {"value": blocked, "unit": "ms", "kind": "reference", "cores": reference_threads(), "host_cores_available": os.cpu_count(), "sample": "whole workload"}
    if rank == 0:
        emit(line)


# ---- C5: reshard-on-load -------------------------------------------------------------------------------------------
def run_c5(ctx: Ctx, T, impl_desc: str) -> None:
    a, rank, world, device = ctx.args, ctx.rank, ctx.world, ctx.device
    rows, cols = a.c5_rows, W.C5_COLS
    split = -(-rows // world)
    lo = min(rank * split, rows)
    n = max(0, min(split, rows - lo))
    t = torch.empty(n, cols, device=device)
    for b in range(0, n, 1 << 20):
        t[b:b + (1 << 20)] = W.c5_content(lo + b, min(1 << 20, n - b), cols, device)
    app = {"emb": T.StateDict(table=W.c5_sharded(t, lo, rows, cols, rank, device))}
    payload = rows * cols * 4
    for w in range(max(1, min(a.warmup, 2))):
        T.Snapshot.take(ctx.path(f"warm{w}"), app)
        ctx.cleanup(f"warm{w}")
    save_ms = []
    for k in range(a.steps):
        ms, _ = ctx.timed(lambda: T.Snapshot.take(ctx.path(f"snap{k}"), app))
        save_ms.append(ms)
        if k + 1 < a.steps:
            ctx.cleanup(f"snap{k}")
    keep = f"snap{a.steps - 1}"
    del t, app
    torch.cuda.empty_cache()
    # restore at half the world size on a sub-group; the other ranks idle
    half = max(1, world // 2)
    sub = dist.new_group(list(range(half))) if world > 1 else None
    restore_ms, ok, restored = [], True, {}
    if rank < half:
        split2 = -(-rows // half)
        lo2 = min(rank * split2, rows)
        n2 = max(0, min(split2, rows - lo2))
        t2 = torch.zeros(n2, cols, device=device)
        app2 = {"emb": T.StateDict(table=W.c5_sharded(t2, lo2, rows, cols, rank, device, process_group=sub))}
        snap = T.Snapshot(ctx.path(keep), pg=sub) if sub is not None else T.Snapshot(ctx.path(keep))
        for rep in range(1 + a.steps):  # one untimed warm-up restore, then --steps timed ones
            t2.zero_()
            if sub is not None:
                dist.barrier(group=sub, device_ids=[device.index]) if dist.get_backend() == "nccl" else dist.barrier(group=sub)
            _sync(device)
            t0 = time.perf_counter()
            snap.restore(app2)
            _sync(device)
            dt = (time.perf_counter() - t0) * 1e3
            if rep:
                restore_ms.append(dt)
        for b in range(0, n2, 1 << 20):
            m = min(1 << 20, n2 - b)
            ok = ok and bool(torch.equal(t2[b:b + m], W.c5_content(lo2 + b, m, cols, device)))
        restored = {f"restored.{rank}.emb.table": t2}
    r_ms = ctx.max(mean(restore_ms) if restore_ms else 0.0)
    ok = bool(ctx.min(1.0 if ok else 0.0))
    dump_outputs(ctx, ctx.path(keep), restored)
    ctx.cleanup(keep)
    s_ms = mean(save_ms)
    config = {"workload": f"C5: row-wise ShardedTensor {rows} x {cols} fp32 ({payload / 1e9:.1f} GB) saved at world_size {world}, restored at world_size {half} (reshard-on-load)",
              "world_size": world, "restore_world_size": half, "payload_bytes_total": int(payload), "target_fs": a.target_fs, "_dtype": "fp32 (byte copy)",
              "l2": "per-rank shards (>= 2 GB) exceed the 126 MB L2"}
    line = common_line(ctx, impl_desc, "reshard_restore_GBps", payload / 1e9 / (r_ms / 1e3), "GB/s", r_ms, config)
    line["e2e"] = {"value": line["value"], "unit": "GB/s", "ms_per_step": r_ms, "timed_restores": len(restore_ms), "h2d_bytes_per_step": int(payload // half), "d2h_bytes_per_step": 0,
                   "definition": "Snapshot.restore wall clock on the restoring ranks (file reads, host->device copies, scatter into the 2x larger local shard), max over ranks"}
    line["save"] = {"value": payload / 1e9 / (s_ms / 1e3), "unit": "GB/s", "ms": s_ms}
    line["verified_every_element_on_restoring_ranks"] = ok
    if a.impl == "ours":
        line["gpu_launches"] = int(_engine(T, device).stats()["kernels_launched"])
    else:
        line["cpu_baseline"] = {"value": line["value"], "unit": "GB/s", "kind": "reference", "cores": reference_threads(), "host_cores_available": os.cpu_count(), "sample": "whole workload"}
    if rank == 0:
        emit(line)


# ---- C1: single-process 1 GiB fp32 nn.Linear on the CPU (the reference's own CPU-runnable case, no GPU involved) ----
def run_c1(ctx: Ctx, T, impl_desc: str) -> None:
    a = ctx.args
    torch.manual_seed(0)
    n = 1024 if a.cpu_dryrun else 16384
    model = torch.nn.Linear(n, n)
    app = {"model": model}
    payload = sum(t.numel() * t.element_size() for t in model.state_dict().values())
    for w in range(a.warmup):
        T.Snapshot.take(ctx.path(f"warm{w}"), app)
        ctx.cleanup(f"warm{w}")
    take_ms, cpu = [], CpuMeter()
    for k in range(a.steps):
        cpu.start()
        t0 = time.perf_counter()
        T.Snapshot.take(ctx.path(f"step{k}"), app)
        take_ms.append((time.perf_counter() - t0) * 1e3)
        cpu.stop()
        if k + 1 < a.steps:
            ctx.cleanup(f"step{k}")
    keep = f"step{a.steps - 1}"
    want = {k: v.clone() for k, v in model.state_dict().items()}
    restore_ms = []
    for _ in range(min(a.steps, 3)):
        with torch.no_grad():
            for v in model.state_dict().values():
                v.zero_()
        t0 = time.perf_counter()
        T.Snapshot(ctx.path(keep)).restore(app)
        restore_ms.append((time.perf_counter() - t0) * 1e3)
    ok = all(torch.equal(want[k], v) for k, v in model.state_dict().items())
    dump_outputs(ctx, ctx.path(keep))
    ctx.cleanup(keep)
    ms = mean(take_ms)
    config = {"workload": f"C1: single-process Snapshot.take of a 1 GiB fp32 nn.Linear({n},{n}) state_dict held on the CPU to local fs (no GPU on the path)",
              "world_size": 1, "payload_bytes_total": int(payload), "target_fs": a.target_fs, "_dtype": "fp32 (byte copy)", "semantics": "returned (no fsync)",
              "l2": "n/a (host path)"}
    line = common_line(ctx, impl_desc, "checkpoint_save_GBps", payload / 1e9 / (ms / 1e3), "GB/s", ms, config)
    line["n_gpus"] = 0
    line["e2e"] = {"value": line["value"], "unit": "GB/s", "ms_per_step": ms, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "definition": "Snapshot.take wall clock; host tensors, host engine"}
    line["steps_ms"] = [round(x, 1) for x in take_ms]
    line["restore"] = {"value": payload / 1e9 / (mean(restore_ms) / 1e3), "unit": "GB/s", "ms": mean(restore_ms), "timed_restores": len(restore_ms), "verified": ok}
    line["host_cpu_during_take"] = cpu.report()
    line["gpu_launches"] = 0
    if a.impl == "reference":
        line["cpu_baseline"] = {"value": line["value"], "unit": "GB/s", "kind": "reference", "cores": cpu.report()["cores_busy_avg"], "host_cores_available": os.cpu_count(), "sample": "whole workload"}
    emit(line)


RUNNERS = {"c1": run_c1, "c2": run_c2, "c3": run_c3, "c4": run_c4, "c5": run_c5}


def fs_kind(path: str) -> str:
    try:
        best, kind = "", "?"
        with open("/proc/mounts") as f:
            for ln in f:
                dev, mnt, typ = ln.split()[:3]
                if path.startswith(mnt) and len(mnt) > len(best):
                    best, kind = mnt, f"{typ} ({dev}) at {mnt}"
        return kind
    except OSError:
        return "?"


def main() -> None:
    global _REAL_STDOUT
    if os.environ.get("BENCH_DUMP_AFTER"):  # debugging aid for hangs: dump every thread's stack after N seconds
        import faulthandler

        faulthandler.dump_traceback_later(float(os.environ["BENCH_DUMP_AFTER"]), exit=True)
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # NCCL prints its version banner on fd 1
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=sorted(RUNNERS), default="c3")
    ap.add_argument("--layout", choices=["sharded", "dtensor", "plain"], default="sharded")
    ap.add_argument("--dir", default=None, help="target directory (default: $TSNAP_BENCH_DIR or a temp dir under /tmp)")
    ap.add_argument("--ref-sample-gib", type=int, default=4, help="bounded sample for the cpu_baseline leg of the engine arm")
    ap.add_argument("--ncu-traffic-bytes", type=float, default=None)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--trace-dir", default=None, help="write the per-chunk timeline of one extra take/restore here")
    ap.add_argument("--trace-tag", default="c3")
    ap.add_argument("--c4-steps-during", type=int, default=8)
    ap.add_argument("--c5-rows", type=int, default=W.C5_ROWS)
    ap.add_argument("--cpu-dryrun", action="store_true", help="developer aid: run the code paths on CPU tensors with shrunken shapes (no GPU box needed); never a measurement")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write the tensors the last timed step computed as DIR/<name>.npy (<= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.cpu_dryrun and args.c5_rows == W.C5_ROWS:
        args.c5_rows = 100_000

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.cpu_dryrun or args.config == "c1":
        device = torch.device("cpu")
    elif not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback for device tensors")
    else:
        device = torch.device("cuda", local_rank)
        torch.cuda.set_device(device)
    T, impl_desc = load_impl(args.impl)
    if T is None:
        if rank == 0:
            emit({"impl": "reference", "unavailable": impl_desc})
        return
    store_file = None
    if world > 1:
        if args.cpu_dryrun:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=device)
    else:
        store_file = tempfile.NamedTemporaryFile(delete=False)
        dist.init_process_group("gloo", init_method=f"file://{store_file.name}", rank=0, world_size=1)
    base = args.dir or os.environ.get("TSNAP_BENCH_DIR")
    made = False
    if base is None:
        box = [tempfile.mkdtemp(prefix="tsnap_bench_", dir="/tmp") if rank == 0 else None]
        if world > 1:
            dist.broadcast_object_list(box, src=0)
        base = box[0]
        made = True
    os.makedirs(base, exist_ok=True)
    args.target_fs = fs_kind(os.path.abspath(base))
    ctx = Ctx(args, rank, world, local_rank, device, base)
    try:
        RUNNERS[args.config](ctx, T, impl_desc)
    finally:
        if dist.is_initialized():
            try:
                ctx.barrier()
            except Exception:
                pass
        if rank == 0 and made:
            shutil.rmtree(base, ignore_errors=True)
        if dist.is_initialized():
            dist.destroy_process_group()
        if store_file is not None:
            try:
                os.unlink(store_file.name)
            except OSError:
                pass


if __name__ == "__main__":
    main()
