"""Round-2 GPU tests: parity at BASELINE scale against the oracle and against snapshots of the UNMODIFIED reference
(tests/golden/, oracle/gen_golden.py), the engine underneath the unmodified reference with CUDA tensors (install() +
cross-restore both ways), arena-less / bounded-arena / nearly-full-HBM operation, O_DIRECT file I/O, restore ordering
against the caller's stream, timeline + probes."""
import gzip
import hashlib
import json
import os
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist

pytestmark = pytest.mark.gpu

import torchsnapshot_b200 as B  # noqa: E402
from benchmarks import workloads as W  # noqa: E402
from oracle import ref_port as R  # noqa: E402
from tests.util import canonicalize, det_tensor, snapshot_digest, wire_bytes  # noqa: E402
from torchsnapshot_b200 import _native as N  # noqa: E402
from torchsnapshot_b200.flatten import flatten  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden")
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pg():
    if not dist.is_initialized():
        f = tempfile.NamedTemporaryFile(delete=False)
        dist.init_process_group("gloo", init_method=f"file://{f.name}", rank=0, world_size=1)
    yield
    if dist.is_initialized():
        dist.destroy_process_group()


@pytest.fixture()
def fresh_engines():
    """Tests that configure the engine through the environment get their own engine and leave none behind."""
    saved = {k: os.environ.get(k) for k in ("TSNAP_B200_ENGINE_FLAGS", "TSNAP_B200_HBM_STAGING_BYTES", "TSNAP_B200_ENGINE_ARENA", "TSNAP_B200_PINNED_SLOTS", "TSNAP_B200_PINNED_SLOT_BYTES")}
    N.reset_engines()
    yield
    N.reset_engines()
    for k, v in saved.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


@pytest.fixture()
def ref():
    if not os.path.isdir(os.path.join(REF_DIR, "torchsnapshot")):
        pytest.skip("oracle/_ref not staged (oracle/make_ref.sh needs a checkout of the reference)")
    sys.path.insert(0, REF_DIR)
    try:
        import torchsnapshot
    finally:
        sys.path.remove(REF_DIR)
    yield torchsnapshot
    B.uninstall()


def _sha_files(root):
    out = {}
    for dp, _, fs in os.walk(root):
        for f in fs:
            if f == ".snapshot_metadata":
                continue
            h = hashlib.sha256()
            with open(os.path.join(dp, f), "rb") as fh:
                while True:
                    b = fh.read(1 << 24)
                    if not b:
                        break
                    h.update(b)
            out[os.path.relpath(os.path.join(dp, f), root)] = (os.path.getsize(os.path.join(dp, f)), h.hexdigest())
    return out


def _assert_snapshot_equals_oracle(snap_dir, entries, files, prefix="0/"):
    """manifest == oracle plan, sha256(file) == sha256(oracle image) for every payload file (slab names canonicalised)."""
    meta = json.load(open(os.path.join(snap_dir, ".snapshot_metadata")))["manifest"]
    got_manifest, got_names = canonicalize(meta)  # slab files: batched/<uuid4> -> batched/<k> by first appearance
    want_manifest, want_names = canonicalize({f"{prefix}{k}": v for k, v in entries.items()})
    for path, e in want_manifest.items():
        assert got_manifest[path] == e, path
    on_disk = {got_names.get(p, p): v for p, v in _sha_files(snap_dir).items()}
    for loc, blob in files.items():
        assert on_disk[want_names.get(loc, loc)] == (len(blob), hashlib.sha256(blob).hexdigest()), loc


# ---- parity at BASELINE scale --------------------------------------------------------------------------------------
def test_c3_rank_shard_matches_oracle_at_full_size(tmp_path, pg):
    """One rank of C3 at world_size 8 (2.0 GB, 291 ShardedTensors -> 16 GPU slabs): every payload file's sha256 equals
    the oracle's image (serialize_view of each piece at its byte_range), manifest == oracle plan."""
    world, rank = 8, 3
    local = W.build_llama_local(rank, world, torch.device(DEV))
    # the ShardedTensor API validates that the shards of all ranks tile the global tensor; the saved bytes only depend on
    # the local shard, so this rank's 2 GB shard is saved as the only shard of a 1-rank job (offsets 0: they only name files)
    from torch.distributed._shard.sharded_tensor import Shard, ShardedTensor, ShardMetadata

    state, flat = {}, {}
    for name, (t, shape, lo) in local.items():
        off = [0] * len(shape)
        md = ShardMetadata(shard_offsets=off, shard_sizes=list(t.shape), placement=f"rank:0/{DEV}")
        state[name] = ShardedTensor._init_from_local_shards([Shard(tensor=t, metadata=md)], tuple(t.shape))
        flat[f"model/{name}"] = R.ShardedSpec([(t, off, list(t.shape))], dim=0)
    payload = sum(t.numel() * 2 for t, _, _ in local.values())
    assert payload > 2_000_000_000
    k0 = B.get_engine(0).stats()["kernels_launched"]
    B.Snapshot.take(str(tmp_path / "s"), {"model": B.StateDict(**state)})
    assert B.get_engine(0).stats()["kernels_launched"] > k0
    entries, files = R.plan_save(flat)
    assert sum(len(b) for b in files.values()) == payload
    _assert_snapshot_equals_oracle(str(tmp_path / "s"), entries, files)


def _device_job_stats():
    """Stats of the engine job that touched the GPU (a mixed CPU/GPU state also has a host-only job for the CPU tensors)."""
    from torchsnapshot_b200 import scheduler as S

    jobs = S.LAST_STATS.get("save") or [{}]
    return max(jobs, key=lambda j: (j.get("n_kernel_launches", 0), j.get("direct_bytes", 0), j.get("payload_bytes", 0)))


def _c2_flat(app_state):
    flat = {}
    for key in ("model", "optim"):
        _, f = flatten(app_state[key].state_dict(), prefix=key)
        flat.update({k: v for k, v in f.items() if isinstance(v, torch.Tensor)})
    return flat


def test_c2_layout_matches_oracle(tmp_path, pg):
    """C2 (ResNet-50 state_dict + Adam with CPU `step` scalars, ~800 tensors, 0-d int64 members, unpadded slabs):
    manifest and every slab image equal the oracle's.  This is the layout that runs the LSU kernel and the CPU-slab chain."""
    app_state, kw, payload = W.build_c2(B, 0, 1, torch.device(DEV), 0)
    k0 = B.get_engine(0).stats()["kernels_launched"]
    B.Snapshot.take(str(tmp_path / "s"), app_state)  # per-rank state: request order == state_dict order (oracle models this)
    st = _device_job_stats()
    flat = _c2_flat(app_state)
    entries, files = R.plan_save(flat)
    assert sum(len(b) for b in files.values()) == payload
    _assert_snapshot_equals_oracle(str(tmp_path / "s"), entries, files)
    assert sum(1 for v in flat.values() if v.is_cuda) > 600 and B.get_engine(0).stats()["kernels_launched"] > k0
    assert st["n_tiles_lsu"] > 0, "unpadded slab members must exercise the LSU kernel"


def test_c2_replicated_equals_unmodified_reference_on_cuda(tmp_path, pg):
    """replicated=['**'] sends every request through the partitioner (which reorders them, T:partitioner.py:194-211)
    before the batcher: compare with the UNMODIFIED reference run on the same CUDA app_state (its snapshot's digest,
    tests/golden/c2_replicated_cuda.json.gz) — manifests and every payload file must be identical."""
    app_state, kw, payload = W.build_c2(B, 0, 1, torch.device(DEV), 0)
    B.Snapshot.take(str(tmp_path / "ours"), app_state, **kw)
    d_ours = snapshot_digest(str(tmp_path / "ours"))
    with gzip.open(os.path.join(GOLDEN, "c2_replicated_cuda.json.gz"), "rt") as f:
        d_ref = json.load(f)
    assert d_ours["manifest"] == d_ref["manifest"]
    assert d_ours["files"] == d_ref["files"]
    assert sum(f["nbytes"] for f in d_ours["files"].values() if "nbytes" in f) == payload


# ---- the engine underneath the unmodified reference, CUDA tensors --------------------------------------------------
MIXED_KNOBS = {"slab": 1 << 16, "max_chunk": 1 << 20}


def _mixed_cuda_state():
    return {
        # (an even element count: the reference truncates bf16 tensors with an odd count, DESIGN.md "divergences")
        "w": det_tensor((514, 257), torch.bfloat16, 1).to(DEV),
        "w_t": det_tensor((300, 200), torch.float32, 2).to(DEV).t(),
        "cols": det_tensor((128, 96), torch.float32, 3).to(DEV)[:, 7:50],
        "i": det_tensor((1001,), torch.int64, 4).to(DEV),
        "flag": det_tensor((3,), torch.bool, 5).to(DEV),
        "big": det_tensor((1 << 20,), torch.float32, 6).to(DEV),
        "step": torch.tensor(3.0),
    }


def test_install_under_unmodified_reference_with_cuda_tensors(ref, tmp_path, pg):
    """reference Snapshot.take/restore with the engine installed == reference alone == this package's Snapshot,
    byte for byte, and snapshots restore across implementations in both directions."""
    from tests.cases import apply_knobs

    state = _mixed_cuda_state()
    with apply_knobs(MIXED_KNOBS):
        # 1. the reference alone (its own pageable tensor.to('cpu') path)
        ref.Snapshot.take(str(tmp_path / "ref"), {"m": ref.StateDict(**state)})
        # 2. the reference with the engine installed underneath
        eng = B.get_engine(0)
        k0, w0 = eng.stats()["kernels_launched"], eng.stats()["bytes_written"]
        B.install(ref)
        ref.Snapshot.take(str(tmp_path / "inst"), {"m": ref.StateDict(**state)})
        assert eng.stats()["kernels_launched"] > k0 and eng.stats()["bytes_written"] > w0, "the engine was not on the path"
        # restore through the installed engine
        tgt = ref.StateDict(**{k: torch.zeros_like(v) for k, v in state.items()})
        r0 = eng.stats()["bytes_read"]
        ref.Snapshot(str(tmp_path / "inst")).restore({"m": tgt})
        assert eng.stats()["bytes_read"] > r0
        for k, v in state.items():
            assert wire_bytes(v) == wire_bytes(tgt[k]), k
        B.uninstall()
        # 3. this package's own Snapshot
        B.Snapshot.take(str(tmp_path / "ours"), {"m": B.StateDict(**state)})
        d_ref, d_inst, d_ours = (snapshot_digest(str(tmp_path / n)) for n in ("ref", "inst", "ours"))
        assert d_ref["manifest"] == d_inst["manifest"] == d_ours["manifest"]
        assert d_ref["files"] == d_inst["files"] == d_ours["files"]
        # cross-restore: reference reader <- engine-written snapshot, engine reader <- reference-written snapshot
        t1 = ref.StateDict(**{k: torch.zeros_like(v) for k, v in state.items()})
        ref.Snapshot(str(tmp_path / "ours")).restore({"m": t1})
        t2 = B.StateDict(**{k: torch.zeros_like(v) for k, v in state.items()})
        B.Snapshot(str(tmp_path / "ref")).restore({"m": t2})
        for k, v in state.items():
            assert wire_bytes(v) == wire_bytes(t1[k]) == wire_bytes(t2[k]), k


def test_mixed_cuda_state_equals_unmodified_reference_snapshot(tmp_path, pg):
    """This package's snapshot of the mixed CUDA state == the UNMODIFIED reference's snapshot of it (digest stored in
    tests/golden/mixed_cuda.json), and it restores bit for bit."""
    from tests.cases import apply_knobs

    state = _mixed_cuda_state()
    with open(os.path.join(GOLDEN, "mixed_cuda.json")) as f:
        d_ref = json.load(f)
    assert d_ref["knobs"] == MIXED_KNOBS
    with apply_knobs(MIXED_KNOBS):
        snap = B.Snapshot.take(str(tmp_path / "ours"), {"m": B.StateDict(**state)})
        d_ours = snapshot_digest(str(tmp_path / "ours"))
        assert d_ours["manifest"] == d_ref["manifest"]
        assert d_ours["files"] == d_ref["files"]
        tgt = B.StateDict(**{k: torch.zeros_like(v) for k, v in state.items()})
        snap.restore({"m": tgt})
    for k, v in state.items():
        assert wire_bytes(v) == wire_bytes(tgt[k]), k


# ---- HBM staging: arena-less, bounded, engine-owned, nearly full device ----------------------------------------------
def _save_and_check(tmp_path, tag, state, expect=None):
    snap = B.Snapshot.take(str(tmp_path / tag), {"m": B.StateDict(**state)})
    st = _device_job_stats()
    flat = {k: v for k, v in flatten(state, "m")[1].items() if isinstance(v, torch.Tensor)}
    slab = int(os.environ.get("TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE", R.DEFAULT_SLAB_THRESHOLD))
    entries, files = R.plan_save(flat, slab_threshold=slab)
    _assert_snapshot_equals_oracle(str(tmp_path / tag), entries, files)
    tgt = B.StateDict(**{k: torch.zeros_like(v) for k, v in state.items()})
    snap.restore({"m": tgt})
    for k, v in state.items():
        assert wire_bytes(v) == wire_bytes(tgt[k]), k
    if expect:
        expect(st)
    return st


def test_arena_less_mode_drains_dense_members_from_live_tensors(tmp_path, fresh_engines):
    os.environ["TSNAP_B200_ENGINE_FLAGS"] = str(N.ENGINE_NO_ARENA)
    dense = {f"d{i}": det_tensor((1 << 18,), torch.float32, i).to(DEV) for i in range(6)}
    dense["odd"] = det_tensor((333,), torch.uint8, 9).to(DEV)  # shifts every later slab member off 16 B alignment
    dense["tail"] = det_tensor((100_003,), torch.int16, 10).to(DEV)

    def all_direct(st):
        assert st["arena_bytes"] == 0 and st["direct_bytes"] == st["payload_bytes"] and st["n_kernel_launches"] == 0

    _save_and_check(tmp_path, "dense", dense, all_direct)
    # strided members cannot be drained without staging: they get a (small) arena of their own, the rest stays direct
    mixed = dict(dense)
    mixed["cols"] = det_tensor((4096, 512), torch.float32, 11).to(DEV)[:, 64:320]  # 4 MiB strided -> its own file

    def partly(st):
        assert 0 < st["arena_bytes"] and st["direct_bytes"] > 0 and st["n_kernel_launches"] >= 1

    os.environ["TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE"] = str(1 << 20)
    try:
        _save_and_check(tmp_path, "mixed", mixed, partly)
    finally:
        del os.environ["TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE"]


def test_bounded_arena_multi_wave_through_the_api(tmp_path, fresh_engines):
    os.environ["TSNAP_B200_HBM_STAGING_BYTES"] = str(64 << 20)
    state = {f"p{i}": det_tensor((6 << 20,), torch.float32, i).to(DEV) for i in range(12)}  # 12 x 24 MiB

    def waves(st):
        assert st["arena_bytes"] <= (64 << 20) and st["n_waves"] >= 4 and st["direct_bytes"] == 0

    os.environ["TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE"] = str(1 << 20)
    try:
        _save_and_check(tmp_path, "s", state, waves)
    finally:
        del os.environ["TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE"]


def test_engine_owned_arena_for_c_callers(tmp_path, fresh_engines):
    os.environ["TSNAP_B200_ENGINE_ARENA"] = "1"
    state = {f"p{i}": det_tensor((1 << 20,), torch.float32, i).to(DEV) for i in range(5)}
    _save_and_check(tmp_path, "s", state, lambda st: st["arena_bytes"] > 0)
    import time

    eng = B.get_engine(0)
    deadline = time.time() + 5
    while eng.stats()["hbm_arena_bytes"] and time.time() < deadline:
        time.sleep(0.05)
    assert eng.stats()["hbm_arena_bytes"] == 0, "an idle engine must give its own arena back"


def test_take_with_nearly_full_hbm_still_bit_exact(tmp_path, fresh_engines):
    """The reference degrades to a CPU slab when its GPU slab allocation OOMs (T:batcher.py:144-152); the engine
    degrades to draining straight from the live tensors.  Fill the device to within ~1 GiB and save 1.5 GiB."""
    state = {f"p{i}": det_tensor((32 << 20,), torch.float32, i).to(DEV) for i in range(12)}  # 12 x 128 MiB = 1.5 GiB
    state["cols"] = det_tensor((2048, 512), torch.float32, 77).to(DEV)[:, 3:300]
    torch.cuda.empty_cache()
    free_b, _ = torch.cuda.mem_get_info(0)
    hog = torch.empty(max(0, free_b - (1 << 30)), dtype=torch.uint8, device=DEV)
    try:
        def degraded(st):
            assert st["direct_bytes"] >= 12 * (128 << 20), st
            assert st["arena_bytes"] < (1 << 30)

        _save_and_check(tmp_path, "s", state, degraded)
    finally:
        del hog
        torch.cuda.empty_cache()


# ---- O_DIRECT ---------------------------------------------------------------------------------------------------------
def test_odirect_files_are_identical(tmp_path, fresh_engines):
    os.environ["TSNAP_B200_ENGINE_FLAGS"] = str(N.ENGINE_ODIRECT)
    os.environ["TSNAP_B200_PINNED_SLOT_BYTES"] = str(1 << 20)
    state = {
        "a": det_tensor((3 * (1 << 20) + 4097,), torch.uint8, 1).to(DEV),  # ragged tail, not a block multiple
        "b": det_tensor((1 << 19,), torch.float32, 2).to(DEV),
        "c": det_tensor((777,), torch.int16, 3).to(DEV),
        "d": det_tensor((100, 300), torch.float32, 4).to(DEV)[:, 5:77],
    }
    os.environ["TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE"] = str(1 << 16)
    try:
        _save_and_check(tmp_path, "s", state)
        # byte-range reads out of a slab through O_DIRECT (unaligned offsets are widened to blocks)
        snap = B.Snapshot(str(tmp_path / "s"))
        out = torch.zeros(777, dtype=torch.int16, device=DEV)
        snap.read_object("0/m/c", obj_out=out)
        assert wire_bytes(out) == wire_bytes(state["c"])
    finally:
        del os.environ["TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE"]


# ---- ordering of a restore against the caller's stream -------------------------------------------------------------
def test_restore_is_ordered_after_work_queued_on_the_callers_stream(tmp_path):
    """Work already queued on the current stream that writes the destination (an init kernel, an optimizer step) must
    not land after the restored bytes — the reference's dst.copy_() runs on that stream (T:io_preparers/tensor.py:358-360)."""
    n = 64 << 20
    src = torch.arange(n, dtype=torch.float32, device=DEV)
    snap = B.Snapshot.take(str(tmp_path / "s"), {"m": B.StateDict(x=src)})
    dst = torch.zeros(n, dtype=torch.float32, device=DEV)
    a = torch.randn(8192, 8192, device=DEV)
    torch.cuda.synchronize()
    for _ in range(40):  # ~hundreds of ms of queued work, then a late writer to the destination
        a = (a @ a).clamp_(-1, 1)
    dst.fill_(-1.0)
    snap.restore({"m": B.StateDict(x=dst)})
    torch.cuda.synchronize()
    assert torch.equal(dst, src)
    # the seam used under third-party storage plugins (tsnap_consume) obeys the same rule
    eng = B.get_engine(0)
    buf = bytearray(wire_bytes(src[: 1 << 20]))
    dst2 = torch.zeros(1 << 20, dtype=torch.float32, device=DEV)
    for _ in range(40):
        a = (a @ a).clamp_(-1, 1)
    dst2.fill_(-1.0)
    eng.consume(buf, [N.load_desc(dst2, 0)])
    torch.cuda.synchronize()
    assert torch.equal(dst2, src[: 1 << 20])


# ---- timeline + probes ---------------------------------------------------------------------------------------------
def test_timeline_shows_the_pipeline_overlapping(tmp_path, fresh_engines):
    from torchsnapshot_b200 import scheduler as S
    from torchsnapshot_b200 import timeline as TL

    os.environ["TSNAP_B200_ENGINE_FLAGS"] = str(N.ENGINE_TRACE)
    os.environ["TSNAP_B200_PINNED_SLOT_BYTES"] = str(8 << 20)
    state = {f"p{i}": torch.randn(16 << 20, device=DEV) for i in range(16)}  # 1 GiB
    B.Snapshot.take(str(tmp_path / "w"), {"m": B.StateDict(**state)})
    snap = B.Snapshot.take(str(tmp_path / "s"), {"m": B.StateDict(**state)})
    tr = S.LAST_STATS["save_trace"][0]
    kinds = {r["kind"] for r in tr}
    assert {"plan", "kernel", "d2h", "pwrite"} <= kinds
    assert sum(r["bytes"] for r in tr if r["kind"] == "d2h") == sum(r["bytes"] for r in tr if r["kind"] == "pwrite") == 1 << 30
    s = TL.summarize(tr)
    assert s["overlap"]["d2h&pwrite"]["both_busy_ms"] > 0, s  # writes run while later chunks are still crossing the link
    json.loads(TL.to_chrome_trace(tr))
    snap.restore({"m": B.StateDict(**{k: torch.zeros_like(v) for k, v in state.items()})})
    lt = S.LAST_STATS["load_trace"][0]
    assert {"pread", "h2d", "kernel"} <= {r["kind"] for r in lt}
    eng = B.get_engine(0)
    assert eng.probe(N.PROBE_D2H, 1 << 30) > 5 and eng.probe(N.PROBE_H2D, 1 << 30) > 5
    d = str(tmp_path / "probe")
    os.makedirs(d)
    assert eng.probe(N.PROBE_WRITE, 1 << 29, d) > 0.1 and eng.probe(N.PROBE_READ, 1 << 29, d) > 0.1


# ---- cast / quantize fused into the pack kernel, through the public API ----------------------------------------------
def test_cast_and_quantize_on_save_on_gpu(tmp_path):
    import struct

    torch.manual_seed(1)
    w = torch.randn(2048, 1031, device=DEV)
    st = {"w": w, "wt": torch.randn(300, 200, device=DEV).t(), "h": torch.randn(4099, device=DEV).half(), "i": torch.arange(100, device=DEV)}
    # cast: payload == tensor.to(bf16) computed by torch on the same device, no processed tensor materialised
    eng = B.get_engine(0)
    k0 = eng.stats()["kernels_launched"]
    snap = B.Snapshot.take(str(tmp_path / "c"), {"m": B.StateDict(**st)}, _custom_tensor_prepare_func=B.cast_on_save(torch.bfloat16, only="m/w*"))
    assert eng.stats()["kernels_launched"] > k0
    man = snap.get_manifest()
    for k in ("w", "wt"):
        assert man[f"0/m/{k}"].dtype == "torch.bfloat16"
        assert open(tmp_path / "c" / man[f"0/m/{k}"].location, "rb").read() == wire_bytes(st[k].to(torch.bfloat16)), k
    assert man["0/m/h"].dtype == "torch.float16"
    # quantize: int_repr of torch.quantize_per_tensor on the same device + the reference's 16-byte trailer
    for qdt in (torch.qint8, torch.quint8):
        hook = B.quantize_on_save(qdt, only="m/[wh]*")
        path = tmp_path / f"q{qdt}".replace(".", "_")
        snap = B.Snapshot.take(str(path), {"m": B.StateDict(**st)}, _custom_tensor_prepare_func=hook)
        man = snap.get_manifest()
        for k in ("w", "wt", "h"):
            _, scale, zp = hook.tsnap_quant(f"m/{k}", st[k])
            q = torch.quantize_per_tensor(st[k].float().contiguous(), scale, zp, qdt)
            want = bytes(q.int_repr().cpu().numpy().tobytes()) + struct.pack("d", q.q_scale()) + struct.pack("q", q.q_zero_point())
            got = open(path / man[f"0/m/{k}"].location, "rb").read()
            assert len(got) == len(want)
            ndiff = sum(a != b for a, b in zip(got, want))
            assert ndiff == 0, (qdt, k, ndiff)
        tgt = B.StateDict(w=torch.zeros_like(w), wt=torch.zeros(200, 300, device=DEV), h=torch.zeros(4099, device=DEV).half(), i=torch.zeros(100, dtype=torch.long, device=DEV))
        snap.restore({"m": tgt})
        _, scale, _ = hook.tsnap_quant("m/w", w)
        assert (tgt["w"] - w).abs().max().item() <= scale * 0.5 + 1e-6 and torch.equal(tgt["i"], st["i"])


def test_host_memory_budget_bounds_the_ring_slots_in_flight(tmp_path, fresh_engines, monkeypatch):
    """TORCHSNAPSHOT_PER_RANK_MEMORY_BUDGET_BYTES (T:scheduler.py:47-58) is honoured by the native path: a job never
    holds more pinned slots than the budget allows, and the snapshot is still bit-exact."""
    os.environ["TSNAP_B200_PINNED_SLOT_BYTES"] = str(1 << 20)
    os.environ["TSNAP_B200_PINNED_SLOTS"] = "32"
    monkeypatch.setenv("TORCHSNAPSHOT_PER_RANK_MEMORY_BUDGET_BYTES", str(6 << 20))
    state = {f"p{i}": det_tensor((4 << 20,), torch.float32, i).to(DEV) for i in range(4)}  # 64 MiB

    def bounded(st):
        assert 1 <= st["max_slots_in_flight"] <= 6, st["max_slots_in_flight"]

    _save_and_check(tmp_path, "s", state, bounded)
    monkeypatch.delenv("TORCHSNAPSHOT_PER_RANK_MEMORY_BUDGET_BYTES")
    st = _save_and_check(tmp_path, "t", state)
    assert st["max_slots_in_flight"] > 6  # without the budget the ring is used freely
