"""N>1 path on CPU: two gloo ranks exercise replicated-state partitioning, per-rank state, sharded state,
the manifest gather/consolidation, the store-based async commit and restore at a different world size; the manifest
is compared with the one the unmodified reference wrote for the same job (tests/golden/two_rank_replicated.json)."""
import json
import os
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.util import det_tensor, snapshot_digest, wire_bytes

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _rep_state():
    rep = {f"layer{i}.weight": det_tensor((40 + i, 16), torch.float32, 10 + i) for i in range(6)}  # identical on all ranks
    rep["big"] = det_tensor((64, 64), torch.float64, 99)  # chunked at the 8 KiB override below
    return rep


def _build_state(rank: int, world: int):
    from torch.distributed._shard.sharded_tensor import Shard, ShardedTensor, ShardMetadata

    rep = _rep_state()
    own = {"counter": torch.tensor([rank], dtype=torch.int64), "noise": det_tensor((34,), torch.bfloat16, 500 + rank), "tag": f"rank{rank}"}
    rows, cols = 24, 10
    full = det_tensor((rows, cols), torch.float32, 77)
    step = rows // world
    local = full[rank * step : (rank + 1) * step].contiguous()
    st = ShardedTensor._init_from_local_shards(
        [Shard(tensor=local, metadata=ShardMetadata(shard_offsets=[rank * step, 0], shard_sizes=[step, cols], placement=f"rank:{rank}/cpu"))], (rows, cols)
    )
    return rep, own, st, full


def _worker(rank: int, world: int, store_path: str, root: str, ref_parent, mode: str):
    """ref_parent: None for this package, else the directory holding the reference's torchsnapshot package
    (oracle/gen_golden.py)."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["LOCAL_WORLD_SIZE"] = str(world)  # as torchrun sets it: ranks share the host-wide pool of I/O tokens
    os.environ["TSNAP_B200_HOST_IO_TOKENS"] = "3"  # fewer tokens than workers: the semaphore path is exercised
    os.environ["TORCHSNAPSHOT_MAX_CHUNK_SIZE_BYTES_OVERRIDE"] = "8192"
    os.environ["TORCHSNAPSHOT_SLAB_SIZE_THRESHOLD_BYTES_OVERRIDE"] = "4096"
    dist.init_process_group("gloo", init_method=f"file://{store_path}", rank=rank, world_size=world)
    if ref_parent:
        sys.path.insert(0, ref_parent)
        os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
        import torchsnapshot as M
    else:
        import torchsnapshot_b200 as M
    rep, own, st, full = _build_state(rank, world)
    app = {"rep": M.StateDict(**rep), "own": M.StateDict(**own), "emb": M.StateDict(table=st)}
    path = os.path.join(root, "snap")
    if mode == "async":
        M.Snapshot.async_take(path, app, replicated=["rep/**"]).wait()
    else:
        M.Snapshot.take(path, app, replicated=["rep/**"])
    dist.barrier()
    # restore into zeroed targets on the same world size
    rep2, own2, st2, _ = _build_state(rank, world)
    for v in list(rep2.values()) + [own2["counter"], own2["noise"]]:
        v.zero_()
    st2.local_shards()[0].tensor.zero_()
    own2["tag"] = ""
    tgt = {"rep": M.StateDict(**rep2), "own": M.StateDict(**own2), "emb": M.StateDict(table=st2)}
    M.Snapshot(path).restore(tgt)
    for k, v in rep.items():
        assert wire_bytes(v) == wire_bytes(tgt["rep"][k]), k
    assert tgt["own"]["tag"] == f"rank{rank}" and int(tgt["own"]["counter"]) == rank
    assert wire_bytes(own["noise"]) == wire_bytes(tgt["own"]["noise"])
    assert wire_bytes(st.local_shards()[0].tensor) == wire_bytes(st2.local_shards()[0].tensor)
    dist.barrier()
    dist.destroy_process_group()


def _run(world, ref_parent, mode, root):
    store = tempfile.NamedTemporaryFile(delete=False)
    mp.spawn(_worker, args=(world, store.name, root, ref_parent, mode), nprocs=world, join=True)
    if os.path.exists(store.name):
        os.unlink(store.name)


def _no_duplicate_locations(root):
    meta = json.load(open(os.path.join(root, "snap", ".snapshot_metadata")))
    seen = {}
    for path, e in meta["manifest"].items():
        if e["type"] == "Tensor":
            tes = [e]
        elif e["type"] == "ChunkedTensor":
            tes = [c["tensor"] for c in e["chunks"]]
        elif e["type"] == "ShardedTensor":
            tes = [s["tensor"] for s in e["shards"]]
        else:
            continue
        for te in tes:
            key = (te["location"], tuple(te["byte_range"] or ()))
            assert key not in seen, f"{path} and {seen[key]} share {key}"
            seen[key] = path
    return meta


@pytest.mark.parametrize("mode", ["sync", "async"])
def test_two_rank_take_restore(mode, tmp_path):
    _run(2, None, mode, str(tmp_path))
    meta = _no_duplicate_locations(str(tmp_path))
    assert meta["world_size"] == 2
    # replicated entries live under rank 0 only; the chunked one is stitched back together
    assert "0/rep/layer0.weight" in meta["manifest"] and "1/rep/layer0.weight" not in meta["manifest"]
    big = meta["manifest"]["0/rep/big"]
    assert big["type"] == "ChunkedTensor" and sum(c["sizes"][0] for c in big["chunks"]) == 64
    assert "1/own/counter" in meta["manifest"] and "0/emb/table" in meta["manifest"] and "1/emb/table" in meta["manifest"]
    # the write load was split: both ranks wrote replicated payload
    files = [os.path.relpath(os.path.join(dp, f), tmp_path / "snap") for dp, _, fs in os.walk(tmp_path / "snap") for f in fs]
    assert any(f.startswith("batched/") for f in files)

    # elasticity: a single fresh process (world size 1) restores replicated + the whole sharded table
    import torchsnapshot_b200 as B

    snap = B.Snapshot(str(tmp_path / "snap"))
    rep, full = _rep_state(), det_tensor((24, 10), torch.float32, 77)
    tgt = B.StateDict(**{k: torch.zeros_like(v) for k, v in rep.items()})
    snap.restore({"rep": tgt})
    for k, v in rep.items():
        assert wire_bytes(v) == wire_bytes(tgt[k]), k
    assert wire_bytes(snap.read_object("0/emb/table")) == wire_bytes(full)
    assert snap.read_object("1/own/tag") == "rank1"


def scrubbed_manifest(digest):
    """The manifest without what is hash-order dependent: chunk-level assignment of identical chunked tensors iterates
    a Python set (T:partitioner.py:119-124), so the rank that writes each chunk of "big" is hash-order dependent in
    BOTH implementations; compare everything except which slab those chunks, and the slab members numbered after
    them, landed in."""
    m = json.loads(json.dumps(digest["manifest"]))
    for c in m["0/rep/big"]["chunks"]:
        c["tensor"]["location"] = "*"
        c["tensor"]["byte_range"] = None
    for e in m.values():
        if e.get("type") == "Tensor" and str(e["location"]).startswith("batched/"):
            e["location"], e["byte_range"] = "*", None
    return m


def test_two_rank_manifest_equals_reference(tmp_path):
    ours = tmp_path / "ours"
    ours.mkdir()
    _run(2, None, "sync", str(ours))
    a = snapshot_digest(str(ours / "snap"))
    theirs = json.load(open(os.path.join(GOLDEN, "two_rank_replicated.json")))
    assert a["manifest"].keys() == theirs["manifest"].keys()
    sa = scrubbed_manifest(a)
    for k in sa:
        assert sa[k] == theirs["manifest"][k], k
    assert sum(v.get("nbytes", 0) for v in a["files"].values()) == theirs["payload_nbytes"]


def _subgroup_worker(rank: int, world: int, store_path: str, root: str):
    """Ranks that took a different number of async snapshots (a take on a sub-group, then one on WORLD) must still
    agree on the commit rendezvous of the WORLD take (it used to be tagged by a process-global counter)."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    dist.init_process_group("gloo", init_method=f"file://{store_path}", rank=rank, world_size=world)
    import torchsnapshot_b200 as M

    sub = dist.new_group([0, 1])
    t = det_tensor((50, 7), torch.float32, rank)
    if rank in (0, 1):
        M.Snapshot.async_take(os.path.join(root, "sub"), {"s": M.StateDict(t=t)}, pg=sub).wait()
        assert os.path.exists(os.path.join(root, "sub", ".snapshot_metadata"))
    snap = M.Snapshot.async_take(os.path.join(root, "world"), {"s": M.StateDict(t=t)}).wait()
    dist.barrier()
    out = M.StateDict(t=torch.zeros(50, 7))
    snap.restore({"s": out})
    assert wire_bytes(out["t"]) == wire_bytes(t)
    # a second take on the same groups keeps working (keys of the first were cleared, tags advance per group)
    M.Snapshot.async_take(os.path.join(root, "world2"), {"s": M.StateDict(t=t)}).wait()
    dist.barrier()
    dist.destroy_process_group()


def test_async_commit_tags_are_per_process_group(tmp_path):
    store = tempfile.NamedTemporaryFile(delete=False)
    mp.spawn(_subgroup_worker, args=(3, store.name, str(tmp_path)), nprocs=3, join=True)
    assert os.path.exists(tmp_path / "world" / ".snapshot_metadata") and os.path.exists(tmp_path / "world2" / ".snapshot_metadata")
