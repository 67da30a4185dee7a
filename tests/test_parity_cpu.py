"""Product path on CPU tensors (host engine, native file I/O) against the reference's golden outputs:
the whole ``.snapshot_metadata`` (containers, primitives, tensor entries, slab byte ranges) and the
sha256 of every raw payload file must be identical; plus restoring snapshots the reference wrote
(tests/golden/ref_snapshots/)."""
import json
import os
import shutil
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist

import torchsnapshot_b200 as B
from tests.cases import CASES, SHARDED_CASES, apply_knobs, build_sharded
from tests.util import det_tensor, snapshot_digest, wire_bytes

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _golden(name):
    return json.load(open(os.path.join(GOLDEN, f"{name}.json")))


def assert_matches_golden(dig, gold):
    assert dig["version"] == gold["version"] and dig["world_size"] == gold["world_size"]
    assert list(dig["manifest"].keys()) == list(gold["manifest"].keys())
    for k in gold["manifest"]:
        assert dig["manifest"][k] == gold["manifest"][k], k
    assert set(dig["files"]) == set(gold["files"])
    for k, v in gold["files"].items():
        if not v.get("opaque"):
            assert dig["files"][k] == v, k


@pytest.fixture(scope="module")
def pg():
    if not dist.is_initialized():
        f = tempfile.NamedTemporaryFile(delete=False)
        dist.init_process_group("gloo", init_method=f"file://{f.name}", rank=0, world_size=1)
    yield
    if dist.is_initialized():
        dist.destroy_process_group()


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("mode", ["take", "async_take"])
def test_take_matches_reference_golden(name, mode, tmp_path):
    build, knobs = CASES[name]
    state = build("cpu")
    with apply_knobs(knobs):
        if mode == "take":
            B.Snapshot.take(str(tmp_path / "snap"), {"state": B.StateDict(**state)})
        else:
            B.Snapshot.async_take(str(tmp_path / "snap"), {"state": B.StateDict(**state)}).wait()
    assert_matches_golden(snapshot_digest(str(tmp_path / "snap")), _golden(name))


@pytest.mark.parametrize("name", sorted(CASES))
def test_restore_round_trip(name, tmp_path):
    build, knobs = CASES[name]
    state = build("cpu")
    with apply_knobs(knobs):
        snap = B.Snapshot.take(str(tmp_path / "snap"), {"state": B.StateDict(**state)})
        from torchsnapshot_b200.flatten import flatten

        target = build("cpu")
        _, flat_t = flatten(target, "x")
        for v in flat_t.values():
            if isinstance(v, torch.Tensor):
                v.zero_()
        tgt = B.StateDict(**target)
        snap.restore({"state": tgt})
    _, a = flatten(state, "x")
    _, b = flatten(dict(tgt), "x")
    assert list(a) == list(b)
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert wire_bytes(a[k]) == wire_bytes(b[k]), k
        else:
            assert a[k] == b[k], k


@pytest.mark.parametrize("name", sorted(SHARDED_CASES))
def test_sharded_take_matches_golden_and_reshards(name, tmp_path, pg):
    _, knobs = SHARDED_CASES[name]
    state = build_sharded(name, "cpu")
    with apply_knobs(knobs):
        snap = B.Snapshot.take(str(tmp_path / "snap"), {"state": B.StateDict(**state)})
        assert_matches_golden(snapshot_digest(str(tmp_path / "snap")), _golden(name))
        # restore into a different sharding of the same tables (reshard-on-load)
        other = "sharded_dim1" if name == "sharded_dim0" else "sharded_dim0"
        specs, _ = SHARDED_CASES[name]
        from torch.distributed._shard.sharded_tensor import Shard, ShardedTensor, ShardMetadata

        targets = {}
        for i, (rows, cols, dt, dim, n) in enumerate(specs):
            odim, on = 1 - dim, n + 1
            extent = (rows, cols)[odim]
            step = -(-extent // on)
            shards = []
            for lo in range(0, extent, step):
                ln = min(step, extent - lo)
                off, sz = [0, 0], [rows, cols]
                off[odim], sz[odim] = lo, ln
                shards.append(Shard(tensor=torch.zeros(sz, dtype=dt), metadata=ShardMetadata(shard_offsets=off, shard_sizes=sz, placement="rank:0/cpu")))
            targets[f"table_{i}"] = ShardedTensor._init_from_local_shards(shards, (rows, cols))
        tgt = B.StateDict(**targets)
        snap.restore({"state": tgt})
        for i, (rows, cols, dt, dim, n) in enumerate(specs):
            full = det_tensor((rows, cols), dt, 900 + i)
            for sh in tgt[f"table_{i}"].local_shards():
                o, s = sh.metadata.shard_offsets, sh.metadata.shard_sizes
                assert wire_bytes(full[o[0] : o[0] + s[0], o[1] : o[1] + s[1]]) == wire_bytes(sh.tensor)
            # no runtime object: the whole table is materialised on the host
            got = snap.read_object(f"0/state/table_{i}")
            assert wire_bytes(got) == wire_bytes(full)


def test_empty_and_odd_bf16_tensors_are_supported(tmp_path):
    # shapes the reference cannot persist (empty tensors: T:serialization.py:204 raises; CPU bfloat16 with an
    # odd element count: truncated by T:serialization.py:208-230) — checked against the oracle instead
    from oracle import ref_port as R

    state = {"e": torch.empty(0, 4), "b1": det_tensor((), torch.bfloat16, 1), "b7": det_tensor((7,), torch.bfloat16, 2), "f": det_tensor((3,), torch.float32, 3)}
    snap = B.Snapshot.take(str(tmp_path / "s"), {"state": B.StateDict(**state)})
    entries, files = R.plan_save({f"state/{k}": v for k, v in state.items()})
    meta = json.load(open(tmp_path / "s" / ".snapshot_metadata"))["manifest"]
    (slab,) = [f for f in os.listdir(tmp_path / "s" / "batched")]
    assert (tmp_path / "s" / "batched" / slab).read_bytes() == files["batched/0"]
    for k, e in entries.items():
        got = dict(meta[f"0/{k}"])
        got["location"] = "batched/0"
        assert got == e
    tgt = B.StateDict(e=torch.ones(0, 4), b1=torch.zeros((), dtype=torch.bfloat16), b7=torch.zeros(7, dtype=torch.bfloat16), f=torch.zeros(3))
    snap.restore({"state": tgt})
    for k in state:
        assert wire_bytes(state[k]) == wire_bytes(tgt[k])


def test_cast_on_save_via_prepare_func(tmp_path):
    # the reference traces the prepare func into the entry but stages the unprocessed tensor
    # (T:io_preparers/tensor.py:59-81 vs 241-258); here the payload is the processed tensor's bytes
    w = det_tensor((33, 17), torch.float32, 5).view(torch.int32).float() / 7.0
    state = {"w": w}

    def to_bf16(path, t, tracing):
        return t.to(torch.bfloat16)

    snap = B.Snapshot.take(str(tmp_path / "s"), {"state": B.StateDict(**state)}, _custom_tensor_prepare_func=to_bf16)
    e = snap.get_manifest()["0/state/w"]
    assert e.dtype == "torch.bfloat16" and e.serializer == "buffer_protocol"
    assert (tmp_path / "s" / e.location).read_bytes() == wire_bytes(w.to(torch.bfloat16))
    got = snap.read_object("0/state/w")
    assert got.dtype == torch.bfloat16 and wire_bytes(got) == wire_bytes(w.to(torch.bfloat16))
    # restoring into an fp32 parameter converts on load, like Tensor.copy_ does in the reference
    tgt = B.StateDict(w=torch.zeros(33, 17))
    snap.restore({"state": tgt})
    assert torch.equal(tgt["w"], w.to(torch.bfloat16).float())


def test_missing_metadata_means_no_snapshot(tmp_path):
    with pytest.raises(RuntimeError, match="snapshot_metadata"):
        B.Snapshot(str(tmp_path / "nope")).get_manifest()


def test_failed_write_leaves_no_metadata(tmp_path):
    # commit protocol: payload first, metadata last (T:snapshot.py:202-209; tests/test_async_take.py:58-66)
    blocker = tmp_path / "snap"
    blocker.mkdir()
    (blocker / "0").write_text("a file where a directory is needed")
    (blocker / "batched").write_text("a file where a directory is needed")
    with pytest.raises(Exception):
        B.Snapshot.take(str(blocker), {"state": B.StateDict(a=torch.ones(1 << 20))})
    assert not (blocker / ".snapshot_metadata").exists()
    pending = B.Snapshot.async_take(str(blocker), {"state": B.StateDict(a=torch.ones(1 << 20))})
    with pytest.raises(RuntimeError):
        pending.wait()
    assert not (blocker / ".snapshot_metadata").exists()


@pytest.mark.parametrize("name", ["dtypes_and_views", "chunked_slabbed", "model_adam"])
def test_interchangeable_with_live_reference(name, tmp_path):
    """Against the reference's recorded output, not a live run of it: what this package writes is, file for file, the
    snapshot the unmodified reference wrote for the same state (stored by oracle/gen_golden.py; torch_save pickles are
    compared as present, not byte for byte), and this package restores the reference's snapshot.  The other direction
    is test_reference_restores_what_this_package_wrote."""
    from torchsnapshot_b200.flatten import flatten

    build, knobs = CASES[name]
    state = build("cpu")

    def zeros():
        t = build("cpu")
        for v in flatten(t, "x")[1].values():
            if isinstance(v, torch.Tensor):
                v.zero_()
        return t

    shutil.copytree(os.path.join(GOLDEN, "ref_snapshots", name), tmp_path / "theirs")
    with apply_knobs(knobs):
        B.Snapshot.take(str(tmp_path / "ours"), {"state": B.StateDict(**state)})
        assert snapshot_digest(str(tmp_path / "ours")) == snapshot_digest(str(tmp_path / "theirs"))
        # we read what the reference wrote
        t2 = B.StateDict(**zeros())
        B.Snapshot(str(tmp_path / "theirs")).restore({"state": t2})
    a = flatten(state, "x")[1]
    got = flatten(dict(t2), "x")[1]
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert wire_bytes(a[k]) == wire_bytes(got[k]), k
        else:
            assert a[k] == got[k], k


REF_PARENT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF_PARENT, "torchsnapshot")), reason="reference not staged (oracle/make_ref.sh)")
@pytest.mark.parametrize("name", ["dtypes_and_views", "chunked_slabbed", "model_adam"])
def test_reference_restores_what_this_package_wrote(name, tmp_path):
    """The unmodified reference (the copy build() stages under oracle/_ref) reads this package's snapshot."""
    sys.path.insert(0, REF_PARENT)
    os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")
    try:
        import torchsnapshot as ref
    finally:
        sys.path.remove(REF_PARENT)
    from torchsnapshot_b200.flatten import flatten

    build, knobs = CASES[name]
    state = build("cpu")
    target = build("cpu")
    for v in flatten(target, "x")[1].values():
        if isinstance(v, torch.Tensor):
            v.zero_()
    with apply_knobs(knobs):
        B.Snapshot.take(str(tmp_path / "ours"), {"state": B.StateDict(**state)})
        t1 = ref.StateDict(**target)
        ref.Snapshot(str(tmp_path / "ours")).restore({"state": t1})
    a, got = flatten(state, "x")[1], flatten(dict(t1), "x")[1]
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert wire_bytes(a[k]) == wire_bytes(got[k]), k
        else:
            assert a[k] == got[k], k


def test_restore_detects_missing_and_truncated_payload(tmp_path):
    state = {"a": torch.arange(100_000, dtype=torch.float32), "b": torch.ones(10)}
    with apply_knobs({"no_batching": 1}):
        B.Snapshot.take(str(tmp_path / "s"), {"state": B.StateDict(**state)})
        victim = tmp_path / "s" / "0" / "state" / "a"
        data = victim.read_bytes()
        victim.write_bytes(data[: len(data) // 2])  # truncated file: a short read must not pass silently
        with pytest.raises(Exception):
            B.Snapshot(str(tmp_path / "s")).restore({"state": B.StateDict(a=torch.zeros(100_000), b=torch.zeros(10))})
        victim.unlink()
        with pytest.raises(Exception):
            B.Snapshot(str(tmp_path / "s")).restore({"state": B.StateDict(a=torch.zeros(100_000), b=torch.zeros(10))})


def test_concurrent_takes_from_two_threads(tmp_path):
    import threading

    states = [{f"t{i}": det_tensor((1000 + i, 37), torch.float32, 10 * k + i) for i in range(20)} for k in range(2)]
    errs = []

    def work(k):
        try:
            for rep in range(3):
                snap = B.Snapshot.take(str(tmp_path / f"s{k}_{rep}"), {"state": B.StateDict(**states[k])})
                tgt = B.StateDict(**{n: torch.zeros_like(v) for n, v in states[k].items()})
                snap.restore({"state": tgt})
                for n, v in states[k].items():
                    assert wire_bytes(v) == wire_bytes(tgt[n]), n
        except Exception as e:  # pragma: no cover
            errs.append(e)

    ts = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
