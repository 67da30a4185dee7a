"""Generates tests/golden/ by running the UNMODIFIED reference (pytorch/torchsnapshot) on the deterministic inputs of
the test-suite.  Run it after build(), with the directory that holds the reference's ``torchsnapshot`` package:

    PYTHONDONTWRITEBYTECODE=1 python oracle/gen_golden.py REFERENCE_DIR [OUT_DIR]

The reference does not travel with the repository; its outputs do, as these fixtures: canonical manifest + sha256 of
every raw payload file, a few whole snapshots it wrote, and the chunk plans it computed.  Payload bytes do not depend
on the device the tensors live on, so the CPU fixtures pin the CUDA path too.  On a machine with a GPU the fixtures of
the CUDA-only tests (C2 app_state, mixed CUDA state) are written as well."""
import gzip
import json
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from tests.cases import CASES, SHARDED_CASES, apply_knobs, build_sharded  # noqa: E402
from tests.util import snapshot_digest  # noqa: E402

# cases whose whole snapshot is stored, so that the suite restores what the reference wrote (tests/test_parity_cpu.py)
STORED_SNAPSHOTS = ("dtypes_and_views", "chunked_slabbed", "model_adam")


def _dump(out, name, obj, compress=False, indent=1):
    if compress:
        with gzip.GzipFile(os.path.join(out, f"{name}.json.gz"), "wb", mtime=0) as f:
            f.write(json.dumps(obj, sort_keys=False).encode())
    else:
        with open(os.path.join(out, f"{name}.json"), "w") as f:
            json.dump(obj, f, indent=indent, sort_keys=False)


def take_digest(ref, out, name, app_state, knobs, keep_snapshot=False, compress=False, **kw):
    with tempfile.TemporaryDirectory() as d, apply_knobs(knobs):
        path = os.path.join(d, "snap")
        ref.Snapshot.take(path, app_state, **kw)
        dig = snapshot_digest(path)
        if keep_snapshot:
            dst = os.path.join(out, "ref_snapshots", name)
            shutil.rmtree(dst, ignore_errors=True)
            shutil.copytree(path, dst)
    dig["knobs"] = knobs
    dig["generator"] = {"reference": "pytorch/torchsnapshot", "torch": torch.__version__}
    _dump(out, name, dig, compress)
    print(f"{name}: {len(dig['manifest'])} entries, {len(dig['files'])} files")


def chunk_plans():
    """The reference's chunk_tensor / subdivide_shard plans for 25 seeded random shapes and byte limits."""
    from torchsnapshot.io_preparers.chunked_tensor import ChunkedTensorIOPreparer
    from torchsnapshot.io_preparers.sharded_tensor import ShardedTensorIOPreparer

    g = torch.Generator().manual_seed(1234)
    cases = []
    for _ in range(25):
        shape = [int(x) for x in torch.randint(1, 40, (int(torch.randint(1, 4, (1,), generator=g)),), generator=g)]
        t = torch.zeros(shape, dtype=torch.float32)
        limit = int(torch.randint(16, 4000, (1,), generator=g))
        chunks = [[list(c.offsets), list(c.sizes)] for c in ChunkedTensorIOPreparer.chunk_tensor(t, chunk_sz_bytes=limit)]
        dim = int(torch.randint(0, len(shape), (1,), generator=g))
        sub = [[list(o), list(s)] for _, o, s in ShardedTensorIOPreparer.subdivide_shard(t, [0] * len(shape), shape, dim, limit)]
        cases.append({"shape": shape, "limit": limit, "dim": dim, "chunks": chunks, "subdivide": sub})
    return {"elem_size": 4, "cases": cases}


def main(ref_parent, out):
    os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")
    sys.path.insert(0, ref_parent)
    import torchsnapshot as ref  # the reference

    assert os.path.abspath(ref.__file__).startswith(os.path.abspath(ref_parent)), ref.__file__
    os.makedirs(out, exist_ok=True)

    for name, (build, knobs) in CASES.items():
        take_digest(ref, out, name, {"state": ref.StateDict(**build("cpu"))}, knobs, keep_snapshot=name in STORED_SNAPSHOTS)
    _dump(out, "chunk_plans", chunk_plans(), indent=None)

    store = tempfile.NamedTemporaryFile(delete=False)
    dist.init_process_group("gloo", init_method=f"file://{store.name}", rank=0, world_size=1)
    for name, (_, knobs) in SHARDED_CASES.items():
        take_digest(ref, out, name, {"state": ref.StateDict(**build_sharded(name, "cpu"))}, knobs)
    from torch.distributed.device_mesh import init_device_mesh

    from tests.test_dtensor_cpu import DTENSOR_KNOBS, _state

    take_digest(ref, out, "dtensor", {"m": ref.StateDict(**_state(init_device_mesh("cpu", (1,)))[0])}, DTENSOR_KNOBS)

    if torch.cuda.is_available():
        from benchmarks import workloads as W
        from tests.test_round2_gpu import MIXED_KNOBS, _mixed_cuda_state

        take_digest(ref, out, "mixed_cuda", {"m": ref.StateDict(**_mixed_cuda_state())}, MIXED_KNOBS)
        app_state, kw, _ = W.build_c2(ref, 0, 1, torch.device("cuda:0"), 0)
        take_digest(ref, out, "c2_replicated_cuda", app_state, {}, compress=True, **kw)
    dist.destroy_process_group()

    # two gloo ranks, replicated + per-rank + sharded state (tests/test_multirank_cpu.py)
    from tests.test_multirank_cpu import _run, scrubbed_manifest

    with tempfile.TemporaryDirectory() as d:
        _run(2, ref_parent, "sync", d)
        dig = snapshot_digest(os.path.join(d, "snap"))
    files = [v["nbytes"] for v in dig["files"].values() if "nbytes" in v]
    _dump(out, "two_rank_replicated", {"manifest": scrubbed_manifest(dig), "payload_nbytes": sum(files), "generator": {"reference": "pytorch/torchsnapshot", "torch": torch.__version__}})
    print("two_rank_replicated:", len(dig["manifest"]), "entries")


if __name__ == "__main__":
    if len(sys.argv) < 2 or not os.path.isdir(os.path.join(sys.argv[1], "torchsnapshot")):
        raise SystemExit(__doc__)
    main(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "tests", "golden"))
