"""DTensor leg (FSDP2 / HSDP layouts) on a 1-rank CPU mesh: entries, payload and restore, against the oracle's byte
image and against what the unmodified reference wrote for the same state (tests/golden/dtensor.json)."""
import json
import os
import tempfile

import pytest
import torch
import torch.distributed as dist

import torchsnapshot_b200 as B
from oracle import ref_port as R
from tests.cases import apply_knobs
from tests.util import det_tensor, snapshot_digest, wire_bytes

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
DTENSOR_KNOBS = {"max_shard": 1000}


@pytest.fixture(scope="module")
def mesh():
    if not dist.is_initialized():
        f = tempfile.NamedTemporaryFile(delete=False)
        dist.init_process_group("gloo", init_method=f"file://{f.name}", rank=0, world_size=1)
    from torch.distributed.device_mesh import init_device_mesh

    yield init_device_mesh("cpu", (1,))
    if dist.is_initialized():
        dist.destroy_process_group()


def _state(mesh):
    from torch.distributed.tensor import DTensor, Replicate, Shard

    w = det_tensor((48, 20), torch.float32, 1)
    e = det_tensor((30, 16), torch.bfloat16, 2)
    return {
        "w": DTensor.from_local(w.clone(), mesh, [Shard(0)], run_check=False),
        "e": DTensor.from_local(e.clone(), mesh, [Shard(1)], run_check=False),
        "r": DTensor.from_local(det_tensor((7, 5), torch.int64, 3), mesh, [Replicate()], run_check=False),
    }, {"w": w, "e": e}


def test_dtensor_take_restore_and_layout(mesh, tmp_path):
    from torch.distributed.tensor import DTensor, Shard

    state, raw = _state(mesh)
    with apply_knobs(DTENSOR_KNOBS):
        snap = B.Snapshot.take(str(tmp_path / "s"), {"m": B.StateDict(**state)})
    man = snap.get_manifest()
    ew = man["0/m/w"]
    assert ew.type == "DTensor" and ew.mesh == [0] and ew.dim_map == [[0], [-1]]
    # 48 x 20 fp32 = 3840 B at a 1000 B limit: rows of 80 B -> 12 rows per piece -> 4 pieces (subdivide_shard)
    assert [s.sizes for s in ew.shards] == [[12, 20]] * 4 and [s.offsets for s in ew.shards] == [[0, 0], [12, 0], [24, 0], [36, 0]]
    # payload of the slab == oracle byte image of the pieces, in order
    blob = b"".join(R.serialize_view(raw["w"][o : o + 12]) for o in (0, 12, 24, 36))
    (slab,) = os.listdir(tmp_path / "s" / "batched")
    data = (tmp_path / "s" / "batched" / slab).read_bytes()
    lo = ew.shards[0].tensor.byte_range[0]
    assert data[lo : lo + len(blob)] == blob
    # restore into zeroed DTensors
    tgt = {k: DTensor.from_local(torch.zeros_like(v.to_local()), mesh, v.placements, run_check=False) for k, v in state.items()}
    snap.restore({"m": B.StateDict(**tgt)})
    for k in state:
        assert wire_bytes(state[k].to_local()) == wire_bytes(tgt[k].to_local()), k


def test_dtensor_matches_live_reference(mesh, tmp_path):
    """Against the reference's recorded output, not a live run of it: manifest and payload equal the unmodified
    reference's snapshot of the same state (tests/golden/dtensor.json, made by oracle/gen_golden.py)."""
    state, _ = _state(mesh)
    with apply_knobs(DTENSOR_KNOBS):
        B.Snapshot.take(str(tmp_path / "ours"), {"m": B.StateDict(**state)})
    theirs = json.load(open(os.path.join(GOLDEN, "dtensor.json")))
    assert theirs["knobs"] == DTENSOR_KNOBS
    assert snapshot_digest(str(tmp_path / "ours")) == {k: theirs[k] for k in ("version", "world_size", "manifest", "files")}
