"""Pins the oracle (oracle/ref_port.py): golden fixtures made by the unmodified reference, the
known-answer plans asserted by the reference's own tests, and the chunk plans the reference computed for
random shapes (tests/golden/chunk_plans.json)."""
import json
import os

import pytest
import torch

from oracle import ref_port as R
from tests.cases import CASES, SHARDED_CASES
from tests.util import ALL_RAW_DTYPES, canonicalize, det_tensor, wire_bytes

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _golden(name):
    return json.load(open(os.path.join(GOLDEN, f"{name}.json")))


def _flatten(state):
    from torchsnapshot_b200.flatten import flatten

    return flatten(state, prefix="state")[1]


def _oracle_digest(flat, knobs):
    import hashlib

    entries, files = R.plan_save(
        flat,
        rank=0,
        max_chunk=knobs.get("max_chunk", R.DEFAULT_MAX_CHUNK),
        max_shard=knobs.get("max_shard", R.DEFAULT_MAX_SHARD),
        slab_threshold=knobs.get("slab", R.DEFAULT_SLAB_THRESHOLD),
        batching=not knobs.get("no_batching", 0),
    )
    manifest, names = canonicalize({f"0/{k}": v for k, v in entries.items()})
    digests = {names.get(loc, loc): {"nbytes": len(b), "sha256": hashlib.sha256(b).hexdigest()} for loc, b in files.items()}
    return manifest, digests


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_reproduces_reference_goldens(name):
    build, knobs = CASES[name]
    gold = _golden(name)
    flat = {k: v for k, v in _flatten(build("cpu")).items() if isinstance(v, torch.Tensor)}
    manifest, digests = _oracle_digest(flat, knobs)
    for path, entry in manifest.items():
        assert gold["manifest"][path] == entry, path
    tensor_paths = {p for p, e in gold["manifest"].items() if e["type"] in ("Tensor", "ChunkedTensor")}
    assert tensor_paths == set(manifest)
    for loc, d in digests.items():
        assert gold["files"][loc] == d, loc
    assert {k for k, v in gold["files"].items() if not v.get("opaque")} == set(digests)


@pytest.mark.parametrize("name", sorted(SHARDED_CASES))
def test_oracle_reproduces_sharded_goldens(name):
    specs, knobs = SHARDED_CASES[name]
    gold = _golden(name)
    flat = {}
    for i, (rows, cols, dt, dim, n) in enumerate(specs):
        full = det_tensor((rows, cols), dt, 900 + i)
        extent = (rows, cols)[dim]
        step = -(-extent // n)
        shards = []
        for lo in range(0, extent, step):
            ln = min(step, extent - lo)
            off, sz = [0, 0], [rows, cols]
            off[dim], sz[dim] = lo, ln
            shards.append((full.narrow(dim, lo, ln).contiguous(), off, sz))
        flat[f"state/table_{i}"] = R.ShardedSpec(shards, dim)
    manifest, digests = _oracle_digest(flat, knobs)
    for path, entry in manifest.items():
        assert gold["manifest"][path] == entry, path
    for loc, d in digests.items():
        assert gold["files"][loc] == d, loc


def test_known_answer_chunk_plans():
    # reference tests/test_chunked_tensor_io_preparer.py:52-103
    assert R.chunk_plan([], 4, 512 << 20) == [([0], [1])]
    assert R.chunk_plan([7, 10], 4, 120) == [([0, 0], [3, 10]), ([3, 0], [3, 10]), ([6, 0], [1, 10])]
    assert R.chunk_plan([7, 10], 4, 180) == [([0, 0], [4, 10]), ([4, 0], [3, 10])]
    assert R.chunk_plan([10, 10], 4, 150) == [([0, 0], [4, 10]), ([4, 0], [4, 10]), ([8, 0], [2, 10])]
    # C1 of BASELINE.json: 1 GiB fp32 Linear weight -> two 512 MiB chunks (SURVEY.md §8)
    assert R.chunk_plan([16384, 16384], 4) == [([0, 0], [8192, 16384]), ([8192, 0], [8192, 16384])]


def test_known_answer_shard_subdivision():
    # reference tests/test_sharded_tensor_io_preparer.py:212-297: 256 / 256 / 86 / 86 / 1 pieces
    assert len(R.subdivide_plan([0, 0], [256, 128], 0, 4, 128 * 4)) == 256
    assert len(R.subdivide_plan([0, 0], [128, 256], 1, 4, 128 * 4)) == 256
    assert len(R.subdivide_plan([0, 0], [256, 128], 0, 4, 128 * 4 * 3)) == 86
    assert len(R.subdivide_plan([0, 0], [128, 256], 1, 4, 128 * 4 * 3)) == 86
    assert len(R.subdivide_plan([0, 0], [256, 128], 0, 4, 1 << 30)) == 1
    # C5 of BASELINE.json: 2 GB row shard [3_906_250, 128] fp32 -> 4 pieces, 1_048_576 rows each but the last
    pieces = R.subdivide_plan([0, 0], [3_906_250, 128], 0, 4)
    assert [p[2][0] for p in pieces] == [1_048_576, 1_048_576, 1_048_576, 760_522]


def test_slab_assignment_rules():
    # `>=` opens a new slab; a tensor >= threshold is never batched; CPU and GPU chains are independent
    reqs = [("a", 60, False, True), ("b", 40, False, True), ("c", 100, False, True), ("g", 50, True, True), ("d", 39, False, True), ("o", 5, False, False)]
    passthrough, slabs = R.slab_assign(reqs, threshold=100)
    assert passthrough == ["c", "o"]
    assert slabs == [
        {"cuda": False, "members": [("a", 0, 60)]},
        {"cuda": False, "members": [("b", 0, 40), ("d", 40, 79)]},
        {"cuda": True, "members": [("g", 0, 50)]},
    ]


def test_overlap_region_matches_narrow_semantics():
    full = torch.arange(20 * 30).reshape(20, 30)
    saved = ([4, 10], [10, 15])
    cur = ([8, 0], [12, 18])
    assert R.boxes_overlap(*saved, *cur)
    region = R.overlap_region(saved[0], saved[1], cur[0], cur[1])
    s = full[4:14, 10:25]
    c = full[8:20, 0:18]
    for d, so, co, n in region:
        s = s.narrow(d, so, n)
        c = c.narrow(d, co, n)
    assert torch.equal(s, c) and s.numel() == 6 * 8
    assert not R.boxes_overlap([0, 0], [4, 4], [4, 0], [4, 4])


def test_serialize_view_every_dtype_and_layout():
    for i, dt in enumerate(ALL_RAW_DTYPES):
        t = det_tensor((6, 9, 4), dt, i)
        for v in (t, t.permute(2, 0, 1), t[1:5, ::2, 1:], t[3], t[:, 4, 2], t.reshape(-1)[3:100], t[0, 0, 0]):
            assert R.serialize_view(v) == wire_bytes(v)
    e = torch.randn(3, 1).expand(3, 4)
    assert R.serialize_view(e) == wire_bytes(e)
    assert R.serialize_view(torch.empty(0, 3)) == b""


def test_ref_pipeline_round_trip_and_bytes(tmp_path):
    tensors = {f"t{i}": det_tensor((50 + i, 7), [torch.float32, torch.int16, torch.bfloat16][i % 3], i) for i in range(12)}
    tensors["big"] = det_tensor((64, 33), torch.float64, 99)
    pipe = R.RefPipeline(str(tmp_path), slab_threshold=4096, max_chunk=6000)
    index = pipe.save(tensors)
    flat = {f"{k}": v for k, v in tensors.items()}
    entries, files = R.plan_save(flat, max_chunk=6000, slab_threshold=4096)
    for loc, blob in files.items():
        assert (tmp_path / loc).read_bytes() == blob, loc
    out = {k: torch.zeros_like(v) for k, v in tensors.items()}
    pipe.load(index, out)
    for k in tensors:
        assert wire_bytes(tensors[k]) == wire_bytes(out[k]), k


def test_oracle_against_live_reference():
    """Against the reference's recorded output, not a live run of it: the chunk_tensor / subdivide_shard plans the
    unmodified reference computed for 25 seeded random shapes and byte limits (tests/golden/chunk_plans.json, made by
    oracle/gen_golden.py) equal the oracle's."""
    gold = _golden("chunk_plans")
    assert len(gold["cases"]) == 25
    for c in gold["cases"]:
        shape, limit, dim = c["shape"], c["limit"], c["dim"]
        assert [[list(o), list(s)] for o, s in R.chunk_plan(shape, gold["elem_size"], limit)] == c["chunks"], c
        got = R.subdivide_plan([0] * len(shape), shape, dim, gold["elem_size"], limit)
        assert [[list(o), list(s)] for _, o, s in got] == c["subdivide"], c
