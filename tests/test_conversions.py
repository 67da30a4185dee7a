"""Fused float casts, cast-on-load and quantise-on-save against an exact reference written in numpy.

The reference is independent of torch and of the engine:

* every source widens exactly to float64 (fp16 through np.float16, bf16 as ``uint32(bits) << 16`` viewed as float32);
* float destinations follow torch's conversion semantics: fp32 and fp16 round to nearest even, overflow becomes inf;
  an fp64 source reaches fp16 and bf16 through fp32, i.e. it is rounded twice (torch has no direct double -> half
  conversion); bf16 rounds the fp32 bits with ``(u + 0x7FFF + ((u >> 16) & 1)) >> 16``;
* non-NaN results must match bitwise (signed zeros and infinities included); a NaN input must give some NaN, whose
  payload is not compared (torch's own CPU paths disagree on it);
* quantisation has one reference per device, because torch's CPU (FBGEMM) and CUDA kernels differ at ties:
  CUDA computes ``rint(double(x) / scale) + zp``, the CPU ``zp + rint(x * float(1 / float(scale)))`` in float32;
  both clamp before converting to an integer.

Each matrix runs through the host planner (``host_execute``) and, on a GPU, through the pack / scatter kernels
(``Engine.stage`` for saves, ``Engine.consume`` and ``Engine.scatter_device`` for loads).  torch's own ``.to()`` and
``quantize_per_tensor`` on the same device are checked against the same reference, so a disagreement shows which
side moved."""
import functools
import struct
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist

import torchsnapshot_b200 as B
from tests.util import wire_bytes
from torchsnapshot_b200 import _native as N

F16, BF16, F32, F64 = torch.float16, torch.bfloat16, torch.float32, torch.float64
FLOATS = (F16, BF16, F32, F64)
PAIRS = [(s, d) for s in FLOATS for d in FLOATS if s != d]
_NAME = {F16: "f16", BF16: "bf16", F32: "f32", F64: "f64"}
_UINT = {F16: np.uint16, BF16: np.uint16, F32: np.uint32, F64: np.uint64}
_SINT = {F16: np.int16, BF16: np.int16, F32: np.int32, F64: np.int64}
_TINT = {F16: torch.int16, BF16: torch.int16, F32: torch.int32, F64: torch.int64}
ESZ = {F16: 2, BF16: 2, F32: 4, F64: 8}
TILE = 128 * 1024  # kTileLsu: destination bytes per LSU tile
OFFSETS = (0, 1, 2, 3, 6, 8, 16)


def _pair_id(p):
    return f"{_NAME[p[0]]}-{_NAME[p[1]]}"


SAVE_EXEC = ["host", pytest.param("device", marks=pytest.mark.gpu)]
LOAD_EXEC = ["host", pytest.param("consume", marks=pytest.mark.gpu), pytest.param("scatter", marks=pytest.mark.gpu)]


# ---- exact reference ---------------------------------------------------------------------------------------------
def widen(bits: np.ndarray, src: torch.dtype) -> np.ndarray:
    """Exact float64 value of every element."""
    with np.errstate(invalid="ignore"):  # NaN inputs widen to NaN
        return _widen(bits, src)


def _widen(bits: np.ndarray, src: torch.dtype) -> np.ndarray:
    if src == F16:
        return bits.view(np.float16).astype(np.float64)
    if src == BF16:
        return (bits.astype(np.uint32) << 16).view(np.float32).astype(np.float64)
    if src == F32:
        return bits.view(np.float32).astype(np.float64)
    return bits.view(np.float64).copy()


def narrow(x: np.ndarray, dst: torch.dtype) -> np.ndarray:
    """Bits of ``dst`` for float64 values that are exact values of the source dtype (torch's semantics: anything
    narrower than fp32 is reached through fp32)."""
    with np.errstate(over="ignore", invalid="ignore"):
        if dst == F64:
            return x.view(np.uint64).copy()
        f = x.astype(np.float32)
        if dst == F32:
            return f.view(np.uint32)
        if dst == F16:
            return f.astype(np.float16).view(np.uint16)
        u = f.view(np.uint32).astype(np.uint64)
        return (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF).astype(np.uint16)


def is_nan_bits(b: np.ndarray, dt: torch.dtype) -> np.ndarray:
    if dt == F16:
        return ((b & 0x7C00) == 0x7C00) & ((b & 0x03FF) != 0)
    if dt == BF16:
        return ((b & 0x7F80) == 0x7F80) & ((b & 0x007F) != 0)
    return np.isnan(b.view(np.float32 if dt == F32 else np.float64))


def assert_cast(got: np.ndarray, src_bits: np.ndarray, src: torch.dtype, dst: torch.dtype, what: str) -> None:
    """``got`` (bits of ``dst``) is the conversion of ``src_bits`` (bits of ``src``), element by element."""
    x = widen(src_bits, src)
    want = narrow(x, dst)
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, got.shape, want.shape)
    nan = np.isnan(x)
    bad = np.where(nan, ~is_nan_bits(got, dst), got != want)
    if bad.any():
        idx = np.flatnonzero(bad)
        first = ", ".join(f"[{i}] {int(src_bits[i]):#x} ({x[i]!r}): got {int(got[i]):#x}, want {int(want[i]):#x}" for i in idx[:6])
        raise AssertionError(f"{what} {_NAME[src]}->{_NAME[dst]}: {idx.size} of {got.size} elements wrong; {first}")


def quant_ref(x32: np.ndarray, scale: float, zp: int, qdtype: torch.dtype, device: bool) -> np.ndarray:
    """int_repr bytes of per-tensor affine quantisation of float32 values (NaN is undefined in torch and not used)."""
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        if device:
            r = np.rint(x32.astype(np.float64) / scale) + zp
        else:
            inv = np.float32(1.0) / np.float32(scale)
            r = np.rint(x32.astype(np.float32) * inv).astype(np.float64) + zp
    lo, hi = (-128, 127) if qdtype == torch.qint8 else (0, 255)
    return np.clip(r, lo, hi).astype(np.int64).astype(np.int8 if qdtype == torch.qint8 else np.uint8).view(np.uint8)


# ---- conversions between numpy bits, tensors and wire bytes ------------------------------------------------------
def tensor_of(bits: np.ndarray, dt: torch.dtype, device="cpu") -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(bits).view(_SINT[dt]).copy()).view(dt).to(device)


def bits_of(t: torch.Tensor) -> np.ndarray:
    """C-order bits of a float tensor (any layout, any device)."""
    return t.detach().cpu().contiguous().view(_TINT[t.dtype]).numpy().view(_UINT[t.dtype]).reshape(-1).copy()


def bits_in(wire: bytes, dt: torch.dtype, offset: int, n: int) -> np.ndarray:
    return np.frombuffer(wire, dtype=_UINT[dt], count=n, offset=offset).copy()


# ---- value sets --------------------------------------------------------------------------------------------------
def _f32_bits(values) -> np.ndarray:
    return np.asarray(values, dtype=np.float32).view(np.uint32)


def _both_signs(bits: np.ndarray, sign: int) -> np.ndarray:
    bits = np.asarray(bits, dtype=type(sign))
    return np.concatenate([bits, bits | sign])


def _double_rounding_f64() -> np.ndarray:
    """fp64 values next to every fp16 and bf16 rounding midpoint (including the overflow thresholds) that round
    *onto* the midpoint in fp32, so that rounding through fp32 ties to even where a single rounding would not."""
    h = np.arange(0x7C00, dtype=np.uint16).view(np.float16).astype(np.float64)  # every finite fp16 >= 0
    mids16 = np.concatenate([(h[:-1] + h[1:]) / 2, [65520.0]])
    b = widen(np.arange(0x7F80, dtype=np.uint16), BF16)  # every finite bf16 >= 0
    mids_b = np.concatenate([(b[:-1] + b[1:]) / 2, [float(np.uint32(0x7F7F8000).view(np.float32))]])
    out = []
    for m in (mids16, mids_b):
        # steps well below half an fp32 ulp of m: float32(m +- step) == m
        for rel in (2.0**-52, 2.0**-40, 2.0**-27):
            step = np.maximum(m * rel, 5e-324)
            out += [m + step, m - step]
    v = np.concatenate(out)
    v = v[v > 0]
    return _both_signs(v.view(np.uint64), np.uint64(1 << 63))


@functools.lru_cache(maxsize=None)
def _specials(src: torch.dtype) -> np.ndarray:
    """Hand-picked edge values: signed zeros, subnormals, ties of every destination, overflow boundaries, inf, NaN."""
    if src == F16:
        s = [0x0000, 0x0001, 0x0002, 0x0003, 0x03FF, 0x0400, 0x0401, 0x3C00, 0x3C01, 0x3555, 0x7BFE, 0x7BFF, 0x7C00, 0x7C01, 0x7E00, 0x7FFF, 0x1000, 0x2E66]
        return _both_signs(s, np.uint16(0x8000))
    if src == BF16:
        s = [0x0000, 0x0001, 0x007F, 0x0080, 0x0081, 0x3F80, 0x3F81, 0x3EAB, 0x3300, 0x3340, 0x3380, 0x33C0, 0x477F, 0x4780, 0x7F7E, 0x7F7F, 0x7F80, 0x7F81, 0x7FC0, 0x7FFF]
        return _both_signs(s, np.uint16(0x8000))
    if src == F32:
        ties = [0x3F808000, 0x3F818000, 0x3F807FFF, 0x3F808001, 0x7F7F8000, 0x7F7F7FFF, 0x7F7E8000, 0x00008000, 0x00018000, 0x3F801000, 0x3F803000]
        fp16 = [65504.0, np.nextafter(np.float32(65520.0), np.float32(0)), 65520.0, 65536.0, 2.0**-24, 2.0**-25, 3 * 2.0**-25, 3 * 2.0**-26, 5 * 2.0**-26, 2.0**-14, 1.0 + 2.0**-11, 1.0 + 3 * 2.0**-11]
        fp16_bits = list(_f32_bits(fp16))
        fp16_bits += [int(b) + d for b in _f32_bits([2.0**-25, 3 * 2.0**-25, 65520.0]) for d in (-1, 1)]
        edge = [0x00000000, 0x00000001, 0x00000002, 0x007FFFFF, 0x00400000, 0x00800000, 0x7F7FFFFF, 0x7F800000, 0x7F800001, 0x7FC00000, 0x7FFFFFFF, 0x3F800000, 0x3EAAAAAB]
        return _both_signs(ties + fp16_bits + edge, np.uint32(0x80000000))
    fmax = float(np.finfo(np.float32).max)
    half_ulp = 2.0**103  # half an fp32 ulp at FLT_MAX: FLT_MAX + half_ulp is the overflow tie
    vals = [0.0, 5e-324, 1e-320, 2.2250738585072009e-308, 2.2250738585072014e-308, 1e-300, 1.0, 1 + 2.0**-11 + 2.0**-40, 65519.999, 2.0**-25 + 2.0**-60,
            1 + 2.0**-8 + 2.0**-40, 1 + 2.0**-8 - 2.0**-40, 65504.0, 65520.0, 2.0**-149, 2.0**-150, 1.5 * 2.0**-149, 2.0**-126,
            fmax, np.nextafter(fmax, np.inf), np.nextafter(fmax, 0.0), fmax + half_ulp, np.nextafter(fmax + half_ulp, 0.0), np.nextafter(fmax + half_ulp, np.inf),
            2.0**128, 1e300, float(np.finfo(np.float64).max), np.inf]
    bits = list(np.asarray(vals, dtype=np.float64).view(np.uint64))
    bits += [0x7FF8000000000000, 0x7FF0000000000001, 0x7FFFFFFFFFFFFFFF, 0x000FFFFFFFFFFFFF]
    return _both_signs(bits, np.uint64(1 << 63))


@functools.lru_cache(maxsize=None)
def full_values(src: torch.dtype) -> np.ndarray:
    """The exhaustive / dense sweep of a source dtype, specials included."""
    if src in (F16, BF16):
        return np.arange(1 << 16, dtype=np.uint64).astype(np.uint16)
    if src == F32:
        hi = np.arange(1 << 16, dtype=np.uint32) << 16
        lo = np.array([0x0000, 0x0001, 0x7FFF, 0x8000, 0x8001, 0xFFFF], dtype=np.uint32)
        return np.concatenate([(hi[:, None] | lo[None, :]).reshape(-1), _specials(F32)])
    rng = np.random.default_rng(20261017)
    n = 1 << 20
    sign = rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(63)
    mant = rng.integers(0, 1 << 52, n, dtype=np.uint64)
    # a quarter over every biased exponent (zero/subnormal and inf/NaN included), the rest where fp32, fp16 and bf16
    # round, overflow and flush
    exp = np.concatenate([rng.integers(0, 2048, n // 4, dtype=np.uint64), rng.integers(1023 - 160, 1023 + 132, n - n // 4, dtype=np.uint64)])
    rand = sign | (exp << np.uint64(52)) | mant
    return np.concatenate([_specials(F64), _double_rounding_f64(), rand])


def compact_values(src: torch.dtype, n: int = 12288) -> np.ndarray:
    """Specials plus a deterministic sample of the full sweep: what the layout tests move."""
    full, spec = full_values(src), _specials(src)
    pick = np.random.default_rng(7).choice(full.size, max(0, n - spec.size), replace=False)
    return np.concatenate([spec, full[np.sort(pick)]])[:n]


# ---- executors ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engine():
    eng = N.Engine(device=0, io_threads=2, pinned_slot_bytes=4 << 20, pinned_slots=4)
    yield eng
    eng.close()


def _dev(executor: str) -> str:
    return "cpu" if executor == "host" else "cuda:0"


def run_save(request, executor: str, members, nbytes: int) -> bytes:
    """members: [(tensor, wire_offset, wire_dtype, qparams)] -> the wire image.  The tensors stay referenced by
    ``members`` until the copy has returned (descriptors hold raw pointers)."""
    descs = [N.save_desc(t, off, wire_dtype=wd, qparams=qp) for t, off, wd, qp in members]
    if executor == "host":
        slack = 32
        wire = torch.full((nbytes + slack,), 0xA5, dtype=torch.uint8)
        N.host_execute(descs, wire)
        out = bytes(wire.numpy())
        assert out[nbytes:] == b"\xa5" * slack, "write past the end of the image"
        return out[:nbytes]
    eng = request.getfixturevalue("engine")
    sb = eng.stage(descs, nbytes, stream=torch.cuda.current_stream().cuda_stream, keepalive=[m[0] for m in members])
    try:
        return bytes(sb.wait())
    finally:
        sb.release()


def run_load(request, executor: str, wire: bytes, members) -> None:
    """members: [(destination view, wire_offset, wire_dtype, wire_strides)]."""
    descs = [N.load_desc(t, off, wire_dtype=wd, wire_strides=ws) for t, off, wd, ws in members]
    if executor == "host":
        buf = torch.frombuffer(bytearray(wire), dtype=torch.uint8).clone()  # 64 B aligned: offsets decide alignment
        N.host_execute(descs, buf)
        return
    eng = request.getfixturevalue("engine")
    if executor == "consume":
        eng.consume(wire, descs)
    else:
        w = torch.frombuffer(bytearray(wire), dtype=torch.uint8).to("cuda:0")
        eng.scatter_device(w, descs)
    torch.cuda.synchronize()


def _check_torch_to(bits, src, dst, device, what):
    """torch's own conversion on the same device agrees with the reference."""
    assert_cast(bits_of(tensor_of(bits, src, device).to(dst)), bits, src, dst, f"torch .to() on {device}, {what}")


# ---- float casts on save -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("executor", SAVE_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_save_full_sweep(request, executor, pair):
    """Every value of the sweep, dense and 16 B aligned (the vectorised path for fp32 <-> fp16/bf16), at numel % 8 of
    0 and 5 so that the ragged tail is exercised; the larger images span several 128 KiB tiles."""
    src, dst = pair
    dev = _dev(executor)
    vals = full_values(src)
    spec = _specials(src)
    for tail in (0, 5):
        n = vals.size + 8 + (tail - vals.size) % 8
        bits = np.concatenate([vals, np.resize(spec, n - vals.size)])  # pad with specials: they also land in the tail
        assert bits.size % 8 == tail
        t = tensor_of(bits, src, dev)
        nbytes = n * ESZ[dst]
        if src != F64:
            assert nbytes > TILE
        got = run_save(request, executor, [(t, 0, dst, None)], nbytes)
        assert_cast(bits_in(got, dst, 0, n), bits, src, dst, f"{executor} dense numel={n}")
    _check_torch_to(vals, src, dst, dev, "full sweep")


@pytest.mark.parametrize("executor", SAVE_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_save_specials_in_the_ragged_tail(request, executor, pair):
    """One member of 8 + 5 elements per group of five specials: every special value passes once through the vectorised
    body and once through the scalar tail of the same member, and all members share one image."""
    src, dst = pair
    dev = _dev(executor)
    spec = _specials(src)
    k = -(-spec.size // 5)
    members, keep, off = [], [], 0
    for j in range(k):
        tail = np.resize(np.roll(spec, -5 * j), 5)
        body = np.resize(np.roll(spec, -5 * j - 5), 8)
        bits = np.concatenate([body, tail])
        t = tensor_of(bits, src, dev)
        members.append((t, off, dst, None))
        keep.append(bits)
        off += -(-13 * ESZ[dst] // 16) * 16  # 16 B aligned members: the vectorised path applies to each
    got = run_save(request, executor, members, off)
    for (t, o, _, _), bits in zip(members, keep):
        assert_cast(bits_in(got, dst, o, 13), bits, src, dst, f"{executor} tail member at {o}")
    _check_torch_to(spec, src, dst, dev, "specials")


def _layouts(flat: torch.Tensor):
    """Views of one value tensor that take the scalar path: narrowed along dim 1, transposed, and a stepped 3-D
    permute (several outer dims); plus a view whose single run is larger than one tile."""
    n = flat.numel()
    c = 96
    r = n // c
    m2 = flat[: r * c].view(r, c)
    m3 = flat[: 16 * 24 * 32].view(16, 24, 32)
    return {
        "narrow1": m2[:, 3:90],
        "t": m2.t(),
        "permute3": m3[:, ::2, 1:].permute(2, 0, 1),
        "rows": m2[1:-1],
    }


@pytest.mark.parametrize("executor", SAVE_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_save_strided_views(request, executor, pair):
    src, dst = pair
    dev = _dev(executor)
    vals = compact_values(src)
    base = tensor_of(vals, src, dev)
    for name, v in _layouts(base).items():
        n = v.numel()
        got = run_save(request, executor, [(v, 0, dst, None)], n * ESZ[dst])
        assert_cast(bits_in(got, dst, 0, n), bits_of(v), src, dst, f"{executor} {name}")


@pytest.mark.parametrize("executor", SAVE_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_save_to_misaligned_wire_offsets(request, executor, pair):
    """The destination sits at every small byte offset, so element stores are misaligned (byte-wise stores); a
    uint8 member fills the bytes in front, and nothing may be written around the cast member."""
    src, dst = pair
    dev = _dev(executor)
    vals = compact_values(src, 4096 + 5)
    t = tensor_of(vals, src, dev)
    strided = t[: 64 * 64].view(64, 64).t()
    for off in OFFSETS:
        for v in (t, strided):
            members = []
            lead = torch.arange(off, dtype=torch.uint8, device=dev) + 1
            if off:
                members.append((lead, 0, None, None))
            members.append((v, off, dst, None))
            n = v.numel()
            got = run_save(request, executor, members, off + n * ESZ[dst])
            assert got[:off] == bytes(range(1, off + 1)), off
            assert_cast(bits_in(got, dst, off, n), bits_of(v), src, dst, f"{executor} wire offset {off}, stride {v.stride()}")


# ---- float casts on load -----------------------------------------------------------------------------------------
_SENTINEL = {F16: 0x7E5A, BF16: 0x7F5A, F32: 0x7F85A5A5, F64: 0x7FF5A5A5A5A5A5A5}  # NaNs no conversion produces


def _sentinel(shape, dt, dev):
    return tensor_of(np.full(int(np.prod(shape)), _SENTINEL[dt], dtype=_UINT[dt]), dt, dev).view(shape)


def _assert_only_view_written(base: torch.Tensor, view_of):
    mask = torch.zeros(base.shape, dtype=torch.bool)
    view_of(mask).fill_(True)
    outside = bits_of(base)[~mask.reshape(-1).numpy()]
    assert (outside == _SENTINEL[base.dtype]).all(), "load wrote outside its destination view"


@pytest.mark.parametrize("executor", LOAD_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_load_full_sweep(request, executor, pair):
    """Wire of ``src`` -> dense ``dst`` tensor (Tensor.copy_ semantics), every value of the sweep."""
    src, dst = pair
    dev = _dev(executor)
    vals = full_values(src)
    for tail in (0, 5):
        n = vals.size + 8 + (tail - vals.size) % 8
        bits = np.concatenate([vals, np.resize(_specials(src), n - vals.size)])
        out = _sentinel((n,), dst, dev)
        run_load(request, executor, bits.tobytes(), [(out, 0, src, None)])
        assert_cast(bits_of(out), bits, src, dst, f"{executor} dense numel={n}")
    # Tensor.copy_ is what the reference's restore does
    want = _sentinel((vals.size,), dst, dev)
    want.copy_(tensor_of(vals, src, dev))
    assert_cast(bits_of(want), vals, src, dst, f"torch copy_ on {dev}")


@pytest.mark.parametrize("executor", LOAD_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_load_from_misaligned_wire_offsets(request, executor, pair):
    """The saved piece starts at every small byte offset of the wire (slab members are packed without padding), so
    the source elements are misaligned; destinations are dense and strided views."""
    src, dst = pair
    dev = _dev(executor)
    vals = compact_values(src, 4096 + 5)
    for off in OFFSETS:
        wire = bytes(range(0x40, 0x40 + off)) + vals.tobytes() + b"\x5a" * 8
        out = _sentinel((vals.size,), dst, dev)
        run_load(request, executor, wire, [(out, off, src, None)])
        assert_cast(bits_of(out), vals, src, dst, f"{executor} dense from wire offset {off}")
        base = _sentinel((64, 80), dst, dev)
        view_of = lambda b: b[:, 5:69].t()  # noqa: E731
        run_load(request, executor, wire, [(view_of(base), off, src, None)])
        assert_cast(bits_of(view_of(base)), vals[: 64 * 64], src, dst, f"{executor} strided from wire offset {off}")
        _assert_only_view_written(base, view_of)


@pytest.mark.parametrize("executor", LOAD_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_load_strided_destinations(request, executor, pair):
    src, dst = pair
    dev = _dev(executor)
    vals = compact_values(src)
    shapes = {k: v.shape for k, v in _layouts(torch.empty(vals.size)).items()}
    for name, shape in shapes.items():
        base = _sentinel((vals.size,), dst, dev)
        view = _layouts(base)[name]
        assert view.shape == shape
        n = view.numel()
        run_load(request, executor, vals[:n].tobytes(), [(view, 0, src, None)])
        assert_cast(bits_of(view), vals[:n], src, dst, f"{executor} {name}")
        _assert_only_view_written(base, lambda b: _layouts(b)[name])


@pytest.mark.parametrize("executor", LOAD_EXEC)
@pytest.mark.parametrize("pair", PAIRS, ids=_pair_id)
def test_cast_on_load_reshard_sub_box(request, executor, pair):
    """Reshard-on-load with a cast: the destination receives rows 10:30, cols 8:40 of a saved [40, 64] piece
    (``wire_strides``) into a narrowed view of a bigger local shard; the piece sits at an aligned and an odd offset."""
    src, dst = pair
    dev = _dev(executor)
    piece = compact_values(src, 40 * 64).reshape(40, 64)
    for base_off in (0, 3):
        wire = b"\x11" * base_off + piece.tobytes()
        local = _sentinel((50, 100), dst, dev)
        view_of = lambda b: b[5:25, 20:52]  # noqa: E731
        off = base_off + (10 * 64 + 8) * ESZ[src]
        run_load(request, executor, wire, [(view_of(local), off, src, [64, 1])])
        assert_cast(bits_of(view_of(local)), piece[10:30, 8:40].reshape(-1), src, dst, f"{executor} sub-box at {base_off}")
        _assert_only_view_written(local, view_of)


# ---- quantise-on-save --------------------------------------------------------------------------------------------
SCALES = (2.0**-2, 0.1, 1.0 / 3.0, 1e-3)
ZERO_POINTS = {torch.qint8: (0, 3, -5), torch.quint8: (0, 7, 128)}


def _quant_inputs(scale: float, zp: int, qdtype, src) -> np.ndarray:
    """k*scale and (k+0.5)*scale for k in -300..300 (exact ties when scale is a power of two), signed zeros, the
    smallest subnormal of ``src``, values past both clamp ends, +-1e30, +-inf; returned as bits of ``src``."""
    k = np.arange(-300, 301, dtype=np.float64)
    lo, hi = (-128, 127) if qdtype == torch.qint8 else (0, 255)
    sub = {F16: 2.0**-24, BF16: 2.0**-133, F32: 2.0**-149, F64: 5e-324}[src]
    extra = [0.0, -0.0, sub, -sub, (lo - zp - 5.5) * scale, (hi - zp + 5.5) * scale, (lo - zp - 0.5) * scale, (hi - zp + 0.5) * scale, 1e30, -1e30, np.inf, -np.inf]
    x = torch.from_numpy(np.concatenate([k * scale, (k + 0.5) * scale, extra])).to(src)
    return bits_of(x)


@pytest.mark.parametrize("executor", SAVE_EXEC)
@pytest.mark.parametrize("src", FLOATS, ids=lambda d: _NAME[d])
@pytest.mark.parametrize("qdtype", [torch.qint8, torch.quint8], ids=["qint8", "quint8"])
def test_quantize_on_save_matches_reference(request, executor, src, qdtype):
    """Every (scale, zero_point) as one member of a single image, dense and strided members alternating, behind a
    3-byte member: each payload is followed by exactly ``struct.pack("<dq", scale, zp)`` and the next member."""
    dev = _dev(executor)
    members, expect, keep = [], [], []
    lead = torch.tensor([1, 2, 3], dtype=torch.uint8, device=dev)
    members.append((lead, 0, None, None))
    expect.append(b"\x01\x02\x03")
    off = 3
    for i, (scale, zp) in enumerate((s, z) for s in SCALES for z in ZERO_POINTS[qdtype]):
        bits = _quant_inputs(scale, zp, qdtype, src)
        x = tensor_of(bits, src, dev)
        if i % 2:
            holder = torch.zeros(bits.size, 3, dtype=src, device=dev)
            holder[:, 1] = x
            x = holder[:, 1]  # element stride 3
        keep.append(x)
        members.append((x, off, qdtype, (scale, zp)))
        x32 = widen(bits, src).astype(np.float32)
        want = quant_ref(x32, scale, zp, qdtype, device=executor != "host")
        q = torch.quantize_per_tensor(x.float().contiguous(), scale, zp, qdtype)
        # torch's vectorised CPU kernel adds the zero point in int32 after rounding, which wraps for |x / scale| near
        # 2^31 and beyond (-inf with zero point -5 gives 127): torch is compared only where that sum is defined
        defined = np.ones(bits.size, dtype=bool) if dev != "cpu" else np.abs(x32.astype(np.float64) / scale) < 2.0**30
        tq = q.int_repr().cpu().numpy().view(np.uint8)
        assert np.array_equal(tq[defined], want[defined]), f"torch.quantize_per_tensor on {dev} disagrees with the reference ({scale}, {zp})"
        expect.append(want.tobytes() + struct.pack("<dq", scale, zp))
        off += bits.size + 16
    tail = torch.tensor([9, 8, 7, 6, 5], dtype=torch.int8, device=dev)
    members.append((tail, off, None, None))
    expect.append(bytes([9, 8, 7, 6, 5]))
    off += 5
    got = run_save(request, executor, members, off)
    pos = 0
    for m, e in zip(members, expect):
        assert got[pos : pos + len(e)] == e, (m[1], m[2], m[3])
        pos += len(e)


# ---- mixed members in one image ----------------------------------------------------------------------------------
@pytest.mark.parametrize("executor", SAVE_EXEC)
def test_mixed_members_in_one_image_and_back(request, executor):
    """Plain copies, casts of every kind of layout and a quantised member back to back at odd offsets in one image;
    then the casts are restored from that image in one call (load executors: host / consume)."""
    dev = _dev(executor)
    f32 = tensor_of(compact_values(F32, 13), F32, dev)
    f64 = tensor_of(compact_values(F64, 36 * 5), F64, dev).view(36, 5)
    bf = tensor_of(compact_values(BF16, 1003), BF16, dev)
    h = tensor_of(compact_values(F16, 40 * 3), F16, dev).view(40, 3)
    qb = _quant_inputs(0.1, 3, torch.qint8, F32)
    q = tensor_of(np.concatenate([qb[280:300], qb[-12:], qb[900:905]]), F32, dev)  # 37 values, both clamp ends
    plan = [
        (torch.tensor([7, 8, 9], dtype=torch.uint8, device=dev), None, None),
        (f32, BF16, None),
        (q, torch.qint8, (0.1, 3)),
        (f64.t(), F16, None),
        (torch.arange(5, dtype=torch.int32, device=dev), None, None),
        (bf[1::2], F32, None),
        (h, F64, None),
        (f32[:5], F16, None),
    ]
    members, off = [], 0
    for t, wd, qp in plan:
        members.append((t, off, wd, qp))
        off += t.numel() + 16 if qp else t.numel() * (ESZ[wd] if wd else t.element_size())
    got = run_save(request, executor, members, off)
    pos = 0
    for t, o, wd, qp in members:
        assert o == pos
        n = t.numel()
        if qp:
            want = quant_ref(widen(bits_of(t), F32).astype(np.float32), *qp, torch.qint8, device=executor != "host")
            assert got[o : o + n + 16] == want.tobytes() + struct.pack("<dq", *qp)
            pos += n + 16
        elif wd is None:
            assert got[o : o + n * t.element_size()] == wire_bytes(t)
            pos += n * t.element_size()
        else:
            assert_cast(bits_in(got, wd, o, n), bits_of(t), t.dtype, wd, f"member at {o}")
            pos += n * ESZ[wd]
    assert pos == len(got)

    # restore every cast member (wire dtype -> the original dtype) from the same image, in one call
    loads, outs = [], []
    for t, o, wd, qp in members:
        if wd is None or qp:
            continue
        out = _sentinel(tuple(t.shape), t.dtype, dev)
        loads.append((out, o, wd, None))
        outs.append((out, bits_in(got, wd, o, t.numel()), wd))
    run_load(request, "host" if executor == "host" else "consume", got, loads)
    for out, wbits, wd in outs:
        assert_cast(bits_of(out), wbits, wd, out.dtype, "restore from the mixed image")


# ---- through the public API --------------------------------------------------------------------------------------
API_DEV = ["cpu", pytest.param("cuda:0", marks=pytest.mark.gpu)]


@pytest.fixture(scope="module")
def pg():
    if not dist.is_initialized():
        f = tempfile.NamedTemporaryFile(delete=False)
        dist.init_process_group("gloo", init_method=f"file://{f.name}", rank=0, world_size=1)
    yield
    if dist.is_initialized():
        dist.destroy_process_group()


def _payload(root, entry) -> bytes:
    data = open(root / entry.location, "rb").read()
    br = entry.byte_range
    return data if br is None else data[br[0] : br[1]]


def _double_rounding_tensor(n: int = 4096) -> torch.Tensor:
    v = _double_rounding_f64()
    pick = np.random.default_rng(3).choice(v.size, n, replace=False)
    head = np.array([1 + 2.0**-11 + 2.0**-40, 65519.999, 2.0**-25 + 2.0**-60]).view(np.uint64)
    return tensor_of(np.concatenate([head, v[np.sort(pick)]]), F64)


@pytest.mark.parametrize("dev", API_DEV)
def test_cast_on_save_fp64_to_fp16_rounds_like_torch(dev, tmp_path):
    """cast_on_save's payload is exactly ``tensor.to(dtype)``: for fp64 -> fp16 that is a rounding through fp32."""
    x = _double_rounding_tensor().to(dev)
    snap = B.Snapshot.take(str(tmp_path / "s"), {"m": B.StateDict(x=x)}, _custom_tensor_prepare_func=B.cast_on_save(F16))
    e = snap.get_manifest()["0/m/x"]
    assert e.dtype == "torch.float16"
    data = _payload(tmp_path / "s", e)
    assert data == wire_bytes(x.to(F16))
    assert_cast(np.frombuffer(data, dtype=np.uint16), bits_of(x), F64, F16, "cast_on_save payload")


def _sharded(t: torch.Tensor):
    from torch.distributed._shard.sharded_tensor import Shard, ShardedTensor, ShardMetadata

    md = ShardMetadata(shard_offsets=[0] * t.dim(), shard_sizes=list(t.shape), placement=f"rank:0/{t.device}")
    return ShardedTensor._init_from_local_shards([Shard(tensor=t, metadata=md)], tuple(t.shape))


@pytest.mark.parametrize("dev", API_DEV)
@pytest.mark.parametrize("pair", [(BF16, F32), (F64, F16)], ids=_pair_id)
def test_sharded_restore_casts_from_an_odd_slab_offset(dev, pair, tmp_path, pg):
    """A ShardedTensor shard batched behind a 3-byte tensor starts at an odd byte of the slab; restoring it into a
    target of another dtype converts like Tensor.copy_."""
    src, dst = pair
    if src == F64:
        w = _double_rounding_tensor(32).view(5, 7).to(dev)
    else:
        w = tensor_of(compact_values(src, 35), src, dev).view(5, 7)
    st = {"a": torch.tensor([1, 2, 3], dtype=torch.uint8, device=dev), "w": _sharded(w)}
    snap = B.Snapshot.take(str(tmp_path / "s"), {"m": B.StateDict(**st)})
    (shard,) = snap.get_manifest()["0/m/w"].shards
    assert shard.tensor.byte_range[0] % 2 == 1, shard.tensor.byte_range  # the case under test
    tgt = {"a": torch.zeros(3, dtype=torch.uint8, device=dev), "w": _sharded(torch.zeros(5, 7, dtype=dst, device=dev))}
    snap.restore({"m": B.StateDict(**tgt)})
    got = tgt["w"].local_shards()[0].tensor
    assert wire_bytes(got) == wire_bytes(w.to(dst))
    assert_cast(bits_of(got), bits_of(w), src, dst, "sharded restore")
    assert torch.equal(tgt["a"], st["a"])


@pytest.mark.parametrize("dev", API_DEV)
@pytest.mark.parametrize("qdtype", [torch.qint8, torch.quint8], ids=["qint8", "quint8"])
def test_quantize_on_save_saturates_like_torch(dev, qdtype, tmp_path):
    """Values far beyond the clamp (1e30, +-inf) saturate to the right end, with custom qparams."""
    scale, zp = 0.1, (3 if qdtype == torch.qint8 else 7)
    x = torch.tensor([1e30, -1e30, float("inf"), float("-inf"), 3e9, -3e9, 0.25, -0.35, 12.7, -12.8, 1e-40, 0.0] * 3, device=dev)
    hook = B.quantize_on_save(qdtype, qparams=lambda path, t: (scale, zp))
    snap = B.Snapshot.take(str(tmp_path / "s"), {"m": B.StateDict(x=x)}, _custom_tensor_prepare_func=hook)
    e = snap.get_manifest()["0/m/x"]
    assert e.serializer == "per_tensor_qtensor"
    q = torch.quantize_per_tensor(x.float(), scale, zp, qdtype)
    want = q.int_repr().cpu().numpy().tobytes() + struct.pack("<dq", scale, zp)
    assert _payload(tmp_path / "s", e) == want
    ref = quant_ref(x.cpu().numpy(), scale, zp, qdtype, device=dev != "cpu")
    assert want[: x.numel()] == ref.tobytes()


def test_host_quantise_checks_room_for_the_trailer():
    """A quantising member needs numel + 16 bytes of wire: the host planner refuses a buffer without room for the
    [scale][zero_point] trailer instead of writing past it."""
    x = torch.linspace(-1, 1, 24)
    wire = torch.zeros(24 + 15, dtype=torch.uint8)
    with pytest.raises(N.NativeError, match="exceeds the wire buffer"):
        N.host_execute([N.save_desc(x, 0, wire_dtype=torch.qint8, qparams=(0.01, 0))], wire)
    wire = torch.zeros(24 + 16, dtype=torch.uint8)
    N.host_execute([N.save_desc(x, 0, wire_dtype=torch.qint8, qparams=(0.01, 0))], wire)
    assert bytes(wire[24:].numpy()) == struct.pack("<dq", 0.01, 0)
