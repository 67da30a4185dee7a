"""Plain-tensor leg of the hot path.

Reference behaviour being replaced (T:io_preparers/tensor.py):
  * prepare_write (50-89)   -> TensorEntry + one WriteReq whose stager owns the (view of the) tensor
  * stage_buffer (240-271)  -> pageable ``tensor.to("cpu")`` in a thread, then a memoryview
  * consume_buffer (331-340)-> frombuffer + ``dst.copy_(src)`` (pageable H2D)
Here the stager/consumer only *describe* the copy (``native_descs``); the engine executes all of them
together: one pack/scatter kernel launch, pinned ring, native file I/O.  The asyncio methods remain
for storage plugins the engine cannot drive directly and run the same kernels through the stage /
consume seam of the C ABI."""
from __future__ import annotations

import asyncio
import math
from concurrent.futures import Executor
from typing import Any, Callable, List, Optional, Tuple, Union

import torch

from .. import _native
from ..io_types import BufferConsumer, BufferStager, BufferType, Future, ReadReq, WriteReq
from ..manifest import ChunkedTensorEntry, TensorEntry
from ..serialization import (
    BUFFER_PROTOCOL_SUPPORTED_DTYPES,
    SUPPORTED_QUANTIZED_DTYPES,
    Serializer,
    dtype_to_element_size,
    dtype_to_string,
    string_to_dtype,
    tensor_from_memoryview,
    torch_load_from_bytes,
    torch_save_as_bytes,
)

RAW = Serializer.BUFFER_PROTOCOL.value
PICKLED = Serializer.TORCH_SAVE.value
from ..prepare import PER_TENSOR_QTENSOR, fused_quant_of  # noqa: E402
from ..serialization import per_tensor_qtensor_from_bytes  # noqa: E402
PrepareFunc = Callable[[torch.Tensor, bool], torch.Tensor]


def entry_nbytes(entry: TensorEntry) -> int:
    n = dtype_to_element_size(string_to_dtype(entry.dtype))
    for s in entry.shape:
        n *= s
    if entry.serializer == PER_TENSOR_QTENSOR:
        n += 16  # [q_scale: double][q_zero_point: int64] behind the int_repr bytes (T:serialization.py:278-310)
    return n


def engine_for(t: torch.Tensor) -> "_native.Engine":
    if t.is_cuda:
        return _native.get_engine(t.device.index if t.device.index is not None else torch.cuda.current_device())
    return _native.get_engine(-1)


def current_stream_of(t: torch.Tensor) -> Optional[int]:
    return torch.cuda.current_stream(t.device).cuda_stream if t.is_cuda else None


class TensorBufferStager(BufferStager):
    def __init__(
        self,
        tensor: torch.Tensor,
        entry: TensorEntry,
        is_async_snapshot: bool = False,
        _tensor_prepare_func: Optional[PrepareFunc] = None,
    ) -> None:
        self.tensor = tensor
        self.entry = entry
        self.is_async_snapshot = is_async_snapshot
        self._tensor_prepare_func = _tensor_prepare_func
        # (qdtype, scale, zero_point) when the entry is a quantise-on-save one: the pack kernel quantises
        self.qparams = fused_quant_of(_tensor_prepare_func, tensor) if entry.serializer == PER_TENSOR_QTENSOR else None

    # ---- engine-facing description ------------------------------------------------------------
    def is_raw(self) -> bool:
        return self.entry.serializer == RAW

    def source(self) -> torch.Tensor:
        """The tensor whose bytes are persisted.  With a prepare func this is the *processed* tensor:
        the payload then matches ``entry.dtype`` (the reference stages the unprocessed tensor here,
        T:io_preparers/tensor.py:241-258, which makes such snapshots unreadable; see DESIGN.md)."""
        t = self.tensor.detach()
        if self._tensor_prepare_func is not None:
            t = self._tensor_prepare_func(t, False).detach()
        return t

    def wire_nbytes(self) -> int:
        return entry_nbytes(self.entry)

    def native_descs(self, wire_offset: int) -> Tuple[List["_native.CopyDesc"], List[torch.Tensor]]:
        if self.qparams is not None:
            t = self.tensor.detach()
            if self.is_async_snapshot and t.device.type == "cpu":
                t = t.clone()
            qdtype, scale, zp = self.qparams
            return [_native.save_desc(t, wire_offset, wire_dtype=qdtype, qparams=(scale, zp))], [t]
        t = self.source()
        if t.numel() == 0:
            return [], []
        if _native.needs_contiguous_copy(t):
            t = t.contiguous()
        elif self.is_async_snapshot and t.device.type == "cpu":
            # host memory is read while the snapshot drains in the background: take a private copy so
            # that later in-place updates (e.g. Adam's CPU `step` counters) cannot leak into it
            t = t.clone()
        return [_native.save_desc(t, wire_offset)], [t]

    # ---- asyncio seam ---------------------------------------------------------------------------
    async def stage_buffer(self, executor: Optional[Executor] = None) -> BufferType:
        if not self.is_raw() and self.qparams is None:
            # complex / quantized tensors: unchanged torch.save path (out of scope of the engine)
            t = self.source()
            cpu = t.cpu() if t.device.type != "cpu" else t
            if cpu.numel() != cpu.untyped_storage().nbytes() // max(cpu.element_size(), 1):
                cpu = cpu.clone()
            return torch_save_as_bytes(cpu)
        descs, keep = self.native_descs(0)
        nbytes = self.wire_nbytes()
        if not descs:
            return memoryview(b"")
        t = keep[0]
        staged = engine_for(t).stage(descs, nbytes, stream=current_stream_of(t), keepalive=keep)
        if executor is not None:
            return await asyncio.get_running_loop().run_in_executor(executor, staged.wait)
        return staged.wait()

    def get_staging_cost_bytes(self) -> int:
        n = entry_nbytes(self.entry)
        return n if self.is_raw() else 2 * n


class TensorBufferConsumer(BufferConsumer):
    def __init__(self, tensor: torch.Tensor, entry: TensorEntry) -> None:
        self.tensor = tensor
        self.entry = entry

    def is_raw(self) -> bool:
        return self.entry.serializer == RAW and _raw_castable(string_to_dtype(self.entry.dtype), self.tensor.dtype)

    def wire_nbytes(self) -> int:
        return entry_nbytes(self.entry)

    def native_descs(self, wire_offset: int) -> Tuple[List["_native.CopyDesc"], List[torch.Tensor]]:
        """The destination receives the whole saved tensor (dtype-converting when they differ)."""
        dst = self.tensor.detach()
        if dst.numel() == 0:
            return [], []
        if list(dst.shape) != list(self.entry.shape):
            raise RuntimeError(f"shape mismatch: saved {self.entry.shape}, destination {list(dst.shape)}")
        return [_native.load_desc(dst, wire_offset, wire_dtype=string_to_dtype(self.entry.dtype))], [dst]

    @staticmethod
    def deserialize_tensor(buf: bytes, entry: TensorEntry) -> torch.Tensor:
        if entry.serializer == PICKLED:
            return torch_load_from_bytes(buf)
        if entry.serializer == RAW:
            return tensor_from_memoryview(memoryview(buf), dtype=string_to_dtype(entry.dtype), shape=entry.shape)
        if entry.serializer == PER_TENSOR_QTENSOR:
            return per_tensor_qtensor_from_bytes(bytes(buf), string_to_dtype(entry.dtype), list(entry.shape))
        raise ValueError(f"Unrecognized serializer: {entry.serializer}.")

    async def consume_buffer(self, buf: bytes, executor: Optional[Executor] = None) -> None:
        def work() -> None:
            if self.is_raw():
                descs, _ = self.native_descs(0)
                if descs:
                    engine_for(self.tensor).consume(buf, descs)
            else:
                tensor_copy(self.tensor, self.deserialize_tensor(buf, self.entry))

        if executor is not None:
            await asyncio.get_running_loop().run_in_executor(executor, work)
        else:
            work()

    def get_consuming_cost_bytes(self) -> int:
        n = entry_nbytes(self.entry)
        return n if self.is_raw() else 2 * n


_FLOATS = (torch.float16, torch.bfloat16, torch.float32, torch.float64)


def _raw_castable(src: torch.dtype, dst: torch.dtype) -> bool:
    """dtype pairs the scatter kernel handles itself; others fall back to Tensor.copy_ semantics."""
    if src == dst:
        return src in BUFFER_PROTOCOL_SUPPORTED_DTYPES
    return src in _FLOATS and dst in _FLOATS


def _q_params_equal(a: torch.Tensor, b: torch.Tensor) -> bool:
    if a.qscheme() != b.qscheme():
        return False
    if a.qscheme() == torch.per_tensor_affine:
        return a.q_scale() == b.q_scale() and a.q_zero_point() == b.q_zero_point()
    return (
        a.q_per_channel_axis() == b.q_per_channel_axis()
        and torch.equal(a.q_per_channel_scales(), b.q_per_channel_scales())
        and torch.equal(a.q_per_channel_zero_points(), b.q_per_channel_zero_points())
    )


def tensor_copy(dst: torch.Tensor, src: torch.Tensor) -> None:
    """``dst.copy_(src)`` with the reference's quantized-tensor caveat (T:io_preparers/tensor.py:385-409): a quantized
    copy moves the storage and the qparams, so a view of a larger tensor (a chunk) whose qparams differ from the
    source's gets the dequantized values instead; with equal qparams the integer values are copied as they are."""
    if src.is_quantized and (
        not dst.is_quantized
        or dst.qscheme() != src.qscheme()
        or dst.dtype != src.dtype
        or (dst._is_view() and not _q_params_equal(dst, src))
    ):
        src = src.dequantize()
    dst.detach().copy_(src)


class TensorIOPreparer:
    @staticmethod
    def prepare_write(
        storage_path: str,
        tensor: torch.Tensor,
        is_async_snapshot: bool = False,
        _tensor_prepare_func: Optional[PrepareFunc] = None,
    ) -> Tuple[TensorEntry, List[WriteReq]]:
        traced = tensor if _tensor_prepare_func is None else _tensor_prepare_func(tensor, True)
        if traced.shape != tensor.shape:
            raise RuntimeError(
                "_tensor_prepare_func shouldn't change the tensor's shape "
                f"(changed from {tensor.shape} to {traced.shape})."
            )
        serializer = RAW if traced.dtype in BUFFER_PROTOCOL_SUPPORTED_DTYPES else PICKLED
        if _tensor_prepare_func is not None and fused_quant_of(_tensor_prepare_func, tensor) is not None:
            serializer = PER_TENSOR_QTENSOR  # int_repr + 16-byte trailer, produced by the pack kernel
        entry = TensorEntry(
            location=storage_path,
            serializer=serializer,
            dtype=dtype_to_string(traced.dtype),
            shape=list(traced.shape),
            replicated=False,
        )
        stager = TensorBufferStager(tensor, entry, is_async_snapshot, _tensor_prepare_func)
        return entry, [WriteReq(path=storage_path, buffer_stager=stager)]

    @staticmethod
    def get_tensor_size_from_entry(entry: TensorEntry) -> int:
        return entry_nbytes(entry)

    @staticmethod
    def can_load_inplace(entry: Union[TensorEntry, ChunkedTensorEntry], obj: Any) -> bool:
        if not isinstance(obj, torch.Tensor) or list(entry.shape) != list(obj.shape):
            return False
        if getattr(entry, "serializer", None) == PER_TENSOR_QTENSOR and obj.dtype in _FLOATS:
            return True  # dequantised into the float tensor it was quantised from (tensor_copy)
        return string_to_dtype(entry.dtype) == obj.dtype

    @staticmethod
    def empty_tensor_from_entry(entry: Union[TensorEntry, ChunkedTensorEntry]) -> torch.Tensor:
        dtype = string_to_dtype(entry.dtype)
        if dtype in SUPPORTED_QUANTIZED_DTYPES:
            raise RuntimeError("Allocating an empty quantized tensor is not supported yet.")
        return torch.empty(entry.shape, dtype=dtype)

    @classmethod
    def prepare_read(
        cls,
        entry: TensorEntry,
        tensor_out: Optional[torch.Tensor] = None,
        buffer_size_limit_bytes: Optional[int] = None,
    ) -> Tuple[List[ReadReq], Future[torch.Tensor]]:
        if tensor_out is None or not cls.can_load_inplace(entry, tensor_out):
            tensor_out = cls.empty_tensor_from_entry(entry)
        if buffer_size_limit_bytes is not None and entry.serializer == RAW:
            return cls.prepare_read_tiled(entry, tensor_out, buffer_size_limit_bytes)
        rr = ReadReq(path=entry.location, byte_range=entry.byte_range_tuple, buffer_consumer=TensorBufferConsumer(tensor_out, entry))
        return [rr], Future(obj=tensor_out)

    @classmethod
    def prepare_read_tiled(
        cls, entry: TensorEntry, tensor_out: torch.Tensor, buffer_size_limit_bytes: int
    ) -> Tuple[List[ReadReq], Future[torch.Tensor]]:
        """Budgeted read: the payload is consumed in <= limit sized byte ranges (T:io_preparers/tensor.py:128-181).
        Tiles are runs of dim-0 slices of the flattened destination when it is dense, rows otherwise."""
        total = entry_nbytes(entry)
        n_tiles = max(1, math.ceil(total / max(buffer_size_limit_bytes, 1)))
        try:
            target = tensor_out.view(-1)
        except RuntimeError:
            target = tensor_out
        if target.dim() == 0:
            target = target.reshape(1)
        esz = dtype_to_element_size(string_to_dtype(entry.dtype))
        base = entry.byte_range[0] if entry.byte_range is not None else 0
        length = target.shape[0]
        step = max(1, math.ceil(length / n_tiles)) if length else 1
        reqs: List[ReadReq] = []
        cursor = 0
        for lo in range(0, length, step):
            piece = target.narrow(0, lo, min(step, length - lo))
            nb = piece.numel() * esz
            piece_entry = TensorEntry(entry.location, entry.serializer, entry.dtype, list(piece.shape), entry.replicated)
            reqs.append(
                ReadReq(
                    path=entry.location,
                    byte_range=(base + cursor, base + cursor + nb),
                    buffer_consumer=TensorBufferConsumer(piece, piece_entry),
                )
            )
            cursor += nb
        return reqs, Future(obj=tensor_out)
