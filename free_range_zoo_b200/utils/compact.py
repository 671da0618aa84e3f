"""Compact observation format for policies that read observations on the host.

``env.gather_observations(compact=True)`` and ``env.step_host(..., observations='compact')`` return a
``CompactObservations``: the same observations as ``gather_observations()``, encoded on the device
(``frz_observe_compact``, include/frz_obs.h) so that fewer bytes cross the link:

- integer arrays are narrowed to int8 / int16 when a bound the configuration guarantees fits (chosen once, from the
  configuration alone, by each domain's ``_compact_schema()``); ``counts`` is uint8 while the capacity is <= 255 rows;
- masks are bits: environment b's bits start on byte ``mask_offsets[b]``, bit ``g * counts[b] + t`` (LSB first) is
  group g's (agent g's) entry for task t;
- columns that are configuration constants are not downloaded (wildfire ``self_obs``: only the suppressant column) and
  are put back by ``unpack()``.

The encoders write device staging buffers whose live bytes the library then stores into page-locked host buffers
(through their device mapping, 16-byte stores, sizes read on the device: one synchronisation); the host buffers are
overwritten by the next download.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Tuple

import numpy as np
import torch

from free_range_zoo_b200 import _lib

_TYPE_CODES = {torch.int32: _lib.OBS_I32, torch.int16: _lib.OBS_I16, torch.int8: _lib.OBS_I8, torch.uint8: _lib.OBS_U8,
               torch.float32: _lib.OBS_F32}
_KIND_CODES = {'dense': _lib.OBS_DENSE, 'rows': _lib.OBS_ROWS, 'mask': _lib.OBS_MASK_BITS}


def narrow_dtype(bound: int) -> torch.dtype:
    """The narrowest signed type holding every value of [-bound, bound]: int8, int16, else int32 (no narrowing)."""
    bound = int(bound)
    if bound <= 127:
        return torch.int8
    if bound <= 32767:
        return torch.int16
    return torch.int32


def count_dtype(capacity: int) -> torch.dtype:
    """Type of the per-environment live-row counts, which lie in [0, capacity]."""
    return torch.uint8 if int(capacity) <= 255 else narrow_dtype(capacity)


def mask_offsets(counts: np.ndarray, groups: int) -> np.ndarray:
    """int64 [B + 1]: first byte of every environment's mask bits (each environment's range is byte-aligned)."""
    sizes = (int(groups) * np.asarray(counts, dtype=np.int64) + 7) // 8
    return np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)


@dataclass(frozen=True)
class Array:
    """One array of the download.  ``src`` is the padded device array; its layout is stated, never inferred:
    dense: [B, rows, src_columns] (a [B, rows] array has one column); rows / mask: [B, groups, rows, src_columns]
    with ``rows`` padded rows per (environment, group), of which the first counts[b] are live."""
    name: str
    kind: str
    src: torch.Tensor
    dtype: torch.dtype  # compact element type
    groups: int
    rows: int
    src_columns: int
    column_first: int
    columns: int
    fill: Optional[torch.Tensor] = None  # dense column selection: [rows, src_columns] values of the other columns


def dense(name: str, src: torch.Tensor, bound: Optional[int] = None, columns: Optional[Tuple[int, int]] = None,
          fill: Optional[torch.Tensor] = None) -> Array:
    """A whole [B, ...] array.  ``bound``: |value| <= bound for an int32 array (None = keep the type); ``columns`` =
    (first, count) of the last dimension to download, the others being ``fill`` ([rows, src_columns] constants)."""
    src_columns = src.shape[-1] if src.dim() == 3 else 1
    rows = math.prod(src.shape[1:]) // max(src_columns, 1)
    first, count = columns if columns is not None else (0, src_columns)
    if (columns is None) != (fill is None):
        raise ValueError(f'{name}: a column selection needs the values of the other columns')
    dtype = src.dtype if bound is None else narrow_dtype(bound)
    return Array(name, 'dense', src, dtype, 1, rows, src_columns, first, count, fill)


def rows(name: str, src: torch.Tensor, bound: int) -> Array:
    """Live rows of an int32 [B, capacity, columns] array whose values satisfy |value| <= bound."""
    B, capacity, columns = src.shape
    return Array(name, 'rows', src, narrow_dtype(bound), 1, capacity, columns, 0, columns)


def mask(name: str, src: torch.Tensor, groups: int) -> Array:
    """A uint8 [B, groups, stride] mask of which entries [b, g, :counts[b]] are live, downloaded as bits."""
    if src.dim() != 3 or src.shape[1] != groups or src.dtype != torch.uint8:
        raise ValueError(f'{name}: expected a uint8 [B, {groups}, stride] mask, got {tuple(src.shape)} {src.dtype}')
    return Array(name, 'mask', src, torch.uint8, groups, src.shape[2], 1, 0, 1)


@dataclass(frozen=True)
class Schema:
    """A domain's compact format: ``capacity`` = most live rows an environment can have, the arrays, and the groups
    of its masks (one mask bit per (group, live row))."""
    capacity: int
    arrays: List[Array]
    mask_groups: int = 1


class CompactObservations:
    """Observations of one download in the compact format (page-locked host tensors, overwritten by the next one).

    ``counts`` [B] (uint8 up to 255 rows, else int16 / int32) live rows per environment; ``offsets`` int32 [B + 1]
    their exclusive prefix sum; ``total`` = offsets[B]; ``mask_offsets`` int64 [B + 1] first byte of each
    environment's mask bits; ``bytes`` = bytes that crossed the link.  ``obs[name]`` is one array:

    - dense arrays: [B, ...] like ``gather_observations()``, narrowed; a column selection keeps only its columns
      (wildfire ``self_obs``: the suppressant, [B, A]);
    - row arrays (``task_obs``): [total, columns] narrowed live rows, environment b's rows at ``offsets[b]``;
    - masks (``action_mask`` / ``task_mask``): uint8 bytes; environment b's bit g * counts[b] + t (LSB first) of the
      bytes from ``mask_offsets[b]`` on is agent g's entry for task t.

    ``unpack()`` returns exactly what ``gather_observations()`` returns (same keys, dtypes, shapes and values)."""

    def __init__(self, schema: Schema, counts: torch.Tensor, offsets: torch.Tensor, buffers: Dict[str, torch.Tensor],
                 mask_bytes: Optional[int] = None):
        self.schema = schema
        self.counts = counts
        self.offsets = offsets
        self.total = int(offsets[-1])
        self._mask_offsets = None
        self.arrays: Dict[str, torch.Tensor] = {}
        moved = counts.numel() * counts.element_size() + offsets.numel() * 4
        for array in schema.arrays:
            buffer = buffers[array.name]
            if array.kind == 'dense':
                shape = tuple(array.src.shape) if array.fill is None else tuple(array.src.shape[:-1]) + (array.columns, )
                if array.fill is not None and array.columns == 1:
                    shape = shape[:-1]
                view = buffer[:math.prod(shape)].view(shape)
            elif array.kind == 'rows':
                view = buffer[:self.total * array.groups * array.columns].view(self.total * array.groups, array.columns)
            else:
                view = buffer[:int(self.mask_offsets[-1]) if mask_bytes is None else mask_bytes]
            self.arrays[array.name] = view
            moved += view.numel() * view.element_size()
        self.bytes = moved

    @property
    def mask_offsets(self) -> torch.Tensor:
        if self._mask_offsets is None:
            self._mask_offsets = torch.from_numpy(mask_offsets(self.counts.numpy(), self.schema.mask_groups))
        return self._mask_offsets

    def __getitem__(self, name: str) -> torch.Tensor:
        return self.arrays[name]

    def keys(self):
        return self.arrays.keys()

    def unpack(self) -> Dict[str, Any]:
        """The packed observations of ``gather_observations()``, rebuilt bit for bit on the host."""
        counts = self.counts.to(torch.int32, copy=True)
        B, total = counts.shape[0], self.total
        out: Dict[str, Any] = {'counts': counts, 'offsets': self.offsets.clone(), 'total': total, 'bytes': self.bytes}
        for array in self.schema.arrays:
            narrow = self.arrays[array.name]
            if array.kind == 'dense':
                if array.fill is None:
                    out[array.name] = narrow.to(array.src.dtype, copy=True).view(array.src.shape)
                    continue
                full = array.fill.to(array.src.dtype).expand(B, array.rows, array.src_columns).clone()
                full[:, :, array.column_first:array.column_first + array.columns] = \
                    narrow.reshape(B, array.rows, array.columns).to(array.src.dtype)
                out[array.name] = full.view(array.src.shape)
            elif array.kind == 'rows':
                out[array.name] = narrow.to(array.src.dtype, copy=True)
            else:
                out[array.name] = torch.from_numpy(_unpack_bits(narrow.numpy(), counts.numpy(),
                                                                self.mask_offsets.numpy(), array.groups))
        return out


def _unpack_bits(bits: np.ndarray, counts: np.ndarray, offsets: np.ndarray, groups: int) -> np.ndarray:
    """uint8 [total * groups]: the bit string of every environment, without the (< 8) padding bits that end each
    environment's byte range -- i.e. entry g * counts[b] + t of environment b's block, in environment order."""
    per_env = groups * counts.astype(np.int64)
    unpacked = np.unpackbits(bits[:int(offsets[-1])], bitorder='little')
    padding = 8 * np.diff(offsets) - per_env  # 0 .. 7 per environment
    keep = np.ones(unpacked.shape[0], dtype=bool)
    ends = 8 * offsets[:-1] + per_env
    for k in range(7):
        keep[ends[padding > k] + k] = False
    return unpacked[keep]


class CompactDownload:
    """Device staging, page-locked host buffers, scratch and the ``FrzObsDownload`` block of one environment (built
    once): the encoders write the staging, the library moves its live bytes to the host buffers."""

    def __init__(self, schema: Schema, counts: torch.Tensor, key: Any = None):
        B, dev = counts.shape[0], counts.device
        self.key = key
        counts_array = Array('counts', 'dense', counts, count_dtype(schema.capacity), 1, 1, 1, 0, 1)
        self.schema = schema
        self.device_offsets = torch.zeros(B + 1, dtype=torch.int32, device=dev)
        self.offsets = torch.zeros(B + 1, dtype=torch.int32).pin_memory()
        self.status = torch.zeros(4, dtype=torch.int32).pin_memory()  # overflow flag, live rows, mask bytes
        self.scan = torch.zeros(2 * (B + 1), dtype=torch.int32, device=dev)
        self.scratch = torch.zeros(2 * ((B + 1023) // 1024 + 1), dtype=torch.int32, device=dev)
        self.buffers: Dict[str, torch.Tensor] = {}
        self.staging: Dict[str, torch.Tensor] = {}
        live = [counts_array] + [array for array in schema.arrays if array.src.numel() > 0]
        descriptors = (_lib.ObsArray * len(live))()
        for at, array in enumerate(live):
            if array.kind == 'mask':
                elements = B * ((array.groups * array.rows + 7) // 8)
            else:
                elements = B * array.groups * array.rows * array.columns
            self.buffers[array.name] = torch.empty(max(elements, 1), dtype=array.dtype).pin_memory()
            self.staging[array.name] = torch.empty(max(elements, 1), dtype=array.dtype, device=dev)
            d = descriptors[at]
            d.src, d.dst, d.host = array.src.data_ptr(), self.staging[array.name].data_ptr(), self.buffers[array.name].data_ptr()
            d.kind, d.src_type, d.dst_type = _KIND_CODES[array.kind], _TYPE_CODES[array.src.dtype], _TYPE_CODES[array.dtype]
            d.groups, d.capacity, d.src_columns = array.groups, array.rows, array.src_columns
            d.column_first, d.columns = array.column_first, array.columns
        for array in schema.arrays:  # arrays with no elements (e.g. no attackers) download nothing
            self.buffers.setdefault(array.name, torch.empty(0, dtype=array.dtype))
        self.descriptors = descriptors
        block = _lib.ObsDownload()
        block.counts, block.offsets, block.host_offsets = counts.data_ptr(), self.device_offsets.data_ptr(), self.offsets.data_ptr()
        block.scan, block.scratch, block.status = self.scan.data_ptr(), self.scratch.data_ptr(), self.status.data_ptr()
        block.arrays = ctypes.cast(descriptors, ctypes.POINTER(_lib.ObsArray))
        block.array_count = len(live)
        block.mask_groups = schema.mask_groups
        self.block = block

    def result(self) -> CompactObservations:
        """The download as observations; call after the stream it was enqueued on has been synchronised."""
        if int(self.status[0]):
            raise ValueError('an observation value lies outside the bound its compact type was chosen from (the state '
                             'does not match the configuration); use observations=True / gather_observations()')
        return CompactObservations(self.schema, self.buffers['counts'], self.offsets, self.buffers, int(self.status[2]))
