"""``np.savetxt``'s default text for many arrays at once, formatted on the device (``csrc/ste_text.cu``).

Every value becomes CPython's ``'%.18e' % x`` (19 significant digits, correctly rounded, ties to even; ``inf``,
``-inf``, ``nan``), followed by ``' '`` or, after a row's last column, ``'\\n'`` - byte for byte what ``np.savetxt(path, X)``
writes.  A :class:`Table` describes one file kind across many ships; :func:`format_tables` converts a whole set of them
in two launches around one ``torch.cumsum`` and returns the text and the byte offset of every (ship, table) file.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence, Tuple

import numpy as np
import torch

from . import _native as nat

#: Bytes of the longest field and its separator: ``-1.234567890123456789e-308 ``.
MAX_VALUE_BYTES = nat.STE_TEXT_MAX_VALUE_BYTES


@dataclass
class Table:
    """One file kind: the value at (row ``r``, column ``c``) of ship ``i`` is ``base[r // row_div, planes[c], track[i]]``.

    ``base`` is a contiguous float64 CUDA tensor ``[rows][row_stride][tracks]`` (the kernels' SoA layout), ``track`` an
    int32 CUDA tensor with one column of ``base`` per ship."""

    base: torch.Tensor
    track: torch.Tensor
    planes: Sequence[int]
    row_div: int = 1

    def native(self) -> nat.SteTextTable:
        if self.base.dim() != 3 or self.base.dtype != torch.float64:
            raise ValueError("Table.base must be a float64 tensor [rows][row_stride][tracks]")
        if self.track.dtype != torch.int32:
            raise ValueError("Table.track must be int32")
        for name, t in (("base", self.base), ("track", self.track)):
            if not t.is_cuda or not t.is_contiguous():   # ld and the plane stride are taken from the shape
                raise ValueError(f"Table.{name} must be a contiguous CUDA tensor")
        t = nat.SteTextTable()
        t.base, t.track = nat.ptr(self.base), nat.ptr(self.track)
        t.ld = t.n_tracks = self.base.shape[2]
        t.row_stride, t.row_div, t.n_cols = self.base.shape[1], int(self.row_div), len(self.planes)
        for c, p in enumerate(self.planes[: nat.STE_TEXT_MAX_COLS]):
            t.plane[c] = int(p)
        return t


def format_tables(tables: Sequence[Table], value_start: torch.Tensor, n_values: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Text of every value of ``tables``: segment ``g = ship * len(tables) + table`` holds the values
    ``[value_start[g], value_start[g + 1])`` (int64 CUDA, row-major rows of ``len(planes)`` values).

    Returns ``(text, offsets)`` on the device: ``text`` (uint8, at least as long as the text) and ``offsets`` (int64,
    ``len(value_start)`` entries) with the text of segment ``g`` at ``text[offsets[g]:offsets[g + 1]]``."""
    lib = nat.load()
    dev = value_start.device
    if any(t.base.device != dev or t.track.device != dev for t in tables):
        raise ValueError("every table must live on the device of value_start")
    n_items = (value_start.numel() - 1) // max(len(tables), 1)
    arr = (nat.SteTextTable * max(len(tables), 1))(*[t.native() for t in tables])
    with torch.cuda.device(dev):   # the launches, the scan and the gather on one stream of the data's device
        digits = torch.empty(n_values, dtype=torch.int64, device=dev)
        meta = torch.empty(n_values, dtype=torch.int32, device=dev)
        length = torch.empty(n_values, dtype=torch.int32, device=dev)
        stream = nat.current_stream()
        nat.check(lib.ste_text_convert_f64(arr, len(tables), n_items, nat.ptr(value_start), n_values, nat.ptr(digits), nat.ptr(meta),
                                           nat.ptr(length), stream))
        end = torch.cumsum(length, 0, dtype=torch.int64)
        text = torch.empty(max(n_values, 1) * MAX_VALUE_BYTES, dtype=torch.uint8, device=dev)
        nat.check(lib.ste_text_write(n_values, nat.ptr(digits), nat.ptr(meta), nat.ptr(end), nat.ptr(text), text.numel(), stream))
        offsets = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), end])[value_start]
    return text, offsets


def format_values(x: torch.Tensor) -> bytes:
    """``''.join('%.18e\\n' % v for v in x)`` for a 1-D float64 CUDA tensor, formatted on the device."""
    if not x.is_cuda:
        raise ValueError("format_values formats CUDA tensors")
    x = x.reshape(-1, 1, 1).to(torch.float64).contiguous()
    n = x.shape[0]
    track = torch.zeros(1, dtype=torch.int32, device=x.device)
    value_start = torch.tensor([0, n], dtype=torch.int64, device=x.device)
    with torch.cuda.device(x.device):
        text, offsets = format_tables([Table(x, track, [0])], value_start, n)
        return text[: int(offsets[-1])].cpu().numpy().tobytes()


def diagonal_planes(cov_planes: int) -> np.ndarray:
    """Planes of a covariance row's diagonal: packed 4 x 4 (10 planes) or row-major n x n."""
    if cov_planes == 10:
        return np.array([0, 4, 7, 9])
    n = int(round(cov_planes ** 0.5))
    if n * n != cov_planes:
        raise ValueError(f"{cov_planes} covariance planes are neither packed 4 x 4 nor n x n")
    return np.arange(n) * (n + 1)
