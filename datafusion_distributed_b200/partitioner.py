"""Host mirror of the producer half: Partitioning::Hash + BatchPartitioner.

Names follow the reference's operator surface
(`Partitioning::Hash(exprs, n)`, `scale_partitioning`,
src/execution_plans/common.rs:17-26; `BatchPartitioner` is DataFusion's).
All compute goes through the C ABI into the CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _native as nv
from .device import DeviceColumn, WorkerContext, columns_to_c


@dataclass(frozen=True)
class Partitioning:
    """`Partitioning::Hash(exprs, n)` restricted to column-reference exprs."""

    key_cols: Tuple[int, ...]
    partition_count: int

    @staticmethod
    def Hash(key_cols: Sequence[int], n: int) -> "Partitioning":
        return Partitioning(tuple(int(k) for k in key_cols), int(n))


def scale_partitioning(p: Partitioning, f) -> Partitioning:
    """src/execution_plans/common.rs:17-26 — Hash(exprs, p) -> Hash(exprs, f(p))."""
    return Partitioning(p.key_cols, int(f(p.partition_count)))


class HashPartitioner:
    """≙ `BatchPartitioner::try_new(Partitioning::Hash(..), ..)` on one GPU."""

    def __init__(self, ctx: WorkerContext, partitioning: Partitioning, seeds: Optional[Sequence[int]] = None):
        self.ctx = ctx
        self.partitioning = partitioning
        self._h = C.c_void_p()
        keys = (C.c_int32 * len(partitioning.key_cols))(*partitioning.key_cols)
        seeds_arr = (C.c_uint64 * 4)(*seeds) if seeds is not None else None
        nv.check(nv.lib().dfd_partitioner_create(ctx.handle, partitioning.partition_count, keys,
                                                 len(partitioning.key_cols), seeds_arr, C.byref(self._h)))
        ctx._adopt(self)

    def set_key_hash_mode(self, key_index: int, mode: int):
        """Interval(DayTime) / Interval(MonthDayNano) keys hash field by field (`dfd_partitioner_set_key_hash_mode`)."""
        nv.check(nv.lib().dfd_partitioner_set_key_hash_mode(self._h, key_index, mode))

    def set_key_dictionary(self, key_index: int, dictionary_values):
        """Key column `key_index` holds dictionary INDICES of `dictionary_values` (a pyarrow Array, or None to make the key
        plain again): hash the values once on the device (`dfd_hash_columns_device`) and let rows take
        dict_hashes[index] (`dfd_partitioner_set_key_dictionary`) — DataFusion's hash_dictionary."""
        if not hasattr(self, "_dicts"):
            self._dicts = {}
        if dictionary_values is None:
            nv.check(nv.lib().dfd_partitioner_set_key_dictionary(self._h, key_index, None, None))
            self._dicts.pop(key_index, None)
            return
        vals = DeviceColumn.from_arrow(self.ctx, dictionary_values)
        n = len(dictionary_values)
        hashes = self.ctx.alloc(max(n * 8, 8))
        nv.check(nv.lib().dfd_hash_columns_device(self.ctx.handle, columns_to_c([vals]), 1, n, None, hashes.ptr))
        nv.check(nv.lib().dfd_partitioner_set_key_dictionary(self._h, key_index, hashes.ptr, vals.validity or None))
        self._dicts[key_index] = (vals, hashes)  # keep the device buffers alive

    @property
    def num_partitions(self) -> int:
        return self.partitioning.partition_count

    def close(self):
        if self._h and self.ctx.handle:  # (the context destroys its children first)
            nv.lib().dfd_partitioner_destroy(self._h)
        self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def part_starts_device_ptr(self) -> int:
        """Device address of the int64 part_starts[N+1] of the last dense `partition()` call."""
        return nv.lib().dfd_partitioner_part_starts_device(self._h) or 0

    def partition_ids(self, cols: Sequence[DeviceColumn], n_rows: int) -> np.ndarray:
        """dest[i] = create_hashes(keys)[i] % N, computed on the GPU."""
        out = self.ctx.alloc(max(n_rows * 4, 4))
        nv.check(nv.lib().dfd_partition_ids_device(self._h, columns_to_c(cols), len(cols), n_rows, out.ptr))
        return out.download(np.uint32, n_rows)

    def partition(self, cols: Sequence[DeviceColumn], n_rows: int, out_cols: Optional[List[DeviceColumn]] = None,
                  sync: bool = True):
        """Partition device columns; returns (out_cols, part_starts[N+1] | None)."""
        if out_cols is None:
            out_cols = [DeviceColumn.empty_like(self.ctx, c, n_rows) for c in cols]
        starts = (C.c_int64 * (self.num_partitions + 1))() if sync else None
        nv.check(nv.lib().dfd_partition_device(self._h, columns_to_c(cols), len(cols), n_rows,
                                               columns_to_c(out_cols), starts))
        return out_cols, (np.frombuffer(starts, dtype=np.int64).copy() if sync else None)

    # -- single-pass form (region layout) ------------------------------------------
    def default_region_rows(self, n_rows: int, slack: float = 0.25) -> int:
        """Rows reserved per destination: the fair share plus `slack`, rounded up to 32 rows
        (aligned region starts).  A destination that outgrows it triggers the exact re-run."""
        N = self.num_partitions
        fair = -(-max(n_rows, 1) // N)
        return (int(fair * (1.0 + slack)) + 32 + 31) // 32 * 32

    def partition_onepass(self, cols: Sequence[DeviceColumn], n_rows: int, region_rows: Optional[int] = None,
                          out_cols: Optional[List[DeviceColumn]] = None, sync: bool = True):
        """`dfd_partition_device_onepass`: one kernel, no histogram pass.  Destination p is rows
        [starts[p], starts[p] + counts[p]) of every output column (starts[p] = p * region_rows unless the
        call fell back to / re-ran with the dense layout).  Returns (out_cols, starts[N], counts[N]);
        with sync=False the arrays are None and `collect()` fetches them."""
        N = self.num_partitions
        if region_rows is None:
            region_rows = self.default_region_rows(n_rows)
        if out_cols is None:
            out_cols = [DeviceColumn.empty_like(self.ctx, c, N * region_rows) for c in cols]
        starts = (C.c_int64 * N)() if sync else None
        counts = (C.c_int64 * N)() if sync else None
        nv.check(nv.lib().dfd_partition_device_onepass(self._h, columns_to_c(cols), len(cols), n_rows, columns_to_c(out_cols),
                                                       region_rows, starts, counts))
        if not sync:
            return out_cols, None, None
        return out_cols, np.frombuffer(starts, dtype=np.int64).copy(), np.frombuffer(counts, dtype=np.int64).copy()

    def collect(self):
        """Complete an asynchronous `partition_onepass(sync=False)`: (starts[N], counts[N])."""
        N = self.num_partitions
        starts, counts = (C.c_int64 * N)(), (C.c_int64 * N)()
        nv.check(nv.lib().dfd_partitioner_collect(self._h, starts, counts))
        return np.frombuffer(starts, dtype=np.int64).copy(), np.frombuffer(counts, dtype=np.int64).copy()


class PartialReduceExec:
    """≙ AggregateExec(mode = PartialReduce) above the producers' hash RepartitionExec
    (src/distributed_planner/partial_reduce_below_network_shuffles.rs:17-100): merges rows with equal group keys inside
    each destination partition of a partitioned device table (`dfd_partial_reduce_device`).

    Group keys may be fixed-width, Boolean, Utf8, LargeUtf8 or Binary columns, and keys and states may be nullable: NULL
    is a group value, null states are skipped, and a state is null when every input state of its group is.  An output
    column is nullable iff its `validity` is set; the default outputs (`DeviceColumn.empty_like`) get a validity bitmap
    exactly when the input column has one, and string outputs a byte capacity equal to the input's byte count, which
    the reduced keys never exceed."""

    def __init__(self, ctx: WorkerContext, key_cols: Sequence[int], agg_ops: Sequence[int]):
        """agg_ops[c] = nv.AGG_* for state column c, -1 for the group-key columns."""
        self.ctx, self.key_cols, self.agg_ops = ctx, [int(k) for k in key_cols], [int(a) for a in agg_ops]

    def reduce(self, cols: Sequence[DeviceColumn], n_rows: int, part_starts_device: int, num_partitions: int,
               out_cols: Optional[List[DeviceColumn]] = None):
        """-> (out_cols, out_part_starts[N+1]); `part_starts_device` = device pointer to the input's int64 part_starts[N+1]."""
        if out_cols is None:
            out_cols = [DeviceColumn.empty_like(self.ctx, c, n_rows) for c in cols]
        keys = (C.c_int32 * len(self.key_cols))(*self.key_cols)
        ops = (C.c_int32 * len(self.agg_ops))(*self.agg_ops)
        starts = (C.c_int64 * (num_partitions + 1))()
        nv.check(nv.lib().dfd_partial_reduce_device(self.ctx.handle, columns_to_c(cols), len(cols), n_rows, keys, len(self.key_cols), ops,
                                                    part_starts_device, num_partitions, columns_to_c(out_cols), starts, None))
        return out_cols, np.frombuffer(starts, dtype=np.int64).copy()
