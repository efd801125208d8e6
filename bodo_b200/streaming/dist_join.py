"""Sharded (multi-GPU) streaming hash join: the host side of build_parallel / probe_parallel.

Reference: join_build_consume_batch shuffles the build rows a rank does not own to hash_to_rank(key)
(bodo/libs/streaming/_join.cpp:3243-3300) and, once the build is complete, turns the join into a BROADCAST join when the
global build table is small (:3317-3405: all-gather the build table, mark it replicated, probe rows then stay where they
are; threshold get_bcast_join_threshold() = 10 MiB, BODO_BCAST_JOIN_THRESHOLD, bodo/libs/_hash_join.cpp:448-459);
join_probe_consume_batch shuffles the probe rows of a partitioned build side the same way.

Here, per rank (one process per GPU, torch.distributed / NCCL for the plumbing):

    build  batches are staged on the device; at the last batch the ranks all-reduce the build size and either
           all-gather the build table (broadcast join) or hash-partition it with the CUDA radix partition
           (b200_shuffle_partition) and exchange it with one all-to-all-v per buffer; the local JoinState then builds
           on the rows this rank owns (or on the whole table);
    probe  every batch is hash-partitioned and exchanged the same way when both sides are partitioned; a REPLICATED probe
           side against a partitioned build keeps only the rows whose key this rank owns (no exchange); against a replicated
           (or broadcast) build side the batch is probed as it is.

The calls are collective, as in the reference: every rank calls build / probe the same number of times (ranks that ran out of
input keep calling with empty batches until the is_last call, bodo/pandas/_pipeline.cpp:453-457).
Placement is the reference's: (uint32) XXH3_64(key, SEED_HASH_PARTITION) % n_pes, and for 2..4 key columns hash_keys of the
tuple (the further columns folded in with hash_combine_boost) % n_pes.
"""

from __future__ import annotations

import os

import numpy as np

from .. import _lib
from ..shuffle import exchange_table, partition_device, with_schema_validity
from ..table import ArrTypes, Column, Table, np_dtype_of, to_device  # noqa: F401 (to_device is re-exported)
from . import join as J


def bcast_join_threshold() -> int:
    """get_bcast_join_threshold (bodo/libs/_hash_join.cpp:448-459): bytes, BODO_BCAST_JOIN_THRESHOLD overrides."""
    v = int(os.environ.get("BODO_BCAST_JOIN_THRESHOLD", 10 * 1024 * 1024))
    if v < 0:
        raise _lib.B200Error("hash_join: bcast_join_threshold < 0")
    return v


def _as_tensor(x, dev):
    import torch

    return x if hasattr(x, "is_cuda") else torch.as_tensor(x, device=dev)


def concat_device(tables, device: int) -> Table:
    """Row-wise concatenation of device batches of one schema (validity bitmaps are re-packed through byte masks)."""
    import torch

    dev = torch.device("cuda", device)
    first = tables[0]
    cols = []
    for ci in range(first.n_cols):
        parts = [_as_tensor(t.columns[ci].data, dev)[: t.columns[ci].length] for t in tables]
        data = torch.cat(parts) if len(parts) > 1 else parts[0]
        validity = None
        if any(t.columns[ci].validity is not None for t in tables):
            bits = []
            for t in tables:
                c = t.columns[ci]
                if c.validity is None:
                    bits.append(torch.ones(c.length, dtype=torch.bool, device=dev))
                else:
                    vb = _as_tensor(c.validity, dev)
                    idx = torch.arange(c.length, device=dev)
                    bits.append(((vb[idx >> 3] >> (idx & 7).to(torch.uint8)) & 1).bool())
            m = torch.cat(bits)
            n = m.numel()
            pad = torch.zeros(((n + 63) // 64) * 64 + 64, dtype=torch.uint8, device=dev)
            pad[:n] = m.to(torch.uint8)
            w = (pad.view(-1, 8) * (1 << torch.arange(8, device=dev, dtype=torch.uint8))).sum(1).to(torch.uint8)
            validity = w
        c0 = first.columns[ci]
        arr = ArrTypes.NULLABLE_INT_BOOL if (validity is not None or c0.arr_type == ArrTypes.NULLABLE_INT_BOOL) else c0.arr_type
        cols.append(Column(data, validity, c0.c_type, arr, int(data.numel())))
    return Table(cols, list(first.names))


def all_gather_table(table: Table, device: int, group=None) -> Table:
    """gather_table(..., all_gather=true) (bodo/libs/_distributed.cpp): every rank ends up with the rows of all ranks."""
    import torch
    import torch.distributed as dist

    dev = torch.device("cuda", device)
    n_pes = dist.get_world_size(group)
    n = torch.tensor([table.n_rows], dtype=torch.int64, device=dev)
    counts = torch.empty(n_pes, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(counts, n, group=group)
    counts = [int(x) for x in counts.cpu().tolist()]
    mx = max(counts + [1])
    table = with_schema_validity(table)
    parts = []
    for r in range(n_pes):
        parts.append([])
    cols_out = []
    for c in table.columns:
        d = _as_tensor(c.data, dev)[: c.length]
        buf = torch.zeros(mx, dtype=d.dtype, device=dev)
        buf[: c.length] = d
        out = torch.empty(n_pes * mx, dtype=d.dtype, device=dev)
        dist.all_gather_into_tensor(out, buf, group=group)
        data = torch.cat([out[r * mx: r * mx + counts[r]] for r in range(n_pes)])
        validity = None
        if c.validity is not None:
            idx = torch.arange(c.length, device=dev)
            vb = _as_tensor(c.validity, dev)
            m = torch.zeros(mx, dtype=torch.uint8, device=dev)
            m[: c.length] = (vb[idx >> 3] >> (idx & 7).to(torch.uint8)) & 1
            mo = torch.empty(n_pes * mx, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(mo, m, group=group)
            mm = torch.cat([mo[r * mx: r * mx + counts[r]] for r in range(n_pes)])
            nn = mm.numel()
            pad = torch.zeros(((nn + 63) // 64) * 64 + 64, dtype=torch.uint8, device=dev)
            pad[:nn] = mm
            validity = (pad.view(-1, 8) * (1 << torch.arange(8, device=dev, dtype=torch.uint8))).sum(1).to(torch.uint8)
        cols_out.append(Column(data, validity, c.c_type, c.arr_type, int(data.numel())))
    return Table(cols_out, list(table.names))


class DistJoinState:
    """Drop-in for JoinState when build_parallel / probe_parallel is set (same verbs through streaming.join)."""

    def __init__(self, operator_id, build_key_inds, probe_key_inds, build_colnames, probe_colnames, build_outer, probe_outer,
                 output_batch_size, expected_build_rows, device, stream, is_na_equal=False, build_parallel=False, probe_parallel=False,
                 force_broadcast=False, process_group=None, is_mark_join=False, is_anti_join=False):
        import torch
        import torch.distributed as dist

        if not dist.is_initialized():
            raise _lib.B200Error("Streaming Join: build_parallel / probe_parallel need an initialised torch.distributed process group")
        self.group = process_group
        self.n_pes = dist.get_world_size(process_group)
        self.rank = dist.get_rank(process_group)
        self.build_parallel = bool(build_parallel) and self.n_pes > 1
        self.probe_parallel = bool(probe_parallel) and self.n_pes > 1
        self.force_broadcast = bool(force_broadcast)
        self.build_outer = bool(build_outer)
        self.device = device if device is not None else torch.cuda.current_device()
        self.local = J.JoinState(operator_id, build_key_inds, probe_key_inds, build_colnames, probe_colnames, build_outer, probe_outer,
                                 output_batch_size, expected_build_rows, self.device, stream, is_na_equal=is_na_equal,
                                 is_mark_join=is_mark_join, is_anti_join=is_anti_join)
        self.probe_outer = bool(probe_outer)
        # bloom filter + key bounds over the build keys of ALL ranks, applied to probe rows before they are shuffled (the
        # reference's use_bloom_filter probe path, _join.cpp:3460-3600); B200_JOIN_BLOOM=0 disables it.  The filter is built for
        # single-column keys only, so a multi-column join skips it
        self.build_key = self.local.build_key_inds
        self.probe_key = self.local.probe_key_inds
        self.use_filter = (os.environ.get("B200_JOIN_BLOOM", "1") != "0" and not probe_outer and not is_mark_join and not is_anti_join
                           and len(self.build_key) == 1)
        self.filter_ready = False
        self._build_batches = []
        self.is_broadcast = False
        self.metrics = {"build_rows_in": 0, "build_rows_local": 0, "probe_rows_in": 0, "probe_rows_local": 0, "broadcast": 0}

    # handle / metrics pass-throughs so get_metric / delete work on both kinds of state
    @property
    def handle(self):
        return self.local.handle

    def _keys_first(self, table: Table, keys) -> Table:
        order = list(keys) + [i for i in range(table.n_cols) if i not in keys]
        return table.select(order), order

    def _shuffle(self, table: Table, keys) -> Table:
        """Rows to their owners (hash_keys of the key tuple); returns the rows this rank owns, in the table's original column order."""
        import torch

        kf, order = self._keys_first(to_device(table, self.device), keys)
        part, counts = partition_device(with_schema_validity(kf), len(keys), self.n_pes)
        torch.cuda.current_stream().synchronize()
        recv = exchange_table(part, counts, self.group)
        inv = [order.index(i) for i in range(len(order))]
        return recv.select(inv)

    def _owned_only(self, table: Table, keys) -> Table:
        """Replicated input against a partitioned other side: keep the rows whose key this rank owns (no exchange)."""
        import torch

        kf, order = self._keys_first(to_device(table, self.device), keys)
        part, counts = partition_device(with_schema_validity(kf), len(keys), self.n_pes)
        torch.cuda.current_stream().synchronize()
        lo = sum(counts[: self.rank])
        n = counts[self.rank]
        blo = sum((c + 7) // 8 for c in counts[: self.rank])
        cols = []
        for c in part.columns:
            v = None
            if c.validity is not None:  # per-destination bitmaps are byte aligned: segment `rank` starts at byte blo
                v = c.validity[blo: blo + (n + 7) // 8 + 8].contiguous()
            cols.append(Column(c.data[lo: lo + n], v, c.c_type, c.arr_type, n))
        inv = [order.index(i) for i in range(len(order))]
        return Table(cols, list(part.names)).select(inv)

    def build_consume(self, table: Table, is_last: bool):
        import torch
        import torch.distributed as dist

        self.metrics["build_rows_in"] += table.n_rows
        if not self.build_parallel:
            return J.join_build_consume_batch(self.local, table, is_last)
        if table.n_rows or not self._build_batches:
            self._build_batches.append(to_device(table, self.device))
        if not is_last:
            return False, True
        whole = concat_device(self._build_batches, self.device) if len(self._build_batches) > 1 else self._build_batches[0]
        self._build_batches = []
        # broadcast decision (_join.cpp:3323-3336): both sides partitioned, global build size under the threshold (or forced);
        # a build-outer join keeps the partitioned form (every rank would emit the unmatched build rows otherwise)
        nbytes = sum(whole.n_rows * np_dtype_of(c.c_type).itemsize for c in whole.columns)
        g = torch.tensor([nbytes], dtype=torch.int64, device=torch.device("cuda", self.device))
        dist.all_reduce(g, group=self.group)
        if self.probe_parallel and not self.build_outer and (self.force_broadcast or int(g.item()) < bcast_join_threshold()):
            mine = all_gather_table(whole, self.device, self.group)
            self.is_broadcast = True
            self.metrics["broadcast"] = 1
        else:
            mine = self._shuffle(whole, self.build_key)
        self.metrics["build_rows_local"] = mine.n_rows
        res = J.join_build_consume_batch(self.local, mine, True)
        if self.use_filter and self.probe_parallel and not self.is_broadcast:
            self._build_global_filter()
        return res

    def _build_global_filter(self):
        """Union of the ranks' bloom filters (same block count everywhere) and the global key bounds."""
        import torch
        import torch.distributed as dist

        dev = torch.device("cuda", self.device)
        tot = torch.tensor([self.metrics["build_rows_local"]], dtype=torch.int64, device=dev)
        dist.all_reduce(tot, group=self.group)
        n_blocks = int(tot.item()) // 32 + 1
        words, (mn, mx) = J.build_runtime_filter(self.local, n_blocks)
        gathered = torch.empty(self.n_pes * words.numel(), dtype=words.dtype, device=dev)
        dist.all_gather_into_tensor(gathered, words, group=self.group)  # NCCL has no bitwise-or reduction
        acc = gathered.view(self.n_pes, -1)[0].clone()
        for r in range(1, self.n_pes):
            acc |= gathered.view(self.n_pes, -1)[r]
        words.copy_(acc)
        lo = torch.tensor([mn], dtype=torch.int64, device=dev)
        hi = torch.tensor([mx], dtype=torch.int64, device=dev)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=self.group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=self.group)
        _lib.check(_lib.lib().b200_join_set_key_bounds(self.local.handle, int(lo.item()), int(hi.item())), "runtime_join_filter")
        self.filter_ready = True
        self.metrics["filter"] = 1

    def probe_consume(self, table: Table, is_last: bool, produce_output: bool = True, used_cols=None):
        self.metrics["probe_rows_in"] += table.n_rows
        partitioned_build = self.build_parallel and not self.is_broadcast
        if partitioned_build and self.probe_parallel:
            if self.filter_ready and table.n_rows:
                table = J.runtime_join_filter((self,), to_device(table, self.device), (self.probe_key,))
                self.metrics["probe_rows_after_filter"] = self.metrics.get("probe_rows_after_filter", 0) + table.n_rows
            table = self._shuffle(table, self.probe_key)
        elif partitioned_build:
            table = self._owned_only(table, self.probe_key)
        self.metrics["probe_rows_local"] += table.n_rows
        return J.join_probe_consume_batch(self.local, table, is_last, produce_output, used_cols)
