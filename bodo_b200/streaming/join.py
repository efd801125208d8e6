"""Streaming hash join operator API — the host-side mirror of bodo/libs/streaming/join.py.

Same verbs and calling protocol as the reference (init_join_state :991-1100, join_build_consume_batch
:1270-1330, join_probe_consume_batch :1838-1950, delete_join_state :1959), so the reference's streaming join
test loops (bodo/tests/test_streaming/test_join.py) carry over.  The work happens in libbodo_b200.so.

Output column order is the reference's: kept build-table columns first, then kept probe-table columns
(both in logical input order, the key columns included on each side unless dropped through used/kept cols).

A join takes 1..4 integer / date key columns per side, the same number on both sides; key position j of the build side is
compared with key position j of the probe side, and both must have the same byte width.  Runtime join filters are built for
single-column keys only.
"""

from __future__ import annotations

from .. import _lib
from .._lib import ffi
from ..table import CTable, Table, table_from_ctable

MAX_KEYS = 4  # equi-join key columns per side (the C state's n_keys limit, as for the groupby and the shuffle)


class JoinState:
    def __init__(self, operator_id, build_key_inds, probe_key_inds, build_colnames, probe_colnames, build_outer, probe_outer,
                 output_batch_size, expected_build_rows, device, stream, is_na_equal=False, build_parallel=False, probe_parallel=False,
                 is_mark_join=False, is_anti_join=False):
        self.operator_id = int(operator_id)
        self.is_mark_join = bool(is_mark_join)
        self.is_anti_join = bool(is_anti_join)
        self.build_key_inds = tuple(int(k) for k in build_key_inds)
        self.probe_key_inds = tuple(int(k) for k in probe_key_inds)
        nk = len(self.build_key_inds)
        if not 1 <= nk <= MAX_KEYS or len(self.probe_key_inds) != nk:
            raise _lib.B200Error(f"Streaming Join: between 1 and {MAX_KEYS} equi-join keys per side, the same number on both sides, are "
                                 f"supported (got {nk} build and {len(self.probe_key_inds)} probe keys)")
        self.build_colnames = list(build_colnames) if build_colnames is not None else None
        self.probe_colnames = list(probe_colnames) if probe_colnames is not None else None
        self.build_outer = bool(build_outer)
        self.probe_outer = bool(probe_outer)
        self.is_na_equal = bool(is_na_equal)
        self.build_parallel = bool(build_parallel)
        self.probe_parallel = bool(probe_parallel)
        self.output_batch_size = int(output_batch_size)
        self.expected_build_rows = int(expected_build_rows)
        self.device = device
        self.stream = int(stream)
        self.handle = None
        self.build_schema = None  # (c_types, arr_types) of the physical (keys-first) build table
        self.build_indices = None
        self.probe_indices = None
        self.build_names = None
        self._out = None

    def _physical(self, table: Table, key_inds):
        others = [i for i in range(table.n_cols) if i not in key_inds]
        return list(key_inds) + others

    def _init_c(self, build: Table):
        """Create the C state at the first build batch (the probe schema is adopted from the first probe batch, so build
        batches go straight to the device and the build overlaps whatever produces them)."""
        L = _lib.lib()
        _lib.require_gpu()
        bct, bat = self.build_schema
        if self.device is None:
            import torch

            self.device = build.device if build.device >= 0 else torch.cuda.current_device()
        h = L.b200_join_state_init(self.operator_id, ffi.new("int8_t[]", bct), ffi.new("int8_t[]", bat), len(bct),
                                   ffi.NULL, ffi.NULL, 0, len(self.build_key_inds), int(self.build_outer), int(self.probe_outer), int(self.is_na_equal),
                                   self.output_batch_size, self.device, self.expected_build_rows, ffi.cast("void*", self.stream))
        self.handle = _lib.check_ptr(h, "init_join_state")
        if self.is_mark_join or self.is_anti_join:
            _lib.check(L.b200_join_set_kind(self.handle, int(self.is_mark_join), int(self.is_anti_join)), "init_join_state")


def init_join_state(operator_id, build_key_inds, probe_key_inds, build_colnames, probe_colnames, build_outer, probe_outer,
                    interval_build_columns=None, force_broadcast=False, op_pool_size_bytes=-1, non_equi_condition=None,
                    build_parallel=False, probe_parallel=False, *, output_batch_size=32768, expected_build_rows=0, device=None,
                    stream=0, is_na_equal=False, is_mark_join=False, is_anti_join=False) -> JoinState:
    """Mirror of bodo.libs.streaming.join.init_join_state (join.py:991-1100).  Interval joins and non-equi conditions are
    out of scope (SURVEY.md §2.1 row 3) and must be left at their defaults.

    `is_na_equal` is HashJoinState's option: False is what this door constructs in the reference (join_state_init_py_entry,
    _join.cpp:4087-4136: NA keys never match); the pandas door (bodo/pandas/physical/join.h:267, here PhysicalJoin / merge)
    passes True.  `build_parallel` / `probe_parallel` say that the side is row-distributed over the ranks of the default
    torch.distributed process group: non-owned rows are shuffled to hash_to_rank(key) before they reach the local join
    (_join.cpp:3243-3300), or — `force_broadcast`, or a build side below the broadcast threshold — the build side is
    all-gathered instead (:3317-3405)  (see bodo_b200/streaming/dist_join.py).

    `is_mark_join` (HashJoinState's ctor argument, _join.h:287) / `is_anti_join` (the probe's template argument, selected by the
    reference's planner for LEFT ANTI joins, bodo/pandas/physical/join.h:151): a mark join emits every probe row once, without
    build columns, plus a trailing boolean column that says whether the row has a match; an anti join emits the probe rows
    that have none."""
    if interval_build_columns not in (None, (), []) or non_equi_condition is not None:
        raise _lib.B200Error("Streaming Join: interval / non-equi joins are not supported by bodo_b200")
    g = lambda x: getattr(x, "meta", x)
    if build_parallel or probe_parallel:
        from .dist_join import DistJoinState

        return DistJoinState(operator_id, g(build_key_inds), g(probe_key_inds), g(build_colnames), g(probe_colnames), build_outer,
                             probe_outer, output_batch_size, expected_build_rows, device, stream, is_na_equal=is_na_equal,
                             build_parallel=build_parallel, probe_parallel=probe_parallel, force_broadcast=force_broadcast,
                             is_mark_join=is_mark_join, is_anti_join=is_anti_join)
    return JoinState(operator_id, g(build_key_inds), g(probe_key_inds), g(build_colnames), g(probe_colnames), build_outer,
                     probe_outer, output_batch_size, expected_build_rows, device, stream, is_na_equal=is_na_equal,
                     is_mark_join=is_mark_join, is_anti_join=is_anti_join)


def join_build_consume_batch(join_state: JoinState, table: Table, is_last: bool):
    """Mirror of join_build_consume_batch (join.py:1270-1330): returns (is_last, request_input)."""
    if hasattr(join_state, "build_consume"):  # sharded state (build_parallel / probe_parallel): dist_join.DistJoinState
        return join_state.build_consume(table, is_last)
    st = join_state
    if st.build_indices is None:
        st.build_indices = st._physical(table, st.build_key_inds)
        cols = [table.columns[i] for i in st.build_indices]
        st.build_schema = ([c.c_type for c in cols], [c.arr_type for c in cols])
        st.build_names = [table.names[i] for i in st.build_indices]
    phys = table.select(st.build_indices)
    if st.handle is None:
        st._init_c(phys)
    return _feed_build(st, phys, is_last), True


def _feed_build(st: JoinState, phys: Table, is_last: bool) -> bool:
    L = _lib.lib()
    ct = CTable(phys)
    req = ffi.new("int32_t*")
    rc = _lib.check(L.b200_join_build_consume_batch(st.handle, ct.ptr, int(bool(is_last)), req), "join_build_consume_batch")
    return bool(rc)


def join_probe_consume_batch(join_state: JoinState, table: Table, is_last: bool, produce_output: bool = True, used_cols=None):
    """Mirror of join_probe_consume_batch (join.py:1838-1950): returns (out_table, is_last, request_input).
    used_cols = (kept_build_cols, kept_probe_cols) as logical column indices, or None to keep everything."""
    if hasattr(join_state, "probe_consume"):
        return join_state.probe_consume(table, is_last, produce_output, used_cols)
    st = join_state
    L = _lib.lib()
    if st.build_indices is None or st.handle is None:
        raise _lib.B200Error("join_probe_consume_batch called before any build batch was consumed")
    if st.probe_indices is None:
        st.probe_indices = st._physical(table, st.probe_key_inds)
    phys = table.select(st.probe_indices)
    if used_cols is None:
        kb_logical = sorted(st.build_indices)
        kp_logical = sorted(st.probe_indices)
    else:
        kb_logical, kp_logical = list(used_cols[0]), list(used_cols[1])
    if st.is_mark_join:
        kb_logical = []  # a mark join does not output build table columns
    kb = [st.build_indices.index(i) for i in kb_logical]
    kp = [st.probe_indices.index(i) for i in kp_logical]
    names = [st.build_names[j] for j in kb] + [phys.names[j] for j in kp]
    # unique output names (a key named the same on both sides appears twice, like pandas' _x/_y without renaming)
    seen, uniq = set(), []
    for nm in names:
        cand, k = nm, 1
        while cand in seen:
            cand = f"{nm}_{k}"; k += 1
        seen.add(cand); uniq.append(cand)
    if st.is_mark_join:
        uniq.append("")  # the mark column is unnamed in the reference too (physical/join.h:317)
    ct = CTable(phys)
    ncols = len(kb) + len(kp) + (1 if st.is_mark_join else 0)
    st._out_cols = ffi.new("b200_column[]", max(ncols, 1))
    st._out = ffi.new("b200_table*")
    st._out.cols = st._out_cols
    total = ffi.new("int64_t*")
    out_last = ffi.new("int32_t*")
    _lib.check(L.b200_join_probe_consume_batch(st.handle, ct.ptr, ffi.new("uint64_t[]", kb or [0]), len(kb),
                                               ffi.new("uint64_t[]", kp or [0]), len(kp), st._out, total, int(bool(is_last)), out_last),
               "join_probe_consume_batch")
    out = table_from_ctable(st._out, ncols, uniq, owner=st)
    return out, bool(out_last[0]), True


def delete_join_state(join_state: JoinState) -> None:
    join_state = getattr(join_state, "local", join_state)
    if join_state.handle is not None:
        _lib.lib().b200_delete_join_state(join_state.handle)
        join_state.handle = None


def _require_single_key_filter(st: JoinState, key_idxs=(0,)) -> None:
    if len(st.build_key_inds) > 1 or len(key_idxs) > 1:
        raise _lib.B200Error(f"runtime_join_filter: multi-column runtime join filters are not built yet (this join has "
                             f"{max(len(st.build_key_inds), len(key_idxs))} key columns; single-column keys only)")


def build_runtime_filter(join_state, n_bloom_blocks: int = 0):
    """Build the bloom filter + key bounds of a finished build side; returns (bloom words as a device tensor aliasing the
    state's memory, (key_min, key_max)).  Sharded joins OR / min / max these across ranks (dist_join.DistJoinState does)."""
    import torch

    st = getattr(join_state, "local", join_state)
    _require_single_key_filter(st)
    L = _lib.lib()
    ptr = ffi.new("void**")
    nb = ffi.new("int64_t*")
    mm = ffi.new("int64_t[2]")
    _lib.check(L.b200_join_build_filter(st.handle, int(n_bloom_blocks), ptr, nb, mm), "runtime_join_filter")
    from ..table import DeviceArray

    words = torch.as_tensor(DeviceArray(int(ffi.cast("uintptr_t", ptr[0])), int(nb[0]) * 8, "int32", st.device, owner=st), device=torch.device("cuda", st.device))
    return words, (int(mm[0]), int(mm[1]))


def runtime_join_filter(join_states, table: Table, join_keys_idxs, process_col_bitmasks=None) -> Table:
    """Mirror of bodo.libs.streaming.join.runtime_join_filter (join.py:1392-1415; C++ HashJoinState::RuntimeFilter): drop the
    rows of `table` that cannot find a partner in the (finished) build sides of `join_states`.  join_keys_idxs[k] = (index of the
    column of `table` that corresponds to the join key of state k,), -1 = no such column (no filter for that state);
    process_col_bitmasks[k] = (apply the column-level min / max filter,).  The bloom filter is applied whenever the key column
    is present, as in the reference.  Device-resident tables only (host batches: bodo_b200.table.to_device first)."""
    import torch

    from ..expr import col
    from ..physical import filter_project_table

    for k, js in enumerate(join_states):
        _require_single_key_filter(getattr(js, "local", js), tuple(join_keys_idxs[k]))
    if table.device < 0:
        raise _lib.B200Error("runtime_join_filter: the table must be device resident")
    L = _lib.lib()
    dev = torch.device("cuda", table.device)
    keep_all = None
    for k, js in enumerate(join_states):
        st = getattr(js, "local", js)
        kc = int(join_keys_idxs[k][0])
        if kc < 0 or st.probe_outer:
            continue
        use_mm = True if process_col_bitmasks is None else bool(process_col_bitmasks[k][0])
        keep = torch.empty(table.n_rows + 8, dtype=torch.uint8, device=dev)
        ct = CTable(table)
        _lib.check(L.b200_join_runtime_filter(st.handle, ct.ptr, kc, int(use_mm), 1, ffi.cast("uint8_t*", keep.data_ptr())), "runtime_join_filter")
        keep_all = keep if keep_all is None else keep_all & keep
    if keep_all is None:
        return table
    return filter_project_table(table, keep_all[: table.n_rows])


def get_metric(join_state: JoinState, which: int) -> int:
    join_state = getattr(join_state, "local", join_state)
    return int(_lib.lib().b200_join_get_metric(join_state.handle, which))
