"""Physical-operator layer — the Python mirror of the reference's pipeline protocol ("door 2",
bodo/pandas/physical/operator.h:46-50,247-458; aggregate.h:65-365; join.h:58-744; _pipeline.cpp:389-466).

    OperatorResult.{NEED_MORE_INPUT, HAVE_MORE_OUTPUT, FINISHED}
    PhysicalReadPandas / PhysicalReadArrow / PhysicalReadParquet : sources (batches of host columns)
    PhysicalAggregate : sink of one pipeline (ConsumeBatch) and source of the next (ProduceBatch)
    PhysicalJoin      : sink for the build side, ProcessBatch for the probe side
    Pipeline          : while not finished: batch = source.ProduceBatch(); ... sink.ConsumeBatch(batch)

plus two helpers that run those pipelines over pandas frames the way bodo.pandas does for
`df.groupby(keys)[cols].agg(...)` and `left.merge(right, on=...)` (PhysicalReadPandas slices the frame into
STREAMING_BATCH_SIZE-row Arrow batches, bodo/pandas/physical/read_pandas.h:13-120).  All computation happens in
libbodo_b200.so; this module only moves batches between operators.
"""

from __future__ import annotations

import enum
from typing import Iterable, Sequence

from .streaming import groupby as G
from .streaming import join as J
from .table import Table

STREAMING_BATCH_SIZE = 32768  # bodo/libs/streaming/_shuffle.h:27-31


class OperatorResult(enum.Enum):
    NEED_MORE_INPUT = 0
    HAVE_MORE_OUTPUT = 1
    FINISHED = 2


class PhysicalReadPandas:
    """Source: slices a pandas DataFrame into batch_size-row batches (read_pandas.h:13-120)."""

    def __init__(self, df, batch_size: int = STREAMING_BATCH_SIZE):
        self.table = Table.from_pandas(df)
        self.batch_size = batch_size
        self.cur = 0

    def ProduceBatch(self):
        n = self.table.n_rows
        batch = self.table.slice(self.cur, self.cur + self.batch_size)
        self.cur += self.batch_size
        return batch, (OperatorResult.FINISHED if self.cur >= n else OperatorResult.HAVE_MORE_OUTPUT)


class PhysicalReadArrow:
    """Source over an in-memory pyarrow Table: batch_size-row zero-copy slices (the Arrow half of
    PhysicalReadPandas, read_pandas.h:13-120: the reference converts every pandas slice to Arrow first)."""

    def __init__(self, table, batch_size: int = STREAMING_BATCH_SIZE):
        self.arrow = table.combine_chunks()
        self.batch_size = batch_size
        self.cur = 0

    def ProduceBatch(self):
        n = self.arrow.num_rows
        batch = Table.from_arrow(self.arrow.slice(self.cur, self.batch_size))
        self.cur += self.batch_size
        return batch, (OperatorResult.FINISHED if self.cur >= n else OperatorResult.HAVE_MORE_OUTPUT)


class PhysicalReadParquet:
    """Source over a Parquet file or dataset directory (host side of physical/read_parquet.h:31-210 — the reference
    streams Arrow record batches out of its ParquetReader; here pyarrow's reader produces them).  Only the selected
    columns are decoded; every batch has at most batch_size rows; an empty dataset yields one empty, FINISHED batch."""

    def __init__(self, path: str, columns: Sequence[str] | None = None, batch_size: int = STREAMING_BATCH_SIZE):
        import pyarrow.dataset as ds

        self.dataset = ds.dataset(path, format="parquet")
        self.columns = list(columns) if columns is not None else None
        self.schema = self.dataset.schema
        self._it = iter(self.dataset.to_batches(columns=self.columns, batch_size=batch_size))
        self._next = self._pull()

    def _pull(self):
        for rb in self._it:
            if rb.num_rows:
                return rb
        return None

    def ProduceBatch(self):
        import pyarrow as pa

        cur = self._next
        if cur is None:  # empty dataset
            names = self.columns if self.columns is not None else list(self.schema.names)
            empty = pa.table({n: pa.array([], type=self.schema.field(n).type) for n in names})
            return Table.from_arrow(empty), OperatorResult.FINISHED
        self._next = self._pull()
        return Table.from_arrow(cur), (OperatorResult.FINISHED if self._next is None else OperatorResult.HAVE_MORE_OUTPUT)


def _infer_ctype(e, col_ctypes: dict) -> int:
    """Storage type of an expression's value: a bare column keeps its type, arithmetic is FLOAT64 as soon as a float (or a
    true division) is involved and INT64 otherwise, comparisons / logic are BOOL."""
    from .table import CTypes

    if e.op == "col":
        return col_ctypes[e.value]
    if e.op == "const_i64":
        return CTypes.INT64
    if e.op == "const_f64" or e.op in ("div", "to_f64"):
        return CTypes.FLOAT64
    if e.op in ("lt", "le", "gt", "ge", "eq", "ne", "and", "or", "not", "is_null"):
        return CTypes.BOOL
    if e.op == "to_i64":
        return CTypes.INT64
    kinds = [_infer_ctype(a, col_ctypes) for a in e.args]
    return CTypes.FLOAT64 if any(k in (CTypes.FLOAT64, CTypes.FLOAT32) for k in kinds) else CTypes.INT64


class PhysicalFilterProject:
    """Filter + projection in one device pass (bodo/pandas/physical/filter.h + project.h with their expression trees,
    expression.{h,cpp}): `predicate` (bodo_b200.expr.Expr or None) selects rows, `outputs` = [(name, Expr)] are the columns of
    the result (col("x") passes a column through).  Host batches are staged to the device first; the result is a device batch."""

    def __init__(self, predicate, outputs, device: int | None = None, stream: int = 0):
        self.predicate = predicate
        self.outputs = list(outputs)
        self.device = device
        self.stream = stream
        self._compiled = None

    def _compile(self, batch: Table):
        from . import _lib
        from .expr import compile_program

        col_index = {n: i for i, n in enumerate(batch.names)}
        col_ctypes = {n: c.c_type for n, c in zip(batch.names, batch.columns)}
        exprs = ([self.predicate] if self.predicate is not None else []) + [e for _, e in self.outputs]
        prog, starts = compile_program(exprs, col_index)
        ffi = _lib.ffi
        cprog = ffi.new("b200_expr_instr[]", len(prog))
        for i, (op, arg) in enumerate(prog):
            cprog[i].op = op
            cprog[i].arg = arg
        pred_start = starts[0] if self.predicate is not None else -1
        out_starts = starts[1:] if self.predicate is not None else starts
        out_ct = [_infer_ctype(e, col_ctypes) for _, e in self.outputs]
        self._compiled = (cprog, len(prog), pred_start, ffi.new("int32_t[]", out_starts or [0]), out_ct)

    def ProcessBatch(self, batch: Table, prev: OperatorResult):
        import torch

        from . import _lib
        from .table import to_device
        from .table import ArrTypes, Column, CTable, np_dtype_of

        dev_i = self.device if self.device is not None else (batch.device if batch.device >= 0 else torch.cuda.current_device())
        batch = to_device(batch, dev_i)
        if self._compiled is None:
            self._compile(batch)
        cprog, n_instr, pred_start, out_starts, out_ct = self._compiled
        dev = torch.device("cuda", dev_i)
        n = batch.n_rows
        cols = []
        for ct in out_ct:
            dt = getattr(torch, str(np_dtype_of(ct)))
            cols.append(Column(torch.empty(max(n, 1), dtype=dt, device=dev), torch.zeros((n + 31) // 32 * 4 + 8, dtype=torch.uint8, device=dev), ct,
                               ArrTypes.NULLABLE_INT_BOOL, n))
        out = Table(cols, [nm for nm, _ in self.outputs])
        cin, cout = CTable(batch), CTable(out)
        L, ffi = _lib.lib(), _lib.ffi
        kept = _lib.check(int(L.b200_filter_project(cin.ptr, cprog, n_instr, pred_start, out_starts, len(out_ct), cout.ptr, ffi.cast("void*", self.stream))),
                          "filter + projection")
        res = Table([Column(c.data[:kept], c.validity, c.c_type, c.arr_type, kept) for c in cols], list(out.names))
        return res, (OperatorResult.FINISHED if prev == OperatorResult.FINISHED else OperatorResult.NEED_MORE_INPUT)


def filter_project_table(table: Table, keep) -> Table:
    """Rows of a device-resident `table` whose entry in `keep` (uint8 device tensor, one byte per row) is non-zero, through the
    fused filter kernel (used by streaming.join.runtime_join_filter)."""
    from .expr import col
    from .table import ArrTypes, Column, CTypes

    ext = Table(list(table.columns) + [Column(keep, None, CTypes.BOOL, ArrTypes.NUMPY, table.n_rows)], list(table.names) + ["__keep"])
    op = PhysicalFilterProject(col("__keep"), [(n, col(n)) for n in table.names], device=table.device)
    out, _ = op.ProcessBatch(ext, OperatorResult.NEED_MORE_INPUT)
    return out


class PhysicalReadArrowDevice:
    """Source over an in-memory pyarrow Table that hands out DEVICE batches; string columns named in `dict_builders`
    ({column: DictionaryBuilder}) travel as dictionary ids unified against the builder (bodo_b200.dictionary), everything else
    as its fixed-width Arrow buffers (the H2D half of the reference's convertTableToGPU, bodo/pandas/physical/operator.cpp:293-380)."""

    def __init__(self, table, batch_size: int = STREAMING_BATCH_SIZE, device: int = 0, dict_builders: dict | None = None):
        self.arrow = table.combine_chunks()
        self.batch_size = batch_size
        self.device = device
        self.dict_builders = dict_builders or {}
        self.cur = 0

    def ProduceBatch(self):
        from .table import to_device

        n = self.arrow.num_rows
        sl = self.arrow.slice(self.cur, self.batch_size)
        self.cur += self.batch_size
        plain = [nm for nm in sl.schema.names if nm not in self.dict_builders]
        t = to_device(Table.from_arrow(sl.select(plain)), self.device) if plain else Table([], [])
        cols, names = [], []
        for nm in sl.schema.names:
            if nm in self.dict_builders:
                cols.append(self.dict_builders[nm].unify(sl.column(nm), self.device))
            else:
                cols.append(t.columns[plain.index(nm)])
            names.append(nm)
        return Table(cols, names), (OperatorResult.FINISHED if self.cur >= n else OperatorResult.HAVE_MORE_OUTPUT)


class PhysicalAggregate:
    """Groupby sink/source (aggregate.h:65-365). `aggs` = [(func_name, input_column_index or None for size)]."""

    def __init__(self, key_inds: Sequence[int], aggs: Sequence[tuple], dropna: bool = True, parallel: bool = False, **kw):
        fnames = tuple(f for f, _ in aggs)
        f_in_offsets, f_in_cols = [0], []
        for _, c in aggs:
            if c is not None:
                f_in_cols.append(c)
            f_in_offsets.append(len(f_in_cols))
        self.state = G.init_groupby_state(-1, tuple(key_inds), fnames, tuple(f_in_offsets), tuple(f_in_cols), parallel=parallel,
                                          dropna=dropna, **kw)
        self.finished_build = False

    def ConsumeBatch(self, batch: Table, prev: OperatorResult) -> OperatorResult:
        is_last = prev == OperatorResult.FINISHED
        global_last, _ = G.groupby_build_consume_batch(self.state, batch, is_last, True)
        self.finished_build = global_last
        return OperatorResult.FINISHED if global_last else OperatorResult.NEED_MORE_INPUT

    def ProduceBatch(self):
        out, last = G.groupby_produce_output_batch(self.state, True)
        return out, (OperatorResult.FINISHED if last else OperatorResult.HAVE_MORE_OUTPUT)

    def Finalize(self):
        G.delete_groupby_state(self.state)


def _key_tuple(keys) -> tuple:
    """One key (an int or a column name) or a sequence of them, as a tuple."""
    import numbers

    return (keys,) if isinstance(keys, (str, numbers.Integral)) else tuple(keys)


class PhysicalJoin:
    """Hash join: sink for build batches, ProcessBatch for probe batches (join.h:58-744).  `build_key` / `probe_key`: one column
    index or a sequence of 1..4 (a multi-column equi-join: position j of one side is compared with position j of the other)."""

    def __init__(self, build_key, probe_key, build_names, probe_names, how: str = "inner", **kw):
        build_outer = how in ("right", "outer")   # the build side is the RIGHT table (reference convention)
        probe_outer = how in ("left", "outer")
        if how == "anti":   # LEFT ANTI: probe rows without a partner (physical/join.h:151: no build columns in the output)
            kw["is_anti_join"] = True
        elif how == "mark":
            kw["is_mark_join"] = True
        kw.setdefault("is_na_equal", True)  # pandas merge semantics: NA joins NA (bodo/pandas/physical/join.h:267)
        bk, pk = tuple(int(k) for k in _key_tuple(build_key)), tuple(int(k) for k in _key_tuple(probe_key))
        self.state = J.init_join_state(-1, bk, pk, tuple(build_names), tuple(probe_names), build_outer, probe_outer, **kw)

    def ConsumeBatch(self, batch: Table, prev: OperatorResult) -> OperatorResult:
        is_last = prev == OperatorResult.FINISHED
        J.join_build_consume_batch(self.state, batch, is_last)
        return OperatorResult.FINISHED if is_last else OperatorResult.NEED_MORE_INPUT

    def ProcessBatch(self, batch: Table, prev: OperatorResult):
        is_last = prev == OperatorResult.FINISHED
        out, out_last, _ = J.join_probe_consume_batch(self.state, batch, is_last, True)
        return out, (OperatorResult.FINISHED if out_last else OperatorResult.NEED_MORE_INPUT)

    def Finalize(self):
        J.delete_join_state(self.state)


class ResultCollector:
    """PhysicalResultCollector: concatenates output batches into one pandas frame."""

    def __init__(self):
        self.frames = []

    def ConsumeBatch(self, batch: Table, prev: OperatorResult) -> OperatorResult:
        self.frames.append(batch.to_pandas())
        return OperatorResult.FINISHED if prev == OperatorResult.FINISHED else OperatorResult.NEED_MORE_INPUT

    def result(self):
        import pandas as pd

        return pd.concat(self.frames, ignore_index=True) if self.frames else pd.DataFrame()


def run_pipeline(source, between: Iterable, sink) -> None:
    """Pipeline::Execute (bodo/pandas/_pipeline.cpp:389-466): push batches source -> between ops -> sink."""
    finished = False
    while not finished:
        batch, res = source.ProduceBatch()
        for op in between:
            batch, res2 = op.ProcessBatch(batch, res)
            if res == OperatorResult.FINISHED and res2 != OperatorResult.FINISHED:
                res2 = OperatorResult.FINISHED
            res = res2
        sink.ConsumeBatch(batch, res)
        finished = res == OperatorResult.FINISHED


def groupby_agg(df, by, aggs: Sequence[tuple], dropna: bool = True, batch_size: int = STREAMING_BATCH_SIZE, **kw):
    """df.groupby(by, as_index=False, dropna=dropna).agg(...) through the streaming operators.

    aggs: [(out_name, column, func)] with func in {'sum','count','mean','min','max','size'}.
    Returns a pandas DataFrame (group order unspecified, as in the reference)."""
    by = [by] if isinstance(by, str) else list(by)
    cols = list(df.columns)
    used = list(by)
    for _, c, _ in aggs:
        if c is not None and c not in used:
            used.append(c)
    sub = df[used]
    key_inds = [used.index(k) for k in by]
    agg_spec = [(f, None if f == "size" or c is None else used.index(c)) for _, c, f in aggs]
    op = PhysicalAggregate(key_inds, agg_spec, dropna=dropna, **kw)
    run_pipeline(PhysicalReadPandas(sub, batch_size), [], op)
    coll = ResultCollector()
    run_pipeline(op, [], coll)
    op.Finalize()
    out = coll.result()
    out.columns = by + [name for name, _, _ in aggs]
    return out


def groupby_agg_parquet(path: str, by, aggs: Sequence[tuple], dropna: bool = True, batch_size: int = STREAMING_BATCH_SIZE, **kw):
    """bodo.pandas.read_parquet(path).groupby(by, as_index=False, dropna=dropna).agg(...): PhysicalReadParquet feeding
    PhysicalAggregate.  Only the key and aggregated columns are decoded (column pruning, as the reference's planner does
    for ReadParquet under an aggregate).  Same `aggs` format and result shape as groupby_agg."""
    by = [by] if isinstance(by, str) else list(by)
    used = list(by)
    for _, c, _ in aggs:
        if c is not None and c not in used:
            used.append(c)
    key_inds = [used.index(k) for k in by]
    agg_spec = [(f, None if f == "size" or c is None else used.index(c)) for _, c, f in aggs]
    op = PhysicalAggregate(key_inds, agg_spec, dropna=dropna, **kw)
    run_pipeline(PhysicalReadParquet(path, used, batch_size), [], op)
    coll = ResultCollector()
    run_pipeline(op, [], coll)
    op.Finalize()
    out = coll.result()
    out.columns = by + [name for name, _, _ in aggs]
    return out


def merge(left, right, left_on, right_on, how: str = "inner", batch_size: int = STREAMING_BATCH_SIZE, **kw):
    """left.merge(right, left_on=..., right_on=..., how=...) through the streaming join (right = build side).
    `left_on` / `right_on`: a column name or equally long lists of 1..4 names (a multi-column join).
    Output columns: right's columns then left's columns (the reference's build-then-probe order), renamed on clashes."""
    from ._lib import B200Error

    lon, ron = _key_tuple(left_on), _key_tuple(right_on)
    if len(lon) != len(ron):
        raise B200Error(f"merge: left_on and right_on must have the same length (got {len(lon)} and {len(ron)})")
    rcols, lcols = list(right.columns), list(left.columns)
    op = PhysicalJoin(tuple(rcols.index(c) for c in ron), tuple(lcols.index(c) for c in lon), rcols, lcols, how=how, **kw)
    run_pipeline(PhysicalReadPandas(right, batch_size), [], op)
    coll = ResultCollector()
    run_pipeline(PhysicalReadPandas(left, batch_size), [op], coll)
    op.Finalize()
    return coll.result()
