"""GPU parity tests for multi-column equi-join keys (2..4 key columns).

Reference: every distinct key tuple over both sides is mapped to a dense int64 id (groupby(..., dropna=False).ngroup(), so NA
and 0 stay distinct); under is_na_equal=False a row with an NA in any key column is marked invalid; the oracle's single-key
hash join then runs on the ids.  Where pandas can express the join (is_na_equal=True) the result is also compared with
DataFrame.merge.  Comparison: sorted row-set equality, bit-exact, over (validity, value) of every output column."""

import os
import socket

import numpy as np
import pandas as pd
import pytest
import torch

from bodo_b200.streaming.join import (delete_join_state, get_metric, init_join_state, join_build_consume_batch,
                                      join_probe_consume_batch)
from bodo_b200.table import CTypes, Table
from tests.helpers import table_to_device

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
I64_MIN = np.iinfo(np.int64).min


# ---- helpers -------------------------------------------------------------------------------------------------------------
def host_cols(t: Table):
    """[(values, valid)] of every column of a (host or device) table."""
    out = []
    for c in t.columns:
        m = c.valid_mask_numpy()
        out.append((np.asarray(c.values_numpy()).copy(), np.ones(c.length, bool) if m is None else m.copy()))
    return out


def frame_cols(df: pd.DataFrame):
    out = []
    for name in df.columns:
        s = df[name]
        if hasattr(s.array, "_mask"):
            out.append((np.asarray(s.array._data), ~np.asarray(s.array._mask)))
        else:
            v = s.to_numpy()
            out.append((v, ~np.isnan(v) if v.dtype.kind == "f" else np.ones(len(s), bool)))
    return out


def canon(cols):
    """(n_rows, 2 * n_cols) int64 matrix of (valid, value with NA -> 0) per column, rows sorted."""
    arrs = []
    for v, m in cols:
        v = np.asarray(v)
        v = v.astype(np.float64).view(np.int64) if v.dtype.kind == "f" else v.astype(np.int64)
        arrs += [m.astype(np.int64), np.where(m, v, 0)]
    mat = np.stack(arrs, axis=1)
    return mat[np.lexsort(mat.T[::-1])]


def assert_rowset_equal(got_cols, exp_cols):
    g, e = canon(got_cols), canon(exp_cols)
    assert g.shape == e.shape, (g.shape, e.shape)
    np.testing.assert_array_equal(g, e)


def key_values(t: Table, k: int):
    c = t.columns[k]
    m = c.valid_mask_numpy()
    m = np.ones(c.length, bool) if m is None else m
    return np.where(m, np.asarray(c.values_numpy()).astype(np.int64), 0), m


def ref_join(oracle, bt: Table, bk, pt: Table, pk, build_outer=False, probe_outer=False, is_na_equal=True):
    """(build_idx, probe_idx) of the join on the key tuples, -1 = NULL side."""
    nb, nk = bt.n_rows, len(bk)
    kf = {}
    for j in range(nk):
        bv, bm = key_values(bt, bk[j])
        pv, pm = key_values(pt, pk[j])
        kf[j] = pd.arrays.IntegerArray(np.concatenate([bv, pv]), ~np.concatenate([bm, pm]))
    kf = pd.DataFrame(kf)
    ids = kf.groupby(list(range(nk)), dropna=False, sort=False).ngroup().to_numpy(np.int64)
    valid = ~kf.isna().any(axis=1).to_numpy()
    bvalid, pvalid = (None, None) if is_na_equal else (valid[:nb], valid[nb:])
    return oracle.hash_join(ids[:nb], bvalid, ids[nb:], pvalid, build_outer, probe_outer, is_na_equal)


def take_cols(cols, idx):
    out = []
    for v, m in cols:
        if len(v) == 0:
            out.append((np.zeros(len(idx), v.dtype), np.zeros(len(idx), bool)))
            continue
        sel = np.where(idx >= 0, idx, 0)
        out.append((v[sel], m[sel] & (idx >= 0)))
    return out


def expected(bt, pt, bi, pi, kept_b=None, kept_p=None):
    bc, pc = host_cols(bt), host_cols(pt)
    kept_b = range(len(bc)) if kept_b is None else kept_b
    kept_p = range(len(pc)) if kept_p is None else kept_p
    return take_cols([bc[j] for j in kept_b], bi) + take_cols([pc[j] for j in kept_p], pi)


def run_join(bt, pt, bk, pk, build_outer=False, probe_outer=False, batch_size=None, to_device=False, used_cols=None, is_na_equal=True,
             **kind):
    """Streaming loop over build then probe batches; returns (output columns, metric 5 = fused probe batches)."""
    st = init_join_state(-1, bk, pk, tuple(bt.names), tuple(pt.names), build_outer, probe_outer, is_na_equal=is_na_equal, **kind)
    bs = batch_size or max(bt.n_rows, pt.n_rows, 1)
    it, last = 0, False
    while not last:
        b = bt.slice(it * bs, (it + 1) * bs)
        last = (it + 1) * bs >= bt.n_rows
        it += 1
        join_build_consume_batch(st, table_to_device(b) if to_device else b, last)
    parts, it, last = [], 0, False
    while not last:
        p = pt.slice(it * bs, (it + 1) * bs)
        last = (it + 1) * bs >= pt.n_rows
        it += 1
        out, _, _ = join_probe_consume_batch(st, table_to_device(p) if to_device else p, last, True, used_cols)
        parts.append(host_cols(out))  # the output aliases the state's buffers until the next call
    fused = get_metric(st, 5)
    delete_join_state(st)
    cols = [(np.concatenate([p[j][0] for p in parts]), np.concatenate([p[j][1] for p in parts])) for j in range(len(parts[0]))]
    return cols, fused


def as_date(t: Table, names):
    """Re-tag int32 columns as DATE (int32 days), the storage the join sees for date32 data."""
    for j, nm in enumerate(t.names):
        if nm in names:
            assert t.columns[j].c_type == CTypes.INT32
            t.columns[j].c_type = CTypes.DATE
    return t


# key dtypes per key count: every width (8, 4, 2, 1 bytes) and a date column appear
KEY_DTYPES = {2: ["Int64", "UInt8"], 3: ["date32", "UInt8", "Int16"], 4: ["Int64", "Int32", "Int16", "date32"]}
KEY_CARD = {"Int64": 25, "Int32": 4, "Int16": 3, "UInt8": 3, "date32": 3}


def make_sides(rng, nk, nb, npr, na_rate=0.04):
    """Build side: [k_{nk-1}, bpay, k_{nk-2}, ..., k_0]; probe side: [ppay, k_0, ..., k_{nk-1}, pf].  Keys sit at non-leading,
    differently ordered logical positions; tuples repeat on both sides (many-to-many); the first and last key columns have NAs."""
    dts = KEY_DTYPES[nk]

    def key(j, n):
        dt = dts[j]
        lo = -KEY_CARD[dt] // 2 if dt in ("Int64", "Int32", "Int16") else 0
        v = rng.integers(lo, lo + KEY_CARD[dt], n)
        s = pd.Series(pd.array(v, dtype="Int32" if dt == "date32" else dt))
        if j in (0, nk - 1):
            s[rng.random(n) < na_rate] = pd.NA
        return s

    bnames = [f"bk{nk - 1}", "bpay"] + [f"bk{j}" for j in range(nk - 2, -1, -1)]
    bdata = {f"bk{j}": key(j, nb) for j in range(nk)}
    bdata["bpay"] = pd.Series(pd.array(rng.integers(-(1 << 40), 1 << 40, nb), dtype="Int64"))
    bdata["bpay"][rng.random(nb) < 0.1] = pd.NA
    bdf = pd.DataFrame({n: bdata[n] for n in bnames})
    pnames = ["ppay"] + [f"pk{j}" for j in range(nk)] + ["pf"]
    pdata = {f"pk{j}": key(j, npr) for j in range(nk)}
    pdata["ppay"] = pd.Series(pd.array(rng.integers(0, 1 << 50, npr), dtype="Int64"))  # masked: pandas' outer merge keeps it integer
    pdata["pf"] = pd.Series(pd.array(rng.random(npr), dtype="Float64"))
    pdf = pd.DataFrame({n: pdata[n] for n in pnames})
    bk = tuple(bnames.index(f"bk{j}") for j in range(nk))
    pk = tuple(pnames.index(f"pk{j}") for j in range(nk))
    dates = {f"bk{j}" for j in range(nk) if dts[j] == "date32"} | {f"pk{j}" for j in range(nk) if dts[j] == "date32"}
    return bdf, pdf, bk, pk, as_date(Table.from_pandas(bdf), dates), as_date(Table.from_pandas(pdf), dates)


HOW = {"inner": (False, False), "left": (True, False), "right": (False, True), "outer": (True, True)}  # build.merge(probe, how)


# ---- join kinds ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nk", [2, 3, 4])
@pytest.mark.parametrize("is_na_equal", [False, True])
@pytest.mark.parametrize("to_device", [False, True])
@pytest.mark.parametrize("how", ["inner", "left", "right", "outer"])
def test_join_kinds_on_key_tuples(gpu_lib, oracle, nk, is_na_equal, to_device, how):
    rng = np.random.default_rng(100 * nk + 10 * is_na_equal + to_device)
    bdf, pdf, bk, pk, bt, pt = make_sides(rng, nk, 700, 1100)
    bo, po = HOW[how]
    got, _ = run_join(bt, pt, bk, pk, bo, po, batch_size=300, to_device=to_device, is_na_equal=is_na_equal)
    bi, pi = ref_join(oracle, bt, bk, pt, pk, bo, po, is_na_equal)
    assert_rowset_equal(got, expected(bt, pt, bi, pi))
    if is_na_equal:  # pandas merge: NA joins NA
        m = bdf.merge(pdf, left_on=[bdf.columns[k] for k in bk], right_on=[pdf.columns[k] for k in pk], how=how)
        assert_rowset_equal(got, frame_cols(m))
    assert len(got[0][0]) > 0


@pytest.mark.parametrize("is_na_equal", [False, True])
def test_tuple_comparison_is_column_by_column(gpu_lib, oracle, is_na_equal):
    """Tuples that share every column but one; (NA, 1) vs (0, 1) and (1, NA) vs (1, 0) never match; INT64_MIN and 0 as key
    values (INT64_MIN is the single-key table's free-slot value, an ordinary value for tuples)."""
    na = pd.NA
    b1 = pd.array([7, 7, 7, 7, na, 0, 1, 1, I64_MIN, 0, I64_MIN, 5], dtype="Int64")
    b2 = pd.array([0, 1, 2, 3, 1, 1, na, 0, 0, I64_MIN, I64_MIN, na], dtype="Int64")
    p1 = pd.array([7, 7, 7, 7, 7, 0, na, 1, 1, I64_MIN, 0, I64_MIN, 0, 5, 6], dtype="Int64")
    p2 = pd.array([3, 2, 9, 1, 0, 1, 1, 0, na, 0, I64_MIN, I64_MIN, 0, na, na], dtype="Int64")
    bdf = pd.DataFrame({"bv": np.arange(len(b1), dtype=np.int64), "b2": b2, "b1": b1})
    pdf = pd.DataFrame({"p1": p1, "p2": p2, "pv": np.arange(len(p1), dtype=np.int64) + 100})
    bt, pt = Table.from_pandas(bdf), Table.from_pandas(pdf)
    got, _ = run_join(bt, pt, (2, 1), (0, 1), is_na_equal=is_na_equal)
    bi, pi = ref_join(oracle, bt, (2, 1), pt, (0, 1), is_na_equal=is_na_equal)
    assert_rowset_equal(got, expected(bt, pt, bi, pi))
    pairs = {(int(b), int(p) - 100) for b, p in zip(got[0][0], got[5][0])}
    exp_pairs = {(0, 4), (1, 3), (2, 1), (3, 0), (5, 5), (7, 7), (8, 9), (9, 10), (10, 11)}
    if is_na_equal:
        exp_pairs |= {(4, 6), (6, 8), (11, 13)}  # (NA, 1) = (NA, 1); (1, NA) = (1, NA); (5, NA) = (5, NA)
    assert pairs == exp_pairs
    if is_na_equal:
        m = bdf.merge(pdf, left_on=["b1", "b2"], right_on=["p1", "p2"])
        assert_rowset_equal(got, frame_cols(m))


@pytest.mark.parametrize("is_na_equal", [False, True])
def test_concurrent_claims_of_one_tuple(gpu_lib, oracle, is_na_equal):
    """100 k build rows over 3 distinct tuples: every row races for the same three slots; per-tuple output counts are exact."""
    rng = np.random.default_rng(3)
    nb = 100_000
    which = rng.integers(0, 3, nb)
    k1 = pd.array(np.array([11, 11, 12])[which], dtype="Int64")
    k2 = pd.array(np.array([5, 6, 5])[which].astype(np.int32), dtype="Int32")
    k2[which == 2] = pd.NA  # the third tuple is (12, NA)
    bdf = pd.DataFrame({"k1": k1, "k2": k2, "row": np.arange(nb, dtype=np.int64)})
    pdf = pd.DataFrame({"k1": pd.array([11, 11, 12, 12, 11], dtype="Int64"), "k2": pd.array([5, 6, None, 5, 7], dtype="Int32")})
    bt, pt = Table.from_pandas(bdf), Table.from_pandas(pdf)
    got, fused = run_join(bt, pt, (0, 1), (0, 1), to_device=True, is_na_equal=is_na_equal)
    assert fused == 0
    counts = np.bincount(which, minlength=3)
    probe_tuple = got[3][0] * 100 + np.where(got[4][1], got[4][0], 99)
    assert len(probe_tuple) == counts[0] + counts[1] + (counts[2] if is_na_equal else 0)
    assert (probe_tuple == 1105).sum() == counts[0] and (probe_tuple == 1106).sum() == counts[1]
    assert (probe_tuple == 1299).sum() == (counts[2] if is_na_equal else 0)
    assert np.array_equal(np.sort(got[2][0][probe_tuple == 1105]), np.flatnonzero(which == 0))
    bi, pi = ref_join(oracle, bt, (0, 1), pt, (0, 1), is_na_equal=is_na_equal)
    assert_rowset_equal(got, expected(bt, pt, bi, pi))


# ---- fused probe for unique build tuples ----------------------------------------------------------------------------------
@pytest.mark.parametrize("is_na_equal", [False, True])
def test_unique_build_tuples_take_the_fused_probe(gpu_lib, oracle, is_na_equal):
    """Unique build tuples + inner join: join_probe_fast_mk_kernel (metric 5 counts its batches); duplicate tuples at the same
    size take the general path (metric 5 == 0).  Kept-column subsets and reordered probe columns included."""
    rng = np.random.default_rng(17)
    nb, npr = 200_000, 1_000_000
    perm = rng.permutation(nb).astype(np.int64)
    b2 = pd.array((perm % 7).astype(np.int32), dtype="Int32")
    b2[(perm % 7 == 3) & ((perm // 7) % 50 == 0)] = pd.NA  # (k1, NA) replaces (k1, 3): tuples stay unique
    build = pd.DataFrame({"b_pay": rng.integers(-(1 << 50), 1 << 50, nb), "k2": b2, "k1": perm // 7,
                          "b_small": rng.integers(-100, 100, nb).astype(np.int16)})
    pv = rng.integers(0, 2 * nb, npr)
    p2 = pd.array((pv % 7).astype(np.int32), dtype="Int32")
    p2[rng.random(npr) < 0.01] = pd.NA
    probe = pd.DataFrame({"k1": pv // 7, "p1": rng.random(npr), "k2": p2, "p_pay": rng.integers(0, 1 << 40, npr)})
    bt, pt = Table.from_pandas(build), Table.from_pandas(probe)
    bk, pk = (2, 1), (0, 2)
    bi, pi = ref_join(oracle, bt, bk, pt, pk, is_na_equal=is_na_equal)
    got, fused = run_join(bt, pt, bk, pk, batch_size=300_000, to_device=True, is_na_equal=is_na_equal)
    assert fused >= 1, "the fused multi-key probe was expected to run for unique build tuples"
    assert_rowset_equal(got, expected(bt, pt, bi, pi))
    assert len(got[0][0]) > 0.3 * npr
    used = ([2, 0], [3, 1])  # build: k1, b_pay; probe: p_pay, p1
    got2, fused2 = run_join(bt, pt, bk, pk, batch_size=300_000, to_device=True, used_cols=used, is_na_equal=is_na_equal)
    assert fused2 >= 1
    assert_rowset_equal(got2, expected(bt, pt, bi, pi, kept_b=[2, 0], kept_p=[3, 1]))
    # duplicate build tuples at the same size: general path
    dup = build.copy()
    dup.loc[::1000, "k1"] = dup.k1.iloc[1::1000].to_numpy()[: len(dup.loc[::1000])]
    dup.loc[::1000, "k2"] = dup.k2.iloc[1::1000].to_numpy()[: len(dup.loc[::1000])]
    dt = Table.from_pandas(dup)
    got3, fused3 = run_join(dt, pt, bk, pk, batch_size=300_000, to_device=True, is_na_equal=is_na_equal)
    assert fused3 == 0
    bi3, pi3 = ref_join(oracle, dt, bk, pt, pk, is_na_equal=is_na_equal)
    assert_rowset_equal(got3, expected(dt, pt, bi3, pi3))


# ---- anti / mark ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("is_na_equal", [False, True])
@pytest.mark.parametrize("to_device", [False, True])
def test_anti_and_mark_joins_on_two_keys(gpu_lib, oracle, is_na_equal, to_device):
    rng = np.random.default_rng(22)
    nb, npr = 5_000, 40_000
    build = pd.DataFrame({"k1": pd.array(rng.integers(0, 60, nb), dtype="Int64"), "b1": rng.integers(0, 100, nb),
                          "k2": pd.array(rng.integers(0, 50, nb).astype(np.int32), dtype="Int32")})
    build.loc[::300, "k1"] = pd.NA
    build.loc[::410, "k2"] = pd.NA
    probe = pd.DataFrame({"p1": rng.random(npr), "k2": pd.array(rng.integers(0, 60, npr).astype(np.int32), dtype="Int32"),
                          "k1": pd.array(rng.integers(0, 90, npr), dtype="Int64"), "p2": rng.integers(0, 1 << 40, npr)})
    probe.loc[::777, "k1"] = pd.NA
    probe.loc[::555, "k2"] = pd.NA
    bt, pt = Table.from_pandas(build), Table.from_pandas(probe)
    bk, pk = (0, 2), (2, 1)
    bi, pi = ref_join(oracle, bt, bk, pt, pk, is_na_equal=is_na_equal)
    has = np.zeros(npr, bool)
    has[pi] = True
    if is_na_equal:  # has a partner in pandas terms as well
        m = build[["k1", "k2"]].drop_duplicates().merge(probe.reset_index()[["index", "k1", "k2"]], on=["k1", "k2"])
        assert np.array_equal(np.sort(m["index"].to_numpy()), np.flatnonzero(has))
    anti, _ = run_join(bt, pt, bk, pk, batch_size=15_000, to_device=to_device, used_cols=([], [0, 1, 2, 3]), is_na_equal=is_na_equal,
                       is_anti_join=True)
    assert_rowset_equal(anti, take_cols(host_cols(pt), np.flatnonzero(~has)))
    mark, _ = run_join(bt, pt, bk, pk, batch_size=15_000, to_device=to_device, used_cols=([], [0, 1, 2, 3]), is_na_equal=is_na_equal,
                       is_mark_join=True)
    assert len(mark) == 5 and len(mark[4][0]) == npr
    # a mark join keeps the probe rows in order: row i of the output is probe row i
    np.testing.assert_array_equal(mark[4][0].astype(bool), has)
    np.testing.assert_array_equal(mark[3][0], probe.p2.to_numpy())


# ---- pandas door -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("how", ["inner", "left", "right", "outer"])
def test_physical_merge_with_key_lists_matches_pandas(gpu_lib, how):
    from bodo_b200.physical import merge

    rng = np.random.default_rng(31)
    left = pd.DataFrame({"x": pd.array(rng.random(3000), dtype="Float64"), "a": pd.array(rng.integers(0, 30, 3000), dtype="Int64"),
                         "b": pd.array(rng.integers(0, 4, 3000).astype(np.int32), dtype="Int32")})
    left.loc[::97, "a"] = pd.NA
    right = pd.DataFrame({"c": pd.array(rng.integers(0, 40, 400), dtype="Int64"), "y": pd.array(rng.integers(0, 1000, 400), dtype="Int64"),
                          "d": pd.array(rng.integers(0, 4, 400).astype(np.int32), dtype="Int32")})
    right.loc[::31, "c"] = pd.NA
    got = merge(left, right, left_on=["a", "b"], right_on=["c", "d"], how=how, batch_size=512)
    exp = right.merge(left, left_on=["c", "d"], right_on=["a", "b"], how={"left": "right", "right": "left"}.get(how, how))
    assert list(got.columns) == ["c", "y", "d", "x", "a", "b"]
    assert_rowset_equal(frame_cols(got), frame_cols(exp))
    # a single-key merge through the same door is unchanged
    got1 = merge(left, right, left_on="a", right_on="c", how=how, batch_size=512)
    exp1 = right.merge(left, left_on="c", right_on="a", how={"left": "right", "right": "left"}.get(how, how))
    assert_rowset_equal(frame_cols(got1), frame_cols(exp1))


def _run_physical_join(build_src, probe_src, bk, pk, build_names, probe_names):
    from bodo_b200.physical import PhysicalJoin, ResultCollector, run_pipeline

    op = PhysicalJoin(bk, pk, build_names, probe_names)
    run_pipeline(build_src, [], op)
    coll = ResultCollector()
    run_pipeline(probe_src, [op], coll)
    op.Finalize()
    return coll.result()


def test_dictionary_encoded_string_tuple_keys_on_the_tpch_fixture(gpu_lib):
    """lineitem (probe) joined with a small dimension table on (L_RETURNFLAG, L_LINESTATUS): both string keys travel as ids
    unified against one DictionaryBuilder per key column; decoded, the rows equal pandas' merge on the strings.  Then
    (L_ORDERKEY int32, L_SHIPDATE date32) against a table derived from lineitem."""
    import pyarrow as pa
    import pyarrow.parquet as pq

    from bodo_b200.dictionary import DictionaryBuilder
    from bodo_b200.physical import PhysicalReadArrow, PhysicalReadArrowDevice

    at = pq.read_table(os.path.join(GOLDEN, "tpch_q1_lineitem.parquet"))
    li = at.select(["L_RETURNFLAG", "L_LINESTATUS", "L_ORDERKEY", "L_QUANTITY"])
    dim = pa.table({"RF": ["N", "A", "R", "N", "N", "Z"], "LS": ["O", "F", "F", "F", "O", "O"], "w": np.arange(6, dtype=np.int64)})
    builders = {"RF": DictionaryBuilder(), "LS": DictionaryBuilder()}
    builders["L_RETURNFLAG"], builders["L_LINESTATUS"] = builders["RF"], builders["LS"]  # one shared builder per key column
    got = _run_physical_join(PhysicalReadArrowDevice(dim, 4, 0, {"RF": builders["RF"], "LS": builders["LS"]}),
                             PhysicalReadArrowDevice(li, 8192, 0, {"L_RETURNFLAG": builders["RF"], "L_LINESTATUS": builders["LS"]}),
                             (0, 1), (0, 1), dim.schema.names, li.schema.names)
    dec = {0: builders["RF"], 1: builders["LS"], 3: builders["RF"], 4: builders["LS"]}
    got = pd.DataFrame({j: dec[j].decode(got.iloc[:, j].to_numpy(dtype="int64")) if j in dec else got.iloc[:, j] for j in range(got.shape[1])})
    exp = dim.to_pandas().merge(li.to_pandas(), left_on=["RF", "LS"], right_on=["L_RETURNFLAG", "L_LINESTATUS"])
    rows = lambda df: sorted(map(tuple, df.astype(object).itertuples(index=False, name=None)))
    assert len(got) == len(exp) > 0
    assert rows(got) == rows(exp)
    # (int32, date32) keys: a derived table of distinct (orderkey, shipdate) pairs of every 7th row, with a payload
    lp = at.select(["L_ORDERKEY", "L_SHIPDATE", "L_QUANTITY"]).to_pandas()
    der = lp.iloc[::7, :2].drop_duplicates().reset_index(drop=True)
    der["pay"] = np.arange(len(der), dtype=np.int64)
    der_at = pa.Table.from_pandas(der, schema=pa.schema([("L_ORDERKEY", pa.int32()), ("L_SHIPDATE", pa.date32()), ("pay", pa.int64())]),
                                  preserve_index=False)
    got2 = _run_physical_join(PhysicalReadArrow(der_at, 1000), PhysicalReadArrow(at.select(["L_ORDERKEY", "L_SHIPDATE", "L_QUANTITY"]), 4096),
                              (0, 1), (0, 1), der_at.schema.names, ["L_ORDERKEY", "L_SHIPDATE", "L_QUANTITY"])
    exp2 = der.merge(lp, on=["L_ORDERKEY", "L_SHIPDATE"])
    norm = lambda s: pd.to_datetime(s).dt.strftime("%Y-%m-%d") if s.dtype.kind in "MO" else s.astype("float64")
    g2 = pd.DataFrame({i: norm(got2.iloc[:, i]) for i in range(got2.shape[1])})
    e2 = exp2[["L_ORDERKEY", "L_SHIPDATE", "pay", "L_ORDERKEY", "L_SHIPDATE", "L_QUANTITY"]]
    e2 = pd.DataFrame({i: norm(e2.iloc[:, i]) for i in range(e2.shape[1])})
    assert len(g2) == len(e2) >= len(der)
    assert rows(g2) == rows(e2)


# ---- sharded ---------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _mk_join_worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from bodo_b200.shuffle import hash_keys_table
        from oracle import oracle as O

        rng = np.random.default_rng(78)  # same global tables on every rank; each rank feeds its own row slice
        nb, npr = 30_000, 120_000
        build = pd.DataFrame({"b1": rng.integers(0, 1 << 40, nb), "k2": pd.array(rng.integers(0, 40, nb).astype(np.int32), dtype="Int32"),
                              "k1": rng.integers(0, 2_000, nb).astype(np.int64)})
        build.loc[rng.random(nb) < 0.05, "k2"] = pd.NA
        probe = pd.DataFrame({"k1": rng.integers(0, 3_000, npr).astype(np.int64), "p1": rng.integers(0, 1 << 40, npr),
                              "k2": pd.array(rng.integers(0, 40, npr).astype(np.int32), dtype="Int32")})
        probe.loc[rng.random(npr) < 0.05, "k2"] = pd.NA
        bk, pk = (2, 1), (0, 2)
        gb, gp = Table.from_pandas(build), Table.from_pandas(probe)
        results = {}
        for name, kw, bo, po in (("shuffle", {}, False, False), ("shuffle-outer", {}, True, True),
                                 ("broadcast", {"force_broadcast": True}, False, True)):
            os.environ["BODO_BCAST_JOIN_THRESHOLD"] = "0" if name != "broadcast" else str(10 << 20)
            st = init_join_state(-1, bk, pk, tuple(build.columns), tuple(probe.columns), bo, po, build_parallel=True,
                                 probe_parallel=True, device=rank, is_na_equal=True, **kw)
            bchunk, pchunk = (nb + world - 1) // world, (npr + world - 1) // world
            mb = gb.slice(rank * bchunk, min((rank + 1) * bchunk, nb))
            mp_ = gp.slice(rank * pchunk, min((rank + 1) * pchunk, npr))
            half = mb.n_rows // 2
            join_build_consume_batch(st, mb.slice(0, half), False)
            join_build_consume_batch(st, mb.slice(half, mb.n_rows), True)
            parts, misplaced = [], 0
            cuts = [0, mp_.n_rows // 3, mp_.n_rows]
            for b in range(2):
                out, _, _ = join_probe_consume_batch(st, mp_.slice(cuts[b], cuts[b + 1]), b == 1, True)
                parts.append(host_cols(out))
                if name != "broadcast" and out.n_rows:  # every build row sits on hash_keys(k1, k2) % n_pes
                    _, dest = hash_keys_table(out.select([2, 1]), 2, world)
                    present = parts[-1][0][1]  # b1 is non-null: False only on NULL-extended rows
                    misplaced += int((dest.cpu().numpy()[present] != rank).sum())
            met = dict(st.metrics)
            delete_join_state(st)
            got = [(np.concatenate([p[j][0] for p in parts]), np.concatenate([p[j][1] for p in parts])) for j in range(len(parts[0]))]
            allg, allm, allp = [None] * world, [None] * world, [None] * world
            dist.all_gather_object(allg, got)
            dist.all_gather_object(allm, met)
            dist.all_gather_object(allp, misplaced)
            if rank == 0:
                union = [(np.concatenate([g[j][0] for g in allg]), np.concatenate([g[j][1] for g in allg])) for j in range(len(got))]
                bi, pi = ref_join(O, gb, bk, gp, pk, bo, po, True)
                g, e = canon(union), canon(expected(gb, gp, bi, pi))
                ok = g.shape == e.shape and bool(np.array_equal(g, e))
                kf = table_to_device(gb.select([2, 1]), rank)
                _, gdest = hash_keys_table(kf, 2, world)
                owners = np.bincount(gdest.cpu().numpy(), minlength=world).tolist()
                local = [m["build_rows_local"] for m in allm]
                results[name] = (ok, [m["broadcast"] for m in allm], [m.get("filter", 0) for m in allm], sum(allp),
                                 local == owners if name != "broadcast" else local == [nb] * world)
        q.put((rank, results))
    except Exception:
        import traceback

        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_sharded_two_key_join_shuffle_and_broadcast_nccl(gpu_lib):
    """build_parallel / probe_parallel with (int64, int32) keys: rows go to hash_keys(tuple) % n_pes (the reference's hash_keys,
    which b200_shuffle_partition computes), or the build side is all-gathered; the union of the ranks' outputs equals the
    reference join of the global tables, and no bloom filter is built for the tuple keys."""
    import torch.multiprocessing as mp

    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_mk_join_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=500) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for r in res:
        assert isinstance(r[1], dict), r
    r0 = [r for r in res if r[0] == 0][0][1]
    for name, bcast in (("shuffle", 0), ("shuffle-outer", 0), ("broadcast", 1)):
        ok, bc, filt, misplaced, placed = r0[name]
        assert ok, name
        assert bc == [bcast] * world and filt == [0] * world and misplaced == 0 and placed, (name, r0[name])
