"""CPU tests (no GPU): pin the oracle against the committed golden vectors of the reference's own tests and against
the reference's vendored xxHash known-answer vectors."""

import json
import os

import numpy as np
import pandas as pd
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    return json.load(open(os.path.join(GOLD, name)))


def _col(vals, dtype):
    arr = np.array([0 if v is None else v for v in vals], dtype=dtype)
    valid = np.array([v is not None for v in vals], dtype=bool)
    return arr, (None if valid.all() else valid)


@pytest.mark.parametrize("case", _load("groupby.json")["cases"], ids=lambda c: c["name"])
def test_oracle_groupby_matches_reference_goldens(oracle, case):
    is_float = any(isinstance(v, float) for v in case["val"])
    key, kvalid = _col(case["key"], np.int64)
    val, vvalid = _col(case["val"], np.float64 if is_float else np.int64)
    f = case["func"]
    r = oracle.groupby(key, kvalid, [f], [val], [vvalid], dropna=case["dropna"], batch_size=3)
    exp = case["expected"]
    ecols = list(exp.keys())
    ekey, eval_ = exp[ecols[0]], exp[ecols[1]]
    got = {}
    for k, kv, d, dv in zip(r["keys"], r["key_valid"], r["cols"][0][0], r["cols"][0][1]):
        got[int(k) if kv else None] = (float(d) if d.dtype.kind == "f" else int(d)) if dv else None
    assert set(got) == set(ekey)
    for k, e in zip(ekey, eval_):
        g = got[k]
        if e is None or (isinstance(e, float) and np.isnan(e)):
            assert g is None or (isinstance(g, float) and np.isnan(g)), (k, g, e)
        elif isinstance(e, float):
            assert g == pytest.approx(e, rel=1e-12, abs=0), (k, g, e)
        else:
            assert g == e, (k, g, e)


@pytest.mark.parametrize("case", _load("join.json")["cases"], ids=lambda c: c["name"])
def test_oracle_join_matches_reference_goldens(oracle, case):
    def keys(spec):
        if isinstance(spec, str):
            return np.arange(int(spec.split(":")[1]), dtype=np.int64)
        return np.array(spec, dtype=np.int64)
    bk, pk = keys(case["build_key"]), keys(case["probe_key"])
    bi, pi = oracle.hash_join(bk, None, pk, None, case["build_outer"], case["probe_outer"], True)
    assert len(bi) == case["n_rows"]
    ksum = int(bk[bi[bi >= 0]].sum() + pk[pi[pi >= 0]].sum())
    assert ksum == case["key_sum"]
    m = (bi >= 0) & (pi >= 0)
    assert (bk[bi[m]] == pk[pi[m]]).all()


def test_oracle_hash_matches_reference_known_answers(oracle):
    L = oracle.lib()
    for vec in _load("xxh3_hash_inner_32.json")["vectors"]:
        seed = vec["seed"]
        for k, h in zip(vec["keys64"], vec["hash64"]):
            assert L.oracle_hash_inner_32_i64(k, seed) == h
        for k, h in zip(vec["keys32"], vec["hash32"]):
            assert L.oracle_hash_inner_32_i32(k, seed) == h


def test_oracle_groupby_vs_pandas_random(oracle):
    rng = np.random.default_rng(0)
    n = 50_000
    k = rng.integers(0, 500, n).astype(np.int64)
    vi = rng.integers(-1000, 1000, n).astype(np.int64)
    vf = rng.random(n)
    vf[rng.random(n) < 0.05] = np.nan
    df = pd.DataFrame({"k": k, "vi": vi, "vf": vf})
    r = oracle.groupby(k, None, ["sum", "count", "min", "max", "mean", "sum", "count", "size"], [vi, vi, vi, vi, vi, vf, vf, vi], batch_size=977)
    o = pd.DataFrame({"k": r["keys"], **{f"f{j}": c[0] for j, c in enumerate(r["cols"])}}).sort_values("k").reset_index(drop=True)
    g = df.groupby("k")
    np.testing.assert_array_equal(o.f0, g.vi.sum().to_numpy())
    np.testing.assert_array_equal(o.f1, g.vi.count().to_numpy())
    np.testing.assert_array_equal(o.f2, g.vi.min().to_numpy())
    np.testing.assert_array_equal(o.f3, g.vi.max().to_numpy())
    np.testing.assert_allclose(o.f4, g.vi.mean().to_numpy(), rtol=1e-12)
    np.testing.assert_allclose(o.f5, g.vf.sum().to_numpy(), rtol=1e-9)
    np.testing.assert_array_equal(o.f6, g.vf.count().to_numpy())
    np.testing.assert_array_equal(o.f7, g.size().to_numpy())


def test_oracle_sharded_groupby_partitions_groups(oracle):
    # the union over ranks of the sharded oracle equals the single-rank oracle; every key sits on hash_to_rank(key)
    k, v = oracle.synth_fill(0, 100_000, 3000, 5)
    full = oracle.groupby(k, None, ["sum", "count"], [v, v])
    seen = {}
    for rank in range(4):
        part = oracle.groupby(k, None, ["sum", "count"], [v, v], n_pes=4, rank=rank)
        dest = oracle.hash_to_rank(part["keys"], None, 4)
        assert (dest == rank).all()
        for kk, s, c in zip(part["keys"], part["cols"][0][0], part["cols"][1][0]):
            assert kk not in seen
            seen[int(kk)] = (int(s), int(c))
    assert seen == {int(kk): (int(s), int(c)) for kk, s, c in zip(full["keys"], full["cols"][0][0], full["cols"][1][0])}


def test_oracle_mt_baseline_matches_single_thread(oracle):
    k, v = oracle.synth_fill(0, 300_000, 10_000, 9)
    ng, cs = oracle.groupby_sum_count_mt(k, v, 4, batch=4096)
    assert ng == len(np.unique(k))
    assert cs[1] == len(k) and cs[0] == int(v.sum()) % (1 << 64)


def test_synth_generators_agree(oracle):
    from bodo_b200 import synth
    k1, v1 = oracle.synth_fill(12345, 10_000, 777, 3)
    k2, v2 = synth.numpy_fill(12345, 10_000, 777, 3)
    np.testing.assert_array_equal(k1, k2)
    np.testing.assert_array_equal(v1, v2)


# ---- multi-column / float key hashing (SURVEY.md §8 a2) ---------------------------------------------------------------
def test_py_hash_double_matches_the_interpreter(oracle):
    # the reference hashes float keys through CPython's _Py_HashDouble (bodo/libs/_array_hash.cpp:119-170); the oracle's
    # restatement is pinned against hash(float) of the interpreter running the tests (same algorithm since 3.2; NaN
    # hashes by identity since 3.10 and the reference passes a NULL identity -> 0)
    import math
    import random
    import struct

    L = oracle.lib()
    vals = [0.0, -0.0, 1.0, -1.0, 0.5, 1e300, -1e300, 1e-300, 5e-324, float("inf"), float("-inf"), math.pi, 2.0**61, 2.0**61 - 1,
            2.0**62 + 12345.0, -7.25, 1 / 3, 123456789.0, -2.0**31]
    rnd = random.Random(7)
    vals += [rnd.uniform(-1e6, 1e6) for _ in range(500)]
    vals += [struct.unpack("<d", struct.pack("<Q", rnd.getrandbits(64)))[0] for _ in range(3000)]
    for v in vals:
        if math.isnan(v):
            assert L.oracle_py_hash_double(v) == 0
        else:
            assert L.oracle_py_hash_double(v) == hash(v), v
    assert L.oracle_py_hash_double(float("nan")) == 0
    # float key hash = hash_inner_32 of that Py_hash_t
    assert L.oracle_hash_inner_32_f64(2.5, 0xB0D01289) == L.oracle_hash_inner_32_i64(hash(2.5), 0xB0D01289)


def test_hash_combine_boost_is_one_murmur3_round(oracle):
    # hash_combine_boost (bodo/libs/_array_hash.cpp:41-56) is the body round of MurmurHash3_x86_32: seed -> one 4-byte
    # block -> finalizer must reproduce the published MurmurHash3 verification vectors
    L = oracle.lib()

    def fmix32(h):
        h ^= h >> 16
        h = (h * 0x85EBCA6B) & 0xFFFFFFFF
        h ^= h >> 13
        h = (h * 0xC2B2AE35) & 0xFFFFFFFF
        return h ^ (h >> 16)

    def murmur3_one_block(k1, seed):
        return fmix32(L.oracle_hash_combine_boost(seed, k1) ^ 4)

    assert murmur3_one_block(0xFFFFFFFF, 0) == 0x76293B50
    assert murmur3_one_block(0x87654321, 0) == 0xF55B516B
    assert murmur3_one_block(0x87654321, 0x5082EDEE) == 0x2362F9DE


def test_hash_keys_first_column_hashed_rest_combined(oracle):
    rng = np.random.default_rng(2)
    k0, k1, k2 = (rng.integers(-2**40, 2**40, 1000) for _ in range(3))
    v1 = rng.random(1000) > 0.1
    L = oracle.lib()
    seed = oracle.SEED_HASH_PARTITION
    one = oracle.hash_keys([k0])
    assert [int(x) for x in one[:50]] == [L.oracle_hash_inner_32_i64(int(x), seed) for x in k0[:50]]
    three = oracle.hash_keys([k0, k1, k2], [None, v1, None])
    na = L.oracle_hash_inner_32_i64(1, seed)
    for i in range(0, 1000, 37):
        h = L.oracle_hash_inner_32_i64(int(k0[i]), seed)
        h = L.oracle_hash_combine_boost(h, L.oracle_hash_inner_32_i64(int(k1[i]), seed) if v1[i] else na)
        h = L.oracle_hash_combine_boost(h, L.oracle_hash_inner_32_i64(int(k2[i]), seed))
        assert int(three[i]) == h
    # column order matters (the combine is not commutative), equal rows hash equally
    assert not np.array_equal(oracle.hash_keys([k0, k1]), oracle.hash_keys([k1, k0]))
    assert np.array_equal(oracle.hash_keys([k0[:10], k1[:10]]), oracle.hash_keys([k0[:10].copy(), k1[:10].copy()]))
