"""GPU parity tests for the row->rank radix partition: placement identical to the reference's
hash_to_rank(XXH3(key, SEED_HASH_PARTITION)) and bit-identical stable scatter versus the oracle."""

import json
import os

import numpy as np
import pandas as pd
import pytest
import torch

from bodo_b200 import _lib
from bodo_b200._lib import ffi
from bodo_b200.shuffle import partition_device
from bodo_b200.table import CTable, Table
from tests.helpers import table_to_device

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _device_hash_to_rank(gpu_lib, keys, n_pes):
    t = table_to_device(Table.from_pandas(pd.DataFrame({"k": keys})))
    dest = torch.empty(len(keys), dtype=torch.int32, device="cuda")
    ct = CTable(t)  # keep the cffi structs alive for the duration of the call
    _lib.check(gpu_lib.b200_hash_to_rank(ct.ptr, n_pes, ffi.cast("int32_t*", dest.data_ptr()), ffi.NULL))
    return dest.cpu().numpy()


@pytest.mark.parametrize("n_pes", [1, 2, 3, 8, 64])
@pytest.mark.parametrize("key_dtype", [np.int64, np.int32])
def test_hash_to_rank_matches_reference_placement(gpu_lib, oracle, n_pes, key_dtype):
    rng = np.random.default_rng(0)
    keys = rng.integers(np.iinfo(key_dtype).min, np.iinfo(key_dtype).max, 100_003).astype(key_dtype)
    got = _device_hash_to_rank(gpu_lib, keys, n_pes)
    if key_dtype == np.int64:
        np.testing.assert_array_equal(got, oracle.hash_to_rank(keys, None, n_pes))
    L = oracle.lib()
    f = L.oracle_hash_inner_32_i64 if key_dtype == np.int64 else L.oracle_hash_inner_32_i32
    np.testing.assert_array_equal(got[:5000], [f(int(k), oracle.SEED_HASH_PARTITION) % n_pes for k in keys[:5000]])
    # the reference's own vendored xxHash: its known-answer vectors for the partition seed
    width = "64" if key_dtype == np.int64 else "32"
    vec = next(v for v in json.load(open(os.path.join(GOLDEN, "xxh3_hash_inner_32.json")))["vectors"]
               if v["seed"] == oracle.SEED_HASH_PARTITION)
    got = _device_hash_to_rank(gpu_lib, np.array(vec["keys" + width], dtype=key_dtype), n_pes)
    np.testing.assert_array_equal(got, np.array(vec["hash" + width], dtype=np.uint64) % n_pes)


@pytest.mark.parametrize("n_pes", [2, 8, 5])
@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 100_000, 1_000_001])
def test_partition_bit_identical_to_oracle(gpu_lib, oracle, n_pes, n):
    rng = np.random.default_rng(n + n_pes)
    keys = rng.integers(0, 1 << 40, n).astype(np.int64)
    valid = rng.random(n) > 0.05
    df = pd.DataFrame({"k": pd.array(keys, dtype="Int64"), "a": rng.random(n), "b": rng.integers(-5, 5, n).astype(np.int32),
                       "c": pd.array(rng.integers(0, 100, n), dtype="Int64")})
    df.loc[~valid, "k"] = pd.NA
    df.loc[rng.random(n) < 0.1, "c"] = pd.NA
    t = Table.from_pandas(df)
    part, counts, perm = partition_device(table_to_device(t), 1, n_pes, want_perm=True)
    ecounts, eperm = oracle.shuffle_partition(keys, valid, n_pes)
    assert counts == list(ecounts)
    np.testing.assert_array_equal(perm.cpu().numpy(), eperm)
    # every column (and its per-destination re-packed bitmap) equals the oracle's permutation of the input
    for ci, c in enumerate(t.columns):
        np.testing.assert_array_equal(part.columns[ci].data.cpu().numpy(), c.data[eperm])
        if c.validity is not None:
            mask = c.valid_mask_numpy()[eperm]
            bm = part.columns[ci].validity.cpu().numpy()
            off_rows, off_bytes = 0, 0
            for cnt in counts:
                seg = np.unpackbits(bm[off_bytes: off_bytes + (cnt + 7) // 8], bitorder="little")[:cnt].astype(bool)
                np.testing.assert_array_equal(seg, mask[off_rows: off_rows + cnt])
                off_rows += cnt
                off_bytes += (cnt + 7) // 8


@pytest.mark.parametrize("counts", [[5], [0, 9, 0], [8, 8, 8], [1, 31, 32, 33, 0, 70001], [3] * 64])
def test_merge_segment_bitmaps(gpu_lib, counts):
    from bodo_b200.shuffle import merge_segment_bitmaps
    rng = np.random.default_rng(sum(counts))
    masks = [rng.random(c) > 0.4 for c in counts]
    segs = [np.packbits(m, bitorder="little") for m in masks]
    buf = np.concatenate(segs + [np.zeros(8, dtype=np.uint8)])
    out = merge_segment_bitmaps(torch.from_numpy(buf).cuda(), counts).cpu().numpy()
    n = sum(counts)
    got = np.unpackbits(out, bitorder="little")[:n].astype(bool)
    np.testing.assert_array_equal(got, np.concatenate(masks) if n else np.zeros(0, dtype=bool))


def test_multi_key_and_float_key_hashing_match_the_reference_functions(gpu_lib, oracle):
    """hash_keys over several key columns (hash_combine_boost, bodo/libs/_array_hash.cpp:41-56,1599-1621) and over float keys
    (_Py_HashDouble, :119-170) on the device against the oracle's restatements, which tests/test_oracle.py pins against the
    published MurmurHash3 vectors and the interpreter's own hash(float)."""
    from bodo_b200.shuffle import hash_keys_table
    rng = np.random.default_rng(5)
    n = 50_021
    k0 = rng.integers(-(1 << 62), 1 << 62, n).astype(np.int64)
    k1 = rng.integers(0, 1000, n).astype(np.int64)
    k2 = rng.integers(-5, 5, n).astype(np.int64)
    v1 = rng.random(n) > 0.1
    df = pd.DataFrame({"a": k0, "b": pd.array(k1, dtype="Int64"), "c": k2})
    df.loc[~v1, "b"] = pd.NA
    t = table_to_device(Table.from_pandas(df))
    for nk in (1, 2, 3):
        h, dest = hash_keys_table(t, nk, 7)
        exp = oracle.hash_keys([k0, k1, k2][:nk], [None, v1, None][:nk])
        np.testing.assert_array_equal(h.cpu().numpy().view(np.uint32), exp)
        np.testing.assert_array_equal(dest.cpu().numpy(), (exp % 7).astype(np.int32))
    # float keys: special values, integers-as-floats (hash equal to the int's), tiny / huge magnitudes
    f = np.concatenate([np.array([0.0, -0.0, 1.0, -1.0, 0.5, 1e300, -1e-300, np.inf, -np.inf, np.nan, 2.0 ** 61, 2.0 ** 61 - 1, 3.0, 1 / 3]),
                        rng.standard_normal(3000) * 10.0 ** rng.integers(-30, 30, 3000)])
    L = oracle.lib()
    import ctypes as C
    L.oracle_hash_inner_32_f64.restype = C.c_uint32
    L.oracle_hash_inner_32_f64.argtypes = [C.c_double, C.c_uint32]
    L.oracle_hash_combine_boost.restype = C.c_uint32
    L.oracle_hash_combine_boost.argtypes = [C.c_uint32, C.c_uint32]
    expf = np.array([L.oracle_hash_inner_32_f64(float(x), 0xB0D01289) for x in f], dtype=np.uint32)
    ki = rng.integers(0, 50, len(f)).astype(np.int64)
    tf = table_to_device(Table.from_pandas(pd.DataFrame({"f": f, "i": ki, "g": f.astype(np.float32)})))
    h1, _ = hash_keys_table(tf, 1, 3)
    np.testing.assert_array_equal(h1.cpu().numpy().view(np.uint32), expf)
    # (float64, int64, float32) composite: first hashed, the others folded in
    ei = oracle.hash_keys([ki])
    eg = np.array([L.oracle_hash_inner_32_f64(float(np.float32(x)), 0xB0D01289) for x in f], dtype=np.uint32)
    exp3 = np.array([L.oracle_hash_combine_boost(L.oracle_hash_combine_boost(int(a), int(b)), int(c)) for a, b, c in zip(expf, ei, eg)], dtype=np.uint32)
    h3, _ = hash_keys_table(tf, 3, 3)
    np.testing.assert_array_equal(h3.cpu().numpy().view(np.uint32), exp3)


def test_partition_on_two_keys_bit_identical_to_oracle_placement(gpu_lib, oracle):
    rng = np.random.default_rng(9)
    n, n_pes = 120_007, 6
    a = rng.integers(0, 300, n).astype(np.int64)
    b = rng.integers(0, 7, n).astype(np.int64)
    df = pd.DataFrame({"a": a, "b": b, "x": rng.random(n)})
    part, counts, perm = partition_device(table_to_device(Table.from_pandas(df)), 2, n_pes, want_perm=True)
    dest = (oracle.hash_keys([a, b]) % n_pes).astype(np.int64)
    eperm = np.argsort(dest, kind="stable")  # stable counting sort by destination = fill_send_array order
    assert counts == [int((dest == d).sum()) for d in range(n_pes)]
    np.testing.assert_array_equal(perm.cpu().numpy(), eperm)
    np.testing.assert_array_equal(part.columns[2].data.cpu().numpy(), df["x"].to_numpy()[eperm])
