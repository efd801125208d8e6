"""ctypes loader for the CPU oracle (oracle/bodo_oracle.c).  TEST INFRASTRUCTURE ONLY.

May be imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs,
never by anything under bodo_b200/ (see the header of bodo_oracle.c).
"""

from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

FT = {"size": 4, "sum": 6, "count": 7, "mean": 14, "min": 15, "max": 16}
CT = {
    np.dtype("int8"): 0, np.dtype("uint8"): 1, np.dtype("int32"): 2, np.dtype("uint32"): 3, np.dtype("int64"): 4,
    np.dtype("float32"): 5, np.dtype("float64"): 6, np.dtype("uint64"): 7, np.dtype("int16"): 8, np.dtype("uint16"): 9,
}
SEED_HASH_PARTITION = 0xB0D01289


class _OCol(C.Structure):
    _fields_ = [("data", C.c_void_p), ("valid", C.c_void_p), ("ctype", C.c_int32), ("pad", C.c_int32)]


def build(force: bool = False) -> None:
    """Compile the oracle (and oracle/_ref when /root/reference is present)."""
    so = os.path.join(_HERE, "libbodo_oracle.so")
    src = os.path.join(_HERE, "bodo_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "all"], stdout=subprocess.DEVNULL)
    elif os.path.exists("/root/reference/bodo/libs/vendored/xxhash.h") and not os.path.exists(
        os.path.join(_HERE, "_ref", "libref_xxh3.so")
    ):
        subprocess.check_call(["make", "-C", _HERE, "ref"], stdout=subprocess.DEVNULL)


def lib():
    global _LIB
    if _LIB is None:
        build()
        L = C.CDLL(os.path.join(_HERE, "libbodo_oracle.so"))
        L.oracle_groupby_run.restype = C.c_void_p
        L.oracle_groupby_run.argtypes = [C.c_int64, C.POINTER(_OCol), C.c_int32, C.c_void_p, C.POINTER(_OCol),
                                         C.c_int32, C.c_int64, C.c_int32, C.c_int32]
        L.oracle_groupby_ngroups.restype = C.c_int64
        L.oracle_groupby_ngroups.argtypes = [C.c_void_p]
        L.oracle_groupby_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.oracle_groupby_free.argtypes = [C.c_void_p]
        L.oracle_hash_inner_32_i64.restype = C.c_uint32
        L.oracle_hash_inner_32_i64.argtypes = [C.c_int64, C.c_uint32]
        L.oracle_hash_inner_32_i32.restype = C.c_uint32
        L.oracle_hash_inner_32_i32.argtypes = [C.c_int32, C.c_uint32]
        L.oracle_hash_to_rank.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_void_p]
        L.oracle_hash_combine_boost.restype = C.c_uint32
        L.oracle_hash_combine_boost.argtypes = [C.c_uint32, C.c_uint32]
        L.oracle_py_hash_double.restype = C.c_int64
        L.oracle_py_hash_double.argtypes = [C.c_double]
        L.oracle_hash_inner_32_f64.restype = C.c_uint32
        L.oracle_hash_inner_32_f64.argtypes = [C.c_double, C.c_uint32]
        L.oracle_hash_keys_i64.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_void_p]
        L.oracle_shuffle_partition.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
        L.oracle_hash_join.restype = C.c_int64
        L.oracle_hash_join.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64]
        L.oracle_groupby_sum_count_mt.restype = C.c_int64
        L.oracle_groupby_sum_count_mt.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p]
        L.oracle_synth_fill.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_uint64]
        _LIB = L
    return _LIB


def _bitmap(valid):
    """bool array -> Arrow validity bitmap (uint8, LSB first) or None."""
    if valid is None:
        return None
    v = np.asarray(valid, dtype=bool)
    return np.packbits(v, bitorder="little")


def _ocol(arr, valid_bm, keep):
    a = np.ascontiguousarray(arr)
    keep.append(a)
    c = _OCol()
    c.data = a.ctypes.data
    if valid_bm is not None:
        keep.append(valid_bm)
        c.valid = valid_bm.ctypes.data
    else:
        c.valid = None
    c.ctype = CT[a.dtype]
    return c


def groupby(keys, key_valid, funcs, vals, val_valids=None, dropna=True, batch_size=32768, n_pes=1, rank=0):
    """Run the oracle groupby.

    keys: int64/int32 array; key_valid: bool array or None; funcs: list of names; vals: list of arrays
    (one per func; ignored for 'size'); val_valids: list of bool arrays / None.
    Returns dict(keys, key_valid, cols=[(data, valid)]) in first-appearance group order.
    """
    L = lib()
    keep = []
    n = len(keys)
    kc = _ocol(keys, _bitmap(key_valid), keep)
    nf = len(funcs)
    ft = np.array([FT[f] for f in funcs], dtype=np.int32)
    vcols = (_OCol * max(nf, 1))()
    for j in range(nf):
        vv = None if val_valids is None else val_valids[j]
        vcols[j] = _ocol(vals[j], _bitmap(vv), keep)
    h = L.oracle_groupby_run(n, C.byref(kc), nf, ft.ctypes.data, vcols, int(dropna), batch_size, n_pes, rank)
    ng = L.oracle_groupby_ngroups(h)
    out_keys = np.empty(ng, dtype=np.int64)
    out_kv = np.empty(ng, dtype=np.uint8)
    raw = [np.empty(ng, dtype=np.int64) for _ in range(nf)]
    valid = [np.empty(ng, dtype=np.uint8) for _ in range(nf)]
    dptr = (C.c_void_p * max(nf, 1))(*[r.ctypes.data for r in raw])
    vptr = (C.c_void_p * max(nf, 1))(*[v.ctypes.data for v in valid])
    L.oracle_groupby_fetch(h, out_keys.ctypes.data, out_kv.ctypes.data, dptr, vptr)
    L.oracle_groupby_free(h)
    cols = []
    for j, f in enumerate(funcs):
        in_float = np.asarray(vals[j]).dtype.kind == "f"
        is_f = f == "mean" or (f in ("sum", "min", "max") and in_float)
        data = raw[j].view(np.float64) if is_f else raw[j]
        cols.append((data, valid[j].astype(bool)))
    return {"keys": out_keys, "key_valid": out_kv.astype(bool), "cols": cols}


def hash_to_rank(keys, key_valid, n_pes, seed=SEED_HASH_PARTITION):
    k = np.ascontiguousarray(keys, dtype=np.int64)
    bm = _bitmap(key_valid)
    out = np.empty(len(k), dtype=np.int32)
    lib().oracle_hash_to_rank(k.ctypes.data, None if bm is None else bm.ctypes.data, len(k), n_pes, seed, out.ctypes.data)
    return out


def hash_keys(key_cols, key_valids=None, seed=SEED_HASH_PARTITION):
    """hash_keys over 1..n int64 key columns (first hashed, the rest combined); returns uint32 hashes."""
    cols = [np.ascontiguousarray(k, dtype=np.int64) for k in key_cols]
    n = len(cols[0])
    bms = [_bitmap(v) for v in (key_valids or [None] * len(cols))]
    kp = (C.c_void_p * len(cols))(*[c.ctypes.data for c in cols])
    vp = (C.c_void_p * len(cols))(*[None if b is None else b.ctypes.data for b in bms])
    out = np.empty(n, dtype=np.uint32)
    lib().oracle_hash_keys_i64(kp, vp, len(cols), n, seed, out.ctypes.data)
    return out


def shuffle_partition(keys, key_valid, n_pes):
    """Returns (send_counts, perm): rows perm[...] grouped by destination rank, stable within a rank."""
    k = np.ascontiguousarray(keys, dtype=np.int64)
    bm = _bitmap(key_valid)
    counts = np.zeros(n_pes, dtype=np.int64)
    perm = np.empty(len(k), dtype=np.int64)
    lib().oracle_shuffle_partition(k.ctypes.data, None if bm is None else bm.ctypes.data, len(k), n_pes,
                                   counts.ctypes.data, perm.ctypes.data)
    return counts, perm


def hash_join(bkeys, bvalid, pkeys, pvalid, build_outer=False, probe_outer=False, na_equal=True):
    """Returns (build_idx, probe_idx) int64 arrays; -1 marks the NULL side of an outer row."""
    bk = np.ascontiguousarray(bkeys, dtype=np.int64)
    pk = np.ascontiguousarray(pkeys, dtype=np.int64)
    bbm, pbm = _bitmap(bvalid), _bitmap(pvalid)
    args = [bk.ctypes.data, None if bbm is None else bbm.ctypes.data, len(bk), pk.ctypes.data,
            None if pbm is None else pbm.ctypes.data, len(pk), int(build_outer), int(probe_outer), int(na_equal)]
    n = lib().oracle_hash_join(*args, None, None, 0)
    bi = np.empty(n, dtype=np.int64)
    pi = np.empty(n, dtype=np.int64)
    lib().oracle_hash_join(*args, bi.ctypes.data, pi.ctypes.data, n)
    return bi, pi


def groupby_sum_count_mt(keys, vals, n_threads, batch=32768):
    """Multi-threaded SPMD baseline; returns (n_groups, (sum_of_sums, sum_of_counts, xor_of_keys))."""
    k = np.ascontiguousarray(keys, dtype=np.int64)
    v = np.ascontiguousarray(vals, dtype=np.int64)
    cs = np.zeros(3, dtype=np.uint64)
    ng = lib().oracle_groupby_sum_count_mt(k.ctypes.data, v.ctypes.data, len(k), n_threads, batch, cs.ctypes.data)
    return ng, tuple(int(x) for x in cs)


def synth_fill(row_start, n, n_groups, seed):
    k = np.empty(n, dtype=np.int64)
    v = np.empty(n, dtype=np.int64)
    lib().oracle_synth_fill(k.ctypes.data, v.ctypes.data, row_start, n, n_groups, seed)
    return k, v
