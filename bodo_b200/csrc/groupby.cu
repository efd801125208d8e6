// groupby.cu — streaming hash groupby/aggregate on one B200 (sm_100a).
//
// Replaces GroupbyState + groupby_agg_build_consume_batch + FinalizeBuild of the reference
// (bodo/libs/streaming/_groupby.cpp:2554-3031, 4325-4457, 4062-4256) and the aggregate kernels of
// bodo/libs/groupby/_groupby_agg_funcs.h.  Design (see DESIGN.md):
//   * one persistent open-addressing table per state (linear probing, load <= 0.5, int64 keys,
//     SoA accumulator columns), instead of the reference's per-batch update table + combine;
//   * the consume kernel fuses hash + find-or-insert + every aggregate update of a row;
//   * rows whose insert would overfill the table are appended to a fail list; the host grows/rehashes
//     the table and replays only those rows (the reference's transactional retry,
//     _groupby.cpp:3309-3341, without the partition split);
//   * finalize compacts occupied slots and evaluates the output columns (mean_eval etc.).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <memory>
#include <vector>

#include <cooperative_groups.h>

#include "common.cuh"

namespace b200 {

constexpr long long EMPTY_KEY = (long long)0x8000000000000000ULL;  // INT64_MIN marks a free slot
constexpr int MAX_OPS = 16;
constexpr int64_t CHUNK_ROWS = 1ll << 28;  // rows per consume chunk (bounds the fail list of the direct path at 1 GiB)

enum OpKind : int { K_SUM_I64 = 0, K_SUM_F64, K_COUNT, K_SIZE, K_MEAN, K_MIN_I64, K_MAX_I64, K_MIN_F64, K_MAX_F64,
                    K_SUMSQ_F64, K_SUMCUBE_F64,  // hidden accumulators: sum of squares / cubes (as double) of the non-NA values
                    // first / last non-NA value in row order (aggfunc<first / last>, _groupby_agg_funcs.h:594-611): a0 = value
                    // bits, a1 = sequence number of the row that supplied it (see groupby_firstlast_fix_kernel)
                    K_FIRST, K_LAST,
                    K_NUNIQUE,  // number of distinct non-NA values: filled at finalize from a nested (key, value) distinct state
                    // evaluation-only kinds of composite functions (accumulators: a K_MEAN pair + K_SUMSQ (+ K_SUMCUBE))
                    E_VAR, E_STD, E_VAR_POP, E_STD_POP, E_SKEW };

struct OpDesc {
    int kind;
    int in_ctype;
    const void* in_data;
    const uint8_t* in_valid;
    void* a0;  // main accumulator column (8 B / slot)
    void* a1;  // second accumulator (mean count, min/max seen-count) or nullptr
};

struct ConsumeArgs {
    const void* key_data;
    const uint8_t* key_valid;
    int key_ctype;
    int dropna;
    int64_t n_rows;
    const uint32_t* index_list;  // nullptr: rows [0, n_rows); else replay of the listed rows
    long long* tkeys;
    uint64_t cap;  // power of two; slot cap = NA key, slot cap + 1 = the key equal to EMPTY_KEY
    long long* counters;  // [0] groups in table, [1] failed rows, [2] cursor, [3] NA present, [4] EMPTY_KEY present
    long long group_limit;
    uint32_t* fail_list;
    unsigned long long seq_base;  // first / last: sequence number of row 0 of this launch, minus 1 (rank << 44 | rows consumed so far)
    int n_ops;
    OpDesc ops[MAX_OPS];
};

// find-or-insert with linear probing over 8-byte key slots; returns the slot, or UINT64_MAX when the table is at
// its group limit (group_limit < 0 disables the limit: rehash into a table that is known to be large enough).
// Measured on B200 (scratch/ubench2.cu, profiles/r01_ubench2.txt): a 4-key bucket fetched with one 256-bit load
// is SLOWER than this (29 vs 40 Grows/s) — L2 random-request rate, not probe-chain latency, is the limit.
__device__ __forceinline__ uint64_t find_or_insert(long long* __restrict__ tkeys, uint64_t cap, long long key,
                                                   long long* counters, long long group_limit) {
    uint64_t mask = cap - 1;
    uint64_t s = (key_hash(key) >> 32) & mask;
    for (uint64_t probes = 0; probes <= mask; probes++) {
        long long k = __ldcg(tkeys + s);
        if (k == key) return s;
        if (k == EMPTY_KEY) {
            // take a ticket first so the table can never exceed group_limit (probing always terminates).  The lanes of the warp
            // that stand here together take their tickets with ONE atomic (coalesced group): a flush of 10^6 new groups is 10^6
            // tickets on a single address otherwise (measured 0.17 ms per operator state)
            if (group_limit >= 0) {
                const cooperative_groups::coalesced_group cgp = cooperative_groups::coalesced_threads();
                long long t = 0;
                if (cgp.thread_rank() == 0) t = (long long)atomicAdd((unsigned long long*)&counters[0], (unsigned long long)cgp.size());
                t = cgp.shfl(t, 0) + (long long)cgp.thread_rank();
                if (t >= group_limit) {
                    atomicAdd((unsigned long long*)&counters[0], (unsigned long long)-1ll);
                    return ~0ull;
                }
            }
            long long prev = atomicCAS((unsigned long long*)(tkeys + s), (unsigned long long)EMPTY_KEY,
                                       (unsigned long long)key);
            if (prev == EMPTY_KEY) return s;
            if (group_limit >= 0) atomicAdd((unsigned long long*)&counters[0], (unsigned long long)-1ll);  // lost the race
            if (prev == key) return s;
        }
        s = (s + 1) & mask;
    }
    return ~0ull;
}

// lookup only; UINT64_MAX when the key is not in the table
__device__ __forceinline__ uint64_t find_only(const long long* __restrict__ tkeys, uint64_t cap, long long key) {
    uint64_t mask = cap - 1;
    uint64_t s = (key_hash(key) >> 32) & mask;
    for (uint64_t probes = 0; probes <= mask; probes++) {
        long long k = __ldcg(tkeys + s);
        if (k == key) return s;
        if (k == EMPTY_KEY) return ~0ull;
        s = (s + 1) & mask;
    }
    return ~0ull;
}
// value of a first / last input as the 8 bytes kept in the accumulator (integers sign / zero extended, floats as double)
__device__ __forceinline__ bool firstlast_value(const OpDesc& op, int64_t row, unsigned long long& bits) {
    if (op.in_ctype == CT_FLOAT64 || op.in_ctype == CT_FLOAT32) {
        const double v = load_as_f64(op.in_data, op.in_ctype, row);
        bits = (unsigned long long)__double_as_longlong(v);
        return !isnan(v);
    }
    bits = (unsigned long long)load_int_as_i64(op.in_data, op.in_ctype, row);
    return true;
}

template <typename A>
__device__ __forceinline__ void apply_ops(const A& a, uint64_t slot, int64_t row) {
#pragma unroll 1
    for (int j = 0; j < a.n_ops; j++) {
        const OpDesc& op = a.ops[j];
        if (op.kind == K_SIZE) {  // size_agg (_groupby_agg_funcs.h:661-669): counts every row
            atomicAdd((unsigned long long*)op.a0 + slot, 1ull);
            continue;
        }
        if (!bit_valid(op.in_valid, row)) continue;  // nullable input: skip NA (do_apply_to_column.cpp:1796-1823)
        switch (op.kind) {
            case K_SUM_I64:  // casted_aggfunc sum: int64 accumulate, wraparound (_groupby_agg_funcs.h:176-190)
                atomicAdd((unsigned long long*)op.a0 + slot, (unsigned long long)load_int_as_i64(op.in_data, op.in_ctype, row));
                break;
            case K_COUNT: {  // count_agg (:644-657): non-NA values (NaN is NA for floats)
                bool ok = true;
                if (op.in_ctype == CT_FLOAT64 || op.in_ctype == CT_FLOAT32) ok = !isnan(load_as_f64(op.in_data, op.in_ctype, row));
                if (ok) atomicAdd((unsigned long long*)op.a0 + slot, 1ull);
                break;
            }
            case K_SUM_F64: {
                double v = load_as_f64(op.in_data, op.in_ctype, row);
                if (!isnan(v)) atomicAdd((double*)op.a0 + slot, v);
                break;
            }
            case K_MEAN: {  // mean_agg (:673-689): double sum + uint64 count
                double v = load_as_f64(op.in_data, op.in_ctype, row);
                if (!isnan(v)) {
                    atomicAdd((double*)op.a0 + slot, v);
                    atomicAdd((unsigned long long*)op.a1 + slot, 1ull);
                }
                break;
            }
            case K_SUMSQ_F64: case K_SUMCUBE_F64: {  // skew_agg's m2 / m3 (:723-745); var / std use m2 with the K_MEAN pair
                double v = load_as_f64(op.in_data, op.in_ctype, row);
                if (!isnan(v)) atomicAdd((double*)op.a0 + slot, op.kind == K_SUMSQ_F64 ? v * v : v * v * v);
                break;
            }
            case K_FIRST: case K_LAST: {  // phase 1: which row supplies the value (phase 2 writes it, groupby_firstlast_fix_kernel)
                unsigned long long bits;
                if (firstlast_value(op, row, bits)) {
                    const unsigned long long seq = a.seq_base + (unsigned long long)row + 1ull;
                    if (op.kind == K_FIRST) atomicMin((unsigned long long*)op.a1 + slot, seq);
                    else atomicMax((unsigned long long*)op.a1 + slot, seq);
                }
                break;
            }
            case K_MIN_I64:
                atomicMin((long long*)op.a0 + slot, (long long)load_int_as_i64(op.in_data, op.in_ctype, row));
                if (op.a1) atomicAdd((unsigned long long*)op.a1 + slot, 1ull);
                break;
            case K_MAX_I64:
                atomicMax((long long*)op.a0 + slot, (long long)load_int_as_i64(op.in_data, op.in_ctype, row));
                if (op.a1) atomicAdd((unsigned long long*)op.a1 + slot, 1ull);
                break;
            case K_MIN_F64: {
                double v = load_as_f64(op.in_data, op.in_ctype, row);
                if (!isnan(v)) {
                    atomicMin((unsigned long long*)op.a0 + slot, f64_to_ordered(v));
                    if (op.a1) atomicAdd((unsigned long long*)op.a1 + slot, 1ull);
                }
                break;
            }
            case K_MAX_F64: {
                double v = load_as_f64(op.in_data, op.in_ctype, row);
                if (!isnan(v)) {
                    atomicMax((unsigned long long*)op.a0 + slot, f64_to_ordered(v));
                    if (op.a1) atomicAdd((unsigned long long*)op.a1 + slot, 1ull);
                }
                break;
            }
        }
    }
}

// Generic fused consume kernel: any key/value types, any mix of aggregates, nullable columns.
__global__ void __launch_bounds__(256) groupby_consume_kernel(const __grid_constant__ ConsumeArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_rows; i += stride) {
        int64_t row = a.index_list ? (int64_t)a.index_list[i] : i;
        bool kvalid = bit_valid(a.key_valid, row);
        uint64_t slot;
        if (!kvalid) {
            if (a.dropna) continue;  // filter_na_keys (_groupby.cpp:4278-4309)
            slot = a.cap;
            a.counters[3] = 1;
        } else {
            long long key = load_int_as_i64(a.key_data, a.key_ctype, row);
            if (key == EMPTY_KEY) {
                slot = a.cap + 1;
                a.counters[4] = 1;
            } else {
                slot = find_or_insert(a.tkeys, a.cap, key, a.counters, a.group_limit);
                if (slot == ~0ull) {
                    unsigned long long f = atomicAdd((unsigned long long*)&a.counters[1], 1ull);
                    a.fail_list[f] = (uint32_t)row;
                    continue;
                }
            }
        }
        apply_ops(a, slot, row);
    }
}

// first / last, phase 2 (after every row of the launch — replays included — has been applied): the row whose sequence number
// won the atomicMin / atomicMax writes its value.  Two passes because (value, sequence) cannot be updated by one atomic.
__global__ void __launch_bounds__(256) groupby_firstlast_fix_kernel(const __grid_constant__ ConsumeArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t row = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; row < a.n_rows; row += stride) {
        uint64_t slot;
        if (!bit_valid(a.key_valid, row)) { if (a.dropna) continue; slot = a.cap; }
        else {
            const long long key = load_int_as_i64(a.key_data, a.key_ctype, row);
            slot = key == EMPTY_KEY ? a.cap + 1 : find_only(a.tkeys, a.cap, key);
            if (slot == ~0ull) continue;
        }
        const unsigned long long seq = a.seq_base + (unsigned long long)row + 1ull;
#pragma unroll 1
        for (int j = 0; j < a.n_ops; j++) {
            const OpDesc& op = a.ops[j];
            if (op.kind != K_FIRST && op.kind != K_LAST) continue;
            if (!bit_valid(op.in_valid, row)) continue;
            unsigned long long bits;
            if (firstlast_value(op, row, bits) && ((const unsigned long long*)op.a1)[slot] == seq) ((unsigned long long*)op.a0)[slot] = bits;
        }
    }
}

// Specialised consume kernel for the headline shape: non-null int64 key, non-null int64 value,
// aggregates drawn from {sum, count, size} of that one value column (BASELINE.json C1/C2).
// Two rows per thread per iteration through 128-bit loads; the aggregate updates are `red` (no return).
template <bool HAS_SUM, bool HAS_CNT>
__global__ void __launch_bounds__(256) groupby_consume_i64_sumcount_kernel(
    const long long* __restrict__ keys, const long long* __restrict__ vals, int64_t n_rows, long long* tkeys, uint64_t cap,
    unsigned long long* acc_sum, unsigned long long* acc_cnt, long long* counters, long long group_limit,
    uint32_t* fail_list) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x * 2;
    int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 2;
    for (; i < n_rows; i += stride) {
        long long k[2], v[2];
        int m = 2;
        if (i + 1 < n_rows) {
            longlong2 kk = __ldcs(reinterpret_cast<const longlong2*>(keys + i));
            k[0] = kk.x; k[1] = kk.y;
            if (HAS_SUM) { longlong2 vv = __ldcs(reinterpret_cast<const longlong2*>(vals + i)); v[0] = vv.x; v[1] = vv.y; }
        } else {
            k[0] = keys[i]; k[1] = 0; m = 1;
            if (HAS_SUM) { v[0] = vals[i]; v[1] = 0; }
        }
#pragma unroll
        for (int r = 0; r < 2; r++) {
            if (r >= m) break;
            uint64_t sl;
            if (k[r] == EMPTY_KEY) {
                sl = cap + 1;
                counters[4] = 1;
            } else {
                sl = find_or_insert(tkeys, cap, k[r], counters, group_limit);
                if (sl == ~0ull) {
                    unsigned long long f = atomicAdd((unsigned long long*)&counters[1], 1ull);
                    fail_list[f] = (uint32_t)(i + r);
                    continue;
                }
            }
            if (HAS_SUM) atomicAdd(acc_sum + sl, (unsigned long long)v[r]);
            if (HAS_CNT) atomicAdd(acc_cnt + sl, 1ull);
        }
    }
}

__global__ void fill_u64_kernel(unsigned long long* p, uint64_t n, unsigned long long v) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}

struct RehashArgs {
    const long long* old_keys;
    uint64_t old_cap;
    long long* new_keys;
    uint64_t new_cap;
    int n_acc;
    const unsigned long long* old_acc[2 * MAX_OPS];
    unsigned long long* new_acc[2 * MAX_OPS];
};
// grow: re-insert every occupied slot (and the two special slots) into the new arrays
__global__ void rehash_kernel(const __grid_constant__ RehashArgs a) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < a.old_cap + 2; s += stride) {
        uint64_t ns;
        if (s >= a.old_cap) {
            ns = a.new_cap + (s - a.old_cap);
        } else {
            long long k = a.old_keys[s];
            if (k == EMPTY_KEY) continue;
            ns = find_or_insert(a.new_keys, a.new_cap, k, nullptr, -1);
        }
        for (int j = 0; j < a.n_acc; j++) a.new_acc[j][ns] = a.old_acc[j][s];
    }
}

// ---- finalize: compact occupied slots, then evaluate output columns ----
// n_pes > 1: only the groups this rank OWNS (hash_to_rank(key) == rank) are output — after the fused exchange the table still
// holds the partial aggregates of groups that were sent to their owners (they are never touched again: received rows only
// carry keys this rank owns)
__global__ void compact_slots_kernel(const long long* __restrict__ tkeys, uint64_t cap, const long long* counters,
                                     long long* cursor, uint64_t* slot_of_out, int n_pes, int rank) {
    const bool na_present = counters[3] != 0, empty_present = counters[4] != 0;
    const uint32_t na_hash = (uint32_t)xxh3_64_short(1ull, 8, SEED_HASH_PARTITION);  // hash_na_val (_array_hash.cpp:22-29)
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s0 = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s0 < ((cap + 2 + 31) & ~31ull); s0 += stride) {
        bool occ = false;
        if (s0 < cap) occ = tkeys[s0] != EMPTY_KEY;
        else if (s0 == cap) occ = na_present;
        else if (s0 == cap + 1) occ = empty_present;
        if (occ && n_pes > 1) {
            const uint32_t h = s0 == cap ? na_hash : (uint32_t)key_hash(s0 < cap ? tkeys[s0] : EMPTY_KEY);
            occ = hash_to_rank_u32(h, n_pes) == rank;
        }
        unsigned m = __ballot_sync(0xffffffffu, occ);
        int lane = threadIdx.x & 31;
        long long base = 0;
        if (lane == 0 && m) base = (long long)atomicAdd((unsigned long long*)cursor, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (occ) slot_of_out[base + __popc(m & ((1u << lane) - 1))] = s0;
    }
}

struct OutDesc {
    int kind;       // OpKind
    int out_ctype;  // CType of the output column
    const void* a0;
    const void* a1;
    const void* b0;  // composite functions: sum of squares
    const void* c0;  //                      sum of cubes
    void* out_data;
    uint32_t* out_valid;  // validity bitmap as 32-bit words, or nullptr when the column has no nulls
};
struct EvalArgs {
    const long long* tkeys;
    uint64_t cap;
    const uint64_t* slot_of_out;
    const long long* n_out_ptr;  // number of compacted slots (device counter written by compact_slots_kernel)
    int key_ctype;
    void* out_keys;
    uint32_t* out_key_valid;  // nullptr unless the NA-key group can exist
    int n_ops;
    OutDesc ops[MAX_OPS];
};

__device__ __forceinline__ void store_int_typed(void* p, int ct, int64_t i, long long v) {
    switch (ct) {
        case CT_INT64: case CT_UINT64: case CT_DATETIME: case CT_TIMEDELTA: ((long long*)p)[i] = v; break;
        case CT_INT32: case CT_UINT32: case CT_DATE: ((int32_t*)p)[i] = (int32_t)v; break;
        case CT_INT16: case CT_UINT16: ((int16_t*)p)[i] = (int16_t)v; break;
        case CT_INT8: case CT_UINT8: case CT_BOOL: ((int8_t*)p)[i] = (int8_t)v; break;
    }
}
__device__ __forceinline__ void store_f_typed(void* p, int ct, int64_t i, double v) {
    if (ct == CT_FLOAT32) ((float*)p)[i] = (float)v; else ((double*)p)[i] = v;
}

// eval_groupby_funcs_helper (_groupby.cpp:396-457) + output null rules (aggfunc_output_initialize_kernel,
// groupby/_groupby_common.cpp:50-74: sum/count/size valid, min/max/mean NULL when nothing was seen).
__global__ void eval_output_kernel(const __grid_constant__ EvalArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_out = *a.n_out_ptr;
    int64_t n_round = (n_out + 31) & ~31ll;
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n_round; p += stride) {
        bool in = p < n_out;
        uint64_t s = in ? a.slot_of_out[p] : 0;
        bool key_ok = true;
        if (in && a.tkeys) {  // single-key tables only (multi-key tables write their key columns in eval_mk_keys_kernel)
            long long key = s < a.cap ? a.tkeys[s] : (s == a.cap ? 0 : EMPTY_KEY);
            key_ok = s != a.cap;
            store_int_typed(a.out_keys, a.key_ctype, p, key);
        }
        if (a.out_key_valid) {
            unsigned m = __ballot_sync(0xffffffffu, in && key_ok);
            if ((threadIdx.x & 31) == 0) a.out_key_valid[p >> 5] = m;
        }
#pragma unroll 1
        for (int j = 0; j < a.n_ops; j++) {
            const OutDesc& op = a.ops[j];
            bool valid = in;
            if (in) {
                switch (op.kind) {
                    case K_SUM_I64: case K_COUNT: case K_SIZE: case K_NUNIQUE:
                        store_int_typed(op.out_data, op.out_ctype, p, ((const long long*)op.a0)[s]);
                        break;
                    case K_SUM_F64:
                        store_f_typed(op.out_data, op.out_ctype, p, ((const double*)op.a0)[s]);
                        break;
                    case K_MEAN: {  // mean_eval (do_apply_to_column.cpp:880-913)
                        unsigned long long c = ((const unsigned long long*)op.a1)[s];
                        valid = c > 0;
                        store_f_typed(op.out_data, op.out_ctype, p, valid ? ((const double*)op.a0)[s] / (double)c : __longlong_as_double(0x7ff8000000000000ll));
                        break;
                    }
                    case E_VAR: case E_STD: case E_VAR_POP: case E_STD_POP: {
                        // var_eval / std_eval (groupby/_groupby_eval.h:71-95).  The reference carries Welford's (count, mean,
                        // M2); the device carries the power sums (atomics cannot run Welford's recurrence) and forms
                        // M2 = sum x^2 - (sum x)^2 / n here — equal up to rounding unless |mean| >> spread (tests state the bound)
                        const double n = (double)((const unsigned long long*)op.a1)[s];
                        const double s1 = ((const double*)op.a0)[s], s2 = ((const double*)op.b0)[s];
                        const bool pop = op.kind == E_VAR_POP || op.kind == E_STD_POP;
                        valid = pop ? n >= 1 : n >= 2;
                        double m2 = s2 - s1 * s1 / n;
                        if (m2 < 0) m2 = 0;
                        double r = valid ? m2 / (pop ? n : n - 1) : __longlong_as_double(0x7ff8000000000000ll);
                        if (valid && (op.kind == E_STD || op.kind == E_STD_POP)) r = sqrt(r);
                        store_f_typed(op.out_data, op.out_ctype, p, r);
                        break;
                    }
                    case E_SKEW: {  // skew_eval (groupby/_groupby_eval.h:110-137), same power sums as the reference
                        const unsigned long long cnt = ((const unsigned long long*)op.a1)[s];
                        const double n = (double)cnt, m1 = ((const double*)op.a0)[s], m2 = ((const double*)op.b0)[s], m3 = ((const double*)op.c0)[s];
                        valid = cnt >= 3;
                        double r = __longlong_as_double(0x7ff8000000000000ll);
                        if (valid) {
                            const double mean = m1 / n;
                            const double num = m3 - 3.0 * m2 * mean + 2.0 * n * mean * mean * mean;
                            const double den = pow(m2 - mean * m1, 1.5);
                            if (num == 0.0 || fabs(den) < 1e-14 || isnan(den) || log2(fabs(den)) - log2(fabs(num)) < -20) r = 0.0;
                            else r = (n * pow(n - 1, 1.5) / (n - 2)) * num / den / (n - 1);
                        }
                        store_f_typed(op.out_data, op.out_ctype, p, r);
                        break;
                    }
                    case K_FIRST: case K_LAST: {  // NA when the group never saw a non-NA value (nullable / float outputs)
                        const unsigned long long q = ((const unsigned long long*)op.a1)[s];
                        const bool seen = op.kind == K_FIRST ? q != ~0ull : q != 0ull;
                        const unsigned long long bits = ((const unsigned long long*)op.a0)[s];
                        valid = seen;
                        if (op.out_ctype == CT_FLOAT32 || op.out_ctype == CT_FLOAT64)
                            store_f_typed(op.out_data, op.out_ctype, p, seen ? __longlong_as_double((long long)bits) : __longlong_as_double(0x7ff8000000000000ll));
                        else store_int_typed(op.out_data, op.out_ctype, p, seen ? (long long)bits : 0);
                        break;
                    }
                    case K_MIN_I64: case K_MAX_I64: {
                        if (op.a1) valid = ((const unsigned long long*)op.a1)[s] > 0;
                        store_int_typed(op.out_data, op.out_ctype, p, valid ? ((const long long*)op.a0)[s] : 0);
                        break;
                    }
                    case K_MIN_F64: case K_MAX_F64: {
                        unsigned long long e = ((const unsigned long long*)op.a0)[s];
                        bool seen = op.kind == K_MIN_F64 ? (e != ~0ull) : (e != 0ull);
                        if (op.a1) valid = seen;
                        store_f_typed(op.out_data, op.out_ctype, p, seen ? ordered_to_f64(e) : __longlong_as_double(0x7ff8000000000000ll));
                        break;
                    }
                }
            }
            if (op.out_valid) {
                unsigned m = __ballot_sync(0xffffffffu, valid);
                if ((threadIdx.x & 31) == 0) op.out_valid[p >> 5] = m;
            }
        }
    }
}

// ---- multi-rank exchange: pack partial aggregates per destination rank -------------------------
// Wire format of one partial row (all fields 8 bytes): [key][flags: bit0 = key valid][a0, a1 of op 0]...
// Only accumulators that exist are sent (row width = 16 + 8 * n_acc).
struct PackArgs {
    const long long* tkeys;
    uint64_t cap;
    const uint64_t* slot_of_out;
    int64_t n_out;
    int n_pes;
    int n_acc;
    const unsigned long long* acc[2 * MAX_OPS];
    long long* dest_count;   // n_pes (histogram pass) / running cursors (scatter pass)
    unsigned long long* out; // packed rows
    int row_words;
    int pass;                // 0 = histogram, 1 = scatter
};
__global__ void pack_partials_kernel(const __grid_constant__ PackArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    uint32_t na_hash = (uint32_t)xxh3_64_short(1ull, 8, SEED_HASH_PARTITION);  // hash_na_val (_array_hash.cpp:22-29)
    int lane = threadIdx.x & 31;
    int64_t n_round = (a.n_out + 31) & ~31ll;
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n_round; p += stride) {
        bool in = p < a.n_out;
        uint64_t s = in ? a.slot_of_out[p] : 0;
        long long key = s < a.cap ? a.tkeys[s] : (s == a.cap ? 0 : EMPTY_KEY);
        bool kvalid = s != a.cap;
        uint32_t h = kvalid ? (uint32_t)key_hash(key) : na_hash;
        int d = in ? hash_to_rank_u32(h, a.n_pes) : -1;
        // warp-aggregated cursor: one atomic per (warp, destination) instead of one per row
        unsigned peers = __match_any_sync(0xffffffffu, d);
        int leader = __ffs(peers) - 1;
        int rank_in_peers = __popc(peers & ((1u << lane) - 1));
        long long base = 0;
        if (in && lane == leader) base = (long long)atomicAdd((unsigned long long*)&a.dest_count[d], (unsigned long long)__popc(peers));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (in && a.pass == 1) {
            unsigned long long* o = a.out + (base + rank_in_peers) * a.row_words;
            o[0] = (unsigned long long)key;
            o[1] = kvalid ? 1ull : 0ull;
            for (int j = 0; j < a.n_acc; j++) o[2 + j] = a.acc[j][s];
        }
    }
}

struct CombineArgs {
    const unsigned long long* in;
    int64_t n_rows;
    int row_words;
    long long* tkeys;
    uint64_t cap;
    long long* counters;
    long long group_limit;
    uint32_t* fail_list;
    const uint32_t* index_list;
    int n_ops;
    int kinds[MAX_OPS];
    void* a0[MAX_OPS];
    void* a1[MAX_OPS];
};
// combine step (get_combine_func, groupby/_groupby_update.cpp:41-57): count/size/mean -> sum, min -> min, max -> max
// merges the accumulator words r[0 ...] of one partial row into `slot`
__device__ __forceinline__ void combine_apply(const CombineArgs& a, uint64_t slot, const unsigned long long* r) {
    {
        int w = 0;
        for (int j = 0; j < a.n_ops; j++) {
            unsigned long long v0 = r[w++];
            unsigned long long v1 = a.a1[j] ? r[w++] : 0;
            switch (a.kinds[j]) {
                case K_SUM_I64: case K_COUNT: case K_SIZE: case K_NUNIQUE: atomicAdd((unsigned long long*)a.a0[j] + slot, v0); break;
                case K_SUM_F64: case K_SUMSQ_F64: case K_SUMCUBE_F64: atomicAdd((double*)a.a0[j] + slot, __longlong_as_double((long long)v0)); break;
                case K_MEAN:
                    atomicAdd((double*)a.a0[j] + slot, __longlong_as_double((long long)v0));
                    atomicAdd((unsigned long long*)a.a1[j] + slot, v1);
                    break;
                case K_MIN_I64: atomicMin((long long*)a.a0[j] + slot, (long long)v0); break;
                case K_MAX_I64: atomicMax((long long*)a.a0[j] + slot, (long long)v0); break;
                case K_MIN_F64: atomicMin((unsigned long long*)a.a0[j] + slot, v0); break;
                case K_MAX_F64: atomicMax((unsigned long long*)a.a0[j] + slot, v0); break;
                // first / last: the partial with the smallest / largest sequence number wins (sequence numbers carry the rank in
                // their high bits: rank order, then row order, as the reference's rank-ordered combine); its value is written by
                // combine_firstlast_fix_kernel once every partial of the batch has been applied
                case K_FIRST: if (v1 != ~0ull) atomicMin((unsigned long long*)a.a1[j] + slot, v1); break;
                case K_LAST: if (v1 != 0ull) atomicMax((unsigned long long*)a.a1[j] + slot, v1); break;
            }
            if (a.a1[j] && a.kinds[j] != K_MEAN && a.kinds[j] != K_FIRST && a.kinds[j] != K_LAST) atomicAdd((unsigned long long*)a.a1[j] + slot, v1);
        }
    }
}
__device__ __forceinline__ void combine_one_row(const CombineArgs& a, int64_t row) {
    const unsigned long long* r = a.in + row * a.row_words;
    long long key = (long long)r[0];
    bool kvalid = r[1] & 1;
    uint64_t slot;
    if (!kvalid) { slot = a.cap; a.counters[3] = 1; }
    else if (key == EMPTY_KEY) { slot = a.cap + 1; a.counters[4] = 1; }
    else {
        slot = find_or_insert(a.tkeys, a.cap, key, a.counters, a.group_limit);
        if (slot == ~0ull) {
            unsigned long long f = atomicAdd((unsigned long long*)&a.counters[1], 1ull);
            a.fail_list[f] = (uint32_t)row;
            return;
        }
    }
    combine_apply(a, slot, r + 2);
}
__global__ void combine_partials_kernel(const __grid_constant__ CombineArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_rows; i += stride)
        combine_one_row(a, a.index_list ? (int64_t)a.index_list[i] : i);
}
// first / last, phase 2 of the combine step: the partial whose sequence number won writes its value
__device__ __forceinline__ void combine_firstlast_fix_row(const CombineArgs& a, int64_t row) {
    const unsigned long long* r = a.in + row * a.row_words;
    const long long key = (long long)r[0];
    uint64_t slot;
    if (!(r[1] & 1)) slot = a.cap;
    else if (key == EMPTY_KEY) slot = a.cap + 1;
    else { slot = find_only(a.tkeys, a.cap, key); if (slot == ~0ull) return; }
    int w = 2;
    for (int j = 0; j < a.n_ops; j++) {
        const unsigned long long v0 = r[w++];
        const unsigned long long v1 = a.a1[j] ? r[w++] : 0;
        if ((a.kinds[j] == K_FIRST && v1 != ~0ull) || (a.kinds[j] == K_LAST && v1 != 0ull))
            if (((const unsigned long long*)a.a1[j])[slot] == v1) ((unsigned long long*)a.a0[j])[slot] = v0;
    }
}
__global__ void combine_firstlast_fix_kernel(const __grid_constant__ CombineArgs a, const unsigned long long* hdr, int n_pes, long long cap_rows) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (hdr == nullptr) {  // one contiguous run of partial rows
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_rows; i += stride) combine_firstlast_fix_row(a, i);
        return;
    }
    for (int s = 0; s < n_pes; s++) {  // the segments of a receive slab (see xchg_combine_slab_kernel)
        if (hdr[s] >> 63) return;  // overflow flag: nobody combined
        const int64_t n = (int64_t)(hdr[s] & ~(1ull << 63));
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) combine_firstlast_fix_row(a, (int64_t)s * cap_rows + i);
    }
}

// ---- fused exchange: pack + all-to-all in ONE kernel over peer memory (NVLink stores), combine straight out of the slab ----
// Every rank owns a receive slab in symmetric memory (mapped into every peer's address space): a header of n_pes counts
// followed by n_pes segments of cap_rows partial rows, segment s written by rank s.  xchg_pack_remote_kernel walks the local
// table once and stores every group that another rank owns straight into that owner's slab (no send buffer, no count
// exchange, no host round trip); xchg_post_counts_kernel then tells every peer how many rows it got; after a device-side
// barrier across the ranks, xchg_combine_slab_kernel merges the received rows into the local table.  A sender whose share for
// some destination exceeds cap_rows flags that in EVERY peer's header; then no rank combines and the host falls back to the
// NCCL exchange (the local tables are still intact).
constexpr unsigned long long XCHG_OVERFLOW = 1ull << 63;
constexpr int XCHG_HDR_BYTES = 256;
struct XchgPackArgs {
    const long long* tkeys;
    uint64_t cap;
    const long long* counters;
    int n_pes, rank;
    int n_acc;
    const unsigned long long* acc[2 * MAX_OPS];
    int row_words;
    unsigned long long* cursors;      // [n_pes] rows packed per destination (device)
    void* const* peer_slabs;          // [n_pes] device pointers to every rank's slab (own slab included)
    long long cap_rows;
};
__global__ void xchg_pack_remote_kernel(const __grid_constant__ XchgPackArgs a) {
    const bool na_present = a.counters[3] != 0, empty_present = a.counters[4] != 0;
    const uint32_t na_hash = (uint32_t)xxh3_64_short(1ull, 8, SEED_HASH_PARTITION);
    const int lane = threadIdx.x & 31;
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < ((a.cap + 2 + 31) & ~31ull); s += stride) {
        bool occ = false;
        if (s < a.cap) occ = a.tkeys[s] != EMPTY_KEY;
        else if (s == a.cap) occ = na_present;
        else if (s == a.cap + 1) occ = empty_present;
        const long long key = s < a.cap ? (occ ? a.tkeys[s] : 0) : (s == a.cap ? 0 : EMPTY_KEY);
        const bool kvalid = s != a.cap;
        const uint32_t h = kvalid ? (uint32_t)key_hash(key) : na_hash;
        int d = occ ? hash_to_rank_u32(h, a.n_pes) : -1;
        if (d == a.rank) d = -1;  // owned here: stays in the table
        // warp-aggregated cursor: one atomic per (warp, destination)
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int leader = __ffs(peers) - 1;
        const int rank_in_peers = __popc(peers & ((1u << lane) - 1));
        unsigned long long base = 0;
        if (d >= 0 && lane == leader) base = atomicAdd(&a.cursors[d], (unsigned long long)__popc(peers));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (d >= 0) {
            const unsigned long long pos = base + rank_in_peers;
            if (pos < (unsigned long long)a.cap_rows) {
                unsigned long long* o = (unsigned long long*)((char*)a.peer_slabs[d] + XCHG_HDR_BYTES) + ((size_t)a.rank * a.cap_rows + pos) * a.row_words;
                o[0] = (unsigned long long)key;
                o[1] = kvalid ? 1ull : 0ull;
                for (int j = 0; j < a.n_acc; j++) o[2 + j] = a.acc[j][s];
            }
        }
    }
}
__global__ void xchg_post_counts_kernel(const unsigned long long* cursors, void* const* peer_slabs, int n_pes, int rank, long long cap_rows) {
    const int d = threadIdx.x;
    const unsigned long long c = d < n_pes ? cursors[d] : 0ull;
    const bool any_over = __any_sync(0xffffffffu, c > (unsigned long long)cap_rows);
    if (d < n_pes) ((unsigned long long*)peer_slabs[d])[rank] = (c > (unsigned long long)cap_rows ? (unsigned long long)cap_rows : c) | (any_over ? XCHG_OVERFLOW : 0ull);
}
__global__ void xchg_combine_slab_kernel(const __grid_constant__ CombineArgs a, const unsigned long long* hdr, int n_pes, long long cap_rows) {
    // a.in = first row of segment 0; flat row index = source * cap_rows + r (also what the fail list records)
    bool over = false;
    for (int s = 0; s < n_pes; s++) over |= (hdr[s] & XCHG_OVERFLOW) != 0;
    if (over) { if (blockIdx.x == 0 && threadIdx.x == 0) a.counters[7] = 1; return; }  // every rank sees the same flags: nobody combines
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int s = 0; s < n_pes; s++) {
        const int64_t n = (int64_t)(hdr[s] & ~XCHG_OVERFLOW);
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) combine_one_row(a, (int64_t)s * cap_rows + i);
    }
}

// ---- multi-column keys (2..4 integer key columns; SURVEY.md §8f "next" row 1, the reference's select-distinct /
// multi-key groupby: bodo/tests/test_streaming/test_groupby.py:111-177) -----------------------------------------
// A slot is claimed through a 64-bit tag word (hash of the key tuple, bit 63 set; 0 = empty, 1 = being written): the
// claiming thread CASes empty -> locked, writes the key columns + NA mask of the slot, fences and publishes the tag.
// Readers that find their own tag compare the full tuple (so the result is exact, the tag only prunes); readers that
// find `locked` re-read the slot.  Aggregate updates are the single-key kernel's apply_ops.
constexpr int MAX_KEYS = 4;

struct MkArgs {
    int nk;
    const void* key_data[MAX_KEYS];
    const uint8_t* key_valid[MAX_KEYS];
    int key_ctype[MAX_KEYS];
    int dropna;
    int64_t n_rows;
    const uint32_t* index_list;
    unsigned long long* tags;
    long long* mk[MAX_KEYS];
    unsigned char* mkmask;  // bit j = key column j is valid (not NA) in this group's key
    uint64_t cap;
    long long* counters;
    long long group_limit;
    uint32_t* fail_list;
    int n_ops;
    OpDesc ops[MAX_OPS];
    unsigned long long seq_base;  // unused (first / last are single-key only); apply_ops reads it
};

template <typename A>
__device__ __forceinline__ uint64_t find_or_insert_mk(const A& a, const long long* keys, unsigned int mask, unsigned long long tag) {
    const uint64_t m = a.cap - 1;
    uint64_t s = (tag >> 20) & m;
    for (uint64_t probes = 0; probes <= m;) {
        unsigned long long t = ld_acquire_u64(a.tags + s);
        if (t == tag) {
            bool eq = __ldcg(a.mkmask + s) == (unsigned char)mask;
            for (int j = 0; j < a.nk && eq; j++) eq = __ldcg(a.mk[j] + s) == keys[j];
            if (eq) return s;
        } else if (t == TAG_EMPTY) {
            if (a.group_limit >= 0) {
                long long tk = atomicAdd((unsigned long long*)&a.counters[0], 1ull);
                if (tk >= a.group_limit) { atomicAdd((unsigned long long*)&a.counters[0], (unsigned long long)-1ll); return ~0ull; }
            }
            unsigned long long old = atomicCAS(a.tags + s, TAG_EMPTY, TAG_LOCKED);
            if (old == TAG_EMPTY) {
                for (int j = 0; j < a.nk; j++) a.mk[j][s] = keys[j];
                a.mkmask[s] = (unsigned char)mask;
                __threadfence();
                atomicExch(a.tags + s, tag);  // publish
                return s;
            }
            if (a.group_limit >= 0) atomicAdd((unsigned long long*)&a.counters[0], (unsigned long long)-1ll);
            continue;  // somebody else took the slot: look at it again
        } else if (t == TAG_LOCKED) {
            continue;  // being written: re-read
        }
        s = (s + 1) & m;
        probes++;
    }
    return ~0ull;
}

__global__ void __launch_bounds__(256) groupby_consume_mk_kernel(const __grid_constant__ MkArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_rows; i += stride) {
        int64_t row = a.index_list ? (int64_t)a.index_list[i] : i;
        long long keys[MAX_KEYS];
        unsigned int mask = 0;
        for (int j = 0; j < a.nk; j++) {
            bool v = bit_valid(a.key_valid[j], row);
            keys[j] = v ? (long long)load_int_as_i64(a.key_data[j], a.key_ctype[j], row) : 0;
            mask |= v ? (1u << j) : 0u;
        }
        if (a.dropna && mask != (1u << a.nk) - 1u) continue;  // any NA key column drops the row (pandas dropna=True)
        uint64_t slot = find_or_insert_mk(a, keys, mask, mk_tag(keys, mask, a.nk));
        if (slot == ~0ull) {
            unsigned long long f = atomicAdd((unsigned long long*)&a.counters[1], 1ull);
            a.fail_list[f] = (uint32_t)row;
            continue;
        }
        apply_ops(a, slot, row);
    }
}

struct RehashMkArgs {
    int nk;
    const unsigned long long* old_tags; const long long* old_mk[MAX_KEYS]; const unsigned char* old_mask; uint64_t old_cap;
    unsigned long long* tags; long long* mk[MAX_KEYS]; unsigned char* mkmask; uint64_t cap;
    long long* counters; long long group_limit;  // group_limit < 0: no limit
    int n_acc;
    const unsigned long long* old_acc[2 * MAX_OPS];
    unsigned long long* new_acc[2 * MAX_OPS];
};
__global__ void rehash_mk_kernel(const __grid_constant__ RehashMkArgs a) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < a.old_cap; s += stride) {
        unsigned long long t = a.old_tags[s];
        if (!(t >> 63)) continue;
        long long keys[MAX_KEYS];
        for (int j = 0; j < a.nk; j++) keys[j] = a.old_mk[j][s];
        uint64_t ns = find_or_insert_mk(a, keys, a.old_mask[s], t);
        for (int j = 0; j < a.n_acc; j++) a.new_acc[j][ns] = a.old_acc[j][s];
    }
}
// Ownership of a multi-column key: hash_keys of the tuple exactly as the reference computes it on the original columns
// (sizeof(T) raw bytes per integer column, NA -> hash_na_val, hash_combine_boost for the further columns), from the
// widened int64 values the table stores.
struct MkOwner {
    int nk, n_pes, rank;
    int own_nk;  // 0: ownership by the hash of all key columns (the reference's hash_keys); 1: by the FIRST key column alone, hashed
                 // like a single-key state's key (nunique's nested (key, value) state: a key's pairs live where the key lives)
    const long long* mk[MAX_KEYS];
    const unsigned char* mkmask;
    int key_ctype[MAX_KEYS];
};
__device__ __forceinline__ uint32_t mk_ref_hash(const long long* keys, unsigned int mask, int nk, const int* ctypes) {
    const uint32_t na_hash = (uint32_t)xxh3_64_short(1ull, 8, SEED_HASH_PARTITION);
    uint32_t h = 0;
    for (int j = 0; j < nk; j++) {
        const uint32_t hj = !((mask >> j) & 1u) ? na_hash
                           : ctype_size(ctypes[j]) == 8 ? (uint32_t)xxh3_64_short((uint64_t)keys[j], 8, SEED_HASH_PARTITION)
                                                        : (uint32_t)xxh3_64_short((uint64_t)(uint32_t)keys[j], 4, SEED_HASH_PARTITION);
        h = j == 0 ? hj : hash_combine_boost(h, hj);
    }
    return h;
}
__device__ __forceinline__ uint32_t mk_owner_hash(const MkOwner& ow, const long long* keys, unsigned int mask) {
    if (ow.own_nk == 1) return (mask & 1u) ? (uint32_t)key_hash(keys[0]) : (uint32_t)xxh3_64_short(1ull, 8, SEED_HASH_PARTITION);
    return mk_ref_hash(keys, mask, ow.nk, ow.key_ctype);
}
// nunique: one thread per distinct (key, value) pair of the nested state; pairs whose value is NA do not count
struct NuniqueArgs {
    const long long* pk; const long long* pv; const unsigned char* pmask; const uint64_t* slot_of_out; long long n_pairs;
    long long* tkeys; uint64_t cap; long long* counters; int dropna;
    int n_acc; unsigned long long* acc[MAX_OPS];
};
__global__ void nunique_count_kernel(const __grid_constant__ NuniqueArgs a) {
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < a.n_pairs; p += (long long)gridDim.x * blockDim.x) {
        const uint64_t s = a.slot_of_out[p];
        const unsigned int m = a.pmask[s];
        if (!(m & 2u)) continue;  // NA value
        uint64_t slot;
        if (!(m & 1u)) { if (a.dropna) continue; slot = a.cap; a.counters[3] = 1; }
        else {
            const long long key = a.pk[s];
            if (key == EMPTY_KEY) { slot = a.cap + 1; a.counters[4] = 1; }
            else { slot = find_only(a.tkeys, a.cap, key); if (slot == ~0ull) continue; }  // (every key of a pair is a group of the outer table)
        }
        for (int j = 0; j < a.n_acc; j++) atomicAdd(a.acc[j] + slot, 1ull);
    }
}
__global__ void compact_mk_kernel(const unsigned long long* __restrict__ tags, uint64_t cap, long long* cursor, uint64_t* slot_of_out,
                                  const __grid_constant__ MkOwner ow) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s0 = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s0 < ((cap + 31) & ~31ull); s0 += stride) {
        bool occ = s0 < cap && (tags[s0] >> 63);
        if (occ && ow.n_pes > 1) {  // only the groups this rank owns (see compact_slots_kernel)
            long long keys[MAX_KEYS];
            for (int j = 0; j < ow.nk; j++) keys[j] = ow.mk[j][s0];
            occ = hash_to_rank_u32(mk_owner_hash(ow, keys, ow.mkmask[s0]), ow.n_pes) == ow.rank;
        }
        unsigned m = __ballot_sync(0xffffffffu, occ);
        int lane = threadIdx.x & 31;
        long long base = 0;
        if (lane == 0 && m) base = (long long)atomicAdd((unsigned long long*)cursor, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (occ) slot_of_out[base + __popc(m & ((1u << lane) - 1))] = s0;
    }
}
// ---- fused exchange for multi-column keys: wire row = [key 0 .. key nk-1][NA mask][accumulators] ----
struct XchgPackMkArgs {
    MkOwner ow;
    const unsigned long long* tags;
    uint64_t cap;
    int n_acc;
    const unsigned long long* acc[2 * MAX_OPS];
    int row_words;
    unsigned long long* cursors;
    void* const* peer_slabs;
    long long cap_rows;
};
__global__ void xchg_pack_remote_mk_kernel(const __grid_constant__ XchgPackMkArgs a) {
    const int lane = threadIdx.x & 31;
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < ((a.cap + 31) & ~31ull); s += stride) {
        const bool occ = s < a.cap && (a.tags[s] >> 63);
        long long keys[MAX_KEYS];
        unsigned int mask = 0;
        int d = -1;
        if (occ) {
            for (int j = 0; j < a.ow.nk; j++) keys[j] = a.ow.mk[j][s];
            mask = a.ow.mkmask[s];
            d = hash_to_rank_u32(mk_owner_hash(a.ow, keys, mask), a.ow.n_pes);
            if (d == a.ow.rank) d = -1;
        }
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int leader = __ffs(peers) - 1;
        const int rank_in_peers = __popc(peers & ((1u << lane) - 1));
        unsigned long long base = 0;
        if (d >= 0 && lane == leader) base = atomicAdd(&a.cursors[d], (unsigned long long)__popc(peers));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (d >= 0) {
            const unsigned long long pos = base + rank_in_peers;
            if (pos < (unsigned long long)a.cap_rows) {
                unsigned long long* o = (unsigned long long*)((char*)a.peer_slabs[d] + XCHG_HDR_BYTES) + ((size_t)a.ow.rank * a.cap_rows + pos) * a.row_words;
                for (int j = 0; j < a.ow.nk; j++) o[j] = (unsigned long long)keys[j];
                o[a.ow.nk] = mask;
                for (int j = 0; j < a.n_acc; j++) o[a.ow.nk + 1 + j] = a.acc[j][s];
            }
        }
    }
}
// combine of received multi-key rows: hdr != nullptr: the slab's n_pes segments; else the rows listed in c.index_list
__global__ void xchg_combine_mk_kernel(const __grid_constant__ MkArgs m, const __grid_constant__ CombineArgs c, const unsigned long long* hdr,
                                       int n_pes, long long cap_rows) {
    auto one = [&](int64_t row) {
        const unsigned long long* r = c.in + row * c.row_words;
        long long keys[MAX_KEYS];
        for (int j = 0; j < m.nk; j++) keys[j] = (long long)r[j];
        const unsigned int mask = (unsigned int)r[m.nk];
        const uint64_t slot = find_or_insert_mk(m, keys, mask, mk_tag(keys, mask, m.nk));
        if (slot == ~0ull) {
            unsigned long long f = atomicAdd((unsigned long long*)&c.counters[1], 1ull);
            c.fail_list[f] = (uint32_t)row;
            return;
        }
        combine_apply(c, slot, r + m.nk + 1);
    };
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (hdr == nullptr) {
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < c.n_rows; i += stride) one((int64_t)c.index_list[i]);
        return;
    }
    bool over = false;
    for (int s = 0; s < n_pes; s++) over |= (hdr[s] & XCHG_OVERFLOW) != 0;
    if (over) { if (blockIdx.x == 0 && threadIdx.x == 0) c.counters[7] = 1; return; }
    for (int s = 0; s < n_pes; s++) {
        const int64_t n = (int64_t)(hdr[s] & ~XCHG_OVERFLOW);
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) one((int64_t)s * cap_rows + i);
    }
}

struct EvalMkKeysArgs {
    int nk;
    const long long* mk[MAX_KEYS];
    const unsigned char* mkmask;
    const uint64_t* slot_of_out;
    const long long* n_out_ptr;
    int key_ctype[MAX_KEYS];
    void* out_keys[MAX_KEYS];
    uint32_t* out_key_valid[MAX_KEYS];  // nullptr for non-nullable key columns
};
__global__ void eval_mk_keys_kernel(const __grid_constant__ EvalMkKeysArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_out = *a.n_out_ptr;
    int64_t n_round = (n_out + 31) & ~31ll;
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n_round; p += stride) {
        bool in = p < n_out;
        uint64_t s = in ? a.slot_of_out[p] : 0;
        unsigned int mask = in ? a.mkmask[s] : 0;
        for (int j = 0; j < a.nk; j++) {
            if (in) store_int_typed(a.out_keys[j], a.key_ctype[j], p, a.mk[j][s]);
            if (a.out_key_valid[j]) {
                unsigned m = __ballot_sync(0xffffffffu, in && ((mask >> j) & 1));
                if ((threadIdx.x & 31) == 0) a.out_key_valid[j][p >> 5] = m;
            }
        }
    }
}

// ================================================================================================
// SM-partitioned groupby (SPG): the fast path for cardinalities whose accumulators fit the chip's
// aggregate shared memory (≈148 x 10k groups).  Motivation (profiles/r01_ubench*.txt): two global `red`s per
// row cap the direct kernel at ≈85 Grows/s and the key probe halves that again (L2 random-request rate), while
// 32-bit shared-memory atomics sustain the full HBM stream rate.  So rows travel to the SM that owns their key:
//
//   K1 spg_partition_tma_kernel : every CTA fetches TILE-row tiles with TMA bulk copies, counting-sorts them by owner
//        (= mulhi(hash, n_owners)) in shared memory, reserves one run per owner with a single global atomic per
//        (tile, owner) and copies the runs out with coalesced 16-byte stores -> owner buckets of (key, value) rows in HBM.
//   K2 spg_aggregate_kernel : one CTA per owner streams its bucket into a shared-memory hash table (key CAS,
//        SUM = two native 32-bit atomics with carry, COUNT = one), then flushes the table into the state's
//        global table with the ordinary find-or-insert + `red` (each key has one owner: <= n_groups per launch).
//   Algorithmic HBM traffic: 16 B/row read + 16 B/row bucket write + 16 B/row bucket read.
// A persistent single-kernel variant (L2-resident inboxes, inter-CTA barriers) was measured slower
// (profiles/r01_spg_persistent.txt): per-chunk work per SM is too small to amortise the barrier latency.
// Rows that do not fit (bucket overflow under skew, shared table full, marker key) take the direct global path
// inside the same kernels; rows that cannot even be inserted there (global table at its limit) are appended to
// a retry list in the partial-aggregate wire format and replayed by combine_partials_kernel after the table grew.
constexpr int SPG_THREADS = 1024;   // K2 (aggregate) threads per CTA
constexpr int SPG_TILE = 2048;
constexpr int SPG_MAX_OWNERS = 256;
// K1 reserves one run per owner per tile with a global atomic on the owner's row counter: ~10^7 atomics per launch.  With
// the 148 counters packed into ten cache lines K1's speed depended on where the array happened to land (0.80 ms against
// 1.00 ms per 2^27 rows for the same SASS after an unrelated allocation moved it), so every counter gets its own line.
constexpr int SPG_CNT_STRIDE = 16;
constexpr int SPG_STASH = 1024;     // K2: linear-probing stash slots for keys whose two buckets are full

struct SpgArgs {
    const long long* keys;
    const long long* vals;
    int64_t n_rows;
    int n_owners;
    // global table (state)
    long long* tkeys;
    uint64_t cap;
    unsigned long long* acc_sum;
    unsigned long long* acc_cnt;
    long long* counters;  // [0] groups, [1] retry rows, [4] marker key present
    long long group_limit;
    // owner buckets
    longlong2* bucket;            // [n_owners][bucket_cap]
    unsigned long long* bucket_cnt;  // [n_owners * SPG_CNT_STRIDE] rows appended per owner (may exceed bucket_cap: the excess
                                     // went the direct way); one counter per 128-byte line, see SPG_CNT_STRIDE
    long long bucket_cap;
    unsigned long long* retry;  // partial-aggregate rows [key][1][a0 of func 0][a0 of func 1]
    long long* retry_ctr;       // number of rows in `retry`
    int sum_first;              // order of the two accumulators in the wire format
    int ns;                     // shared-memory table slots (K2)
    int n_pass;                 // K2 passes over each owner bucket (pass p keeps the keys of sub-range p): > 1 when the
                                // estimated cardinality exceeds what the shared tables hold at once
    int reserve_tickets;  // K2n flush: the global table is empty — a CTA reserves the group tickets of all its slots with one atomic
    const long long* hot_tab;   // [SPG_HOT_SLOTS] heavy-hitter keys found by spg_hot_sample_kernel (EMPTY_KEY = free), or null
    const int* n_hot;           // number of keys in hot_tab (device memory: K1 reads it, the host never waits for it)
};

// cheap in-kernel hash for owner / shared-table slot (placement inside one GPU is free to choose; the rank
// placement that must match the reference uses xxh3, see shuffle.cu)
__device__ __forceinline__ uint64_t spg_hash(long long key) {
    uint64_t x = (uint64_t)key;
    return (x ^ (x >> 29)) * 0x9E3779B97F4A7C15ULL;
}
__device__ __forceinline__ unsigned int spg_owner(uint64_t h, int n_owners) { return __umulhi((unsigned int)(h >> 32), (unsigned int)n_owners); }
__device__ __forceinline__ unsigned int spg_slot(uint64_t h, int ns) { return __umulhi((unsigned int)(h >> 20), (unsigned int)ns); }

template <bool HAS_SUM, bool HAS_CNT>
__device__ __forceinline__ void spg_retry_row(const SpgArgs& a, long long key, unsigned long long sum, unsigned long long cnt) {
    unsigned long long f = atomicAdd((unsigned long long*)a.retry_ctr, 1ull);
    unsigned long long* r = a.retry + f * 4;
    r[0] = (unsigned long long)key; r[1] = 1ull;
    if (HAS_SUM && HAS_CNT) { r[2] = a.sum_first ? sum : cnt; r[3] = a.sum_first ? cnt : sum; }
    else { r[2] = HAS_SUM ? sum : cnt; r[3] = 0; }
}
template <bool HAS_SUM, bool HAS_CNT>
__device__ __forceinline__ void spg_direct_apply(const SpgArgs& a, long long key, unsigned long long sum, unsigned long long cnt) {
    uint64_t sl;
    if (key == EMPTY_KEY) { sl = a.cap + 1; a.counters[4] = 1; }
    else {
        sl = find_or_insert(a.tkeys, a.cap, key, a.counters, a.group_limit);
        if (sl == ~0ull) { spg_retry_row<HAS_SUM, HAS_CNT>(a, key, sum, cnt); return; }
    }
    if (HAS_SUM && sum) atomicAdd(a.acc_sum + sl, sum);
    if (HAS_CNT && cnt) atomicAdd(a.acc_cnt + sl, cnt);
}

// ---- steps shared by the K1 / K2 kernels of SPG, SPG-N (spgn.cuh) and SPG-G (spgg.cuh) -------------------------
// Force-inlined: the kernels were tuned with these steps written out, and `__noinline__` cold paths measured slower.

// K1: exclusive scan of a tile's class histogram hist[0, C) by warp 0 into lbase[0, C); lbase[C] = the tile's rows
__device__ __forceinline__ void spg_scan_hist(const unsigned int* hist, unsigned int* lbase, int C, int tid) {
    if (tid < 32) {
        unsigned int carry = 0;
        for (int base = 0; base < C; base += 32) {
            int j = base + tid;
            unsigned int x = j < C ? hist[j] : 0u, inc = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { unsigned int y = __shfl_up_sync(0xffffffffu, inc, d); if (tid >= d) inc += y; }
            if (j < C) lbase[j] = carry + inc - x;
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (tid == 0) lbase[C] = carry;
    }
}

// K2 shared tables are two-choice bucketed hash tables + stash: NB two-slot buckets, then SPG_STASH stash slots.
// The two candidate buckets of the key whose spg_hash is h:
__device__ __forceinline__ void spg_buckets(uint64_t h, unsigned int NB, unsigned int& b1, unsigned int& b2) {
    b1 = __umulhi((unsigned int)(h >> 20), NB);
    b2 = __umulhi(((unsigned int)h ^ (unsigned int)(h >> 44)) * 0x9E3779B1u, NB);  // low word of h remixed: independent of b1's bits 20..51 enough
    b2 = b2 == b1 ? (b1 + 1 == NB ? 0u : b1 + 1) : b2;
}
// the slot holding `key` in bucket b1 (slots c1.x, c1.y) or b2 (c2.x, c2.y), each read with one shared load; -1 = neither
template <typename P, typename K>
__device__ __forceinline__ int spg_find_slot(const P& c1, const P& c2, unsigned int b1, unsigned int b2, K key) {
    return c1.x == key ? (int)(2 * b1) : c1.y == key ? (int)(2 * b1 + 1) : c2.x == key ? (int)(2 * b2) : c2.y == key ? (int)(2 * b2 + 1) : -1;
}
// K2 slow path: the key's candidate slot, else a free candidate slot claimed by CAS, else find-or-insert in the stash behind
// the NS bucket slots; -1 = no room (the caller sends the row the direct way).  Balanced allocation: a new key goes to the
// EMPTIER of its two buckets (0.9 % of the keys overflow into the stash at 50 % load where first-fit left 2.2 % there —
// every row of a stash-resident key comes through here), and the four CAS attempts are skipped when both buckets are full
// (buckets never lose keys), so a stash-resident key costs two loads and one stash probe instead of four failed CAS round
// trips.  SPG-N's K2n has its own 32-bit copy, see spgn_aggregate_kernel.
__device__ __forceinline__ int spg_slow_slot(long long* skeys, int NS, unsigned int NB, long long key) {
    unsigned int b1, b2;
    spg_buckets(spg_hash(key), NB, b1, b2);
    const unsigned long long uk = (unsigned long long)key;
    const ulonglong2 c1 = *reinterpret_cast<const ulonglong2*>(skeys + 2 * b1);
    const ulonglong2 c2 = *reinterpret_cast<const ulonglong2*>(skeys + 2 * b2);
    const int f1 = (c1.x == (unsigned long long)EMPTY_KEY) + (c1.y == (unsigned long long)EMPTY_KEY);
    const int f2 = (c2.x == (unsigned long long)EMPTY_KEY) + (c2.y == (unsigned long long)EMPTY_KEY);
    int s = spg_find_slot(c1, c2, b1, b2, uk);
    if (s < 0 && f1 + f2 > 0) {
        const unsigned int first = f2 > f1 ? b2 : b1, second = f2 > f1 ? b1 : b2;
        const unsigned int cand[4] = {2 * first, 2 * first + 1, 2 * second, 2 * second + 1};
#pragma unroll
        for (int c = 0; c < 4 && s < 0; c++) {
            unsigned long long old = atomicCAS((unsigned long long*)&skeys[cand[c]], (unsigned long long)EMPTY_KEY, uk);
            if (old == (unsigned long long)EMPTY_KEY || old == uk) s = (int)cand[c];
        }
    }
    if (s < 0) {
        unsigned int st = (unsigned int)NS + ((unsigned int)(spg_hash(key) >> 12) & (SPG_STASH - 1));
        for (int probes = 0; probes < SPG_STASH && s < 0; probes++) {
            unsigned long long kk = (unsigned long long)skeys[st];
            if (kk == (unsigned long long)EMPTY_KEY) {
                unsigned long long old = atomicCAS((unsigned long long*)&skeys[st], (unsigned long long)EMPTY_KEY, uk);
                if (old == (unsigned long long)EMPTY_KEY) { s = (int)st; break; }
                kk = old;
            }
            if (kk == uk) { s = (int)st; break; }
            st = st + 1 == (unsigned int)NS + SPG_STASH ? (unsigned int)NS : st + 1;
        }
    }
    return s;
}

// ---- heavy hitters (skewed keys) ----------------------------------------------------------------------------
// A key that carries more than ~1/1024 of the rows (Zipf-like inputs: the top key of Zipf(1.1) over 1 M groups carries
// 12 %) would overload its owner: the bucket overflows into the direct path, where every row is a global atomic on ONE
// address (measured 10 Grows/s against 88 uniform).  Such keys are found once per operator state by counting a strided
// sample of the first launch (spg_hot_sample_kernel) and are then aggregated inside K1, in a per-CTA shared-memory
// accumulator table (two-slot buckets: one 16-byte load per row), and never reach the owner buckets.
constexpr int SPG_HOT_SLOTS = 128, SPG_HOT_BUCKETS = SPG_HOT_SLOTS / 2;
constexpr int SPG_HOT_SAMPLE = 1 << 15;  // sampled rows (one CTA counts them: the cost is per operator state, ~0.1 ms)
constexpr int SPG_HOT_TAB = 8192;        // counting-table slots of the sample kernel
constexpr size_t SPG_HOT_SAMPLE_SMEM = (size_t)SPG_HOT_TAB * 12 + SPG_HOT_SLOTS * 8;
__device__ __forceinline__ unsigned int spg_hot_bucket(uint64_t h) { return (unsigned int)(h >> 8) & (SPG_HOT_BUCKETS - 1); }

__global__ void __launch_bounds__(1024, 1) spg_hot_sample_kernel(const long long* keys, const long long* vals, int64_t n_rows, long long* hot_tab, int* n_hot) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    long long* tk = (long long*)smem_raw;                  // SPG_HOT_TAB keys
    unsigned int* tc = (unsigned int*)(tk + SPG_HOT_TAB);  // their sample counts
    long long* hk = (long long*)(tc + SPG_HOT_TAB);        // SPG_HOT_SLOTS: the hot table being built
    __shared__ unsigned int fill, nh, nwide;
    const int tid = threadIdx.x;
    for (int s = tid; s < SPG_HOT_TAB; s += 1024) { tk[s] = EMPTY_KEY; tc[s] = 0; }
    for (int s = tid; s < SPG_HOT_SLOTS; s += 1024) hk[s] = EMPTY_KEY;
    if (tid == 0) { fill = 0; nh = 0; nwide = 0; }
    __syncthreads();
    // the sample = 32 evenly spaced blocks of 1024 contiguous rows (one coalesced 8 KB read per block and column: a row-strided
    // sample touched a different DRAM page and TLB entry with every load and took 0.26 ms for 32 Ki rows)
    const int64_t S = n_rows < SPG_HOT_SAMPLE ? n_rows : SPG_HOT_SAMPLE;
    const int64_t block_stride = S == SPG_HOT_SAMPLE ? n_rows / (SPG_HOT_SAMPLE / 1024) : 1024;
    constexpr int ILP = 4;
    for (int64_t i0 = tid; i0 < S; i0 += 1024 * ILP) {
        long long kv[ILP];
#pragma unroll
        for (int u = 0; u < ILP; u++) {
            const int64_t i = i0 + (int64_t)u * 1024;
            const int64_t row = (i >> 10) * block_stride + (i & 1023);
            kv[u] = i < S ? keys[row] : EMPTY_KEY;
            // SPG-N (spgn.cuh): does this sampled row fit an (int32, int32) bucket row?
            if (i < S) {
                const long long v = vals ? vals[row] : 0;
                if (kv[u] != (long long)(int)kv[u] || (int)kv[u] == (int)0x80000000 || v != (long long)(int)v) atomicAdd(&nwide, 1u);
            }
        }
#pragma unroll
        for (int u = 0; u < ILP; u++) {
            const long long k = kv[u];
            if (k == EMPTY_KEY) continue;
            unsigned int s = (unsigned int)(spg_hash(k) >> 40) & (SPG_HOT_TAB - 1);
            for (int probes = 0; probes < 8; probes++) {  // heavy hitters arrive while the table is empty: short probes suffice
                long long kk = *(volatile long long*)&tk[s];
                if (kk == EMPTY_KEY) {
                    // the table only has to hold the heavy hitters, which show up early: stop admitting keys at 50 % load
                    if (*(volatile unsigned int*)&fill >= SPG_HOT_TAB / 2) break;
                    kk = (long long)atomicCAS((unsigned long long*)&tk[s], (unsigned long long)EMPTY_KEY, (unsigned long long)k);
                    if (kk == EMPTY_KEY) { atomicAdd(&fill, 1u); kk = k; }
                }
                if (kk == k) { atomicAdd(&tc[s], 1u); break; }
                s = (s + 1) & (SPG_HOT_TAB - 1);
            }
        }
    }
    __syncthreads();
    const unsigned int T = S >= (16 << 10) ? (unsigned int)(S >> 10) : 16u;  // hot = at least 1/1024 of the sample
    // admit candidates heaviest first (four count bands); a candidate whose two-slot bucket is taken stays an ordinary key
    for (int band = 3; band >= 0; band--) {
        const unsigned int lo = T << band, hi = band == 3 ? 0xffffffffu : (T << (band + 1));
        for (int s = tid; s < SPG_HOT_TAB; s += 1024) {
            const unsigned int c = tc[s];
            if (c < lo || c >= hi) continue;
            const long long k = tk[s];
            const unsigned int hb = spg_hot_bucket(spg_hash(k));
            unsigned long long old = atomicCAS((unsigned long long*)&hk[2 * hb], (unsigned long long)EMPTY_KEY, (unsigned long long)k);
            if (old != (unsigned long long)EMPTY_KEY) old = atomicCAS((unsigned long long*)&hk[2 * hb + 1], (unsigned long long)EMPTY_KEY, (unsigned long long)k);
            if (old == (unsigned long long)EMPTY_KEY) atomicAdd(&nh, 1u);
        }
        __syncthreads();
    }
    for (int s = tid; s < SPG_HOT_SLOTS; s += 1024) hot_tab[s] = hk[s];
    if (tid == 0) { n_hot[0] = (int)nh; n_hot[1] = (int)nwide; }
}

// K1: partition rows into owner buckets.  The tile's key and value slabs are fetched with cp.async.bulk (TMA, SASS UBLKCP)
// into a shared-memory staging area while the previous tile is being copied out, completion is signalled on an mbarrier
// (expect_tx / complete_tx), so no warp ever stalls on an HBM load and no row lives in registers across a barrier.  Then:
// hash, shared-memory histogram, run reservation, staging, coalesced 16-byte copy-out.  grid = persistent (SPG_TCTAS CTAs
// per SM), tiles are taken grid-stride.
constexpr int SPG_TTHREADS = 512;  // K1 threads per CTA (4 rows per thread per tile)
constexpr int SPG_TCTAS = 3;       // K1 CTAs per SM

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

template <bool HAS_SUM, bool HAS_CNT, bool HOT = false>
__global__ void __launch_bounds__(SPG_TTHREADS, SPG_TCTAS) spg_partition_tma_kernel(const __grid_constant__ SpgArgs a) {
    extern __shared__ __align__(128) unsigned char smem_tma_raw[];  // own name: the other kernels declare smem_raw with 16-byte alignment
    long long* raw_k = (long long*)smem_tma_raw;                               // [SPG_TILE] keys
    long long* raw_v = raw_k + SPG_TILE;                                       // [SPG_TILE] values
    longlong2* stage = (longlong2*)(raw_v + SPG_TILE);                         // SPG_TILE x 16
    unsigned long long* gbase = (unsigned long long*)(stage + SPG_TILE);      // SPG_MAX_OWNERS x 8
    uint64_t* mbar = (uint64_t*)(gbase + SPG_MAX_OWNERS);                      // 2 mbarriers (one used)
    unsigned int* hist = (unsigned int*)(mbar + 2);                            // SPG_MAX_OWNERS
    unsigned int* lbase = hist + SPG_MAX_OWNERS;                               // SPG_MAX_OWNERS + 1
    unsigned char* stage_owner = (unsigned char*)(lbase + SPG_MAX_OWNERS + 4);  // SPG_TILE
    long long* hkeys = (long long*)(stage_owner + SPG_TILE);                   // SPG_HOT_SLOTS heavy-hitter keys ...
    unsigned int* hlo = (unsigned int*)(hkeys + SPG_HOT_SLOTS);                // ... and this CTA's partial sums / row counts
    unsigned int* hhi = hlo + SPG_HOT_SLOTS;
    unsigned int* hcnt = hhi + SPG_HOT_SLOTS;
    const int G = a.n_owners, tid = threadIdx.x;
    constexpr bool hot_on = HOT;  // separate instantiation: the uniform-key kernel carries none of this (its SASS is the
                                  // kernel tuned before heavy hitters existed)
    if (hot_on)
        for (int s = tid; s < SPG_HOT_SLOTS; s += SPG_TTHREADS) { hkeys[s] = a.hot_tab[s]; hlo[s] = 0; hhi[s] = 0; hcnt[s] = 0; }
    constexpr int ROWS = SPG_TILE / SPG_TTHREADS;
    const int64_t n_tiles = (a.n_rows + SPG_TILE - 1) / SPG_TILE;
    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);  // unused (one raw tile buffer); initialised anyway, which keeps K1's SASS the tuned kernel's
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int j = tid; j < G; j += SPG_TTHREADS) hist[j] = 0;
    __syncthreads();
    // full tiles come in through TMA; a trailing partial tile is loaded with ordinary loads
    auto issue = [&](int64_t t) {
        const int64_t r0 = t * SPG_TILE;
        if (r0 + SPG_TILE <= a.n_rows && tid == 0) {
            mbar_expect_tx(&mbar[0], (HAS_SUM ? 2u : 1u) * SPG_TILE * 8u);
            tma_load_1d(raw_k, a.keys + r0, SPG_TILE * 8u, &mbar[0]);
            if (HAS_SUM) tma_load_1d(raw_v, a.vals + r0, SPG_TILE * 8u, &mbar[0]);
        }
    };
    uint32_t phase = 0;
    int64_t t = blockIdx.x;
    if (t < n_tiles) issue(t);
    for (; t < n_tiles; t += gridDim.x) {
        const int64_t r0 = t * SPG_TILE;
        const int64_t tn = t + gridDim.x;
        const bool full = r0 + SPG_TILE <= a.n_rows;
        if (full) {
            while (!mbar_try_wait(&mbar[0], phase)) {}
            phase ^= 1;
        } else {
            for (int j = tid; j < SPG_TILE; j += SPG_TTHREADS) {
                int64_t i = r0 + j;
                raw_k[j] = i < a.n_rows ? a.keys[i] : 0;
                raw_v[j] = (HAS_SUM && i < a.n_rows) ? a.vals[i] : 0;
            }
            __syncthreads();
        }
        int o[ROWS];
        unsigned int rk[ROWS];
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
            const int j = r * SPG_TTHREADS + tid;
            o[r] = -1;
            if (r0 + j >= a.n_rows) continue;
            const long long k = raw_k[j];
            if (k == EMPTY_KEY) { spg_direct_apply<HAS_SUM, HAS_CNT>(a, k, HAS_SUM ? (unsigned long long)raw_v[j] : 0ull, 1ull); continue; }
            const uint64_t h = spg_hash(k);
            if (hot_on) {  // heavy hitter: aggregate here, the row never reaches an owner bucket
                const unsigned int hb = spg_hot_bucket(h);
                const ulonglong2 hk2 = *reinterpret_cast<const ulonglong2*>(hkeys + 2 * hb);
                const int hs = hk2.x == (unsigned long long)k ? (int)(2 * hb) : hk2.y == (unsigned long long)k ? (int)(2 * hb + 1) : -1;
                if (hs >= 0) {
                    if (HAS_SUM) {
                        const unsigned long long v = (unsigned long long)raw_v[j];
                        const unsigned int lo = (unsigned int)v;
                        unsigned int hi = (unsigned int)(v >> 32);
                        const unsigned int old = atomicAdd(&hlo[hs], lo);
                        hi += (old + lo < old) ? 1u : 0u;
                        if (hi) atomicAdd(&hhi[hs], hi);
                    }
                    atomicAdd(&hcnt[hs], 1u);  // rows, also when only SUM is asked for: the group has to exist
                    continue;
                }
            }
            o[r] = (int)spg_owner(h, G);
            rk[r] = atomicAdd(&hist[o[r]], 1u);
        }
        __syncthreads();
        // reserve one run per owner: the global atomic's round trip (~1 us) is kept in a register and only waited for
        // after the staging pass, which needs the local prefix sums but not the global run start
        unsigned long long my_gbase = 0;
        if (tid >= SPG_TTHREADS - G) { int ow = tid - (SPG_TTHREADS - G); unsigned int cnt = hist[ow]; if (cnt) my_gbase = atomicAdd(&a.bucket_cnt[ow * SPG_CNT_STRIDE], (unsigned long long)cnt); }
        spg_scan_hist(hist, lbase, G, tid);
        __syncthreads();
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
            if (o[r] < 0) continue;
            const int j = r * SPG_TTHREADS + tid;
            unsigned int p = lbase[o[r]] + rk[r];
            stage[p] = make_longlong2(raw_k[j], HAS_SUM ? raw_v[j] : 0);
            stage_owner[p] = (unsigned char)o[r];
        }
        // publish run start minus local start, so the copy-out computes its destination with one add
        if (tid >= SPG_TTHREADS - G) { int ow = tid - (SPG_TTHREADS - G); gbase[ow] = my_gbase - lbase[ow]; }
        __syncthreads();  // the raw tile is free from here on
        if (tn < n_tiles) issue(tn);  // the next tile streams in during the copy-out
        const unsigned int n_tile = lbase[G];
        for (unsigned int p = tid; p < n_tile; p += SPG_TTHREADS) {
            unsigned int ow = stage_owner[p];
            unsigned long long off = gbase[ow] + p;
            longlong2 row = stage[p];
            if (off < (unsigned long long)a.bucket_cap) a.bucket[(size_t)ow * a.bucket_cap + off] = row;
            else spg_direct_apply<HAS_SUM, HAS_CNT>(a, row.x, (unsigned long long)row.y, 1ull);
        }
        for (int j = tid; j < G; j += SPG_TTHREADS) hist[j] = 0;
        __syncthreads();
    }
    if (hot_on) {  // this CTA's heavy-hitter partials -> global table (n_hot atomics per CTA)
        __syncthreads();
        for (int s = tid; s < SPG_HOT_SLOTS; s += SPG_TTHREADS)
            if (hcnt[s]) spg_direct_apply<HAS_SUM, HAS_CNT>(a, hkeys[s], (unsigned long long)hlo[s] | ((unsigned long long)hhi[s] << 32), (unsigned long long)hcnt[s]);
    }
}

// K2: one CTA per owner aggregates its bucket in shared memory, then flushes into the global table.
//
// Shared table = two-choice bucketed hash table + stash: every key has two candidate buckets of two slots (one 16-byte
// shared load each), so the hot lookup is two unconditional loads + four compares, no probe loop and no divergence
// (a linear-probing table spent > 50 % of its issue slots on loop control with ~15 of 32 lanes active,
// profiles/r01_spg_ncu_summary.txt; a collision-free key set runs the same loop 1.65x faster, scratch/ubench3.cu).
// Everything else — first appearance of a key (CAS into a free candidate slot), keys whose four candidates are taken
// (~2 % at this load: linear-probing stash behind the buckets), a full stash (direct global path), a non-zero high word
// of the sum — is parked and handled once per iteration behind the hot path.  Two racing inserts may put one key into
// both of its buckets: harmless, both partial sums are flushed into the same global group.
template <bool HAS_SUM, bool HAS_CNT>
__global__ void __launch_bounds__(SPG_THREADS, 1) spg_aggregate_kernel(const __grid_constant__ SpgArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NS = a.ns, NT = a.ns + SPG_STASH, tid = threadIdx.x, me = blockIdx.x;  // NS bucket slots + stash
    // 16 bytes per slot: key, low 32 bits of the sum (biased by 2^31 so sums of small positive AND negative values stay away
    // from the 32-bit wrap points), count.  The high word of an addition (value bits 32..63 plus the carry out of the low
    // word) is almost always zero; when it is not it is added straight to the global table: SUM stays exact mod 2^64.
    long long* skeys = (long long*)smem_raw;          // NT x 8
    unsigned int* slo = (unsigned int*)(skeys + NT);  // NT x 4
    unsigned int* scnt = slo + NT;
    const unsigned int NB = (unsigned int)NS / 2;
    const unsigned int NP = (unsigned int)a.n_pass, GP = (unsigned int)gridDim.x * NP;

    auto add = [&](int s, long long key, long long val) {
        if (HAS_SUM) {
            unsigned int lo = (unsigned int)(unsigned long long)val, hi = (unsigned int)((unsigned long long)val >> 32);
            unsigned int old = atomicAdd(&slo[s], lo);
            hi += (old + lo < old) ? 1u : 0u;  // carry of this very addition
            if (hi) spg_direct_apply<HAS_SUM, HAS_CNT>(a, key, (unsigned long long)hi << 32, 0ull);
        }
        if (HAS_CNT) atomicAdd(&scnt[s], 1u);
    };
    // slow path (spg_slow_slot), else the direct global path
    auto slow_upsert = [&](long long key, long long val) {
        const int s = spg_slow_slot(skeys, NS, NB, key);
        if (s < 0) { spg_direct_apply<HAS_SUM, HAS_CNT>(a, key, (unsigned long long)val, 1ull); return; }
        add(s, key, val);
    };

    unsigned long long n_in = a.bucket_cnt[me * SPG_CNT_STRIDE];
    if (n_in > (unsigned long long)a.bucket_cap) n_in = (unsigned long long)a.bucket_cap;
    const longlong2* src = a.bucket + (size_t)me * a.bucket_cap;
    constexpr int U = 4;  // independent bucket loads in flight per thread
    // rows of this thread: src[first + u * SPG_THREADS], u = 0..U-1, valid while < n_in
    auto process = [&](unsigned long long first, unsigned int pass, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;  // FULL: all U rows of every thread are in range (no padding checks)
        longlong2 row[U];
        int sl[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            unsigned long long p = first + (unsigned long long)u * SPG_THREADS;
            row[u] = (FULL || p < n_in) ? __ldcs(src + p) : make_longlong2(EMPTY_KEY, 0);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {  // hot lookups: branch-free
            unsigned int b1, b2;
            spg_buckets(spg_hash(row[u].x), NB, b1, b2);
            const ulonglong2 k1 = *reinterpret_cast<const ulonglong2*>(skeys + 2 * b1);
            const ulonglong2 k2 = *reinterpret_cast<const ulonglong2*>(skeys + 2 * b2);
            sl[u] = spg_find_slot(k1, k2, b1, b2, (unsigned long long)row[u].x);
            if (!FULL && row[u].x == EMPTY_KEY) sl[u] = -2;  // padding lane
            // multi-pass: owner = mulhi(hash_hi, G) = mulhi(hash_hi, G * NP) / NP; this pass keeps sub-range `pass` only
            if (NP > 1 && __umulhi((unsigned int)(spg_hash(row[u].x) >> 32), GP) - (unsigned int)me * NP != pass) sl[u] = -2;
        }
        long long pk = 0, pv = 0;
        bool parked = false;
#pragma unroll
        for (int u = 0; u < U; u++) {
            if (sl[u] >= 0) add(sl[u], row[u].x, row[u].y);
            else if (sl[u] == -1) {
                if (!parked) { pk = row[u].x; pv = row[u].y; parked = true; }
                else slow_upsert(row[u].x, row[u].y);  // second slow row of this thread in one iteration: rare
            }
        }
        if (parked) slow_upsert(pk, pv);
    };
    const unsigned long long step = (unsigned long long)U * SPG_THREADS;
    const unsigned long long n_full = n_in / step * step;
    for (unsigned int pass = 0; pass < NP; pass++) {
        for (int s = tid; s < NT; s += SPG_THREADS) { skeys[s] = EMPTY_KEY; slo[s] = 0x80000000u; scnt[s] = 0; }
        __syncthreads();
        for (unsigned long long base = 0; base < n_full; base += step) process(base + tid, pass, std::true_type{});
        if (n_full < n_in) process(n_full + tid, pass, std::false_type{});
        __syncthreads();
        // flush the shared table into the state's global table
        for (int s = tid; s < NT; s += SPG_THREADS) {
            long long key = skeys[s];
            if (key == EMPTY_KEY) continue;
            unsigned long long sum = (unsigned long long)slo[s] - 0x80000000ull;  // remove the bias (wraps mod 2^64)
            spg_direct_apply<HAS_SUM, HAS_CNT>(a, key, sum, (unsigned long long)scnt[s]);
        }
        __syncthreads();
    }
}

#include "spgn.cuh"  // SPG-N: narrow (int32 key, int32 value) bucket rows: 32 instead of 48 B/row of HBM traffic
#include "spgg.cuh"  // SPG-G: the same two kernels for nullable / 4-byte / mean / min / max signatures

// ---- low-cardinality kernel (LC): every CTA keeps a private shared-memory table of ALL groups ----------------
// Used when the (estimated) number of groups fits one CTA's table (<= LC_SLOTS / 2), e.g. BASELINE.json configs[0]
// (20 M rows, 30 groups) where every row of a warp hits one of a handful of hot keys.  Rows are pre-aggregated inside
// the warp when the whole warp holds ONE key (hot key / clustered input): the warp's SUM is formed with four
// __reduce_add_sync (REDUX) over 16-bit limbs (exact: 32 lanes x 65535 < 2^32 per limb, limbs recombined mod 2^64),
// its COUNT is popc(active), and one lane touches the shared table; otherwise each lane updates the CTA-private table
// (CAS-probe + native 32-bit atomics with carry).  One pass over the input: 16 B/row of HBM traffic, no global atomics
// until the final flush.
constexpr int LC_THREADS = 512;
// per-CTA table slots (20 B each); groups beyond LC_SLOTS / 2 take the direct path.  Two instantiations: 1024 slots
// (3 CTAs = 1536 threads per SM, for <= 256 expected groups) and 4096 slots (2 CTAs per SM, <= 1024 expected groups).
constexpr int LC_SLOTS_BIG = 4096, LC_SLOTS_SMALL = 1024;

template <bool HAS_SUM, bool HAS_CNT, int LC_SLOTS, int MIN_CTAS>
__global__ void __launch_bounds__(LC_THREADS, MIN_CTAS) groupby_lowcard_kernel(const __grid_constant__ SpgArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    long long* lkeys = (long long*)smem_raw;                 // LC_SLOTS x 8
    unsigned int* llo = (unsigned int*)(lkeys + LC_SLOTS);  // low / high words of the sum, count
    unsigned int* lhi = llo + LC_SLOTS;
    unsigned int* lcnt = lhi + LC_SLOTS;
    unsigned int* misc = lcnt + LC_SLOTS;
    const int tid = threadIdx.x, lane = tid & 31;
    for (int s = tid; s < LC_SLOTS; s += LC_THREADS) { lkeys[s] = EMPTY_KEY; llo[s] = 0; lhi[s] = 0; lcnt[s] = 0; }
    if (tid == 0) misc[0] = 0;
    __syncthreads();

    auto leader_upsert = [&](long long key, unsigned long long sum, unsigned int cnt) {
        unsigned int s = (unsigned int)(spg_hash(key) >> 32) & (LC_SLOTS - 1);
        bool done = false;
        for (int probes = 0; probes < LC_SLOTS; probes++) {
            long long kk = lkeys[s];
            if (kk == EMPTY_KEY) {
                unsigned int t = atomicAdd(&misc[0], 1u);
                if (t >= LC_SLOTS / 2) { atomicSub(&misc[0], 1u); break; }
                long long prev = (long long)atomicCAS((unsigned long long*)&lkeys[s], (unsigned long long)EMPTY_KEY, (unsigned long long)key);
                if (prev == EMPTY_KEY) { done = true; break; }
                atomicSub(&misc[0], 1u);
                kk = prev;
            }
            if (kk == key) { done = true; break; }
            s = (s + 1) & (LC_SLOTS - 1);
        }
        if (!done) { spg_direct_apply<HAS_SUM, HAS_CNT>(a, key, sum, (unsigned long long)cnt); return; }
        if (HAS_SUM) {
            unsigned int lo = (unsigned int)sum, hi = (unsigned int)(sum >> 32);
            unsigned int old = atomicAdd(&llo[s], lo);
            hi += (old + lo < old) ? 1u : 0u;
            if (hi) atomicAdd(&lhi[s], hi);
        }
        if (HAS_CNT) atomicAdd(&lcnt[s], cnt);
    };

    // warp-uniform trip count (bounds checked per row): the warp collectives below need converged warps
    const int64_t stride = (int64_t)gridDim.x * LC_THREADS * 2;
    const int64_t n_round = (a.n_rows + 63) & ~63ll;
    for (int64_t i = ((int64_t)blockIdx.x * LC_THREADS + tid) * 2; i < n_round; i += stride) {
        long long k[2] = {0, 0}, v[2] = {0, 0};
        bool ok[2] = {i < a.n_rows, i + 1 < a.n_rows};
        if (ok[1]) {
            longlong2 kk = __ldcs(reinterpret_cast<const longlong2*>(a.keys + i));
            k[0] = kk.x; k[1] = kk.y;
            if (HAS_SUM) { longlong2 vv = __ldcs(reinterpret_cast<const longlong2*>(a.vals + i)); v[0] = vv.x; v[1] = vv.y; }
        } else if (ok[0]) {
            k[0] = a.keys[i];
            if (HAS_SUM) v[0] = a.vals[i];
        }
#pragma unroll
        for (int r = 0; r < 2; r++) {
            if (ok[r] && k[r] == EMPTY_KEY) { spg_direct_apply<HAS_SUM, HAS_CNT>(a, k[r], (unsigned long long)v[r], 1ull); ok[r] = false; }
            const unsigned act = __ballot_sync(0xffffffffu, ok[r]);
            if (!ok[r]) continue;
            // warp-uniform shortcut (one hot key, sorted / clustered input): reduce the whole warp with REDUX and let one
            // lane update the table.  Otherwise every lane updates the CTA table itself: for >= ~30 distinct keys per warp
            // a __match_any_sync based pre-aggregation was measured 3-5x slower (it serialises over the distinct keys).
            const long long k0 = __shfl_sync(act, k[r], __ffs(act) - 1);
            const bool uniform = __all_sync(act, k[r] == k0) && act != (1u << (__ffs(act) - 1));
            if (uniform) {
                unsigned long long sum = 0;
                if (HAS_SUM) {
                    const unsigned long long u = (unsigned long long)v[r];
                    const unsigned int l0 = __reduce_add_sync(act, (unsigned int)(u & 0xffffu));
                    const unsigned int l1 = __reduce_add_sync(act, (unsigned int)((u >> 16) & 0xffffu));
                    const unsigned int l2 = __reduce_add_sync(act, (unsigned int)((u >> 32) & 0xffffu));
                    const unsigned int l3 = __reduce_add_sync(act, (unsigned int)(u >> 48));
                    sum = (unsigned long long)l0 + ((unsigned long long)l1 << 16) + ((unsigned long long)l2 << 32) + ((unsigned long long)l3 << 48);
                }
                if (lane == __ffs(act) - 1) leader_upsert(k0, sum, (unsigned int)__popc(act));
            } else {
                leader_upsert(k[r], (unsigned long long)v[r], 1u);
            }
        }
    }
    __syncthreads();
    for (int s = tid; s < LC_SLOTS; s += LC_THREADS) {
        long long key = lkeys[s];
        if (key == EMPTY_KEY) continue;
        unsigned long long sum = (unsigned long long)llo[s] | ((unsigned long long)lhi[s] << 32);
        spg_direct_apply<HAS_SUM, HAS_CNT>(a, key, sum, (unsigned long long)lcnt[s]);
    }
}

// ================================================================================================
// Host side
// ================================================================================================

// One user-visible aggregate: evaluated from the accumulators of `prim[0..n_prim)` (indices into the primitive list)
struct OutSpec {
    int ftype;
    int kind;        // OpKind used by eval_output_kernel
    int prim[3];
    int n_prim;
    int out_ctype, out_arrtype;
};

struct FuncSpec {
    int ftype;
    int in_col;  // physical input column or -1 (size)
    int in_ctype;
    int in_arrtype;
    int kind;
    int out_ctype;
    int out_arrtype;
    bool has_a1;
    unsigned long long init0;
    unsigned long long init1 = 0;  // initial value of the second accumulator
};

class GroupbyState {
   public:
    int device;
    cudaStream_t stream;
    cudaStream_t copy_stream = nullptr;
    int n_cols;
    std::vector<int8_t> c_types, arr_types;
    int n_funcs;                  // primitive accumulator functions (what the kernels, the table and the exchange see)
    std::vector<FuncSpec> funcs;
    int n_outs = 0;               // aggregates the caller asked for (output columns)
    std::vector<OutSpec> outs;
    bool dropna, parallel;
    bool has_firstlast = false;
    int owner_nk = 0;  // see MkOwner::own_nk
    // nunique: one nested distinct state over (key, value) per value column; `prims` = the K_NUNIQUE accumulators it feeds
    struct NuInner { int in_col; std::unique_ptr<GroupbyState> st; std::vector<int> prims; };
    std::vector<NuInner> nu_inner;
    bool nu_applied = false;
    int n_pes, rank;
    int64_t output_batch_size;
    int sms;

    uint64_t cap = 0;
    int nk = 1;  // number of key columns (2..4 = multi-key table: d_tags / d_mk / d_mkmask instead of d_keys)
    DevBuf d_tags, d_mk[MAX_KEYS], d_mkmask;
    DevBuf d_out_mk[MAX_KEYS], d_out_mk_valid[MAX_KEYS];
    DevBuf d_keys;
    std::vector<DevBuf> d_a0, d_a1;
    DevBuf d_counters;
    long long* h_counters = nullptr;  // pinned
    PooledBuf d_fail;
    int64_t n_groups = 0;

    // host-input staging (double buffered, per used column)
    std::vector<DevBuf> stage[2];
    cudaEvent_t stage_free[2] = {nullptr, nullptr}, stage_ready[2] = {nullptr, nullptr};

    // finalize / output
    bool finalized = false;
    int64_t n_out = 0, out_cursor = 0;
    DevBuf d_slot_of_out, d_out_keys, d_out_key_valid;
    std::vector<DevBuf> d_out_data, d_out_valid;
    // exchange
    DevBuf d_dest_count;
    std::vector<long long> h_dest_count;
    int64_t packed_rows = 0;

    // host-side time accounting (printed at delete when B200_TRACE is set)
    double t_ctor = 0, t_grow = 0, t_alloc = 0, t_spg = 0, t_finalize = 0;
    static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
    // metrics
    int64_t rows_consumed = 0, rebuilds = 0, launches = 0, fail_rows = 0;
    bool build_done = false;
    // optional per-launch timing of the consume kernel (bench.py roofline): CUDA events on `stream`
    bool profiling = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    int64_t consume_launches = 0;
    double consume_kernel_us() {
        double us = 0;
        for (auto& pr : prof_events) {
            float ms = 0;
            if (cudaEventSynchronize(pr.second) == cudaSuccess && cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) us += ms * 1000.0;
        }
        return us;
    }

    GroupbyState(const int8_t* ct, const int8_t* at, int n_arrs, const int32_t* ftypes, const int32_t* f_in_offsets,
                 const int32_t* f_in_cols, int n_funcs_, uint64_t n_keys, int64_t out_bs, bool parallel_, bool dropna_,
                 int device_, int n_pes_, int rank_, int64_t expected_groups, cudaStream_t stream_)
        : device(device_), stream(stream_), n_cols(n_arrs), n_funcs(0), n_outs(n_funcs_), dropna(dropna_), parallel(parallel_),
          n_pes(n_pes_), rank(rank_), output_batch_size(out_bs) {
        B200_REQUIRE(n_keys >= 1 && n_keys <= (uint64_t)MAX_KEYS, "b200 groupby: between 1 and 4 key columns are supported");
        nk = (int)n_keys;
        B200_REQUIRE(n_arrs >= 1, "b200 groupby: empty build schema");
        B200_REQUIRE(n_funcs_ <= 2 * MAX_OPS, "b200 groupby: too many aggregate functions");
        c_types.assign(ct, ct + n_arrs);
        arr_types.assign(at, at + n_arrs);
        B200_REQUIRE(n_arrs >= nk, "b200 groupby: fewer columns than keys");
        for (int kc = 0; kc < nk; kc++) {
            int kct = c_types[kc];
            B200_REQUIRE(ctype_size(kct) > 0 && !ctype_is_float(kct), "b200 groupby: key columns must be integer/date typed");
            B200_REQUIRE(arr_types[kc] == ARR_NUMPY || arr_types[kc] == ARR_NULLABLE, "b200 groupby: unsupported key array type");
        }
        if (!parallel) { n_pes = 1; rank = 0; }
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        sms = num_sms(device);
        for (int j = 0; j < n_outs; j++) {
            FuncSpec f{};
            f.ftype = ftypes[j];
            int n_in = f_in_offsets[j + 1] - f_in_offsets[j];
            B200_REQUIRE(n_in <= 1, "b200 groupby: functions with more than one input column are not supported");
            f.in_col = n_in == 1 ? f_in_cols[f_in_offsets[j]] : -1;
            if (f.ftype != FT_SIZE) B200_REQUIRE(f.in_col >= nk && f.in_col < n_arrs, "b200 groupby: bad f_in_cols entry");
            f.in_ctype = f.in_col >= 0 ? c_types[f.in_col] : CT_INT64;
            f.in_arrtype = f.in_col >= 0 ? arr_types[f.in_col] : ARR_NUMPY;
            B200_REQUIRE(f.in_arrtype == ARR_NUMPY || f.in_arrtype == ARR_NULLABLE, "b200 groupby: unsupported value array type");
            B200_REQUIRE(ctype_size(f.in_ctype) > 0, "b200 groupby: unsupported value dtype");
            bool isf = ctype_is_float(f.in_ctype);
            f.has_a1 = false;
            f.init0 = 0;
            // output typing: get_groupby_output_dtype (groupby/_groupby_common.cpp:561-668)
            switch (f.ftype) {
                case FT_SIZE: f.kind = K_SIZE; f.out_ctype = CT_INT64; f.out_arrtype = ARR_NUMPY; break;
                case FT_COUNT: f.kind = K_COUNT; f.out_ctype = CT_INT64; f.out_arrtype = ARR_NUMPY; break;
                case FT_SUM:
                    f.kind = isf ? K_SUM_F64 : K_SUM_I64;
                    f.out_ctype = isf ? f.in_ctype : (ctype_is_signed_int(f.in_ctype) || f.in_ctype == CT_BOOL ? CT_INT64 : CT_UINT64);
                    f.out_arrtype = f.in_ctype == CT_BOOL ? ARR_NULLABLE : f.in_arrtype;
                    break;
                case FT_MEAN: f.kind = K_MEAN; f.out_ctype = CT_FLOAT64; f.out_arrtype = ARR_NULLABLE; f.has_a1 = true; break;
                case FT_MIN: case FT_MAX: {
                    B200_REQUIRE(f.in_ctype != CT_UINT64, "b200 groupby: min/max of uint64 is not supported");
                    bool mn = f.ftype == FT_MIN;
                    f.kind = isf ? (mn ? K_MIN_F64 : K_MAX_F64) : (mn ? K_MIN_I64 : K_MAX_I64);
                    f.out_ctype = f.in_ctype; f.out_arrtype = f.in_arrtype;
                    f.has_a1 = f.in_arrtype == ARR_NULLABLE;
                    if (isf) f.init0 = mn ? ~0ull : 0ull;
                    else f.init0 = mn ? (unsigned long long)INT64_MAX : (unsigned long long)INT64_MIN;
                    break;
                }
                case FT_NUNIQUE: {
                    // nunique_computation (bodo/libs/groupby/_groupby_col_set.cpp:1771-1810): distinct non-NA values per group
                    B200_REQUIRE(nk == 1, "b200 groupby: nunique is supported for single-column keys");
                    B200_REQUIRE(!isf, "b200 groupby: nunique of a float column is not supported (integer / date / bool value columns)");
                    f.kind = K_NUNIQUE; f.out_ctype = CT_INT64; f.out_arrtype = ARR_NUMPY;
                    size_t q = 0;
                    while (q < nu_inner.size() && nu_inner[q].in_col != f.in_col) q++;
                    if (q == nu_inner.size()) { nu_inner.emplace_back(); nu_inner[q].in_col = f.in_col; }
                    nu_inner[q].prims.push_back((int)funcs.size());
                    break;
                }
                case FT_FIRST: case FT_LAST:
                    B200_REQUIRE(nk == 1, "b200 groupby: first / last are supported for single-column keys");
                    f.kind = f.ftype == FT_FIRST ? K_FIRST : K_LAST;
                    f.out_ctype = f.in_ctype; f.out_arrtype = f.in_arrtype;
                    f.has_a1 = true; f.init1 = f.ftype == FT_FIRST ? ~0ull : 0ull;
                    has_firstlast = true;
                    break;
                case FT_VAR: case FT_STD: case FT_VAR_POP: case FT_STD_POP: case FT_SKEW: {
                    // composite: a K_MEAN pair (sum, count) + sum of squares (+ sum of cubes), all over the same input column
                    OutSpec o{};
                    o.ftype = f.ftype;
                    o.kind = f.ftype == FT_VAR ? E_VAR : f.ftype == FT_STD ? E_STD : f.ftype == FT_VAR_POP ? E_VAR_POP : f.ftype == FT_STD_POP ? E_STD_POP : E_SKEW;
                    o.out_ctype = CT_FLOAT64; o.out_arrtype = ARR_NULLABLE;
                    const int kinds[3] = {K_MEAN, K_SUMSQ_F64, K_SUMCUBE_F64};
                    o.n_prim = f.ftype == FT_SKEW ? 3 : 2;
                    for (int q = 0; q < o.n_prim; q++) {
                        FuncSpec pf = f;
                        pf.kind = kinds[q]; pf.has_a1 = q == 0; pf.out_ctype = CT_FLOAT64; pf.out_arrtype = ARR_NULLABLE;
                        // composites (and a plain mean) over the same input column share their accumulator columns
                        int found = -1;
                        for (int e = 0; e < (int)funcs.size(); e++)
                            if (funcs[e].kind == pf.kind && funcs[e].in_col == pf.in_col) { found = e; break; }
                        if (found < 0) { found = (int)funcs.size(); funcs.push_back(pf); }
                        o.prim[q] = found;
                    }
                    outs.push_back(o);
                    continue;
                }
                default:
                    throw Error("b200 groupby: unsupported aggregate function ftype=" + std::to_string(f.ftype) +
                                " (supported: size, sum, count, nunique, mean, min, max, first, last, var, std, var_pop, std_pop, skew)");
            }
            OutSpec o{};
            o.ftype = f.ftype; o.kind = f.kind; o.prim[0] = (int)funcs.size(); o.n_prim = 1; o.out_ctype = f.out_ctype; o.out_arrtype = f.out_arrtype;
            outs.push_back(o);
            funcs.push_back(f);
        }
        n_funcs = (int)funcs.size();
        B200_REQUIRE(n_funcs <= MAX_OPS, "b200 groupby: too many aggregate functions (composite ones count their accumulator columns)");
        d_a0.resize(n_funcs); d_a1.resize(n_funcs);
        d_out_data.resize(n_outs); d_out_valid.resize(n_outs);
        d_counters.alloc(8 * sizeof(long long));
        B200_CUDA(cudaMemsetAsync(d_counters.p, 0, 8 * sizeof(long long), stream));
        h_counters = (long long*)pinned_acquire(8 * sizeof(long long));
        expected_groups_hint = expected_groups > 0 ? expected_groups : 0;
        uint64_t want = 1ull << 16;
        if (expected_groups > 0) { while (want < (uint64_t)expected_groups * 2) want <<= 1; }
        else want = 1ull << 21;
        double t0 = now();
        alloc_table(want, d_keys, d_a0, d_a1);
        if (nk > 1) alloc_mk(want, d_tags, d_mk, d_mkmask);
        cap = want;
        for (auto& ni : nu_inner) {  // nested distinct states over (key, value); their groups are owned where the KEY is owned
            const int8_t ict[2] = {c_types[0], c_types[ni.in_col]}, iat[2] = {arr_types[0], arr_types[ni.in_col]};
            const int32_t no_off[1] = {0};
            ni.st.reset(new GroupbyState(ict, iat, 2, nullptr, no_off, nullptr, 0, 2, 1ll << 40, parallel, /*dropna=*/false, device, n_pes, rank,
                                         expected_groups > 0 ? expected_groups * 4 : 0, stream));
            ni.st->owner_nk = 1;
        }
        t_ctor = now() - t0;
    }

    ~GroupbyState() {
        cudaSetDevice(device);
        scratch_set_stream(stream);
        cudaStreamSynchronize(stream);
        if (getenv("B200_TRACE"))
            fprintf(stderr, "[b200 groupby state] ctor %.3f ms, grow %.3f ms (%lld rebuilds), spg alloc %.3f ms, spg loop %.3f ms, finalize %.3f ms, cap %llu\n",
                    t_ctor * 1e3, t_grow * 1e3, (long long)rebuilds, t_alloc * 1e3, t_spg * 1e3, t_finalize * 1e3, (unsigned long long)cap);
        if (copy_stream) { cudaStreamSynchronize(copy_stream); cudaStreamDestroy(copy_stream); }
        for (int b = 0; b < 2; b++) { if (stage_free[b]) cudaEventDestroy(stage_free[b]); if (stage_ready[b]) cudaEventDestroy(stage_ready[b]); }
        pinned_release(h_counters, 8 * sizeof(long long));
        pinned_release(h_spg, 24 * sizeof(long long));
        for (int b = 0; b < 2; b++) if (spg_ev[b]) cudaEventDestroy(spg_ev[b]);
        for (auto& pr : prof_events) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
    }

    int grid_for(int64_t n, int per_thread = 1, int block = 256) const {
        int64_t want = (n + (int64_t)block * per_thread - 1) / ((int64_t)block * per_thread);
        int64_t maxg = (int64_t)sms * 8;  // 8 resident CTAs of 256 threads per SM
        return (int)std::max<int64_t>(1, std::min(want, maxg));
    }

    void fill(void* p, uint64_t n, unsigned long long v) {
        if (v == 0) { B200_CUDA(cudaMemsetAsync(p, 0, n * 8, stream)); return; }
        fill_u64_kernel<<<grid_for((int64_t)n), 256, 0, stream>>>((unsigned long long*)p, n, v);
        launches++;
    }

    void alloc_table(uint64_t c, DevBuf& keys, std::vector<DevBuf>& a0, std::vector<DevBuf>& a1) {
        B200_REQUIRE(c <= (1ull << 32), "b200 groupby: hash table would exceed 2^32 slots");
        if (nk == 1) {
            keys.alloc((c + 2) * 8);
            fill(keys.p, c + 2, (unsigned long long)EMPTY_KEY);
        }
        for (int j = 0; j < n_funcs; j++) {
            a0[j].alloc((c + 2) * 8);
            fill(a0[j].p, c + 2, funcs[j].init0);
            if (funcs[j].has_a1) { a1[j].alloc((c + 2) * 8); fill(a1[j].p, c + 2, funcs[j].init1); }
        }
    }

    void read_counters() {
        B200_CUDA(cudaMemcpyAsync(h_counters, d_counters.p, 8 * sizeof(long long), cudaMemcpyDeviceToHost, stream));
        B200_CUDA(cudaStreamSynchronize(stream));
        n_groups = h_counters[0];
    }

    void grow(uint64_t new_cap) {
        double t0 = now();
        struct Acc { double& t; double t0; ~Acc() { t += now() - t0; } } acc{t_grow, t0};
        if (nk > 1) { grow_mk(new_cap); return; }
        DevBuf nkeys; std::vector<DevBuf> na0(n_funcs), na1(n_funcs);
        alloc_table(new_cap, nkeys, na0, na1);
        RehashArgs ra{};
        ra.old_keys = d_keys.as<long long>(); ra.old_cap = cap; ra.new_keys = nkeys.as<long long>(); ra.new_cap = new_cap;
        int n = 0;
        for (int j = 0; j < n_funcs; j++) {
            ra.old_acc[n] = d_a0[j].as<unsigned long long>(); ra.new_acc[n++] = na0[j].as<unsigned long long>();
            if (funcs[j].has_a1) { ra.old_acc[n] = d_a1[j].as<unsigned long long>(); ra.new_acc[n++] = na1[j].as<unsigned long long>(); }
        }
        ra.n_acc = n;
        rehash_kernel<<<grid_for((int64_t)cap + 2), 256, 0, stream>>>(ra);
        launches++;
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaStreamSynchronize(stream));  // old arrays are freed below
        d_keys = std::move(nkeys);
        for (int j = 0; j < n_funcs; j++) { d_a0[j] = std::move(na0[j]); d_a1[j] = std::move(na1[j]); }
        cap = new_cap;
        rebuilds++;
    }
    // grow the table (at least doubling it) until n_groups + pending groups fit under its group limit of cap / 2
    void grow_to_hold(int64_t pending) {
        uint64_t nc = cap;
        while (nc < 2ull * (uint64_t)(n_groups + pending)) nc <<= 1;
        if (nc == cap) nc <<= 1;
        grow(nc);
    }

    // ---- multi-key table management ----
    void alloc_mk(uint64_t c, DevBuf& tags, DevBuf* mk, DevBuf& mask) {
        tags.alloc(c * 8);
        B200_CUDA(cudaMemsetAsync(tags.p, 0, c * 8, stream));
        for (int j = 0; j < nk; j++) mk[j].alloc(c * 8);
        mask.alloc(c);
    }
    void grow_mk(uint64_t new_cap) {
        DevBuf ntags, nmk[MAX_KEYS], nmask, dummy;
        std::vector<DevBuf> na0(n_funcs), na1(n_funcs);
        alloc_table(new_cap, dummy, na0, na1);
        alloc_mk(new_cap, ntags, nmk, nmask);
        RehashMkArgs ra{};
        ra.nk = nk; ra.old_tags = d_tags.as<unsigned long long>(); ra.old_mask = d_mkmask.as<unsigned char>(); ra.old_cap = cap;
        ra.tags = ntags.as<unsigned long long>(); ra.mkmask = nmask.as<unsigned char>(); ra.cap = new_cap;
        ra.counters = d_counters.as<long long>(); ra.group_limit = -1;
        for (int j = 0; j < nk; j++) { ra.old_mk[j] = d_mk[j].as<long long>(); ra.mk[j] = nmk[j].as<long long>(); }
        int n = 0;
        for (int j = 0; j < n_funcs; j++) {
            ra.old_acc[n] = d_a0[j].as<unsigned long long>(); ra.new_acc[n++] = na0[j].as<unsigned long long>();
            if (funcs[j].has_a1) { ra.old_acc[n] = d_a1[j].as<unsigned long long>(); ra.new_acc[n++] = na1[j].as<unsigned long long>(); }
        }
        ra.n_acc = n;
        rehash_mk_kernel<<<grid_for((int64_t)cap), 256, 0, stream>>>(ra);
        launches++;
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaStreamSynchronize(stream));
        d_tags = std::move(ntags); d_mkmask = std::move(nmask);
        for (int j = 0; j < nk; j++) d_mk[j] = std::move(nmk[j]);
        for (int j = 0; j < n_funcs; j++) { d_a0[j] = std::move(na0[j]); d_a1[j] = std::move(na1[j]); }
        cap = new_cap;
        rebuilds++;
    }
    void consume_mk(const std::vector<const void*>& data, const std::vector<const uint8_t*>& valid, int64_t n) {
        bool could_fail = (int64_t)(cap / 2) - n_groups_bound < n;
        if (could_fail) d_fail.ensure(device, (size_t)n * 4);
        auto launch = [&](const uint32_t* index_list, int64_t rows) {
            MkArgs a{};
            a.nk = nk; a.dropna = dropna ? 1 : 0; a.n_rows = rows; a.index_list = index_list;
            for (int j = 0; j < nk; j++) { a.key_data[j] = data[j]; a.key_valid[j] = valid[j]; a.key_ctype[j] = c_types[j]; a.mk[j] = d_mk[j].as<long long>(); }
            a.tags = d_tags.as<unsigned long long>(); a.mkmask = d_mkmask.as<unsigned char>(); a.cap = cap;
            a.counters = d_counters.as<long long>(); a.group_limit = (long long)(cap / 2); a.fail_list = d_fail.as<uint32_t>();
            a.n_ops = n_funcs;
            for (int j = 0; j < n_funcs; j++) {
                const FuncSpec& f = funcs[j];
                a.ops[j].kind = f.kind; a.ops[j].in_ctype = f.in_ctype;
                a.ops[j].in_data = f.in_col >= 0 ? data[f.in_col] : nullptr;
                a.ops[j].in_valid = f.in_col >= 0 ? valid[f.in_col] : nullptr;
                a.ops[j].a0 = d_a0[j].p; a.ops[j].a1 = f.has_a1 ? d_a1[j].p : nullptr;
            }
            groupby_consume_mk_kernel<<<grid_for(rows), 256, 0, stream>>>(a);
            launches++; consume_launches += index_list == nullptr;
            B200_CUDA(cudaGetLastError());
        };
        launch(nullptr, n);
        settle(n, could_fail, launch);
        if (!could_fail) n_groups_bound += n; else n_groups_bound = n_groups;
        rows_consumed += n;
    }

    // After a launch that may have failed rows: grow + replay until every row is in.
    template <typename Replay>
    void settle(int64_t chunk_rows, bool could_fail, Replay replay) {
        if (!could_fail) return;
        read_counters();
        while (h_counters[1] > 0) {
            int64_t nf = h_counters[1];
            fail_rows += nf;
            grow_to_hold(nf);
            // the fail list becomes the index list of the replay; it cannot fail again (room for nf new groups)
            DevBuf replay_list;
            replay_list.alloc((size_t)nf * 4);
            B200_CUDA(cudaMemcpyAsync(replay_list.p, d_fail.p, (size_t)nf * 4, cudaMemcpyDeviceToDevice, stream));
            B200_CUDA(cudaMemsetAsync((char*)d_counters.p + 8, 0, 8, stream));
            replay(replay_list.as<uint32_t>(), nf);
            read_counters();
        }
        (void)chunk_rows;
    }

    // ---- SM-partitioned fast path (SPG) ----
    static constexpr int64_t SPG_LAUNCH_ROWS = 1ll << 27;
    PooledBuf d_bucket;
    DevBuf d_bucket_cnt;
    int spg_owners = 0, spg_ns = 0;
    size_t spg_smem = 0;
    int spg_state = -1;  // -1 not probed, 0 unavailable/disabled, 1 ready
    int64_t spg_launches = 0, spg_retry_rows = 0, lc_launches = 0;
    int64_t expected_groups_hint = 0;

    // Calls f(std::bool_constant<HAS_SUM>, std::bool_constant<HAS_CNT>) for the accumulators of the int64 fast path: sum and
    // count, sum only or count only (sum_j / cnt_j < 0: not asked for).  These are the three instantiations of its kernels.
    template <typename F>
    static void with_sum_cnt(int sum_j, int cnt_j, F&& f) {
        if (sum_j >= 0 && cnt_j >= 0) f(std::true_type{}, std::true_type{});
        else if (sum_j >= 0) f(std::true_type{}, std::false_type{});
        else f(std::false_type{}, std::true_type{});
    }
    // ... and f for each of the three
    template <typename F>
    static void for_each_sum_cnt(F&& f) {
        f(std::true_type{}, std::true_type{});
        f(std::true_type{}, std::false_type{});
        f(std::false_type{}, std::true_type{});
    }

    bool spg_probe() {
        if (spg_state >= 0) return spg_state == 1;
        spg_state = 0;
        const char* env = getenv("B200_SPG");
        if (env && env[0] == '0') return false;
        int max_smem = 0;
        cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
        if (sms > SPG_MAX_OWNERS - 1 || max_smem < 64 * 1024) return false;
        spg_ns = ((int)(((size_t)max_smem - 64) / 16) - SPG_STASH) & ~1;
        spg_smem = (size_t)(spg_ns + SPG_STASH) * 16 + 16;
        // opt a kernel in to `bytes` of dynamic shared memory; false (error cleared) when the device refuses
        auto smem_ok = [](const void* f, size_t bytes) {
            if (cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess) return true;
            cudaGetLastError();
            return false;
        };
        bool ok = true;
        for_each_sum_cnt([&](auto S, auto C) {
            constexpr bool HS = decltype(S)::value, HC = decltype(C)::value;
            ok = ok && smem_ok((const void*)spg_aggregate_kernel<HS, HC>, spg_smem) &&
                 smem_ok((const void*)spg_partition_tma_kernel<HS, HC>, spg_tma_smem()) &&
                 smem_ok((const void*)spg_partition_tma_kernel<HS, HC, true>, spg_tma_smem(true));
        });
        if (!ok) return false;
        {   // SPG-N (spgn.cuh): narrow bucket rows
            spgn_ns = ((int)(((size_t)max_smem - 256) / 12) - SPG_STASH) & ~1;  // (K2n also has a few static shared words)
            spgn_smem = (size_t)(spgn_ns + SPG_STASH) * 12 + 16;
            spgn_enabled = true;
            for_each_sum_cnt([&](auto S, auto C) {
                constexpr bool HS = decltype(S)::value, HC = decltype(C)::value;
                if (!smem_ok((const void*)spgn_partition_kernel<HS, HC>, spgn_part_smem())) spgn_enabled = false;
                if (!smem_ok((const void*)spgn_aggregate_kernel<HS, HC>, spgn_smem)) spgn_enabled = false;
            });
            const char* e8 = getenv("B200_SPG_NARROW");
            if (e8 && e8[0] == '0') spgn_enabled = false;
        }
        {   // SPG-G (spgg.cuh): generic signatures
            spgg_enabled = 2 * sms <= GEN_CLS;  // classes of K1g's counting sort: at least owners + owners
            const void* gp[6] = {(const void*)spgg_partition_kernel<8, 8>, (const void*)spgg_partition_kernel<8, 4>, (const void*)spgg_partition_kernel<8, 0>,
                                 (const void*)spgg_partition_kernel<4, 8>, (const void*)spgg_partition_kernel<4, 4>, (const void*)spgg_partition_kernel<4, 0>};
            for (auto f : gp)
                if (!smem_ok(f, GEN_K1_SMEM)) spgg_enabled = false;
            for (int v = 0; v < 4; v++) {  // v = mm + 2 * nn
                const int sb = 16 + ((v & 1) ? 16 : 0) + ((v & 2) ? 4 : 0);
                spgg_ns[v] = ((int)(((size_t)max_smem - 64) / sb) - SPG_STASH) & ~1;
                spgg_smem[v] = (size_t)(spgg_ns[v] + SPG_STASH) * sb + 16;
            }
            const void* ga[8] = {(const void*)spgg_aggregate_kernel<false, false, false>, (const void*)spgg_aggregate_kernel<true, false, false>,
                                 (const void*)spgg_aggregate_kernel<false, true, false>, (const void*)spgg_aggregate_kernel<true, true, false>,
                                 (const void*)spgg_aggregate_kernel<false, false, true>, (const void*)spgg_aggregate_kernel<true, false, true>,
                                 (const void*)spgg_aggregate_kernel<false, true, true>, (const void*)spgg_aggregate_kernel<true, true, true>};
            for (int q = 0; q < 8; q++)  // q = sum + 2 * mm + 4 * nn
                if (!smem_ok(ga[q], spgg_smem[q >> 1])) spgg_enabled = false;
            const char* e7 = getenv("B200_SPG_GEN");
            if (e7 && e7[0] == '0') spgg_enabled = false;
        }
        if (!smem_ok((const void*)spg_hot_sample_kernel, SPG_HOT_SAMPLE_SMEM)) return false;
        { const char* e4 = getenv("B200_SPG_HOT"); spg_hot_enabled = !(e4 && e4[0] == '0'); }
        d_hot.alloc((size_t)SPG_HOT_SLOTS * 8 + 16);
        for_each_sum_cnt([&](auto S, auto C) {
            ok = ok && smem_ok((const void*)groupby_lowcard_kernel<decltype(S)::value, decltype(C)::value, LC_SLOTS_BIG, 2>, (size_t)LC_SLOTS_BIG * 20 + 64);
        });
        if (!ok) return false;
        { const char* e3 = getenv("B200_LC"); lc_enabled = !(e3 && e3[0] == '0'); }
        spg_owners = sms;  // one owner (bucket + shared table) per SM
        d_bucket_cnt.alloc((size_t)std::max(2 * spg_owners, GEN_CLS) * SPG_CNT_STRIDE * 8);  // SPG-G: one counter per class of K1g
        spg_state = 1;
        return true;
    }

    bool lc_enabled = true, lowcard_small = false;
    // SPG-N: narrow bucket rows (spgn.cuh)
    int spgn_ns = 0;
    size_t spgn_smem = 0;
    bool spgn_enabled = false;
    int spg_sample_wide = -1;  // sampled rows of the first launch that do NOT fit (int32 key, int32 value); -1 = not sampled
    int64_t spgn_launches = 0;
    static size_t spgn_part_smem() { return (size_t)SPGN_TILE * (16 + 8 + 1) + SPG_MAX_OWNERS * 16 + 16 + (2 * SPG_MAX_OWNERS + 4) * 4 + 256; }
    int64_t spgn_group_capacity() const { return (int64_t)spg_owners * (spgn_ns * 7 / 10); }
    int spgg_ns[4] = {0, 0, 0, 0};  // K2g table slots, by slot layout v = (min/max fields) + 2 * (NA-value counter)
    size_t spgg_smem[4] = {0, 0, 0, 0};
    bool spgg_enabled = true;      // B200_SPG_GEN=0 disables the generic SM-partitioned path
    int64_t spgg_launches = 0;
    int spg_n_hot = 0;
    bool spg_hot_enabled = true, spg_hot_sampled = false;  // heavy-hitter table: sampled once per state, at its first SPG launch
    DevBuf d_hot;                                           // [SPG_HOT_SLOTS] keys + n_hot (int)
    int spg_passes = 1;
    static constexpr int SPG_MAX_PASSES = 24;
    // K2 passes needed for `est` groups (each pass holds spg_group_capacity() groups); 0 = too many for the SPG path
    int spg_pass_count(int64_t est) const {
        int64_t p = (est + spg_group_capacity() - 1) / spg_group_capacity();
        return p <= 1 ? 1 : (p <= SPG_MAX_PASSES ? (int)p : 0);
    }
    static size_t spg_tma_smem(bool hot = false) { return (size_t)SPG_TILE * (16 + 16 + 1) + SPG_MAX_OWNERS * 8 + 16 + (2 * SPG_MAX_OWNERS + 4) * 4 + (hot ? SPG_HOT_SLOTS * 20 : 0) + 256; }
    bool lc_pick(int64_t est) { lowcard_small = est <= LC_SLOTS_SMALL / 4; return lc_enabled && est <= LC_SLOTS_BIG / 4; }
    // groups the shared-memory tables of all owners are expected to hold together (two-choice buckets work well up to ~70 %)
    int64_t spg_group_capacity() const { return (int64_t)spg_owners * (spg_ns * 7 / 10); }

    // One SPG launch pair in flight while the host inspects the previous one (two retry lists / counter slots), so
    // the GPU never idles on the host's counter read-back.
    PooledBuf d_retry2[2];
    long long* h_spg = nullptr;  // pinned: [slot][8] counter snapshots
    cudaEvent_t spg_ev[2] = {nullptr, nullptr};

    int64_t spgn_wide_rows = 0;  // rows that did not fit the narrow format so far (device counter 5)
    void spg_finish(int slot, int sum_j, int cnt_j) {
        B200_CUDA(cudaEventSynchronize(spg_ev[slot]));
        const long long* hc = h_spg + slot * 8;
        n_groups = hc[0];
        spgn_wide_rows = hc[5];
        int64_t nr = hc[1 + 5 * slot];  // retry rows of that launch: counters[1] (slot 0) / counters[6] (slot 1)
        while (nr > 0) {
            // rows / partials that found the global table full: grow, then merge them like received partial rows
            spg_retry_rows += nr;
            B200_CUDA(cudaStreamSynchronize(stream));  // the other in-flight launch uses the table we are about to replace
            read_counters();
            int64_t pending = h_counters[1] + h_counters[6];
            // the snapshot this call was made on may be stale: the other slot's spg_finish already grew the table and merged
            // BOTH retry lists (their live counters are 0 then) — nothing left to do, and no second grow
            if (pending == 0) break;
            grow_to_hold(pending + (int64_t)spg_owners * spg_ns);
            for (int sl = 0; sl < 2; sl++) {
                int64_t cnt = h_counters[1 + 5 * sl];
                if (cnt == 0) continue;
                B200_CUDA(cudaMemsetAsync((char*)d_counters.p + 8 * (1 + 5 * sl), 0, 8, stream));
                CombineArgs c{};
                c.in = d_retry2[sl].as<unsigned long long>(); c.n_rows = cnt; c.row_words = 4;
                d_fail.ensure(device, (size_t)cnt * 4);
                c.tkeys = d_keys.as<long long>(); c.cap = cap; c.counters = d_counters.as<long long>(); c.group_limit = (long long)(cap / 2);
                c.fail_list = d_fail.as<uint32_t>(); c.index_list = nullptr; c.n_ops = 0;  // cannot fail: the table was grown for all pending rows
                // wire order = function order of the (at most two) accumulators
                int order[2] = {sum_j, cnt_j};
                if (sum_j >= 0 && cnt_j >= 0 && cnt_j < sum_j) std::swap(order[0], order[1]);
                if (order[0] < 0) std::swap(order[0], order[1]);
                for (int q = 0; q < 2; q++) if (order[q] >= 0) { c.kinds[c.n_ops] = K_SUM_I64; c.a0[c.n_ops] = d_a0[order[q]].p; c.a1[c.n_ops] = nullptr; c.n_ops++; }
                combine_partials_kernel<<<grid_for(cnt), 256, 0, stream>>>(c);
                launches++;
                B200_CUDA(cudaGetLastError());
            }
            read_counters();
            nr = 0;
        }
    }

    void consume_spg(const long long* keys, const long long* vals, int64_t n, int sum_j, int cnt_j, bool lowcard = false, int64_t est_groups = 0) {
        if (!h_spg) {
            h_spg = (long long*)pinned_acquire(24 * sizeof(long long));  // [slot][8] counter snapshots + n_hot read-back
            for (int b = 0; b < 2; b++) B200_CUDA(cudaEventCreateWithFlags(&spg_ev[b], cudaEventDisableTiming));
        }
        double tspg0 = now();
        struct Acc2 { double& t; double t0; ~Acc2() { t += now() - t0; } } acc2{t_spg, tspg0};
        B200_REQUIRE(((uintptr_t)keys & 15) == 0 && ((uintptr_t)vals & 15) == 0,
                     "internal: the SM-partitioned groupby takes 16-byte aligned columns (K1 fetches tiles with TMA bulk copies)");
        read_counters();  // exact group count before the first launch
        n_groups_bound = n_groups;
        if (!lowcard && !spg_hot_sampled) {
            // once per state: count a sample of this call's keys (heavy hitters) and test the sampled rows against the narrow-row
            // format; the host reads back both verdicts
            int* d_nhot = (int*)(d_hot.as<long long>() + SPG_HOT_SLOTS);
            spg_hot_sample_kernel<<<1, 1024, SPG_HOT_SAMPLE_SMEM, stream>>>(keys, vals, n, d_hot.as<long long>(), d_nhot);
            B200_CUDA(cudaMemcpyAsync(h_spg + 16, d_nhot, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream));
            B200_CUDA(cudaStreamSynchronize(stream));
            spg_n_hot = spg_hot_enabled ? ((int*)(h_spg + 16))[0] : 0;
            spg_sample_wide = ((int*)(h_spg + 16))[1];
            spg_hot_sampled = true;
            launches++;
        }
        // narrow bucket rows are half the bytes: twice the rows per launch for the same scratch, half the per-launch flushes
        const bool narrow_call = spgn_enabled && !lowcard && spg_n_hot == 0 && spg_sample_wide == 0;
        const int64_t launch_rows = narrow_call ? 2 * SPG_LAUNCH_ROWS : SPG_LAUNCH_ROWS;
        int64_t li = 0;
        for (int64_t r0 = 0; r0 < n; r0 += launch_rows, li++) {
            int slot = (int)(li & 1);
            int64_t rows = std::min(launch_rows, n - r0);
            // no pre-growing: a flush that finds the global table at its limit lands in the retry list and is merged
            // after the table grew (spg_finish), exactly like rows of the direct path
            // uniform keys put rows / owners rows in every bucket (sd = sqrt of that); 12.5 % + 4096 rows head room,
            // anything beyond (skew) takes the direct path inside K1
            const int64_t bucket_cap = (rows / spg_owners) + (rows / spg_owners) / 8 + 4096;
            double ta = now();
            d_bucket.ensure(device, (size_t)spg_owners * bucket_cap * 16);  // K2 of the previous launch precedes K1 of this one in stream order
            d_retry2[slot].ensure(device, ((size_t)rows + (size_t)spg_owners * spg_ns) * 32);
            t_alloc += now() - ta;
            B200_CUDA(cudaMemsetAsync(d_bucket_cnt.p, 0, (size_t)spg_owners * SPG_CNT_STRIDE * 8, stream));
            SpgArgs a{};
            a.keys = keys + r0; a.vals = vals ? vals + r0 : nullptr; a.n_rows = rows; a.n_owners = spg_owners;
            a.tkeys = d_keys.as<long long>(); a.cap = cap;
            a.acc_sum = sum_j >= 0 ? d_a0[sum_j].as<unsigned long long>() : nullptr;
            a.acc_cnt = cnt_j >= 0 ? d_a0[cnt_j].as<unsigned long long>() : nullptr;
            a.counters = d_counters.as<long long>(); a.group_limit = (long long)(cap / 2);
            a.retry_ctr = d_counters.as<long long>() + 1 + 5 * slot;
            a.bucket = d_bucket.as<longlong2>(); a.bucket_cnt = d_bucket_cnt.as<unsigned long long>(); a.bucket_cap = bucket_cap;
            a.retry = d_retry2[slot].as<unsigned long long>();
            a.sum_first = (sum_j >= 0 && cnt_j >= 0 && sum_j < cnt_j) ? 1 : 0; a.ns = spg_ns; a.n_pass = spg_passes;
            cudaEvent_t ev0 = nullptr, ev1 = nullptr;
            if (profiling) { B200_CUDA(cudaEventCreate(&ev0)); B200_CUDA(cudaEventCreate(&ev1)); B200_CUDA(cudaEventRecord(ev0, stream)); }
            if (lowcard) {
                const bool small = lowcard_small;
                int gl = (int)std::min<int64_t>((int64_t)sms * (small ? 3 : 2), (rows + LC_THREADS * 2 - 1) / (LC_THREADS * 2));
                size_t lsm = (size_t)(small ? LC_SLOTS_SMALL : LC_SLOTS_BIG) * 20 + 64;
                with_sum_cnt(sum_j, cnt_j, [&](auto S, auto C) {
                    constexpr bool HS = decltype(S)::value, HC = decltype(C)::value;
                    if (small) groupby_lowcard_kernel<HS, HC, LC_SLOTS_SMALL, 3><<<gl, LC_THREADS, lsm, stream>>>(a);
                    else groupby_lowcard_kernel<HS, HC, LC_SLOTS_BIG, 2><<<gl, LC_THREADS, lsm, stream>>>(a);
                });
                lc_launches++;
            } else {
                int g1 = (int)std::min<int64_t>((int64_t)sms * SPG_TCTAS, (rows + SPG_TILE - 1) / SPG_TILE);
                const bool hot = spg_hot_enabled && spg_n_hot > 0;
                if (hot) { a.hot_tab = d_hot.as<long long>(); a.n_hot = (const int*)(d_hot.as<long long>() + SPG_HOT_SLOTS); }
                const size_t tsm = spg_tma_smem(hot);
                // SPG-N: the sample found only rows that fit (int32 key, int32 value), and the rows that did not so far are rare
                const bool narrow = spgn_enabled && !hot && spg_sample_wide == 0 && spgn_wide_rows * 64 <= rows_consumed;
                if (narrow) {
                    a.ns = spgn_ns;
                    // first flush into an empty table: per-CTA ticket reservation, but only with >= 25 % head room under the group
                    // limit — a reservation transiently over-counts (slots that hold one key twice), and a CTA that then finds the
                    // limit reached would send its groups to the retry list and make the host grow the table for nothing (seen on
                    // 8 GPUs: 1 M groups against a limit of 2^20 cost 1.4 ms per state in some runs)
                    a.reserve_tickets = (n_groups_bound == 0 && li == 0 && est_groups > 0 && est_groups + est_groups / 4 <= (int64_t)(cap / 2)) ? 1 : 0;
                    const int64_t est_n = std::max<int64_t>(est_groups, 1);
                    a.n_pass = (int)std::min<int64_t>(SPG_MAX_PASSES, std::max<int64_t>(1, (est_n + spgn_group_capacity() - 1) / spgn_group_capacity()));
                    a.bucket_cap = bucket_cap & ~1ll;
                    const size_t nsm = spgn_part_smem();
                    const int gn = (int)std::min<int64_t>((int64_t)sms * SPGN_CTAS, (rows + SPGN_TILE - 1) / SPGN_TILE);
                    with_sum_cnt(sum_j, cnt_j, [&](auto S, auto C) {
                        constexpr bool HS = decltype(S)::value, HC = decltype(C)::value;
                        spgn_partition_kernel<HS, HC><<<gn, SPG_TTHREADS, nsm, stream>>>(a);
                        spgn_aggregate_kernel<HS, HC><<<spg_owners, SPG_THREADS, spgn_smem, stream>>>(a);
                    });
                    spgn_launches++;
                } else {
                    with_sum_cnt(sum_j, cnt_j, [&](auto S, auto C) {
                        constexpr bool HS = decltype(S)::value, HC = decltype(C)::value;
                        if (hot) spg_partition_tma_kernel<HS, HC, true><<<g1, SPG_TTHREADS, tsm, stream>>>(a);
                        else spg_partition_tma_kernel<HS, HC><<<g1, SPG_TTHREADS, tsm, stream>>>(a);
                        spg_aggregate_kernel<HS, HC><<<spg_owners, SPG_THREADS, spg_smem, stream>>>(a);
                    });
                }
            }
            B200_CUDA(cudaGetLastError());
            if (ev0) { B200_CUDA(cudaEventRecord(ev1, stream)); prof_events.emplace_back(ev0, ev1); }
            B200_CUDA(cudaMemcpyAsync(h_spg + slot * 8, d_counters.p, 8 * sizeof(long long), cudaMemcpyDeviceToHost, stream));
            B200_CUDA(cudaEventRecord(spg_ev[slot], stream));
            launches += 2; consume_launches++; spg_launches++;
            rows_consumed += rows;
            if (li > 0) spg_finish(1 - slot, sum_j, cnt_j);  // inspect the previous launch while this one runs
        }
        if (li > 0) spg_finish((int)((li - 1) & 1), sum_j, cnt_j);
        read_counters();
        n_groups_bound = n_groups;
    }

    // ---- SPG-G: the SM-partitioned path for generic signatures (spgg.cuh) ----
    struct GenSig { int vcol = -1; bool has_sum = false, has_mm = false, has_nn = false; int layout = 0; };
    static bool gen_int_ok(int ct) { const int sz = ctype_size(ct); return (sz == 4 || sz == 8) && !ctype_is_float(ct) && ct != CT_UINT64; }
    bool gen_signature(const std::vector<const void*>& data, const std::vector<const uint8_t*>& valid, GenSig& gs) const {
        if (nk != 1 || n_funcs < 1 || n_funcs > GEN_MAX_F || !gen_int_ok(c_types[0])) return false;
        bool has_size = false;
        for (auto& f : funcs) {
            switch (f.kind) {
                case K_SIZE: has_size = true; continue;
                case K_COUNT: break;
                case K_SUM_I64: case K_MEAN: gs.has_sum = true; break;
                case K_MIN_I64: case K_MAX_I64: gs.has_mm = true; break;
                default: return false;
            }
            if (!gen_int_ok(f.in_ctype)) return false;
            if (gs.vcol >= 0 && gs.vcol != f.in_col) return false;
            gs.vcol = f.in_col;
        }
        // tiles (columns and validity bitmaps) are fetched with TMA bulk copies: 16-byte aligned sources
        if (((uintptr_t)data[0] & 15) || ((uintptr_t)valid[0] & 15)) return false;
        if (gs.vcol >= 0 && (((uintptr_t)data[gs.vcol] & 15) || ((uintptr_t)valid[gs.vcol] & 15))) return false;
        gs.has_nn = gs.vcol >= 0 && valid[gs.vcol] != nullptr && has_size;
        gs.layout = (gs.has_mm ? 1 : 0) + (gs.has_nn ? 2 : 0);
        return true;
    }
    int64_t spgg_group_capacity(int layout) const { return (int64_t)spg_owners * (spgg_ns[layout] * 7 / 10); }
    int spgg_pass_count(int64_t est, int layout) const {
        int64_t p = (est + spgg_group_capacity(layout) - 1) / spgg_group_capacity(layout);
        return p <= 1 ? 1 : (p <= SPG_MAX_PASSES ? (int)p : 0);
    }
    static constexpr int64_t GEN_LAUNCH_ROWS = 1ll << 27;
    PooledBuf d_nbucket;  // key-only buckets of the rows whose value is NA

    void consume_spg_gen(const std::vector<const void*>& data, const std::vector<const uint8_t*>& valid, int64_t n, const GenSig& gs, int passes) {
        double tspg0 = now();
        struct Acc2 { double& t; double t0; ~Acc2() { t += now() - t0; } } acc2{t_spg, tspg0};
        const int kct = c_types[0], vct = gs.vcol >= 0 ? c_types[gs.vcol] : CT_INT64;
        const int ks = ctype_size(kct), vs = gs.vcol >= 0 ? ctype_size(vct) : 0;
        const int mm = gs.layout;
        const bool v_nullable = gs.vcol >= 0 && valid[gs.vcol] != nullptr;
        // multi-pass: K1g partitions straight into owners x passes buckets when its class table has room for them
        const int n_vo = (passes > 1 && spg_owners * passes + (v_nullable ? spg_owners : 0) <= GEN_CLS) ? spg_owners * passes : spg_owners;
        for (int64_t r0 = 0; r0 < n; r0 += GEN_LAUNCH_ROWS) {
            const int64_t rows = std::min(GEN_LAUNCH_ROWS, n - r0);
            // a bucket holds rows / owners rows (NA-value buckets: at most that) however many buckets the valued rows spread over
            const int64_t bucket_cap = (rows / spg_owners) + (rows / spg_owners) / 8 + 4096;
            double ta = now();
            d_bucket.ensure(device, (size_t)n_vo * bucket_cap * 16);
            if (v_nullable) d_nbucket.ensure(device, (size_t)spg_owners * bucket_cap * 8);
            d_retry2[0].ensure(device, ((size_t)rows + (size_t)spg_owners * (spgg_ns[mm] + SPG_STASH) * passes) * GEN_RETRY_WORDS * 8);
            t_alloc += now() - ta;
            B200_CUDA(cudaMemsetAsync(d_bucket_cnt.p, 0, (size_t)(n_vo + spg_owners) * SPG_CNT_STRIDE * 8, stream));
            auto make_args = [&]() {
                SpgGenArgs g{};
                g.s.n_rows = rows; g.s.n_owners = spg_owners;
                g.s.tkeys = d_keys.as<long long>(); g.s.cap = cap; g.s.counters = d_counters.as<long long>(); g.s.group_limit = (long long)(cap / 2);
                g.s.retry_ctr = d_counters.as<long long>() + 1; g.s.retry = d_retry2[0].as<unsigned long long>();
                g.s.bucket = d_bucket.as<longlong2>(); g.s.bucket_cnt = d_bucket_cnt.as<unsigned long long>(); g.s.bucket_cap = bucket_cap;
                g.s.ns = spgg_ns[mm]; g.s.n_pass = passes;
                g.nbucket = v_nullable ? d_nbucket.as<long long>() : nullptr; g.n_vo = n_vo;
                g.kdata = (const char*)data[0] + r0 * ks; g.kvalid = valid[0] ? valid[0] + r0 / 8 : nullptr;
                g.vdata = gs.vcol >= 0 ? (const char*)data[gs.vcol] + r0 * vs : nullptr;
                g.vvalid = (gs.vcol >= 0 && valid[gs.vcol]) ? valid[gs.vcol] + r0 / 8 : nullptr;
                g.k_signed = ctype_is_signed_int(kct) ? 1 : 0; g.v_signed = ctype_is_signed_int(vct) ? 1 : 0;
                g.dropna = dropna ? 1 : 0;
                g.fl.n = n_funcs;
                for (int j = 0; j < n_funcs; j++) {
                    g.fl.kind[j] = funcs[j].kind; g.fl.a0[j] = d_a0[j].as<unsigned long long>();
                    g.fl.a1[j] = funcs[j].has_a1 ? d_a1[j].as<unsigned long long>() : nullptr;
                }
                return g;
            };
            SpgGenArgs g = make_args();
            cudaEvent_t ev0 = nullptr, ev1 = nullptr;
            if (profiling) { B200_CUDA(cudaEventCreate(&ev0)); B200_CUDA(cudaEventCreate(&ev1)); B200_CUDA(cudaEventRecord(ev0, stream)); }
            const int g1 = (int)std::min<int64_t>((int64_t)sms * SPG_TCTAS, (rows + SPG_TILE - 1) / SPG_TILE);
            const size_t psm = GEN_K1_SMEM;
            if (ks == 8 && vs == 8) spgg_partition_kernel<8, 8><<<g1, SPG_TTHREADS, psm, stream>>>(g);
            else if (ks == 8 && vs == 4) spgg_partition_kernel<8, 4><<<g1, SPG_TTHREADS, psm, stream>>>(g);
            else if (ks == 8) spgg_partition_kernel<8, 0><<<g1, SPG_TTHREADS, psm, stream>>>(g);
            else if (vs == 8) spgg_partition_kernel<4, 8><<<g1, SPG_TTHREADS, psm, stream>>>(g);
            else if (vs == 4) spgg_partition_kernel<4, 4><<<g1, SPG_TTHREADS, psm, stream>>>(g);
            else spgg_partition_kernel<4, 0><<<g1, SPG_TTHREADS, psm, stream>>>(g);
#define B200_SPGG_K2(S, M, N) spgg_aggregate_kernel<S, M, N><<<spg_owners, SPG_THREADS, spgg_smem[mm], stream>>>(g)
            switch ((gs.has_sum ? 1 : 0) + (gs.has_mm ? 2 : 0) + (gs.has_nn ? 4 : 0)) {
                case 0: B200_SPGG_K2(false, false, false); break;
                case 1: B200_SPGG_K2(true, false, false); break;
                case 2: B200_SPGG_K2(false, true, false); break;
                case 3: B200_SPGG_K2(true, true, false); break;
                case 4: B200_SPGG_K2(false, false, true); break;
                case 5: B200_SPGG_K2(true, false, true); break;
                case 6: B200_SPGG_K2(false, true, true); break;
                default: B200_SPGG_K2(true, true, true); break;
            }
#undef B200_SPGG_K2
            B200_CUDA(cudaGetLastError());
            if (ev0) { B200_CUDA(cudaEventRecord(ev1, stream)); prof_events.emplace_back(ev0, ev1); }
            launches += 2; consume_launches++; spg_launches++; spgg_launches++;
            rows_consumed += rows;
            read_counters();
            while (h_counters[1] > 0) {  // partials that found the global table at its limit: grow, replay them
                const int64_t nr = h_counters[1];
                spg_retry_rows += nr;
                grow_to_hold(nr);
                d_retry2[1].ensure(device, (size_t)nr * GEN_RETRY_WORDS * 8);
                B200_CUDA(cudaMemcpyAsync(d_retry2[1].p, d_retry2[0].p, (size_t)nr * GEN_RETRY_WORDS * 8, cudaMemcpyDeviceToDevice, stream));
                B200_CUDA(cudaMemsetAsync((char*)d_counters.p + 8, 0, 8, stream));
                SpgGenArgs g2 = make_args();
                spgg_replay_kernel<<<grid_for(nr), 256, 0, stream>>>(g2, d_retry2[1].as<unsigned long long>(), (long long)nr);
                launches++;
                B200_CUDA(cudaGetLastError());
                read_counters();
            }
        }
        n_groups_bound = n_groups;
    }

    // Consume rows [0, n) of device-resident columns.
    void consume_device_chunk(const std::vector<const void*>& data, const std::vector<const uint8_t*>& valid, int64_t n) {
        if (n == 0) return;
        if (nk > 1) { consume_mk(data, valid, n); return; }
        // fast path: non-null int64 key + {sum, count/size} over one non-null int64 value column
        bool fast = c_types[0] == CT_INT64 && valid[0] == nullptr && n_funcs >= 1;
        int sum_j = -1, cnt_j = -1, vcol = -1;
        for (int j = 0; j < n_funcs && fast; j++) {
            const FuncSpec& f = funcs[j];
            if (f.kind == K_SUM_I64 && f.in_ctype == CT_INT64 && valid[f.in_col] == nullptr && sum_j < 0) {
                sum_j = j; vcol = f.in_col;
            } else if ((f.kind == K_SIZE || (f.kind == K_COUNT && !ctype_is_float(f.in_ctype) && valid[f.in_col] == nullptr)) && cnt_j < 0) {
                cnt_j = j;
            } else {
                fast = false;
            }
        }
        if (fast && (((uintptr_t)data[0] & 15) || (vcol >= 0 && ((uintptr_t)data[vcol] & 15)))) fast = false;
        // SM-partitioned path: big batches whose (estimated) cardinality fits the chip's shared memory
        if (fast && n >= (1 << 20) && spg_probe()) {
            const char* env = getenv("B200_SPG");
            bool force = env && env[0] == '1';
            int64_t est = std::max(expected_groups_hint, n_groups);
            if (!force && est == 0 && rows_consumed == 0) {
                // cardinality unknown: learn it from a prefix through the direct kernel
                int64_t prefix = std::min<int64_t>(n, 1 << 20);
                std::vector<const void*> d2(data); std::vector<const uint8_t*> v2(valid);
                consume_direct(d2, v2, prefix, fast, sum_j, cnt_j, vcol, /*force_count=*/true);
                est = n_groups;
                if (prefix == n) return;
                for (int c = 0; c < n_cols; c++) if (data[c]) d2[c] = (const char*)data[c] + prefix * ctype_size(c_types[c]);
                if (spg_pass_count(est) > 0) { spg_passes = spg_pass_count(est); consume_spg((const long long*)d2[0], vcol >= 0 ? (const long long*)d2[vcol] : nullptr, n - prefix, sum_j, cnt_j, lc_pick(est), est); }
                else consume_direct(d2, v2, n - prefix, fast, sum_j, cnt_j, vcol, false);
                return;
            }
            if (force || spg_pass_count(est) > 0) {
                spg_passes = std::max(1, spg_pass_count(est));
                consume_spg((const long long*)data[0], vcol >= 0 ? (const long long*)data[vcol] : nullptr, n, sum_j, cnt_j, est > 0 && lc_pick(est), est);
                return;
            }
        }
        // generic signatures (nullable / 4-byte keys or values / mean / min / max over one integer column): same two-kernel path
        if (!fast && n >= (1 << 20) && spg_probe() && spgg_enabled) {
            GenSig gs;
            if (gen_signature(data, valid, gs)) {
                int64_t est = std::max(expected_groups_hint, n_groups);
                std::vector<const void*> d2(data); std::vector<const uint8_t*> v2(valid);
                int64_t left = n;
                if (est == 0 && rows_consumed == 0) {  // cardinality unknown: learn it from a prefix through the direct kernel
                    const int64_t prefix = std::min<int64_t>(n, 1 << 20);
                    consume_direct(data, valid, prefix, false, -1, -1, -1, /*force_count=*/true);
                    est = n_groups;
                    if (prefix == n) return;
                    for (int c = 0; c < n_cols; c++) {
                        if (data[c]) d2[c] = (const char*)data[c] + prefix * ctype_size(c_types[c]);
                        if (valid[c]) v2[c] = valid[c] + prefix / 8;
                    }
                    left = n - prefix;
                }
                // below ~1000 groups the owners are unevenly loaded (and there is no low-cardinality generic kernel): direct path
                if (est > LC_SLOTS_BIG / 4 && spgg_pass_count(est, gs.layout) > 0 && left >= (1 << 16)) {
                    consume_spg_gen(d2, v2, left, gs, spgg_pass_count(est, gs.layout));
                    return;
                }
                consume_direct(d2, v2, left, false, -1, -1, -1, false);
                return;
            }
        }
        consume_direct(data, valid, n, fast, sum_j, cnt_j, vcol, false);
    }

    void consume_direct(const std::vector<const void*>& data, const std::vector<const uint8_t*>& valid, int64_t n, bool fast, int sum_j,
                        int cnt_j, int vcol, bool force_count) {
        bool could_fail = force_count || (int64_t)(cap / 2) - n_groups_bound < n;
        if (could_fail) d_fail.ensure(device, (size_t)n * 4);
        // table pointers are looked up at launch time: grow() replaces them between a launch and its replay
        auto launch = [&](const uint32_t* index_list, int64_t rows) {
            long long* ctr = d_counters.as<long long>();
            long long limit = (long long)(cap / 2);
            cudaEvent_t ev0 = nullptr, ev1 = nullptr;
            if (profiling && index_list == nullptr) {
                B200_CUDA(cudaEventCreate(&ev0)); B200_CUDA(cudaEventCreate(&ev1));
                B200_CUDA(cudaEventRecord(ev0, stream));
            }
            if (fast && index_list == nullptr) {
                int g = grid_for(rows, 2);
                const long long* k = (const long long*)data[0];
                const long long* v = vcol >= 0 ? (const long long*)data[vcol] : nullptr;
                unsigned long long* as = sum_j >= 0 ? d_a0[sum_j].as<unsigned long long>() : nullptr;
                unsigned long long* ac = cnt_j >= 0 ? d_a0[cnt_j].as<unsigned long long>() : nullptr;
                with_sum_cnt(sum_j, cnt_j, [&](auto S, auto C) {
                    groupby_consume_i64_sumcount_kernel<decltype(S)::value, decltype(C)::value>
                        <<<g, 256, 0, stream>>>(k, v, rows, d_keys.as<long long>(), cap, as, ac, ctr, limit, d_fail.as<uint32_t>());
                });
            } else {
                ConsumeArgs a = generic_args(data, valid, index_list, rows);
                groupby_consume_kernel<<<grid_for(rows), 256, 0, stream>>>(a);
            }
            launches++;
            if (index_list == nullptr) consume_launches++;
            if (ev0) { B200_CUDA(cudaEventRecord(ev1, stream)); prof_events.emplace_back(ev0, ev1); }
            B200_CUDA(cudaGetLastError());
        };
        launch(nullptr, n);
        settle(n, could_fail, launch);
        if (has_firstlast) {  // every row is in (replays included): the rows that won first / last write their values
            groupby_firstlast_fix_kernel<<<grid_for(n), 256, 0, stream>>>(generic_args(data, valid, nullptr, n));
            launches++;
            B200_CUDA(cudaGetLastError());
        }
        if (!could_fail) n_groups_bound += n;  // upper bound without a device round trip
        else n_groups_bound = n_groups;
        rows_consumed += n;
    }
    ConsumeArgs generic_args(const std::vector<const void*>& data, const std::vector<const uint8_t*>& valid, const uint32_t* index_list, int64_t rows) {
        ConsumeArgs a{};
        a.key_data = data[0]; a.key_valid = valid[0]; a.key_ctype = c_types[0]; a.dropna = dropna ? 1 : 0;
        a.n_rows = rows; a.index_list = index_list; a.tkeys = d_keys.as<long long>(); a.cap = cap;
        a.counters = d_counters.as<long long>(); a.group_limit = (long long)(cap / 2); a.fail_list = d_fail.as<uint32_t>(); a.n_ops = n_funcs;
        // rank-major sequence numbers: rows of a lower rank come first (the reference's row-block distribution), then row order
        a.seq_base = ((unsigned long long)rank << 44) + (unsigned long long)rows_consumed;
        for (int j = 0; j < n_funcs; j++) {
            const FuncSpec& f = funcs[j];
            a.ops[j].kind = f.kind; a.ops[j].in_ctype = f.in_ctype;
            a.ops[j].in_data = f.in_col >= 0 ? data[f.in_col] : nullptr;
            a.ops[j].in_valid = f.in_col >= 0 ? valid[f.in_col] : nullptr;
            a.ops[j].a0 = d_a0[j].p; a.ops[j].a1 = f.has_a1 ? d_a1[j].p : nullptr;
        }
        return a;
    }

    int64_t n_groups_bound = 0;  // upper bound on groups in the table known to the host
    int64_t untracked_groups = 0;  // upper bound of groups inserted without ticket counting (combine with guaranteed room)
    bool stage_recorded[2] = {false, false};

    void consume(const b200_table* t) {
        B200_REQUIRE(!build_done, "b200 groupby: consume after the build was finished");
        B200_REQUIRE(t->n_cols == n_cols, "b200 groupby: batch has a different number of columns than the build schema");
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        int64_t n = t->n_rows;
        std::vector<bool> used(n_cols, false);
        for (int kc = 0; kc < nk; kc++) used[kc] = true;
        for (auto& f : funcs) if (f.in_col >= 0) used[f.in_col] = true;
        for (int c = 0; c < n_cols; c++) {
            if (!used[c]) continue;
            B200_REQUIRE(t->cols[c].c_type == c_types[c], "b200 groupby: batch column dtype differs from the build schema");
            B200_REQUIRE(n == 0 || t->cols[c].data != nullptr, "b200 groupby: null data pointer");
        }
        for (auto& ni : nu_inner) {  // nunique: the (key, value) pairs of this batch go to the nested distinct state
            b200_column pc[2] = {t->cols[0], t->cols[ni.in_col]};
            b200_table pt{};
            pt.n_cols = 2; pt.n_rows = n; pt.cols = pc; pt.device = t->device;
            ni.st->consume(&pt);
            B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        }
        if (coalesce(t, n)) return;  // small batch of the fast-path signature: buffered until a launch is worth it
        flush_coalesced();
        if (t->device >= 0) {
            B200_REQUIRE(t->device == device, "b200 groupby: batch lives on a different device than the state");
            for (int64_t r0 = 0; r0 < n; r0 += CHUNK_ROWS) {
                int64_t rows = std::min(CHUNK_ROWS, n - r0);
                B200_REQUIRE(r0 % 8 == 0, "internal: chunk offset must be byte aligned for validity bitmaps");
                std::vector<const void*> data(n_cols, nullptr);
                std::vector<const uint8_t*> valid(n_cols, nullptr);
                for (int c = 0; c < n_cols; c++) {
                    if (!used[c]) continue;
                    data[c] = (const char*)t->cols[c].data + r0 * ctype_size(c_types[c]);
                    valid[c] = t->cols[c].validity ? t->cols[c].validity + r0 / 8 : nullptr;
                }
                consume_device_chunk(data, valid, rows);
            }
            return;
        }
        // host batch: pinned or pageable host memory, staged through two device buffers per column so the
        // H2D copy of chunk c+1 overlaps the kernel of chunk c (replaces convertTableToGPU,
        // bodo/pandas/physical/operator.cpp:293-380).
        const int64_t HCHUNK = 1ll << 24;  // 16 Mi rows (128 MiB per 8-byte column)
        if (!copy_stream) {
            B200_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
            for (int b = 0; b < 2; b++) {
                B200_CUDA(cudaEventCreateWithFlags(&stage_free[b], cudaEventDisableTiming));
                B200_CUDA(cudaEventCreateWithFlags(&stage_ready[b], cudaEventDisableTiming));
                stage[b].resize(2 * n_cols);
            }
        }
        int64_t nchunks = (n + HCHUNK - 1) / HCHUNK;
        for (int64_t ci = 0; ci < nchunks; ci++) {
            int b = (int)(ci & 1);
            int64_t r0 = ci * HCHUNK, rows = std::min(HCHUNK, n - r0);
            if (stage_recorded[b]) B200_CUDA(cudaStreamWaitEvent(copy_stream, stage_free[b], 0));
            std::vector<const void*> data(n_cols, nullptr);
            std::vector<const uint8_t*> valid(n_cols, nullptr);
            for (int c = 0; c < n_cols; c++) {
                if (!used[c]) continue;
                size_t isz = ctype_size(c_types[c]);
                stage[b][2 * c].ensure((size_t)std::min(HCHUNK, n) * isz);
                B200_CUDA(cudaMemcpyAsync(stage[b][2 * c].p, (const char*)t->cols[c].data + r0 * isz, rows * isz, cudaMemcpyHostToDevice, copy_stream));
                data[c] = stage[b][2 * c].p;
                if (t->cols[c].validity) {
                    stage[b][2 * c + 1].ensure((size_t)(std::min(HCHUNK, n) + 7) / 8 + 8);
                    B200_CUDA(cudaMemcpyAsync(stage[b][2 * c + 1].p, t->cols[c].validity + r0 / 8, (rows + 7) / 8, cudaMemcpyHostToDevice, copy_stream));
                    valid[c] = stage[b][2 * c + 1].as<uint8_t>();
                }
            }
            B200_CUDA(cudaEventRecord(stage_ready[b], copy_stream));
            B200_CUDA(cudaStreamWaitEvent(stream, stage_ready[b], 0));
            consume_device_chunk(data, valid, rows);
            B200_CUDA(cudaEventRecord(stage_free[b], stream));
            stage_recorded[b] = true;
        }
    }

    // ---- coalescing of small streaming batches ----
    // The reference streams 32 768-row batches (bodo/libs/streaming/_shuffle.h:27-31); the SM-partitioned and low-cardinality
    // kernels want >= 2^20 rows per launch.  Batches of the fast-path signature (non-null int64 key, SUM / COUNT / SIZE over one
    // non-null int64 value column) below that size are appended to a device-side buffer (one D2D or H2D copy per column) and
    // consumed together when the buffer is full, when a batch of another shape arrives, or when the build ends.
    static constexpr int64_t CO_MIN_BATCH = 1ll << 20, CO_ROWS = 1ll << 22;
    DevBuf co_key, co_val;
    int64_t co_n = 0, co_batches = 0;
    int co_vcol = -1;
    bool coalesce(const b200_table* t, int64_t n) {
        if (n == 0 || n >= CO_MIN_BATCH || nk != 1 || n_funcs < 1 || c_types[0] != CT_INT64 || t->cols[0].validity != nullptr) return false;
        { const char* e = getenv("B200_COALESCE"); if (e && e[0] == '0') return false; }
        int vcol = -1;
        for (auto& f : funcs) {
            if (f.kind == K_SIZE) continue;
            if (!((f.kind == K_SUM_I64 || f.kind == K_COUNT) && f.in_ctype == CT_INT64 && t->cols[f.in_col].validity == nullptr)) return false;
            if (vcol >= 0 && vcol != f.in_col) return false;
            vcol = f.in_col;
        }
        if (!spg_probe()) return false;
        if (co_n > 0 && (co_vcol != vcol || co_n + n > CO_ROWS)) flush_coalesced();
        co_vcol = vcol;
        co_key.ensure((size_t)CO_ROWS * 8);
        if (vcol >= 0) co_val.ensure((size_t)CO_ROWS * 8);
        const cudaMemcpyKind kind = t->device >= 0 ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        if (t->device >= 0) B200_REQUIRE(t->device == device, "b200 groupby: batch lives on a different device than the state");
        B200_CUDA(cudaMemcpyAsync(co_key.as<long long>() + co_n, t->cols[0].data, (size_t)n * 8, kind, stream));
        if (vcol >= 0) B200_CUDA(cudaMemcpyAsync(co_val.as<long long>() + co_n, t->cols[vcol].data, (size_t)n * 8, kind, stream));
        if (kind == cudaMemcpyHostToDevice) B200_CUDA(cudaStreamSynchronize(stream));  // the caller may reuse its host batch right away
        co_n += n;
        co_batches++;
        if (co_n + CO_MIN_BATCH > CO_ROWS) flush_coalesced();
        return true;
    }
    void flush_coalesced() {
        if (co_n == 0) return;
        std::vector<const void*> data(n_cols, nullptr);
        std::vector<const uint8_t*> valid(n_cols, nullptr);
        data[0] = co_key.p;
        if (co_vcol >= 0) data[co_vcol] = co_val.p;
        const int64_t n = co_n;
        co_n = 0;
        consume_device_chunk(data, valid, n);
    }

    // ---- finalize ----
    // Compacts the occupied slots (owned_only: of the groups this rank owns).  No host synchronisation: the output is sized by
    // the table's group limit (cap / 2 + the two special slots), the count stays on the device (counters[2]).
    int64_t max_out_bound() const { return (int64_t)(cap / 2) + 2; }
    void compact(bool owned_only = false) {
        int64_t max_out = max_out_bound();
        d_slot_of_out.ensure((size_t)max_out * 8);
        B200_CUDA(cudaMemsetAsync((char*)d_counters.p + 16, 0, 8, stream));
        if (nk > 1)
            compact_mk_kernel<<<grid_for((int64_t)cap), 256, 0, stream>>>(d_tags.as<unsigned long long>(), cap, d_counters.as<long long>() + 2, d_slot_of_out.as<uint64_t>(),
                                                                           mk_owner(owned_only));
        else
            compact_slots_kernel<<<grid_for((int64_t)cap + 2), 256, 0, stream>>>(d_keys.as<long long>(), cap, d_counters.as<long long>(),
                                                                                      d_counters.as<long long>() + 2, d_slot_of_out.as<uint64_t>(),
                                                                                      owned_only ? n_pes : 1, rank);
        launches++;
        B200_CUDA(cudaGetLastError());
        n_out = -1;  // known on the device (counters[2]); the host learns it with the next counter read-back
    }

    // nunique: count the distinct (key, value) pairs of every nested state into the outer table.  On the sharded path the host
    // has exchanged the nested states first (their pairs are owned where the key is owned) and the outer table already holds
    // the groups this rank owns.
    void apply_nunique() {
        if (nu_applied || nu_inner.empty()) return;
        for (auto& ni : nu_inner) {
            GroupbyState& in = *ni.st;
            B200_REQUIRE(!(parallel && n_pes > 1) || in.xchg_fused, "b200 groupby: nunique on the sharded path: exchange the nested states (b200_groupby_inner_state) before the outer finalize");
            const int64_t n_pairs = in.finalize();
            B200_REQUIRE(n_pairs >= 0, "b200 groupby: nunique: the nested exchange overflowed its slab");
            B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
            if (n_pairs == 0) continue;
            NuniqueArgs a{};
            a.pk = in.d_mk[0].as<long long>(); a.pv = in.d_mk[1].as<long long>(); a.pmask = in.d_mkmask.as<unsigned char>();
            a.slot_of_out = in.d_slot_of_out.as<uint64_t>(); a.n_pairs = n_pairs;
            a.tkeys = d_keys.as<long long>(); a.cap = cap; a.counters = d_counters.as<long long>(); a.dropna = dropna ? 1 : 0;
            a.n_acc = (int)ni.prims.size();
            for (int j = 0; j < a.n_acc; j++) a.acc[j] = d_a0[ni.prims[j]].as<unsigned long long>();
            nunique_count_kernel<<<grid_for(n_pairs), 256, 0, stream>>>(a);
            launches++;
            B200_CUDA(cudaGetLastError());
        }
        nu_applied = true;
    }

    int64_t finalize() {
        if (finalized) return n_out;
        double tf0 = now();
        struct Acc3 { double& t; double t0; ~Acc3() { t += now() - t0; } } acc3{t_finalize, tf0};
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        flush_coalesced();
        apply_nunique();
        compact(/*owned_only=*/parallel && n_pes > 1);
        const int64_t max_out = max_out_bound();
        EvalArgs e{};
        e.tkeys = nk == 1 ? d_keys.as<long long>() : nullptr; e.cap = cap; e.slot_of_out = d_slot_of_out.as<uint64_t>(); e.n_out_ptr = d_counters.as<long long>() + 2;
        e.key_ctype = c_types[0];
        size_t words = (size_t)((max_out + 31) / 32 + 1);
        if (nk == 1) {
            d_out_keys.ensure((size_t)(max_out + 32) * ctype_size(c_types[0]));
            e.out_keys = d_out_keys.p;
            bool key_nullable = arr_types[0] == ARR_NULLABLE;
            if (key_nullable) { d_out_key_valid.ensure(words * 4); e.out_key_valid = d_out_key_valid.as<uint32_t>(); }
        } else {
            EvalMkKeysArgs k{};
            k.nk = nk; k.mkmask = d_mkmask.as<unsigned char>(); k.slot_of_out = d_slot_of_out.as<uint64_t>(); k.n_out_ptr = d_counters.as<long long>() + 2;
            for (int j = 0; j < nk; j++) {
                k.mk[j] = d_mk[j].as<long long>(); k.key_ctype[j] = c_types[j];
                d_out_mk[j].ensure((size_t)(max_out + 32) * ctype_size(c_types[j]));
                k.out_keys[j] = d_out_mk[j].p;
                if (arr_types[j] == ARR_NULLABLE) { d_out_mk_valid[j].ensure(words * 4); k.out_key_valid[j] = d_out_mk_valid[j].as<uint32_t>(); }
            }
            eval_mk_keys_kernel<<<grid_for(max_out), 256, 0, stream>>>(k);
            launches++;
        }
        e.n_ops = n_outs;
        for (int j = 0; j < n_outs; j++) {
            const OutSpec& o = outs[j];
            const int p0 = o.prim[0];
            d_out_data[j].ensure((size_t)(max_out + 32) * 8);
            e.ops[j].kind = o.kind; e.ops[j].out_ctype = o.out_ctype; e.ops[j].a0 = d_a0[p0].p;
            e.ops[j].a1 = funcs[p0].has_a1 ? d_a1[p0].p : nullptr; e.ops[j].out_data = d_out_data[j].p;
            e.ops[j].b0 = o.n_prim > 1 ? d_a0[o.prim[1]].p : nullptr;
            e.ops[j].c0 = o.n_prim > 2 ? d_a0[o.prim[2]].p : nullptr;
            if (o.out_arrtype == ARR_NULLABLE) { d_out_valid[j].ensure(words * 4); e.ops[j].out_valid = d_out_valid[j].as<uint32_t>(); }
        }
        eval_output_kernel<<<grid_for(max_out), 256, 0, stream>>>(e);
        launches++;
        B200_CUDA(cudaGetLastError());
        read_counters();  // one synchronisation: the output is complete and n_out is known
        if (xchg_fused) {
            if (h_counters[7] != 0) {  // some rank's share did not fit its slab segment: nobody combined, the NCCL exchange takes over
                B200_CUDA(cudaMemsetAsync((char*)d_counters.p + 56, 0, 8, stream));
                xchg_fused = false;
                return -2;
            }
            if (h_counters[1] > 0) {
                // received rows that found the table at its group limit: grow, merge them from the slab (still intact), evaluate again
                int64_t nf = h_counters[1];
                fail_rows += nf;
                grow_to_hold(nf);
                DevBuf replay_list;
                replay_list.alloc((size_t)nf * 4);
                B200_CUDA(cudaMemcpyAsync(replay_list.p, d_fail.p, (size_t)nf * 4, cudaMemcpyDeviceToDevice, stream));
                B200_CUDA(cudaMemsetAsync((char*)d_counters.p + 8, 0, 8, stream));
                CombineArgs c = combine_args((const unsigned long long*)((const char*)xchg_slab + XCHG_HDR_BYTES), nf, /*group_limit=*/-1);
                c.index_list = replay_list.as<uint32_t>();
                if (nk > 1) { c.row_words = nk + 1 + acc_count(); MkArgs m = mk_table_args(); m.group_limit = -1; xchg_combine_mk_kernel<<<grid_for(nf), 256, 0, stream>>>(m, c, nullptr, n_pes, 0); }
                else
                combine_partials_kernel<<<grid_for(nf), 256, 0, stream>>>(c);
                if (has_firstlast) {  // over the whole slab again (idempotent): the table moved when it grew
                    CombineArgs cf = combine_args((const unsigned long long*)((const char*)xchg_slab + XCHG_HDR_BYTES), 0, -1);
                    combine_firstlast_fix_kernel<<<grid_for(1 << 20), 256, 0, stream>>>(cf, (const unsigned long long*)xchg_slab, n_pes, xchg_cap_rows);
                }
                launches++;
                B200_CUDA(cudaGetLastError());
                B200_CUDA(cudaStreamSynchronize(stream));
                return finalize();
            }
        }
        n_out = h_counters[2];
        finalized = true;
        out_cursor = 0;
        return n_out;
    }

    MkOwner mk_owner(bool owned_only) {
        MkOwner o{};
        o.nk = nk; o.n_pes = owned_only ? n_pes : 1; o.rank = rank; o.mkmask = d_mkmask.as<unsigned char>(); o.own_nk = owner_nk;
        for (int j = 0; j < nk; j++) { o.mk[j] = d_mk[j].as<long long>(); o.key_ctype[j] = c_types[j]; }
        return o;
    }
    MkArgs mk_table_args() {
        MkArgs a{};
        a.nk = nk; a.tags = d_tags.as<unsigned long long>(); a.mkmask = d_mkmask.as<unsigned char>(); a.cap = cap;
        for (int j = 0; j < nk; j++) a.mk[j] = d_mk[j].as<long long>();
        a.counters = d_counters.as<long long>(); a.group_limit = (long long)(cap / 2); a.fail_list = d_fail.as<uint32_t>();
        return a;
    }
    // ---- fused exchange (see xchg_pack_remote_kernel) ----
    bool xchg_fused = false;
    const void* xchg_slab = nullptr;
    long long xchg_cap_rows = 0;
    DevBuf d_xchg_cursors;
    CombineArgs combine_args(const unsigned long long* in, int64_t n_rows, long long group_limit) {
        CombineArgs c{};
        c.in = in; c.n_rows = n_rows; c.row_words = 2 + acc_count();
        c.tkeys = d_keys.as<long long>(); c.cap = cap; c.counters = d_counters.as<long long>(); c.group_limit = group_limit;
        c.fail_list = d_fail.as<uint32_t>(); c.index_list = nullptr; c.n_ops = n_funcs;
        for (int j = 0; j < n_funcs; j++) { c.kinds[j] = funcs[j].kind; c.a0[j] = d_a0[j].p; c.a1[j] = funcs[j].has_a1 ? d_a1[j].p : nullptr; }
        return c;
    }
    int64_t xchg_row_bytes() const { return (int64_t)((nk == 1 ? 2 : nk + 1) + acc_count()) * 8; }
    void exchange_fused_pack(void* const* peer_slabs_dev, int64_t cap_rows) {
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        flush_coalesced();
        build_done = true;
        d_xchg_cursors.ensure((size_t)std::max(n_pes, 32) * 8);
        B200_CUDA(cudaMemsetAsync(d_xchg_cursors.p, 0, (size_t)std::max(n_pes, 32) * 8, stream));
        if (nk > 1) {
            XchgPackMkArgs p{};
            p.ow = mk_owner(true); p.tags = d_tags.as<unsigned long long>(); p.cap = cap;
            int n = 0;
            for (int j = 0; j < n_funcs; j++) {
                p.acc[n++] = d_a0[j].as<unsigned long long>();
                if (funcs[j].has_a1) p.acc[n++] = d_a1[j].as<unsigned long long>();
            }
            p.n_acc = n; p.row_words = nk + 1 + n; p.cursors = d_xchg_cursors.as<unsigned long long>(); p.peer_slabs = peer_slabs_dev; p.cap_rows = cap_rows;
            xchg_pack_remote_mk_kernel<<<grid_for((int64_t)cap), 256, 0, stream>>>(p);
            xchg_post_counts_kernel<<<1, 32, 0, stream>>>(d_xchg_cursors.as<unsigned long long>(), peer_slabs_dev, n_pes, rank, cap_rows);
            launches += 2;
            B200_CUDA(cudaGetLastError());
            return;
        }
        XchgPackArgs p{};
        p.tkeys = d_keys.as<long long>(); p.cap = cap; p.counters = d_counters.as<long long>(); p.n_pes = n_pes; p.rank = rank;
        int n = 0;
        for (int j = 0; j < n_funcs; j++) {
            p.acc[n++] = d_a0[j].as<unsigned long long>();
            if (funcs[j].has_a1) p.acc[n++] = d_a1[j].as<unsigned long long>();
        }
        p.n_acc = n; p.row_words = 2 + n; p.cursors = d_xchg_cursors.as<unsigned long long>(); p.peer_slabs = peer_slabs_dev; p.cap_rows = cap_rows;
        xchg_pack_remote_kernel<<<grid_for((int64_t)cap + 2), 256, 0, stream>>>(p);
        xchg_post_counts_kernel<<<1, 32, 0, stream>>>(d_xchg_cursors.as<unsigned long long>(), peer_slabs_dev, n_pes, rank, cap_rows);
        launches += 2;
        B200_CUDA(cudaGetLastError());
    }
    void exchange_fused_combine(const void* my_slab, int64_t cap_rows) {
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        d_fail.ensure(device, (size_t)n_pes * (size_t)cap_rows * 4);
        CombineArgs c = combine_args((const unsigned long long*)((const char*)my_slab + XCHG_HDR_BYTES), 0, (long long)(cap / 2));
        if (nk > 1) { c.row_words = nk + 1 + acc_count(); xchg_combine_mk_kernel<<<grid_for(std::min<int64_t>(cap_rows, 1 << 22)), 256, 0, stream>>>(mk_table_args(), c, (const unsigned long long*)my_slab, n_pes, cap_rows); }
        else
        xchg_combine_slab_kernel<<<grid_for(std::min<int64_t>(cap_rows, 1 << 22)), 256, 0, stream>>>(c, (const unsigned long long*)my_slab, n_pes, cap_rows);
        if (has_firstlast) { combine_firstlast_fix_kernel<<<grid_for(std::min<int64_t>(cap_rows, 1 << 22)), 256, 0, stream>>>(c, (const unsigned long long*)my_slab, n_pes, cap_rows); launches++; }
        launches++;
        B200_CUDA(cudaGetLastError());
        xchg_fused = true;
        xchg_slab = my_slab; xchg_cap_rows = cap_rows;
        untracked_groups = 0;
    }

    int acc_count() const { int n = 0; for (auto& f : funcs) n += f.has_a1 ? 2 : 1; return n; }

    // ---- exchange ----
    int64_t shuffle_prepare(int64_t* send_counts) {
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        B200_REQUIRE(nk == 1, "b200 groupby: multi-column keys on the sharded path use the fused exchange (symmetric memory); the NCCL form handles single-column keys");
        flush_coalesced();
        build_done = true;
        compact(/*owned_only=*/false);
        read_counters();
        n_out = h_counters[2];
        d_dest_count.ensure((size_t)n_pes * 8);
        B200_CUDA(cudaMemsetAsync(d_dest_count.p, 0, (size_t)n_pes * 8, stream));
        PackArgs p = pack_args();
        p.pass = 0; p.out = nullptr;
        if (n_out > 0) { pack_partials_kernel<<<grid_for(n_out), 256, 0, stream>>>(p); launches++; B200_CUDA(cudaGetLastError()); }
        h_dest_count.assign(n_pes, 0);
        B200_CUDA(cudaMemcpyAsync(h_dest_count.data(), d_dest_count.p, (size_t)n_pes * 8, cudaMemcpyDeviceToHost, stream));
        B200_CUDA(cudaStreamSynchronize(stream));
        for (int d = 0; d < n_pes; d++) send_counts[d] = h_dest_count[d];
        packed_rows = n_out;
        return (int64_t)(2 + acc_count()) * 8;
    }
    PackArgs pack_args() {
        PackArgs p{};
        p.tkeys = d_keys.as<long long>(); p.cap = cap; p.slot_of_out = d_slot_of_out.as<uint64_t>(); p.n_out = n_out; p.n_pes = n_pes;
        int n = 0;
        for (int j = 0; j < n_funcs; j++) {
            p.acc[n++] = d_a0[j].as<unsigned long long>();
            if (funcs[j].has_a1) p.acc[n++] = d_a1[j].as<unsigned long long>();
        }
        p.n_acc = n; p.row_words = 2 + n; p.dest_count = d_dest_count.as<long long>();
        return p;
    }
    void shuffle_pack(void* send_buf) {
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        // exclusive scan of the per-destination counts -> running cursors
        std::vector<long long> offs(n_pes, 0);
        long long run = 0;
        for (int d = 0; d < n_pes; d++) { offs[d] = run; run += h_dest_count[d]; }
        B200_CUDA(cudaMemcpyAsync(d_dest_count.p, offs.data(), (size_t)n_pes * 8, cudaMemcpyHostToDevice, stream));
        PackArgs p = pack_args();
        p.pass = 1; p.out = (unsigned long long*)send_buf;
        if (n_out > 0) { pack_partials_kernel<<<grid_for(n_out), 256, 0, stream>>>(p); launches++; B200_CUDA(cudaGetLastError()); }
        // the table now only has to hold the groups this rank owns: clear it for the combine step
        B200_CUDA(cudaStreamSynchronize(stream));  // offs is a stack buffer
        fill(d_keys.p, cap + 2, (unsigned long long)EMPTY_KEY);
        for (int j = 0; j < n_funcs; j++) { fill(d_a0[j].p, cap + 2, funcs[j].init0); if (funcs[j].has_a1) fill(d_a1[j].p, cap + 2, funcs[j].init1); }
        B200_CUDA(cudaMemsetAsync(d_counters.p, 0, 8 * sizeof(long long), stream));
        n_groups = 0; n_groups_bound = 0; untracked_groups = 0;
    }
    void shuffle_combine(const void* recv, int64_t n_rows) {
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        if (n_rows == 0) return;
        B200_REQUIRE(n_rows < (1ll << 32), "b200 groupby: too many partial rows in one combine call");
        bool could_fail = (int64_t)(cap / 2) - n_groups_bound < n_rows;
        if (could_fail) d_fail.ensure(device, (size_t)n_rows * 4);
        auto launch = [&](const uint32_t* index_list, int64_t rows) {
            CombineArgs c{};
            c.in = (const unsigned long long*)recv; c.n_rows = rows; c.row_words = 2 + acc_count();
            // with room guaranteed the per-insert ticket (one atomic on a single counter per new group: ~170 us for 1 M
            // groups) is skipped; the groups are accounted for as `untracked_groups` until the next compaction counts them
            c.tkeys = d_keys.as<long long>(); c.cap = cap; c.counters = d_counters.as<long long>(); c.group_limit = could_fail ? (long long)(cap / 2) : -1;
            c.fail_list = d_fail.as<uint32_t>(); c.index_list = index_list; c.n_ops = n_funcs;
            for (int j = 0; j < n_funcs; j++) { c.kinds[j] = funcs[j].kind; c.a0[j] = d_a0[j].p; c.a1[j] = funcs[j].has_a1 ? d_a1[j].p : nullptr; }
            combine_partials_kernel<<<grid_for(rows), 256, 0, stream>>>(c);
            launches++;
            B200_CUDA(cudaGetLastError());
        };
        launch(nullptr, n_rows);
        settle(n_rows, could_fail, launch);
        if (has_firstlast) {
            CombineArgs c = combine_args((const unsigned long long*)recv, n_rows, -1);
            combine_firstlast_fix_kernel<<<grid_for(n_rows), 256, 0, stream>>>(c, nullptr, 0, 0);
            launches++;
            B200_CUDA(cudaGetLastError());
        }
        if (!could_fail) { n_groups_bound += n_rows; untracked_groups += n_rows; } else n_groups_bound = n_groups + untracked_groups;
    }

    int produce(b200_table* out, int32_t* out_is_last, bool produce_output) {
        if (!finalized && finalize() == -2)
            throw Error("b200 groupby: the fused exchange overflowed its slab; run the prepare/pack/combine exchange and finalize again before producing output");
        int64_t bs = output_batch_size > 0 ? output_batch_size : n_out;
        if (bs % 32 != 0 && bs < n_out) bs = (bs + 31) & ~31ll;  // validity bitmaps are sliced at word granularity
        int64_t rows = produce_output ? std::min(bs, n_out - out_cursor) : 0;
        B200_REQUIRE(out->cols != nullptr, "b200 groupby: out->cols must point to n_keys + n_funcs descriptors");
        out->n_rows = rows; out->n_cols = nk + n_outs; out->device = device;
        int64_t off = out_cursor;
        for (int kc = 0; kc < nk; kc++) {
            b200_column& k = out->cols[kc];
            const DevBuf& kd = nk == 1 ? d_out_keys : d_out_mk[kc];
            const DevBuf& kv = nk == 1 ? d_out_key_valid : d_out_mk_valid[kc];
            k.data = (char*)kd.p + off * ctype_size(c_types[kc]);
            k.validity = arr_types[kc] == ARR_NULLABLE ? kv.as<uint8_t>() + off / 8 : nullptr;
            k.length = rows; k.c_type = c_types[kc]; k.arr_type = arr_types[kc];
        }
        for (int j = 0; j < n_outs; j++) {
            b200_column& c = out->cols[nk + j];
            c.data = (char*)d_out_data[j].p + off * ctype_size(outs[j].out_ctype);
            c.validity = outs[j].out_arrtype == ARR_NULLABLE ? d_out_valid[j].as<uint8_t>() + off / 8 : nullptr;
            c.length = rows; c.c_type = outs[j].out_ctype; c.arr_type = outs[j].out_arrtype;
        }
        out_cursor += rows;
        *out_is_last = out_cursor >= n_out ? 1 : 0;
        return 0;
    }
};

}  // namespace b200

using b200::GroupbyState;

#define B200_TRY try {
#define B200_CATCH(retval)                              \
    }                                                   \
    catch (const std::exception& e) {                   \
        b200::set_last_error(e.what());                 \
        return retval;                                  \
    }

extern "C" {

void* b200_groupby_state_init(int64_t operator_id, const int8_t* build_arr_c_types, const int8_t* build_arr_array_types,
                              int32_t n_build_arrs, const int32_t* ftypes, const int32_t* f_in_offsets,
                              const int32_t* f_in_cols, int32_t n_funcs, uint64_t n_keys, int64_t output_batch_size,
                              int32_t parallel, int32_t pandas_drop_na, int32_t device, int32_t n_pes, int32_t myrank,
                              int64_t expected_groups, void* stream) {
    (void)operator_id;
    B200_TRY
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw b200::Error("b200 groupby: no CUDA device available (this path has no CPU fallback)");
    B200_REQUIRE(device >= 0 && device < ndev, "b200 groupby: bad device ordinal");
    return new GroupbyState(build_arr_c_types, build_arr_array_types, n_build_arrs, ftypes, f_in_offsets, f_in_cols, n_funcs,
                            n_keys, output_batch_size, parallel != 0, pandas_drop_na != 0, device, n_pes, myrank,
                            expected_groups, (cudaStream_t)stream);
    B200_CATCH(nullptr)
}

int b200_groupby_build_consume_batch(void* state, const b200_table* in_table, int32_t is_last, int32_t is_final_pipeline,
                                     int32_t* request_input) {
    (void)is_final_pipeline;
    B200_TRY
    B200_REQUIRE(state && in_table, "b200 groupby: null state or table");
    auto* s = (GroupbyState*)state;
    s->consume(in_table);
    if (request_input) *request_input = 1;
    if (is_last && !s->parallel) s->build_done = true;
    return is_last ? 1 : 0;
    B200_CATCH(-1)
}

int64_t b200_groupby_shuffle_prepare(void* state, int64_t* send_row_counts) {
    B200_TRY
    return ((GroupbyState*)state)->shuffle_prepare(send_row_counts);
    B200_CATCH(-1)
}
int64_t b200_groupby_shuffle_send_bytes(void* state) {
    auto* s = (GroupbyState*)state;
    return s->packed_rows * (int64_t)(2 + s->acc_count()) * 8;
}
int b200_groupby_shuffle_pack(void* state, void* send_buf) {
    B200_TRY
    ((GroupbyState*)state)->shuffle_pack(send_buf);
    return 0;
    B200_CATCH(-1)
}
int64_t b200_groupby_exchange_row_bytes(void* state) { return ((GroupbyState*)state)->xchg_row_bytes(); }
int b200_groupby_exchange_fused_pack(void* state, void* const* peer_slabs_dev, int64_t cap_rows) {
    B200_TRY
    B200_REQUIRE(state && peer_slabs_dev && cap_rows > 0, "b200 groupby: bad fused-exchange arguments");
    ((GroupbyState*)state)->exchange_fused_pack(peer_slabs_dev, cap_rows);
    return 0;
    B200_CATCH(-1)
}
int b200_groupby_exchange_fused_combine(void* state, const void* my_slab, int64_t cap_rows) {
    B200_TRY
    B200_REQUIRE(state && my_slab && cap_rows > 0, "b200 groupby: bad fused-exchange arguments");
    ((GroupbyState*)state)->exchange_fused_combine(my_slab, cap_rows);
    return 0;
    B200_CATCH(-1)
}
int b200_groupby_shuffle_combine(void* state, const void* recv_buf, int64_t n_recv_rows) {
    B200_TRY
    ((GroupbyState*)state)->shuffle_combine(recv_buf, n_recv_rows);
    return 0;
    B200_CATCH(-1)
}
int32_t b200_groupby_num_inner_states(void* state) { return state ? (int32_t)((GroupbyState*)state)->nu_inner.size() : 0; }
void* b200_groupby_inner_state(void* state, int32_t i) {
    auto* s = (GroupbyState*)state;
    if (!s || i < 0 || i >= (int32_t)s->nu_inner.size()) { b200::set_last_error("b200_groupby_inner_state: bad arguments"); return nullptr; }
    return s->nu_inner[i].st.get();
}

int64_t b200_groupby_finalize(void* state) {
    B200_TRY
    return ((GroupbyState*)state)->finalize();
    B200_CATCH(-1)
}
int b200_groupby_produce_output_batch(void* state, b200_table* out, int32_t* out_is_last, int32_t produce_output) {
    B200_TRY
    B200_REQUIRE(state && out && out_is_last, "b200 groupby: null argument");
    return ((GroupbyState*)state)->produce(out, out_is_last, produce_output != 0);
    B200_CATCH(-1)
}
void b200_delete_groupby_state(void* state) { delete (GroupbyState*)state; }

int64_t b200_groupby_get_metric(void* state, int32_t which) {
    auto* s = (GroupbyState*)state;
    switch (which) {
        case 0: return s->finalized ? s->n_out : s->n_groups;
        case 1: return (int64_t)s->cap;
        case 2: return s->rows_consumed;
        case 3: return s->rebuilds;
        case 4: return s->launches;
        case 5: return s->fail_rows;
        case 6: return (int64_t)s->consume_kernel_us();
        case 7: return s->consume_launches;
        case 8: return s->spg_launches;
        case 9: return s->spg_retry_rows;
        case 10: return s->lc_launches;
        case 11: return s->co_batches;
        case 12: return s->spgg_launches;
        case 14: return s->spgn_launches;
        case 13: { cudaSetDevice(s->device); s->read_counters(); return s->n_groups + s->untracked_groups; }  // exact (synchronises the stream)
        case 100: s->profiling = true; return 0;
        default: return -1;
    }
}

}  // extern "C"
