// join.cu — streaming hash join on one B200 (sm_100a).
//
// Replaces HashJoinState / JoinPartition of the reference (bodo/libs/streaming/_join.cpp):
//   build  : join_build_consume_batch (:3134-3443) appends batches to device-resident build columns; on the
//            last batch BuildHashTable (:381-437) + FinalizeGroups (:439-512) become three kernels:
//            insert+count (one table slot per distinct key, rows-per-key counter), exclusive scan (CSR
//            groups_offsets), fill (CSR groups = build row ids).  Keys with exactly one build row keep the
//            row id in the slot itself, so the common 1:N probe needs no CSR lookup.
//   probe  : join_probe_consume_batch (:3459-3900): pass A looks up every probe row and writes its match count,
//            a scan turns counts into output offsets, pass B expands the matches and gathers the kept build and
//            probe columns straight into the output columns (produce_probe_output :729-827 +
//            ChunkedTableBuilder::AppendJoinOutput fused; no (build_idx, probe_idx) pair vectors in HBM,
//            unlike the cuDF path bodo/libs/streaming/cuda_join.cpp:543-612).
//   outer  : probe_table_outer emits unmatched probe rows with NULL build columns; build_table_outer tracks
//            matched build rows and emits the unmatched ones after the last probe batch.
// NA keys: `is_na_equal` is a state option, as in the reference's HashJoinState.  true (the pandas door,
// bodo/pandas/physical/join.h:267): NA joins NA.  false (the default of join_state_init_py_entry, SQL semantics): rows
// with an NA key never match — they are filtered from the build table unless it is the outer side
// (_join.cpp:3180 filter_na_values) and only survive as NULL-extended rows of an outer join.
// Key columns: 1..4 (HashJoinState's n_keys), the first n_keys columns of each side.  One key column uses the key-valued table
// below; a tuple of 2..4 uses a tag table whose slots point at a representative build row (see "multi-column keys").  With
// is_na_equal = false a row with an NA in ANY key column matches nothing (filter_na_values works over all keys); with true, NA
// equals NA at the same key position and never equals a value.
#include <algorithm>
#include <type_traits>
#include <vector>

#include "common.cuh"

namespace b200 {

constexpr long long J_EMPTY = (long long)0x8000000000000000ULL;
constexpr int J_MAX_COLS = 32;
constexpr uint32_t J_NONE = 0xffffffffu;

// ---- exclusive scan u32 -> u64 (reduce / scan-of-sums / scan), tile = 2048 elements per CTA ----
constexpr int SCAN_TILE = 2048;
__global__ void __launch_bounds__(256) scan_reduce_kernel(const uint32_t* in, int64_t n, unsigned long long* block_sums) {
    __shared__ unsigned long long sh[256];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    unsigned long long s = 0;
    for (int k = threadIdx.x; k < SCAN_TILE; k += 256) { int64_t i = base + k; if (i < n) s += in[i]; }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) block_sums[blockIdx.x] = sh[0];
}
__global__ void __launch_bounds__(1024) scan_sums_kernel(unsigned long long* block_sums, int64_t nb, unsigned long long* total) {
    // single CTA: each thread owns a contiguous run of block sums
    __shared__ unsigned long long sh[1024];
    int64_t per = (nb + 1023) / 1024;
    int64_t b0 = threadIdx.x * per, b1 = b0 + per < nb ? b0 + per : nb;
    unsigned long long s = 0;
    for (int64_t b = b0; b < b1; b++) s += block_sums[b];
    sh[threadIdx.x] = s;
    __syncthreads();
    // inclusive Hillis-Steele over 1024 partials
    for (int o = 1; o < 1024; o <<= 1) {
        unsigned long long v = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
        __syncthreads();
        sh[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned long long run = threadIdx.x ? sh[threadIdx.x - 1] : 0;
    for (int64_t b = b0; b < b1; b++) { unsigned long long v = block_sums[b]; block_sums[b] = run; run += v; }
    if (threadIdx.x == 1023) *total = sh[1023];
}
__global__ void __launch_bounds__(256) scan_apply_kernel(const uint32_t* in, int64_t n, const unsigned long long* block_sums,
                                                         unsigned long long* out) {
    __shared__ unsigned long long sh[256];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    constexpr int PER = SCAN_TILE / 256;
    uint32_t v[PER];
    unsigned long long s = 0;
    int64_t i0 = base + (int64_t)threadIdx.x * PER;
#pragma unroll
    for (int k = 0; k < PER; k++) { v[k] = (i0 + k < n) ? in[i0 + k] : 0; s += v[k]; }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        unsigned long long t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
        __syncthreads();
        sh[threadIdx.x] += t;
        __syncthreads();
    }
    unsigned long long run = block_sums[blockIdx.x] + (threadIdx.x ? sh[threadIdx.x - 1] : 0);
#pragma unroll
    for (int k = 0; k < PER; k++) { if (i0 + k < n) out[i0 + k] = run; run += v[k]; }
}

struct Scanner {
    DevBuf sums, total;
    unsigned long long* h_total = nullptr;
    ~Scanner() { pinned_release(h_total, 8); }
    // out[i] = sum_{j<i} in[j]; returns the grand total (synchronises the stream)
    unsigned long long run(const uint32_t* in, int64_t n, unsigned long long* out, cudaStream_t st, int64_t* launches) {
        if (!h_total) h_total = (unsigned long long*)pinned_acquire(8);
        if (n == 0) return 0;
        int64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
        sums.ensure((size_t)nb * 8);
        total.ensure(8);
        scan_reduce_kernel<<<(unsigned)nb, 256, 0, st>>>(in, n, sums.as<unsigned long long>());
        scan_sums_kernel<<<1, 1024, 0, st>>>(sums.as<unsigned long long>(), nb, total.as<unsigned long long>());
        scan_apply_kernel<<<(unsigned)nb, 256, 0, st>>>(in, n, sums.as<unsigned long long>(), out);
        *launches += 3;
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaMemcpyAsync(h_total, total.p, 8, cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        return *h_total;
    }
};

// ---- hash table ----
struct SlotInfo { uint32_t cnt; uint32_t first; };  // rows with this key; one of those rows (row id)

__device__ __forceinline__ uint64_t j_hash_slot(long long key, uint64_t mask) {
    return (xxh3_64_short((uint64_t)key, 8, SEED_HASH_JOIN) >> 32) & mask;
}
// capacity >= 2 * n_build, so an insert always finds a free slot
__device__ __forceinline__ uint32_t j_find_or_insert(long long* tkeys, uint64_t cap, long long key) {
    uint64_t mask = cap - 1, s = j_hash_slot(key, mask);
    while (true) {
        long long k = __ldcg(tkeys + s);
        if (k == key) return (uint32_t)s;
        if (k == J_EMPTY) {
            long long prev = (long long)atomicCAS((unsigned long long*)(tkeys + s), (unsigned long long)J_EMPTY, (unsigned long long)key);
            if (prev == J_EMPTY || prev == key) return (uint32_t)s;
        }
        s = (s + 1) & mask;
    }
}
__device__ __forceinline__ uint32_t j_find(const long long* __restrict__ tkeys, uint64_t cap, long long key) {
    uint64_t mask = cap - 1, s = j_hash_slot(key, mask);
    while (true) {
        long long k = __ldg(tkeys + s);
        if (k == key) return (uint32_t)s;
        if (k == J_EMPTY) return J_NONE;
        s = (s + 1) & mask;
    }
}

// BuildHashTable: slot per distinct key, num_rows_in_group, build_row_to_group_map (= row_slot)
__global__ void join_insert_count_kernel(const void* key_data, int key_ctype, const uint8_t* key_valid_bytes, int64_t n,
                                         long long* tkeys, uint64_t cap, SlotInfo* info, uint32_t* row_slot, int na_equal) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        uint32_t s;
        if (key_valid_bytes && !key_valid_bytes[i]) {
            if (!na_equal) { row_slot[i] = J_NONE; continue; }  // never matches: belongs to no group
            s = (uint32_t)cap;  // NA group
        } else {
            long long key = load_int_as_i64(key_data, key_ctype, i);
            s = key == J_EMPTY ? (uint32_t)cap + 1 : j_find_or_insert(tkeys, cap, key);
        }
        row_slot[i] = s;
        atomicAdd(&info[s].cnt, 1u);
        info[s].first = (uint32_t)i;  // any row of the group; exact when cnt == 1
    }
}
__global__ void join_slot_counts_kernel(const SlotInfo* info, uint64_t n_slots, uint32_t* cnt_multi) {
    // CSR only holds groups with more than one row
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < n_slots; s += stride) {
        uint32_t c = info[s].cnt;
        cnt_multi[s] = c > 1 ? c : 0;
    }
}
// FinalizeGroups: groups[offs[slot] + k] = k-th build row of the slot's key
__global__ void join_fill_groups_kernel(const uint32_t* row_slot, int64_t n, const SlotInfo* info, const unsigned long long* offs,
                                        uint32_t* fill, uint32_t* groups) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        uint32_t s = row_slot[i];
        if (s != J_NONE && info[s].cnt > 1) groups[offs[s] + atomicAdd(&fill[s], 1u)] = (uint32_t)i;
    }
}

// probe pass A: slot + match count per probe row
// mode 0: inner / outer join; 1: anti join (a probe row goes out, once and with NULL build columns, iff it has NO match:
// the is_anti_join template of the reference's probe, _join.cpp:763-767); 2: mark join (every probe row goes out once, without
// build columns; mark[i] says whether it has a match, _join.cpp:3668-3693)
__global__ void join_probe_count_kernel(const void* key_data, int key_ctype, const uint8_t* key_valid, int64_t n,
                                        const long long* tkeys, uint64_t cap, const SlotInfo* info, int probe_outer,
                                        uint32_t* pslot, uint32_t* pcnt, int na_equal, int mode, uint8_t* mark) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        uint32_t s;
        if (!bit_valid(key_valid, i)) s = na_equal ? (uint32_t)cap : J_NONE;
        else {
            long long key = load_int_as_i64(key_data, key_ctype, i);
            s = key == J_EMPTY ? (uint32_t)cap + 1 : j_find(tkeys, cap, key);
        }
        uint32_t c = s == J_NONE ? 0 : info[s].cnt;
        if (c == 0) s = J_NONE;
        if (mode == 1) { pslot[i] = J_NONE; pcnt[i] = c ? 0u : 1u; continue; }
        if (mode == 2) { pslot[i] = J_NONE; pcnt[i] = 1u; mark[i] = c ? 1 : 0; continue; }
        pslot[i] = s;
        pcnt[i] = c ? c : (probe_outer ? 1u : 0u);
    }
}

// ---- multi-column keys (2..4 key columns) ----
// A tuple maps to a slot through the slot's tag word (mk_tag, common.cuh: 0 = free, 1 = being claimed, bit 63 = published tag of
// the widened key values + NA mask).  The claiming row writes itself into SlotInfo.first before it publishes the tag, and first is
// never overwritten: it is the slot's representative row.  A reader that finds its own tag compares the NA mask and every key
// value with that row in the build columns, which stay on the device for the state's lifetime, so the table holds no key columns.
// NA is part of the tuple, so there is no NA slot and no free-slot-marker slot.  Everything that only sees slots and row ids
// (counts, CSR groups, gather, outer tail) is the single-key code.
constexpr int J_MAX_KEYS = MAX_HASH_KEYS;
struct JKeys {  // the key columns of one side: validity is one byte per row on the build side, a bitmap on the probe side
    const void* data[J_MAX_KEYS];
    const uint8_t* valid[J_MAX_KEYS];
    int ctype[J_MAX_KEYS];
};
// row i's tuple widened to int64 (NA positions read as 0); returns the NA mask, bit j set = key j valid
template <int NK, bool BYTE_VALID>
__device__ __forceinline__ unsigned int j_load_tuple(const JKeys& k, int64_t i, long long (&keys)[NK]) {
    unsigned int mask = 0;
#pragma unroll
    for (int j = 0; j < NK; j++) {
        const bool v = BYTE_VALID ? (k.valid[j] == nullptr || k.valid[j][i] != 0) : bit_valid(k.valid[j], i);
        keys[j] = v ? (long long)load_int_as_i64(k.data[j], k.ctype[j], i) : 0;
        mask |= v ? (1u << j) : 0u;
    }
    return mask;
}
template <int NK>
__device__ __forceinline__ bool j_tuple_eq(const JKeys& b, uint32_t brow, const long long (&keys)[NK], unsigned int mask) {
    long long bk[NK];
    bool eq = j_load_tuple<NK, true>(b, brow, bk) == mask;
#pragma unroll
    for (int j = 0; j < NK; j++) eq = eq && bk[j] == keys[j];
    return eq;
}
// BuildHashTable for tuples: the claim protocol of the multi-key groupby (find_or_insert_mk); row_slot as in the single-key kernel
template <int NK>
__global__ void join_insert_count_mk_kernel(const __grid_constant__ JKeys b, int64_t n, unsigned long long* tags, uint64_t cap, SlotInfo* info,
                                            uint32_t* row_slot, int na_equal) {
    const uint64_t m = cap - 1;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        long long keys[NK];
        const unsigned int mask = j_load_tuple<NK, true>(b, i, keys);
        if (!na_equal && mask != (1u << NK) - 1u) { row_slot[i] = J_NONE; continue; }  // an NA in any key column: never matches
        const unsigned long long tag = mk_tag(keys, mask, NK);
        uint64_t s = (tag >> 20) & m;
        while (true) {
            const unsigned long long t = ld_acquire_u64(tags + s);
            if (t == tag) {
                if (j_tuple_eq<NK>(b, __ldcg(&info[s].first), keys, mask)) break;
            } else if (t == TAG_EMPTY) {
                if (atomicCAS(tags + s, TAG_EMPTY, TAG_LOCKED) == TAG_EMPTY) {
                    info[s].first = (uint32_t)i;
                    __threadfence();
                    atomicExch(tags + s, tag);  // publish
                    break;
                }
                continue;  // another row claimed the slot meanwhile: look at it again
            } else if (t == TAG_LOCKED) {
                continue;  // being claimed: re-read
            }
            s = (s + 1) & m;
        }
        row_slot[i] = (uint32_t)s;
        atomicAdd(&info[s].cnt, 1u);
    }
}
template <int NK>
__device__ __forceinline__ uint32_t j_find_mk(const unsigned long long* __restrict__ tags, uint64_t cap, const SlotInfo* __restrict__ info,
                                              const JKeys& b, const long long (&keys)[NK], unsigned int mask) {
    const uint64_t m = cap - 1;
    const unsigned long long tag = mk_tag(keys, mask, NK);
    for (uint64_t s = (tag >> 20) & m;; s = (s + 1) & m) {
        const unsigned long long t = __ldg(tags + s);
        if (t == tag && j_tuple_eq<NK>(b, info[s].first, keys, mask)) return (uint32_t)s;
        if (t == TAG_EMPTY) return J_NONE;
    }
}
// probe pass A for tuples: same outputs and modes as join_probe_count_kernel
template <int NK>
__global__ void join_probe_count_mk_kernel(const __grid_constant__ JKeys p, const __grid_constant__ JKeys b, int64_t n, const unsigned long long* tags,
                                           uint64_t cap, const SlotInfo* info, int probe_outer, uint32_t* pslot, uint32_t* pcnt, int na_equal, int mode,
                                           uint8_t* mark) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        long long keys[NK];
        const unsigned int mask = j_load_tuple<NK, false>(p, i, keys);
        uint32_t s = na_equal || mask == (1u << NK) - 1u ? j_find_mk<NK>(tags, cap, info, b, keys, mask) : J_NONE;
        uint32_t c = s == J_NONE ? 0 : info[s].cnt;
        if (c == 0) s = J_NONE;
        if (mode == 1) { pslot[i] = J_NONE; pcnt[i] = c ? 0u : 1u; continue; }
        if (mode == 2) { pslot[i] = J_NONE; pcnt[i] = 1u; mark[i] = c ? 1 : 0; continue; }
        pslot[i] = s;
        pcnt[i] = c ? c : (probe_outer ? 1u : 0u);
    }
}

struct GatherArgs {
    int64_t n_probe;
    const uint32_t* pslot;
    const unsigned long long* poff;
    const SlotInfo* info;
    const unsigned long long* goffs;
    const uint32_t* groups;
    uint8_t* bmatched;  // build_outer: matched flags per build row, else nullptr
    int n_b, n_p;       // kept build / probe columns
    const void* b_data[J_MAX_COLS]; const uint8_t* b_valid[J_MAX_COLS]; int b_size[J_MAX_COLS];
    const void* p_data[J_MAX_COLS]; const uint8_t* p_valid[J_MAX_COLS]; int p_size[J_MAX_COLS];
    void* ob_data[J_MAX_COLS]; uint8_t* ob_valid[J_MAX_COLS];  // output columns (validity: one byte per row or nullptr)
    void* op_data[J_MAX_COLS]; uint8_t* op_valid[J_MAX_COLS];
};
__device__ __forceinline__ void copy_item(void* dst, int64_t d, const void* src, int64_t s, int size) {
    switch (size) {
        case 8: ((uint64_t*)dst)[d] = ((const uint64_t*)src)[s]; break;
        case 4: ((uint32_t*)dst)[d] = ((const uint32_t*)src)[s]; break;
        case 2: ((uint16_t*)dst)[d] = ((const uint16_t*)src)[s]; break;
        default: ((uint8_t*)dst)[d] = ((const uint8_t*)src)[s]; break;
    }
}
__device__ __forceinline__ void zero_item(void* dst, int64_t d, int size) {
    switch (size) {
        case 8: ((uint64_t*)dst)[d] = 0; break;
        case 4: ((uint32_t*)dst)[d] = 0; break;
        case 2: ((uint16_t*)dst)[d] = 0; break;
        default: ((uint8_t*)dst)[d] = 0; break;
    }
}
// probe pass B: expand matches and gather both sides into the output columns (build validity is byte-per-row)
__global__ void __launch_bounds__(256) join_probe_gather_kernel(const __grid_constant__ GatherArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_probe; i += stride) {
        uint32_t s = a.pslot[i];
        unsigned long long o = a.poff[i];
        uint32_t c = s == J_NONE ? 0 : a.info[s].cnt;
        uint32_t reps = c ? c : (a.poff[i + 1] - o ? 1u : 0u);  // outer probe row without match: one NULL-build row
        for (uint32_t q = 0; q < reps; q++) {
            int64_t orow = (int64_t)(o + q);
            if (c) {
                uint32_t brow = c == 1 ? a.info[s].first : a.groups[a.goffs[s] + q];
                if (a.bmatched) a.bmatched[brow] = 1;
                for (int k = 0; k < a.n_b; k++) {
                    copy_item(a.ob_data[k], orow, a.b_data[k], brow, a.b_size[k]);
                    if (a.ob_valid[k]) a.ob_valid[k][orow] = a.b_valid[k] ? a.b_valid[k][brow] : 1;
                }
            } else {
                for (int k = 0; k < a.n_b; k++) { zero_item(a.ob_data[k], orow, a.b_size[k]); a.ob_valid[k][orow] = 0; }
            }
            for (int k = 0; k < a.n_p; k++) {
                copy_item(a.op_data[k], orow, a.p_data[k], i, a.p_size[k]);
                if (a.op_valid[k]) a.op_valid[k][orow] = bit_valid(a.p_valid[k], i) ? 1 : 0;
            }
        }
    }
}

// build_outer tail: unmatched build rows with NULL probe columns
__global__ void join_unmatched_flags_kernel(const uint8_t* bmatched, int64_t n, uint32_t* flags) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) flags[i] = bmatched[i] ? 0u : 1u;
}
struct TailArgs {
    int64_t n_build;
    const uint32_t* flags;
    const unsigned long long* off;
    int n_b, n_p;
    const void* b_data[J_MAX_COLS]; const uint8_t* b_valid[J_MAX_COLS]; int b_size[J_MAX_COLS];
    int p_size[J_MAX_COLS];
    void* ob_data[J_MAX_COLS]; uint8_t* ob_valid[J_MAX_COLS];
    void* op_data[J_MAX_COLS]; uint8_t* op_valid[J_MAX_COLS];
};
__global__ void join_unmatched_emit_kernel(const __grid_constant__ TailArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_build; i += stride) {
        if (!a.flags[i]) continue;
        int64_t orow = (int64_t)a.off[i];
        for (int k = 0; k < a.n_b; k++) {
            copy_item(a.ob_data[k], orow, a.b_data[k], i, a.b_size[k]);
            if (a.ob_valid[k]) a.ob_valid[k][orow] = a.b_valid[k] ? a.b_valid[k][i] : 1;
        }
        for (int k = 0; k < a.n_p; k++) { zero_item(a.op_data[k], orow, a.p_size[k]); a.op_valid[k][orow] = 0; }
    }
}

__global__ void expand_bitmap_kernel(const uint8_t* bitmap, int64_t n, uint8_t* bytes) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) bytes[i] = bit_valid(bitmap, i) ? 1 : 0;
}
__global__ void pack_bitmap_kernel(const uint8_t* bytes, int64_t n, uint32_t* words) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t n_round = (n + 31) & ~31ll;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_round; i += stride) {
        unsigned m = __ballot_sync(0xffffffffu, i < n && bytes[i]);
        if ((threadIdx.x & 31) == 0) words[i >> 5] = m;
    }
}
__global__ void fill_i64_kernel(long long* p, uint64_t n, long long v) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}

// ---- fast path: unique build keys + inner join --------------------------------------------------
// One 16-byte slot {key, first_row, cnt} (one 32-byte sector per lookup instead of two), the non-key build columns
// packed row-major in 8-byte fields (one sector per matched row instead of one per column), and a single fused kernel:
// lookup -> warp-aggregated output cursor -> gather both sides straight into the output columns. No per-row slot /
// count / offset arrays and no scan. Output order follows the cursor (unspecified, as in the reference).
struct __align__(16) Slot16 { long long key; uint32_t first; uint32_t cnt; };

__global__ void join_make_slots16_kernel(const long long* tkeys, const SlotInfo* info, uint64_t n_slots, Slot16* out) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < n_slots; s += stride) {
        Slot16 e; e.key = tkeys[s]; e.first = info[s].first; e.cnt = info[s].cnt;
        out[s] = e;
    }
}
struct PackPayloadArgs {
    int64_t n_build;
    int n_fields;
    const void* src[J_MAX_COLS];
    int size[J_MAX_COLS];
    unsigned long long* out;  // n_build x n_fields 8-byte fields
};
__global__ void join_pack_payload_kernel(const __grid_constant__ PackPayloadArgs a) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n_build; i += stride)
        for (int f = 0; f < a.n_fields; f++) {
            unsigned long long v = 0;
            switch (a.size[f]) {
                case 8: v = ((const uint64_t*)a.src[f])[i]; break;
                case 4: v = ((const uint32_t*)a.src[f])[i]; break;
                case 2: v = ((const uint16_t*)a.src[f])[i]; break;
                default: v = ((const uint8_t*)a.src[f])[i]; break;
            }
            a.out[i * a.n_fields + f] = v;
        }
}
struct FastProbeArgs {
    int64_t n_probe;
    const void* key_data; int key_ctype; const uint8_t* key_valid;
    const Slot16* slots; uint64_t cap;
    const unsigned long long* bpack; int n_fields;
    unsigned long long* cursor;
    int n_b, n_p;
    int na_equal;
    int b_field[J_MAX_COLS];               // kept build col -> payload field index, -1 = the key column
    const uint8_t* b_valid[J_MAX_COLS]; int b_size[J_MAX_COLS];
    const void* p_data[J_MAX_COLS]; const uint8_t* p_valid[J_MAX_COLS]; int p_size[J_MAX_COLS];
    void* ob_data[J_MAX_COLS]; uint8_t* ob_valid[J_MAX_COLS];
    void* op_data[J_MAX_COLS]; uint8_t* op_valid[J_MAX_COLS];
};
__device__ __forceinline__ void store_sized(void* dst, int64_t d, unsigned long long v, int size) {
    switch (size) {
        case 8: ((uint64_t*)dst)[d] = v; break;
        case 4: ((uint32_t*)dst)[d] = (uint32_t)v; break;
        case 2: ((uint16_t*)dst)[d] = (uint16_t)v; break;
        default: ((uint8_t*)dst)[d] = (uint8_t)v; break;
    }
}
__global__ void __launch_bounds__(256) join_probe_fast_kernel(const __grid_constant__ FastProbeArgs a) {
    // tile = 1024 probe rows per CTA iteration (4 per thread); ONE global cursor atomic per tile (a cursor atomic per
    // warp serialises on a single L2 address: measured 117 ms for 1e9 probe rows, dominated by that atomic)
    constexpr int R = 4, NW = 8, TILE = 256 * R;
    __shared__ unsigned int wcnt[R * NW];
    __shared__ unsigned int woff[R * NW];
    __shared__ unsigned long long tile_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t mask = a.cap - 1;
    const int64_t n_tiles = (a.n_probe + TILE - 1) / TILE;
    for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        long long key[R];
        uint32_t brow[R];
        unsigned int rank[R];
        bool match[R], kvalid[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int64_t i = t * TILE + r * 256 + threadIdx.x;
            match[r] = false; kvalid[r] = true; key[r] = 0; brow[r] = 0;
            if (i < a.n_probe) {
                kvalid[r] = bit_valid(a.key_valid, i);
                key[r] = load_int_as_i64(a.key_data, a.key_ctype, i);
                if (!kvalid[r]) { if (a.na_equal) { Slot16 e = a.slots[a.cap]; match[r] = e.cnt > 0; brow[r] = e.first; } }
                else if (key[r] == J_EMPTY) { Slot16 e = a.slots[a.cap + 1]; match[r] = e.cnt > 0; brow[r] = e.first; }
                else {
                    uint64_t s = j_hash_slot(key[r], mask);
                    while (true) {
                        int4 raw = __ldg(reinterpret_cast<const int4*>(a.slots + s));
                        long long k = ((long long)(unsigned int)raw.x) | ((long long)raw.y << 32);
                        if (k == key[r]) { match[r] = (unsigned int)raw.w > 0; brow[r] = (unsigned int)raw.z; break; }
                        if (k == J_EMPTY) break;
                        s = (s + 1) & mask;
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            unsigned m = __ballot_sync(0xffffffffu, match[r]);
            rank[r] = __popc(m & ((1u << lane) - 1));
            if (lane == 0) wcnt[r * NW + warp] = __popc(m);
        }
        __syncthreads();
        if (warp == 0) {  // exclusive scan of the 32 (row-slot, warp) counts, one cursor atomic for the tile
            unsigned int x = wcnt[lane], inc = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { unsigned int y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
            woff[lane] = inc - x;
            if (lane == 31) tile_base = inc ? atomicAdd(a.cursor, (unsigned long long)inc) : 0ull;
        }
        __syncthreads();
        const unsigned long long base = tile_base;
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (!match[r]) continue;
            const int64_t i = t * TILE + r * 256 + threadIdx.x;
            const int64_t orow = (int64_t)(base + woff[r * NW + warp] + rank[r]);
            const unsigned long long* fields = a.bpack + (size_t)brow[r] * a.n_fields;
            for (int k2 = 0; k2 < a.n_b; k2++) {
                int f = a.b_field[k2];
                unsigned long long v = f < 0 ? (unsigned long long)key[r] : __ldg(fields + f);
                store_sized(a.ob_data[k2], orow, v, a.b_size[k2]);
                if (a.ob_valid[k2]) a.ob_valid[k2][orow] = f < 0 ? (kvalid[r] ? 1 : 0) : (a.b_valid[k2] ? a.b_valid[k2][brow[r]] : 1);
            }
            for (int k2 = 0; k2 < a.n_p; k2++) {
                copy_item(a.op_data[k2], orow, a.p_data[k2], i, a.p_size[k2]);
                if (a.op_valid[k2]) a.op_valid[k2][orow] = bit_valid(a.p_valid[k2], i) ? 1 : 0;
            }
        }
        __syncthreads();
    }
}
// Fused probe for unique build tuples: join_probe_fast_kernel's tiles, cursor and ballot ranks over a Slot16 table whose key word is
// the tuple's tag.  The packed build row holds every build column, keys first, so the tuple check and the gather read one row.
struct FastProbeMkArgs {
    int64_t n_probe;
    JKeys pk;                                    // probe key columns (bitmaps)
    const uint8_t* bk_valid[J_MAX_KEYS];         // build key validity (one byte per row), nullptr = all valid
    unsigned long long bk_bits[J_MAX_KEYS];      // low-bit mask of each key's width: packed fields are zero-extended raw bits
    const Slot16* slots; uint64_t cap;
    const unsigned long long* bpack; int n_fields;
    unsigned long long* cursor;
    int n_b, n_p;
    int na_equal;
    int b_field[J_MAX_COLS];                     // kept build col -> packed field
    const uint8_t* b_valid[J_MAX_COLS]; int b_size[J_MAX_COLS];
    const void* p_data[J_MAX_COLS]; const uint8_t* p_valid[J_MAX_COLS]; int p_size[J_MAX_COLS];
    void* ob_data[J_MAX_COLS]; uint8_t* ob_valid[J_MAX_COLS];
    void* op_data[J_MAX_COLS]; uint8_t* op_valid[J_MAX_COLS];
};
// (the minimum-blocks hint only steers ptxas' allocation: without it the NK = 3 instance spills 16 bytes at 40 registers)
template <int NK>
__global__ void __launch_bounds__(256, 4) join_probe_fast_mk_kernel(const __grid_constant__ FastProbeMkArgs a) {
    constexpr int R = 4, NW = 8, TILE = 256 * R;
    __shared__ unsigned int wcnt[R * NW];
    __shared__ unsigned int woff[R * NW];
    __shared__ unsigned long long tile_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t mask = a.cap - 1;
    const int64_t n_tiles = (a.n_probe + TILE - 1) / TILE;
    for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        uint32_t brow[R];
        unsigned int rank[R];
        bool match[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int64_t i = t * TILE + r * 256 + threadIdx.x;
            match[r] = false; brow[r] = 0;
            long long keys[NK];
            const unsigned int na = i < a.n_probe ? j_load_tuple<NK, false>(a.pk, i, keys) : 0u;
            if (i < a.n_probe && (a.na_equal || na == (1u << NK) - 1u)) {
                const unsigned long long tag = mk_tag(keys, na, NK);
                uint64_t s = (tag >> 20) & mask;
                while (true) {
                    int4 raw = __ldg(reinterpret_cast<const int4*>(a.slots + s));
                    const unsigned long long k = (unsigned long long)(unsigned int)raw.x | ((unsigned long long)(unsigned int)raw.y << 32);
                    if (k == TAG_EMPTY) break;
                    if (k == tag) {
                        const uint32_t row = (unsigned int)raw.z;
                        const unsigned long long* fields = a.bpack + (size_t)row * a.n_fields;
                        bool eq = true;
#pragma unroll
                        for (int j = 0; j < NK; j++) {
                            const bool bv = a.bk_valid[j] == nullptr || a.bk_valid[j][row] != 0;
                            eq = eq && bv == (((na >> j) & 1u) != 0) && (!bv || __ldg(fields + j) == ((unsigned long long)keys[j] & a.bk_bits[j]));
                        }
                        if (eq) { match[r] = (unsigned int)raw.w > 0; brow[r] = row; break; }
                    }
                    s = (s + 1) & mask;
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            unsigned m = __ballot_sync(0xffffffffu, match[r]);
            rank[r] = __popc(m & ((1u << lane) - 1));
            if (lane == 0) wcnt[r * NW + warp] = __popc(m);
        }
        __syncthreads();
        if (warp == 0) {
            unsigned int x = wcnt[lane], inc = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { unsigned int y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
            woff[lane] = inc - x;
            if (lane == 31) tile_base = inc ? atomicAdd(a.cursor, (unsigned long long)inc) : 0ull;
        }
        __syncthreads();
        const unsigned long long base = tile_base;
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (!match[r]) continue;
            const int64_t i = t * TILE + r * 256 + threadIdx.x;
            const int64_t orow = (int64_t)(base + woff[r * NW + warp] + rank[r]);
            const unsigned long long* fields = a.bpack + (size_t)brow[r] * a.n_fields;
            for (int k2 = 0; k2 < a.n_b; k2++) {
                store_sized(a.ob_data[k2], orow, __ldg(fields + a.b_field[k2]), a.b_size[k2]);
                if (a.ob_valid[k2]) a.ob_valid[k2][orow] = a.b_valid[k2] ? a.b_valid[k2][brow[r]] : 1;
            }
            for (int k2 = 0; k2 < a.n_p; k2++) {
                copy_item(a.op_data[k2], orow, a.p_data[k2], i, a.p_size[k2]);
                if (a.op_valid[k2]) a.op_valid[k2][orow] = bit_valid(a.p_valid[k2], i) ? 1 : 0;
            }
        }
        __syncthreads();
    }
}

// ---- inline-payload probe: the specialisation for all-8-byte, bitmap-free schemas with at most two build payload columns ----
// Slot32 = {key, f0, f1, first | cnt << 32}: key AND payload of a unique-key build row sit in ONE 32-byte sector, so a probe
// row costs one random sector instead of two (Slot16 + packed payload row).  All coalesced loads of a tile (key and the kept
// probe columns, 4 rows per thread) are issued before the first dependent table access.
struct __align__(32) Slot32 { long long key; unsigned long long f0, f1; uint32_t first; uint32_t cnt; };
constexpr int J_INL_MAX_P = 4;
struct InlineProbeArgs {
    int64_t n_probe;
    const long long* key;
    const Slot32* slots; uint64_t cap;
    unsigned long long* cursor;
    int n_b;                       // kept build columns (<= 3)
    int b_field[4];                // -1 = key, 0 / 1 = payload field
    unsigned long long* ob[4];
    const unsigned long long* p[J_INL_MAX_P];  // kept probe columns (the key column included when kept)
    unsigned long long* op[J_INL_MAX_P];
};
// Direct build of the Slot32 table (no separate key table / slot-info / CSR passes): one random 32-byte sector per build row.
// A row claims its slot with a CAS on the key word, counts itself in the slot and, when it is the first row of that key,
// writes the payload.  A second row of any key raises *dup: the host then falls back to the general build (CSR groups).
__global__ void join_fill_slots32_kernel(Slot32* slots, uint64_t n_slots) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const ulonglong4 e = make_ulonglong4((unsigned long long)J_EMPTY, 0ull, 0ull, 0ull);
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < n_slots; s += stride) reinterpret_cast<ulonglong4*>(slots)[s] = e;
}
__global__ void __launch_bounds__(256) join_build_inline_kernel(const long long* __restrict__ keys, const unsigned long long* __restrict__ f0, const unsigned long long* __restrict__ f1,
                                                                int64_t n, int64_t row0, Slot32* slots, uint64_t cap, int* dup) {
    constexpr int R = 4;
    const uint64_t mask = cap - 1;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * R;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x * R + threadIdx.x; i0 < n; i0 += stride) {
        long long key[R], k0[R];
        uint64_t s[R];
#pragma unroll
        for (int r = 0; r < R; r++) { const int64_t i = i0 + r * 256; key[r] = i < n ? __ldcs(keys + i) : 0; }
#pragma unroll
        for (int r = 0; r < R; r++) {  // the R first probes are in flight together
            s[r] = key[r] == J_EMPTY ? cap + 1 : j_hash_slot(key[r], mask);
            k0[r] = __ldcg(&slots[s[r]].key);
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int64_t i = i0 + r * 256;
            if (i >= n) continue;
            bool won = false;  // this row claimed a free slot (it is the first row of its key)
            if (key[r] != J_EMPTY) {
                long long k = k0[r];
                while (true) {
                    if (k == J_EMPTY) {
                        const long long prev = (long long)atomicCAS((unsigned long long*)&slots[s[r]].key, (unsigned long long)J_EMPTY, (unsigned long long)key[r]);
                        if (prev == J_EMPTY) { won = true; break; }
                        k = prev;
                    }
                    if (k == key[r]) break;  // another row holds this key: duplicate
                    s[r] = (s[r] + 1) & mask;
                    k = __ldcg(&slots[s[r]].key);
                }
            } else {
                won = atomicAdd(&slots[s[r]].cnt, 1u) == 0;  // marker-key slot: its key word stays the free-slot pattern
            }
            if (won) {  // the rest of the sector: f0 (8 B), then {f1, first, cnt = 1} (16 B)
                slots[s[r]].f0 = f0 ? __ldcs(f0 + i) : 0ull;
                const unsigned long long f1v = f1 ? __ldcs(f1 + i) : 0ull;
                *reinterpret_cast<ulonglong2*>(&slots[s[r]].f1) = make_ulonglong2(f1v, (unsigned long long)(uint32_t)(row0 + i) | (1ull << 32));
            } else *dup = 1;
        }
    }
}
__global__ void join_slots16_from32_kernel(const Slot32* in, uint64_t n_slots, Slot16* out) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < n_slots; s += stride) {
        Slot16 e; e.key = in[s].key; e.first = in[s].first; e.cnt = in[s].cnt;
        out[s] = e;
    }
}
template <int NF, int NPK>
__global__ void __launch_bounds__(256) join_probe_inline_kernel(const __grid_constant__ InlineProbeArgs a) {
    constexpr int R = 4, NW = 8, TILE = 256 * R;
    __shared__ unsigned int wcnt[R * NW];
    __shared__ unsigned int woff[R * NW];
    __shared__ unsigned long long tile_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t mask = a.cap - 1;
    const int64_t n_tiles = (a.n_probe + TILE - 1) / TILE;
    for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        long long key[R];
        unsigned long long pv[NPK][R], f0[R], f1[R];
        unsigned int rank[R];
        bool match[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int64_t i = t * TILE + r * 256 + threadIdx.x;
            const bool in = i < a.n_probe;
            key[r] = in ? __ldcs(a.key + i) : 0;
#pragma unroll
            for (int c = 0; c < NPK; c++) pv[c][r] = in ? __ldcs(a.p[c] + i) : 0ull;
        }
        // first probe of all R rows: the R random 256-bit slot loads (one sector, one request each) are in flight together;
        // a data-dependent probe loop per row would serialise them
        uint64_t sl[R];
        unsigned long long w0[R], w1[R], w2[R], w3[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            sl[r] = key[r] == J_EMPTY ? a.cap + 1 : j_hash_slot(key[r], mask);
            asm volatile("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(w0[r]), "=l"(w1[r]), "=l"(w2[r]), "=l"(w3[r]) : "l"(a.slots + sl[r]));
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int64_t i = t * TILE + r * 256 + threadIdx.x;
            match[r] = false; f0[r] = 0; f1[r] = 0;
            if (i >= a.n_probe) continue;
            while (true) {
                if ((long long)w0[r] == key[r]) {
                    if (NF >= 1) f0[r] = w1[r];
                    if (NF >= 2) f1[r] = w2[r];
                    match[r] = (unsigned int)(w3[r] >> 32) > 0;
                    break;
                }
                if ((long long)w0[r] == J_EMPTY || sl[r] > mask) break;  // free slot, or the marker-key slot (cap + 1) without a build row
                sl[r] = (sl[r] + 1) & mask;  // collision (about one row in four at this load factor): next slot
                asm volatile("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(w0[r]), "=l"(w1[r]), "=l"(w2[r]), "=l"(w3[r]) : "l"(a.slots + sl[r]));
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            unsigned m = __ballot_sync(0xffffffffu, match[r]);
            rank[r] = __popc(m & ((1u << lane) - 1));
            if (lane == 0) wcnt[r * NW + warp] = __popc(m);
        }
        __syncthreads();
        if (warp == 0) {
            unsigned int x = wcnt[lane], inc = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { unsigned int y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
            woff[lane] = inc - x;
            if (lane == 31) tile_base = inc ? atomicAdd(a.cursor, (unsigned long long)inc) : 0ull;
        }
        __syncthreads();
        const unsigned long long base = tile_base;
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (!match[r]) continue;
            const int64_t orow = (int64_t)(base + woff[r * NW + warp] + rank[r]);
            for (int k2 = 0; k2 < a.n_b; k2++) {
                const int f = a.b_field[k2];
                a.ob[k2][orow] = f < 0 ? (unsigned long long)key[r] : (f == 0 ? f0[r] : f1[r]);
            }
#pragma unroll
            for (int c = 0; c < NPK; c++) a.op[c][orow] = pv[c][r];
        }
        __syncthreads();
    }
}

// ---- runtime join filter (reference: HashJoinState::RuntimeFilter, bodo/libs/streaming/_join.h:1060-1095; bloom filter
// bodo/libs/gpu_bloom_filter.cu:60-201; key min / max bodo/libs/streaming/_join.cpp:3199-3238) ----
// Split-block bloom filter: a key selects one 32-byte block (one sector) with the high hash word and sets / tests one bit in each
// of its eight 32-bit words (eight odd multipliers of the low hash word, the Parquet / Impala scheme).  ~8 bits per build key.
__device__ __forceinline__ void bloom_masks(uint32_t h, uint32_t (&m)[8]) {
    const uint32_t salt[8] = {0x47b6137bu, 0x44974d91u, 0x8824ad5bu, 0xa2b7289du, 0x705495c7u, 0x2df1424bu, 0x9efc4947u, 0x5c6bfb31u};
#pragma unroll
    for (int j = 0; j < 8; j++) m[j] = 1u << ((h * salt[j]) >> 27);
}
__global__ void join_bloom_add_kernel(const void* key_data, int key_ctype, const uint8_t* key_valid_bytes, int64_t n, uint32_t* bloom, uint64_t n_blocks,
                                      long long* minmax) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    long long mn = INT64_MAX, mx = INT64_MIN;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        if (key_valid_bytes && !key_valid_bytes[i]) continue;
        const long long key = load_int_as_i64(key_data, key_ctype, i);
        mn = key < mn ? key : mn; mx = key > mx ? key : mx;
        const uint64_t h = xxh3_64_short((uint64_t)key, 8, SEED_HASH_JOIN);
        uint32_t m[8];
        bloom_masks((uint32_t)h, m);
        uint32_t* blk = bloom + (size_t)(__umul64hi(h, n_blocks)) * 8;
#pragma unroll
        for (int j = 0; j < 8; j++) atomicOr(blk + j, m[j]);
    }
    for (int d = 16; d; d >>= 1) {
        const long long a = __shfl_xor_sync(0xffffffffu, mn, d), b = __shfl_xor_sync(0xffffffffu, mx, d);
        mn = a < mn ? a : mn; mx = b > mx ? b : mx;
    }
    if ((threadIdx.x & 31) == 0 && mn <= mx) { atomicMin(minmax, mn); atomicMax(minmax + 1, mx); }
}
// keep[i] = 1 iff row i can still find a partner: key not NA, inside [min, max] of the build keys, bloom hit
__global__ void join_runtime_filter_kernel(const void* key_data, int key_ctype, const uint8_t* key_valid, int64_t n, const uint32_t* bloom, uint64_t n_blocks,
                                           long long mn, long long mx, int use_minmax, int use_bloom, uint8_t* keep) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        bool k = bit_valid(key_valid, i);
        if (k) {
            const long long key = load_int_as_i64(key_data, key_ctype, i);
            if (use_minmax && (key < mn || key > mx)) k = false;
            if (k && use_bloom) {
                const uint64_t h = xxh3_64_short((uint64_t)key, 8, SEED_HASH_JOIN);
                uint32_t m[8];
                bloom_masks((uint32_t)h, m);
                const uint4* blk = reinterpret_cast<const uint4*>(bloom + (size_t)(__umul64hi(h, n_blocks)) * 8);
                const uint4 lo = __ldg(blk), hi = __ldg(blk + 1);
                k = (lo.x & m[0]) && (lo.y & m[1]) && (lo.z & m[2]) && (lo.w & m[3]) && (hi.x & m[4]) && (hi.y & m[5]) && (hi.z & m[6]) && (hi.w & m[7]);
            }
        }
        keep[i] = k ? 1 : 0;
    }
}

// ================================================================================================
struct GrowCol {  // growable device column (geometric growth, copy on grow)
    DevBuf buf;
    size_t used = 0;
    void append(const void* src, size_t nbytes, bool src_is_host, cudaStream_t st) {
        if (used + nbytes > buf.bytes) {
            DevBuf nb;
            nb.alloc(std::max<size_t>((used + nbytes) * 2, 1 << 16));
            if (used) B200_CUDA(cudaMemcpyAsync(nb.p, buf.p, used, cudaMemcpyDeviceToDevice, st));
            B200_CUDA(cudaStreamSynchronize(st));
            buf = std::move(nb);
        }
        if (nbytes) B200_CUDA(cudaMemcpyAsync((char*)buf.p + used, src, nbytes, src_is_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, st));
        used += nbytes;
    }
    void reserve(size_t n) { if (n > buf.bytes) { B200_REQUIRE(used == 0, "internal: reserve after append"); buf.alloc(n); } }
};

class JoinState {
   public:
    int device; cudaStream_t stream; int sms;
    std::vector<int8_t> b_ct, b_at, p_ct, p_at;
    int n_b, n_p;
    int nk = 1;  // key columns: the first nk columns of each side
    bool build_outer, probe_outer;
    bool na_equal = false;  // is_na_equal of the reference's HashJoinState
    int64_t output_batch_size;
    // build side
    std::vector<GrowCol> bcol, bvalid;  // data; validity as one byte per row (empty when the column has none so far)
    std::vector<bool> b_has_valid;
    int64_t n_build = 0;
    bool build_final = false;
    uint64_t cap = 0;
    DevBuf d_tkeys, d_info, d_row_slot, d_cnt_multi, d_goffs, d_groups, d_fill, d_bmatched;  // d_tkeys: keys, or tuple tags (nk > 1)
    DevBuf d_slots16, d_bpack, d_cursor;  // fast path (unique build keys, inner join)
    DevBuf d_slots32;                      // inline-payload table (all-8-byte bitmap-free build schema, <= 2 payload columns)
    bool fast_ready = false, inline_ready = false;
    int64_t inline_probes = 0, inline_builds = 0;
    // join kind (set_kind, before the first build batch): mark join / probe-side anti join (reference: is_mark_join member,
    // is_anti_join template argument of the probe)
    bool mark = false, anti = false;
    DevBuf d_mark, d_mark_valid;
    // runtime join filter, built on demand from the build keys
    DevBuf d_bloom, d_minmax;
    uint64_t bloom_blocks = 0;
    long long key_min = INT64_MAX, key_max = INT64_MIN;
    int64_t filter_rows_in = 0, filter_rows_kept = 0;
    unsigned long long* h_cursor = nullptr;
    int64_t fast_probes = 0;
    Scanner scan;
    // probe scratch + output
    DevBuf d_pslot, d_pcnt, d_poff, d_stage_valid;
    std::vector<DevBuf> stage_data, stage_valid;   // device copies of host probe batches
    std::vector<DevBuf> out_data, out_vbytes, out_bitmap;
    int64_t launches = 0, probe_rows = 0, out_rows_total = 0;
    bool tail_emitted = false;

    JoinState(const int8_t* bct, const int8_t* bat, int nb, const int8_t* pct, const int8_t* pat, int np, uint64_t n_keys,
              bool bo, bool po, bool na_eq, int64_t obs, int dev, int64_t expected_build_rows, cudaStream_t st)
        : device(dev), stream(st), n_b(nb), n_p(0), build_outer(bo), probe_outer(po), na_equal(na_eq), output_batch_size(obs) {
        B200_REQUIRE(n_keys >= 1 && n_keys <= (uint64_t)J_MAX_KEYS, "b200 join: between 1 and 4 key columns are supported");
        nk = (int)n_keys;
        B200_REQUIRE(nb >= 1 && np >= 0 && nb <= J_MAX_COLS && np <= J_MAX_COLS, "b200 join: between 1 and 32 columns per side");
        B200_REQUIRE(nb >= nk, "b200 join: the build table has fewer columns than key columns");
        b_ct.assign(bct, bct + nb); b_at.assign(bat, bat + nb);
        for (int c = 0; c < nb; c++) B200_REQUIRE(ctype_size(b_ct[c]) > 0, "b200 join: unsupported build column dtype");
        for (int j = 0; j < nk; j++) B200_REQUIRE(!ctype_is_float(b_ct[j]), "b200 join: key columns must be integer/date typed");
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        sms = num_sms(device);
        bcol.resize(nb); bvalid.resize(nb); b_has_valid.assign(nb, false);
        if (expected_build_rows > 0)
            for (int c = 0; c < nb; c++) bcol[c].reserve((size_t)expected_build_rows * ctype_size(b_ct[c]));
        stage_data.resize(nb); stage_valid.resize(nb);
        if (np > 0) set_probe_schema(pct, pat, np);
    }
    // The probe schema may be given at init (n_probe_arrs > 0) or adopted from the first probe batch (n_probe_arrs == 0), so
    // a host layer that only learns it from the data can feed build batches straight away.
    void set_probe_schema(const int8_t* pct, const int8_t* pat, int np) {
        B200_REQUIRE(np >= 1 && np <= J_MAX_COLS, "b200 join: between 1 and 32 columns per side");
        p_ct.assign(pct, pct + np); p_at.assign(pat, pat + np); n_p = np;
        for (int c = 0; c < np; c++) B200_REQUIRE(ctype_size(p_ct[c]) > 0, "b200 join: unsupported probe column dtype");
        B200_REQUIRE(np >= nk, "b200 join: the probe table has fewer columns than key columns");
        for (int j = 0; j < nk; j++) {
            // sharded placement hashes each key's sizeof(T) raw bytes, so both sides must agree on the width at every position
            B200_REQUIRE(!ctype_is_float(p_ct[j]), "b200 join: key columns must be integer/date typed");
            B200_REQUIRE(ctype_size(b_ct[j]) == ctype_size(p_ct[j]),
                         nk == 1 ? std::string("b200 join: build and probe key widths differ")
                                 : "b200 join: build and probe key widths differ at key position " + std::to_string(j));
        }
        out_data.resize(n_b + np); out_vbytes.resize(n_b + np); out_bitmap.resize(n_b + np);
        if ((int)stage_data.size() < std::max(n_b, np)) { stage_data.resize(std::max(n_b, np)); stage_valid.resize(std::max(n_b, np)); }
    }
    ~JoinState() { cudaSetDevice(device); scratch_set_stream(stream); cudaStreamSynchronize(stream); pinned_release(h_cursor, 8); }

    int grid_for(int64_t n) const { return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)sms * 8)); }

    // multi-key kernels are instantiated per key count; f(std::integral_constant<int, NK>) launches one
    template <typename F> void with_nk(F&& f) const {
        switch (nk) {
            case 2: f(std::integral_constant<int, 2>()); break;
            case 3: f(std::integral_constant<int, 3>()); break;
            default: f(std::integral_constant<int, 4>()); break;
        }
    }
    JKeys build_keys() const {
        JKeys k{};
        for (int j = 0; j < nk; j++) { k.data[j] = bcol[j].buf.p; k.valid[j] = b_has_valid[j] ? bvalid[j].buf.as<uint8_t>() : nullptr; k.ctype[j] = b_ct[j]; }
        return k;
    }
    JKeys probe_keys(const std::vector<const void*>& data, const std::vector<const uint8_t*>& valid) const {
        JKeys k{};
        for (int j = 0; j < nk; j++) { k.data[j] = data[j]; k.valid[j] = valid[j]; k.ctype[j] = p_ct[j]; }
        return k;
    }

    void set_kind(bool is_mark, bool is_anti) {
        B200_REQUIRE(n_build == 0 && !build_final, "b200 join: the join kind must be set before the first build batch");
        B200_REQUIRE(!(is_mark && is_anti), "b200 join: a join is a mark join or an anti join, not both");
        B200_REQUIRE(!(is_mark || is_anti) || !build_outer, "b200 join: mark / anti joins do not emit build rows (build_table_outer must be false)");
        mark = is_mark; anti = is_anti;
    }

    // ---- runtime join filter ----
    // n_blocks: 32-byte bloom blocks (0 = one per 32 build rows, ~8 bits per key); ranks that will OR their filters together
    // pass the same value.  Also computes the min / max of the (non-NA) build keys.
    void require_single_key_filter() const {
        B200_REQUIRE(nk == 1, "b200 join: the runtime join filter is built for single-column join keys only (this state joins on " + std::to_string(nk) + " key columns)");
    }
    void build_filter(uint64_t n_blocks) {
        require_single_key_filter();
        B200_REQUIRE(build_final, "b200 join: runtime filter before the build side was finished");
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        bloom_blocks = n_blocks ? n_blocks : (uint64_t)n_build / 32 + 1;
        d_bloom.alloc(bloom_blocks * 32);
        B200_CUDA(cudaMemsetAsync(d_bloom.p, 0, bloom_blocks * 32, stream));
        d_minmax.alloc(16);
        const long long init[2] = {INT64_MAX, INT64_MIN};
        B200_CUDA(cudaMemcpyAsync(d_minmax.p, init, 16, cudaMemcpyHostToDevice, stream));
        if (n_build > 0) {
            join_bloom_add_kernel<<<grid_for(n_build), 256, 0, stream>>>(bcol[0].buf.p, b_ct[0], b_has_valid[0] ? bvalid[0].buf.as<uint8_t>() : nullptr, n_build,
                                                                        d_bloom.as<uint32_t>(), bloom_blocks, d_minmax.as<long long>());
            launches++;
            B200_CUDA(cudaGetLastError());
        }
        long long h[2];
        B200_CUDA(cudaMemcpyAsync(h, d_minmax.p, 16, cudaMemcpyDeviceToHost, stream));
        B200_CUDA(cudaStreamSynchronize(stream));
        key_min = h[0]; key_max = h[1];
    }
    void runtime_filter(const b200_table* t, int key_col, bool use_minmax, bool use_bloom, uint8_t* keep) {
        require_single_key_filter();
        B200_REQUIRE(t->device == device, "b200 join: runtime_filter takes a device-resident table on the state's device");
        B200_REQUIRE(key_col >= 0 && key_col < t->n_cols, "b200 join: runtime_filter: bad key column");
        B200_REQUIRE(ctype_size(t->cols[key_col].c_type) == ctype_size(b_ct[0]) && !ctype_is_float(t->cols[key_col].c_type), "b200 join: runtime_filter: key column type differs from the build key");
        if (!d_bloom.p) build_filter(0);
        B200_CUDA(cudaSetDevice(device));
        const int64_t n = t->n_rows;
        if (n == 0) return;
        join_runtime_filter_kernel<<<grid_for(n), 256, 0, stream>>>(t->cols[key_col].data, t->cols[key_col].c_type, t->cols[key_col].validity, n, d_bloom.as<uint32_t>(),
                                                                   bloom_blocks, key_min, key_max, use_minmax ? 1 : 0, use_bloom ? 1 : 0, keep);
        launches++;
        B200_CUDA(cudaGetLastError());
        filter_rows_in += n;
    }

    // device pointers for a batch (host batches are staged to the device first)
    void stage_batch(const b200_table* t, int ncols, const std::vector<int8_t>& cts, std::vector<const void*>& data,
                     std::vector<const uint8_t*>& valid) {
        data.assign(ncols, nullptr); valid.assign(ncols, nullptr);
        int64_t n = t->n_rows;
        for (int c = 0; c < ncols; c++) {
            B200_REQUIRE(t->cols[c].c_type == cts[c], "b200 join: batch column dtype differs from the schema");
            if (t->device >= 0) {
                B200_REQUIRE(t->device == device, "b200 join: batch lives on another device");
                data[c] = t->cols[c].data; valid[c] = t->cols[c].validity;
            } else {
                size_t nbytes = (size_t)n * ctype_size(cts[c]);
                stage_data[c].ensure(nbytes + 8);
                if (nbytes) B200_CUDA(cudaMemcpyAsync(stage_data[c].p, t->cols[c].data, nbytes, cudaMemcpyHostToDevice, stream));
                data[c] = stage_data[c].p;
                if (t->cols[c].validity) {
                    stage_valid[c].ensure((size_t)(n + 7) / 8 + 8);
                    B200_CUDA(cudaMemcpyAsync(stage_valid[c].p, t->cols[c].validity, (size_t)(n + 7) / 8, cudaMemcpyHostToDevice, stream));
                    valid[c] = stage_valid[c].as<uint8_t>();
                }
            }
        }
    }

    void build_consume(const b200_table* t, bool is_last) {
        B200_REQUIRE(!build_final, "b200 join: build batch after the build was finalized");
        B200_REQUIRE(t->n_cols == n_b, "b200 join: build batch has a different number of columns than the schema");
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        int64_t n = t->n_rows;
        // slot ids and build row ids are 32-bit; cap = next power of two >= 2 * n_build, and cap + 2 must stay below 2^32
        B200_REQUIRE(n_build + n <= (1ll << 30), "b200 join: build side is limited to 2^30 rows per GPU");
        if (n > 0) {
            std::vector<const void*> data; std::vector<const uint8_t*> valid;
            stage_batch(t, n_b, b_ct, data, valid);
            for (int c = 0; c < n_b; c++) {
                bcol[c].append(data[c], (size_t)n * ctype_size(b_ct[c]), false, stream);
                bool has = valid[c] != nullptr;
                if (has && !b_has_valid[c]) {  // first batch with a bitmap: earlier rows were all valid
                    b_has_valid[c] = true;
                    if (n_build) { DevBuf ones; ones.alloc((size_t)n_build); B200_CUDA(cudaMemsetAsync(ones.p, 1, (size_t)n_build, stream)); bvalid[c].append(ones.p, (size_t)n_build, false, stream); B200_CUDA(cudaStreamSynchronize(stream)); }
                }
                if (b_has_valid[c]) {
                    d_stage_valid.ensure((size_t)n);
                    if (has) { expand_bitmap_kernel<<<grid_for(n), 256, 0, stream>>>(valid[c], n, d_stage_valid.as<uint8_t>()); launches++; }
                    else B200_CUDA(cudaMemsetAsync(d_stage_valid.p, 1, (size_t)n, stream));
                    bvalid[c].append(d_stage_valid.p, (size_t)n, false, stream);
                }
            }
            B200_CUDA(cudaStreamSynchronize(stream));  // staging buffers are reused by the next batch
            n_build += n;
        }
        if (is_last) finalize_build();
    }

    // Inline-payload build attempt (unique keys expected): true when the Slot32 table is complete, false when a key repeats
    // (or the schema does not qualify: multi-column keys never do) and the general build has to run.
    bool try_inline_build(uint64_t n_slots) {
        const int nf = n_b - 1;
        bool ok = nk == 1 && n_build > 0 && nf <= 2 && !build_outer && !probe_outer && !(getenv("B200_JOIN_INLINE") && getenv("B200_JOIN_INLINE")[0] == '0');
        for (int c = 0; c < n_b; c++) ok = ok && ctype_size(b_ct[c]) == 8 && !b_has_valid[c];
        if (!ok) return false;
        d_slots32.alloc(n_slots * sizeof(Slot32));
        d_cursor.alloc(8);
        B200_CUDA(cudaMemsetAsync(d_cursor.p, 0, 8, stream));
        join_fill_slots32_kernel<<<grid_for((int64_t)n_slots), 256, 0, stream>>>(d_slots32.as<Slot32>(), n_slots);
        join_build_inline_kernel<<<(int)std::max<int64_t>(1, std::min<int64_t>((n_build + 1023) / 1024, (int64_t)sms * 8)), 256, 0, stream>>>(bcol[0].buf.as<long long>(), nf > 0 ? bcol[1].buf.as<unsigned long long>() : nullptr,
                                                                       nf > 1 ? bcol[2].buf.as<unsigned long long>() : nullptr, n_build, 0, d_slots32.as<Slot32>(), cap,
                                                                       (int*)d_cursor.p);
        launches += 2;
        B200_CUDA(cudaGetLastError());
        if (!h_cursor) h_cursor = (unsigned long long*)pinned_acquire(8);
        B200_CUDA(cudaMemcpyAsync(h_cursor, d_cursor.p, 8, cudaMemcpyDeviceToHost, stream));
        B200_CUDA(cudaStreamSynchronize(stream));
        if (*h_cursor != 0) { d_slots32.release(); return false; }  // duplicate build keys
        return true;
    }
    // Slot16 table + packed payload of the two-sector fast kernel, derived on demand when a probe batch does not qualify for the
    // inline kernel (bitmaps, narrow columns) after an inline build
    void ensure_fast_tables() {
        if (d_slots16.p) return;
        const uint64_t n_slots = cap + 2;
        d_slots16.alloc(n_slots * sizeof(Slot16));
        join_slots16_from32_kernel<<<grid_for((int64_t)n_slots), 256, 0, stream>>>(d_slots32.as<Slot32>(), n_slots, d_slots16.as<Slot16>());
        const int nf = n_b - 1;
        d_bpack.alloc((size_t)std::max<int64_t>(n_build * std::max(nf, 1), 1) * 8);
        if (nf > 0) {
            PackPayloadArgs pa{};
            pa.n_build = n_build; pa.n_fields = nf; pa.out = d_bpack.as<unsigned long long>();
            for (int c = 1; c < n_b; c++) { pa.src[c - 1] = bcol[c].buf.p; pa.size[c - 1] = ctype_size(b_ct[c]); }
            join_pack_payload_kernel<<<grid_for(n_build), 256, 0, stream>>>(pa);
        }
        launches += 2;
        B200_CUDA(cudaGetLastError());
    }

    void finalize_build() {
        cap = 1024;
        while (cap < 2ull * (uint64_t)n_build) cap <<= 1;
        uint64_t n_slots = cap + 2;
        if (!mark && !anti && try_inline_build(n_slots)) {
            d_goffs.alloc(8); d_groups.alloc(8);
            fast_ready = true; inline_ready = true; inline_builds++;
            build_final = true;
            return;
        }
        d_tkeys.alloc(n_slots * 8);
        if (nk == 1) fill_i64_kernel<<<grid_for((int64_t)n_slots), 256, 0, stream>>>(d_tkeys.as<long long>(), n_slots, J_EMPTY);
        else B200_CUDA(cudaMemsetAsync(d_tkeys.p, 0, n_slots * 8, stream));  // every tag TAG_EMPTY
        d_info.alloc(n_slots * sizeof(SlotInfo));
        B200_CUDA(cudaMemsetAsync(d_info.p, 0, n_slots * sizeof(SlotInfo), stream));
        d_row_slot.alloc((size_t)std::max<int64_t>(n_build, 1) * 4);
        if (nk == 1) launches++;
        if (n_build > 0) {
            if (nk == 1)
                join_insert_count_kernel<<<grid_for(n_build), 256, 0, stream>>>(bcol[0].buf.p, b_ct[0], b_has_valid[0] ? bvalid[0].buf.as<uint8_t>() : nullptr,
                                                                               n_build, d_tkeys.as<long long>(), cap, d_info.as<SlotInfo>(), d_row_slot.as<uint32_t>(), na_equal ? 1 : 0);
            else
                with_nk([&](auto k) {
                    join_insert_count_mk_kernel<decltype(k)::value><<<grid_for(n_build), 256, 0, stream>>>(build_keys(), n_build, d_tkeys.as<unsigned long long>(), cap,
                                                                                                           d_info.as<SlotInfo>(), d_row_slot.as<uint32_t>(), na_equal ? 1 : 0);
                });
            d_cnt_multi.alloc(n_slots * 4);
            join_slot_counts_kernel<<<grid_for((int64_t)n_slots), 256, 0, stream>>>(d_info.as<SlotInfo>(), n_slots, d_cnt_multi.as<uint32_t>());
            launches += 2;
            d_goffs.alloc((n_slots + 1) * 8);
            unsigned long long n_multi = scan.run(d_cnt_multi.as<uint32_t>(), (int64_t)n_slots, d_goffs.as<unsigned long long>(), stream, &launches);
            d_groups.alloc((size_t)std::max<unsigned long long>(n_multi, 1) * 4);
            if (n_multi > 0) {
                d_fill.alloc(n_slots * 4);
                B200_CUDA(cudaMemsetAsync(d_fill.p, 0, n_slots * 4, stream));
                join_fill_groups_kernel<<<grid_for(n_build), 256, 0, stream>>>(d_row_slot.as<uint32_t>(), n_build, d_info.as<SlotInfo>(), d_goffs.as<unsigned long long>(),
                                                                              d_fill.as<uint32_t>(), d_groups.as<uint32_t>());
                launches++;
            }
            d_cnt_multi.release(); d_fill.release(); d_row_slot.release();
            if (n_multi == 0 && !build_outer && !probe_outer && !mark && !anti && n_b >= 1) {
                // every key (incl. the NA / marker groups) has exactly one build row: set up the fused probe path.  Single key: Slot16.key
                // is the key and the packed rows hold the non-key columns; multi-key: Slot16.key is the tuple's tag and the packed rows
                // hold every column (the tuple check reads the keys from there)
                d_slots16.alloc(n_slots * sizeof(Slot16));
                join_make_slots16_kernel<<<grid_for((int64_t)n_slots), 256, 0, stream>>>(d_tkeys.as<long long>(), d_info.as<SlotInfo>(), n_slots, d_slots16.as<Slot16>());
                const int c0 = nk == 1 ? 1 : 0;
                int nf = n_b - c0;
                d_bpack.alloc((size_t)std::max<int64_t>(n_build * std::max(nf, 1), 1) * 8);
                if (nf > 0) {
                    PackPayloadArgs pa{};
                    pa.n_build = n_build; pa.n_fields = nf; pa.out = d_bpack.as<unsigned long long>();
                    for (int c = c0; c < n_b; c++) { pa.src[c - c0] = bcol[c].buf.p; pa.size[c - c0] = ctype_size(b_ct[c]); }
                    join_pack_payload_kernel<<<grid_for(n_build), 256, 0, stream>>>(pa);
                }
                d_cursor.alloc(8);
                if (!h_cursor) h_cursor = (unsigned long long*)pinned_acquire(8);
                launches += 2;
                fast_ready = true;
                d_tkeys.release(); d_info.release();  // the general-path table is not needed any more
            }
        } else {
            d_goffs.alloc(8); d_groups.alloc(8);
        }
        if (build_outer) { d_bmatched.alloc((size_t)std::max<int64_t>(n_build, 1)); B200_CUDA(cudaMemsetAsync(d_bmatched.p, 0, (size_t)std::max<int64_t>(n_build, 1), stream)); }
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaStreamSynchronize(stream));
        build_final = true;
    }

    // describes output column k (0..n_kb-1 build, then probe) in `out`
    void describe_out(b200_table* out, const std::vector<int>& kb, const std::vector<int>& kp, int64_t rows) {
        out->n_rows = rows; out->n_cols = (int)(kb.size() + kp.size()); out->device = device;
        for (size_t k = 0; k < kb.size() + kp.size(); k++) {
            bool is_b = k < kb.size();
            int src = is_b ? kb[k] : kp[k - kb.size()];
            b200_column& c = out->cols[k];
            c.data = out_data[k].p; c.length = rows;
            c.c_type = is_b ? b_ct[src] : p_ct[src];
            bool nullable = out_vbytes[k].p != nullptr && out_has_valid[k];
            c.validity = nullable ? out_bitmap[k].as<uint8_t>() : nullptr;
            c.arr_type = nullable ? ARR_NULLABLE : (is_b ? b_at[src] : p_at[src]);
        }
    }
    std::vector<bool> out_has_valid;

    int64_t probe_fast(const b200_table* t, const std::vector<int>& kb, const std::vector<int>& kp, const std::vector<const void*>& data,
                       const std::vector<const uint8_t*>& valid, b200_table* out) {
        int64_t n = t->n_rows;
        int n_out_cols = (int)(kb.size() + kp.size());
        out_has_valid.assign(n_out_cols, false);
        for (int k = 0; k < n_out_cols; k++) {
            bool is_b = k < (int)kb.size();
            int src = is_b ? kb[k] : kp[k - kb.size()];
            out_has_valid[k] = is_b ? (src == 0 && nk == 1 ? (valid[0] != nullptr || b_at[0] == ARR_NULLABLE) : (b_has_valid[src] || b_at[src] == ARR_NULLABLE))
                                    : (valid[src] != nullptr || p_at[src] == ARR_NULLABLE);
            out_data[k].ensure((size_t)(n + 32) * ctype_size(is_b ? b_ct[src] : p_ct[src]));  // matches <= probe rows
            if (out_has_valid[k]) { out_vbytes[k].ensure((size_t)n + 32); out_bitmap[k].ensure((size_t)((n + 31) / 32 + 1) * 4); }
        }
        int64_t rows = 0;
        if (n > 0 && nk > 1) {
            FastProbeMkArgs f{};
            f.n_probe = n; f.pk = probe_keys(data, valid);
            for (int j = 0; j < nk; j++) {
                f.bk_valid[j] = b_has_valid[j] ? bvalid[j].buf.as<uint8_t>() : nullptr;
                f.bk_bits[j] = ctype_size(b_ct[j]) == 8 ? ~0ull : (1ull << (8 * ctype_size(b_ct[j]))) - 1;
            }
            f.slots = d_slots16.as<Slot16>(); f.cap = cap; f.bpack = d_bpack.as<unsigned long long>(); f.n_fields = n_b;
            f.cursor = d_cursor.as<unsigned long long>(); f.n_b = (int)kb.size(); f.n_p = (int)kp.size(); f.na_equal = na_equal ? 1 : 0;
            for (int k = 0; k < n_out_cols; k++) {
                bool is_b = k < (int)kb.size();
                int src = is_b ? kb[k] : kp[k - kb.size()];
                if (is_b) {
                    f.b_field[k] = src; f.b_size[k] = ctype_size(b_ct[src]);
                    f.b_valid[k] = b_has_valid[src] ? bvalid[src].buf.as<uint8_t>() : nullptr;
                    f.ob_data[k] = out_data[k].p; f.ob_valid[k] = out_has_valid[k] ? out_vbytes[k].as<uint8_t>() : nullptr;
                } else {
                    int j = k - (int)kb.size();
                    f.p_data[j] = data[src]; f.p_valid[j] = valid[src]; f.p_size[j] = ctype_size(p_ct[src]);
                    f.op_data[j] = out_data[k].p; f.op_valid[j] = out_has_valid[k] ? out_vbytes[k].as<uint8_t>() : nullptr;
                }
            }
            B200_CUDA(cudaMemsetAsync(d_cursor.p, 0, 8, stream));
            const int gridp = (int)std::min<int64_t>((int64_t)sms * 8, (n + 1023) / 1024);
            with_nk([&](auto c) { join_probe_fast_mk_kernel<decltype(c)::value><<<gridp, 256, 0, stream>>>(f); });
        } else if (n > 0) {
            FastProbeArgs f{};
            f.n_probe = n; f.key_data = data[0]; f.key_ctype = p_ct[0]; f.key_valid = valid[0];
            f.slots = d_slots16.as<Slot16>(); f.cap = cap; f.bpack = d_bpack.as<unsigned long long>(); f.n_fields = std::max(n_b - 1, 1);
            f.cursor = d_cursor.as<unsigned long long>(); f.n_b = (int)kb.size(); f.n_p = (int)kp.size(); f.na_equal = na_equal ? 1 : 0;
            for (int k = 0; k < n_out_cols; k++) {
                bool is_b = k < (int)kb.size();
                int src = is_b ? kb[k] : kp[k - kb.size()];
                if (is_b) {
                    f.b_field[k] = src - 1; f.b_size[k] = ctype_size(b_ct[src]);
                    f.b_valid[k] = (src > 0 && b_has_valid[src]) ? bvalid[src].buf.as<uint8_t>() : nullptr;
                    f.ob_data[k] = out_data[k].p; f.ob_valid[k] = out_has_valid[k] ? out_vbytes[k].as<uint8_t>() : nullptr;
                } else {
                    int j = k - (int)kb.size();
                    f.p_data[j] = data[src]; f.p_valid[j] = valid[src]; f.p_size[j] = ctype_size(p_ct[src]);
                    f.op_data[j] = out_data[k].p; f.op_valid[j] = out_has_valid[k] ? out_vbytes[k].as<uint8_t>() : nullptr;
                }
            }
            B200_CUDA(cudaMemsetAsync(d_cursor.p, 0, 8, stream));
            // inline-payload variant: every column of this batch 8 bytes wide and bitmap-free, 1..4 kept probe columns
            bool inl = inline_ready && valid[0] == nullptr && kp.size() >= 1 && kp.size() <= (size_t)J_INL_MAX_P && kb.size() <= 4;
            for (int src : kp) inl = inl && ctype_size(p_ct[src]) == 8 && valid[src] == nullptr;
            for (int k = 0; k < n_out_cols; k++) inl = inl && !out_has_valid[k];  // (a nullable-typed column without a bitmap still gets one)
            const int gridp = (int)std::min<int64_t>((int64_t)sms * 8, (n + 1023) / 1024);
            if (inl) {
                InlineProbeArgs ia{};
                ia.n_probe = n; ia.key = (const long long*)data[0]; ia.slots = d_slots32.as<Slot32>(); ia.cap = cap;
                ia.cursor = d_cursor.as<unsigned long long>(); ia.n_b = (int)kb.size();
                for (size_t k = 0; k < kb.size(); k++) { ia.b_field[k] = kb[k] - 1; ia.ob[k] = out_data[k].as<unsigned long long>(); }
                for (size_t j = 0; j < kp.size(); j++) { ia.p[j] = (const unsigned long long*)data[kp[j]]; ia.op[j] = out_data[kb.size() + j].as<unsigned long long>(); }
                const int nf = n_b - 1;
#define B200_INL(NF, NPK) join_probe_inline_kernel<NF, NPK><<<gridp, 256, 0, stream>>>(ia)
#define B200_INL_NF(NF) do { switch (kp.size()) { case 1: B200_INL(NF, 1); break; case 2: B200_INL(NF, 2); break; case 3: B200_INL(NF, 3); break; default: B200_INL(NF, 4); break; } } while (0)
                if (nf <= 0) B200_INL_NF(0); else if (nf == 1) B200_INL_NF(1); else B200_INL_NF(2);
#undef B200_INL_NF
#undef B200_INL
                inline_probes++;
            } else {
                ensure_fast_tables();
                f.slots = d_slots16.as<Slot16>(); f.bpack = d_bpack.as<unsigned long long>();
                join_probe_fast_kernel<<<gridp, 256, 0, stream>>>(f);
            }
        }
        if (n > 0) {
            launches++; fast_probes++;
            B200_CUDA(cudaGetLastError());
            B200_CUDA(cudaMemcpyAsync(h_cursor, d_cursor.p, 8, cudaMemcpyDeviceToHost, stream));
            B200_CUDA(cudaStreamSynchronize(stream));
            rows = (int64_t)*h_cursor;
            for (int k = 0; k < n_out_cols; k++)
                if (out_has_valid[k] && rows > 0) { pack_bitmap_kernel<<<grid_for(rows), 256, 0, stream>>>(out_vbytes[k].as<uint8_t>(), rows, out_bitmap[k].as<uint32_t>()); launches++; }
            B200_CUDA(cudaGetLastError());
            B200_CUDA(cudaStreamSynchronize(stream));
        }
        describe_out(out, kb, kp, rows);
        probe_rows += n; out_rows_total += rows;
        return rows;
    }

    int64_t probe_consume(const b200_table* t, const uint64_t* kept_b, int64_t n_kb, const uint64_t* kept_p, int64_t n_kp,
                          b200_table* out, bool is_last) {
        B200_REQUIRE(build_final, "b200 join: probe before the build side was finished (is_last build batch)");
        if (n_p == 0) {  // adopt the probe schema from the first probe batch
            B200_REQUIRE(t->n_cols >= 1 && t->n_cols <= J_MAX_COLS, "b200 join: between 1 and 32 columns per side");
            std::vector<int8_t> ct(t->n_cols), at(t->n_cols);
            for (int c = 0; c < t->n_cols; c++) { ct[c] = (int8_t)t->cols[c].c_type; at[c] = (int8_t)t->cols[c].arr_type; }
            set_probe_schema(ct.data(), at.data(), t->n_cols);
        }
        B200_REQUIRE(t->n_cols == n_p, "b200 join: probe batch has a different number of columns than the schema");
        B200_REQUIRE(out->cols != nullptr, "b200 join: out->cols must point to n_kept_build + n_kept_probe descriptors");
        B200_CUDA(cudaSetDevice(device)); scratch_set_stream(stream);
        std::vector<int> kb, kp;
        for (int64_t k = 0; k < n_kb; k++) { B200_REQUIRE((int)kept_b[k] < n_b, "b200 join: bad kept build column"); kb.push_back((int)kept_b[k]); }
        for (int64_t k = 0; k < n_kp; k++) { B200_REQUIRE((int)kept_p[k] < n_p, "b200 join: bad kept probe column"); kp.push_back((int)kept_p[k]); }
        int n_out_cols = (int)(kb.size() + kp.size());
        B200_REQUIRE(n_out_cols + (mark ? 1 : 0) <= J_MAX_COLS, "b200 join: too many output columns");
        B200_REQUIRE(!mark || kb.empty(), "b200 join: a mark join does not output build table columns (bodo/pandas/physical/join.h:309-316)");
        int64_t n = t->n_rows;
        std::vector<const void*> data; std::vector<const uint8_t*> valid;
        stage_batch(t, n_p, p_ct, data, valid);
        if (fast_ready) return probe_fast(t, kb, kp, data, valid, out);
        // pass A + scan
        unsigned long long n_match = 0;
        d_pslot.ensure((size_t)(n + 1) * 4); d_pcnt.ensure((size_t)(n + 1) * 4); d_poff.ensure((size_t)(n + 2) * 8);
        if (n > 0) {
            if (mark) { d_mark.ensure((size_t)n + 32); d_mark_valid.ensure((size_t)(n + 7) / 8 + 32); B200_CUDA(cudaMemsetAsync(d_mark_valid.p, 0xff, (size_t)(n + 7) / 8 + 8, stream)); }
            if (nk == 1)
                join_probe_count_kernel<<<grid_for(n), 256, 0, stream>>>(data[0], p_ct[0], valid[0], n, d_tkeys.as<long long>(), cap, d_info.as<SlotInfo>(),
                                                                         probe_outer ? 1 : 0, d_pslot.as<uint32_t>(), d_pcnt.as<uint32_t>(), na_equal ? 1 : 0,
                                                                         anti ? 1 : (mark ? 2 : 0), mark ? d_mark.as<uint8_t>() : nullptr);
            else
                with_nk([&](auto c) {
                    join_probe_count_mk_kernel<decltype(c)::value><<<grid_for(n), 256, 0, stream>>>(
                        probe_keys(data, valid), build_keys(), n, d_tkeys.as<unsigned long long>(), cap, d_info.as<SlotInfo>(), probe_outer ? 1 : 0,
                        d_pslot.as<uint32_t>(), d_pcnt.as<uint32_t>(), na_equal ? 1 : 0, anti ? 1 : (mark ? 2 : 0), mark ? d_mark.as<uint8_t>() : nullptr);
                });
            launches++;
            B200_CUDA(cudaMemsetAsync(d_pcnt.as<uint32_t>() + n, 0, 4, stream));
            n_match = scan.run(d_pcnt.as<uint32_t>(), n + 1, d_poff.as<unsigned long long>(), stream, &launches);
        }
        // unmatched build rows go out with the last probe batch
        unsigned long long n_tail = 0;
        DevBuf tail_flags, tail_off;
        if (is_last && build_outer && !tail_emitted && n_build > 0) {
            tail_flags.alloc((size_t)(n_build + 1) * 4); tail_off.alloc((size_t)(n_build + 2) * 8);
        }
        // which output columns carry validity: nullable inputs, NULL-extended sides of an outer join
        out_has_valid.assign(n_out_cols, false);
        for (int k = 0; k < n_out_cols; k++) {
            bool is_b = k < (int)kb.size();
            int src = is_b ? kb[k] : kp[k - kb.size()];
            out_has_valid[k] = is_b ? (b_has_valid[src] || b_at[src] == ARR_NULLABLE || probe_outer || anti)
                                    : (valid[src] != nullptr || p_at[src] == ARR_NULLABLE || build_outer);
        }
        auto ensure_out = [&](int64_t rows) {
            for (int k = 0; k < n_out_cols; k++) {
                bool is_b = k < (int)kb.size();
                int src = is_b ? kb[k] : kp[k - kb.size()];
                out_data[k].ensure((size_t)(rows + 32) * ctype_size(is_b ? b_ct[src] : p_ct[src]));
                if (out_has_valid[k]) { out_vbytes[k].ensure((size_t)rows + 32); out_bitmap[k].ensure((size_t)((rows + 31) / 32 + 1) * 4); }
            }
        };
        // pass B needs bmatched complete before the tail is computed, so: gather first, then the tail
        GatherArgs g{};
        g.n_probe = n; g.pslot = d_pslot.as<uint32_t>(); g.poff = d_poff.as<unsigned long long>(); g.info = d_info.as<SlotInfo>();
        g.goffs = d_goffs.as<unsigned long long>(); g.groups = d_groups.as<uint32_t>(); g.bmatched = build_outer ? d_bmatched.as<uint8_t>() : nullptr;
        g.n_b = (int)kb.size(); g.n_p = (int)kp.size();
        // the tail size is only known after the gather; grow the output (keeping the gathered rows) if needed
        ensure_out((int64_t)n_match);
        for (int k = 0; k < n_out_cols; k++) {
            bool is_b = k < (int)kb.size();
            int src = is_b ? kb[k] : kp[k - kb.size()];
            if (is_b) {
                int j = k;
                g.b_data[j] = bcol[src].buf.p; g.b_valid[j] = b_has_valid[src] ? bvalid[src].buf.as<uint8_t>() : nullptr; g.b_size[j] = ctype_size(b_ct[src]);
                g.ob_data[j] = out_data[k].p; g.ob_valid[j] = out_has_valid[k] ? out_vbytes[k].as<uint8_t>() : nullptr;
            } else {
                int j = k - (int)kb.size();
                g.p_data[j] = data[src]; g.p_valid[j] = valid[src]; g.p_size[j] = ctype_size(p_ct[src]);
                g.op_data[j] = out_data[k].p; g.op_valid[j] = out_has_valid[k] ? out_vbytes[k].as<uint8_t>() : nullptr;
            }
        }
        if (n > 0 && n_match > 0) { join_probe_gather_kernel<<<grid_for(n), 256, 0, stream>>>(g); launches++; B200_CUDA(cudaGetLastError()); }
        if (tail_flags.p) {
            join_unmatched_flags_kernel<<<grid_for(n_build), 256, 0, stream>>>(d_bmatched.as<uint8_t>(), n_build, tail_flags.as<uint32_t>());
            B200_CUDA(cudaMemsetAsync(tail_flags.as<uint32_t>() + n_build, 0, 4, stream));
            launches++;
            n_tail = scan.run(tail_flags.as<uint32_t>(), n_build + 1, tail_off.as<unsigned long long>(), stream, &launches);
            tail_emitted = true;
            if (n_tail > 0) {
                // grow output columns, preserving the rows already gathered
                for (int k = 0; k < n_out_cols; k++) {
                    bool is_b = k < (int)kb.size();
                    int src = is_b ? kb[k] : kp[k - kb.size()];
                    size_t isz = ctype_size(is_b ? b_ct[src] : p_ct[src]);
                    size_t need = (size_t)(n_match + n_tail + 32) * isz;
                    if (need > out_data[k].bytes) {
                        DevBuf nb; nb.alloc(need);
                        B200_CUDA(cudaMemcpyAsync(nb.p, out_data[k].p, (size_t)n_match * isz, cudaMemcpyDeviceToDevice, stream));
                        B200_CUDA(cudaStreamSynchronize(stream));
                        out_data[k] = std::move(nb);
                    }
                    if (out_has_valid[k]) {
                        size_t needv = (size_t)(n_match + n_tail) + 32;
                        if (needv > out_vbytes[k].bytes) {
                            DevBuf nb; nb.alloc(needv);
                            B200_CUDA(cudaMemcpyAsync(nb.p, out_vbytes[k].p, (size_t)n_match, cudaMemcpyDeviceToDevice, stream));
                            B200_CUDA(cudaStreamSynchronize(stream));
                            out_vbytes[k] = std::move(nb);
                        }
                        out_bitmap[k].ensure((size_t)((n_match + n_tail + 31) / 32 + 1) * 4);
                    }
                }
                TailArgs ta{};
                ta.n_build = n_build; ta.flags = tail_flags.as<uint32_t>(); ta.off = tail_off.as<unsigned long long>();
                ta.n_b = (int)kb.size(); ta.n_p = (int)kp.size();
                for (int k = 0; k < n_out_cols; k++) {
                    bool is_b = k < (int)kb.size();
                    int src = is_b ? kb[k] : kp[k - kb.size()];
                    size_t isz = ctype_size(is_b ? b_ct[src] : p_ct[src]);
                    if (is_b) {
                        ta.b_data[k] = bcol[src].buf.p; ta.b_valid[k] = b_has_valid[src] ? bvalid[src].buf.as<uint8_t>() : nullptr; ta.b_size[k] = (int)isz;
                        ta.ob_data[k] = (char*)out_data[k].p + n_match * isz; ta.ob_valid[k] = out_has_valid[k] ? out_vbytes[k].as<uint8_t>() + n_match : nullptr;
                    } else {
                        int j = k - (int)kb.size();
                        ta.p_size[j] = (int)isz;
                        ta.op_data[j] = (char*)out_data[k].p + n_match * isz; ta.op_valid[j] = out_vbytes[k].as<uint8_t>() + n_match;
                    }
                }
                join_unmatched_emit_kernel<<<grid_for(n_build), 256, 0, stream>>>(ta);
                launches++;
                B200_CUDA(cudaGetLastError());
            }
        }
        int64_t rows = (int64_t)(n_match + n_tail);
        for (int k = 0; k < n_out_cols; k++)
            if (out_has_valid[k] && rows > 0) { pack_bitmap_kernel<<<grid_for(rows), 256, 0, stream>>>(out_vbytes[k].as<uint8_t>(), rows, out_bitmap[k].as<uint32_t>()); launches++; }
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaStreamSynchronize(stream));
        describe_out(out, kb, kp, rows);
        if (mark) {  // the mark column: BOOL, nullable array type, every row valid; output row i is probe row i
            b200_column& c = out->cols[n_out_cols];
            c.data = d_mark.p; c.validity = d_mark_valid.as<uint8_t>(); c.length = rows; c.c_type = CT_BOOL; c.arr_type = ARR_NULLABLE;
            out->n_cols = n_out_cols + 1;
        }
        probe_rows += n; out_rows_total += rows;
        return rows;
    }
};

}  // namespace b200

using b200::JoinState;

extern "C" {

void* b200_join_state_init(int64_t operator_id, const int8_t* build_arr_c_types, const int8_t* build_arr_array_types,
                           int32_t n_build_arrs, const int8_t* probe_arr_c_types, const int8_t* probe_arr_array_types,
                           int32_t n_probe_arrs, uint64_t n_keys, int32_t build_table_outer, int32_t probe_table_outer,
                           int32_t is_na_equal, int64_t output_batch_size, int32_t device, int64_t expected_build_rows, void* stream) {
    (void)operator_id;
    try {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw b200::Error("b200 join: no CUDA device available (this path has no CPU fallback)");
        B200_REQUIRE(device >= 0 && device < ndev, "b200 join: bad device ordinal");
        return new JoinState(build_arr_c_types, build_arr_array_types, n_build_arrs, probe_arr_c_types, probe_arr_array_types, n_probe_arrs,
                             n_keys, build_table_outer != 0, probe_table_outer != 0, is_na_equal != 0, output_batch_size, device, expected_build_rows, (cudaStream_t)stream);
    } catch (const std::exception& e) { b200::set_last_error(e.what()); return nullptr; }
}

int b200_join_build_consume_batch(void* state, const b200_table* in_table, int32_t is_last, int32_t* request_input) {
    try {
        B200_REQUIRE(state && in_table, "b200 join: null state or table");
        ((JoinState*)state)->build_consume(in_table, is_last != 0);
        if (request_input) *request_input = 1;
        return is_last ? 1 : 0;
    } catch (const std::exception& e) { b200::set_last_error(e.what()); return -1; }
}

int b200_join_probe_consume_batch(void* state, const b200_table* in_table, const uint64_t* kept_build_cols, int64_t n_kept_build,
                                  const uint64_t* kept_probe_cols, int64_t n_kept_probe, b200_table* out, int64_t* total_rows,
                                  int32_t is_last, int32_t* out_is_last) {
    try {
        B200_REQUIRE(state && in_table && out, "b200 join: null argument");
        int64_t rows = ((JoinState*)state)->probe_consume(in_table, kept_build_cols, n_kept_build, kept_probe_cols, n_kept_probe, out, is_last != 0);
        if (total_rows) *total_rows = rows;
        if (out_is_last) *out_is_last = is_last ? 1 : 0;
        return 0;
    } catch (const std::exception& e) { b200::set_last_error(e.what()); return -1; }
}

void b200_delete_join_state(void* state) { delete (JoinState*)state; }

int b200_join_set_kind(void* state, int32_t is_mark_join, int32_t is_anti_join) {
    try {
        B200_REQUIRE(state, "b200 join: null state");
        ((JoinState*)state)->set_kind(is_mark_join != 0, is_anti_join != 0);
        return 0;
    } catch (const std::exception& e) { b200::set_last_error(e.what()); return -1; }
}

int b200_join_build_filter(void* state, int64_t n_bloom_blocks, void** bloom_words_dev, int64_t* n_blocks_out, int64_t* key_min_max) {
    try {
        B200_REQUIRE(state && n_bloom_blocks >= 0, "b200 join: bad arguments");
        auto* s = (JoinState*)state;
        s->build_filter((uint64_t)n_bloom_blocks);
        if (bloom_words_dev) *bloom_words_dev = s->d_bloom.p;
        if (n_blocks_out) *n_blocks_out = (int64_t)s->bloom_blocks;
        if (key_min_max) { key_min_max[0] = s->key_min; key_min_max[1] = s->key_max; }
        return 0;
    } catch (const std::exception& e) { b200::set_last_error(e.what()); return -1; }
}

int b200_join_set_key_bounds(void* state, int64_t key_min, int64_t key_max) {
    try {
        B200_REQUIRE(state, "b200 join: null state");
        ((JoinState*)state)->require_single_key_filter();
        ((JoinState*)state)->key_min = key_min; ((JoinState*)state)->key_max = key_max;
        return 0;
    } catch (const std::exception& e) { b200::set_last_error(e.what()); return -1; }
}

int b200_join_runtime_filter(void* state, const b200_table* in_table, int32_t key_col, int32_t use_min_max, int32_t use_bloom, uint8_t* keep_out) {
    try {
        B200_REQUIRE(state && in_table && keep_out, "b200 join: null argument");
        ((JoinState*)state)->runtime_filter(in_table, key_col, use_min_max != 0, use_bloom != 0, keep_out);
        return 0;
    } catch (const std::exception& e) { b200::set_last_error(e.what()); return -1; }
}

int64_t b200_join_get_metric(void* state, int32_t which) {
    auto* s = (JoinState*)state;
    switch (which) {
        case 0: return s->n_build;
        case 1: return (int64_t)s->cap;
        case 2: return s->probe_rows;
        case 3: return s->out_rows_total;
        case 4: return s->launches;
        case 5: return s->fast_probes;
        case 6: return s->inline_probes;
        case 7: return s->inline_builds;
        default: return -1;
    }
}

}  // extern "C"
