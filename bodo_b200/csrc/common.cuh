// common.cuh — shared device/host helpers for libbodo_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include <stdexcept>
#include <string>

#include "../../include/bodo_b200.h"

namespace b200 {

// Bodo_CTypes / bodo_array_type codes (reference: bodo/libs/_bodo_common.h:331-359, :515-532)
enum CType : int { CT_INT8 = 0, CT_UINT8 = 1, CT_INT32 = 2, CT_UINT32 = 3, CT_INT64 = 4, CT_FLOAT32 = 5, CT_FLOAT64 = 6,
                   CT_UINT64 = 7, CT_INT16 = 8, CT_UINT16 = 9, CT_BOOL = 11, CT_DATE = 13, CT_DATETIME = 15,
                   CT_TIMEDELTA = 16 };
enum ArrType : int { ARR_NUMPY = 0, ARR_NULLABLE = 2 };
// Bodo_FTypes (reference: bodo/libs/groupby/_groupby_ftypes.h:17-110)
enum FType : int { FT_SIZE = 4, FT_SUM = 6, FT_COUNT = 7, FT_NUNIQUE = 8, FT_MEAN = 14, FT_MIN = 15, FT_MAX = 16, FT_FIRST = 18, FT_LAST = 19,
                   FT_VAR_POP = 22, FT_STD_POP = 23, FT_VAR = 24, FT_STD = 25, FT_SKEW = 27 };

// hash seeds (reference: bodo/libs/_array_hash.h:8-14)
constexpr uint32_t SEED_HASH_PARTITION = 0xb0d01289u;
constexpr uint32_t SEED_HASH_JOIN = 0xb0d01286u;

void set_last_error(const std::string& msg);

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define B200_CUDA(call)                                                                                       \
    do {                                                                                                      \
        cudaError_t _e = (call);                                                                              \
        if (_e != cudaSuccess)                                                                                \
            throw b200::Error(std::string("CUDA error: ") + cudaGetErrorString(_e) + " in " #call " at " +   \
                              __FILE__ + ":" + std::to_string(__LINE__));                                     \
    } while (0)

#define B200_REQUIRE(cond, msg)                      \
    do {                                             \
        if (!(cond)) throw b200::Error(std::string(msg)); \
    } while (0)

__host__ __device__ inline int ctype_size(int ct) {
    switch (ct) {
        case CT_INT8: case CT_UINT8: case CT_BOOL: return 1;
        case CT_INT16: case CT_UINT16: return 2;
        case CT_INT32: case CT_UINT32: case CT_FLOAT32: case CT_DATE: return 4;
        case CT_INT64: case CT_UINT64: case CT_FLOAT64: case CT_DATETIME: case CT_TIMEDELTA: return 8;
        default: return 0;
    }
}
__host__ __device__ inline bool ctype_is_float(int ct) { return ct == CT_FLOAT32 || ct == CT_FLOAT64; }
inline bool ctype_is_signed_int(int ct) {
    return ct == CT_INT8 || ct == CT_INT16 || ct == CT_INT32 || ct == CT_INT64 || ct == CT_DATE || ct == CT_DATETIME ||
           ct == CT_TIMEDELTA;
}

// ---- device helpers -------------------------------------------------------------------------

__device__ __forceinline__ bool bit_valid(const uint8_t* __restrict__ bm, int64_t i) {
    return bm == nullptr || ((bm[i >> 3] >> (i & 7)) & 1);
}

__device__ __forceinline__ uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }

// XXH3_64bits_withSeed for 4- and 8-byte inputs (XXH3_len_4to8_64b + XXH3_rrmxmx), the function behind the
// reference's hash_inner_32 (bodo/libs/vendored/_murmurhash3.h:59-68, vendored/xxhash.h:4034-4041,4102-4119).
// Restated from the published xxHash algorithm; pinned against the reference's vendored header in
// tests/test_oracle.py (through the oracle) and tests/test_gpu_shuffle.py (this device function).
__host__ __device__ __forceinline__ uint64_t xxh3_64_short(uint64_t raw, int len, uint32_t seed32) {
    uint64_t seed = seed32;
    uint32_t s = (uint32_t)seed;
    uint32_t sw = ((s & 0xffu) << 24) | ((s & 0xff00u) << 8) | ((s >> 8) & 0xff00u) | (s >> 24);
    seed ^= (uint64_t)sw << 32;
    uint32_t in1 = (uint32_t)raw;
    uint32_t in2 = len == 8 ? (uint32_t)(raw >> 32) : (uint32_t)raw;
    const uint64_t bitflip = (0x1cad21f72c81017cULL ^ 0xdb979083e96dd4deULL) - seed;
    uint64_t h = ((uint64_t)in2 + ((uint64_t)in1 << 32)) ^ bitflip;
    h ^= ((h << 49) | (h >> 15)) ^ ((h << 24) | (h >> 40));
    h *= 0x9FB21C651E98DF25ULL;
    h ^= (h >> 35) + (uint64_t)len;
    h *= 0x9FB21C651E98DF25ULL;
    return h ^ (h >> 28);
}

// hash_combine_boost (reference: bodo/libs/_array_hash.cpp:41-56): one 32-bit murmur round folding a further key column's
// hash into the running row hash.
__host__ __device__ __forceinline__ uint32_t hash_combine_boost(uint32_t h1, uint32_t k1) {
    k1 *= 0xcc9e2d51u;
    k1 = (k1 << 15) | (k1 >> 17);
    k1 *= 0x1b873593u;
    h1 ^= k1;
    h1 = (h1 << 13) | (h1 >> 19);
    return h1 * 5u + 0xe6546b64u;
}
// _Py_HashDouble (CPython Python/pyhash.c, what the reference feeds float keys through before hashing the resulting
// Py_hash_t, bodo/libs/_array_hash.cpp:119-170): reduction of the double modulo the Mersenne prime 2^61 - 1; NaN -> 0 (the
// reference passes a NULL identity), +-inf -> +-314159.  Restated from the published algorithm; pinned against the oracle
// (which is pinned against the interpreter's own hash(float)) in tests/test_gpu_shuffle.py.
__host__ __device__ inline int64_t py_hash_double(double v) {
    const int BITS = 61;
    const uint64_t MOD = (1ULL << 61) - 1;
    if (isnan(v)) return 0;
    if (isinf(v)) return v > 0 ? 314159 : -314159;
    int e;
    double m = frexp(v, &e);
    int sign = 1;
    if (m < 0) { sign = -1; m = -m; }
    uint64_t x = 0;
    while (m != 0.0) {
        x = ((x << 28) & MOD) | (x >> (BITS - 28));
        m *= 268435456.0;  // 2^28
        e -= 28;
        uint64_t y = (uint64_t)m;
        m -= (double)y;
        x += y;
        if (x >= MOD) x -= MOD;
    }
    e = e >= 0 ? e % BITS : BITS - 1 - ((-1 - e) % BITS);
    x = ((x << e) & MOD) | (x >> (BITS - e));
    int64_t r = (int64_t)x * sign;
    return r == -1 ? -2 : r;
}

// hash_to_rank (reference: bodo/libs/_shuffle.h:5-7): (uint32) hash % n_pes.
__host__ __device__ __forceinline__ int hash_to_rank_u32(uint32_t h, int n_pes) { return (int)(h % (uint32_t)n_pes); }

// Table-slot hash: the same xxh3 value (one hash per row); ranks use the low 32 bits, slots the high 32
// bits, so the two are independent (a rank's keys all share low32 % P).
__device__ __forceinline__ uint64_t key_hash(int64_t key) { return xxh3_64_short((uint64_t)key, 8, SEED_HASH_PARTITION); }

__device__ __forceinline__ int64_t load_int_as_i64(const void* __restrict__ p, int ct, int64_t i) {
    switch (ct) {
        case CT_INT64: case CT_DATETIME: case CT_TIMEDELTA: case CT_UINT64: return ((const int64_t*)p)[i];
        case CT_INT32: case CT_DATE: return ((const int32_t*)p)[i];
        case CT_UINT32: return ((const uint32_t*)p)[i];
        case CT_INT16: return ((const int16_t*)p)[i];
        case CT_UINT16: return ((const uint16_t*)p)[i];
        case CT_INT8: return ((const int8_t*)p)[i];
        case CT_UINT8: case CT_BOOL: return ((const uint8_t*)p)[i];
        default: return 0;
    }
}
__device__ __forceinline__ double load_as_f64(const void* __restrict__ p, int ct, int64_t i) {
    switch (ct) {
        case CT_FLOAT64: return ((const double*)p)[i];
        case CT_FLOAT32: return (double)((const float*)p)[i];
        default: return (double)load_int_as_i64(p, ct, i);
    }
}

// hash_keys (reference: bodo/libs/_array_hash.cpp:1599-1621) of one row over 1..MAX_HASH_KEYS key columns: the first column is
// hashed (hash_array_inner: sizeof(T) raw bytes of an integer / date column through XXH3, a float column through
// _Py_HashDouble first; NA -> hash_na_val = hash of int64 1), every further column's hash is folded in with
// hash_combine_boost.  Low 32 bits of the XXH3 value, as hash_inner_32 returns them.
constexpr int MAX_HASH_KEYS = 4;
struct KeySet {
    int n_keys;
    const void* data[MAX_HASH_KEYS];
    const uint8_t* valid[MAX_HASH_KEYS];
    int ctype[MAX_HASH_KEYS];
};
__device__ __forceinline__ uint32_t hash_key_column(const void* data, int ct, const uint8_t* valid, int64_t i, uint32_t seed) {
    if (!bit_valid(valid, i)) return (uint32_t)xxh3_64_short(1ull, 8, seed);
    if (ct == CT_FLOAT64 || ct == CT_FLOAT32) return (uint32_t)xxh3_64_short((uint64_t)py_hash_double(load_as_f64(data, ct, i)), 8, seed);
    if (ctype_size(ct) == 8) return (uint32_t)xxh3_64_short((uint64_t)load_int_as_i64(data, ct, i), 8, seed);
    return (uint32_t)xxh3_64_short((uint64_t)(uint32_t)load_int_as_i64(data, ct, i), 4, seed);  // 4-byte keys hash their 4 raw bytes
}
__device__ __forceinline__ uint32_t hash_keys_row(const KeySet& k, int64_t i, uint32_t seed) {
    uint32_t h = hash_key_column(k.data[0], k.ctype[0], k.valid[0], i, seed);
    for (int j = 1; j < k.n_keys; j++) h = hash_combine_boost(h, hash_key_column(k.data[j], k.ctype[j], k.valid[j], i, seed));
    return h;
}

// Key-tuple tables (multi-key groupby, multi-key join): a slot is claimed through a 64-bit tag word, the hash of the widened
// int64 key values and the NA mask (bit j = key column j is valid) with bit 63 set, so a published tag is never TAG_EMPTY or
// TAG_LOCKED.  The claiming thread CASes empty -> locked, writes what readers compare against, fences and publishes the tag.
constexpr unsigned long long TAG_EMPTY = 0ull, TAG_LOCKED = 1ull;

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long mk_tag(const long long* keys, unsigned int mask, int nk) {
    unsigned long long h = 0x9E3779B97F4A7C15ULL ^ mask;
    for (int j = 0; j < nk; j++) h = xxh3_64_short((unsigned long long)keys[j] ^ (h * 0xD1B54A32D192ED03ULL), 8, SEED_HASH_PARTITION + j);
    return h | 0x8000000000000000ULL;
}

// order-preserving double <-> uint64 encoding (so float min/max are native 64-bit integer atomics)
__host__ __device__ __forceinline__ uint64_t f64_to_ordered(double d) {
#ifdef __CUDA_ARCH__
    uint64_t b = (uint64_t)__double_as_longlong(d);
#else
    uint64_t b; memcpy(&b, &d, 8);
#endif
    return b ^ ((b >> 63) ? 0xFFFFFFFFFFFFFFFFULL : 0x8000000000000000ULL);
}
__host__ __device__ __forceinline__ double ordered_to_f64(uint64_t e) {
    uint64_t b = e ^ ((e >> 63) ? 0x8000000000000000ULL : 0xFFFFFFFFFFFFFFFFULL);
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)b);
#else
    double d; memcpy(&d, &b, 8); return d;
#endif
}

// counter-based generator of the synthetic workload (SURVEY.md §8d); mirrored in oracle/bodo_oracle.c
// (oracle_synth_fill) and bodo_b200/synth.py.
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x += 0x9e3779b97f4a7c15ULL;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ULL;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebULL;
    return x ^ (x >> 31);
}

inline int num_sms(int device) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
    return n > 0 ? n : 148;
}

// Scratch buffers (bucket / retry / fail lists: up to GBs) come from a process-wide per-device pool and go back to
// it when a state dies, so creating an operator state per query does not pay cudaMalloc / cudaFree of gigabytes
// (cudaFree of multi-GB blocks is synchronous and costs tens of milliseconds).
// The pool is stream-ordered: a released block remembers an event recorded on the releasing thread's scratch stream
// (scratch_set_stream: every state entry point sets it to the state's stream) and is only handed out again once that
// event has completed.  Pooled bytes are capped (B200_POOL_MAX_BYTES, default 24 GiB; scratch_trim frees on request).
void* scratch_acquire(int device, size_t bytes, size_t* got);
void scratch_release(int device, void* p, size_t bytes);
void scratch_set_stream(cudaStream_t s);
void scratch_trim(int device, size_t keep_bytes);
void* pinned_acquire(size_t bytes);   // small pinned host blocks (counter mirrors), pooled for the same reason
void pinned_release(void* p, size_t bytes);

// RAII device buffer drawn from the pool of the CURRENT device (states call cudaSetDevice first).
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int device = -1;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes), device(o.device) { o.p = nullptr; o.bytes = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { release(); p = o.p; bytes = o.bytes; device = o.device; o.p = nullptr; o.bytes = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() { if (p) scratch_release(device, p, bytes); p = nullptr; bytes = 0; }
    void alloc(size_t n) {
        release();
        if (n == 0) n = 8;
        B200_CUDA(cudaGetDevice(&device));
        p = scratch_acquire(device, n, &bytes);
    }
    void ensure(size_t n) { if (n > bytes) alloc(n); }
    void ensure(int /*dev*/, size_t n) { ensure(n); }
    template <typename T> T* as() const { return (T*)p; }
};
using PooledBuf = DevBuf;

}  // namespace b200
