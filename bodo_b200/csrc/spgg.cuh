// SPG-G: the SM-partitioned groupby path (see groupby.cu, "SM-partitioned groupby") for everything that is not the headline
// signature.  Included by groupby.cu only.
//
//   keys    one integer / date / datetime column of 4 or 8 bytes (not uint64), nullable or not (NA keys: dropped with dropna,
//           else they form the NA group, as in groupby_consume_kernel)
//   values  one integer column of 4 or 8 bytes (not uint64), nullable or not — or none (size only)
//   funcs   any mix of sum, count, size, mean, min, max over that column (mean of integers accumulates the exact integer sum
//           per launch and owner and folds it into the state's double accumulator at the flush; the reference adds doubles row
//           by row, _groupby_agg_funcs.h:673-689 — same value up to the rounding of the partial sums)
//
// K1g is spg_partition_tma_kernel generalised: the tile's raw key / value bytes AND its two validity-bitmap slices (256 B per
// 2048-row tile) come in through TMA (cp.async.bulk + mbarrier), rows are widened to (int64 key, int64 value) when they are
// read from the staging tile.  Rows whose VALUE is NA must still create their group (and count for `size`): they are
// partitioned too, into a second, key-only bucket per owner (class index owner + G in the same counting sort), so no row
// takes a global-memory probe inside K1g.  NA-KEY rows are dropped (dropna) or pre-aggregated per CTA in shared memory and
// added to the NA slot of the state's table once per CTA.  Only rows with the marker key and bucket overflow (skew) take the
// direct path.  K2g is spg_aggregate_kernel's hot loop over a wider slot when min / max are asked for (key, low sum word,
// count, min, max = 32 B instead of 16 B, so the owners hold half as many groups per pass), plus a pass over the owner's
// key-only bucket.  min / max read the slot first and only issue the (CAS-emulated, SASS ATOMS.CAST.SPIN.64) 64-bit shared
// atomic when the row improves the extremum: ~ln(rows per group) times per group.
#pragma once

constexpr int GEN_MAX_F = 8;
struct GenFlush {
    int n;
    int kind[GEN_MAX_F];
    unsigned long long* a0[GEN_MAX_F];
    unsigned long long* a1[GEN_MAX_F];
};

struct SpgGenArgs {
    SpgArgs s;  // table, buckets, retry list, owners / passes (keys, vals, acc_sum, acc_cnt unused); bucket_cnt has 2 x n_owners
                // counters: [owner] rows in the owner's bucket, [n_owners + owner] keys in its NA-value bucket
    long long* nbucket;  // [n_owners][bucket_cap] keys of the rows whose value is NA (null when the value column has no bitmap)
    int n_vo;            // buckets K1g partitions the valued rows into: n_owners (K2g tests every row's pass when n_pass > 1), or
                         // n_owners * n_pass "virtual owners" (bucket me * n_pass + p holds exactly the rows of owner me's pass p,
                         // so a multi-pass K2g still reads every row once); bucket_cnt: [0, n_vo) buckets, [n_vo, n_vo + n_owners) NA-value buckets
    const void* kdata;
    const uint8_t* kvalid;
    const void* vdata;
    const uint8_t* vvalid;
    int k_signed, v_signed;  // 4-byte columns: sign- or zero-extend
    int dropna;
    GenFlush fl;
};
constexpr int GEN_RETRY_WORDS = 8;  // [key][sum][cnt][nnull][min][max][-][-]

// one partial aggregate (sum / cnt / min / max over `cnt` non-NA values, plus `nnull` rows whose value was NA) -> slot `sl`
__device__ __forceinline__ void gen_apply_slot(const GenFlush& f, uint64_t sl, unsigned long long sum, unsigned long long cnt,
                                               unsigned long long nnull, long long mn, long long mx) {
#pragma unroll 1
    for (int j = 0; j < f.n; j++) {
        switch (f.kind[j]) {
            case K_SUM_I64: if (sum) atomicAdd(f.a0[j] + sl, sum); break;
            case K_COUNT: if (cnt) atomicAdd(f.a0[j] + sl, cnt); break;
            case K_SIZE: if (cnt + nnull) atomicAdd(f.a0[j] + sl, cnt + nnull); break;
            case K_MEAN:
                if (sum) atomicAdd((double*)f.a0[j] + sl, (double)(long long)sum);
                if (cnt) atomicAdd(f.a1[j] + sl, cnt);
                break;
            case K_MIN_I64:
                if (cnt) { atomicMin((long long*)f.a0[j] + sl, mn); if (f.a1[j]) atomicAdd(f.a1[j] + sl, cnt); }
                break;
            case K_MAX_I64:
                if (cnt) { atomicMax((long long*)f.a0[j] + sl, mx); if (f.a1[j]) atomicAdd(f.a1[j] + sl, cnt); }
                break;
        }
    }
}

__device__ __forceinline__ void gen_direct_apply(const SpgGenArgs& g, long long key, unsigned long long sum, unsigned long long cnt,
                                              unsigned long long nnull, long long mn, long long mx) {
    const SpgArgs& a = g.s;
    uint64_t sl;
    if (key == EMPTY_KEY) { sl = a.cap + 1; a.counters[4] = 1; }
    else {
        sl = find_or_insert(a.tkeys, a.cap, key, a.counters, a.group_limit);
        if (sl == ~0ull) {  // global table at its limit: park the partial, the host grows the table and replays it
            unsigned long long f = atomicAdd((unsigned long long*)a.retry_ctr, 1ull);
            unsigned long long* r = a.retry + f * GEN_RETRY_WORDS;
            r[0] = (unsigned long long)key; r[1] = sum; r[2] = cnt; r[3] = nnull; r[4] = (unsigned long long)mn; r[5] = (unsigned long long)mx;
            return;
        }
    }
    gen_apply_slot(g.fl, sl, sum, cnt, nnull, mn, mx);
}

__global__ void spgg_replay_kernel(const __grid_constant__ SpgGenArgs g, const unsigned long long* rows, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long* r = rows + i * GEN_RETRY_WORDS;
        gen_direct_apply(g, (long long)r[0], r[1], r[2], r[3], (long long)r[4], (long long)r[5]);
    }
}

constexpr int GEN_CLS = 448;  // counting-sort classes of K1g: n_vo buckets of valued rows + n_owners buckets of NA-value rows
constexpr size_t GEN_K1_SMEM = (size_t)SPG_TILE * 32 + GEN_CLS * 8 + 16 + 32 + GEN_CLS * 4 + (GEN_CLS + 4) * 4 + 2 * (SPG_TILE / 8 + 16) + 64;

template <int BYTES>
__device__ __forceinline__ long long gen_widen(const void* raw, int j, int is_signed) {
    if (BYTES == 8) return ((const long long*)raw)[j];
    const int t = ((const int*)raw)[j];
    return is_signed ? (long long)t : (long long)(unsigned int)t;
}

// K1g: KS / VS = bytes per key / value element (VS = 0: no value column).
template <int KS, int VS>
__global__ void __launch_bounds__(SPG_TTHREADS, SPG_TCTAS) spgg_partition_kernel(const __grid_constant__ SpgGenArgs g) {
    extern __shared__ __align__(128) unsigned char smem_gen_raw[];
    const SpgArgs& a = g.s;
    unsigned char* raw_k = smem_gen_raw;                                          // SPG_TILE x 8 (raw bytes: SPG_TILE x KS used)
    unsigned char* raw_v = raw_k + SPG_TILE * 8;                                  // SPG_TILE x 8
    longlong2* stage = (longlong2*)(raw_v + SPG_TILE * 8);                        // SPG_TILE x 16
    unsigned long long* gbase = (unsigned long long*)(stage + SPG_TILE);         // GEN_CLS x 8
    uint64_t* mbar = (uint64_t*)(gbase + GEN_CLS);                                // 2 mbarriers (one used)
    unsigned long long* na_sum = (unsigned long long*)(mbar + 2);                 // NA-key group, this CTA's partial aggregate
    long long* na_min = (long long*)(na_sum + 1);
    long long* na_max = na_min + 1;
    unsigned int* na_cnt = (unsigned int*)(na_max + 1);                           // [0] non-NA values, [1] NA values
    unsigned int* hist = na_cnt + 2;                                              // GEN_CLS
    unsigned int* lbase = hist + GEN_CLS;                                         // GEN_CLS + 4
    unsigned char* kvb = (unsigned char*)(lbase + GEN_CLS + 4);                   // 256 + 16 validity bytes of the tile's keys
    unsigned char* vvb = kvb + SPG_TILE / 8 + 16;                                 // ... and values
    const bool k_nullable = g.kvalid != nullptr, v_nullable = VS && g.vvalid != nullptr;
    const int G = a.n_owners, NVO = g.n_vo, C = NVO + (v_nullable ? G : 0), tid = threadIdx.x;
    constexpr int ROWS = SPG_TILE / SPG_TTHREADS;
    const int64_t n_tiles = (a.n_rows + SPG_TILE - 1) / SPG_TILE;
    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        *na_sum = 0; *na_min = INT64_MAX; *na_max = INT64_MIN; na_cnt[0] = 0; na_cnt[1] = 0;
    }
    for (int j = tid; j < C; j += SPG_TTHREADS) hist[j] = 0;
    __syncthreads();
    auto issue = [&](int64_t t) {
        const int64_t r0 = t * SPG_TILE;
        if (r0 + SPG_TILE <= a.n_rows && tid == 0) {
            mbar_expect_tx(&mbar[0], (uint32_t)(SPG_TILE * (KS + VS) + (k_nullable ? SPG_TILE / 8 : 0) + (v_nullable ? SPG_TILE / 8 : 0)));
            tma_load_1d(raw_k, (const char*)g.kdata + r0 * KS, SPG_TILE * KS, &mbar[0]);
            if (VS) tma_load_1d(raw_v, (const char*)g.vdata + r0 * VS, SPG_TILE * VS, &mbar[0]);
            if (k_nullable) tma_load_1d(kvb, g.kvalid + r0 / 8, SPG_TILE / 8, &mbar[0]);
            if (v_nullable) tma_load_1d(vvb, g.vvalid + r0 / 8, SPG_TILE / 8, &mbar[0]);
        }
    };
    uint32_t phase = 0;
    int64_t t = blockIdx.x;
    if (t < n_tiles) issue(t);
    for (; t < n_tiles; t += gridDim.x) {
        const int64_t r0 = t * SPG_TILE;
        const int64_t tn = t + gridDim.x;
        if (r0 + SPG_TILE <= a.n_rows) {
            while (!mbar_try_wait(&mbar[0], phase)) {}
            phase ^= 1;
        } else {  // trailing partial tile: ordinary loads of the raw bytes
            const int64_t left = a.n_rows - r0;
            for (int64_t j = tid; j < left * KS; j += SPG_TTHREADS) raw_k[j] = ((const unsigned char*)g.kdata)[r0 * KS + j];
            if (VS) for (int64_t j = tid; j < left * VS; j += SPG_TTHREADS) raw_v[j] = ((const unsigned char*)g.vdata)[r0 * VS + j];
            if (k_nullable) for (int64_t j = tid; j < (left + 7) / 8; j += SPG_TTHREADS) kvb[j] = g.kvalid[r0 / 8 + j];
            if (v_nullable) for (int64_t j = tid; j < (left + 7) / 8; j += SPG_TTHREADS) vvb[j] = g.vvalid[r0 / 8 + j];
            __syncthreads();
        }
        int cls[ROWS];
        unsigned int rk[ROWS];
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
            const int j = r * SPG_TTHREADS + tid;
            cls[r] = -1;
            if (r0 + j >= a.n_rows) continue;
            const bool kok = !k_nullable || ((kvb[j >> 3] >> (j & 7)) & 1);
            const bool vok = !v_nullable || ((vvb[j >> 3] >> (j & 7)) & 1);
            const long long k = gen_widen<KS>(raw_k, j, g.k_signed);
            const long long v = VS ? gen_widen<VS ? VS : 8>(raw_v, j, g.v_signed) : 0;
            if (!kok) {  // NA key: dropped, or this CTA's share of the NA group
                if (!g.dropna) {
                    if (vok) {
                        atomicAdd(na_sum, (unsigned long long)v);
                        atomicAdd(&na_cnt[0], 1u);
                        if (v < *na_min) atomicMin(na_min, v);
                        if (v > *na_max) atomicMax(na_max, v);
                    } else atomicAdd(&na_cnt[1], 1u);
                }
                continue;
            }
            if (k == EMPTY_KEY) { gen_direct_apply(g, k, vok ? (unsigned long long)v : 0ull, vok ? 1ull : 0ull, vok ? 0ull : 1ull, v, v); continue; }
            cls[r] = vok ? (int)spg_owner(spg_hash(k), NVO) : NVO + (int)spg_owner(spg_hash(k), G);
            rk[r] = atomicAdd(&hist[cls[r]], 1u);
        }
        __syncthreads();
        unsigned long long my_gbase = 0;
        if (tid >= SPG_TTHREADS - C) { int c = tid - (SPG_TTHREADS - C); unsigned int cnt = hist[c]; if (cnt) my_gbase = atomicAdd(&a.bucket_cnt[c * SPG_CNT_STRIDE], (unsigned long long)cnt); }
        spg_scan_hist(hist, lbase, C, tid);
        __syncthreads();
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
            if (cls[r] < 0) continue;
            const int j = r * SPG_TTHREADS + tid;
            const unsigned int p = lbase[cls[r]] + rk[r];
            stage[p] = make_longlong2(gen_widen<KS>(raw_k, j, g.k_signed), VS ? gen_widen<VS ? VS : 8>(raw_v, j, g.v_signed) : 0);
        }
        if (tid >= SPG_TTHREADS - C) { int c = tid - (SPG_TTHREADS - C); gbase[c] = my_gbase - lbase[c]; }
        __syncthreads();  // the raw tile is free from here on
        if (tn < n_tiles) issue(tn);  // the next tile streams in during the copy-out
        // the staged rows are sorted by class, valued rows first: a row's class follows from its key and its position
        const unsigned int n_tile = lbase[C], n_valued = lbase[NVO];
        for (unsigned int p = tid; p < n_tile; p += SPG_TTHREADS) {
            const longlong2 row = stage[p];
            const uint64_t h = spg_hash(row.x);
            if (p < n_valued) {
                const unsigned int c = spg_owner(h, NVO);
                const unsigned long long off = gbase[c] + p;
                if (off < (unsigned long long)a.bucket_cap) a.bucket[(size_t)c * a.bucket_cap + off] = row;
                else gen_direct_apply(g, row.x, (unsigned long long)row.y, 1ull, 0ull, row.y, row.y);  // bucket full (skew)
            } else {
                const unsigned int o = spg_owner(h, G);
                const unsigned long long off = gbase[NVO + o] + p;
                if (off < (unsigned long long)a.bucket_cap) g.nbucket[(size_t)o * a.bucket_cap + off] = row.x;
                else gen_direct_apply(g, row.x, 0ull, 0ull, 1ull, 0, 0);
            }
        }
        for (int j = tid; j < C; j += SPG_TTHREADS) hist[j] = 0;
        __syncthreads();
    }
    if (tid == 0 && (na_cnt[0] | na_cnt[1])) {  // NA-key group (slot cap of the state's table)
        a.counters[3] = 1;
        gen_apply_slot(g.fl, a.cap, *na_sum, (unsigned long long)na_cnt[0], (unsigned long long)na_cnt[1], *na_min, *na_max);
    }
}

// K2g: one CTA per owner; slot = key, low sum word (biased, see spg_aggregate_kernel), count [, min, max] [, NA-value rows].
template <bool HAS_SUM, bool HAS_MM, bool HAS_NN>
__global__ void __launch_bounds__(SPG_THREADS, 1) spgg_aggregate_kernel(const __grid_constant__ SpgGenArgs g) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SpgArgs& a = g.s;
    const int NS = a.ns, NT = a.ns + SPG_STASH, tid = threadIdx.x, me = blockIdx.x;
    long long* skeys = (long long*)smem_raw;
    long long* smin = skeys + NT;                                  // HAS_MM only
    long long* smax = smin + (HAS_MM ? NT : 0);
    unsigned int* slo = (unsigned int*)(smax + (HAS_MM ? NT : 0));
    unsigned int* scnt = slo + NT;
    unsigned int* snull = scnt + NT;                               // HAS_NN only
    const unsigned int NB = (unsigned int)NS / 2;
    const unsigned int NP = (unsigned int)a.n_pass, GP = (unsigned int)gridDim.x * NP;
    const bool VO = g.n_vo != a.n_owners;  // bucket me * NP + pass holds exactly this pass's rows
    const bool CHK = NP > 1 && !VO;        // else every row of the owner's bucket is tested against the pass

    auto add = [&](int s, long long key, long long val) {
        if (HAS_SUM) {
            unsigned int lo = (unsigned int)(unsigned long long)val, hi = (unsigned int)((unsigned long long)val >> 32);
            unsigned int old = atomicAdd(&slo[s], lo);
            hi += (old + lo < old) ? 1u : 0u;
            if (hi) gen_direct_apply(g, key, (unsigned long long)hi << 32, 0ull, 0ull, 0, 0);
        }
        atomicAdd(&scnt[s], 1u);
        if (HAS_MM) {
            if (val < smin[s]) atomicMin(&smin[s], val);
            if (val > smax[s]) atomicMax(&smax[s], val);
        }
    };
    auto slow_upsert = [&](long long key, long long val) {
        const int s = spg_slow_slot(skeys, NS, NB, key);
        if (s < 0) { gen_direct_apply(g, key, (unsigned long long)val, 1ull, 0ull, val, val); return; }
        add(s, key, val);
    };

    unsigned long long n_in = 0;
    unsigned long long n_null = g.nbucket ? a.bucket_cnt[(g.n_vo + me) * SPG_CNT_STRIDE] : 0ull;
    if (n_null > (unsigned long long)a.bucket_cap) n_null = (unsigned long long)a.bucket_cap;
    const longlong2* src = nullptr;
    const long long* nsrc = g.nbucket ? g.nbucket + (size_t)me * a.bucket_cap : nullptr;
    constexpr int U = 4;
    auto process = [&](unsigned long long first, unsigned int pass, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        longlong2 row[U];
        int sl[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            unsigned long long p = first + (unsigned long long)u * SPG_THREADS;
            row[u] = (FULL || p < n_in) ? __ldcs(src + p) : make_longlong2(EMPTY_KEY, 0);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            unsigned int b1, b2;
            spg_buckets(spg_hash(row[u].x), NB, b1, b2);
            const ulonglong2 k1 = *reinterpret_cast<const ulonglong2*>(skeys + 2 * b1);
            const ulonglong2 k2 = *reinterpret_cast<const ulonglong2*>(skeys + 2 * b2);
            sl[u] = spg_find_slot(k1, k2, b1, b2, (unsigned long long)row[u].x);
            if (!FULL && row[u].x == EMPTY_KEY) sl[u] = -2;
            if (CHK && __umulhi((unsigned int)(spg_hash(row[u].x) >> 32), GP) - (unsigned int)me * NP != pass) sl[u] = -2;
        }
        long long pk = 0, pv = 0;
        bool parked = false;
#pragma unroll
        for (int u = 0; u < U; u++) {
            if (sl[u] >= 0) add(sl[u], row[u].x, row[u].y);
            else if (sl[u] == -1) {
                if (!parked) { pk = row[u].x; pv = row[u].y; parked = true; }
                else slow_upsert(row[u].x, row[u].y);
            }
        }
        if (parked) slow_upsert(pk, pv);
    };
    const unsigned long long step = (unsigned long long)U * SPG_THREADS;
    for (unsigned int pass = 0; pass < NP; pass++) {
        const unsigned int bi = VO ? (unsigned int)me * NP + pass : (unsigned int)me;
        n_in = a.bucket_cnt[bi * SPG_CNT_STRIDE];
        if (n_in > (unsigned long long)a.bucket_cap) n_in = (unsigned long long)a.bucket_cap;
        src = a.bucket + (size_t)bi * a.bucket_cap;
        const unsigned long long n_full = n_in / step * step;
        for (int s = tid; s < NT; s += SPG_THREADS) {
            skeys[s] = EMPTY_KEY; slo[s] = 0x80000000u; scnt[s] = 0;
            if (HAS_MM) { smin[s] = INT64_MAX; smax[s] = INT64_MIN; }
            if (HAS_NN) snull[s] = 0;
        }
        __syncthreads();
        for (unsigned long long base = 0; base < n_full; base += step) process(base + tid, pass, std::true_type{});
        if (n_full < n_in) process(n_full + tid, pass, std::false_type{});
        // rows whose value is NA: the group has to exist (and the row counts for `size`)
        for (unsigned long long p = tid; p < n_null; p += SPG_THREADS) {
            const long long key = __ldcs(nsrc + p);
            if (NP > 1 && __umulhi((unsigned int)(spg_hash(key) >> 32), GP) - (unsigned int)me * NP != pass) continue;
            const int s = spg_slow_slot(skeys, NS, NB, key);  // looks the four candidates up first
            if (s < 0) gen_direct_apply(g, key, 0ull, 0ull, 1ull, 0, 0);
            else if (HAS_NN) atomicAdd(&snull[s], 1u);
        }
        __syncthreads();
        for (int s = tid; s < NT; s += SPG_THREADS) {
            long long key = skeys[s];
            if (key == EMPTY_KEY) continue;
            unsigned long long sum = HAS_SUM ? (unsigned long long)slo[s] - 0x80000000ull : 0ull;
            gen_direct_apply(g, key, sum, (unsigned long long)scnt[s], HAS_NN ? (unsigned long long)snull[s] : 0ull, HAS_MM ? smin[s] : 0, HAS_MM ? smax[s] : 0);
        }
        __syncthreads();
    }
}
