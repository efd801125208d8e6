// SPG-N: the SM-partitioned groupby kernels (groupby.cu, "SM-partitioned groupby") with NARROW bucket rows.
// Included by groupby.cu only.
//
// The two-kernel path moves 48 B/row through HBM: 16 read + 16 bucket write + 16 bucket read.  When a row's key and value both
// fit 32 bits (dictionary codes, dates, small integers — decided per ROW, sampled per operator state so the variant is only
// chosen when it pays) the owner bucket carries the row as an (int32 key, int32 value) pair: 16 + 8 + 8 = 32 B/row, K1n stages
// and copies out half the bytes, and K2n's shared table shrinks to 12-byte slots (int32 key, low sum word, count) whose
// two-slot buckets are ONE 8-byte shared load each, with 32-bit key compares.  Rows that do not fit (either value outside
// int32, or the key INT32_MIN, which marks a free slot) take the direct global path inside K1n, so the result is exact for any
// input; a.counters[5] counts them and the host drops back to the 16-byte kernels when they are not rare.
// Sums stay exact mod 2^64: the sign-extended value is added as (low word, high word + carry) exactly as in spg_aggregate_kernel.
#pragma once

constexpr int SPGN_EMPTY = (int)0x80000000;
constexpr int SPGN_TILE = 4096;  // rows per K1n tile (8-byte staged rows leave room for twice the 16-byte kernels' tile)
constexpr int SPGN_CTAS = 2;     // K1n CTAs per SM

// find-or-insert for a caller that already holds a group ticket: `inserted` says whether THIS call created the group (else the
// ticket goes back).  The table cannot be full: tickets bound the number of groups by cap / 2.
__device__ __forceinline__ uint64_t spgn_insert_ticketed(long long* __restrict__ tkeys, uint64_t cap, long long key, bool& inserted) {
    const uint64_t mask = cap - 1;
    uint64_t s = (key_hash(key) >> 32) & mask;
    inserted = false;
    while (true) {
        long long k = __ldcg(tkeys + s);
        if (k == EMPTY_KEY) {
            k = (long long)atomicCAS((unsigned long long*)(tkeys + s), (unsigned long long)EMPTY_KEY, (unsigned long long)key);
            if (k == EMPTY_KEY) { inserted = true; return s; }
        }
        if (k == key) return s;
        s = (s + 1) & mask;
    }
}

template <bool HAS_SUM, bool HAS_CNT>
__global__ void __launch_bounds__(SPG_TTHREADS, SPGN_CTAS) spgn_partition_kernel(const __grid_constant__ SpgArgs a) {
    extern __shared__ __align__(128) unsigned char smem_n_raw[];
    long long* raw_k = (long long*)smem_n_raw;                                 // [SPGN_TILE] keys
    long long* raw_v = raw_k + SPGN_TILE;                                       // [SPGN_TILE] values
    int2* stage = (int2*)(raw_v + SPGN_TILE);                                   // SPGN_TILE x 8
    unsigned long long* gbase = (unsigned long long*)(stage + SPGN_TILE);      // SPG_MAX_OWNERS x 8
    uint64_t* mbar = (uint64_t*)(gbase + SPG_MAX_OWNERS);                      // 2 mbarriers (one used)
    unsigned int* hist = (unsigned int*)(mbar + 2);                            // SPG_MAX_OWNERS
    unsigned int* lbase = hist + SPG_MAX_OWNERS;                               // SPG_MAX_OWNERS + 1
    unsigned char* stage_owner = (unsigned char*)(lbase + SPG_MAX_OWNERS + 4);  // SPGN_TILE
    int2** dptr = (int2**)(stage_owner + SPGN_TILE);                            // SPG_MAX_OWNERS: run start - local start, as an address
    unsigned int* tile_over = (unsigned int*)(dptr + SPG_MAX_OWNERS);           // some run of this tile does not fit its bucket
    const int G = a.n_owners, tid = threadIdx.x;
    constexpr int ROWS = SPGN_TILE / SPG_TTHREADS;
    const int64_t n_tiles = (a.n_rows + SPGN_TILE - 1) / SPGN_TILE;
    int2* bucket = reinterpret_cast<int2*>(a.bucket);
    unsigned int wide = 0;
    if (tid == 0) {
        mbar_init(&mbar[0], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        *tile_over = 0;
    }
    for (int j = tid; j < G; j += SPG_TTHREADS) hist[j] = 0;
    __syncthreads();
    auto issue = [&](int64_t t) {
        const int64_t r0 = t * SPGN_TILE;
        if (r0 + SPGN_TILE <= a.n_rows && tid == 0) {
            mbar_expect_tx(&mbar[0], (HAS_SUM ? 2u : 1u) * SPGN_TILE * 8u);
            tma_load_1d(raw_k, a.keys + r0, SPGN_TILE * 8u, &mbar[0]);
            if (HAS_SUM) tma_load_1d(raw_v, a.vals + r0, SPGN_TILE * 8u, &mbar[0]);
        }
    };
    uint32_t phase = 0;
    int64_t t = blockIdx.x;
    if (t < n_tiles) issue(t);
    for (; t < n_tiles; t += gridDim.x) {
        const int64_t r0 = t * SPGN_TILE;
        const int64_t tn = t + gridDim.x;
        const bool full = r0 + SPGN_TILE <= a.n_rows;
        if (full) {
            while (!mbar_try_wait(&mbar[0], phase)) {}
            phase ^= 1;
        } else {
            for (int j = tid; j < SPGN_TILE; j += SPG_TTHREADS) {
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
            if (!full && r0 + j >= a.n_rows) continue;
            const long long k = raw_k[j];
            const long long v = HAS_SUM ? raw_v[j] : 0;
            // both values inside int32 <=> the high words of (x + 2^31) are zero; the key INT32_MIN (low word of k + 2^31 zero) is excluded
            const unsigned long long kb = (unsigned long long)k + 0x80000000ull, vb = (unsigned long long)v + 0x80000000ull;
            const bool narrow = ((kb | vb) >> 32) == 0 && (unsigned int)kb != 0u;
            if (!narrow) { spg_direct_apply<HAS_SUM, HAS_CNT>(a, k, (unsigned long long)v, 1ull); wide++; continue; }
            o[r] = (int)spg_owner(spg_hash(k), G);
            rk[r] = atomicAdd(&hist[o[r]], 1u);
        }
        __syncthreads();
        unsigned long long my_gbase = 0;
        unsigned int my_cnt = 0;
        if (tid >= SPG_TTHREADS - G) { int ow = tid - (SPG_TTHREADS - G); my_cnt = hist[ow]; if (my_cnt) my_gbase = atomicAdd(&a.bucket_cnt[ow * SPG_CNT_STRIDE], (unsigned long long)my_cnt); }
        spg_scan_hist(hist, lbase, G, tid);
        __syncthreads();
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
            if (o[r] < 0) continue;
            const int j = r * SPG_TTHREADS + tid;
            const unsigned int p = lbase[o[r]] + rk[r];
            stage[p] = make_int2((int)raw_k[j], HAS_SUM ? (int)raw_v[j] : 0);
            stage_owner[p] = (unsigned char)o[r];
        }
        if (tid >= SPG_TTHREADS - G) {
            const int ow = tid - (SPG_TTHREADS - G);
            gbase[ow] = my_gbase - lbase[ow];
            dptr[ow] = bucket + ((size_t)ow * a.bucket_cap + my_gbase - lbase[ow]);  // staged position p of this owner's run goes to dptr[ow][p]
            if (my_gbase + my_cnt > (unsigned long long)a.bucket_cap) *tile_over = 1;
        }
        __syncthreads();  // the raw tile is free from here on
        if (tn < n_tiles) issue(tn);
        const unsigned int n_tile = lbase[G];
        if (*tile_over == 0) {  // every run fits (the common case): one owner byte, one address and one 8-byte store per row
            unsigned int p = tid;
            for (; p + SPG_TTHREADS < n_tile; p += 2 * SPG_TTHREADS) {
                const unsigned int o0 = stage_owner[p], o1 = stage_owner[p + SPG_TTHREADS];
                const int2 r0v = stage[p], r1v = stage[p + SPG_TTHREADS];
                dptr[o0][p] = r0v;
                dptr[o1][p + SPG_TTHREADS] = r1v;
            }
            if (p < n_tile) dptr[stage_owner[p]][p] = stage[p];
        } else {
            for (unsigned int p = tid; p < n_tile; p += SPG_TTHREADS) {
                const unsigned int ow = stage_owner[p];
                const unsigned long long off = gbase[ow] + p;
                const int2 row = stage[p];
                if (off < (unsigned long long)a.bucket_cap) bucket[(size_t)ow * a.bucket_cap + off] = row;
                else spg_direct_apply<HAS_SUM, HAS_CNT>(a, (long long)row.x, (unsigned long long)(long long)row.y, 1ull);  // bucket full (skew)
            }
        }
        __syncthreads();  // (tile_over is read above, cleared below)
        for (int j = tid; j < G; j += SPG_TTHREADS) hist[j] = 0;
        if (tid == 0) *tile_over = 0;
        __syncthreads();
    }
    if (wide) atomicAdd((unsigned long long*)&a.counters[5], (unsigned long long)wide);
}

// K2n: slot = int32 key, low sum word (biased by 2^31), count.
template <bool HAS_SUM, bool HAS_CNT>
__global__ void __launch_bounds__(SPG_THREADS, 1) spgn_aggregate_kernel(const __grid_constant__ SpgArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NS = a.ns, NT = a.ns + SPG_STASH, tid = threadIdx.x, me = blockIdx.x;
    int* skeys = (int*)smem_raw;                      // NT x 4
    unsigned int* slo = (unsigned int*)(skeys + NT);  // NT x 4
    unsigned int* scnt = slo + NT;
    const unsigned int NB = (unsigned int)NS / 2;
    const unsigned int NP = (unsigned int)a.n_pass, GP = (unsigned int)gridDim.x * NP;

    auto add = [&](int s, int key, int val) {
        if (HAS_SUM) {
            const unsigned int lo = (unsigned int)val;
            unsigned int hi = val < 0 ? 0xffffffffu : 0u;
            const unsigned int old = atomicAdd(&slo[s], lo);
            hi += (old + lo < old) ? 1u : 0u;
            if (hi) spg_direct_apply<HAS_SUM, HAS_CNT>(a, (long long)key, (unsigned long long)hi << 32, 0ull);
        }
        if (HAS_CNT) atomicAdd(&scnt[s], 1u);
    };
    // spg_slow_slot for 32-bit keys, written out: calling a shared 32-bit instantiation of it changed the register allocation
    // of the count-only kernel (53 -> 55 registers)
    auto slow_upsert = [&](int key, int val) {
        unsigned int b1, b2;
        spg_buckets(spg_hash((long long)key), NB, b1, b2);
        const int2 c1 = *reinterpret_cast<const int2*>(skeys + 2 * b1);
        const int2 c2 = *reinterpret_cast<const int2*>(skeys + 2 * b2);
        const int f1 = (c1.x == SPGN_EMPTY) + (c1.y == SPGN_EMPTY), f2 = (c2.x == SPGN_EMPTY) + (c2.y == SPGN_EMPTY);
        int s = spg_find_slot(c1, c2, b1, b2, key);
        if (s < 0 && f1 + f2 > 0) {
            const unsigned int first = f2 > f1 ? b2 : b1, second = f2 > f1 ? b1 : b2;
            const unsigned int cand[4] = {2 * first, 2 * first + 1, 2 * second, 2 * second + 1};
#pragma unroll
            for (int c = 0; c < 4 && s < 0; c++) {
                const int old = atomicCAS(&skeys[cand[c]], SPGN_EMPTY, key);
                if (old == SPGN_EMPTY || old == key) s = (int)cand[c];
            }
        }
        if (s < 0) {
            unsigned int st = (unsigned int)NS + ((unsigned int)(spg_hash((long long)key) >> 12) & (SPG_STASH - 1));
            for (int probes = 0; probes < SPG_STASH && s < 0; probes++) {
                int kk = skeys[st];
                if (kk == SPGN_EMPTY) {
                    const int old = atomicCAS(&skeys[st], SPGN_EMPTY, key);
                    if (old == SPGN_EMPTY) { s = (int)st; break; }
                    kk = old;
                }
                if (kk == key) { s = (int)st; break; }
                st = st + 1 == (unsigned int)NS + SPG_STASH ? (unsigned int)NS : st + 1;
            }
        }
        if (s < 0) { spg_direct_apply<HAS_SUM, HAS_CNT>(a, (long long)key, (unsigned long long)(long long)val, 1ull); return; }
        add(s, key, val);
    };

    unsigned long long n_in = a.bucket_cnt[me * SPG_CNT_STRIDE];
    if (n_in > (unsigned long long)a.bucket_cap) n_in = (unsigned long long)a.bucket_cap;
    const int2* src = reinterpret_cast<const int2*>(a.bucket) + (size_t)me * a.bucket_cap;  // bucket_cap is even: 16-byte aligned
    constexpr int U = 4;  // rows per thread per iteration, as two 16-byte loads of two adjacent rows
    // unit = two adjacent rows; units of this thread: first + j * SPG_THREADS, j = 0 .. U/2 - 1
    // rows of one iteration: U/2 units of two adjacent rows, unit index first + j * SPG_THREADS
    auto load_rows = [&](unsigned long long first, int2 (&row)[U], auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
#pragma unroll
        for (int j = 0; j < U / 2; j++) {
            const unsigned long long r = 2 * (first + (unsigned long long)j * SPG_THREADS);
            row[2 * j] = row[2 * j + 1] = make_int2(SPGN_EMPTY, 0);
            if (FULL || r + 1 < n_in) {
                const int4 q = __ldcs(reinterpret_cast<const int4*>(src + r));
                row[2 * j] = make_int2(q.x, q.y); row[2 * j + 1] = make_int2(q.z, q.w);
            } else if (r < n_in) row[2 * j] = __ldcs(src + r);
        }
    };
    auto process = [&](const int2 (&row)[U], unsigned int pass, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        int sl[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t h = spg_hash((long long)row[u].x);
            unsigned int b1, b2;
            spg_buckets(h, NB, b1, b2);
            const int2 k1 = *reinterpret_cast<const int2*>(skeys + 2 * b1);
            const int2 k2 = *reinterpret_cast<const int2*>(skeys + 2 * b2);
            const int key = row[u].x;
            sl[u] = spg_find_slot(k1, k2, b1, b2, key);
            if (!FULL && key == SPGN_EMPTY) sl[u] = -2;  // padding lane (INT32_MIN never reaches a bucket)
            if (NP > 1 && __umulhi((unsigned int)(h >> 32), GP) - (unsigned int)me * NP != pass) sl[u] = -2;
        }
        int pk = 0, pv = 0;
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
    const unsigned long long ustep = (unsigned long long)(U / 2) * SPG_THREADS;   // units per CTA iteration
    const unsigned long long full_units = n_in / (2 * ustep) * ustep;              // iterations whose rows are all in range
    for (unsigned int pass = 0; pass < NP; pass++) {
        for (int s = tid; s < NT; s += SPG_THREADS) { skeys[s] = SPGN_EMPTY; slo[s] = 0x80000000u; scnt[s] = 0; }
        __syncthreads();
        // software pipeline: the next iteration's bucket rows are in flight while the current ones are aggregated (the wait for these
        // loads was the largest single stall of the unpipelined loop, 20 % of the samples)
        if (full_units > 0) {
            int2 cur[U], nxt[U];
            load_rows(tid, cur, std::true_type{});
            for (unsigned long long ub = 0; ub < full_units; ub += ustep) {
                if (ub + ustep < full_units) load_rows(ub + ustep + tid, nxt, std::true_type{});
                process(cur, pass, std::true_type{});
#pragma unroll
                for (int u = 0; u < U; u++) cur[u] = nxt[u];
            }
        }
        for (unsigned long long ub = full_units; 2 * ub < n_in; ub += ustep) {
            int2 tail[U];
            load_rows(ub + tid, tail, std::false_type{});
            process(tail, pass, std::false_type{});
        }
        __syncthreads();
        // flush.  First flush of a state (empty global table, a.reserve_tickets): every occupied slot is a NEW group, and 10^6
        // per-insert tickets on one counter cost ~0.2 ms — the CTA takes the tickets of all its slots with ONE atomic and returns
        // the few it did not need (a key that sits in two slots, or that the direct path inserted meanwhile).
        __shared__ unsigned int fl_occ, fl_dup;
        __shared__ int fl_reserved;
        if (tid == 0) { fl_occ = 0; fl_dup = 0; fl_reserved = 0; }
        __syncthreads();
        if (a.reserve_tickets && a.group_limit >= 0) {
            unsigned int mine = 0;
            for (int s = tid; s < NT; s += SPG_THREADS) mine += skeys[s] != SPGN_EMPTY;
            for (int d = 16; d; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
            if ((tid & 31) == 0 && mine) atomicAdd(&fl_occ, mine);
            __syncthreads();
            if (tid == 0 && fl_occ) {
                const long long t = (long long)atomicAdd((unsigned long long*)&a.counters[0], (unsigned long long)fl_occ);
                if (t + (long long)fl_occ <= a.group_limit) fl_reserved = 1;
                else atomicAdd((unsigned long long*)&a.counters[0], (unsigned long long)(-(long long)fl_occ));  // no room: per-insert tickets
            }
            __syncthreads();
        }
        const bool reserved = fl_reserved != 0;
        unsigned int dup = 0;
        for (int s = tid; s < NT; s += SPG_THREADS) {
            const int key = skeys[s];
            if (key == SPGN_EMPTY) continue;
            const unsigned long long sum = (unsigned long long)slo[s] - 0x80000000ull;  // remove the bias (wraps mod 2^64)
            if (!reserved) { spg_direct_apply<HAS_SUM, HAS_CNT>(a, (long long)key, sum, (unsigned long long)scnt[s]); continue; }
            // ticket already held: insert without the limit; a key that was there already gives its ticket back
            bool inserted;
            const uint64_t sl = spgn_insert_ticketed(a.tkeys, a.cap, (long long)key, inserted);
            if (!inserted) dup++;
            if (HAS_SUM && sum) atomicAdd(a.acc_sum + sl, sum);
            if (HAS_CNT && scnt[s]) atomicAdd(a.acc_cnt + sl, (unsigned long long)scnt[s]);
        }
        if (reserved) {
            for (int d = 16; d; d >>= 1) dup += __shfl_xor_sync(0xffffffffu, dup, d);
            if ((tid & 31) == 0 && dup) atomicAdd(&fl_dup, dup);
            __syncthreads();
            if (tid == 0 && fl_dup) atomicAdd((unsigned long long*)&a.counters[0], (unsigned long long)(-(long long)fl_dup));
        }
        __syncthreads();
    }
}
