// spg_harness.cu — times the SPG kernel pair (K1 spg_partition_tma_kernel, K2 spg_aggregate_kernel) in isolation, outside
// the operator state machine, so a kernel change can be timed with one short GPU run.  Development tool, not part
// of the library: it includes groupby.cu to reach the kernels and links misc.cu for the buffer pool.
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -I bodo_b200/csrc \
//        scratch/spg_harness.cu bodo_b200/csrc/misc.cu -o scratch/spg_harness
//   scratch/spg_harness [log2_rows=27] [groups=1000000] [reps=5] [cnt_stride_pad_bytes=0]
//
// Prints per-kernel CUDA-event times (min / median over reps), the achieved fraction of the 16 B/row stream roofline for the
// pair, and checks SUM/COUNT totals against the input (result must be exact).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../bodo_b200/csrc/groupby.cu"

using namespace b200;

__global__ void harness_fill_kernel(long long* keys, long long* vals, int64_t n, uint64_t n_groups) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        keys[i] = (long long)(mix64((uint64_t)i ^ 0x9e3779b97f4a7c15ULL) % n_groups);
        vals[i] = (long long)(mix64((uint64_t)i ^ 0xd1b54a32d192ed03ULL * 2) % 1000) - 500;
    }
}
__global__ void harness_fill_u64(unsigned long long* p, size_t n, unsigned long long v) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void harness_sum_kernel(const long long* v, int64_t n, unsigned long long* out) {
    unsigned long long s = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s += (unsigned long long)v[i];
    atomicAdd(out, s);
}

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); exit(1); } } while (0)

int main(int argc, char** argv) {
    const int lg = argc > 1 ? atoi(argv[1]) : 27;
    const uint64_t groups = argc > 2 ? strtoull(argv[2], nullptr, 10) : 1000000ull;
    const int reps = argc > 3 ? atoi(argv[3]) : 5;
    const size_t pad = argc > 4 ? strtoull(argv[4], nullptr, 10) : 0;  // shifts the owner row counters inside their allocation
    const int64_t rows = 1ll << lg;
    int dev = 0, sms = 0, max_smem = 0;
    CK(cudaSetDevice(dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CK(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const int owners = sms;
    int ns = ((int)(((size_t)max_smem - 64) / 16) - SPG_STASH) & ~1;
    const size_t k2_smem = (size_t)(ns + SPG_STASH) * 16 + 16;
    const size_t k1_smem = GroupbyState::spg_tma_smem();
    const int64_t n_tiles = (rows + SPG_TILE - 1) / SPG_TILE;
    const int g1 = (int)std::min<int64_t>((int64_t)sms * SPG_TCTAS, n_tiles);

    long long *keys, *vals, *tkeys, *counters;
    unsigned long long *acc_sum, *acc_cnt, *bucket_cnt_raw, *retry, *chk;
    longlong2* bucket;
    const uint64_t cap = 1ull << 22;
    CK(cudaMalloc(&keys, rows * 8)); CK(cudaMalloc(&vals, rows * 8));
    CK(cudaMalloc(&tkeys, (cap + 2) * 8)); CK(cudaMalloc(&acc_sum, (cap + 2) * 8)); CK(cudaMalloc(&acc_cnt, (cap + 2) * 8));
    CK(cudaMalloc(&counters, 64)); CK(cudaMalloc(&chk, 16));
    const int64_t bucket_cap = rows / owners + rows / owners / 8 + 4096;
    CK(cudaMalloc(&bucket, (size_t)owners * bucket_cap * 16));
    CK(cudaMalloc(&bucket_cnt_raw, (size_t)owners * SPG_CNT_STRIDE * 8 + pad + 256));
    CK(cudaMalloc(&retry, ((size_t)rows + (size_t)owners * ns) * 32));
    unsigned long long* bucket_cnt = (unsigned long long*)((char*)bucket_cnt_raw + pad);
    harness_fill_kernel<<<sms * 8, 256>>>(keys, vals, rows, groups);
    harness_fill_u64<<<sms * 8, 256>>>((unsigned long long*)tkeys, cap + 2, (unsigned long long)EMPTY_KEY);
    CK(cudaMemset(acc_sum, 0, (cap + 2) * 8)); CK(cudaMemset(acc_cnt, 0, (cap + 2) * 8)); CK(cudaMemset(counters, 0, 64));
    CK(cudaDeviceSynchronize());

    SpgArgs a{};
    a.keys = keys; a.vals = vals; a.n_rows = rows; a.n_owners = owners;
    a.tkeys = tkeys; a.cap = cap; a.acc_sum = acc_sum; a.acc_cnt = acc_cnt; a.counters = counters; a.group_limit = (long long)(cap / 2);
    a.bucket = bucket; a.bucket_cnt = bucket_cnt; a.bucket_cap = bucket_cap; a.retry = retry; a.retry_ctr = counters + 1;
    a.sum_first = 1; a.ns = ns; a.n_pass = 1;

    CK(cudaFuncSetAttribute((const void*)spg_partition_tma_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1_smem));
    CK(cudaFuncSetAttribute((const void*)spg_aggregate_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k2_smem));

    std::vector<float> t1, t2;
    cudaEvent_t e0, e1, e2;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); CK(cudaEventCreate(&e2));
    for (int r = 0; r < reps + 1; r++) {  // the first repetition (table inserts, cold) is not reported
        CK(cudaMemsetAsync(bucket_cnt, 0, (size_t)owners * SPG_CNT_STRIDE * 8));
        CK(cudaEventRecord(e0));
        spg_partition_tma_kernel<true, true><<<g1, SPG_TTHREADS, k1_smem>>>(a);
        CK(cudaEventRecord(e1));
        spg_aggregate_kernel<true, true><<<owners, SPG_THREADS, k2_smem>>>(a);
        CK(cudaEventRecord(e2));
        CK(cudaEventSynchronize(e2));
        CK(cudaGetLastError());
        float a1 = 0, a2 = 0;
        CK(cudaEventElapsedTime(&a1, e0, e1)); CK(cudaEventElapsedTime(&a2, e1, e2));
        if (r > 0) { t1.push_back(a1); t2.push_back(a2); }
    }
    std::sort(t1.begin(), t1.end()); std::sort(t2.begin(), t2.end());
    // totals: SUM of sums and SUM of counts over the table must equal (reps + 1) x the input totals
    CK(cudaMemset(chk, 0, 16));
    harness_sum_kernel<<<sms * 4, 256>>>((const long long*)acc_cnt, (int64_t)cap + 2, chk);
    harness_sum_kernel<<<sms * 4, 256>>>((const long long*)acc_sum, (int64_t)cap + 2, chk + 1);
    unsigned long long h[2], hin = 0, *din;
    CK(cudaMemcpy(h, chk, 16, cudaMemcpyDeviceToHost));
    CK(cudaMalloc(&din, 8)); CK(cudaMemset(din, 0, 8));
    harness_sum_kernel<<<sms * 4, 256>>>(vals, rows, din);
    CK(cudaMemcpy(&hin, din, 8, cudaMemcpyDeviceToHost));
    long long hc[8];
    CK(cudaMemcpy(hc, counters, 64, cudaMemcpyDeviceToHost));
    const bool ok = h[0] == (unsigned long long)rows * (reps + 1) && h[1] == hin * (unsigned long long)(reps + 1) && hc[1] == 0;
    const float m1 = t1[t1.size() / 2], m2 = t2[t2.size() / 2];
    printf("{\"rows\": %lld, \"groups\": %llu, \"k1_ms\": {\"min\": %.4f, \"median\": %.4f}, \"k2_ms\": {\"min\": %.4f, \"median\": %.4f}, "
           "\"pair_grows_per_s\": %.2f, \"roofline_frac\": %.4f, \"table_groups\": %lld, \"retry_rows\": %lld, \"check\": \"%s\"}\n",
           (long long)rows, (unsigned long long)groups, t1[0], m1, t2[0], m2, rows / ((m1 + m2) * 1e-3) / 1e9,
           rows * 16.0 / ((m1 + m2) * 1e-3) / 6574.8e9, hc[0], hc[1], ok ? "ok" : "MISMATCH");
    return ok ? 0 : 3;
}
