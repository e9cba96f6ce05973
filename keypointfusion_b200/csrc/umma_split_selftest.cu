// Self-test + cycle probe of the split-precision GEMM forms in tcgen05.cuh (tests/test_umma_gpu.py):
//   D[128 x N] = A[128 x K] B[N x K]^T with fp32 A, B carried as (hi, lo) bf16 or fp16 planes, A from shared memory or
//   from tensor memory; optional "exact" A (hi plane only).  Also reports cycles of one GEMM and of eight back to back.
#include "tcgen05.cuh"

namespace kpf {

template <int FMT, int K>
__global__ void __launch_bounds__(128)
umma_split_selftest_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ D, int N, int a_tmem, int a_exact,
                           long long* cycles) {
    extern __shared__ __align__(128) unsigned char sm[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int warp_u = warp_index_uniform();
    constexpr int CH = K / 8;
    uint4* sAh = reinterpret_cast<uint4*>(sm);   // [K/8][128]
    uint4* sAl = sAh + CH * 128;
    uint4* sBh = sAl + CH * 128;                 // [K/8][N]
    uint4* sBl = sBh + CH * N;
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot, lane_base = tmem + ((uint32_t)(warp * 32) << 16);
    const uint32_t TA_HI = 256, TA_LO = 256 + 128;   // A planes in tensor memory (K / 2 <= 128 columns each)
    // ---- stage A: thread = row
    for (int kc = 0; kc < CH; ++kc) {
        float v[8];
        for (int i = 0; i < 8; ++i) v[i] = A[(size_t)tid * K + kc * 8 + i];
        uint4 hi, lo;
        split8<FMT>(v, hi, lo);
        if (a_tmem) {
            tmem_st_nw<4>(lane_base + TA_HI + kc * 4, reinterpret_cast<const float*>(&hi));
            tmem_st_nw<4>(lane_base + TA_LO + kc * 4, reinterpret_cast<const float*>(&lo));
        } else {
            sAh[kc * 128 + tid] = hi;
            sAl[kc * 128 + tid] = lo;
        }
    }
    if (a_tmem) tmem_wait_st();
    // ---- stage B
    for (int i = tid; i < N * CH; i += 128) {
        const int r = i % N, kc = i / N;
        float v[8];
        for (int k = 0; k < 8; ++k) v[k] = Bm[(size_t)r * K + kc * 8 + k];
        uint4 hi, lo;
        split8<FMT>(v, hi, lo);
        sBh[kc * N + r] = hi;
        sBl[kc * N + r] = lo;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t idesc = umma_idesc_f16(128, N, false, false, FMT, FMT);
    SmemOp a, b;
    a.hi = smem_u32(sAh); a.lo = a_exact ? 0u : smem_u32(sAl); a.lbo = 128 * 16; a.sbo = 128;
    b.hi = smem_u32(sBh); b.lo = smem_u32(sBl); b.lbo = (uint32_t)N * 16; b.sbo = 128;
    TmemOp at;
    at.hi = tmem + TA_HI; at.lo = a_exact ? NO_PLANE : tmem + TA_LO;
    uint32_t phase = 0;
    for (int reps = 1; reps <= 8; reps *= 8) {
        const long long t0 = clock64();
        if (warp_u == 0) {   // warp-uniform issue: one UTCHMMA per MMA (tcgen05.cuh)
            if (elect_one()) {
                for (int r = 0; r < reps; ++r) {
                    if (a_tmem) umma_gemm3_ts<K>(tmem, at, b, idesc, false);
                    else umma_gemm3_ss<K>(tmem, a, b, idesc, false);
                }
                umma_commit(&bar);
            }
            __syncwarp();
        }
        mbar_wait(&bar, phase);
        phase ^= 1;
        tc_fence_after();
        const long long t1 = clock64();
        if (tid == 0 && cycles) cycles[reps == 1 ? 0 : 1] = t1 - t0;
        __syncthreads();
    }
    for (int c0 = 0; c0 < N; c0 += 16) {
        float v[16];
        tmem_ld<16>(lane_base + c0, v);
        for (int i = 0; i < 16 && c0 + i < N; ++i) D[(size_t)tid * N + c0 + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

using SplitSelftestKernel = void (*)(const float*, const float*, float*, int, int, int, long long*);
template <int FMT>
SplitSelftestKernel split_selftest_kernel(int K) {
    switch (K) {
        case 16: return umma_split_selftest_kernel<FMT, 16>;
        case 32: return umma_split_selftest_kernel<FMT, 32>;
        case 64: return umma_split_selftest_kernel<FMT, 64>;
        case 128: return umma_split_selftest_kernel<FMT, 128>;
        case 256: return umma_split_selftest_kernel<FMT, 256>;
        default: return nullptr;
    }
}

}  // namespace kpf

extern "C" int kpf_umma_split_selftest(const float* A, const float* B, float* D, int N, int K, int fmt, int a_tmem, int a_exact,
                                       long long* cycles, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(N >= 16 && N <= 256 && N % 16 == 0);
    // K in {16, 32, 64, 128, 256}, fmt in {FMT_F16, FMT_BF16}: anything else has no kernel
    const SplitSelftestKernel kern = fmt == FMT_F16 ? split_selftest_kernel<FMT_F16>(K) : fmt == FMT_BF16 ? split_selftest_kernel<FMT_BF16>(K) : nullptr;
    KPF_REQUIRE(kern != nullptr);
    const size_t smem = (size_t)(128 + N) * K * 2 * 2;
    KPF_REQUIRE(smem <= 220 * 1024);
    cudaError_t e = kpf::set_smem(kern, smem);
    if (e != cudaSuccess) return (int)e;
    kern<<<1, 128, smem, stream>>>(A, B, D, N, a_tmem, a_exact, cycles);
    KPF_CHECK_LAUNCH();
    return 0;
}
