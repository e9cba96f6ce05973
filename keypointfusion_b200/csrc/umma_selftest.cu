// Self-test of the tcgen05 building blocks in tcgen05.cuh: one 128 x N x K bf16 GEMM through shared-memory descriptors
// (K-major and MN-major operands), TMEM accumulation and tcgen05.ld read-back.  Used by tests/test_umma_gpu.py.
#include "tcgen05.cuh"

namespace kpf {

__global__ void __launch_bounds__(128)
umma_selftest_kernel(const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ Bm, float* __restrict__ D, int N, int K,
                     int a_mn, int b_mn) {
    extern __shared__ __align__(128) unsigned char sm[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    uint4* sA = reinterpret_cast<uint4*>(sm);                       // 128*K*2 bytes
    uint4* sB = reinterpret_cast<uint4*>(sm + (size_t)128 * K * 2);  // N*K*2 bytes
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    if (tid == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
    }
    // ---- stage A
    if (!a_mn) {  // A given [128][K] row-major -> K-major canonical smem[K/8][128]
        for (int i = tid; i < 128 * (K / 8); i += blockDim.x) {
            const int r = i % 128, kc = i / 128;
            sA[kc * 128 + r] = *reinterpret_cast<const uint4*>(A + (size_t)r * K + kc * 8);
        }
    } else {      // A given [K][128] (M contiguous) -> MN-major canonical smem[K/8][128/8][8]
        for (int i = tid; i < K * 16; i += blockDim.x) {
            const int m8 = i % 16, k = i / 16;
            sA[(k / 8) * 128 + m8 * 8 + (k % 8)] = *reinterpret_cast<const uint4*>(A + (size_t)k * 128 + m8 * 8);
        }
    }
    // ---- stage B
    if (!b_mn) {  // B given [N][K] row-major
        for (int i = tid; i < N * (K / 8); i += blockDim.x) {
            const int r = i % N, kc = i / N;
            sB[kc * N + r] = *reinterpret_cast<const uint4*>(Bm + (size_t)r * K + kc * 8);
        }
    } else {      // B given [K][N] (N contiguous)
        for (int i = tid; i < K * (N / 8); i += blockDim.x) {
            const int n8 = i % (N / 8), k = i / (N / 8);
            sB[(k / 8) * N + n8 * 8 + (k % 8)] = *reinterpret_cast<const uint4*>(Bm + (size_t)k * N + n8 * 8);
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    if (tid == 0) {
        const SmemOp a = smem_op_k_outer(smem_u32(sA), 128, K), b = smem_op_k_outer(smem_u32(sB), N, K);   // either major
        umma_gemm(tmem, a.hi, a.lbo, a.sbo, b.hi, b.lbo, b.sbo, umma_idesc_f16(128, N, a_mn != 0, b_mn != 0, FMT_BF16, FMT_BF16), K, false);
        umma_commit(&bar);
    }
    mbar_wait(&bar, 0);
    tc_fence_after();
    const int row = tid;  // lane == row of D
    for (int c0 = 0; c0 < N; c0 += 32) {
        float v[32];
        tmem_ld<32>(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
        for (int i = 0; i < 32 && c0 + i < N; ++i) D[(size_t)row * N + c0 + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

}  // namespace kpf

extern "C" int kpf_umma_selftest(const void* A, const void* B, float* D, int N, int K, int a_mn, int b_mn, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(N >= 16 && N <= 256 && N % 16 == 0 && K >= 16 && K % 16 == 0);
    const size_t smem = (size_t)(128 + N) * K * 2;
    KPF_REQUIRE(smem <= 200 * 1024);
    cudaError_t e = kpf::set_smem(umma_selftest_kernel, smem);
    if (e != cudaSuccess) return (int)e;
    umma_selftest_kernel<<<1, 128, smem, stream>>>((const __nv_bfloat16*)A, (const __nv_bfloat16*)B, D, N, K, a_mn, b_mn);
    KPF_CHECK_LAUNCH();
    return 0;
}
