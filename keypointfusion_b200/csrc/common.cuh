// Shared device helpers for the KeypointFusion B200 kernels (sm_100a only).
#pragma once
#include <cstdlib>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kpf_b200.h"

#define KPF_CHECK_LAUNCH()                         \
    do {                                           \
        cudaError_t e__ = cudaGetLastError();      \
        if (e__ != cudaSuccess) return (int)e__;   \
    } while (0)

namespace kpf {
// Opt a kernel into `smem` bytes of dynamic shared memory and pin the L1/shared split at "max shared" so that
// back-to-back kernels of one step never ask the SM to re-partition its unified L1 between launches.
template <typename K>
inline cudaError_t set_smem(K* kernel, size_t smem) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
}  // namespace kpf

namespace kpf {
// Programmatic dependent launch (PDL).  A kernel started with launch_pdl() may begin while its predecessor in the stream is still
// running; everything it does before pdl_wait() must therefore (a) read only data no kernel writes (weights, the step's inputs)
// and (b) write nothing to global memory.  pdl_wait() returns once the predecessor grid has completed and its writes are
// visible.  EVERY kernel launched this way calls pdl_wait() before it exits -- completion of kernel k must imply completion of
// kernel k-1, or the chain of dependencies is broken for the kernels behind it.  pdl_launch_dependents() at the top lets the
// successor's CTAs take free SMs and run their own prologue (TMEM allocation, barrier init, weight TMA) early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
}  // namespace kpf

#define KPF_REQUIRE(cond)                          \
    do {                                           \
        if (!(cond)) return KPF_ERR_BAD_ARGUMENT;  \
    } while (0)

namespace kpf {

// ---- exact (non-contracted) arithmetic: the index-producing kernels must follow the oracle's operation
// ---- order bit for bit, so no FMA contraction on those paths.
__device__ __forceinline__ float xadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float xsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float xmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float xdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double xadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double xsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double xmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double xdiv(double a, double b) { return __ddiv_rn(a, b); }

// fp64 adjugate inverse of a row-major 3x3 (oracle: inv3x3_f64). Replaces np.linalg.inv (loader.py:882)
// and torch.linalg.inv (loader.py:781) -- no host sync, no LAPACK.
__device__ __forceinline__ void inv3x3_f64(const float* __restrict__ M, double* __restrict__ out) {
    const double a = M[0], b = M[1], c = M[2], d = M[3], e = M[4], f = M[5], g = M[6], h = M[7], i = M[8];
    const double A = xsub(xmul(e, i), xmul(f, h));
    const double Bc = xsub(xmul(f, g), xmul(d, i));
    const double C = xsub(xmul(d, h), xmul(e, g));
    const double det = xadd(xadd(xmul(a, A), xmul(b, Bc)), xmul(c, C));
    out[0] = xdiv(A, det);
    out[1] = xdiv(xsub(xmul(c, h), xmul(b, i)), det);
    out[2] = xdiv(xsub(xmul(b, f), xmul(c, e)), det);
    out[3] = xdiv(Bc, det);
    out[4] = xdiv(xsub(xmul(a, i), xmul(c, g)), det);
    out[5] = xdiv(xsub(xmul(c, d), xmul(a, f)), det);
    out[6] = xdiv(C, det);
    out[7] = xdiv(xsub(xmul(b, g), xmul(a, h)), det);
    out[8] = xdiv(xsub(xmul(a, e), xmul(b, d)), det);
}

// Per-sample camera / crop parameters in the fp32 form the uvd<->xyz transforms use.
struct CamF {
    float mi[6];      // first two rows of fl32(M^-1)
    float cx, cy, cz; // center (mm)
    float hx, hy, hz; // cube / 2
    float fx, fy, fu, fv;
    float hs;         // img_size / 2
    float flip;
};

__device__ __forceinline__ void load_cam(CamF& c, int b, const float* center, const float* M, const float* cube,
                                         const float* cam, float img_size, float flip) {
    double mi[9];
    inv3x3_f64(M + 9 * b, mi);
#pragma unroll
    for (int k = 0; k < 6; ++k) c.mi[k] = (float)mi[k];
    c.cx = center[3 * b + 0];
    c.cy = center[3 * b + 1];
    c.cz = center[3 * b + 2];
    c.hx = xdiv(cube[3 * b + 0], 2.0f);
    c.hy = xdiv(cube[3 * b + 1], 2.0f);
    c.hz = xdiv(cube[3 * b + 2], 2.0f);
    c.fx = cam[4 * b + 0];
    c.fy = cam[4 * b + 1];
    c.fu = cam[4 * b + 2];
    c.fv = cam[4 * b + 3];
    c.hs = xdiv(img_size, 2.0f);
    c.flip = flip;
}

// uvd (normalised) -> xyz (normalised).  dataloader/loader.py:775-789; oracle: uvd_nl2xyznl.
__device__ __forceinline__ float3 uvd2xyz(const CamF& c, float un, float vn, float dn) {
    const float u = xmul(xadd(un, 1.0f), c.hs);
    const float v = xmul(xadd(vn, 1.0f), c.hs);
    const float d = xadd(xmul(dn, c.hz), c.cz);
    const float xw = xadd(xadd(xmul(c.mi[0], u), xmul(c.mi[1], v)), c.mi[2]);
    const float yw = xadd(xadd(xmul(c.mi[3], u), xmul(c.mi[4], v)), c.mi[5]);
    const float X = xdiv(xmul(xsub(xw, c.fu), d), c.fx);
    const float Y = xdiv(xmul(xmul(c.flip, xsub(yw, c.fv)), d), c.fy);
    float3 o;
    o.x = xdiv(xsub(X, c.cx), c.hx);
    o.y = xdiv(xsub(Y, c.cy), c.hy);
    o.z = xdiv(xsub(d, c.cz), c.hz);
    return o;
}

// normalised cell-centre coordinate 2(i+.5)/fs-1 (model.py:477-481), fp32, fixed order
__device__ __forceinline__ float cell_coord(int i, float fs) {
    return xsub(xdiv(xmul(xadd((float)i, 0.5f), 2.0f), fs), 1.0f);
}

// nearest-neighbour source index of F.interpolate(img,[fs,fs]) (model.py:409): floor(dst * S/fs)
__device__ __forceinline__ int nearest_src(int dst, int S, int fs) {
    int s = (int)floorf((float)dst * ((float)S / (float)fs));
    return s < S - 1 ? s : S - 1;
}

// ---- dtype helpers --------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ---- reductions ------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// block-wide sum/max broadcast to all threads; `scratch` holds >= 32 floats; blockDim.x multiple of 32
__device__ __forceinline__ float block_sum(float v, float* scratch) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    float r = lane < nw ? scratch[lane] : 0.f;
    return warp_sum(r);
}
__device__ __forceinline__ float block_max(float v, float* scratch) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_max(v);
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    float r = lane < nw ? scratch[lane] : -INFINITY;
    return warp_max(r);
}

// ---- mbarrier + bulk-TMA (cp.async.bulk) helpers ---------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped launch (cudaErrorLaunchFailure), never as a hung GPU.
// try_wait may suspend the thread for an implementation-defined time, so the bound is on the clock, not the poll count.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000ll) __trap();  // ~2 s at 2 GHz
    }
}
// 1-D bulk copy global -> shared through the TMA engine (SASS: UBLKCP); bytes % 16 == 0, 16 B aligned.
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// 1-D bulk copy shared -> global through the TMA engine (SASS: UBLKCP), tracked per thread in bulk groups; bytes % 16 == 0, 16 B aligned
__device__ __forceinline__ void tma_bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N bulk groups still reading their shared-memory sources / still pending
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// ---- cp.async (SASS: LDGSTS): 16-byte copies global -> shared, waited for per thread ------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
// .cg: through L2 only; the bytes of the chunk past src_bytes (0..16) are zero filled
__device__ __forceinline__ void cp_async16_cg(void* smem_dst, const void* gmem_src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// at most N committed groups of this thread still pending
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// named barrier `id` (1..15; 0 is __syncthreads) over `nthreads` threads, a multiple of 32
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace kpf
