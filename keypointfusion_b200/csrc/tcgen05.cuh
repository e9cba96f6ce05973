// tcgen05 / TMEM primitives for sm_100a, hand-written inline PTX (no CUTLASS dependency): instruction descriptor, MMA issue,
// synchronisation and TMEM allocation, TMEM <-> register moves, and the split-precision operand planes.
// Descriptor bit layouts follow the PTX ISA "tcgen05 matrix descriptor" / "instruction descriptor" tables.
//
// Shared-memory operand layout used everywhere in this repo: SWIZZLE_NONE ("interleaved") canonical layout with
// 8x16-byte core matrices stored chunk-major:
//   K-major  operand X[rows][K] (bf16): element (r,k) at  (k/8)*LBO + (r/8)*SBO + (r%8)*16 + (k%8)*2
//            with SBO = 128, LBO = rows*16  ==  uint4 smem[K/8][rows]   (one 16-byte chunk = 8 consecutive k)
//   MN-major operand Y[K][MN]  (bf16): element (k,n) at  (k/8)*LBO + (n/8)*SBO + (k%8)*16 + (n%8)*2
//            with SBO = 128, LBO = (MN/8)*128 == uint4 smem[K/8][MN/8][8]  (one chunk = 8 consecutive mn)
// One tcgen05.mma consumes K=16 (two 8-k groups); the descriptor start address advances by 2*LBO per step.
//
// Split-precision GEMMs: an fp32 operand x is carried as TWO 16-bit planes  x = hi + lo  (hi = rn16(x), lo = rn16(x - hi)),
// and a product is three MMAs into the same fp32 TMEM accumulator:  A B^T ~= A_hi B_hi^T + A_lo B_hi^T + A_hi B_lo^T.
// The dropped lo x lo term and the rounding of lo are both 2^-2p relative (p = 8 for bf16 planes, 11 for fp16 planes), so the
// contraction is good to ~2^-16 (bf16) / ~2^-21 (fp16) per product instead of 2^-9 -- what the 0.05 mm joint bar needs
// (DESIGN.md section 2).  An operand that is exactly representable in 16 bits (a bf16 feature map) has no lo plane and its lo
// MMAs are skipped.  The instruction descriptor has separate A / B format fields, but an fp16 x bf16 pairing traps as an illegal
// instruction on sm_100a (measured), so both operands of an MMA use ONE format: where a bf16 feature map is an operand, the other
// side is carried as THREE bf16 planes (24 bits, split3_bf16) instead of two fp16 planes.
//
// A may also come from TENSOR MEMORY (tcgen05.mma [d], [a_tmem], b_desc): row m of A = TMEM lane m, K runs along the columns,
// two 16-bit elements per 32-bit column (low half = even k).  Weights that stay resident for a whole kernel live there, which
// frees their shared memory for the activation planes and removes the A-side shared-memory read from every MMA.
#pragma once
#include "common.cuh"
#include <cuda_fp16.h>

namespace kpf {

// ==== instruction descriptor ==========================================================================================

constexpr int FMT_F16 = 0, FMT_BF16 = 1;   // = the instruction descriptor's a_format / b_format encodings for kind::f16

// 32-bit instruction descriptor for kind::f16, fp32 accumulate, element formats per operand
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N, bool a_mn_major, bool b_mn_major, int a_fmt, int b_fmt) {
    return (1u << 4) /*D=f32*/ | ((uint32_t)a_fmt << 7) | ((uint32_t)b_fmt << 10) | ((a_mn_major ? 1u : 0u) << 15) |
           ((b_mn_major ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ==== MMA issue =======================================================================================================

// One operand plane pair in shared memory.  lo == 0: the operand is exact in 16 bits (no lo plane).
struct SmemOp {
    uint32_t hi, lo;      // shared-memory byte addresses of the two planes
    uint32_t lbo, sbo;    // descriptor strides (layout above)
};
// A operand planes in tensor memory: 16-bit elements, K/2 columns per plane
struct TmemOp {
    uint32_t hi, lo;      // TMEM addresses (lane 0 of the operand, first column); lo == 0xffffffff: no lo plane
};
constexpr uint32_t NO_PLANE = 0xffffffffu;

// ---- MMA issue with the 64-bit shared-memory descriptor kept as two 32-bit halves.  Only the low half (start address | LBO) moves
// along K, by a constant that folds into an immediate once the K loop is unrolled; the 64-bit add-with-carry, the per-iteration
// R2UR of the accumulator address / instruction descriptor and the loop control of the rolled form cost ~16 uniform-datapath
// instructions per MMA (~42 cycles per MMA measured, against a 16-cycle tensor-pipe floor at N = 32).
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
    return ((smem_addr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14); }

__device__ __forceinline__ void umma_issue_ss(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_issue_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 db;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}

// one plane pair over KS = K / 16 steps, fully unrolled
template <int KS>
__device__ __forceinline__ void umma_planes_ss(uint32_t tmem_d, uint32_t a_addr, uint32_t a_lbo, uint32_t a_sbo, uint32_t b_addr,
                                               uint32_t b_lbo, uint32_t b_sbo, uint32_t idesc, uint32_t& acc) {
    const uint32_t al = desc_lo(a_addr, a_lbo), ah = desc_hi(a_sbo), bl = desc_lo(b_addr, b_lbo), bh = desc_hi(b_sbo);
    const uint32_t a_step = (2 * a_lbo) >> 4, b_step = (2 * b_lbo) >> 4;   // start-address field, 16-byte units
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        umma_issue_ss(tmem_d, al + ks * a_step, ah, bl + ks * b_step, bh, idesc, acc);
        acc = 1u;
    }
}
template <int KS>
__device__ __forceinline__ void umma_planes_ts(uint32_t tmem_d, uint32_t a_tmem, uint32_t b_addr, uint32_t b_lbo, uint32_t b_sbo,
                                               uint32_t idesc, uint32_t& acc) {
    const uint32_t bl = desc_lo(b_addr, b_lbo), bh = desc_hi(b_sbo);
    const uint32_t b_step = (2 * b_lbo) >> 4;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        umma_issue_ts(tmem_d, a_tmem + 8 * ks, bl + ks * b_step, bh, idesc, acc);
        acc = 1u;
    }
}

// D[128 x N] (+)= A B^T over K, split precision, both operands from shared memory.  Issued by ONE thread.
// Order: the two small cross terms first, then hi x hi.
template <int K>
__device__ __forceinline__ void umma_gemm3_ss(uint32_t tmem_d, const SmemOp a, const SmemOp b, uint32_t idesc, bool accumulate) {
    static_assert(K % 16 == 0 && K >= 16 && K <= 256, "K must be a multiple of 16 in [16, 256]");
    constexpr int KS = K / 16;
    uint32_t acc = accumulate ? 1u : 0u;
    if (a.lo) umma_planes_ss<KS>(tmem_d, a.lo, a.lbo, a.sbo, b.hi, b.lbo, b.sbo, idesc, acc);
    if (b.lo) umma_planes_ss<KS>(tmem_d, a.hi, a.lbo, a.sbo, b.lo, b.lbo, b.sbo, idesc, acc);
    umma_planes_ss<KS>(tmem_d, a.hi, a.lbo, a.sbo, b.hi, b.lbo, b.sbo, idesc, acc);
}
// Same with A in tensor memory (8 columns per K = 16 step).
template <int K>
__device__ __forceinline__ void umma_gemm3_ts(uint32_t tmem_d, const TmemOp a, const SmemOp b, uint32_t idesc, bool accumulate) {
    static_assert(K % 16 == 0 && K >= 16 && K <= 256, "K must be a multiple of 16 in [16, 256]");
    constexpr int KS = K / 16;
    uint32_t acc = accumulate ? 1u : 0u;
    if (a.lo != NO_PLANE) umma_planes_ts<KS>(tmem_d, a.lo, b.hi, b.lbo, b.sbo, idesc, acc);
    if (b.lo) umma_planes_ts<KS>(tmem_d, a.hi, b.lo, b.lbo, b.sbo, idesc, acc);
    umma_planes_ts<KS>(tmem_d, a.hi, b.hi, b.lbo, b.sbo, idesc, acc);
}

// ---- the rolled single-plane form with a 64-bit descriptor (K5's map GEMMs and the bring-up self-test)
// 64-bit shared-memory matrix descriptor: start[0,14) | LBO[16,30) | SBO[32,46) | version=1 [46,48) | swizzle none
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}

// D[128 x N] (+)= A[128 x K] * B[N x K]^T ; K % 16 == 0.  Issued by ONE thread.  A rolled loop on purpose: the issue
// rate of the tensor pipe (~80 cycles per MMA here), not this loop, bounds it, and the unrolled form costs ~15 SASS
// instructions of descriptor arithmetic per MMA in kernels that are already instruction-fetch bound.
__device__ __forceinline__ void umma_gemm(uint32_t tmem_d, uint32_t a_addr, uint32_t a_lbo, uint32_t a_sbo, uint32_t b_addr,
                                          uint32_t b_lbo, uint32_t b_sbo, uint32_t idesc, int K, bool accumulate) {
    uint64_t ad = umma_smem_desc(a_addr, a_lbo, a_sbo), bd = umma_smem_desc(b_addr, b_lbo, b_sbo);
    const uint64_t a_step = (uint64_t)((2 * a_lbo) >> 4), b_step = (uint64_t)((2 * b_lbo) >> 4);  // start-address field, 16-byte units
#pragma unroll 1
    for (int ks = 0; ks < K / 16; ++ks) {
        umma_bf16(tmem_d, ad, bd, idesc, accumulate || ks > 0);
        ad += a_step;
        bd += b_step;
    }
}

// ==== synchronisation and TMEM allocation =============================================================================

// One lane of a CONVERGENT warp.  MMA / TMA issue code belongs in `if (warp_u == 0) { if (elect_one()) {...} __syncwarp(); }` with
// warp_u = warp_index_uniform(): inside a branch ptxas can prove warp-uniform the descriptors stay in uniform registers and each
// tcgen05.mma is one UTCHMMA; under a divergent `if (tid == 0)` every MMA is wrapped in a ~15-instruction
// ELECT / R2UR.BROADCAST waterfall loop (~100 cycles per MMA, measured).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ int warp_index_uniform() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

// all previously issued tcgen05.mma of this thread arrive on `bar` when complete (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// TMEM allocation: one full warp; ncols power of two in [32,512]; the base address lands in *slot (shared)
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ==== TMEM <-> register moves =========================================================================================
// N consecutive fp32 columns (tcgen05.ld/st 32x32b.xN): thread t of warp w touches TMEM lane 32*(w%4)+t.  The *_nw forms do
// not wait, so several moves can be in flight before one tmem_wait_ld()/tmem_wait_st().  The address must be warp-uniform and
// every call must sit in convergent code (.sync.aligned).

__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

template <int N>
__device__ __forceinline__ void tmem_ld_nw(uint32_t taddr, float* v) {
    static_assert(N == 1 || N == 2 || N == 4 || N == 8 || N == 16 || N == 32 || N == 64, "unsupported width");
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    if constexpr (N == 1) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(taddr));
    } else if constexpr (N == 2) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];"
                     : "=r"(r[0]), "=r"(r[1])
                     : "r"(taddr));
    } else if constexpr (N == 4) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                     : "r"(taddr));
    } else if constexpr (N == 8) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                     : "r"(taddr));
    } else if constexpr (N == 16) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                     : "r"(taddr));
    } else if constexpr (N == 32) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                     : "r"(taddr));
    } else {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
                     : "r"(taddr));
    }
}
// N = 64 is two x32 stores
template <int N>
__device__ __forceinline__ void tmem_st_nw(uint32_t taddr, const float* v) {
    static_assert(N == 2 || N == 4 || N == 8 || N == 16 || N == 32 || N == 64, "unsupported width");
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    if constexpr (N == 64) {
        tmem_st_nw<32>(taddr, v);
        tmem_st_nw<32>(taddr + 32, v + 32);
    } else if constexpr (N == 2) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(r[0]), "r"(r[1])
                     : "memory");
    } else if constexpr (N == 4) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3])
                     : "memory");
    } else if constexpr (N == 8) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                     : "memory");
    } else if constexpr (N == 16) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
                     : "memory");
    } else {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
                     : "memory");
    }
}
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float* v) {
    tmem_ld_nw<N>(taddr, v);
    tmem_wait_ld();
}
template <int N>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const float* v) {
    tmem_st_nw<N>(taddr, v);
    tmem_wait_st();
}

// ==== fp32 -> 16-bit planes ===========================================================================================
__device__ __forceinline__ uint32_t pack2_bf16(float a, float b) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack2_f16(float a, float b) {
    const __half2 v = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&v);
}
// two floats -> one 32-bit word of each plane (low half = first element)
template <int FMT>
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    if constexpr (FMT == FMT_BF16) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        const float2 hf = __bfloat1622float2(h);
        hi = *reinterpret_cast<const uint32_t*>(&h);
        lo = pack2_bf16(a - hf.x, b - hf.y);
    } else {
        const __half2 h = __floats2half2_rn(a, b);
        const float2 hf = __half22float2(h);
        hi = *reinterpret_cast<const uint32_t*>(&h);
        lo = pack2_f16(a - hf.x, b - hf.y);
    }
}
// eight floats -> one 16-byte operand chunk of each plane
template <int FMT>
__device__ __forceinline__ void split8(const float* v, uint4& hi, uint4& lo) {
    split2<FMT>(v[0], v[1], hi.x, lo.x);
    split2<FMT>(v[2], v[3], hi.y, lo.y);
    split2<FMT>(v[4], v[5], hi.z, lo.z);
    split2<FMT>(v[6], v[7], hi.w, lo.w);
}
// fp32 -> three bf16 planes (hi + mid + lo carries 24 mantissa bits, full fp32 range): the partner of a bf16 feature-map operand
__device__ __forceinline__ void split3_bf16(float a, float b, uint32_t& hi, uint32_t& mid, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const float2 hf = __bfloat1622float2(h);
    const float ra = a - hf.x, rb = b - hf.y;
    const __nv_bfloat162 m = __floats2bfloat162_rn(ra, rb);
    const float2 mf = __bfloat1622float2(m);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    mid = *reinterpret_cast<const uint32_t*>(&m);
    lo = pack2_bf16(ra - mf.x, rb - mf.y);
}
__device__ __forceinline__ void split8x3_bf16(const float* v, uint4& hi, uint4& mid, uint4& lo) {
    split3_bf16(v[0], v[1], hi.x, mid.x, lo.x);
    split3_bf16(v[2], v[3], hi.y, mid.y, lo.y);
    split3_bf16(v[4], v[5], hi.z, mid.z, lo.z);
    split3_bf16(v[6], v[7], hi.w, mid.w, lo.w);
}
// D (+)= A B^T with A = a bf16 feature-map operand (one exact plane, or hi + lo of an fp32 map) and B = three bf16 planes at
// b_addr + {0, 1, 2} * b_plane_bytes: A_hi (B_hi + B_mid + B_lo) [+ A_lo (B_hi + B_mid)], smallest terms first.  Issued with the
// rolled umma_gemm (see there).
__device__ __forceinline__ void umma_gemm_map_x3(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo /* 0: none */, uint32_t a_lbo, uint32_t a_sbo,
                                                 uint32_t b_addr, uint32_t b_plane_bytes, uint32_t b_lbo, uint32_t b_sbo, uint32_t idesc, int K,
                                                 bool accumulate) {
    umma_gemm(tmem_d, a_hi, a_lbo, a_sbo, b_addr + 2 * b_plane_bytes, b_lbo, b_sbo, idesc, K, accumulate);
    if (a_lo) umma_gemm(tmem_d, a_lo, a_lbo, a_sbo, b_addr + b_plane_bytes, b_lbo, b_sbo, idesc, K, true);
    umma_gemm(tmem_d, a_hi, a_lbo, a_sbo, b_addr + b_plane_bytes, b_lbo, b_sbo, idesc, K, true);
    if (a_lo) umma_gemm(tmem_d, a_lo, a_lbo, a_sbo, b_addr, b_lbo, b_sbo, idesc, K, true);
    umma_gemm(tmem_d, a_hi, a_lbo, a_sbo, b_addr, b_lbo, b_sbo, idesc, K, true);
}

}  // namespace kpf
