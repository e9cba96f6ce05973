// Point stage of Block_KPFusion on tensor cores (model/model.py:295-320; SURVEY.md 8a rows a7-a9, 8f-2):
//   K4b pcl_joint2offset + K3 4-tap gathers + the four folded Conv1d+BN point embeddings + relu/relu
//   + the softmax-over-points aggregation numerators, in ONE persistent kernel; nothing of [B,N,*] but the final
//   point features e (bf16) ever reaches HBM.
//
//   kpf_repack_features : NCHW (img_feat | img_feat_rgb | img_offset[4J:]) -> channels-last bf16 rows [B,HW,288]
//                         so that one tap of a point is ONE contiguous 576-byte row.
//   kpf_point_embed     : per 128-point tile (512 threads: 4 per point in the gather, 4 column groups per row in the epilogues):
//       A1[128 x 256] = [gather(img_feat) | gather(weight map) | (unit offset xyz, closeness) per joint, xyz]   (bf16, smem)
//       A2[128 x 128] =  gather(img_feat_rgb)
//       e  = relu( relu(A1 W1^T + b1) + A2 W2^T + b2 )                     tcgen05, fp32 accumulators in TMEM
//       p  = exp(w - max_tile w)  (softmax numerators of the gathered weight map, per joint)
//       D[c][j] = sum_n e[n][c] p[n][j]                                    tcgen05 with MN-major operands
//     outputs: e [B,N,128] bf16, and per tile (D, max, sum) partials that the DESA kernel combines flash-style.
//   Weights (96 KB bf16) stay resident in shared memory; CTAs are persistent over tiles.
#include "tcgen05.cuh"

namespace kpf {

constexpr int PE_CP = 288;   // channels per repacked row: 128 depth-branch + 128 rgb-branch + 32 (J weight channels, zero padded)
constexpr int PE_CH = PE_CP / 8;

template <typename T>
__global__ void __launch_bounds__(256)
repack_kernel(const T* __restrict__ f_d, const T* __restrict__ f_rgb, const T* __restrict__ f_w, long long w_bs, int C, int J, int HW,
              __nv_bfloat16* __restrict__ out, __nv_bfloat16* __restrict__ out_lo) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, c0 = blockIdx.y * 32, h0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, h = h0 + tx;
        float v = 0.f;
        if (h < HW) {
            if (c < C) v = to_f32(f_d[((size_t)b * C + c) * HW + h]);
            else if (c < 2 * C) v = to_f32(f_rgb[((size_t)b * C + (c - C)) * HW + h]);
            else if (c - 2 * C < J) v = to_f32(f_w[(size_t)b * w_bs + (size_t)(c - 2 * C) * HW + h]);
        }
        tile[r][tx] = v;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int h = h0 + r, c = c0 + tx;
        if (h < HW && c < PE_CP) {
            const float v = tile[tx][r];
            const __nv_bfloat16 hi = __float2bfloat16_rn(v);
            out[((size_t)b * HW + h) * PE_CP + c] = hi;
            if (out_lo) out_lo[((size_t)b * HW + h) * PE_CP + c] = __float2bfloat16_rn(v - __bfloat162float(hi));   // fp32 maps: second plane
        }
    }
}

// bf16 fast path of the repack (C = 128, HW % 128 == 0): a CTA transposes a [64 channels x 128 cells] block through shared memory
// with 16-byte global accesses on both sides (8 cells of a channel in, 8 channels of a cell out) -- the generic kernel above
// moves 2 bytes per lane.  Channel blocks 0,1 = depth branch, 2,3 = rgb branch, 4 = the J weight channels zero-padded to 32.
constexpr int RP_LD = 128 + 2;   // bf16 elements per staged channel row (+2: consecutive channels land in consecutive banks)
__global__ void __launch_bounds__(256)
repack_bf16_kernel(const __nv_bfloat16* __restrict__ f_d, const __nv_bfloat16* __restrict__ f_rgb, const __nv_bfloat16* __restrict__ f_w,
                   long long w_bs, int J, int HW, __nv_bfloat16* __restrict__ out) {
    __shared__ __align__(16) __nv_bfloat16 tile[64 * RP_LD];
    const int b = blockIdx.z, cb = blockIdx.y, h0 = blockIdx.x * 128, tid = threadIdx.x;
    const int nch = cb < 4 ? 64 : 32;
    // load: thread -> (channel, 8 consecutive cells); a warp reads 2 channels x 256 B
    for (int i = tid; i < nch * 16; i += 256) {
        const int ch = i >> 4, seg = i & 15;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (cb < 2) v = __ldg(reinterpret_cast<const uint4*>(f_d + ((size_t)b * 128 + cb * 64 + ch) * HW + h0) + seg);
        else if (cb < 4) v = __ldg(reinterpret_cast<const uint4*>(f_rgb + ((size_t)b * 128 + (cb - 2) * 64 + ch) * HW + h0) + seg);
        else if (ch < J) v = __ldg(reinterpret_cast<const uint4*>(f_w + (size_t)b * w_bs + (size_t)ch * HW + h0) + seg);
        uint32_t* dst = reinterpret_cast<uint32_t*>(tile + ch * RP_LD + seg * 8);   // 4-byte aligned (RP_LD even)
        dst[0] = v.x;
        dst[1] = v.y;
        dst[2] = v.z;
        dst[3] = v.w;
    }
    __syncthreads();
    // store: thread -> (cell, 8 consecutive channels); a warp writes 128 contiguous bytes of each of 4 (or 8) cell rows
    const int gs = cb < 4 ? 3 : 2, ngrp = 1 << gs;   // 8-channel groups per cell
    for (int i = tid; i < 128 * ngrp; i += 256) {
        const int g = i & (ngrp - 1), cell = i >> gs;
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint16_t lo = *reinterpret_cast<const uint16_t*>(tile + (8 * g + 2 * k) * RP_LD + cell);
            const uint16_t hi = *reinterpret_cast<const uint16_t*>(tile + (8 * g + 2 * k + 1) * RP_LD + cell);
            w[k] = (uint32_t)lo | ((uint32_t)hi << 16);
        }
        *reinterpret_cast<uint4*>(out + ((size_t)b * HW + h0 + cell) * PE_CP + cb * 64 + 8 * g) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

struct PointParams {
    const uint4* feat_hi;    // [B,HW,36] uint4 (288 bf16): repacked maps (hi plane; the only one for bf16 maps)
    const uint4* feat_lo;    // same layout, lo plane of fp32 maps, or null
    const int32_t* idx;      // [B,N,4]
    const float* clos;       // [B,N,4]
    const float* pcl;        // [B,N,3]
    const float* joint;      // [B,J,3]
    const int32_t* order;    // [B,N] processing order of the points (kpf_spatial_order) or null = identity
    const uint4* wmat;       // canonical planes: W1 hi [32][128], W1 lo, W2 hi [16][128], W2 lo
    const float* wvec;       // b1[128], b2[128]
    uint16_t* e_out;         // [B,N,256]: rows [hi 128 | lo 128] 16-bit planes, batch stride e_bs elements (>= N*256: DESA appends its
    long long e_bs;          //   joint rows behind the points)
    float* part_acc;         // [B,T,128,32]   T = N / 64
    float* part_ms;          // [B,T,2,32]  (max, sum)
    // The gathered inputs do not depend on the joints, and both blocks of KPFusion gather the same taps of the same maps
    // (model.py:297-306 runs per block): a launch can store every tile's gathered operand image (stage_out) and a later launch on
    // the same points can load it with the TMA engine instead of gathering again (stage_in).  [B*T][PE_STAGE_BYTES], 16-byte aligned.
    unsigned char* stage_out;
    const unsigned char* stage_in;
    int B, N, J, HW, fmt;
    float kernel_size;
};

__device__ __forceinline__ void bf16x8_fma(float* acc, const uint4& v, float w) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        acc[2 * i] += f.x * w;
        acc[2 * i + 1] += f.y * w;
    }
}

constexpr int PE_NT = 512;
constexpr int PE_ISSUER = 15;   // the warp whose elected lane issues the MMAs: one of group 1 (warps 8-15), which has no softmax work to
                                // do while the MMAs are being issued (tcgen05.mma issue blocks at the tensor pipe's rate)
constexpr int PE_TP = 64;    // points per tile
// TMEM columns: the resident weight planes (A operands, 16-bit pairs), then the two accumulators; after the epilogue has read
// them the accumulator columns are reused for e^T (the aggregation's A operand) and the aggregation accumulator
constexpr uint32_t PE_W1H = 0, PE_W1L = 128, PE_W2H = 256, PE_W2L = 320, PE_ACC1 = 384, PE_ACC2 = 448;
constexpr uint32_t PE_EH = PE_ACC2, PE_EL = PE_ACC2 + 32, PE_ACC3 = PE_ACC1;
// staged tile image: the feature chunks (k-chunks 0..19) of the 8 point groups of both A1 planes, the A2 planes, the raw gathered
// weight-map values (sT: [21][65] f32 + 3 pad)
constexpr int PE_ST_X1 = 20 * 8 * 16;                      // bytes per (plane, point group) run of sX1
constexpr int PE_ST_T = (21 * 65 + 3) * 4;                 // bytes of sT
constexpr int PE_STAGE_BYTES = 16 * PE_ST_X1 + 2 * 1024 * 16 + PE_ST_T;

// The whole point stage, computed TRANSPOSED: D^T[channel][point] = W[channel][k] X[point][k].  The folded weights (K = 384, two
// 16-bit planes) stay in TENSOR MEMORY for the life of the persistent CTA as the A operands; a tile is 64 points whose gathered
// inputs are written as K-major B operand planes; a thread of the epilogue owns one output channel (its TMEM lane) and 16 points.
// STAGE: 0 = gather; 1 = gather and store the tiles' operand images (stage_out); 2 = load them instead of gathering (stage_in).
// A template parameter: the launches that do not stage carry none of its code or registers.
template <int FMT, int STAGE>
__global__ void __launch_bounds__(PE_NT, 1) point_embed_kernel(const PointParams p) {
    constexpr bool ST_OUT = STAGE == 1, ST_IN = STAGE == 2;
    extern __shared__ __align__(128) unsigned char pe_smem[];
    uint4* sX1 = reinterpret_cast<uint4*>(pe_smem);   // 2 planes x [8 point groups][32 k-chunks][8 points]   (K = 256)
    uint4* sX2 = sX1 + 2 * 2048;                       // 2 planes x [8][16][8]                                (K = 128)
    uint4* sP = sX2 + 2 * 1024;                        // 2 planes x MN-major B [8 point groups][4 joint groups][8 points]: softmax numerators
    uint4* sE = sP + 2 * 256;                          // [64 points][32 chunks]: e rows [hi | lo] staged for the coalesced copy-out
    float* sJ = reinterpret_cast<float*>(sE + 2048);   // [32][4] joints of the current sample
    float* sRed = sJ + 128;                            // [32] per-joint tile maxima
    float* sB = sRed + 32;                             // b1[128], b2[128]
    float* sT = sB + 256;                              // [21][65] transposed softmax scratch
    int* sN = reinterpret_cast<int*>(sT + 21 * 65 + 3);   // [2][64] point ids of the tile in flight / being prefetched
    __shared__ __align__(8) uint64_t mma_bar, in_bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = warp_index_uniform();  // MMA issue: one elected lane of warp 0 from warp-uniform code (tcgen05.cuh)
    // gather: warp = 8 points x 4 chunk lanes (64 contiguous bytes of a tap row per point per load; the 8 points fill the 8 rows x
    // 16 B core matrices of the operand, so the stores are conflict free).  Warps 0-7 (grp 0) take the depth-branch and weight-map
    // chunks and the joint offsets, warps 8-15 (grp 1) the rgb-branch chunks of the same 64 points.
    const int r = 8 * (warp & 7) + (lane & 7), sub = lane >> 3, grp = warp >> 3;
    const int q = warp & 3, cg = warp >> 2, ch = 32 * q + lane;   // epilogues: channel ch (TMEM lane), points [16cg, 16cg + 16)
    const int J = p.J, N = p.N, T = N / PE_TP;
    constexpr int fmt = FMT;

    pdl_launch_dependents();
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 0) {
        mbar_init(&mma_bar, 1);
        mbar_init(&in_bar, 1);
        fence_mbar_init();
    }
    for (int i = tid; i < 256; i += PE_NT) sB[i] = p.wvec[i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = tmem_slot, tmem = tmem0 + ((uint32_t)(32 * q) << 16);
    {   // weights -> tensor memory: row ch, 16-bit K elements packed two per column; this thread moves a quarter of each plane
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {   // W1 planes: 32 k-chunks = 128 columns, chunks [8cg, 8cg + 8)
            const uint4* src = p.wmat + pl * 4096;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint4 v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = __ldg(src + (8 * cg + 4 * h + k) * 128 + ch);
                tmem_st_nw<16>(tmem + (pl ? PE_W1L : PE_W1H) + 32 * cg + 16 * h, reinterpret_cast<const float*>(v));
            }
        }
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {   // W2 planes: 16 k-chunks = 64 columns, chunks [4cg, 4cg + 4)
            const uint4* src = p.wmat + 8192 + pl * 2048;
            uint4 v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = __ldg(src + (4 * cg + k) * 128 + ch);
            tmem_st_nw<16>(tmem + (pl ? PE_W2L : PE_W2H) + 16 * cg, reinterpret_cast<const float*>(v));
        }
        tmem_wait_st();
    }
    uint32_t phase = 0;

    // per-point inputs of the tile about to be gathered (prefetched during the previous tile's MMAs)
    int4 id = make_int4(0, 0, 0, 0);
    float4 cw = make_float4(0.f, 0.f, 0.f, 0.f);
    float px = 0.f, py = 0.f, pz = 0.f;
    int tile_par = 0;
    auto fetch_point = [&](int tile, int par) {
        const int b = tile / T, t = tile - b * T;
        const int n_id = p.order ? __ldg(p.order + (size_t)b * N + t * PE_TP + r) : t * PE_TP + r;   // tile = 64 consecutive points of the order
        if (sub == 0 && grp == 0) sN[par * PE_TP + r] = n_id;
        const size_t pn = (size_t)b * N + n_id;
        if (!ST_IN) {
            id = __ldg(reinterpret_cast<const int4*>(p.idx + pn * 4));
            cw = __ldg(reinterpret_cast<const float4*>(p.clos + pn * 4));
        }
        px = __ldg(p.pcl + pn * 3);
        py = __ldg(p.pcl + pn * 3 + 1);
        pz = __ldg(p.pcl + pn * 3 + 2);
    };
    // staged input: warp 0 pulls a tile's image into sX1 (feature chunks) / sX2 / sT with 18 bulk copies, one per lane
    auto load_stage = [&](int tile) {   // call from all lanes of warp 0
        const unsigned char* src = p.stage_in + (size_t)tile * PE_STAGE_BYTES;
        if (lane == 0) mbar_expect_tx(&in_bar, PE_STAGE_BYTES);
        __syncwarp();
        if (lane < 16) tma_bulk_g2s(sX1 + (lane >> 3) * 2048 + (lane & 7) * 256, src + (size_t)lane * PE_ST_X1, PE_ST_X1, &in_bar);
        else if (lane == 16) tma_bulk_g2s(sX2, src + 16 * PE_ST_X1, 2 * 1024 * 16, &in_bar);
        else if (lane == 17) tma_bulk_g2s(sT, src + 16 * PE_ST_X1 + 2 * 1024 * 16, PE_ST_T, &in_bar);
    };
    uint32_t in_phase = 0;
    pdl_wait();   // weights only so far; points, indices and the repacked maps come from the previous kernels
    if ((int)blockIdx.x < p.B * T) {
        fetch_point(blockIdx.x, 0);
        if (ST_IN && warp == 0) load_stage(blockIdx.x);
    }

    for (int tile = blockIdx.x; tile < p.B * T; tile += gridDim.x) {
        const int b = tile / T, t = tile - b * T;
        __syncthreads();  // previous tile's readers of sJ / sRed / sT / sE are done (its MMAs were waited for)
        // ---- K3: 4-tap gathers of this thread's chunks of the 36-chunk row: grp 0 -> depth 0-15 (A1 chunks 0-15) and weight map
        //      32-35 (A1 chunks 16-19 and the softmax); grp 1 -> rgb 16-31 (A2 chunks 0-15)
        float wraw[8];   // grp 0: gathered weight-map channels [8 sub, 8 sub + 8) of this point
        uint4* x1r = sX1 + (r >> 3) * 256 + (r & 7);
        uint4* x2r = sX2 + (r >> 3) * 128 + (r & 7);
        if (ST_IN) {   // the tile's gathered image was staged by an earlier launch: it is (being) copied in by the TMA engine
            mbar_wait(&in_bar, in_phase);
            in_phase ^= 1;
            if (grp == 0) {
#pragma unroll
                for (int k = 0; k < 8; ++k) wraw[k] = 8 * sub + k < J ? sT[(8 * sub + k) * 65 + r] : 0.f;
            }
        } else {
            const size_t rb = (size_t)b * p.HW;
            const uint4 *h0 = p.feat_hi + (rb + id.x) * PE_CH, *h1 = p.feat_hi + (rb + id.y) * PE_CH, *h2 = p.feat_hi + (rb + id.z) * PE_CH,
                        *h3 = p.feat_hi + (rb + id.w) * PE_CH;
            const int nload = grp == 0 ? 5 : 4, c_base = grp == 0 ? 0 : 16;
            uint4 v[5][4];
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                if (u < nload) {
                    const int cc = (u < 4 ? c_base + 4 * u : 32) + sub;
                    v[u][0] = __ldg(h0 + cc);
                    v[u][1] = __ldg(h1 + cc);
                    v[u][2] = __ldg(h2 + cc);
                    v[u][3] = __ldg(h3 + cc);
                }
            }
            float acc[5][8];
#pragma unroll
            for (int u = 0; u < 5; ++u) {
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[u][k] = 0.f;
                if (u < nload) {
                    bf16x8_fma(acc[u], v[u][0], cw.x);
                    bf16x8_fma(acc[u], v[u][1], cw.y);
                    bf16x8_fma(acc[u], v[u][2], cw.z);
                    bf16x8_fma(acc[u], v[u][3], cw.w);
                }
            }
            if (p.feat_lo) {   // fp32 maps: add the lo plane's taps
                const uint4 *l0 = p.feat_lo + (rb + id.x) * PE_CH, *l1 = p.feat_lo + (rb + id.y) * PE_CH, *l2 = p.feat_lo + (rb + id.z) * PE_CH,
                            *l3 = p.feat_lo + (rb + id.w) * PE_CH;
#pragma unroll
                for (int u = 0; u < 5; ++u) {
                    if (u < nload) {
                        const int cc = (u < 4 ? c_base + 4 * u : 32) + sub;
                        bf16x8_fma(acc[u], __ldg(l0 + cc), cw.x);
                        bf16x8_fma(acc[u], __ldg(l1 + cc), cw.y);
                        bf16x8_fma(acc[u], __ldg(l2 + cc), cw.z);
                        bf16x8_fma(acc[u], __ldg(l3 + cc), cw.w);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                if (u < nload) {
                    uint4 oh, ol;
                    split8<FMT>(acc[u], oh, ol);
                    if (grp == 1) {
                        x2r[(4 * u + sub) * 8] = oh;
                        x2r[1024 + (4 * u + sub) * 8] = ol;
                    } else {
                        const int kc = u < 4 ? 4 * u + sub : 16 + sub;
                        x1r[kc * 8] = oh;
                        x1r[2048 + kc * 8] = ol;
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) wraw[k] = acc[4][k];
        }
        // the sample's joints for K4b, stored after the gather: the gather runs at the 128-register cap, and values held across it
        // (these, 1 / kernel_size) spill
        if (tid < J) {
            sJ[4 * tid] = p.joint[((size_t)b * J + tid) * 3];
            sJ[4 * tid + 1] = p.joint[((size_t)b * J + tid) * 3 + 1];
            sJ[4 * tid + 2] = p.joint[((size_t)b * J + tid) * 3 + 2];
        }
        // softmax over the tile's points, step 1: the gathered weights, transposed, for the per-joint maxima
        if (grp == 0 && !ST_IN) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (8 * sub + k < J) sT[(8 * sub + k) * 65 + r] = wraw[k];
        }
        if (ST_OUT) fence_proxy_async();   // the operand chunks and sT are read by the bulk stores below (async proxy)
        __syncthreads();  // sJ, sT visible
        if (ST_OUT && warp == 0 && lane < 18) {   // store this tile's gathered image for a later launch (the 18 runs load_stage reads)
            unsigned char* dst = p.stage_out + (size_t)tile * PE_STAGE_BYTES;
            if (lane < 16) tma_bulk_s2g(dst + (size_t)lane * PE_ST_X1, sX1 + (lane >> 3) * 2048 + (lane & 7) * 256, PE_ST_X1);
            else if (lane == 16) tma_bulk_s2g(dst + 16 * PE_ST_X1, sX2, 2 * 1024 * 16);
            else tma_bulk_s2g(dst + 16 * PE_ST_X1 + 2 * 1024 * 16, sT, PE_ST_T);
            bulk_commit();
        }
        // ---- K4b: items 0..J-1 = [unit offset xyz, closeness] of a joint, item J = the point's xyz; item i fills half (i & 1) of
        //      k-chunk 20 + i / 2 of A1 (ops.pack_point_embed orders W1's columns to match).  The eight threads of a point (four
        //      chunk lanes x two groups) take three items each.  fp32-exact sqrt / divisions: the values feed a split-precision operand.
        {
            const int u = sub + 4 * grp;
            const float inv_ks = 1.f / p.kernel_size;
#pragma unroll
            for (int jj = 0; jj < 3; ++jj) {
                const int j = 3 * u + jj;
                float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;
                if (j < J) {
                    const float ox = sJ[4 * j] - px, oy = sJ[4 * j + 1] - py, oz = sJ[4 * j + 2] - pz;
                    const float dis = sqrtf(ox * ox + oy * oy + oz * oz);
                    const float inv = 1.f / (dis + 1e-8f);
                    const float heat = (p.kernel_size - dis) * inv_ks;
                    const float msk = (heat >= 0.f && pz < 0.99f) ? 1.f : 0.f;
                    o0 = ox * inv * msk;
                    o1 = oy * inv * msk;
                    o2 = oz * inv * msk;
                    o3 = heat * msk;
                } else if (j == J) {
                    o0 = px;
                    o1 = py;
                    o2 = pz;
                }
                uint2 oh, ol;
                split2<FMT>(o0, o1, oh.x, ol.x);
                split2<FMT>(o2, o3, oh.y, ol.y);
                reinterpret_cast<uint2*>(x1r + (20 + (j >> 1)) * 8)[j & 1] = oh;
                reinterpret_cast<uint2*>(x1r + 2048 + (20 + (j >> 1)) * 8)[j & 1] = ol;
            }
        }
        // softmax step 1b: per-joint maximum over the tile's 64 points, 16 threads per joint
        {
            const int rj = tid >> 4, rs = tid & 15;
            float m = -INFINITY;
            if (rj < J) {
#pragma unroll
                for (int i = 0; i < 4; ++i) m = fmaxf(m, sT[rj * 65 + rs + 16 * i]);
            }
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (rs == 0) sRed[rj] = rj < J ? m : -INFINITY;
        }
        // the bulk stores have read their sources: sT is rewritten after the barrier below, the operands by the next tile
        if (ST_OUT && warp == 0 && lane < 18) bulk_wait_read<0>();
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp_u == PE_ISSUER) {
            tc_fence_after();
            if (elect_one()) {
                const uint32_t id64 = umma_idesc_f16(128, PE_TP, false, false, fmt, fmt);
                TmemOp a;
                SmemOp xb;
                // B operands: 128 B between k-chunks, 4096 / 2048 B between 8-point groups
                a.hi = tmem0 + PE_W1H; a.lo = tmem0 + PE_W1L;
                xb.hi = smem_u32(sX1); xb.lo = xb.hi + 2048 * 16; xb.lbo = 128; xb.sbo = 4096;
                umma_gemm3_ts<256>(tmem0 + PE_ACC1, a, xb, id64, false);
                a.hi = tmem0 + PE_W2H; a.lo = tmem0 + PE_W2L;
                xb.hi = smem_u32(sX2); xb.lo = xb.hi + 1024 * 16; xb.lbo = 128; xb.sbo = 2048;
                umma_gemm3_ts<128>(tmem0 + PE_ACC2, a, xb, id64, false);
                umma_commit(&mma_bar);
            }
            __syncwarp();
        }
        // ---- while the MMAs run: next tile's point inputs, and the softmax numerators p = exp(w - max) with their per-joint sums
        const int my_n = sN[tile_par * PE_TP + (tid >> 3)];   // copy-out below: thread = (point tid / 8, 8 chunk lanes)
        if (tile + (int)gridDim.x < p.B * T) fetch_point(tile + gridDim.x, tile_par ^ 1);
        float* ms = p.part_ms + ((size_t)b * T + t) * 64;
        if (grp == 0) {
            float pj[8];   // joints [8 sub, 8 sub + 8) of this point
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int j = 8 * sub + k;
                pj[k] = j < J ? __expf(wraw[k] - sRed[j]) : 0.f;
                if (j < J) sT[j * 65 + r] = pj[k];
            }
            uint4 oh, ol;
            split8<FMT>(pj, oh, ol);
            sP[(r >> 3) * 32 + sub * 8 + (r & 7)] = oh;
            sP[256 + (r >> 3) * 32 + sub * 8 + (r & 7)] = ol;
        }
        if (tid < 32) ms[tid] = sRed[tid];
        if (grp == 0) {   // the numerators and their sums involve only warps 0-7: their own barrier, so nobody waits for the MMA issuer here
            named_bar_sync(1, 256);
            const int rj = tid >> 3, rs = tid & 7;
            float sm_ = 0.f;
            if (rj < J) {
#pragma unroll
                for (int i = 0; i < 8; ++i) sm_ += sT[rj * 65 + rs + 8 * i];
            }
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) sm_ += __shfl_xor_sync(0xffffffffu, sm_, o);
            if (rs == 0) ms[32 + rj] = rj < J ? sm_ : 0.f;
        }
        mbar_wait(&mma_bar, phase);
        phase ^= 1;
        tc_fence_after();
        // ---- epilogue: e = relu(relu(acc1 + b1) + acc2 + b2) for channel ch, points [16cg, 16cg + 16)
        uint32_t eh[8], el[8];
        {
            float a[16], rr[16];
            tmem_ld_nw<16>(tmem + PE_ACC1 + 16 * cg, a);
            tmem_ld_nw<16>(tmem + PE_ACC2 + 16 * cg, rr);
            tmem_wait_ld();
            const float b1 = sB[ch], b2 = sB[128 + ch];
            uint16_t* se = reinterpret_cast<uint16_t*>(sE) + ch;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float e0 = fmaxf(fmaxf(a[2 * i] + b1, 0.f) + rr[2 * i] + b2, 0.f);
                const float e1 = fmaxf(fmaxf(a[2 * i + 1] + b1, 0.f) + rr[2 * i + 1] + b2, 0.f);
                split2<FMT>(e0, e1, eh[i], el[i]);
                // staged rows [point][hi 128 | lo 128]: a warp's 32 channels are 64 contiguous bytes of each
                se[(16 * cg + 2 * i) * 256] = (uint16_t)eh[i];
                se[(16 * cg + 2 * i) * 256 + 128] = (uint16_t)el[i];
                se[(16 * cg + 2 * i + 1) * 256] = (uint16_t)(eh[i] >> 16);
                se[(16 * cg + 2 * i + 1) * 256 + 128] = (uint16_t)(el[i] >> 16);
            }
        }
        tc_fence_before();
        __syncthreads();   // every warp has read its accumulator columns: they are reused for e^T and the aggregation
        tc_fence_after();
        // the main MMAs have completed and everybody is past the softmax sums: sX1 / sX2 / sT are free for the next tile's image
        if (ST_IN && warp == 0 && tile + (int)gridDim.x < p.B * T) {
            fence_proxy_async();
            load_stage(tile + gridDim.x);
        }
        // e^T as the aggregation's A operand in tensor memory: lane = channel, K = the tile's 64 points, 16-bit pairs
        tmem_st_nw<8>(tmem + PE_EH + 8 * cg, reinterpret_cast<const float*>(eh));
        tmem_st_nw<8>(tmem + PE_EL + 8 * cg, reinterpret_cast<const float*>(el));
        tmem_wait_st();
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp_u == PE_ISSUER) {
            tc_fence_after();
            if (elect_one()) {   // D[c][j] = sum_n e[n][c] p[n][j]
                TmemOp a;
                a.hi = tmem0 + PE_EH; a.lo = tmem0 + PE_EL;
                SmemOp pb;
                pb.hi = smem_u32(sP); pb.lo = pb.hi + 256 * 16; pb.lbo = 512; pb.sbo = 128;
                umma_gemm3_ts<PE_TP>(tmem0 + PE_ACC3, a, pb, umma_idesc_f16(128, 32, false, true, fmt, fmt), false);
                umma_commit(&mma_bar);
            }
            __syncwarp();
        }
        {   // copy-out of the staged e rows while the aggregation runs: 8 lanes write 128 contiguous bytes of a 512-byte row
            uint4* dst = reinterpret_cast<uint4*>(p.e_out + (size_t)b * p.e_bs + (size_t)my_n * 256);
            const uint4* src = sE + (tid >> 3) * 32;
#pragma unroll
            for (int k = 0; k < 4; ++k) dst[(tid & 7) + 8 * k] = src[(tid & 7) + 8 * k];
        }
        mbar_wait(&mma_bar, phase);
        phase ^= 1;
        tc_fence_after();
        {   // D[channel = ch][joints 8cg .. 8cg + 8)
            float a[8];
            tmem_ld<8>(tmem + PE_ACC3 + 8 * cg, a);
            float4* o = reinterpret_cast<float4*>(p.part_acc + (((size_t)b * T + t) * 128 + ch) * 32 + 8 * cg);
            o[0] = make_float4(a[0], a[1], a[2], a[3]);
            o[1] = make_float4(a[4], a[5], a[6], a[7]);
        }
        tc_fence_before();
        tile_par ^= 1;
    }
    if (ST_OUT && warp == 0 && lane < 18) bulk_wait<0>();   // the staged images are written
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem0, 512);
}

constexpr size_t PE_SMEM = (size_t)(2 * 2048 + 2 * 1024 + 2 * 256 + 2048) * 16 + (128 + 32 + 256 + 21 * 65 + 3 + 128) * 4;

}  // namespace kpf

extern "C" int kpf_repack_features(const void* f_d, const void* f_rgb, const void* f_w, long long w_batch_stride, int dtype, int B, int C,
                                   int J, int HW, void* out, void* out_lo, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && C == 128 && J >= 1 && J <= 32 && HW >= 1);
    if (B == 0) return 0;
    KPF_REQUIRE((dtype == KPF_F32) == (out_lo != nullptr));   // fp32 maps carry a second (lo) plane, bf16 maps are exact in one
    dim3 grid((HW + 31) / 32, PE_CP / 32, B);
    if (dtype == KPF_F32) {
        kpf::set_smem(repack_kernel<float>, 0);
        repack_kernel<float><<<grid, 256, 0, stream>>>((const float*)f_d, (const float*)f_rgb, (const float*)f_w, w_batch_stride, C, J, HW,
                                                      (__nv_bfloat16*)out, (__nv_bfloat16*)out_lo);
    } else if (dtype == KPF_BF16 && HW % 128 == 0 && ((uintptr_t)f_d % 16) == 0 && ((uintptr_t)f_rgb % 16) == 0 && ((uintptr_t)f_w % 16) == 0 &&
               w_batch_stride % 8 == 0) {
        kpf::set_smem(repack_bf16_kernel, 0);
        repack_bf16_kernel<<<dim3(HW / 128, 5, B), 256, 0, stream>>>((const __nv_bfloat16*)f_d, (const __nv_bfloat16*)f_rgb,
                                                                    (const __nv_bfloat16*)f_w, w_batch_stride, J, HW, (__nv_bfloat16*)out);
    } else if (dtype == KPF_BF16) {
        kpf::set_smem(repack_kernel<__nv_bfloat16>, 0);
        repack_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)f_d, (const __nv_bfloat16*)f_rgb,
                                                              (const __nv_bfloat16*)f_w, w_batch_stride, C, J, HW, (__nv_bfloat16*)out, nullptr);
    } else {
        return KPF_ERR_UNSUPPORTED;
    }
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_point_embed(const void* feat_hi, const void* feat_lo, const int32_t* idx, const float* clos, const float* pcl,
                               const float* joint, const int32_t* order, const void* wmat, const float* wvec, int B, int N, int J, int HW,
                               float kernel_size, int fmt, void* e_out, long long e_batch_stride, float* part_acc, float* part_ms,
                               void* stage_out, const void* stage_in, int num_sms, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(((uintptr_t)stage_out % 16) == 0 && ((uintptr_t)stage_in % 16) == 0 && !(stage_out && stage_in));
    KPF_REQUIRE(B >= 0 && N >= PE_TP && N % PE_TP == 0 && J >= 1 && J <= 21 && HW >= 1 && num_sms >= 1);
    KPF_REQUIRE(fmt == FMT_F16 || fmt == FMT_BF16);
    KPF_REQUIRE(((uintptr_t)feat_hi % 16) == 0 && ((uintptr_t)feat_lo % 16) == 0 && ((uintptr_t)wmat % 16) == 0 && ((uintptr_t)idx % 16) == 0 &&
                ((uintptr_t)clos % 16) == 0 && ((uintptr_t)e_out % 16) == 0);
    if (B == 0) return 0;
    PointParams p;
    p.feat_hi = (const uint4*)feat_hi; p.feat_lo = (const uint4*)feat_lo; p.idx = idx; p.clos = clos; p.pcl = pcl; p.joint = joint; p.order = order;
    p.wmat = (const uint4*)wmat; p.wvec = wvec;
    KPF_REQUIRE(e_batch_stride >= (long long)N * 256 && e_batch_stride % 8 == 0);
    p.e_out = (uint16_t*)e_out; p.e_bs = e_batch_stride; p.part_acc = part_acc; p.part_ms = part_ms; p.B = B; p.N = N; p.J = J; p.HW = HW;
    p.kernel_size = kernel_size; p.fmt = fmt;
    p.stage_out = (unsigned char*)stage_out; p.stage_in = (const unsigned char*)stage_in;
    const int st = stage_out ? 1 : stage_in ? 2 : 0;
    auto kern = fmt == FMT_F16 ? (st == 0 ? point_embed_kernel<FMT_F16, 0> : st == 1 ? point_embed_kernel<FMT_F16, 1> : point_embed_kernel<FMT_F16, 2>)
                               : (st == 0 ? point_embed_kernel<FMT_BF16, 0> : st == 1 ? point_embed_kernel<FMT_BF16, 1> : point_embed_kernel<FMT_BF16, 2>);
    cudaError_t e = kpf::set_smem(kern, PE_SMEM);
    if (e != cudaSuccess) return (int)e;
    const int tiles = B * (N / PE_TP);
    e = kpf::launch_pdl(kern, dim3(tiles < num_sms ? tiles : num_sms), dim3(PE_NT), PE_SMEM, stream, p);
    if (e != cudaSuccess) return (int)e;
    KPF_CHECK_LAUNCH();
    return 0;
}

static_assert(kpf::PE_STAGE_BYTES == KPF_POINT_EMBED_STAGE_BYTES_PER_TILE, "include/kpf_b200.h states the staged tile size");
