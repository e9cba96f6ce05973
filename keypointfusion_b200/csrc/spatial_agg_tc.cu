// K5 on tensor cores: depth-keypoint spatial attention + aggregation, model/model.py:334-344 (with K4c = a10, a11 fused).
// Same math as csrc/spatial_agg.cu (see there for the reference mapping); here both contractions are tcgen05 MMAs:
//
//   GEMM A   S1[hw][j]  = sum_c F[c][hw] Wa[j][c] + sum_j' hm[j'][hw] Wa[j][C+j']        M = 128 cells, N = 32, K = 128 + 32
//   epilogue sw = sigmoid(S1 + ba) -> global ; G[hw][j] = fc_w[hw] (sg GAM + (1-sg) sw)    (thread = cell)
//   GEMM B   out[c][j] += sum_hw relu(F[c][hw]) G[hw][j]                                   M = 128 channels, N = 32, K = 128 cells
//
// Split precision (csrc/tcgen05.cuh): the bf16 feature map is exact in one plane (fp32 maps arrive as two bf16 planes from
// kpf_split_planes); its GEMM partners (Wa's feature part, G) are THREE bf16 planes (both operands of an MMA must share a format);
// the heat map and Wa's heat-map part are two planes in format fmt.  fp32-class results.
// The NCHW feature tile [128 c x 128 hw] is staged ONCE per tile with 16-byte cp.async into the SWIZZLE_NONE canonical
// layout and read by GEMM A as an MN-major A operand (M = hw contiguous) and -- same bytes, LBO/SBO swapped, after an
// in-place relu pass -- by GEMM B as a K-major A operand (K = hw contiguous).  One CTA per sample sweeps its HW/128
// tiles, accumulating out[c][j] in TMEM; the next tile's features are prefetched while the current one is consumed.
#include "tcgen05.cuh"

namespace kpf {

struct SpatialParams {
    const __nv_bfloat16* feat;   // [B,128,HW]  (hi plane)
    const __nv_bfloat16* feat_lo;   // lo plane of an fp32 map, or null
    const float* joints;         // [B,J,3] (uvd)
    const float* depth;
    long long depth_bs;
    int depth_rs, depth_cs;
    const float *center, *M, *cube, *cam;
    const uint4* wa;             // canonical 16-bit planes: Wa[:, :128] as [16][32] x 3 bf16 planes, Wa[:, 128:] as [4][32] hi | lo (fmt)
    const float *ba, *weight_dis, *fc_w, *fc_b, *prev;
    float *sw_out, *feat_j_out;
    int B, J, fs;
    float img_size, flip, hm_std, hm_sigma, gamma;
    float* scratch;   // [B][split][128][32] partial out[c][j]
    int* counters;    // [B], zero on entry, zero again on exit
    int split, fmt;
};

constexpr int K5_NT = 512;   // thread = (cell or channel row = 32 * (warp % 4) + lane, joint group warp / 4 of 8 joints)

template <int FMT>
__global__ void __launch_bounds__(K5_NT, 1) spatial_aggregate_tc_kernel(const SpatialParams p) {
    extern __shared__ __align__(128) unsigned char k5_smem[];
    const bool has_lo = p.feat_lo != nullptr;
    const int NP = has_lo ? 2 : 1;                   // feature planes
    uint4* sHm = reinterpret_cast<uint4*>(k5_smem); // 2 planes x [4][128] heat-map rows, K-major A operand (K = 32 joints)
    const int NBUF = has_lo ? 1 : 2;                 // fp32 maps: two planes per tile leave no room for the prefetch buffer
    uint4* sG = sHm + 1024;                          // 3 bf16 planes x [16][4][8] G, MN-major B operand [K = 128 cells][N = 32]
    uint4* sWa = sG + 1536;                          // [16][32] x 3 bf16 planes, [4][32] hi | lo
    float* sJ = reinterpret_cast<float*>(sWa + 1792); // [32][8]: hm centre (x,y), xyz
    uint4* sF = reinterpret_cast<uint4*>(sJ + 256 + 32);   // [NBUF buffers][NP planes][2048] raw feature tile, index (c/8)*128 + (hw/8)*8 + (c%8)
    uint4* sFr = sF + NBUF * NP * 2048;              // [NP planes][2048] relu copy
    float* sBa = sJ + 256;                           // [32] atten_spatial bias
    float* sD2 = reinterpret_cast<float*>(sFr + NP * 2048);   // [2][32 joints][fs]: ((cell + 0.5 - centre) / std)^2 per column / per row
    constexpr int fmt = FMT;
    __shared__ __align__(8) uint64_t mma_bar;
    __shared__ uint32_t tmem_slot;
    __shared__ CamF cam;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = warp_index_uniform();  // MMA issue: one elected lane of warp 0 from warp-uniform code (tcgen05.cuh)
    const int q = warp & 3, cg = warp >> 2, row = 32 * q + lane;   // TMEM lane `row` (cell / channel), joints [8cg, 8cg + 8)
    const int b = blockIdx.x / p.split, sp = blockIdx.x - b * p.split, J = p.J, fs = p.fs, HW = fs * fs, T = HW / 128;
    const int t_begin = sp * (T / p.split), t_end = t_begin + T / p.split;
    __shared__ int s_last;
    const uint32_t ACC1 = 0, ACC2 = 32;
    pdl_launch_dependents();

    if (warp == 0) tmem_alloc(&tmem_slot, 64);
    if (tid == 0) {
        mbar_init(&mma_bar, 1);
        fence_mbar_init();
        load_cam(cam, b, p.center, p.M, p.cube, p.cam, p.img_size, p.flip);
    }
    for (int i = tid; i < 1792; i += K5_NT) sWa[i] = p.wa[i];
    if (tid < 32) sBa[tid] = tid < J ? p.ba[tid] : 0.f;
    const __nv_bfloat16* fb = p.feat + (size_t)b * 128 * HW;
    const __nv_bfloat16* fbl = has_lo ? p.feat_lo + (size_t)b * 128 * HW : nullptr;
    // tile loader: thread -> (c%8 = tid%8, hw8 = (tid/8)%16, channel group tid/128 + 4i): 16-byte cp.async, 128 contiguous bytes
    // of a channel row per 8 lanes
    // (parts [i0, i1) of the four: the prefetch of the NEXT tile is issued in four parts across an iteration, not as one burst that
    //  fills the memory-instruction queue in front of the geometry's and the epilogues' shared-memory accesses -- see desa_fused.cu)
    auto load_tile = [&](int t, uint4* dst, int i0 = 0, int i1 = 4) {
        const int c8 = tid & 7, hw8 = (tid >> 3) & 15;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (i < i0 || i >= i1) continue;
            const int cgp = (tid >> 7) + 4 * i;
            cp_async16(dst + cgp * 128 + hw8 * 8 + c8, fb + (size_t)(cgp * 8 + c8) * HW + t * 128 + hw8 * 8);
            if (has_lo) cp_async16(dst + 2048 + cgp * 128 + hw8 * 8 + c8, fbl + (size_t)(cgp * 8 + c8) * HW + t * 128 + hw8 * 8);
        }
    };
    load_tile(t_begin, sF);   // features, camera and weights are inputs of the step: fetched before the dependency wait
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_wait();   // joints / prev come from the previous kernels
    if (tid < J) {
        const float* s = p.joints + ((size_t)b * J + tid) * 3;
        sJ[8 * tid + 0] = (s[0] + 1.f) / 2.f * (float)fs;  // generateFeature.py:592-593
        sJ[8 * tid + 1] = (s[1] + 1.f) / 2.f * (float)fs;
        const float3 qj = uvd2xyz(cam, s[0], s[1], s[2]);  // loader.py:800
        sJ[8 * tid + 2] = qj.x;
        sJ[8 * tid + 3] = qj.y;
        sJ[8 * tid + 4] = qj.z;
    }
    const uint32_t tmem0 = tmem_slot, tmem = tmem0 + ((uint32_t)(32 * q) << 16);
    uint32_t phase = 0;
    const float sg = 1.f / (1.f + expf(-p.weight_dis[0]));
    const float inv2s2 = 1.f / (2.f * p.hm_sigma * p.hm_sigma);
    const float ffs = (float)fs;
    __syncthreads();
    // the heat map's squared, std-normalised distances are separable: one division per (joint, column) and (joint, row) instead
    // of two per (joint, cell); the sum and the exponential below are unchanged (bit-identical heat map)
    for (int i = tid; i < 2 * 32 * fs; i += K5_NT) {
        const int ax = i / (32 * fs), j = (i / fs) & 31, c = i - (i / fs) * fs;
        const float dd = j < J ? ((float)c + 0.5f - sJ[8 * j + ax]) / p.hm_std : 0.f;
        sD2[(ax * 32 + j) * fs + c] = dd * dd;
    }
    __syncthreads();

    // depth of this thread's cell, fetched one tile ahead (an L2 round trip at the head of every tile otherwise)
    auto cell_depth = [&](int t) {
        const int m = t * 128 + row, r = m / fs, col = m - r * fs;
        return __ldg(p.depth + (size_t)b * p.depth_bs + (size_t)r * p.depth_rs + (size_t)col * p.depth_cs);
    };
    float d_next = cell_depth(t_begin);
    bool gemm_b_pending = false;   // GEMM B of the previous tile: waited for only where its operands are rewritten
    for (int t = t_begin; t < t_end; ++t) {
        uint4* cur = sF + ((t - t_begin) & (NBUF - 1)) * NP * 2048;
        if (NBUF == 1 && t > t_begin) load_tile(t, sF);   // single buffer: its readers (tile t-1's MMAs) were waited for
        cp_async_wait_all();   // this thread's part of tile t has landed ...
        __syncthreads();       // ... and everybody's; the other buffer's readers (tile t-1) are done
        const bool prefetch = NBUF == 2 && t + 1 < t_end;   // overlaps the whole iteration
        uint4* nxt = sF + ((t + 1 - t_begin) & 1) * NP * 2048;
        if (prefetch) load_tile(t + 1, nxt, 0, 1);
        // ---- per-cell geometry (thread = cell `row`, joints [8cg, 8cg + 8)): heat-map chunk (A operand) and GAM (registers)
        const int m = t * 128 + row, r = m / fs, col = m - r * fs;
        const float d = d_next;
        if (t + 1 < t_end) d_next = cell_depth(t + 1);
        const float3 qc = uvd2xyz(cam, cell_coord(col, ffs), cell_coord(r, ffs), d);   // same arithmetic as the fp32 kernel (spatial_agg.cu)
        float gam[8], hm[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int j = 8 * cg + i;
            if (j < J) {
                hm[i] = expf(-(sD2[j * fs + col] + sD2[(32 + j) * fs + r]) * inv2s2);
                const float ex = qc.x - sJ[8 * j + 2], ey = qc.y - sJ[8 * j + 3], ez = qc.z - sJ[8 * j + 4];
                gam[i] = 1.f / (p.gamma * (ex * ex + ey * ey + ez * ez) + 1.f);
            } else {
                hm[i] = 0.f;
                gam[i] = 0.f;
            }
        }
        if (gemm_b_pending) {   // the geometry above ran under GEMM B of tile t - 1; sHm / sFr / sG are rewritten from here on
            mbar_wait(&mma_bar, phase);
            phase ^= 1;
            tc_fence_after();
            gemm_b_pending = false;
        }
        {
            uint4 oh, ol;
            split8<FMT>(hm, oh, ol);
            sHm[cg * 128 + row] = oh;
            sHm[512 + cg * 128 + row] = ol;
        }
        if (prefetch) load_tile(t + 1, nxt, 1, 2);
        // relu copy for GEMM B (same layout)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            uint4 v = cur[tid + i * K5_NT];
            uint32_t* h = reinterpret_cast<uint32_t*>(&v);
            uint32_t keep[4];   // 0xffff per 16-bit element whose hi plane is positive: relu(hi + lo) keeps or drops both planes together
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                keep[k] = ((h[k] & 0x8000u) ? 0u : 0xffffu) | ((h[k] & 0x80000000u) ? 0u : 0xffff0000u);
                h[k] &= keep[k];
            }
            sFr[tid + i * K5_NT] = v;
            if (has_lo) {
                uint4 l = cur[2048 + tid + i * K5_NT];
                l.x &= keep[0];
                l.y &= keep[1];
                l.z &= keep[2];
                l.w &= keep[3];
                sFr[2048 + tid + i * K5_NT] = l;
            }
        }
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                // GEMM A: A = F tile MN-major (LBO 2048 between channel groups, SBO 128 between cell groups), bf16 plane(s);
                //         B = Wa's feature part, three bf16 planes
                const uint32_t fa = smem_u32(cur);
                umma_gemm_map_x3(tmem0 + ACC1, fa, has_lo ? fa + 2048 * 16 : 0u, 2048, 128, smem_u32(sWa), 512 * 16, 512, 128,
                                 umma_idesc_f16(128, 32, true, false, FMT_BF16, FMT_BF16), 128, false);
                SmemOp a, bo;
                a.hi = smem_u32(sHm); a.lo = a.hi + 512 * 16; a.lbo = 2048; a.sbo = 128;
                bo.hi = smem_u32(sWa + 1536); bo.lo = bo.hi + 128 * 16; bo.lbo = 512; bo.sbo = 128;
                umma_gemm3_ss<32>(tmem0 + ACC1, a, bo, umma_idesc_f16(128, 32, false, false, fmt, fmt), true);
                umma_commit(&mma_bar);
            }
            __syncwarp();
        }
        const float fw = __ldg(p.fc_w + m);
        if (prefetch) load_tile(t + 1, nxt, 2, 3);
        mbar_wait(&mma_bar, phase);
        phase ^= 1;
        tc_fence_after();
        {
            float s1[8];
            tmem_ld<8>(tmem + ACC1 + 8 * cg, s1);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int j = 8 * cg + i;
                if (j < J) {
                    const float swv = 1.f / (1.f + expf(-(s1[i] + sBa[j])));
                    p.sw_out[((size_t)b * J + j) * HW + m] = swv;
                    s1[i] = fw * (sg * gam[i] + (1.f - sg) * swv);  // model.py:337-338 and fc_spatial2joint_feature's weight
                } else {
                    s1[i] = 0.f;
                }
            }
            uint4 oh, om, ol;
            split8x3_bf16(s1, oh, om, ol);
            sG[(row >> 3) * 32 + cg * 8 + (row & 7)] = oh;
            sG[512 + (row >> 3) * 32 + cg * 8 + (row & 7)] = om;
            sG[1024 + (row >> 3) * 32 + cg * 8 + (row & 7)] = ol;
        }
        if (prefetch) load_tile(t + 1, nxt, 3, 4);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                // GEMM B: A = relu(F) tile read K-major (K = cells): LBO 128 between cell groups, SBO 2048 between channel groups
                const uint32_t fr = smem_u32(sFr);
                umma_gemm_map_x3(tmem0 + ACC2, fr, has_lo ? fr + 2048 * 16 : 0u, 128, 2048, smem_u32(sG), 512 * 16, 512, 128,
                                 umma_idesc_f16(128, 32, false, true, FMT_BF16, FMT_BF16), 128, t > t_begin);
                umma_commit(&mma_bar);
            }
            __syncwarp();
        }
        gemm_b_pending = true;
    }
    mbar_wait(&mma_bar, phase);   // the last tile's GEMM B
    phase ^= 1;
    tc_fence_after();
    {
        float o[8];
        tmem_ld<8>(tmem + ACC2 + 8 * cg, o);  // thread = (channel `row`, joints [8cg, 8cg + 8)): this CTA's partial out[c][j]
        if (p.split > 1) {
            // deterministic cross-CTA reduction: publish the partial, the last CTA of the sample sums them in split order
            float4* dst = reinterpret_cast<float4*>(p.scratch + (((size_t)b * p.split + sp) * 128 + row) * 32 + 8 * cg);
            dst[0] = make_float4(o[0], o[1], o[2], o[3]);
            dst[1] = make_float4(o[4], o[5], o[6], o[7]);
            __threadfence();
            __syncthreads();
            if (tid == 0) s_last = (atomicAdd(p.counters + b, 1) == p.split - 1);
            __syncthreads();
            if (s_last) {
                __threadfence();
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] = 0.f;
                for (int qq = 0; qq < p.split; ++qq) {
                    const float4* src = reinterpret_cast<const float4*>(p.scratch + (((size_t)b * p.split + qq) * 128 + row) * 32 + 8 * cg);
                    const float4 v0 = __ldcg(src), v1 = __ldcg(src + 1);
                    o[0] += v0.x;
                    o[1] += v0.y;
                    o[2] += v0.z;
                    o[3] += v0.w;
                    o[4] += v1.x;
                    o[5] += v1.y;
                    o[6] += v1.z;
                    o[7] += v1.w;
                }
                if (tid == 0) p.counters[b] = 0;  // ready for the next launch / graph replay
            }
        }
        if (p.split == 1 || s_last) {
            const float fb0 = p.fc_b[0];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int j = 8 * cg + i;
                if (j < J) {
                    float v = o[i] + fb0;
                    const size_t idx = ((size_t)b * J + j) * 128 + row;
                    if (p.prev) v = fmaxf((v + p.prev[idx]) * 0.5f, 0.f);  // model.py:343-344
                    p.feat_j_out[idx] = v;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem0, 64);
}

}  // namespace kpf

// fp32 -> two bf16 planes (hi = rn(x), lo = rn(x - hi)), elementwise: how an fp32 feature map enters the split-precision kernels
__global__ void __launch_bounds__(256) split_planes_kernel(const float4* __restrict__ x, long long n4, uint2* __restrict__ hi, uint2* __restrict__ lo) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = __ldg(x + i);
        uint2 h, l;
        kpf::split2<kpf::FMT_BF16>(v.x, v.y, h.x, l.x);
        kpf::split2<kpf::FMT_BF16>(v.z, v.w, h.y, l.y);
        hi[i] = h;
        lo[i] = l;
    }
}

extern "C" int kpf_split_planes(const float* x, long long n, void* hi, void* lo, cudaStream_t stream) {
    KPF_REQUIRE(n >= 0 && n % 4 == 0 && ((uintptr_t)x % 16) == 0 && ((uintptr_t)hi % 8) == 0 && ((uintptr_t)lo % 8) == 0);
    if (n == 0) return 0;
    const long long n4 = n / 4;
    const int grid = (int)((n4 + 255) / 256 < 148 * 8 ? (n4 + 255) / 256 : 148 * 8);
    split_planes_kernel<<<grid, 256, 0, stream>>>((const float4*)x, n4, (uint2*)hi, (uint2*)lo);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_spatial_aggregate_tc(const void* feat_rgb, const void* feat_rgb_lo, const float* joints, const float* depth, long long depth_bs, int depth_rs,
                                        int depth_cs, const float* center, const float* M, const float* cube, const float* cam,
                                        const void* wa_packed, const float* ba, const float* weight_dis, const float* fc_w,
                                        const float* fc_b, const float* prev, int B, int C, int J, int fs, float img_size, float flip,
                                        float hm_std, float hm_sigma, float gamma, int fmt, float* sw_out, float* feat_j_out, float* scratch,
                                        int* counters, int split, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && C == 128 && J >= 1 && J <= 32 && fs >= 1 && (fs * fs) % 128 == 0);
    KPF_REQUIRE(((uintptr_t)feat_rgb % 16) == 0 && ((uintptr_t)feat_rgb_lo % 16) == 0 && ((uintptr_t)wa_packed % 16) == 0);
    KPF_REQUIRE(fmt == FMT_F16 || fmt == FMT_BF16);
    if (B == 0) return 0;
    KPF_REQUIRE(split >= 1 && ((fs * fs) / 128) % split == 0 && (split == 1 || (scratch != nullptr && counters != nullptr)));
    SpatialParams p;
    p.feat = (const __nv_bfloat16*)feat_rgb; p.feat_lo = (const __nv_bfloat16*)feat_rgb_lo; p.fmt = fmt; p.joints = joints; p.depth = depth; p.depth_bs = depth_bs; p.depth_rs = depth_rs;
    p.depth_cs = depth_cs; p.center = center; p.M = M; p.cube = cube; p.cam = cam; p.wa = (const uint4*)wa_packed; p.ba = ba;
    p.weight_dis = weight_dis; p.fc_w = fc_w; p.fc_b = fc_b; p.prev = prev; p.sw_out = sw_out; p.feat_j_out = feat_j_out;
    p.scratch = scratch; p.counters = counters; p.split = split;
    p.B = B; p.J = J; p.fs = fs; p.img_size = img_size; p.flip = flip; p.hm_std = hm_std; p.hm_sigma = hm_sigma; p.gamma = gamma;
    const int NP = feat_rgb_lo ? 2 : 1, NBUF = feat_rgb_lo ? 1 : 2;
    const size_t smem = (size_t)(1024 + 1536 + 1792 + (NBUF + 1) * NP * 2048) * 16 + 32 * 8 * 4 + 32 * 4 + (size_t)2 * 32 * fs * 4;
    KPF_REQUIRE(smem <= 227 * 1024);
    auto kern = fmt == FMT_F16 ? spatial_aggregate_tc_kernel<FMT_F16> : spatial_aggregate_tc_kernel<FMT_BF16>;
    cudaError_t e = kpf::set_smem(kern, smem);
    if (e != cudaSuccess) return (int)e;
    {
        cudaError_t le = kpf::launch_pdl(kern, dim3(B * split), dim3(K5_NT), smem, stream, p);
        if (le != cudaSuccess) return (int)le;
    }
    KPF_CHECK_LAUNCH();
    return 0;
}
