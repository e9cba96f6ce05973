// DESA on tensor cores (model/model.py:129-204 + the joint embeddings :323-325), SURVEY.md 8f-1.  Split precision throughout
// (csrc/tcgen05.cuh): every operand is two 16-bit planes, three MMAs per product, so the results are fp32-class.  The point
// features e arrive as rows [hi 128 | lo 128] (kpf_point_embed); the tile kernel keeps each scale's W1 / W2 planes in TENSOR
// MEMORY as the A operands (256 of the 512 columns), which frees their shared memory for the second plane of the activations.
// Two kernels:
//
// desa_prep_kernel   512 threads, two independent roles side by side in one launch:
//             CTA per sample:  combine the point stage's softmax partials (flash-style) -> joint_agg[J][128]
//                              jf = relu(Wj [joint_agg | joint_xyz] + b)    (model.py:323-325)   tcgen05 + fp32 xyz term
//                              jf is also appended, in bf16, as rows N.. of the point-feature tensor e (the joints are members
//                              of the grouped set, model.py:168-169), and cj[s][j] = W1_s jf[j] is computed for every scale
//             CTA per (sample, scale): ball query (pointnet2_ops semantics) of the J joints over the N points + the J joints
//                              themselves -> idx[b][scale][j][nsample]; the scale-0 CTA also writes a padded xyz table
// desa_tile_kernel   persistent, one CTA per SM, 16 worker warps + 1 issuer warp.  Work item = (scale, sample, tile of 128/NS
//             joints), NS = rows grouped per joint = nsample, or 16 / 32 for a scale whose widest ball of the launch holds no more
//             points than that (the padding copies of the first hit are not multiplied: same maxima, fewer tiles); every CTA takes
//             a contiguous, scale-major range so the scale's weights stay resident:
//             X = [feat[idx] - jf[j] | (xyz[idx] - c_j)/r]  ->  h = relu(W1 X + b1)  ->  relu(W2 h + b2)  -> max over nsample,
//             evaluated as h = relu(W1 [feat[idx] | (xyz[idx] - c_j)/r] - cj + b1): layer 1 reads the RAW gathered rows, so the
//             gather is a cp.async copy (128-byte requests) straight into the operand and cj is subtracted in the epilogue.
//             Both GEMMs are computed transposed -- D[c][row] = sum_k W[c][k] X[row][k], weight = M=128 A operand, activations =
//             N operand -- so thread (lane quarter, column group) owns OUTPUT CHANNEL c and DESA's max-pool over the grouped
//             points of a joint is a per-thread register reduction.  Software pipeline per iteration s: GEMM2(s) and GEMM1(s+1)
//             are issued together; while they run the rows of tile s+2 are copied (indices fetched one iteration earlier);
//             then epilogue 2 of s and epilogue 1 of s+1.  One __syncthreads per tile.
//   output    desa_part[b][scale][j][:], jf[b][j][:]; the 512->128 fusion conv follows in kpf_token_stack.
#include "tcgen05.cuh"

namespace kpf {

struct DesaParams {
    uint16_t* e;              // [B][N + J][256] point features, rows = [hi 128 | lo 128] 16-bit planes (kpf_point_embed, batch stride
    long long e_bs;           //   e_bs elements); rows N.. = the joint features (prep)
    const float* part_acc;    // [B,T,128,32]
    const float* part_ms;     // [B,T,2,32]
    const float* pcl;         // [B,N,3]
    const float* joint;       // [B,J,3]
    const uint4* wmat;        // canonical (hi | lo) planes: Wj 2 x [16][128] ; per scale: W1 main 2 x [16][128], W1 tail 2 x [2][128], W2 2 x [16][128]
    const float* wvec;        // bj[128], Wjx[128][4] ; per scale: b1[128], b2[128]
    float* desa_part;         // [B,S,J,128]
    float* jf_out;            // [B,J,128]
    const float* jf_in;       // null, or [B,J,128]: the joints' features are GIVEN (stand-alone DESA.forward); the embedding is skipped
    float* cj;                // scratch [B,S,J,128]: W1_s jf[j] (fp32), subtracted in the tile kernel's layer-1 epilogue
    float4* xyz4;             // scratch [B][N + 32]: xyz of the grouped point set (N points, then the J joints), one 16-byte load each
    uint16_t* idx;            // scratch [B,S,J,nsample] ball-query indices (>= N: one of the joints)
    int* gw;                  // scratch [B,S]: the largest ball population (capped at nsample) among the sample's J balls of a scale
    int B, N, J, T, S, nsample, fmt;
    float radius[4];
};

constexpr int DS_NT = 512;
constexpr int DS_MAT_PER_SCALE = 2 * (2048 + 256 + 2048);
constexpr int DS_XBUF = 2 * (2048 + 128);   // uint4 per activation buffer: main hi | main lo | K tail hi | K tail lo (one 16-byte chunk per row:
                                            // the tail's second k-chunk is all zero and never stored, the descriptor re-reads the first)

// ================================================================================================ prep
// Two roles in one launch: CTAs [0, B) embed the joints of one sample (softmax-partial combine + tcgen05 GEMM); CTAs
// [B, B + B*S) run the ball query of one (sample, scale).  The roles are independent and run side by side on different SMs.
template <int FMT>
__global__ void __launch_bounds__(DS_NT, 1) desa_prep_kernel(const DesaParams p) {
    extern __shared__ __align__(128) unsigned char ds_smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int J = p.J, N = p.N, T = p.T, NS = p.nsample, S = p.S;
    pdl_launch_dependents();

    if ((int)blockIdx.x >= p.B) {
        // ================= ball query (pointnet2_ops: first NS hits in index order, padded with the first hit) =================
        // one CTA per sample, all S scales: the distances are computed once and compared against every radius
        const int b = blockIdx.x - p.B;
        pdl_wait();
        float4* sPcl = reinterpret_cast<float4*>(ds_smem);                          // [N + J] xyz
        uint32_t* sMask = reinterpret_cast<uint32_t*>(sPcl + (N + J + 3) / 4 * 4);   // [S][J][NW] hit words (bit = point)
        __shared__ int sGw[4];
        if (tid < 4) sGw[tid] = 0;
        for (int i = tid; i < N + J; i += DS_NT) {
            const float* s = i < N ? p.pcl + ((size_t)b * N + i) * 3 : p.joint + ((size_t)b * J + (i - N)) * 3;
            sPcl[i] = make_float4(s[0], s[1], s[2], 0.f);
        }
        __syncthreads();
        for (int i = tid; i < N + J; i += DS_NT) p.xyz4[(size_t)b * (N + 32) + i] = sPcl[i];
        // Phase 1: thread = (32-point word, centre): lane = centre j, warp = word.  Every lane walks the word's 32 points (one
        // broadcast shared-memory read per point), computes d2 ONCE in the exact fp32 op order and sets the point's bit in the hit
        // word of every scale whose r^2 it is under.  No ballots, no cross-lane traffic; hit word layout sMask[(sc J + j) NW + word].
        const int NW = (N + J + 31) / 32;
        float r2[4];
#pragma unroll
        for (int sc = 0; sc < 4; ++sc) r2[sc] = xmul(p.radius[sc < S ? sc : 0], p.radius[sc < S ? sc : 0]);
        if (lane < J) {
            const float4 c = sPcl[N + lane];
            for (int wi = warp; wi < NW; wi += DS_NT / 32) {
                uint32_t m0 = 0u, m1 = 0u, m2 = 0u, m3 = 0u;
                const int n0 = wi * 32, cnt = min(32, N + J - n0);
#pragma unroll 4
                for (int i = 0; i < cnt; ++i) {
                    const float4 q = sPcl[n0 + i];
                    const float dx = xsub(c.x, q.x), dy = xsub(c.y, q.y), dz = xsub(c.z, q.z);
                    const float d2 = xadd(xadd(xmul(dx, dx), xmul(dy, dy)), xmul(dz, dz));
                    const uint32_t bit = 1u << i;
                    m0 |= d2 < r2[0] ? bit : 0u;
                    m1 |= d2 < r2[1] ? bit : 0u;
                    m2 |= d2 < r2[2] ? bit : 0u;
                    m3 |= d2 < r2[3] ? bit : 0u;
                }
                sMask[(0 * J + lane) * NW + wi] = m0;
                if (S > 1) sMask[(1 * J + lane) * NW + wi] = m1;
                if (S > 2) sMask[(2 * J + lane) * NW + wi] = m2;
                if (S > 3) sMask[(3 * J + lane) * NW + wi] = m3;
            }
        }
        __syncthreads();
        // Phase 2: one warp per centre: popcount prefix over its hit words, then every lane expands the set bits of its word(s)
        // into their slots
        for (int pj = warp; pj < S * J; pj += DS_NT / 32) {   // pj = sc * J + j: the layout of sMask and of idx[b]
            const uint32_t* wj = sMask + pj * NW;
            uint16_t* out = p.idx + ((size_t)b * S * J + pj) * NS;
            int carry = 0, first = -1;
            for (int w0 = 0; w0 < NW && carry < NS; w0 += 32) {
                const int wi = w0 + lane;
                uint32_t word = wi < NW ? wj[wi] : 0u;
                const int cntw = __popc(word);
                int incl = cntw;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                int slot = carry + incl - cntw;
                const uint32_t nz = __ballot_sync(0xffffffffu, word != 0u);
                if (first < 0 && nz) {
                    const int fl = __ffs(nz) - 1;
                    const uint32_t fw = __shfl_sync(0xffffffffu, word, fl);
                    first = (w0 + fl) * 32 + __ffs(fw) - 1;
                }
                while (word && slot < NS) {
                    const int bit = __ffs(word) - 1;
                    out[slot] = (uint16_t)(wi * 32 + bit);
                    word &= word - 1;
                    ++slot;
                }
                carry += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (first < 0) first = 0;
            const int cnt = carry < NS ? carry : NS;
            for (int s2 = cnt + lane; s2 < NS; s2 += 32) out[s2] = (uint16_t)first;
            if (lane == 0) atomicMax(&sGw[pj / J], cnt);
        }
        // the widest ball of each scale: the tile kernel groups only as many rows per joint as the widest ball of the launch needs
        __syncthreads();
        if (tid < S) p.gw[(size_t)b * S + tid] = sGw[tid];
        return;
    }

    // ================= joint embedding: jf = relu(Wj [joint_agg | joint_xyz] + b)  (model.py:319-325) =================
    uint4* sWj = reinterpret_cast<uint4*>(ds_smem);             // 2 planes x [16][128] K-major A operand: Wj, later W1 of scale 2 (3)
    uint4* sW1 = sWj + 4096;                                     // [2] such buffers: W1 of scales 0 and 1, prefetched at kernel start
    uint4* sAgg = sW1 + 2 * 4096;                                // 2 planes x MN-major B operand [16][4][8]: joint_agg[channel][joint]
    float* sMS = reinterpret_cast<float*>(sAgg + 1024);          // [T][2][32] partial max/sum -> [T][32] factors + den[32]
    float4* sJ = reinterpret_cast<float4*>(sMS + T * 64 + 64);   // [32] joint xyz
    __shared__ __align__(8) uint64_t wbar, w1bar[2], mma_bar;
    __shared__ uint32_t tmem_slot;
    const int warp_u = warp_index_uniform();
    const int b = blockIdx.x;
    if (warp == 0) tmem_alloc(&tmem_slot, 128);   // accumulators: jf [0, 32), cj of the scales in flight [32, 128)
    if (tid == 0) {
        mbar_init(&wbar, 1);
        mbar_init(&w1bar[0], 1);
        mbar_init(&w1bar[1], 1);
        mbar_init(&mma_bar, 1);
        fence_mbar_init();
        mbar_expect_tx(&wbar, 4096 * 16);
        tma_bulk_g2s(sWj, p.wmat, 4096 * 16, &wbar);
        for (int sc = 0; sc < 2 && sc < S; ++sc) {   // the first two scales' W1 (weights: no dependence on the previous kernel)
            mbar_expect_tx(&w1bar[sc], 4096 * 16);
            tma_bulk_g2s(sW1 + sc * 4096, p.wmat + 4096 + (size_t)sc * DS_MAT_PER_SCALE, 4096 * 16, &w1bar[sc]);
        }
    }
    constexpr int fmt = FMT;
    // A = the weight planes in sWj, B = joint_agg / jf planes in sAgg
    const SmemOp opW = smem_op_k_outer(smem_u32(sWj), 128, 128), opA = smem_op_k_outer(smem_u32(sAgg), 32, 128);
    const uint32_t id_jf = umma_idesc_f16(128, 32, false, true, fmt, fmt);
    pdl_wait();   // weights only so far
    if (tid < 32) {
        const float* s = p.joint + ((size_t)b * J + (tid < J ? tid : 0)) * 3;
        sJ[tid] = tid < J ? make_float4(s[0], s[1], s[2], 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const bool given = p.jf_in != nullptr;
    if (!given)
        for (int i = tid; i < T * 64; i += DS_NT) sMS[i] = p.part_ms[(size_t)b * T * 64 + i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = tmem_slot;
    uint32_t mph = 0;   // mma_bar phase
    // scale factors exp(m_t - m) and the softmax denominator, per joint
    if (!given && tid < 32) {
        float m = -INFINITY;
        for (int t = 0; t < T; ++t) m = fmaxf(m, sMS[t * 64 + tid]);
        float den = 0.f;
        for (int t = 0; t < T; ++t) {
            const float f = __expf(sMS[t * 64 + tid] - m);
            den += sMS[t * 64 + 32 + tid] * f;
            sMS[t * 64 + tid] = f;
        }
        sMS[T * 64 + tid] = den;
    }
    __syncthreads();
    // ---- joint_agg[c][j] (softmax over all N points of the gathered weight map): 8 lanes read one channel's 128-byte row of
    //      a partial per load (4 L1 wavefronts per warp load); thread = (channel, 4 joints), two channel halves
    if (!given) {
        const int jq = lane & 7;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int ch = 64 * half + 4 * warp + (lane >> 3);
            float agg[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
            for (int t = 0; t < T; ++t) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(p.part_acc + (((size_t)b * T + t) * 128 + ch) * 32) + jq);
                const float* f = sMS + t * 64 + 4 * jq;
                agg[0] += v.x * f[0];
                agg[1] += v.y * f[1];
                agg[2] += v.z * f[2];
                agg[3] += v.w * f[3];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) agg[j] = (4 * jq + j) < J ? agg[j] / sMS[T * 64 + 4 * jq + j] : 0.f;
            uint2 oh, ol;
            split2<FMT>(agg[0], agg[1], oh.x, ol.x);
            split2<FMT>(agg[2], agg[3], oh.y, ol.y);
            // (k = channel, n = joint), n contiguous: chunk jq / 2 of the row, half jq & 1
            reinterpret_cast<uint2*>(sAgg + (ch >> 3) * 32 + (jq >> 1) * 8 + (ch & 7))[jq & 1] = oh;
            reinterpret_cast<uint2*>(sAgg + 512 + (ch >> 3) * 32 + (jq >> 1) * 8 + (ch & 7))[jq & 1] = ol;
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp_u == 0) {
        tc_fence_after();
        mbar_wait(&wbar, 0);   // (also when the embedding is skipped: the buffer is refilled below)
        if (!given) {
            if (elect_one()) {
                umma_gemm3_ss<128>(tmem0, opW, opA, id_jf, false);
                umma_commit(&mma_bar);
            }
            __syncwarp();
        }
    }
    if (!given) {
        mbar_wait(&mma_bar, mph);
        mph ^= 1;
        tc_fence_after();
    }
    if (tid == 0 && S > 2) {   // Wj has been read (or was never needed): its buffer takes W1 of scale 2 while the epilogue runs
        mbar_expect_tx(&wbar, 4096 * 16);
        tma_bulk_g2s(sWj, p.wmat + 4096 + (size_t)2 * DS_MAT_PER_SCALE, 4096 * 16, &wbar);
    }
    const int q = warp & 3, cg = warp >> 2, ch = 32 * q + lane;   // channel 32q + lane, joints [8cg, 8cg + 8)
    const uint32_t tmem_q = tmem0 + ((uint32_t)(32 * q) << 16);
    {   // jf[j][ch]
        float d[8];
        if (!given) tmem_ld<8>(tmem_q + 8 * cg, d);
        const float bj = p.wvec[ch];
        const float4 wx = *reinterpret_cast<const float4*>(p.wvec + 128 + 4 * ch);
        uint16_t* erow = p.e + (size_t)b * p.e_bs + (size_t)N * 256 + ch;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int j = 8 * cg + i;
            float v = 0.f;
            if (j < J) {
                const float4 c = sJ[j];
                v = given ? __ldg(p.jf_in + ((size_t)b * J + j) * 128 + ch) : fmaxf(d[i] + bj + wx.x * c.x + wx.y * c.y + wx.z * c.z, 0.f);
                if (p.jf_out) p.jf_out[((size_t)b * J + j) * 128 + ch] = v;
                uint32_t h2, l2;   // the joints are points N .. N+J-1 of the grouped set (model.py:168-169)
                split2<FMT>(v, 0.f, h2, l2);
                erow[(size_t)j * 256] = (uint16_t)h2;
                erow[(size_t)j * 256 + 128] = (uint16_t)l2;
            }
            d[i] = v;
        }
        // jf as the B operand [K = channel][N = joint] of the W1 jf GEMMs (same layout as sAgg, whose reader has completed)
        uint4 oh, ol;
        split8<FMT>(d, oh, ol);
        sAgg[(ch >> 3) * 32 + cg * 8 + (ch & 7)] = oh;
        sAgg[512 + (ch >> 3) * 32 + cg * 8 + (ch & 7)] = ol;
    }
    // ---- cj[s][j][:] = W1_s jf[j] for every scale: the tile kernel feeds the RAW gathered point features to its layer-1 GEMM and
    //      subtracts this term in the epilogue ( W1 (feat - jf) = W1 feat - W1 jf ), so its gather is a pure copy
    //      Scales 0..2 are issued back to back into their own accumulators (weights already in shared memory); a fourth scale
    //      reuses buffer 0 afterwards.
    const int S3 = S < 3 ? S : 3;
    fence_proxy_async();   // sAgg (generic-proxy writes) -> the MMAs' async-proxy reads
    tc_fence_before();
    __syncthreads();
    if (warp_u == 0) {
        tc_fence_after();
        for (int sc = 0; sc < S3; ++sc) {
            if (sc < 2) mbar_wait(&w1bar[sc], 0);
            else mbar_wait(&wbar, 1);
            if (elect_one()) {
                const SmemOp w = sc < 2 ? smem_op_k_outer(smem_u32(sW1 + sc * 4096), 128, 128) : opW;
                umma_gemm3_ss<128>(tmem0 + 32 * (sc + 1), w, opA, id_jf, false);
            }
            __syncwarp();
        }
        if (elect_one()) umma_commit(&mma_bar);
        __syncwarp();
    }
    mbar_wait(&mma_bar, mph);
    mph ^= 1;
    tc_fence_after();
    for (int sc = 0; sc < S3; ++sc) {
        float d[8];
        tmem_ld<8>(tmem_q + 32 * (sc + 1) + 8 * cg, d);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int j = 8 * cg + i;
            if (j < J) p.cj[(((size_t)b * S + sc) * J + j) * 128 + ch] = d[i];
        }
    }
    if (S > 3) {   // fourth scale: buffer 0 again (its GEMM has completed), accumulator 1 (read above)
        tc_fence_before();
        __syncthreads();
        if (warp_u == 0) {
            if (elect_one()) {
                mbar_expect_tx(&w1bar[0], 4096 * 16);
                tma_bulk_g2s(sW1, p.wmat + 4096 + (size_t)3 * DS_MAT_PER_SCALE, 4096 * 16, &w1bar[0]);
            }
            __syncwarp();
            tc_fence_after();
            mbar_wait(&w1bar[0], 1);
            if (elect_one()) {
                umma_gemm3_ss<128>(tmem0 + 32, smem_op_k_outer(smem_u32(sW1), 128, 128), opA, id_jf, false);
                umma_commit(&mma_bar);
            }
            __syncwarp();
        }
        mbar_wait(&mma_bar, mph);
        mph ^= 1;
        tc_fence_after();
        float d[8];
        tmem_ld<8>(tmem_q + 32 + 8 * cg, d);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int j = 8 * cg + i;
            if (j < J) p.cj[(((size_t)b * S + 3) * J + j) * 128 + ch] = d[i];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem0, 128);
}

// ================================================================================================ tiles
constexpr int DS_TILE_NT = DS_NT + 32;   // 16 worker warps + one warp that only issues MMAs / TMA copies

struct DesaItem {   // (scale, sample, first joint) of a work item, advanced incrementally (no divisions in the loop)
    int sc, b, j0;
};

template <int FMT>
__global__ void __launch_bounds__(DS_TILE_NT, 1) desa_tile_kernel(const DesaParams p) {
    extern __shared__ __align__(128) unsigned char ds_smem[];
    uint4* sW1t = reinterpret_cast<uint4*>(ds_smem);  // W1's K tail (the xyz columns), 2 planes x [2][128]; W1 main / W2 live in tensor memory
    // Three activation buffers, tile t lives in buffer t % 3 for three iterations: its gathered rows are copied in (K-major B operand of
    // layer 1: 2 planes x [16 row groups][16 k-chunks][8 rows] + 2 planes x tail [16][2][8]); once layer 1 has read them, the layer-1
    // epilogue writes h = relu(.) over the SAME bytes (MN-major B operand of layer 2: 2 planes x [16][16][8]); layer 2 reads it one
    // iteration later.  No separate h buffer, so the epilogue of tile t + 1 never waits for layer 2 of tile t to release one.
    uint4* sX = sW1t + 512;
    float* sPart = reinterpret_cast<float*>(sX + 3 * DS_XBUF);   // [2][4][128] per-column-group maxima
    float4* sXyz = reinterpret_cast<float4*>(sPart + 1024);   // [2][128][2] xyz of a tile's grouped points and of their centres (cp.async staging)
    __shared__ __align__(8) uint64_t wbar, g1_bar, g2_bar;
    __shared__ uint32_t tmem_slot;
    __shared__ int sGw[4], sNs[4], sBase[5];   // per scale: widest ball of the launch, rows grouped per joint, first work item

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int warp_u = warp_index_uniform();
    const bool issuer = warp_u == DS_NT / 32;                     // warp 16: MMA / TMA issue only
    const int q = warp & 3, cg = (warp >> 2) & 3, ch = 32 * q + lane;   // epilogues: channel ch, tile rows [32cg, 32cg + 32)
    // gather: a thread copies its part of tile rows r and r + 64; lane = (row & 3, g8): the eight g8 lanes of a row read 128
    // contiguous bytes per cp.async, i.e. ONE 128-byte request per row half instead of eight 16-byte ones -- the copy is bound by
    // the number of requests the SM can keep in flight, not by bytes
    const int r = 4 * (warp & 15) + (lane & 3), g8 = lane >> 2;
    const int J = p.J, N = p.N, NSTRIDE = p.nsample, S = p.S, B = p.B;
    // Rows grouped per joint.  pointnet2's ball query pads a ball of fewer than nsample hits with copies of its first hit, and a max
    // over copies is the max over the originals: a scale whose widest ball (over the whole launch, desa_prep's gw) holds <= 16 / 32
    // points is grouped NS = 16 / 32 rows per joint instead of nsample -- 8 / 4 joints per 128-row tile, bit-identical maxima, a
    // quarter / half of the tiles.  NS, JPT, TPS, ns_shift are constants of a RUN (items of one scale), set at the top of each run.
    int NS = NSTRIDE, JPT = 128 / NS, TPS = (J + JPT - 1) / JPT;  // joints per tile, tiles per (sample, scale)
    int ns_shift = 31 - __clz(NS);                                // NS is a power of two: joint of tile row x = x >> ns_shift
    const uint32_t ACC1 = 0, ACC2 = 128, TW1_HI = 256, TW1_LO = 320, TW2_HI = 384, TW2_LO = 448;   // TMEM columns
    constexpr int fmt = FMT;
    pdl_launch_dependents();
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 0) {
        mbar_init(&wbar, 1);
        mbar_init(&g1_bar, 1);
        mbar_init(&g2_bar, 1);
        fence_mbar_init();
    }
    if (tid < 4) sGw[tid] = 0;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = tmem_slot, tmem = tmem0 + ((uint32_t)(32 * q) << 16);
    uint32_t g1_phase = 0, g2_phase = 0, w_phase = 0;
    pdl_wait();   // indices, W1 jf terms and point features come from the previous kernels

    for (int i = tid; i < B * S; i += DS_TILE_NT) atomicMax(&sGw[i % S], __ldg(p.gw + i));
    __syncthreads();
    if (tid == 0) {
        int base = 0;
        for (int sc = 0; sc < S; ++sc) {
            int n = 16;
            while (n < sGw[sc]) n <<= 1;
            if (n > NSTRIDE) n = NSTRIDE;
            sNs[sc] = n;
            sBase[sc] = base;
            const int jpt = 128 / n;
            base += B * ((J + jpt - 1) / jpt);
        }
        for (int sc = S; sc < 5; ++sc) sBase[sc] = base;
    }
    __syncthreads();
    const int total = sBase[S];
    const int it0 = (int)((long long)total * blockIdx.x / gridDim.x), it1 = (int)((long long)total * (blockIdx.x + 1) / gridDim.x);

    auto decode = [&](int item) {   // uses the run constants of the item's scale: set_run(scale_of(item)) first
        DesaItem it;
        it.sc = 0;
        while (it.sc + 1 < S && item >= sBase[it.sc + 1]) ++it.sc;
        const int rem = item - sBase[it.sc];
        it.b = rem / TPS;
        it.j0 = (rem - it.b * TPS) * JPT;
        return it;
    };
    auto set_run = [&](int item) {
        int sc = 0;
        while (sc + 1 < S && item >= sBase[sc + 1]) ++sc;
        NS = sNs[sc];
        JPT = 128 / NS;
        TPS = (J + JPT - 1) / JPT;
        ns_shift = 31 - __clz(NS);
    };
    auto advance = [&](DesaItem& it) {
        it.j0 += JPT;
        if (it.j0 >= J) {
            it.j0 = 0;
            if (++it.b == B) {
                it.b = 0;
                ++it.sc;
            }
        }
    };
    // ---- gather side (worker warps): the grouped rows of a tile are copied global -> shared by cp.async, 16 bytes per chunk,
    //      straight into the K-major operand (W1 (feat - jf) = W1 feat - W1 jf: the subtraction happens in the layer-1 epilogue,
    //      so no register staging, no conversion); every stage walks the items with its own cursor
    DesaItem c_idx, c_rows, c_epi, c_max;
    int ii[2] = {0, 0};      // ball-query indices of this thread's two rows for the item whose rows are copied next (< N + J)
    bool tail_ok[2] = {false, false};   // this thread's rows of the tile copied last belong to real joints
    float inv_r = 1.f;       // 1 / radius of the run's scale

    auto fetch_idx = [&]() {
        const uint16_t* base = p.idx + (((size_t)c_idx.b * S + c_idx.sc) * J + c_idx.j0) * NSTRIDE;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int row = r + 64 * h, jo = row >> ns_shift;   // the first NS of a joint's NSTRIDE indices
            ii[h] = c_idx.j0 + jo < J ? (int)__ldg(base + jo * NSTRIDE + (row & (NS - 1))) : 0;
        }
        advance(c_idx);
    };
    // One part of a tile's row copy: part = 4 h + k = 16-byte chunk group k of this thread's row r + 64 h (uses ii; the item cursor is
    // captured by part 0, the group is committed by part 7).  The eight parts are issued at eight points of an iteration, between the
    // pieces of the epilogues, NOT back to back: a burst of 6144 cp.async fills the SM's memory-instruction queue and every warp's
    // next shared-memory / TMEM / global instruction -- i.e. the epilogues -- queues up behind it.  Measured per launch, the kernel alone
    // over L2-resident rows (profiles/probe_kernels.py, same box): one burst 84.1 us, two halves 81, four parts 77.0, eight parts 74.8
    // (with the copy switched off: 57 us).  Inside the running step (four steps in flight, rows partly from DRAM) the gain is within
    // the run-to-run noise: 0.497 vs 0.501 ms per step, means of three alternating runs.
    DesaItem it_copy = {0, 0, 0};
    auto copy_one = [&](int item, int part) {
        if (part == 0) {
            it_copy = c_rows;
            advance(c_rows);
        }
        const int h = part >> 2, k = part & 3;
        const int row = r + 64 * h, jj = it_copy.j0 + (row >> ns_shift);
        const bool ok = jj < J;
        const uint16_t* src = p.e + (size_t)it_copy.b * p.e_bs + (size_t)ii[h] * 256 + 8 * g8;
        uint4* X = sX + (item % 3) * DS_XBUF + (row >> 3) * 128 + g8 * 8 + (row & 7);
        const uint32_t nbytes = ok ? 16u : 0u;
        // 16-byte chunk 8k + g8 of the 512-byte row [hi 128 | lo 128]: k-chunk (8k + g8) & 15 of plane k >> 1; the eight g8 lanes of a row
        // read 128 contiguous bytes = ONE request.  (.cg: the rows stream through L2 only -- measured 9 % faster than .ca, whose L1 is
        // ~30 KB next to 225 KB of shared memory.)  Rows beyond the last joint are zero filled (src-size 0).
        cp_async16_cg(X + (k >> 1) * 2048 + (k & 1) * 64, src + 64 * k, nbytes);
        if (k == 0 && g8 == 0) {   // xyz of the row's point and of its centre -> staging; the tail is built from it one iteration later
            const float4* tab = p.xyz4 + (size_t)it_copy.b * (N + 32);
            float4* st = sXyz + ((item & 1) * 128 + row) * 2;
            cp_async16(st, tab + ii[h]);
            cp_async16(st + 1, tab + N + (ok ? jj : 0));
            tail_ok[h] = ok;
        }
        if (part == 7) cp_async_commit();
    };
    auto store_tail = [&](int item) {   // group_xyz_norm = (xyz[idx] - centre) / radius   model.py:177
        if (g8 != 0) return;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int row = r + 64 * h;
            const float4* st = sXyz + ((item & 1) * 128 + row) * 2;
            const float4 a4 = st[0], c4 = st[1];
            float t8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (tail_ok[h]) {
                t8[0] = (a4.x - c4.x) * inv_r;
                t8[1] = (a4.y - c4.y) * inv_r;
                t8[2] = (a4.z - c4.z) * inv_r;
            }
            uint4* X = sX + (item % 3) * DS_XBUF + 4096 + (row >> 3) * 8 + (row & 7);
            uint4 th, tl;
            split8<FMT>(t8, th, tl);
            X[0] = th;
            X[128] = tl;
        }
    };
    // maxima of a finished tile: combine the column groups of each joint, store
    auto store_max = [&](int item) {
        const DesaItem it = c_max;
        advance(c_max);
        if (tid < JPT * 128) {
            const int g = tid >> 7, c = tid & 127, nc = NS / 32;
            const float* pp = sPart + (item & 1) * 512 + (g * nc) * 128 + c;
            float m = pp[0];
            for (int k = 1; k < nc; ++k) m = fmaxf(m, pp[k * 128]);
            if (it.j0 + g < J) p.desa_part[(((size_t)it.b * S + it.sc) * J + it.j0 + g) * 128 + c] = m;
        }
    };

    // ---- runs of items that share a scale (= weights)
    for (int i0 = it0; i0 < it1;) {
        set_run(i0);
        const DesaItem first = decode(i0);
        const int sc0 = first.sc;
        const int run_end = sBase[sc0 + 1];
        const bool direct = NS <= 32;   // a thread's 32 tile rows hold whole joints: it stores its maxima itself (no sPart, no store_max)
        const int i1 = it1 < run_end ? it1 : run_end;
        c_idx = c_rows = c_epi = c_max = first;
        // every MMA of the previous run has completed (its epilogues ran), so the weight buffers are free
        const uint4* ws = p.wmat + 4096 + (size_t)sc0 * DS_MAT_PER_SCALE;   // W1 main hi | lo, W1 tail hi | lo, W2 hi | lo
        if (issuer) {
            if (elect_one()) {
                mbar_expect_tx(&wbar, 512 * 16);
                tma_bulk_g2s(sW1t, ws + 4096, 512 * 16, &wbar);
            }
            __syncwarp();
        } else {
            // the scale's W1 main / W2 planes -> tensor memory (A operands): row ch = lane 32q + lane, 16-bit K elements packed two
            // per column; this thread moves k-chunks [4cg, 4cg + 4) (16 columns) of each of the four planes
#pragma unroll
            for (int pl = 0; pl < 4; ++pl) {
                const uint4* src = ws + (pl < 2 ? pl * 2048 : 4096 + 512 + (pl - 2) * 2048);
                uint4 v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = __ldg(src + (4 * cg + k) * 128 + ch);
                const uint32_t col = (pl == 0 ? TW1_HI : pl == 1 ? TW1_LO : pl == 2 ? TW2_HI : TW2_LO) + 16 * cg;
                tmem_st_nw<16>(tmem + col, reinterpret_cast<const float*>(v));
            }
            tmem_wait_st();
        }
        const float b1 = p.wvec[128 + 512 + sc0 * 256 + ch], b2 = p.wvec[128 + 512 + sc0 * 256 + 128 + ch];
        inv_r = 1.f / p.radius[sc0];
        bool w_ready = false;
        if (!issuer) fetch_idx();   // fill: indices of i0
        for (int s = i0 - 2; s < i1; ++s) {
            if (s >= i0 - 1) {
                cp_async_wait_group<0>();   // this thread's rows of tile s + 1 have landed
                if (!issuer && s + 1 < i1) store_tail(s + 1);          // ... and their xyz: the operand's K tail
                fence_proxy_async();
                tc_fence_before();
                __syncthreads();
                if (issuer) {
                    tc_fence_after();
                    if (!w_ready) mbar_wait(&wbar, w_phase);
                    if (elect_one()) {
                        // Layer 1 of tile s + 1 goes FIRST: its (long) epilogue then runs under layer 2 of tile s, whose (short) epilogue
                        // follows.  (Layer 2 first left the tensor pipe idle for the whole layer-1 epilogue of every tile; that order was
                        // forced by a single h buffer, which layer 2 of tile s had to release before the epilogue of tile s + 1 could write.)
                        if (s + 1 < i1) {   // layer 1 of tile s + 1: D1[c][row] = W1 [feat - jf | xyz]
                            const uint32_t X = smem_u32(sX + ((s + 1) % 3) * DS_XBUF);
                            const uint32_t id128 = umma_idesc_f16(128, 128, false, false, fmt, fmt);
                            TmemOp a;
                            a.hi = tmem0 + TW1_HI; a.lo = tmem0 + TW1_LO;
                            umma_gemm3_ts<128>(tmem0 + ACC1, a, smem_op_mn_outer(X, 128, 128), id128, false);
                            SmemOp tb = smem_op_k_outer(X + 4096 * 16, 128, 8);   // the tail's one stored k-chunk
                            tb.lbo = 0;   // k-chunk 1 (zero weights) re-reads chunk 0
                            umma_gemm3_ss<16>(tmem0 + ACC1, smem_op_k_outer(smem_u32(sW1t), 128, 16), tb, id128, true);
                            umma_commit(&g1_bar);
                        }
                        if (s >= i0) {   // layer 2 of tile s: D2[c][row] = W2 h
                            TmemOp a;
                            a.hi = tmem0 + TW2_HI; a.lo = tmem0 + TW2_LO;
                            const SmemOp hb = smem_op_k_outer(smem_u32(sX + (s % 3) * DS_XBUF), 128, 128);
                            umma_gemm3_ts<128>(tmem0 + ACC2, a, hb, umma_idesc_f16(128, 128, false, true, fmt, fmt), false);
                            umma_commit(&g2_bar);
                        }
                    }
                    __syncwarp();
                }
                w_ready = true;
                if (!direct && s - 1 >= i0) store_max(s - 1);   // written before the barrier above
            }
            if (!issuer) {
                // gather side: rows of tile s + 2 (its buffer held tile s - 1, whose layer 2 every thread waited for in the previous
                // iteration), indices of s + 3
                const bool fine = s + 2 < i1;   // tile s + 2 exists: its row copy is issued in eight parts across this iteration (copy_one)
                if (fine) copy_one(s + 2, 0);
                // layer-1 bias of tile s + 1 minus the W1 jf term of the joint this thread's 32 rows belong to
                float cjv[2] = {0.f, 0.f};   // per 16-row half (two joints when NS = 16); loaded here, consumed after the layer-2 epilogue
                if (s >= i0 - 1 && s + 1 < i1) {
                    const float* cjb = p.cj + (((size_t)c_epi.b * S + c_epi.sc) * J) * 128 + ch;
                    const int j0h = c_epi.j0 + ((32 * cg) >> ns_shift), j1h = c_epi.j0 + ((32 * cg + 16) >> ns_shift);
                    if (j0h < J) cjv[0] = __ldg(cjb + (size_t)j0h * 128);
                    cjv[1] = j1h == j0h ? cjv[0] : (j1h < J ? __ldg(cjb + (size_t)j1h * 128) : 0.f);
                    advance(c_epi);
                }
                if (fine) {
                    copy_one(s + 2, 1);
                    copy_one(s + 2, 2);
                }
                if (s >= i0 - 1 && s + 1 < i1) {   // layer-1 epilogue of tile s + 1: h[c][row] = relu(D1 + b1) -> MN-major B operand, in place
                    mbar_wait(&g1_bar, g1_phase);
                    g1_phase ^= 1;
                    tc_fence_after();
                    uint4* H = sX + ((s + 1) % 3) * DS_XBUF;   // layer 1 has consumed the rows that lived here
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {   // two 16-column reads: half the live registers of one 32-column read
                        float a[16];
                        tmem_ld<16>(tmem + ACC1 + 32 * cg + 16 * hf, a);
                        const float cjb = b1 - cjv[hf];
#pragma unroll
                        for (int i = 0; i < 16; ++i) a[i] = fmaxf(a[i] + cjb, 0.f);   // relu(W1 feat + tail - W1 jf + b1)
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            uint4 hh, hl;
                            split8<FMT>(a + 8 * c, hh, hl);
                            H[(ch >> 3) * 128 + (4 * cg + 2 * hf + c) * 8 + (ch & 7)] = hh;
                            H[2048 + (ch >> 3) * 128 + (4 * cg + 2 * hf + c) * 8 + (ch & 7)] = hl;
                        }
                        if (fine) copy_one(s + 2, 3 + hf);
                    }
                } else if (fine) {
                    copy_one(s + 2, 3);
                    copy_one(s + 2, 4);
                }
                if (s >= i0) {   // layer-2 epilogue of tile s: max over this thread's 32 grouped points  (model.py:197-198)
                    mbar_wait(&g2_bar, g2_phase);
                    g2_phase ^= 1;
                    tc_fence_after();
                    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        float a[16];
                        tmem_ld<16>(tmem + ACC2 + 32 * cg + 16 * hf, a);
#pragma unroll
                        for (int i = 0; i < 16; ++i) mx[hf] = fmaxf(mx[hf], a[i]);
                        if (fine) copy_one(s + 2, 5 + hf);
                    }
                    if (!direct) {
                        sPart[(s & 1) * 512 + cg * 128 + ch] = fmaxf(fmaxf(mx[0], mx[1]) + b2, 0.f);   // max_i relu(a_i + b2)
                    } else {   // narrow groups: this thread's rows are one joint (NS = 32) or two (NS = 16)
                        const DesaItem it = c_max;
                        advance(c_max);
                        float* dst = p.desa_part + (((size_t)it.b * S + it.sc) * J) * 128 + ch;
                        const int j0h = it.j0 + ((32 * cg) >> ns_shift), j1h = it.j0 + ((32 * cg + 16) >> ns_shift);
                        if (j0h == j1h) {
                            if (j0h < J) dst[(size_t)j0h * 128] = fmaxf(fmaxf(mx[0], mx[1]) + b2, 0.f);
                        } else {
                            if (j0h < J) dst[(size_t)j0h * 128] = fmaxf(mx[0] + b2, 0.f);
                            if (j1h < J) dst[(size_t)j1h * 128] = fmaxf(mx[1] + b2, 0.f);
                        }
                    }
                    tc_fence_before();
                } else if (fine) {
                    copy_one(s + 2, 5);
                    copy_one(s + 2, 6);
                }
                if (fine) copy_one(s + 2, 7);
                if (s + 3 < i1) fetch_idx();
            }
        }
        __syncthreads();
        if (!direct) store_max(i1 - 1);
        w_phase ^= 1;
        i0 = i1;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem0, 512);
}

}  // namespace kpf

extern "C" int kpf_desa_fused(void* e, long long e_batch_stride, const float* part_acc, const float* part_ms, const float* pcl, const float* joint,
                              const void* wmat, const float* wvec, int B, int N, int J, int S, int nsample, float r0, float r1, float r2,
                              float r3, int fmt, const float* jf_in, float* desa_part, float* jf_out, void* scratch, int num_sms,
                              cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && N >= 64 && N % 64 == 0 && N + J <= 65535 && J >= 1 && J <= 32 && S >= 1 && S <= 4);
    KPF_REQUIRE(nsample == 32 || nsample == 64 || nsample == 128);
    KPF_REQUIRE(fmt == FMT_F16 || fmt == FMT_BF16);
    KPF_REQUIRE(((uintptr_t)wmat % 16) == 0 && ((uintptr_t)e % 16) == 0 && ((uintptr_t)part_acc % 16) == 0 && ((uintptr_t)wvec % 16) == 0);
    if (B == 0) return 0;
    KPF_REQUIRE(scratch != nullptr && ((uintptr_t)scratch % 16) == 0 && num_sms >= 1);
    DesaParams p;
    KPF_REQUIRE(e_batch_stride >= (long long)(N + J) * 256 && e_batch_stride % 8 == 0);
    KPF_REQUIRE(jf_in != nullptr || (part_acc != nullptr && part_ms != nullptr));
    p.fmt = fmt; p.jf_in = jf_in;
    p.e = (uint16_t*)e; p.e_bs = e_batch_stride; p.part_acc = part_acc; p.part_ms = part_ms; p.pcl = pcl; p.joint = joint; p.wmat = (const uint4*)wmat;
    p.wvec = wvec; p.desa_part = desa_part; p.jf_out = jf_out; p.B = B; p.N = N; p.J = J; p.T = N / 64;   /* kpf_point_embed's tile = 64 points */ p.S = S; p.nsample = nsample;
    p.radius[0] = r0; p.radius[1] = r1; p.radius[2] = r2; p.radius[3] = r3;
    p.cj = (float*)scratch;
    p.xyz4 = (float4*)((char*)scratch + (size_t)B * S * J * 128 * 4);
    p.idx = (uint16_t*)((char*)scratch + (size_t)B * S * J * 128 * 4 + (size_t)B * (N + 32) * 16);
    p.gw = (int*)((char*)scratch + (size_t)B * S * J * 128 * 4 + (size_t)B * (N + 32) * 16 + (size_t)B * S * J * nsample * 2);
    const int NW = (N + J + 31) / 32;
    const size_t smem_jf = (size_t)(3 * 4096 + 1024) * 16 + (size_t)(p.T * 64 + 64) * 4 + 32 * 16 + 64;
    const size_t smem_bq = (size_t)((N + J + 3) / 4 * 4) * 16 + (size_t)S * J * NW * 4 + 64;
    const size_t smem_a = smem_jf > smem_bq ? smem_jf : smem_bq;
    const size_t smem_b = (size_t)(512 + 3 * DS_XBUF) * 16 + 2 * 512 * 4 + 2 * 128 * 2 * 16 + 64;
    KPF_REQUIRE(smem_a <= 227 * 1024 && smem_b <= 227 * 1024);
    auto prep = fmt == FMT_F16 ? desa_prep_kernel<FMT_F16> : desa_prep_kernel<FMT_BF16>;
    auto tile = fmt == FMT_F16 ? desa_tile_kernel<FMT_F16> : desa_tile_kernel<FMT_BF16>;
    cudaError_t err = kpf::set_smem(prep, smem_a);
    if (err != cudaSuccess) return (int)err;
    err = kpf::set_smem(tile, smem_b);
    if (err != cudaSuccess) return (int)err;
    err = kpf::launch_pdl(prep, dim3(2 * B), dim3(DS_NT), smem_a, stream, p);
    if (err != cudaSuccess) return (int)err;
    KPF_CHECK_LAUNCH();
    const int JPT = 128 / nsample, total = S * B * ((J + JPT - 1) / JPT);
    err = kpf::launch_pdl(tile, dim3(total < num_sms ? total : num_sms), dim3(DS_TILE_NT), smem_b, stream, p);
    if (err != cudaSuccess) return (int)err;
    KPF_CHECK_LAUNCH();
    return 0;
}
