// Keypoint-token transformer stacks on tcgen05 tensor cores, split precision (fp32 operands as two 16-bit planes, three MMAs
// per product, fp32 accumulation in TMEM: csrc/tcgen05.cuh) -- results are fp32-class, which the 0.05 mm joint bar needs.
//
//   encoder : KP_Interaction_TR.forward, model/model.py:45-126 (transformers 4.25.1 BertLayer x L):
//             h = pos_emb + x W_emb^T + b ; L x { self-attention, +res, LN, FFN(gelu), +res, LN } ; pred = cls_head(h) + residual(x)
//             optional prologue: x = relu(W_fu [desa_0 | desa_1 | desa_2 | jf] + b)   (DESA's fusion conv, model.py:160-164, :203)
//   cross   : the live TransformerDecoderLayer of updatedDecoder, model/transfusion_head.py:684-708 / :132-173:
//             Q from anchor + self_posembed, K = V from tokens + cross_posembed, +res(anchor), LN2, FFN(relu), +res, LN3
//   cross + encoder fused: crossTR followed by final_TR on cat([r3d, cross_out]) (model.py:347-349) without leaving the SM.
//
// One CTA = one sample (a latency chain of tiny GEMMs; samples spread over SMs).  Everything is computed TRANSPOSED:
//   D^T[feature][token] = W[feature][k] X[token][k]      weights = the M = 128 A operand, the sample's <= 32 tokens = N = 32,
// so a thread owns ONE feature (its TMEM lane) and 8 tokens (its column group), an activation operand is 8 KB per plane instead
// of the 32 KB a 128-row A operand costs, and an MMA is N = 32 wide.  16 worker warps = 4 lane quarters x 4 token groups.
//   * Attention for all four heads is two MMA groups.  Q^T and K^T come out with lane = 32h + d; they are stored as MN-major
//     operands [K = d][M or N = 32h + token], so ONE 128x128x32 group yields S_h in lanes/columns [32h, 32h+32) (the block
//     diagonal).  P_h goes to rows 32h + t of a K-major B operand, V^T stays in TENSOR MEMORY as the A operand (lane = 32h + d,
//     K = keys), and ONE 128x128x32 group yields O^T_h in the same diagonal blocks.
//   * FFN-1 (hidden 16 or 128) is the one GEMM computed token-major: A = the activation operand read as an MN-major A (rows
//     >= 32 alias other data and only feed unused accumulator lanes), B = W1; FFN-2 is transposed again.
//   * LayerNorm / the regression head reduce over features = over lanes: warp reduce-scatter by shuffles, then four partials
//     per token through shared memory, in a fixed order (deterministic, batch-invariant).
//   * Weights stream through a ring of four 32 KB slots (a 128x128 matrix with both planes = two half-K tiles) filled by a
//     dedicated producer warp with cp.async.bulk; tcgen05.commit on a slot's "empty" barrier hands it back.  Per-layer vectors
//     are double-buffered the same way.  The fp32 residual stream stays in registers.
#include "tcgen05.cuh"

namespace kpf {

constexpr int TS_C = 128;              // hidden size
constexpr int TS_WORKERS = 512;        // 16 worker warps
constexpr int TS_NT = TS_WORKERS + 32; // + the weight producer warp
constexpr int TS_RING = 4;
constexpr int TS_SLOT = 2048;          // uint4 per ring slot (32 KB)
constexpr int TS_MAXG = 64;            // ring entries per program
constexpr int TS_VEC = 10 * TS_C;      // floats of per-layer vectors
constexpr int TS_PLANE = 512;          // uint4 per activation operand plane (128 x 32 x 2 B)
// TMEM columns
constexpr uint32_t ACC_Q = 0, ACC_K = 32, ACC_V = 64, ACC_X = 96, ACC_F = 128, ACC_S = 256, ACC_O = 384;
constexpr uint32_t VT_HI = 128, VT_LO = 144;   // V^T operand planes (16 columns each) share ACC_F's columns: disjoint in time

struct TokParams {
    const float* x;        // encoder input [B,J,D] (no prologue) | cross: anchor [B,J,C]
    const float* y;        // cross: tokens [B,J,C]
    const float* r3d;      // cross+encoder: leading D-128 inputs of the encoder [B,J,D-128]
    const float* desa;     // prologue: [B,3,J,C]
    const float* jf;       // prologue: [B,J,C]
    const uint4* wmat;     // 16-bit canonical half-K tiles, (hi, lo) planes (ops.pack_token_program)
    const int4* wseq;      // per ring entry: (source offset, count) in uint4, layer whose vectors are loaded before it (-1: none)
    const float* wvec;     // fp32 vectors
    float* tokens_out;     // [B,J,C] or null (final hidden states)
    float* pred_out;       // [B,J,3] or null
    float* out_cj;         // cross only: [B,C,J] or null
    float* out_jc;         // cross only: element (b,t,c) at out_jc[(b*J+t)*stride + c0 + c] or null
    int out_jc_stride, out_jc_c0;
    int B, J, D, L, F, pre, cross, Fc, G, fmt;
    // fused exchange step (SURVEY.md 2b row C1): pred is ALSO stored straight into every rank's gathered-joints buffer over NVLink
    const unsigned long long* peer_bases;   // null, or [world] base addresses of the ranks' symmetric exchange buffers
    const int* xstep;                       // device step counter (its parity selects the half of the double-buffered result)
    int world, row0, rows_total;            // this rank's first row and the total rows of the gathered tensor
};

// Exchange buffer layout (identical on every rank; 64-byte header, then two [rows_total, J, 3] f32 halves):
//   u32 arrived : cumulative count of samples whose joints have landed here, from all ranks (system-scope release adds)
constexpr int XCHG_HEADER_FLOATS = 16;

// erf-GELU with Abramowitz-Stegun 7.1.26 (|erf error| <= 1.5e-7)
__device__ __forceinline__ float gelu_erf(float x) {
    const float z = fabsf(x) * 0.70710678118654752f;
    const float t = __fdividef(1.f, 1.f + 0.3275911f * z);
    const float poly = ((((1.061405429f * t - 1.453152027f) * t + 1.421413741f) * t - 0.284496736f) * t + 0.254829592f) * t;
    const float erf_abs = 1.f - poly * __expf(-z * z);
    return 0.5f * x * (1.f + copysignf(erf_abs, x));
}

// Sum v[0..NV) over the 32 lanes of a warp (NV a power of two <= 32) by recursive halving: NV - 1 + (5 - log2 NV) shuffles.
// On return v[0] of lane L holds the total of value index L >> (5 - log2 NV).
template <int NV>
__device__ __forceinline__ void warp_reduce_scatter(float* v, int lane) {
    int off = 16;
#pragma unroll
    for (int n = NV; n > 1; n >>= 1, off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
            const float send = upper ? v[i] : v[i + n / 2];
            const float recv = __shfl_xor_sync(0xffffffffu, send, off);
            v[i] = (upper ? v[i + n / 2] : v[i]) + recv;
        }
    }
#pragma unroll
    for (; off > 0; off >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
}

// FMT: the split format of the operand planes, a template parameter so that every split8 / instruction descriptor folds to one path
// (a run-time format doubled the conversion code of every epilogue; the kernel is instruction-fetch sensitive: `no_instruction`
// was 3 of 11 stall cycles per instruction, profiles/stalls_r2_a.txt)
template <int FMT>
__global__ void __launch_bounds__(TS_NT, 1) token_stack_kernel(const TokParams p) {
    extern __shared__ __align__(128) unsigned char ts_smem[];
    uint4* wslot = reinterpret_cast<uint4*>(ts_smem);   // [4][2048]    weight ring
    uint4* bufX = wslot + TS_RING * TS_SLOT;            // [2][512]     main activation operand: MN-major [K = 128 features][N = 32 tokens]
    uint4* bufY = bufX + 2 * TS_PLANE;                  // [2][512]     cross k_in / prologue source (same layout); FFN hidden, K-major [K/8][32]
    uint4* bufQ = bufY + 2 * TS_PLANE;                  // [2][512]     Q: MN-major A [K = 32 d][M = 32h + t]; then P: K-major B [4][128]
    uint4* bufK = bufQ + 2 * TS_PLANE;                  // [2][512]     K: MN-major B [K = 32 d][N = 32h + k]
    uint4* bufAt = bufK + 2 * TS_PLANE;                 // [2][64]      K-tail of the embedding input, K-major [2][32 tokens]
    float* sVec = reinterpret_cast<float*>(bufAt + 128);   // [2][10][128] per-layer vectors (double buffered)
    float* sRed = sVec + 2 * TS_VEC;                    // [2][4 c][4 q][16] LayerNorm partials (double buffered)
    float* sSum = sRed + 512;                           // [4 c][128]   softmax partial sums of (key group, row)
    float* sHead = sSum + 512;                          // [2][4 q][4 c][32] regression-head partials (x part, h part)
    float* sLead = sHead + 1024;                        // [32][4]      head share of the leading D-128 inputs
    __shared__ __align__(8) uint64_t full[TS_RING], empty[TS_RING], vec_full[2], vec_empty[2], bars[4];
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, q = w & 3, c = (w >> 2) & 3;
    const int f = 32 * q + lane;              // this thread's feature = TMEM lane
    const int J = p.J, C = TS_C, G = p.G;
    constexpr int fmt = FMT;
    const int b = blockIdx.x;
    const int warp_u = warp_index_uniform();
    const bool producer = warp_u == TS_WORKERS / 32;

    pdl_launch_dependents();
    if (warp_u == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 32) {
        for (int i = 0; i < TS_RING; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&vec_full[i], 1);
            mbar_init(&vec_empty[i], 1);
        }
        for (int i = 0; i < 4; ++i) mbar_init(&bars[i], 1);
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = tmem_slot;
    const uint32_t tmem = tmem0 + ((uint32_t)(32 * q) << 16);  // this thread's lane window

    // ---- layout of the fp32 vector blob (ops.pack_token_program)
    const int D = p.D, shift = p.L > 0 ? D - C : 0;
    const float* vp = p.wvec;
    const float *qpos = nullptr, *kpos = nullptr, *cross_vec = nullptr, *bfu = nullptr, *pos = nullptr, *bemb = nullptr,
                *Wres_lead = nullptr, *Wres_feat = nullptr, *bres = nullptr, *Wcls = nullptr, *bcls = nullptr, *enc_vec = nullptr;
    if (p.cross) {
        qpos = vp;
        kpos = qpos + J * C;
        cross_vec = kpos + J * C;
        vp = cross_vec + TS_VEC;
    }
    if (p.pre) {
        bfu = vp;
        vp += C;
    }
    if (p.L > 0) {
        pos = vp;                        // [J][128]
        bemb = pos + J * C;              // [128]
        Wres_lead = bemb + C;            // [3][16]  residual.weight columns of the leading D-128 inputs (zero padded)
        Wres_feat = Wres_lead + 48;      // [3][128] residual.weight columns of the 128 features
        bres = Wres_feat + 3 * C;        // [3] (+1 pad)
        Wcls = bres + 4;                 // [3][128]
        bcls = Wcls + 3 * C;             // [3] (+1 pad)
        enc_vec = bcls + 4;              // [L][10][128]
    }
    const int n_layers = (p.cross ? 1 : 0) + p.L;
    auto layer_vec = [&](int it) { return (p.cross && it == 0) ? cross_vec : enc_vec + (size_t)(it - (p.cross ? 1 : 0)) * TS_VEC; };

    // =========================== weight producer warp ===========================
    if (producer) {
        if (elect_one()) {
            for (int e = 0; e < G; ++e) {
                const int4 s = __ldg(p.wseq + e);
                if (s.z >= 0) {   // this layer's vectors (buffer s.z & 1; its previous user is layer s.z - 2)
                    const int it = s.z;
                    if (it >= 2) mbar_wait(&vec_empty[it & 1], ((it >> 1) - 1) & 1);
                    mbar_expect_tx(&vec_full[it & 1], TS_VEC * 4);
                    tma_bulk_g2s(sVec + (it & 1) * TS_VEC, layer_vec(it), TS_VEC * 4, &vec_full[it & 1]);
                }
                const int slot = e & (TS_RING - 1);
                if (e >= TS_RING) mbar_wait(&empty[slot], ((e >> 2) - 1) & 1);
                mbar_expect_tx(&full[slot], (uint32_t)s.y * 16);
                tma_bulk_g2s(wslot + slot * TS_SLOT, p.wmat + s.x, (uint32_t)s.y * 16, &full[slot]);
            }
        }
        __syncwarp();
        pdl_wait();   // a kernel launched with the PDL attribute must not finish before its predecessor has
        return;       // (the workers' only later __syncthreads-free path: they use named barrier 1 below)
    }

    // =========================== workers ===========================
    // all worker-only synchronisation goes through named barrier 1 (512 threads): the producer warp has left
    auto wsync = [&]() { named_bar_sync(1, 512); };
    uint32_t bar_phase[4] = {0, 0, 0, 0};
    auto wait_bar = [&](int i) {
        mbar_wait(&bars[i], bar_phase[i]);
        bar_phase[i] ^= 1;
        tc_fence_after();
    };
    // operand writes -> async proxy, everybody's TMEM accesses done, then the elected lane issues
    auto sync_for_mma = [&]() {
        fence_proxy_async();
        tc_fence_before();
        wsync();
    };
    int g = 0;   // ring entry cursor (same in every thread)
    auto slot_addr = [&](int e) { return smem_u32(wslot + (e & (TS_RING - 1)) * TS_SLOT); };
    auto wait_full = [&](int e) { mbar_wait(&full[e & (TS_RING - 1)], (e >> 2) & 1); };
    // --- issue helpers: call only from the elected lane of warp 0
    // D^T[acc][128 x 32] (+)= W (ring entries e, e+1: the two half-K tiles, A operand) x act (MN-major B operand, 2 planes)
    auto issue_proj = [&](uint32_t acc, const uint4* act, int e, bool accumulate) {
        const uint32_t id = umma_idesc_f16(128, 32, false, true, fmt, fmt);
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
            wait_full(e + h);
            tc_fence_after();
            const SmemOp a = smem_op_k_outer(slot_addr(e + h), 128, 64), bo = smem_op_k_outer(smem_u32(act) + h * 4096, 32, 128);
            umma_gemm3_ss<64>(tmem0 + acc, a, bo, id, accumulate || h > 0);
            umma_commit(&empty[(e + h) & (TS_RING - 1)]);
        }
    };
    const uint32_t xidx = (uint32_t)((f >> 3) * 32 + c * 8 + (f & 7));   // this thread's chunk of an MN-major [128][32] operand plane
    auto write_act = [&](uint4* buf, const float* v) {   // 8 tokens of feature f -> both planes
        uint4 hi, lo;
        split8<FMT>(v, hi, lo);
        buf[xidx] = hi;
        buf[TS_PLANE + xidx] = lo;
    };
    bool tokv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) tokv[i] = 8 * c + i < J;
    auto load_tok = [&](const float* base, int ld, float* v) {   // v[i] = base[(8c+i)*ld + f] (coalesced over the warp's features)
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = tokv[i] ? __ldg(base + (size_t)(8 * c + i) * ld + f) : 0.f;
    };
    // regression-head partial of 8 tokens x 3 outputs over this warp's 32 features -> sHead[part][q][c][0..24)
    auto head_partial = [&](int part, const float* v, const float* W) {
        float hx[32];
        const float w0 = __ldg(W + f), w1 = __ldg(W + C + f), w2 = __ldg(W + 2 * C + f);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            hx[3 * i] = v[i] * w0;
            hx[3 * i + 1] = v[i] * w1;
            hx[3 * i + 2] = v[i] * w2;
        }
#pragma unroll
        for (int i = 24; i < 32; ++i) hx[i] = 0.f;
        warp_reduce_scatter<32>(hx, lane);
        sHead[((part * 4 + q) * 4 + c) * 32 + lane] = hx[0];
    };

    if (tid < 128) sLead[tid] = 0.f;
    wsync();      // sLead is rewritten by warp 0 in the input stage
    pdl_wait();   // everything above touched only weights; the activations below come from the previous kernel
    float resid[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // fp32 residual stream: feature f of this thread's 8 tokens
    const float qscale = rsqrtf((float)(C / 4));  // head_dim^-0.5, 4 heads
    int red_par = 0;

    // =========================== cross-attention inputs (crossTR) ===========================
    if (p.cross) {
        float a[8], e[8];
        load_tok(p.x + (size_t)b * J * C, C, a);
        load_tok(qpos, C, e);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            resid[i] = a[i];     // residual = anchor (transfusion_head.py:164)
            e[i] += a[i];
        }
        write_act(bufX, e);      // q_in = anchor + self_posembed
        load_tok(p.y + (size_t)b * J * C, C, a);
        load_tok(kpos, C, e);
#pragma unroll
        for (int i = 0; i < 8; ++i) e[i] += a[i];
        write_act(bufY, e);      // k_in = tokens + cross_posembed
    }

    // ---- DESA fusion conv: x = relu(W_fu [desa_0 | desa_1 | desa_2 | jf] + b_fu): four accumulating K = 128 GEMMs (model.py:160-164)
    auto fusion_prologue = [&](float* a) {
        float v[8];
        const float* dsrc = p.desa + (size_t)b * 3 * J * C;
        load_tok(dsrc, C, v);
        write_act(bufX, v);
        load_tok(dsrc + (size_t)J * C, C, v);
        write_act(bufY, v);
        load_tok(dsrc + (size_t)2 * J * C, C, v);
        write_act(bufQ, v);
        load_tok(p.jf + (size_t)b * J * C, C, v);
        write_act(bufK, v);
        sync_for_mma();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                issue_proj(ACC_X, bufX, g, false);
                issue_proj(ACC_X, bufY, g + 2, true);
                issue_proj(ACC_X, bufQ, g + 4, true);
                issue_proj(ACC_X, bufK, g + 6, true);
                umma_commit(&bars[0]);
            }
            __syncwarp();
        }
        g += 8;
        const float bb = __ldg(bfu + f);
        wait_bar(0);
        tmem_ld<8>(tmem + ACC_X + 8 * c, a);
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = tokv[i] ? fmaxf(a[i] + bb, 0.f) : 0.f;
    };
    float pre_a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // the fusion conv's output (one instantiation of the prologue: code size)
    if (p.pre) {
        fusion_prologue(pre_a);
        if (p.L == 0 && p.tokens_out) {   // prologue-only program (stand-alone DESA.forward): the fusion conv's output is the result
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (tokv[i]) p.tokens_out[((size_t)b * J + 8 * c + i) * C + f] = pre_a[i];
        }
    }

    for (int it = 0; it < n_layers; ++it) {
        const bool is_cross = p.cross && it == 0;
        if (it == (p.cross ? 1 : 0) && p.L > 0) {
            // =========================== encoder input stage (KP_Interaction_TR) ===========================
            if (p.pre) {
                head_partial(0, pre_a, Wres_feat);
                write_act(bufX, pre_a);
            }
            if (!p.pre && !p.cross) {
                float v[8];
                load_tok(p.x + (size_t)b * J * D + shift, D, v);
                head_partial(0, v, Wres_feat);
                write_act(bufX, v);
            }
            if (p.cross) head_partial(0, resid, Wres_feat);   // fused crossTR -> final_TR: the features are the cross layer's output
            if (shift > 0 && w == 0) {  // leading (D - 128) inputs: joint coordinates (one thread per token)
                const int t = lane;
                const float* lead = p.cross ? p.r3d + ((size_t)b * J + t) * shift : p.x + ((size_t)b * J + t) * D;
                float tl[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) tl[i] = (t < J && i < shift) ? __ldg(lead + i) : 0.f;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    float s = 0.f;
#pragma unroll
                    for (int i = 0; i < 16; ++i) s += tl[i] * __ldg(Wres_lead + 16 * k + i);
                    sLead[4 * t + k] = s;
                }
                uint4 hi, lo;
                split8<FMT>(tl, hi, lo);
                bufAt[t] = hi;
                bufAt[64 + t] = lo;
                split8<FMT>(tl + 8, hi, lo);
                bufAt[32 + t] = hi;
                bufAt[96 + t] = lo;
            }
            // ---- embedding: h = pos_emb[tok] + x W_emb^T + b_emb      (model.py:56, :88-89)
            sync_for_mma();
            if (warp_u == 0) {
                tc_fence_after();
                if (elect_one()) {
                    issue_proj(ACC_X, bufX, g, false);
                    if (shift > 0) {   // K tail: A = W_emb[:, :shift] (zero padded to 16) [2 chunks][128 rows], B = bufAt K-major
                        wait_full(g + 2);
                        tc_fence_after();
                        const SmemOp a = smem_op_k_outer(slot_addr(g + 2), 128, 16), bo = smem_op_k_outer(smem_u32(bufAt), 32, 16);
                        umma_gemm3_ss<16>(tmem0 + ACC_X, a, bo, umma_idesc_f16(128, 32, false, false, fmt, fmt), true);
                        umma_commit(&empty[(g + 2) & (TS_RING - 1)]);
                    }
                    umma_commit(&bars[0]);
                }
                __syncwarp();
            }
            g += shift > 0 ? 3 : 2;
            float e[8];
            load_tok(pos, C, e);
            const float bb = __ldg(bemb + f);
            wait_bar(0);
            float a[8];
            tmem_ld<8>(tmem + ACC_X + 8 * c, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) resid[i] = a[i] = tokv[i] ? a[i] + bb + e[i] : 0.f;
            write_act(bufX, a);
        }

        const float* sv = sVec + (it & 1) * TS_VEC;
        const uint4* kv_src = is_cross ? bufY : bufX;     // operand the K / V projections read
        const int F = is_cross ? p.Fc : p.F;
        const int act = is_cross ? 0 : 1;                 // relu | erf-gelu
        const float eps = is_cross ? 1e-5f : 1e-12f;

        // ---- K and Q projections back to back (ring order K, Q, V, O: V's weights take the slots K frees, the earliest possible);
        //      V follows S
        sync_for_mma();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                if (it >= 1) mbar_arrive(&vec_empty[(it - 1) & 1]);   // everybody is past the previous layer's vector reads
                issue_proj(ACC_K, kv_src, g, false);
                umma_commit(&bars[1]);
                issue_proj(ACC_Q, bufX, g + 2, false);
                umma_commit(&bars[0]);
            }
            __syncwarp();
        }
        mbar_wait(&vec_full[it & 1], (it >> 1) & 1);       // this layer's vectors have landed
        const float bq = sv[f], bk = sv[C + f], bv = sv[2 * C + f], bo_ = sv[3 * C + f], g1 = sv[4 * C + f], be1 = sv[5 * C + f],
                    b2 = sv[7 * C + f], g2 = sv[8 * C + f], be2 = sv[9 * C + f];
        const float* b1 = sv + 6 * C;
        // chunk of the head-major attention operands: K index d = lane, row 32q + token
        const uint32_t qidx = (uint32_t)((lane >> 3) * 128 + (4 * q + c) * 8 + (lane & 7));
        wait_bar(1);
        {   // K^T -> MN-major B operand of S
            float a[8];
            tmem_ld<8>(tmem + ACC_K + 8 * c, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = tokv[i] ? a[i] + bk : 0.f;
            uint4 hi, lo;
            split8<FMT>(a, hi, lo);
            bufK[qidx] = hi;
            bufK[TS_PLANE + qidx] = lo;
        }
        wait_bar(0);
        {   // Q^T -> MN-major A operand of S
            float a[8];
            tmem_ld<8>(tmem + ACC_Q + 8 * c, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = tokv[i] ? (a[i] + bq) * qscale : 0.f;
            uint4 hi, lo;
            split8<FMT>(a, hi, lo);
            bufQ[qidx] = hi;
            bufQ[TS_PLANE + qidx] = lo;
        }
        // ---- S for all four heads: D[32h+t][32h'+k] = Q_h[t] . K_h'[k] (diagonal blocks h = h' are the scores); then V^T
        sync_for_mma();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                const SmemOp a = smem_op_k_outer(smem_u32(bufQ), 128, 32), bo = smem_op_k_outer(smem_u32(bufK), 128, 32);
                umma_gemm3_ss<32>(tmem0 + ACC_S, a, bo, umma_idesc_f16(128, 128, true, true, fmt, fmt), false);
                umma_commit(&bars[0]);
                issue_proj(ACC_V, kv_src, g + 4, false);
                umma_commit(&bars[1]);
            }
            __syncwarp();
        }
        wait_bar(0);
        {   // softmax of row t = lane of head q: every key group takes the row maximum over all keys and exponentiates its 8 keys;
            // P stays un-normalised, the partial sums meet when O is read out
            float sa[32], own[8];
            tmem_ld_nw<32>(tmem + ACC_S + 32 * q, sa);
            tmem_ld_nw<8>(tmem + ACC_S + 32 * q + 8 * c, own);
            tmem_wait_ld();
            float mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < 32; ++i) mx = fmaxf(mx, i < J ? sa[i] : -INFINITY);
            float psum = 0.f;
            const bool qv = lane < J;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                own[i] = (qv && tokv[i]) ? __expf(own[i] - mx) : 0.f;
                psum += own[i];
            }
            sSum[c * 128 + f] = psum;
            uint4 hi, lo;   // P: K-major B operand [N = 32h + t][K = 32 keys], over the (dead) Q
            split8<FMT>(own, hi, lo);
            bufQ[c * 128 + f] = hi;
            bufQ[TS_PLANE + c * 128 + f] = lo;
        }
        wait_bar(1);
        {   // V^T (lane = 32h + d, K = keys) -> A operand planes in tensor memory
            float a[8];
            tmem_ld<8>(tmem + ACC_V + 8 * c, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = tokv[i] ? a[i] + bv : 0.f;
            uint4 hi, lo;
            split8<FMT>(a, hi, lo);
            tmem_st_nw<4>(tmem + VT_HI + 4 * c, reinterpret_cast<const float*>(&hi));
            tmem_st_nw<4>(tmem + VT_LO + 4 * c, reinterpret_cast<const float*>(&lo));
            tmem_wait_st();
        }
        // ---- O^T for all four heads: D[32h+d][32h'+t] = sum_k V^T_h[d][k] P_h'[t][k]; columns [32h, 32h+32) of lane block h are head h
        sync_for_mma();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                TmemOp a;
                a.hi = tmem0 + VT_HI; a.lo = tmem0 + VT_LO;
                const SmemOp bo = smem_op_k_outer(smem_u32(bufQ), 128, 32);
                umma_gemm3_ts<32>(tmem0 + ACC_O, a, bo, umma_idesc_f16(128, 128, false, false, fmt, fmt), false);
                umma_commit(&bars[0]);
            }
            __syncwarp();
        }
        float inv[8];
        {   // 1 / row sums of this thread's 8 tokens (head q)
            float s8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float4 u0 = *reinterpret_cast<const float4*>(sSum + k * 128 + 32 * q + 8 * c);
                const float4 u1 = *reinterpret_cast<const float4*>(sSum + k * 128 + 32 * q + 8 * c + 4);
                s8[0] += u0.x; s8[1] += u0.y; s8[2] += u0.z; s8[3] += u0.w;
                s8[4] += u1.x; s8[5] += u1.y; s8[6] += u1.z; s8[7] += u1.w;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) inv[i] = tokv[i] ? 1.f / s8[i] : 0.f;
        }
        wait_bar(0);
        {   // O^T -> activation operand of the output projection
            float a[8];
            tmem_ld<8>(tmem + ACC_O + 32 * q + 8 * c, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] *= inv[i];
            write_act(bufX, a);
        }
        // ---- residual + LayerNorm over the features (= lanes) of each token
        auto resid_ln = [&](float bias, float gam, float bet) {
            float v[16];
            tmem_ld<8>(tmem + ACC_X + 8 * c, v);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                v[i] += bias + resid[i];
                resid[i] = v[i];
                v[8 + i] = v[i] * v[i];
            }
            warp_reduce_scatter<16>(v, lane);
            float* red = sRed + red_par * 256;
            red_par ^= 1;
            if ((lane & 1) == 0) red[(c * 4 + q) * 16 + (lane >> 1)] = v[0];
            wsync();
            float st[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) st[i] = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {   // same order in every thread: identical statistics everywhere
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    const float4 u = *reinterpret_cast<const float4*>(red + (c * 4 + k) * 16 + 4 * j4);
                    st[4 * j4] += u.x; st[4 * j4 + 1] += u.y; st[4 * j4 + 2] += u.z; st[4 * j4 + 3] += u.w;
                }
            }
            float y[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float mean = st[i] * (1.f / C);
                const float rstd = rsqrtf(fmaxf(st[8 + i] * (1.f / C) - mean * mean, 0.f) + eps);
                resid[i] = y[i] = tokv[i] ? (resid[i] - mean) * rstd * gam + bet : 0.f;
            }
            write_act(bufX, y);
        };
        sync_for_mma();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                issue_proj(ACC_X, bufX, g + 6, false);
                umma_commit(&bars[0]);
            }
            __syncwarp();
        }
        wait_bar(0);
        resid_ln(bo_, g1, be1);
        // ---- FFN-1, token-major: D[token][F] = X^T W1^T.  A = bufX read as an MN-major A operand (rows >= 32 alias other data
        //      and only produce unused accumulator lanes), B = W1 [N = F][K = 128] K-major
        const int nffn = F == 16 ? 1 : 4;   // ring entries of the FFN weights
        sync_for_mma();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                if (F == 16) {
                    wait_full(g + 8);
                    tc_fence_after();
                    const SmemOp a = smem_op_k_outer(smem_u32(bufX), 32, 128), bo = smem_op_k_outer(slot_addr(g + 8), 16, 128);
                    umma_gemm3_ss<128>(tmem0 + ACC_F, a, bo, umma_idesc_f16(128, 16, true, false, fmt, fmt), false);
                } else {
#pragma unroll 1
                    for (int h = 0; h < 2; ++h) {
                        wait_full(g + 8 + h);
                        tc_fence_after();
                        const SmemOp a = smem_op_k_outer(smem_u32(bufX) + h * 4096, 32, 128), bo = smem_op_k_outer(slot_addr(g + 8 + h), 128, 64);
                        umma_gemm3_ss<64>(tmem0 + ACC_F, a, bo, umma_idesc_f16(128, 128, true, false, fmt, fmt), h > 0);
                        umma_commit(&empty[(g + 8 + h) & (TS_RING - 1)]);
                    }
                }
                umma_commit(&bars[0]);
            }
            __syncwarp();
        }
        wait_bar(0);
        if (q == 0) {   // lanes 0..31 of the accumulator = tokens: the four quarter-0 warps take F/4 hidden units each
            const bool tv = lane < J;
            if (F == 16) {
                float a[4];
                tmem_ld<4>(tmem0 + ACC_F + 4 * c, a);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float u = a[i] + b1[4 * c + i];
                    a[i] = tv ? (act == 1 ? gelu_erf(u) : fmaxf(u, 0.f)) : 0.f;
                }
                uint2 hi, lo;
                split2<FMT>(a[0], a[1], hi.x, lo.x);
                split2<FMT>(a[2], a[3], hi.y, lo.y);
                // hidden operand: K-major B [N = 32 tokens][K = 16]: chunk (k >> 3) * 32 + token
                reinterpret_cast<uint2*>(bufY + (c >> 1) * 32 + lane)[c & 1] = hi;
                reinterpret_cast<uint2*>(bufY + TS_PLANE + (c >> 1) * 32 + lane)[c & 1] = lo;
            } else {
#pragma unroll 1
                for (int j4 = 0; j4 < 4; ++j4) {   // rolled: eight hidden units per trip (code size; this path runs once per program)
                    float a[8];
                    tmem_ld<8>(tmem0 + ACC_F + 32 * c + 8 * j4, a);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float u = a[i] + b1[32 * c + 8 * j4 + i];
                        a[i] = tv ? (act == 1 ? gelu_erf(u) : fmaxf(u, 0.f)) : 0.f;
                    }
                    uint4 hi, lo;
                    split8<FMT>(a, hi, lo);
                    bufY[(4 * c + j4) * 32 + lane] = hi;
                    bufY[TS_PLANE + (4 * c + j4) * 32 + lane] = lo;
                }
            }
        }
        // ---- FFN-2 (transposed again): D^T[feature][token] = W2 [128][F] x hidden [32 tokens][F]
        sync_for_mma();
        if (warp_u == 0) {
            tc_fence_after();
            if (elect_one()) {
                const uint32_t id = umma_idesc_f16(128, 32, false, false, fmt, fmt);
                if (F == 16) {
                    const SmemOp a = smem_op_k_outer(slot_addr(g + 8) + 512 * 16, 128, 16), bo = smem_op_k_outer(smem_u32(bufY), 32, 128);
                    umma_gemm3_ss<16>(tmem0 + ACC_X, a, bo, id, false);
                    umma_commit(&empty[(g + 8) & (TS_RING - 1)]);
                } else {
#pragma unroll 1
                    for (int h = 0; h < 2; ++h) {
                        wait_full(g + 10 + h);
                        tc_fence_after();
                        const SmemOp a = smem_op_k_outer(slot_addr(g + 10 + h), 128, 64), bo = smem_op_k_outer(smem_u32(bufY) + h * 4096, 32, 128);
                        umma_gemm3_ss<64>(tmem0 + ACC_X, a, bo, id, h > 0);
                        umma_commit(&empty[(g + 10 + h) & (TS_RING - 1)]);
                    }
                }
                umma_commit(&bars[0]);
            }
            __syncwarp();
        }
        wait_bar(0);
        resid_ln(b2, g2, be2);
        g += 8 + nffn;
    }

    if (p.cross && p.L == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int t = 8 * c + i;
            if (tokv[i]) {
                if (p.out_cj) p.out_cj[((size_t)b * C + f) * J + t] = resid[i];
                if (p.out_jc) p.out_jc[((size_t)b * J + t) * p.out_jc_stride + p.out_jc_c0 + f] = resid[i];
            }
        }
    }
    if (p.L > 0) {
        // ---- regression head: pred = cls_head(h) + residual(x)   (model.py:122-124), fp32
        head_partial(1, resid, Wcls);
        if (p.tokens_out) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (tokv[i]) p.tokens_out[((size_t)b * J + 8 * c + i) * C + f] = resid[i];
        }
        wsync();
        if (tid < 96 && p.pred_out) {
            const int t = tid / 3, k = tid - 3 * t, cc = t >> 3, i = t & 7;
            if (t < J) {
                float o = __ldg(bres + k) + __ldg(bcls + k) + sLead[4 * t + k];
#pragma unroll
                for (int part = 0; part < 2; ++part)
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) o += sHead[((part * 4 + qq) * 4 + cc) * 32 + 3 * i + k];
                p.pred_out[((size_t)b * J + t) * 3 + k] = o;
                if (p.peer_bases) {   // the exchange step: the same value into every rank's gathered tensor, peer stores over NVLink
                    const size_t off = XCHG_HEADER_FLOATS + ((size_t)(*p.xstep & 1) * p.rows_total + p.row0 + b) * J * 3 + (size_t)t * 3 + k;
                    for (int r = 0; r < p.world; ++r) reinterpret_cast<float*>(p.peer_bases[r])[off] = o;
                }
            }
        }
        if (p.peer_bases && tid < 96) {
            // Only the three warps that stored take part: each makes its peer stores visible system-wide, the three meet at a named
            // barrier, then lane r of warp 0 counts the sample as arrived on rank r -- the fences ordered the stores before the
            // barrier, so relaxed additions suffice and all ranks' counters are updated at once (eight serial release-reductions and a
            // 512-thread system fence cost 22 us per step at 8 GPUs: KPF_EXCHANGE=off vs peer, DESIGN.md section 7).
            __threadfence_system();
            named_bar_sync(2, 96);
            if (tid < p.world) asm volatile("red.relaxed.sys.global.add.u32 [%0], 1;" ::"l"(p.peer_bases[tid]) : "memory");
        }
    }
    tc_fence_before();
    wsync();
    if (warp_u == 0) tmem_dealloc(tmem0, 512);
}

constexpr size_t TS_SMEM = (size_t)(TS_RING * TS_SLOT + 8 * TS_PLANE + 128) * 16 + (size_t)(2 * TS_VEC + 512 + 512 + 1024 + 128) * 4;

}  // namespace kpf

// The receiving side of the fused exchange.  `inflight` (device flag) says whether a step's joints are still on their way:
//   mode 0 (begin a step): if a step is in flight, wait until all `per_step` samples of it have landed here and advance the step counter
//                          (so the wait for step s overlaps nothing but is issued at the START of step s+1, when the other ranks have
//                          long finished step s: no per-step rank skew on the critical path); then mark the new step in flight;
//   mode 1 (flush)       : complete the step in flight, if any (end of a run, or before a consumer reads the gathered tensor).
// One thread; the spin is clock-bounded like every wait in this library.
__global__ void exchange_wait_kernel(const unsigned int* arrived, int* xstep, unsigned int per_step, int* inflight, int mode) {
    if (*inflight) {
        const unsigned int expected = ((unsigned int)*xstep + 1u) * per_step;
        const long long t0 = clock64();
        while (true) {
            unsigned int v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(arrived) : "memory");
            if ((int)(v - expected) >= 0) break;
            if (clock64() - t0 > 8000000000ll) __trap();   // ~4 s: a rank that never arrives is a failed launch, not a hung GPU
        }
        *xstep = *xstep + 1;
    }
    *inflight = mode == 0 ? 1 : 0;
}

extern "C" int kpf_exchange_wait(const void* exchange_buffer, int* xstep, int samples_per_step, int* inflight, int mode, cudaStream_t stream) {
    KPF_REQUIRE(exchange_buffer != nullptr && xstep != nullptr && inflight != nullptr && samples_per_step >= 1 && (mode == 0 || mode == 1));
    exchange_wait_kernel<<<1, 1, 0, stream>>>((const unsigned int*)exchange_buffer, xstep, (unsigned int)samples_per_step, inflight, mode);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_token_stack(const float* x, const float* y, const float* r3d, const float* desa, const float* jf, const void* wmat,
                               const void* wseq, const float* wvec, int n_weights, int cross, int pre, int B, int J, int D, int L, int F,
                               int Fc, int fmt, float* tokens_out, float* pred_out, float* out_cj, float* out_jc, int out_jc_stride,
                               int out_jc_c0, const void* peer_bases, const int* xstep, int world, int row0, int rows_total,
                               cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && J >= 1 && J <= 32 && L >= 0 && (cross || pre || L > 0));
    KPF_REQUIRE(fmt == FMT_F16 || fmt == FMT_BF16);
    if (B == 0) return 0;   // an empty batch has no buffers to validate
    KPF_REQUIRE(L == 0 || F == 16 || F == 128);
    KPF_REQUIRE(!cross || (y != nullptr && (Fc == 16 || Fc == 128)));
    KPF_REQUIRE(L == 0 || D == TS_C || (D > TS_C && D <= TS_C + 16));
    KPF_REQUIRE(!pre || (desa != nullptr && jf != nullptr && !cross && (L == 0 || D == TS_C)));
    KPF_REQUIRE(!(cross && L > 0) || (r3d != nullptr && D > TS_C));
    KPF_REQUIRE(n_weights <= TS_MAXG);
    const int per_cross = 8 + (Fc == 16 ? 1 : 4), per_layer = 8 + (F == 16 ? 1 : 4);
    KPF_REQUIRE(n_weights == (cross ? per_cross : 0) + (pre ? 8 : 0) + (L > 0 ? 2 + (D > TS_C ? 1 : 0) + per_layer * L : 0));
    KPF_REQUIRE(((uintptr_t)wmat % 16) == 0 && ((uintptr_t)wseq % 16) == 0);
    TokParams p;
    p.x = x; p.y = y; p.r3d = r3d; p.desa = desa; p.jf = jf; p.wmat = (const uint4*)wmat; p.wseq = (const int4*)wseq; p.wvec = wvec;
    p.tokens_out = tokens_out; p.pred_out = pred_out; p.out_cj = out_cj; p.out_jc = out_jc; p.out_jc_stride = out_jc_stride;
    p.out_jc_c0 = out_jc_c0; p.B = B; p.J = J; p.D = D; p.L = L; p.F = F; p.pre = pre; p.cross = cross; p.Fc = Fc; p.G = n_weights; p.fmt = fmt;
    KPF_REQUIRE(peer_bases == nullptr || (xstep != nullptr && world >= 1 && row0 >= 0 && row0 + B <= rows_total && L > 0));
    p.peer_bases = (const unsigned long long*)peer_bases; p.xstep = xstep; p.world = world; p.row0 = row0; p.rows_total = rows_total;
    auto kern = fmt == FMT_F16 ? token_stack_kernel<FMT_F16> : token_stack_kernel<FMT_BF16>;
    cudaError_t e = kpf::set_smem(kern, TS_SMEM);
    if (e != cudaSuccess) return (int)e;
    e = kpf::launch_pdl(kern, dim3(B), dim3(TS_NT), TS_SMEM, stream, p);
    if (e != cudaSuccess) return (int)e;
    KPF_CHECK_LAUNCH();
    return 0;
}
