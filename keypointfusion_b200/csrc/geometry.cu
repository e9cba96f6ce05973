// Geometry + per-joint feature kernels (SURVEY.md 8a rows a4-a7, a10, a11, a16; kernels K2, K4a-d).
// All are HBM / ALU bound CUDA-core kernels: coalesced loads, shared-memory staging of the per-sample
// cell cloud, warp-shuffle reductions.  Index-producing arithmetic follows the oracle's fp32 operation
// order without FMA contraction (common.cuh x* helpers) so indices are bit-exact.
#include "common.cuh"

namespace kpf {

// ------------------------------------------------------------------------------------------------
// a5: uvd_nl2xyznl_tensor / xyz_nl2uvdnl_tensor   dataloader/loader.py:775-789, :821-841
// ------------------------------------------------------------------------------------------------
__global__ void uvd2xyz_kernel(const float* __restrict__ uvd, const float* __restrict__ center, const float* __restrict__ M,
                               const float* __restrict__ cube, const float* __restrict__ cam, int P, float img_size, float flip,
                               float* __restrict__ out) {
    const int b = blockIdx.y;
    __shared__ CamF c;
    if (threadIdx.x == 0) load_cam(c, b, center, M, cube, cam, img_size, flip);
    __syncthreads();
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
        const float* s = uvd + ((size_t)b * P + p) * 3;
        const float3 o = uvd2xyz(c, s[0], s[1], s[2]);
        float* d = out + ((size_t)b * P + p) * 3;
        d[0] = o.x;
        d[1] = o.y;
        d[2] = o.z;
    }
}

// The points3DToImg half of xyz_nl2uvdnl_tensor: normalised xyz s -> camera-space point (X, Y, Z) in mm (loader.py:828) and its
// frame pixel (pu, pv) (loader.py:277-288).  Shared by xyz2uvd_kernel (which goes on into the crop) and joints_to_frame_kernel.
struct FramePoint {
    float X, Y, Z, pu, pv;
};

__device__ __forceinline__ FramePoint xyznl_to_frame(const float* s, float cx, float cy, float cz, float sx, float sy, float sz, float fx,
                                                     float fy, float fu, float fv, float flip) {
    FramePoint q;
    q.X = xadd(xdiv(xmul(s[0], sx), 2.0f), cx);  // loader.py:828
    q.Y = xadd(xdiv(xmul(s[1], sy), 2.0f), cy);
    q.Z = xadd(xdiv(xmul(s[2], sz), 2.0f), cz);
    q.pu = xadd(xdiv(xmul(q.X, fx), xadd(q.Z, 1e-8f)), fu);  // loader.py:281-283
    q.pv = xadd(xdiv(xmul(xmul(flip, q.Y), fy), q.Z), fv);   // loader.py:284-286
    return q;
}

__global__ void xyz2uvd_kernel(const float* __restrict__ xyz, const float* __restrict__ center, const float* __restrict__ M,
                               const float* __restrict__ cube, const float* __restrict__ cam, int P, float img_size, float flip,
                               float* __restrict__ out) {
    const int b = blockIdx.y;
    const float* m = M + 9 * b;
    const float cx = center[3 * b], cy = center[3 * b + 1], cz = center[3 * b + 2];
    const float sx = cube[3 * b], sy = cube[3 * b + 1], sz = cube[3 * b + 2];
    const float fx = cam[4 * b], fy = cam[4 * b + 1], fu = cam[4 * b + 2], fv = cam[4 * b + 3];
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
        const FramePoint q = xyznl_to_frame(xyz + ((size_t)b * P + p) * 3, cx, cy, cz, sx, sy, sz, fx, fy, fu, fv, flip);
        const float tu = xadd(xadd(xmul(m[0], q.pu), xmul(m[1], q.pv)), m[2]);
        const float tv = xadd(xadd(xmul(m[3], q.pu), xmul(m[4], q.pv)), m[5]);
        float* d = out + ((size_t)b * P + p) * 3;
        d[0] = xsub(xmul(xdiv(tu, img_size), 2.0f), 1.0f);  // loader.py:831
        d[1] = xsub(xmul(xdiv(tv, img_size), 2.0f), 1.0f);
        d[2] = xdiv(xsub(q.Z, cz), xdiv(sz, 2.0f));         // loader.py:832
    }
}

// Joints back into the frame they were cropped from: uvd_frame (frame pixels u, v and depth in mm) and xyz_cam (camera mm).
// One thread per joint over the flat [B*P] range (P is a hand's 21 joints: a per-sample grid row would idle most of its threads).
__global__ void joints_to_frame_kernel(const float* __restrict__ joints, const float* __restrict__ center, const float* __restrict__ cube,
                                       const float* __restrict__ cam, int B, int P, float flip, float* __restrict__ uvd_frame,
                                       float* __restrict__ xyz_cam) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)B * P) return;
    const int b = (int)(i / P);
    const FramePoint q = xyznl_to_frame(joints + i * 3, center[3 * b], center[3 * b + 1], center[3 * b + 2], cube[3 * b], cube[3 * b + 1],
                                        cube[3 * b + 2], cam[4 * b], cam[4 * b + 1], cam[4 * b + 2], cam[4 * b + 3], flip);
    float* u = uvd_frame + i * 3;
    u[0] = q.pu;
    u[1] = q.pv;
    u[2] = q.Z;
    float* x = xyz_cam + i * 3;
    x[0] = q.X;
    x[1] = q.Y;
    x[2] = q.Z;
}

// ------------------------------------------------------------------------------------------------
// Spatial processing order of a sample's points: the permutation that sorts them by the feature-map cell they project to
// (row-major cell index, point id as tie break -> deterministic).  Not part of the reference; kpf_img2pcl_index and
// kpf_point_embed use it to make neighbouring threads / tiles touch neighbouring cells.  One CTA per sample, bitonic sort of
// (cell << 13 | id) keys in shared memory.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
spatial_order_kernel(const float* __restrict__ pcl, const float* __restrict__ center, const float* __restrict__ M,
                     const float* __restrict__ cube, const float* __restrict__ cam, int N, int npow2, int fs, float img_size, float flip,
                     int32_t* __restrict__ order) {
    extern __shared__ uint32_t so_keys[];
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* m9 = M + 9 * b;
    const float cx = center[3 * b], cy = center[3 * b + 1], cz = center[3 * b + 2];
    const float hx = cube[3 * b] * 0.5f, hy = cube[3 * b + 1] * 0.5f, hz = cube[3 * b + 2] * 0.5f;
    const float fx = cam[4 * b], fy = cam[4 * b + 1], fu = cam[4 * b + 2], fv = cam[4 * b + 3];
    const float sc = (float)fs / img_size;
    for (int i = tid; i < npow2; i += blockDim.x) {
        uint32_t key = 0xFFFFFFFFu;
        if (i < N) {
            const float* s = pcl + ((size_t)b * N + i) * 3;
            const float X = s[0] * hx + cx, Y = s[1] * hy + cy, Z = s[2] * hz + cz;   // loader.py:828
            const float pu = X * fx / (Z + 1e-8f) + fu, pv = flip * Y * fy / Z + fv;  // loader.py:281-286
            const float tu = m9[0] * pu + m9[1] * pv + m9[2], tv = m9[3] * pu + m9[4] * pv + m9[5];
            int cp = (int)(tu * sc), rp = (int)(tv * sc);
            cp = min(max(cp, 0), fs - 1);
            rp = min(max(rp, 0), fs - 1);
            key = ((uint32_t)(rp * fs + cp) << 13) | (uint32_t)i;
        }
        so_keys[i] = key;
    }
    __syncthreads();
    if (npow2 <= (int)blockDim.x) {
        // one key per thread in a register: exchanges inside a warp (j < 32) are shuffles, only the 15 wider ones go through
        // shared memory (keys are unique, so min / max on both sides of an exchange is a consistent compare-swap)
        uint32_t key = tid < npow2 ? so_keys[tid] : 0xFFFFFFFFu;
        for (int k = 2; k <= npow2; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                uint32_t other;
                if (j >= 32) {
                    __syncthreads();
                    if (tid < npow2) so_keys[tid] = key;
                    __syncthreads();
                    other = tid < npow2 ? so_keys[tid ^ j] : key;
                } else {
                    other = __shfl_xor_sync(0xffffffffu, key, j);
                }
                const bool keep_min = ((tid & j) == 0) == ((tid & k) == 0);
                key = keep_min ? min(key, other) : max(key, other);
            }
        }
        if (tid < N) order[(size_t)b * N + tid] = (int32_t)(key & 0x1FFFu);
        return;
    }
    for (int k = 2; k <= npow2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < npow2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint32_t a = so_keys[i], c = so_keys[ixj];
                    if ((a > c) == ((i & k) == 0)) {
                        so_keys[i] = c;
                        so_keys[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
    for (int i = tid; i < N; i += blockDim.x) order[(size_t)b * N + i] = (int32_t)(so_keys[i] & 0x1FFFu);
}

// ------------------------------------------------------------------------------------------------
// K2 / a6: img2pcl_index   dataloader/loader.py:936-967
//   cell cloud of the sample (H*W x float4) lives in shared memory; one thread per point keeps a sorted
//   top-K in registers; ties -> lower cell index (lexicographic (d2, index) order, = the reference's stable ascending scan).
// ------------------------------------------------------------------------------------------------
//   K2_RQ warps share a group of 32 points: warp (group, rq) seeds its list from the point's window and scans the cell rows rq,
//   rq + K2_RQ, ... only; the lists (each the exact top K of the window plus its rows) meet through shared memory and warp rq = 0 merges them
//   (same lexicographic order, duplicates from the shared window dropped by index) -- bit-identical results.  The point of it: 65 k
//   points are 2048 warps, 14 per SM at batch 64, far too few to hide the dependent non-contracted arithmetic; a quarter of the rows
//   per warp gives four times the warps.  Measured: TWO warps per group (K2_RQ = 2, 512 threads = 256 points per CTA) is the optimum,
//   43.4 -> 36.7 us; four lose to their redundant window seeding and the merge (see the launcher).
template <int K, int K2_RQ, int K2_NT>
__global__ void __launch_bounds__(K2_NT)
nearest_cells_kernel(const float* __restrict__ pcl, const float* __restrict__ depth, long long depth_bs, int depth_rs,
                     int depth_cs, const float* __restrict__ center, const float* __restrict__ M,
                     const float* __restrict__ cube, const float* __restrict__ cam, int N, int fs, float img_size, float flip,
                     const int32_t* __restrict__ order, float* __restrict__ closeness, long long* __restrict__ index64,
                     int32_t* __restrict__ index32) {
    extern __shared__ __align__(16) float4 cells[];      // [HW] cell xyz, then [fs][2] per-row bounding boxes (min, max)
    __shared__ CamF c;
    const int b = blockIdx.y, HW = fs * fs;
    float4* rowbox = cells + HW;
    float* mrg_d = reinterpret_cast<float*>(rowbox + 2 * fs);                 // [groups][K2_RQ - 1][K][32] merge lists: distances ...
    int* mrg_i = reinterpret_cast<int*>(mrg_d + (K2_NT / 32 / K2_RQ) * (K2_RQ - 1) * K * 32);   // ... and cell indices
    if (threadIdx.x == 0) load_cam(c, b, center, M, cube, cam, img_size, flip);
    __syncthreads();
    const float ffs = (float)fs;
    for (int m = threadIdx.x; m < HW; m += blockDim.x) {
        const int r = m / fs, col = m - r * fs;
        const float d = __ldg(depth + (size_t)b * depth_bs + (size_t)r * depth_rs + (size_t)col * depth_cs);
        const float3 q = uvd2xyz(c, cell_coord(col, ffs), cell_coord(r, ffs), d);  // ch0 = column, ch1 = row (:948-951)
        cells[m] = make_float4(q.x, q.y, q.z, 0.f);
    }
    __syncthreads();
    // bounding box of every cell row (one warp per row): whole rows are skipped below when no lane of a warp can improve on it
    {
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
        for (int r = w; r < fs; r += nw) {
            float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
            for (int col = lane; col < fs; col += 32) {
                const float4 q = cells[r * fs + col];
                lo[0] = fminf(lo[0], q.x);
                hi[0] = fmaxf(hi[0], q.x);
                lo[1] = fminf(lo[1], q.y);
                hi[1] = fmaxf(hi[1], q.y);
                lo[2] = fminf(lo[2], q.z);
                hi[2] = fmaxf(hi[2], q.z);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
                    hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
                }
            }
            if (lane == 0) {
                rowbox[2 * r] = make_float4(lo[0], lo[1], lo[2], 0.f);
                rowbox[2 * r + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
            }
        }
    }
    __syncthreads();
    constexpr int K2_PTS = K2_NT / K2_RQ;
    const int lane_ = threadIdx.x & 31, warp_ = threadIdx.x >> 5, pgrp = warp_ / K2_RQ, rq = warp_ % K2_RQ;
    const int slot = blockIdx.x * K2_PTS + pgrp * 32 + lane_;
    const bool active = slot < N;   // inactive lanes stay in the loop (warp votes below) but never store
    // optional processing order (kpf_spatial_order): neighbouring threads then hold neighbouring points, so a warp's lanes prune
    // the same rows and take the insertion path at the same cells; the outputs are indexed by the point id either way
    const int n = !active ? 0 : (order ? order[(size_t)b * N + slot] : slot);
    const float* pp = pcl + ((size_t)b * N + n) * 3;
    const float px = pp[0], py = pp[1], pz = pp[2];
    float bd[K];
    int bi[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        bd[k] = INFINITY;
        bi[k] = 0;
    }
    // The result is the K smallest (d2, cell index) pairs in lexicographic order -- exactly what the reference's stable
    // ascending scan with a strict '<' yields -- so cells may be visited in any order.  Seed the list from a 3 x 8 window of
    // cells around the point's own (approximately projected) cell: the K-th best distance is then already tight and the full
    // scan below almost never takes the (divergent, ~25-instruction) insertion path.
    auto insert = [&](float d2, int m) {
        float cd = d2;
        int ci = m;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (cd < bd[k] || (cd == bd[k] && ci < bi[k])) {
                const float td = bd[k];
                const int ti = bi[k];
                bd[k] = cd;
                bi[k] = ci;
                cd = td;
                ci = ti;
            }
        }
    };
    auto dist2 = [&](const float4 q) {
        const float dx = xsub(px, q.x), dy = xsub(py, q.y), dz = xsub(pz, q.z);
        return xadd(xadd(xmul(dx, dx), xmul(dy, dy)), xmul(dz, dz));  // loader.py:956
    };
    const bool windowed = (fs & 3) == 0 && fs >= 8;
    int wr0 = -64, wc0 = -64;   // window origin (rows wr0..wr0+2, columns wc0..wc0+7); far away = no window
    if (windowed) {
        // fast-math projection of the point into the crop (loader.py:281-286, :828-831); only seeds the window
        const float* m9 = M + 9 * b;
        const float X = px * c.hx + c.cx, Y = py * c.hy + c.cy, Z = pz * c.hz + c.cz;
        const float pu = X * c.fx / (Z + 1e-8f) + c.fu, pv = c.flip * Y * c.fy / Z + c.fv;
        const float tu = m9[0] * pu + m9[1] * pv + m9[2], tv = m9[3] * pu + m9[4] * pv + m9[5];
        const float sc = ffs / img_size;
        int cp = (int)(tu * sc), rp = (int)(tv * sc);   // NaN / out of range -> clamped: any window is valid
        cp = min(max(cp, 0), fs - 1);
        rp = min(max(rp, 0), fs - 1);
        wr0 = min(max(rp - 1, 0), fs - 3);
        wc0 = min(max((((cp + 2) >> 2) << 2) - 4, 0), fs - 8);   // multiple of 4: a 4-cell group is inside or outside as a whole
        for (int rr = 0; rr < 3; ++rr) {
            const int m0 = (wr0 + rr) * fs + wc0;
#pragma unroll
            for (int cc = 0; cc < 8; ++cc) insert(dist2(cells[m0 + cc]), m0 + cc);
        }
    }
    // full scan, four cells per iteration: the distance arithmetic of a group is branch-free.  A cell row is skipped when, for
    // every lane of the warp, the distance from its point to the row's bounding box already exceeds its K-th best (with a 1e-4
    // relative margin, far above fp32 rounding, so no candidate -- not even an exact tie -- is ever lost).
    int m = 0;
    if (windowed) {
        for (int row = rq; row < fs; row += K2_RQ) {
            const float4 lo = rowbox[2 * row], hi = rowbox[2 * row + 1];
            const float ex = fmaxf(fmaxf(lo.x - px, px - hi.x), 0.f), ey = fmaxf(fmaxf(lo.y - py, py - hi.y), 0.f),
                        ez = fmaxf(fmaxf(lo.z - pz, pz - hi.z), 0.f);
            const float lb = ex * ex + ey * ey + ez * ez;
            const bool skip = !active || lb > bd[K - 1] * 1.0001f;
            if (__all_sync(0xffffffffu, skip)) continue;
            const bool in_rows = (unsigned)(row - wr0) < 3u;
            for (int col = 0; col < fs; col += 4) {
                const int mm = row * fs + col;
                float d2[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) d2[u] = dist2(cells[mm + u]);
                const float mn = fminf(fminf(d2[0], d2[1]), fminf(d2[2], d2[3]));
                const bool inwin = in_rows && (unsigned)(col - wc0) < 8u;   // already inserted
                if (!inwin && mn <= bd[K - 1]) {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (d2[u] <= bd[K - 1]) insert(d2[u], mm + u);
                }
            }
        }
        m = HW;
    }
    for (m += rq; m < HW; m += K2_RQ) {   // map sizes without the windowed fast path: every K2_RQ-th cell
        const float d2 = dist2(cells[m]);
        if (d2 <= bd[K - 1]) insert(d2, m);
    }
    // ---- merge the four row-quarter lists of a point group (warps rq = 1..3 publish, warp rq = 0 inserts)
    if (rq > 0) {
        float* md = mrg_d + ((pgrp * (K2_RQ - 1) + rq - 1) * K) * 32 + lane_;
        int* mi = mrg_i + ((pgrp * (K2_RQ - 1) + rq - 1) * K) * 32 + lane_;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            md[k * 32] = bd[k];
            mi[k * 32] = bi[k];
        }
    }
    __syncthreads();
    if (rq > 0 || !active) return;
    for (int o = 0; o < K2_RQ - 1; ++o) {
        const float* md = mrg_d + ((pgrp * (K2_RQ - 1) + o) * K) * 32 + lane_;
        const int* mi = mrg_i + ((pgrp * (K2_RQ - 1) + o) * K) * 32 + lane_;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float cd = md[k * 32];
            const int ci = mi[k * 32];
            if (!(cd <= bd[K - 1])) continue;   // cannot enter (also skips the +inf fillers of a short list)
            bool dup = false;                    // a window cell is in every list: the same cell never enters twice
#pragma unroll
            for (int kk = 0; kk < K; ++kk) dup |= bi[kk] == ci && bd[kk] == cd;
            if (!dup) insert(cd, ci);
        }
    }
    float cv[K];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        cv[k] = xdiv(1.0f, xadd(bd[k], 1e-8f));  // loader.py:959
        s = k == 0 ? cv[0] : xadd(s, cv[k]);
    }
    const float den = xadd(s, 1e-8f);  // loader.py:960
    const size_t o = ((size_t)b * N + n) * K;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        closeness[o + k] = xdiv(cv[k], den);
        if (index64) index64[o + k] = bi[k];
        if (index32) index32[o + k] = bi[k];
    }
}

// ------------------------------------------------------------------------------------------------
// K4a / a4: offset2joint_weight   model/model.py:466-500 == util/generateFeature.py:166-195
//   one CTA per (joint, sample); two passes over the 5 channel rows (max, then softmax-weighted sums).
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
offset2joint_kernel(const T* __restrict__ offset, const float* __restrict__ depth, int S, int J, int fs,
                    const float* __restrict__ kernel_vec, float* __restrict__ joint_out) {
    __shared__ float scratch[32];
    const int j = blockIdx.x, b = blockIdx.y, HW = fs * fs;
    const T* base = offset + (size_t)b * 5 * J * HW;
    const T* ux = base + (size_t)(3 * j) * HW;
    const T* heat = base + (size_t)(3 * J + j) * HW;
    const T* wgt = base + (size_t)(4 * J + j) * HW;
    const float* dimg = depth + (size_t)b * S * S;
    const float ks = kernel_vec[j];
    const float ffs = (float)fs;
    float mx = -INFINITY;
    for (int m = threadIdx.x; m < HW; m += blockDim.x) {
        const int r = m / fs, col = m - r * fs;
        const float d = __ldg(dimg + (size_t)nearest_src(r, S, fs) * S + nearest_src(col, S, fs));
        const float w = d > 0.99f ? -1e8f : to_f32(wgt[m]);  // masked_fill(depth.gt(0.99), -1e8)  :488
        mx = fmaxf(mx, w);
    }
    mx = block_max(mx, scratch);
    float se = 0.f, ax = 0.f, ay = 0.f, az = 0.f;
    for (int m = threadIdx.x; m < HW; m += blockDim.x) {
        const int r = m / fs, col = m - r * fs;
        const float d = __ldg(dimg + (size_t)nearest_src(r, S, fs) * S + nearest_src(col, S, fs));
        const float w = d > 0.99f ? -1e8f : to_f32(wgt[m]);
        const float e = expf(w - mx);
        const float msk = d < 0.99f ? 1.f : 0.f;                       // depth.lt(0.99)  :485
        const float dist = ks - (to_f32(heat[m]) * msk) * ks;         // :495
        const float ox = to_f32(ux[m]) * msk, oy = to_f32(ux[HW + m]) * msk, oz = to_f32(ux[2 * HW + m]) * msk;
        se += e;
        ax += (ox * dist + cell_coord(col, ffs)) * e;                 // coords ch0 = column  :481
        ay += (oy * dist + cell_coord(r, ffs)) * e;
        az += (oz * dist + d) * e;
    }
    se = block_sum(se, scratch);
    ax = block_sum(ax, scratch);
    ay = block_sum(ay, scratch);
    az = block_sum(az, scratch);
    if (threadIdx.x == 0) {
        float* o = joint_out + ((size_t)b * J + j) * 3;
        o[0] = ax / se;
        o[1] = ay / se;
        o[2] = az / se;
    }
}

// bf16 fast path of K4a for maps with HW == 8 * blockDim.x cells and fs % 8 == 0.  A CTA takes K4A_JPC joints of one sample; a thread
// owns 8 consecutive cells of a row and reads each channel row of a joint with ONE 16-byte load.  The kernel is a stream over
// 10 KB per joint, so what matters is how many loads are in flight and how few block-wide round trips interrupt them:
//   phase A  the depth of the 8 cells (once per CTA, not per joint) and the weight rows of ALL the CTA's joints -> masked weights in
//            registers, the joints' maxima with one reduction round;
//   phase B  per joint the four remaining rows, the NEXT joint's loads issued before the current joint's arithmetic;
//   phase C  one reduction round for all 4 * K4A_JPC sums.
// Two barriers per CTA instead of two per joint.  Same arithmetic per cell as the generic kernel above.
template <int K4A_JPC, int MINB>
__global__ void __launch_bounds__(128, MINB)
offset2joint_bf16x8_kernel(const __nv_bfloat16* __restrict__ offset, const float* __restrict__ depth, int S, int J, int fs,
                           const float* __restrict__ kernel_vec, float* __restrict__ joint_out) {
    __shared__ float smx[4][K4A_JPC];
    __shared__ float part[4][4 * K4A_JPC];
    __shared__ float coord[128];   // cell_coord(i), i < fs <= 128 (HW = 1024, fs % 8 == 0): fs IEEE divisions per CTA instead of 9 per thread
    const int j0 = blockIdx.x * K4A_JPC, b = blockIdx.y, HW = fs * fs, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const __nv_bfloat16* base = offset + (size_t)b * 5 * J * HW;
    const int m0 = 8 * tid, r = m0 / fs, col0 = m0 - r * fs;
    if (tid < fs) coord[tid] = cell_coord(tid, (float)fs);   // read after the barrier of phase A
    auto row16 = [&](int ch) { return __ldg(reinterpret_cast<const uint4*>(base + (size_t)ch * HW + m0)); };
    // ---- phase A
    uint4 vw[K4A_JPC];
#pragma unroll
    for (int jj = 0; jj < K4A_JPC; ++jj) vw[jj] = j0 + jj < J ? row16(4 * J + j0 + jj) : make_uint4(0, 0, 0, 0);
    uint4 nx[4];   // the first joint's other four rows are already on their way
    nx[0] = row16(3 * j0); nx[1] = row16(3 * j0 + 1); nx[2] = row16(3 * j0 + 2); nx[3] = row16(3 * J + j0);
    // nearest down-sample (model.py:409): floor(dst * (S / fs)) is dst * (S / fs) in integers when fs divides S (the float product is exact)
    const int step = S % fs == 0 ? S / fs : 0;
    const float* drow = depth + (size_t)b * S * S + (size_t)(step ? r * step : nearest_src(r, S, fs)) * S;
    float d[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = __ldg(drow + (step ? (col0 + i) * step : nearest_src(col0 + i, S, fs)));
    float wv[K4A_JPC][8], mx[K4A_JPC];
#pragma unroll
    for (int jj = 0; jj < K4A_JPC; ++jj) {
        const __nv_bfloat16* pw = reinterpret_cast<const __nv_bfloat16*>(&vw[jj]);
        mx[jj] = -INFINITY;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            wv[jj][i] = d[i] > 0.99f ? -1e8f : __bfloat162float(pw[i]);  // masked_fill(depth.gt(0.99), -1e8)  :488
            mx[jj] = fmaxf(mx[jj], wv[jj][i]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx[jj] = fmaxf(mx[jj], __shfl_xor_sync(0xffffffffu, mx[jj], o));
        if (lane == 0) smx[w][jj] = mx[jj];
    }
    __syncthreads();
#pragma unroll
    for (int jj = 0; jj < K4A_JPC; ++jj) mx[jj] = fmaxf(fmaxf(smx[0][jj], smx[1][jj]), fmaxf(smx[2][jj], smx[3][jj]));
    // ---- phase B
    const float cr = coord[r];
    float cc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) cc[i] = coord[col0 + i];
    float acc[K4A_JPC][4];
#pragma unroll
    for (int jj = 0; jj < K4A_JPC; ++jj) {
        const uint4 vx = nx[0], vy = nx[1], vz = nx[2], vh = nx[3];
        if (jj + 1 < K4A_JPC && j0 + jj + 1 < J) {
            const int j = j0 + jj + 1;
            nx[0] = row16(3 * j); nx[1] = row16(3 * j + 1); nx[2] = row16(3 * j + 2); nx[3] = row16(3 * J + j);
        }
        const float ks = j0 + jj < J ? __ldg(kernel_vec + j0 + jj) : 0.f;
        const __nv_bfloat16 *px = reinterpret_cast<const __nv_bfloat16*>(&vx), *py = reinterpret_cast<const __nv_bfloat16*>(&vy),
                            *pz = reinterpret_cast<const __nv_bfloat16*>(&vz), *ph = reinterpret_cast<const __nv_bfloat16*>(&vh);
        float se = 0.f, ax = 0.f, ay = 0.f, az = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float e = expf(wv[jj][i] - mx[jj]);
            // depth.lt(0.99) mask (:485): a masked cell's offsets are zero, i.e. it contributes its own coordinates -- same value as the
            // generic kernel's (o * 0) * dist + c, with one select instead of four multiplications
            const float dist = d[i] < 0.99f ? ks - __bfloat162float(ph[i]) * ks : 0.f;    // :495
            se += e;
            ax += (__bfloat162float(px[i]) * dist + cc[i]) * e;                           // coords ch0 = column  :481
            ay += (__bfloat162float(py[i]) * dist + cr) * e;
            az += (__bfloat162float(pz[i]) * dist + d[i]) * e;
        }
        acc[jj][0] = se; acc[jj][1] = ax; acc[jj][2] = ay; acc[jj][3] = az;
    }
    // ---- phase C
#pragma unroll
    for (int jj = 0; jj < K4A_JPC; ++jj)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float v = acc[jj][k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) part[w][4 * jj + k] = v;
        }
    __syncthreads();
    if (tid < 3 * K4A_JPC) {
        const int jj = tid / 3, k = tid - 3 * jj;
        if (j0 + jj < J) {
            const float se = ((part[0][4 * jj] + part[1][4 * jj]) + part[2][4 * jj]) + part[3][4 * jj];
            const float a = ((part[0][4 * jj + 1 + k] + part[1][4 * jj + 1 + k]) + part[2][4 * jj + 1 + k]) + part[3][4 * jj + 1 + k];
            joint_out[((size_t)b * J + j0 + jj) * 3 + k] = a / se;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K4b / a7: pcl_joint2offset   model/model.py:503-525 -> [B,N,4J] (3J joint-major unit vectors, then J closeness)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pcl_joint2offset_kernel(const float* __restrict__ joint, const float* __restrict__ pcl, const float* __restrict__ kernel_vec,
                        int J, int N, float* __restrict__ out) {
    const int b = blockIdx.y;
    const int j = threadIdx.x;                       // blockDim.x = 32 >= J handled by loop below
    const int n = blockIdx.x * blockDim.y + threadIdx.y;
    if (n >= N) return;
    const float* p = pcl + ((size_t)b * N + n) * 3;
    const float px = p[0], py = p[1], pz = p[2];
    float* o = out + ((size_t)b * N + n) * 4 * J;
    for (int jj = j; jj < J; jj += blockDim.x) {
        const float* q = joint + ((size_t)b * J + jj) * 3;
        const float ox = q[0] - px, oy = q[1] - py, oz = q[2] - pz;
        const float dis = sqrtf(ox * ox + oy * oy + oz * oz);
        const float inv = 1.0f / (dis + 1e-8f);
        const float ks = kernel_vec[jj];
        const float heat = (ks - dis) / ks;
        const float msk = (heat >= 0.f && pz < 0.99f) ? 1.f : 0.f;  // :522
        o[3 * jj + 0] = ox * inv * msk;
        o[3 * jj + 1] = oy * inv * msk;
        o[3 * jj + 2] = oz * inv * msk;
        o[3 * J + jj] = heat * msk;
    }
}

// ------------------------------------------------------------------------------------------------
// K4c / a10: GFM.joint2heatmap   util/generateFeature.py:584-600
// ------------------------------------------------------------------------------------------------
__global__ void joint2heatmap_kernel(const float* __restrict__ joint, int joint_stride, int J, int S, float stdv, float sigma,
                                     float* __restrict__ out) {
    const int bj = blockIdx.y;  // b*J + j
    const float jx = (joint[(size_t)bj * joint_stride + 0] + 1.f) / 2.f * (float)S;
    const float jy = (joint[(size_t)bj * joint_stride + 1] + 1.f) / 2.f * (float)S;
    const float inv2s2 = 1.f / (2.f * sigma * sigma);
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < S * S; m += gridDim.x * blockDim.x) {
        const int r = m / S, col = m - r * S;
        const float dx = ((float)col + 0.5f - jx) / stdv, dy = ((float)r + 0.5f - jy) / stdv;
        out[(size_t)bj * S * S + m] = expf(-(dx * dx + dy * dy) * inv2s2);
    }
}

// ------------------------------------------------------------------------------------------------
// K4c / a11: loader.img2anchor_dis   dataloader/loader.py:791-819 -> GAM [B,J,H,W]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
img2anchor_dis_kernel(const float* __restrict__ joint_uvd, const float* __restrict__ depth, long long depth_bs, int depth_rs,
                      int depth_cs, const float* __restrict__ center, const float* __restrict__ M,
                      const float* __restrict__ cube, const float* __restrict__ cam, int J, int fs, float img_size, float flip,
                      float gamma, float* __restrict__ out) {
    extern __shared__ float jxyz[];  // [J*3]
    __shared__ CamF c;
    const int b = blockIdx.y, HW = fs * fs;
    if (threadIdx.x == 0) load_cam(c, b, center, M, cube, cam, img_size, flip);
    __syncthreads();
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
        const float* s = joint_uvd + ((size_t)b * J + j) * 3;
        const float3 q = uvd2xyz(c, s[0], s[1], s[2]);
        jxyz[3 * j] = q.x;
        jxyz[3 * j + 1] = q.y;
        jxyz[3 * j + 2] = q.z;
    }
    __syncthreads();
    const float ffs = (float)fs;
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < HW; m += gridDim.x * blockDim.x) {
        const int r = m / fs, col = m - r * fs;
        const float d = __ldg(depth + (size_t)b * depth_bs + (size_t)r * depth_rs + (size_t)col * depth_cs);
        const float3 q = uvd2xyz(c, cell_coord(col, ffs), cell_coord(r, ffs), d);
        for (int j = 0; j < J; ++j) {
            const float dx = q.x - jxyz[3 * j], dy = q.y - jxyz[3 * j + 1], dz = q.z - jxyz[3 * j + 2];
            out[((size_t)b * J + j) * HW + m] = 1.f / (gamma * (dx * dx + dy * dy + dz * dz) + 1.f);  // :814-818
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K4d / a16: GFM.joint2offset   util/generateFeature.py:59-84 (eps=1e-8) / model.py:440-463 (eps=0)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
joint2offset_kernel(const float* __restrict__ joint, const float* __restrict__ depth, int S, int J, int fs,
                    const float* __restrict__ kernel_vec, float eps, float* __restrict__ out) {
    extern __shared__ float js[];  // [J*4]: xyz + kernel
    const int b = blockIdx.y, HW = fs * fs;
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
        js[4 * j] = joint[((size_t)b * J + j) * 3];
        js[4 * j + 1] = joint[((size_t)b * J + j) * 3 + 1];
        js[4 * j + 2] = joint[((size_t)b * J + j) * 3 + 2];
        js[4 * j + 3] = kernel_vec[j];
    }
    __syncthreads();
    const float ffs = (float)fs;
    float* ob = out + (size_t)b * 4 * J * HW;
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < HW; m += gridDim.x * blockDim.x) {
        const int r = m / fs, col = m - r * fs;
        const float d = __ldg(depth + (size_t)b * S * S + (size_t)nearest_src(r, S, fs) * S + nearest_src(col, S, fs));
        const float u = cell_coord(col, ffs), v = cell_coord(r, ffs);
        const float fg = d < 0.99f ? 1.f : 0.f;
        for (int j = 0; j < J; ++j) {
            const float ox = js[4 * j] - u, oy = js[4 * j + 1] - v, oz = js[4 * j + 2] - d;
            const float dist = sqrtf(ox * ox + oy * oy + oz * oz + eps);
            const float ks = js[4 * j + 3];
            const float heat = (ks - dist) / ks;
            const float msk = heat >= 0.f ? fg : 0.f;
            ob[(size_t)(3 * j) * HW + m] = ox / dist * msk;
            ob[(size_t)(3 * j + 1) * HW + m] = oy / dist * msk;
            ob[(size_t)(3 * j + 2) * HW + m] = oz / dist * msk;
            ob[(size_t)(3 * J + j) * HW + m] = heat * msk;
        }
    }
}

}  // namespace kpf

using namespace kpf;

extern "C" int kpf_uvd2xyz(const float* uvd, const float* center, const float* M, const float* cube, const float* cam, int B,
                           int P, float img_size, float flip, float* out, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && P >= 0);
    if (B == 0 || P == 0) return 0;
    dim3 grid((P + 255) / 256 > 64 ? 64 : (P + 255) / 256, B);
    uvd2xyz_kernel<<<grid, 256, 0, stream>>>(uvd, center, M, cube, cam, P, img_size, flip, out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_xyz2uvd(const float* xyz, const float* center, const float* M, const float* cube, const float* cam, int B,
                           int P, float img_size, float flip, float* out, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && P >= 0);
    if (B == 0 || P == 0) return 0;
    dim3 grid((P + 255) / 256 > 64 ? 64 : (P + 255) / 256, B);
    xyz2uvd_kernel<<<grid, 256, 0, stream>>>(xyz, center, M, cube, cam, P, img_size, flip, out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_joints_to_frame(const float* joints, const float* center, const float* cube, const float* cam, int B, int P, float flip,
                                   float* uvd_frame_out, float* xyz_cam_out, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && P >= 0);
    const long long n = (long long)B * P;
    if (n == 0) return 0;
    joints_to_frame_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(joints, center, cube, cam, B, P, flip, uvd_frame_out, xyz_cam_out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_spatial_order(const float* pcl, const float* center, const float* M, const float* cube, const float* cam, int B, int N,
                                 int fs, float img_size, float flip, int32_t* order, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && N >= 1 && N <= 8192 && fs >= 1 && fs * fs <= (1 << 19));
    if (B == 0) return 0;
    int npow2 = 1;
    while (npow2 < N) npow2 <<= 1;
    kpf::spatial_order_kernel<<<B, 1024, (size_t)npow2 * 4, stream>>>(pcl, center, M, cube, cam, N, npow2, fs, img_size, flip, order);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_img2pcl_index(const float* pcl, const float* depth, long long depth_bs, int depth_rs, int depth_cs,
                                 const float* center, const float* M, const float* cube, const float* cam, int B, int N, int fs,
                                 float img_size, float flip, int K, const int32_t* order, float* closeness, long long* index64,
                                 int32_t* index32, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && N >= 0 && fs >= 1 && fs * fs <= 8192 && K >= 1 && K <= fs * fs);
    if (B == 0 || N == 0) return 0;
    // (row quarters per point group, threads per CTA): measured at batch 64, S = 128, K = 4 (profiles/probe_k2.py): (1, 256) 43.4 us,
    // (2, 256) 39.4, (2, 512) 36.7, (4, 512) 49.9, (4, 1024) 48.8 -- two warps per point group pay for their second window seeding and
    // the merge, four do not; seeding each warp only from the window rows it scans itself (no redundant seeding) loosens the bound and
    // is far slower (49 / 86 us with two / four warps).
    constexpr int RQ = 2, NT = 512, PTS = NT / RQ;
    dim3 grid((N + PTS - 1) / PTS, B);
    const size_t smem = ((size_t)fs * fs + 2 * (size_t)fs) * sizeof(float4) + (size_t)(NT / 32 / RQ) * (RQ - 1) * K * 32 * 8;
#define KPF_LAUNCH_K2(KK)                                                                                                    \
    case KK: {                                                                                                               \
        cudaError_t e = kpf::set_smem(nearest_cells_kernel<KK, RQ, NT>, smem);                                               \
        if (e != cudaSuccess) return (int)e;                                                                                 \
        nearest_cells_kernel<KK, RQ, NT><<<grid, NT, smem, stream>>>(pcl, depth, depth_bs, depth_rs, depth_cs, center, M, cube, cam, N, \
                                                                     fs, img_size, flip, order, closeness, index64, index32);   \
    } break;
    switch (K) {
        KPF_LAUNCH_K2(1)
        KPF_LAUNCH_K2(2)
        KPF_LAUNCH_K2(3)
        KPF_LAUNCH_K2(4)
        KPF_LAUNCH_K2(5)
        KPF_LAUNCH_K2(6)
        KPF_LAUNCH_K2(7)
        KPF_LAUNCH_K2(8)
        KPF_LAUNCH_K2(9)
        KPF_LAUNCH_K2(16)
        default:
            return KPF_ERR_UNSUPPORTED;
    }
#undef KPF_LAUNCH_K2
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_offset2joint_weight(const void* offset, int dtype, const float* depth, int B, int J, int fs, int S,
                                       const float* kernel_vec, float* joint_out, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && J >= 1 && fs >= 1 && S >= fs);
    if (B == 0) return 0;
    dim3 grid(J, B);
    if (dtype == KPF_F32) {
        kpf::set_smem(offset2joint_kernel<float>, 0);
        offset2joint_kernel<float><<<grid, 256, 0, stream>>>((const float*)offset, depth, S, J, fs, kernel_vec, joint_out);
    } else if (dtype == KPF_BF16 && fs * fs == 8 * 128 && fs % 8 == 0 && ((uintptr_t)offset % 16) == 0) {
        // joints per CTA: 7 amortise the per-CTA setup best once the grid fills the GPU several times over (batch 512: 37 us vs 41 us,
        // 3.0 TB/s); 3 keep enough CTAs at small batches (batch 64: 8.7 us vs 10.1 us) -- profiles/probe_k4a.py
#define KPF_K4A(JPC, MINB)                                                                                                   \
    do {                                                                                                                     \
        kpf::set_smem(offset2joint_bf16x8_kernel<JPC, MINB>, 0);                                                             \
        grid.x = (J + JPC - 1) / JPC;                                                                                        \
        offset2joint_bf16x8_kernel<JPC, MINB><<<grid, 128, 0, stream>>>((const __nv_bfloat16*)offset, depth, S, J, fs, kernel_vec, joint_out); \
    } while (0)
        const bool big = (long long)B * ((J + 6) / 7) >= 4 * 148;
        if (big) KPF_K4A(7, 4);
        else KPF_K4A(3, 5);
#undef KPF_K4A
    } else if (dtype == KPF_BF16) {
        kpf::set_smem(offset2joint_kernel<__nv_bfloat16>, 0);
        offset2joint_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)offset, depth, S, J, fs, kernel_vec, joint_out);
    } else {
        return KPF_ERR_UNSUPPORTED;
    }
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_pcl_joint2offset(const float* joint, const float* pcl, const float* kernel_vec, int B, int J, int N,
                                    float* out, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && J >= 1 && N >= 0);
    if (B == 0 || N == 0) return 0;
    dim3 block(32, 8), grid((N + 7) / 8, B);
    pcl_joint2offset_kernel<<<grid, block, 0, stream>>>(joint, pcl, kernel_vec, J, N, out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_joint2heatmap(const float* joint, int joint_stride, int B, int J, int S, float stdv, float sigma, float* out,
                                 cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && J >= 1 && S >= 1 && joint_stride >= 2);
    if (B == 0) return 0;
    dim3 grid((S * S + 255) / 256 > 16 ? 16 : (S * S + 255) / 256, B * J);
    joint2heatmap_kernel<<<grid, 256, 0, stream>>>(joint, joint_stride, J, S, stdv, sigma, out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_img2anchor_dis(const float* joint_uvd, const float* depth, long long depth_bs, int depth_rs, int depth_cs,
                                  const float* center, const float* M, const float* cube, const float* cam, int B, int J, int fs,
                                  float img_size, float flip, float gamma, float* out, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && J >= 1 && fs >= 1);
    if (B == 0) return 0;
    dim3 grid((fs * fs + 255) / 256, B);
    img2anchor_dis_kernel<<<grid, 256, (size_t)J * 3 * sizeof(float), stream>>>(joint_uvd, depth, depth_bs, depth_rs, depth_cs,
                                                                              center, M, cube, cam, J, fs, img_size, flip, gamma, out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_joint2offset(const float* joint, const float* depth, int B, int J, int S, int fs, const float* kernel_vec,
                                float eps, float* out, cudaStream_t stream) {
    KPF_REQUIRE(B >= 0 && J >= 1 && fs >= 1 && S >= fs);
    if (B == 0) return 0;
    dim3 grid((fs * fs + 255) / 256, B);
    joint2offset_kernel<<<grid, 256, (size_t)J * 4 * sizeof(float), stream>>>(joint, depth, S, J, fs, kernel_vec, eps, out);
    KPF_CHECK_LAUNCH();
    return 0;
}
