// SURVEY 8f-4: evaluation tail on the GPU (train.py:330-386, :470-488; util/generateFeature.py:681-703).
//   err[b][j]    = || (pred - gt) * cube/2 ||                                   (Trainer.xyz2error, mm)
//   pa_err[b][j] = same after the similarity (Procrustes / Umeyama) alignment of pred onto gt  (GFM.rigid_align)
// The reference loops over the batch in Python with a numpy SVD per sample and a .cpu() copy per call; here one thread per
// sample does the 3x3 SVD in fp64 (Jacobi eigen-decomposition of H^T H), so evaluation never leaves the device.
// kpf_eval_accumulate runs the same per-sample code for S stacked joint sets and adds the results into a caller-owned int64
// accumulator in fixed point (2^20 units per mm), so totals are exact and do not depend on batch order, split or rank count.
#include "common.cuh"

namespace kpf {

// eigen-decomposition of a symmetric 3x3 (cyclic Jacobi, fp64): A = V diag(w) V^T, columns of V are eigenvectors
__device__ void jacobi3(double A[3][3], double V[3][3], double w[3]) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) V[i][j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 30; ++sweep) {
        const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
        if (off < 1e-300) break;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                if (fabs(A[p][q]) < 1e-300) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 3; ++k) {
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - s * akq;
                    A[k][q] = s * akp + c * akq;
                }
                for (int k = 0; k < 3; ++k) {
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - s * aqk;
                    A[q][k] = s * apk + c * aqk;
                }
                for (int k = 0; k < 3; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - s * vkq;
                    V[k][q] = s * vkp + c * vkq;
                }
            }
    }
    for (int i = 0; i < 3; ++i) w[i] = A[i][i];
}

// One sample's errors: sink(0, j, err_j) for j = 0..J-1, then, if `aligned`, sink(1, j, pa_err_j) for j = 0..J-1, each the fp32
// value kpf_eval_errors stores.  Both loops run over the same J in every thread, so a sink may use warp collectives.
template <class Sink>
__device__ __forceinline__ void eval_sample(const float* __restrict__ P, const float* __restrict__ G, const float* __restrict__ cube3, int J,
                                            bool aligned, Sink&& sink) {
    const double h[3] = {cube3[0] / 2.0, cube3[1] / 2.0, cube3[2] / 2.0};
    // plain error (the centre cancels in the difference; train.py:480-487)
    for (int j = 0; j < J; ++j) {
        double s = 0;
        for (int k = 0; k < 3; ++k) {
            const double d = ((double)P[3 * j + k] - (double)G[3 * j + k]) * h[k];
            s += d * d;
        }
        sink(0, j, (float)sqrt(s));
    }
    if (!aligned) return;
    // rigid_transform_3D (generateFeature.py:681-697): A = pred, B = gt (normalised coordinates)
    double ca[3] = {0, 0, 0}, cb[3] = {0, 0, 0};
    for (int j = 0; j < J; ++j)
        for (int k = 0; k < 3; ++k) {
            ca[k] += P[3 * j + k];
            cb[k] += G[3 * j + k];
        }
    for (int k = 0; k < 3; ++k) {
        ca[k] /= J;
        cb[k] /= J;
    }
    double H[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}, varP = 0;
    for (int j = 0; j < J; ++j) {
        double a[3], bb[3];
        for (int k = 0; k < 3; ++k) {
            a[k] = P[3 * j + k] - ca[k];
            bb[k] = G[3 * j + k] - cb[k];
            varP += a[k] * a[k];
        }
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) H[r][c] += a[r] * bb[c];
    }
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) H[r][c] /= J;
    varP /= J;
    // SVD H = U diag(s) V^T through the eigen-decomposition of H^T H
    double S[3][3], V[3][3], w[3];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) S[r][c] = H[0][r] * H[0][c] + H[1][r] * H[1][c] + H[2][r] * H[2][c];
    jacobi3(S, V, w);
    int o[3] = {0, 1, 2};  // sort descending
    for (int i = 0; i < 2; ++i)
        for (int k = i + 1; k < 3; ++k)
            if (w[o[k]] > w[o[i]]) {
                const int t = o[i];
                o[i] = o[k];
                o[k] = t;
            }
    double sv[3], Vc[3][3], U[3][3];
    for (int i = 0; i < 3; ++i) {
        sv[i] = sqrt(fmax(w[o[i]], 0.0));
        for (int r = 0; r < 3; ++r) Vc[r][i] = V[r][o[i]];
    }
    for (int i = 0; i < 2; ++i) {
        double n = 0;
        for (int r = 0; r < 3; ++r) {
            U[r][i] = H[r][0] * Vc[0][i] + H[r][1] * Vc[1][i] + H[r][2] * Vc[2][i];
            n += U[r][i] * U[r][i];
        }
        n = sqrt(n);
        for (int r = 0; r < 3; ++r) U[r][i] = n > 0 ? U[r][i] / n : (r == i ? 1.0 : 0.0);
    }
    // third left / right vectors completed as cross products: a proper (det +1) pair; the reflection case is handled by `sgn`
    U[0][2] = U[1][0] * U[2][1] - U[2][0] * U[1][1];
    U[1][2] = U[2][0] * U[0][1] - U[0][0] * U[2][1];
    U[2][2] = U[0][0] * U[1][1] - U[1][0] * U[0][1];
    double v3[3] = {Vc[1][0] * Vc[2][1] - Vc[2][0] * Vc[1][1], Vc[2][0] * Vc[0][1] - Vc[0][0] * Vc[2][1], Vc[0][0] * Vc[1][1] - Vc[1][0] * Vc[0][1]};
    // sign of the third singular pair relative to the true SVD: s3 * (u3 . H v3) ; det(V U^T) = +1 by construction here, so the
    // reference's det(R) < 0 branch corresponds to u3 . (H v3) < 0
    double hv3[3] = {H[0][0] * v3[0] + H[0][1] * v3[1] + H[0][2] * v3[2], H[1][0] * v3[0] + H[1][1] * v3[1] + H[1][2] * v3[2],
                     H[2][0] * v3[0] + H[2][1] * v3[1] + H[2][2] * v3[2]};
    const double dotp = U[0][2] * hv3[0] + U[1][2] * hv3[1] + U[2][2] * hv3[2];
    const double sgn = dotp < 0 ? -1.0 : 1.0;
    for (int r = 0; r < 3; ++r) Vc[r][2] = v3[r];
    // R = V diag(1,1,1) U^T with (u3, v3) right-handed completions == reference R after its reflection fix;  c = (s1+s2+sgn*s3)/varP
    double R[3][3];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r][c] = Vc[r][0] * U[c][0] + Vc[r][1] * U[c][1] + Vc[r][2] * U[c][2];
    const double scale = (sv[0] + sv[1] + sgn * sv[2]) / varP;
    double t[3];
    for (int r = 0; r < 3; ++r) t[r] = -scale * (R[r][0] * ca[0] + R[r][1] * ca[1] + R[r][2] * ca[2]) + cb[r];
    for (int j = 0; j < J; ++j) {
        double s = 0;
        for (int r = 0; r < 3; ++r) {
            const double a2 = scale * (R[r][0] * P[3 * j] + R[r][1] * P[3 * j + 1] + R[r][2] * P[3 * j + 2]) + t[r];
            const double d = (a2 - (double)G[3 * j + r]) * h[r];
            s += d * d;
        }
        sink(1, j, (float)sqrt(s));
    }
}

__global__ void eval_errors_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const float* __restrict__ cube, int B,
                                   int J, float* __restrict__ err, float* __restrict__ pa_err) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    eval_sample(pred + (size_t)b * J * 3, gt + (size_t)b * J * 3, cube + 3 * b, J, pa_err != nullptr,
                [&](int kind, int j, float e) { (kind ? pa_err : err)[(size_t)b * J + j] = e; });
}

// ---- accumulation (kpf_eval_accumulate): one thread per (stage, sample), blockIdx.y = stage, so every warp holds one stage.
// A thread's time is the fp64 code of eval_sample (91 us at B = 64, S = 5 on a B200 at its 1000 W limit); staging the block's inputs
// in shared memory first measured the same (90.0 against 91.4 us), so they are read from global memory as eval_errors reads them.
constexpr int EV_THREADS = 64, EV_MAX_J = 32, EV_MAX_T = 256;
constexpr float EV_CLAMP_MM = 1048576.0f;   // 2^20 mm
constexpr double EV_SCALE = 1048576.0;      // fixed point: 2^20 units per mm

// index of the first threshold >= e (fp32 compare), T when there is none or e is NaN
__device__ __forceinline__ int eval_bin(const float* thr, int T, float e) {
    int lo = 0, hi = T;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (e <= thr[mid])
            hi = mid;
        else
            lo = mid + 1;
    }
    return lo;
}

__global__ void __launch_bounds__(EV_THREADS) eval_accumulate_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                                     const float* __restrict__ cube, const uint8_t* __restrict__ valid,
                                                                     const float* __restrict__ thr, int B, int J, int T,
                                                                     unsigned long long* __restrict__ acc) {
    __shared__ float s_thr[EV_MAX_T];
    __shared__ unsigned long long s_sum[2][EV_MAX_J];
    __shared__ unsigned s_nonfinite[2][EV_MAX_J];
    __shared__ unsigned s_hist[2][EV_MAX_T + 1];
    const int tid = threadIdx.x, lane = tid & 31, stage = blockIdx.y;
    for (int i = tid; i < 2 * EV_MAX_J; i += EV_THREADS) {
        s_sum[i / EV_MAX_J][i % EV_MAX_J] = 0;
        s_nonfinite[i / EV_MAX_J][i % EV_MAX_J] = 0;
    }
    for (int i = tid; i < 2 * (T + 1); i += EV_THREADS) s_hist[i / (T + 1)][i % (T + 1)] = 0;
    for (int i = tid; i < T; i += EV_THREADS) s_thr[i] = thr[i];
    __syncthreads();

    // threads past the batch or on a masked sample run the same loops on a real sample (the sink's warp collectives need every
    // lane) and contribute nothing
    const int b = blockIdx.x * EV_THREADS + tid;
    const bool active = b < B && (valid == nullptr || valid[b] != 0);
    const int bl = b < B ? b : B - 1;
    eval_sample(pred + ((size_t)stage * B + bl) * J * 3, gt + (size_t)bl * J * 3, cube + 3 * bl, J, true, [&](int kind, int j, float e) {
        const bool finite = isfinite(e);
        unsigned long long q = active && finite ? (unsigned long long)llrint((double)fminf(e, EV_CLAMP_MM) * EV_SCALE) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const unsigned nonfinite = __popc(__ballot_sync(0xffffffffu, active && !finite));
        if (lane == 0) {
            if (q) atomicAdd(&s_sum[kind][j], q);
            if (nonfinite) atomicAdd(&s_nonfinite[kind][j], nonfinite);
        }
        if (active) atomicAdd(&s_hist[kind][eval_bin(s_thr, T, e)], 1u);
    });
    const int samples = __syncthreads_count(active);

    // row layout (include/kpf_b200.h): samples | sum err [J] | sum pa [J] | nonfinite err [J] | nonfinite pa [J] | hist err [T+1] | hist pa [T+1]
    unsigned long long* row = acc + (size_t)stage * (1 + 4 * J + 2 * (T + 1));
    if (tid == 0 && samples) atomicAdd(row, (unsigned long long)samples);
    for (int i = tid; i < 2 * J; i += EV_THREADS) {
        const unsigned long long s = s_sum[i / J][i % J];
        const unsigned n = s_nonfinite[i / J][i % J];
        if (s) atomicAdd(row + 1 + i, s);
        if (n) atomicAdd(row + 1 + 2 * J + i, (unsigned long long)n);
    }
    for (int i = tid; i < 2 * (T + 1); i += EV_THREADS) {
        const unsigned n = s_hist[i / (T + 1)][i % (T + 1)];
        if (n) atomicAdd(row + 1 + 4 * J + i, (unsigned long long)n);
    }
}

}  // namespace kpf

extern "C" int kpf_eval_errors(const float* pred, const float* gt, const float* cube, int B, int J, float* err, float* pa_err,
                               cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && J >= 3);
    if (B == 0) return 0;
    eval_errors_kernel<<<(B + 63) / 64, 64, 0, stream>>>(pred, gt, cube, B, J, err, pa_err);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_eval_accumulate(const float* pred, const float* gt, const float* cube, const uint8_t* valid, const float* thresholds, int S,
                                   int B, int J, int T, long long* acc, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(S >= 1 && S <= 8 && B >= 0 && J >= 3 && J <= EV_MAX_J && T >= 1 && T <= EV_MAX_T);
    KPF_REQUIRE(thresholds != nullptr && acc != nullptr);
    if (B == 0) return 0;
    KPF_REQUIRE(pred != nullptr && gt != nullptr && cube != nullptr);
    eval_accumulate_kernel<<<dim3((B + EV_THREADS - 1) / EV_THREADS, S), EV_THREADS, 0, stream>>>(pred, gt, cube, valid, thresholds, B, J, T,
                                                                                                  (unsigned long long*)acc);
    KPF_CHECK_LAUNCH();
    return 0;
}
