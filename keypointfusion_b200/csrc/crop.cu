// SURVEY 8f-3: crop + normalise front end for in-the-wild RGB-D frames (BASELINE config 5), demo_RGBD.py:
//   get_center_from_bbx :253-276, comToBounds :519-529, getCrop :531-569, Crop_Image_deep_pp :410-462,
//   Crop_Image_deep_pp_RGB :464-517, normalize_img :378-385, jointImgTo3D :387-.
// One CTA per box; box b reads frame frame_index[b] (frame b when frame_index is NULL), so several hands of one frame share
// one upload.  An index outside [0,F) is never dereferenced: that box's outputs are NaN.  All integer work (bounds, cv2 INTER_NEAREST source indices, paste offsets, uint16 z-threshold casts)
// is reproduced bit-exactly in fp64 / integer arithmetic; the frame is read once (only the pixels the crop samples).
// HBM-bound and tiny: a 128 x 128 crop touches <= 16384 source pixels of the uint16 frame.
#include "common.cuh"

namespace kpf {

struct CropGeom {
    int xs, xe, ys, ye, szw, szh, px, py;
    double zs, ze, sc, ifx, ify;
};

__device__ __forceinline__ int box_frame(const int32_t* frame_index, int b, int F) {
    const int f = frame_index ? frame_index[b] : b;
    return (f >= 0 && f < F) ? f : -1;
}

// comToBounds + resize size + paste offset (fp64, reference operation order)
__device__ __forceinline__ void crop_geometry(const double* com, const float* size, const double* cam, int dsize, CropGeom& g) {
    const double fx = cam[0], fy = cam[1];
    const double s0 = size[0], s1 = size[1], s2 = size[2];
    g.zs = com[2] - s2 / 2.;
    g.ze = com[2] + s2 / 2.;
    g.xs = (int)floor((com[0] * com[2] / fx - s0 / 2.) / com[2] * fx + 0.5);
    g.xe = (int)floor((com[0] * com[2] / fx + s0 / 2.) / com[2] * fx + 0.5);
    g.ys = (int)floor((com[1] * com[2] / fy - s1 / 2.) / com[2] * fy + 0.5);
    g.ye = (int)floor((com[1] * com[2] / fy + s1 / 2.) / com[2] * fy + 0.5);
    const int wb = g.xe - g.xs, hb = g.ye - g.ys;
    if (wb > hb) {
        g.szw = dsize;
        g.szh = (int)((double)hb * dsize / wb);   // int(hb * dsize[0] / wb): true division then truncation
    } else {
        g.szw = (int)((double)wb * dsize / hb);
        g.szh = dsize;
    }
    g.sc = hb > wb ? g.szh / (double)hb : g.szw / (double)wb;
    g.px = (int)floor(dsize / 2. - g.szw / 2.);
    g.py = (int)floor(dsize / 2. - g.szh / 2.);
    g.ifx = 1.0 / ((double)g.szw / (double)wb);     // cv2.resize: ifx = 1 / inv_scale_x, sx = min(floor(x * ifx), src - 1)
    g.ify = 1.0 / ((double)g.szh / (double)hb);
}

__global__ void __launch_bounds__(256)
center_from_bbox_kernel(const uint16_t* __restrict__ depth, const double* __restrict__ bbox, const int32_t* __restrict__ frame_index,
                        int F, int Hf, int Wf, int upper, int lower, double* __restrict__ center) {
    __shared__ unsigned long long sh[4][8];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int fr = box_frame(frame_index, b, F);
    if (fr < 0) {   // uniform over the CTA
        if (tid < 3) center[3 * b + tid] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    const double* bb = bbox + 4 * b;
    const int x0 = (int)bb[0], x1 = (int)(bb[0] + bb[2]), y0 = (int)bb[1], y1 = (int)(bb[1] + bb[3]);
    const int cx0 = max(x0, 0), cx1 = min(x1, Wf), cy0 = max(y0, 0), cy1 = min(y1, Hf);   // numpy slicing clips at the frame
    const int w = max(cx1 - cx0, 0), h = max(cy1 - cy0, 0);
    unsigned long long sc = 0, sr = 0, sd = 0, cnt = 0;
    const uint16_t* f = depth + (size_t)fr * Hf * Wf;
    for (int i = tid; i < w * h; i += blockDim.x) {
        const int r = i / w, c = i - r * w;
        const int v = f[(size_t)(cy0 + r) * Wf + cx0 + c];
        if (v <= upper && v >= lower) {
            sc += c;
            sr += r;
            sd += v;
            cnt += 1;
        }
    }
    unsigned long long v4[4] = {sc, sr, sd, cnt};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v4[q] += __shfl_xor_sync(0xffffffffu, v4[q], o);
        if ((tid & 31) == 0) sh[q][tid >> 5] = v4[q];
    }
    __syncthreads();
    if (tid == 0) {
        unsigned long long t[4] = {0, 0, 0, 0};
        for (int q = 0; q < 4; ++q)
            for (int k = 0; k < 8; ++k) t[q] += sh[q][k];
        double c0 = 0.0, c1 = 0.0, c2 = 300.0;
        if (t[3] > 0) {
            // np.linspace(0, w, w)[c] = c * w / (w - 1)
            const double stepx = w > 1 ? (double)w / (double)(w - 1) : 0.0, stepy = h > 1 ? (double)h / (double)(h - 1) : 0.0;
            c0 = (double)t[0] * stepx / (double)t[3];
            c1 = (double)t[1] * stepy / (double)t[3];
            c2 = (double)t[2] / (double)t[3];
            if (c2 <= 0) c2 = 300.0;
        }
        center[3 * b + 0] = c0 + bb[0];
        center[3 * b + 1] = c1 + bb[1];
        center[3 * b + 2] = c2;
    }
}

__global__ void __launch_bounds__(256)
crop_depth_kernel(const uint16_t* __restrict__ depth, const double* __restrict__ center, const float* __restrict__ cube,
                  const double* __restrict__ cam, const int32_t* __restrict__ frame_index, int F, int Hf, int Wf, int dsize,
                  float* __restrict__ img_out, float* __restrict__ M_out, float* __restrict__ com3d_out) {
    extern __shared__ float crop[];   // [dsize*dsize]
    __shared__ CropGeom g;
    __shared__ float red[8];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int fr = box_frame(frame_index, b, F);
    if (fr < 0) {   // uniform over the CTA
        const float nan = __int_as_float(0x7fc00000);
        if (tid < 9) M_out[9 * b + tid] = nan;
        if (tid < 3) com3d_out[3 * b + tid] = nan;
        for (int i = tid; i < dsize * dsize; i += blockDim.x) img_out[(size_t)b * dsize * dsize + i] = nan;
        return;
    }
    const double* com = center + 3 * b;
    if (tid == 0) {
        crop_geometry(com, cube + 3 * b, cam + 4 * b, dsize, g);
        // trans = off . scale . trans  (demo_RGBD.py:437-462); jointImgTo3D of the centre
        float* M = M_out + 9 * b;
        M[0] = (float)g.sc; M[1] = 0.f; M[2] = (float)(g.sc * (double)(-g.xs) + (double)g.px);
        M[3] = 0.f; M[4] = (float)g.sc; M[5] = (float)(g.sc * (double)(-g.ys) + (double)g.py);
        M[6] = 0.f; M[7] = 0.f; M[8] = 1.f;
        const double fx = cam[4 * b], fy = cam[4 * b + 1], fu = cam[4 * b + 2], fv = cam[4 * b + 3];
        com3d_out[3 * b + 0] = (float)((com[0] - fu) * com[2] / fx);
        com3d_out[3 * b + 1] = (float)((com[1] - fv) * com[2] / fy);
        com3d_out[3 * b + 2] = (float)com[2];
    }
    __syncthreads();
    const uint16_t* f = depth + (size_t)fr * Hf * Wf;
    const int wb = g.xe - g.xs, hb = g.ye - g.ys;
    const uint16_t zs_cast = (uint16_t)g.zs;   // cropped[msk1] = zstart on a uint16 array
    float mx = 0.f;
    for (int i = tid; i < dsize * dsize; i += blockDim.x) {
        const int oy = i / dsize, ox = i - oy * dsize;
        const int ry = oy - g.py, rx = ox - g.px;
        float val = 0.f;                                   // background filler (:452)
        if (ry >= 0 && ry < g.szh && rx >= 0 && rx < g.szw) {
            int sy = (int)floor((double)ry * g.ify), sx = (int)floor((double)rx * g.ifx);
            sy = min(sy, hb - 1) + g.ys;
            sx = min(sx, wb - 1) + g.xs;
            uint16_t v = (sy >= 0 && sy < Hf && sx >= 0 && sx < Wf) ? f[(size_t)sy * Wf + sx] : (uint16_t)0;   // getCrop pad = 0
            if (v != 0) {
                const bool below = (double)v < g.zs, above = (double)v > g.ze;   // masks from the ORIGINAL crop (:563-566)
                if (below) v = zs_cast;
                if (above) v = 0;
            }
            val = (float)v;
        }
        crop[i] = val;
        mx = fmaxf(mx, val);
    }
    mx = warp_max(mx);
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    float premax = red[0];
#pragma unroll
    for (int k = 1; k < 8; ++k) premax = fmaxf(premax, red[k]);
    // normalize_img (demo_RGBD.py:378-385), numpy dtype semantics: float32 storage, comparisons / the subtraction against
    // float64 scalars in double, the final division in float32
    const double hi = com[2] + (double)cube[3 * b + 2] / 2., lo = com[2] - (double)cube[3 * b + 2] / 2.;
    const float hif = (float)hi, lof = (float)lo, half = (float)((double)cube[3 * b + 2] / 2.);
    for (int i = tid; i < dsize * dsize; i += blockDim.x) {
        float x = crop[i];
        if (x == premax) x = hif;
        if (x == 0.f) x = hif;
        if ((double)x >= hi) x = hif;
        if ((double)x <= lo) x = lof;
        x = (float)((double)x - com[2]);
        img_out[(size_t)b * dsize * dsize + i] = x / half;
    }
}

__global__ void __launch_bounds__(256)
crop_rgb_kernel(const uint8_t* __restrict__ rgb, const double* __restrict__ center, const float* __restrict__ cube,
                const double* __restrict__ cam, const int32_t* __restrict__ frame_index, int F, int Hf, int Wf, int dsize,
                float* __restrict__ out) {
    __shared__ CropGeom g;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int fr = box_frame(frame_index, b, F);
    if (fr < 0) {   // uniform over the CTA
        const float nan = __int_as_float(0x7fc00000);
        for (int i = tid; i < 3 * dsize * dsize; i += blockDim.x) out[(size_t)b * 3 * dsize * dsize + i] = nan;
        return;
    }
    if (tid == 0) crop_geometry(center + 3 * b, cube + 3 * b, cam + 4 * b, dsize, g);
    __syncthreads();
    const uint8_t* f = rgb + (size_t)fr * Hf * Wf * 3;
    const int wb = g.xe - g.xs, hb = g.ye - g.ys;
    for (int i = tid; i < dsize * dsize; i += blockDim.x) {
        const int oy = i / dsize, ox = i - oy * dsize;
        const int ry = oy - g.py, rx = ox - g.px;
        float v0 = 0.f, v1 = 0.f, v2 = 0.f;
        if (ry >= 0 && ry < g.szh && rx >= 0 && rx < g.szw) {
            int sy = (int)floor((double)ry * g.ify), sx = (int)floor((double)rx * g.ifx);
            sy = min(sy, hb - 1) + g.ys;
            sx = min(sx, wb - 1) + g.xs;
            if (sy >= 0 && sy < Hf && sx >= 0 && sx < Wf) {
                const uint8_t* p = f + ((size_t)sy * Wf + sx) * 3;
                v0 = (float)p[0];
                v1 = (float)p[1];
                v2 = (float)p[2];
            }
        }
        // ToTensor() on a float32 HWC array only permutes to CHW; then / 255. (demo_RGBD.py:87); channel order kept (BGR)
        float* o = out + (size_t)b * 3 * dsize * dsize + i;
        o[0] = v0 / 255.f;
        o[(size_t)dsize * dsize] = v1 / 255.f;
        o[(size_t)2 * dsize * dsize] = v2 / 255.f;
    }
}

}  // namespace kpf

extern "C" int kpf_center_from_bbox(const void* depth_u16, const double* bbox, const int32_t* frame_index, int F, int B, int Hf, int Wf,
                                    int upper, int lower, double* center_out, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && F >= 0 && Hf >= 1 && Wf >= 1 && (frame_index != nullptr || F == B));
    if (B == 0) return 0;
    center_from_bbox_kernel<<<B, 256, 0, stream>>>((const uint16_t*)depth_u16, bbox, frame_index, F, Hf, Wf, upper, lower, center_out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_crop_depth(const void* depth_u16, const double* center, const float* cube, const double* cam, const int32_t* frame_index,
                              int F, int B, int Hf, int Wf, int dsize, float* img_out, float* M_out, float* com3d_out, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && F >= 0 && Hf >= 1 && Wf >= 1 && dsize >= 8 && dsize <= 224 && (frame_index != nullptr || F == B));
    if (B == 0) return 0;
    const size_t smem = (size_t)dsize * dsize * sizeof(float);
    cudaError_t e = kpf::set_smem(crop_depth_kernel, smem);
    if (e != cudaSuccess) return (int)e;
    crop_depth_kernel<<<B, 256, smem, stream>>>((const uint16_t*)depth_u16, center, cube, cam, frame_index, F, Hf, Wf, dsize, img_out,
                                                  M_out, com3d_out);
    KPF_CHECK_LAUNCH();
    return 0;
}

extern "C" int kpf_crop_rgb(const void* rgb_u8, const double* center, const float* cube, const double* cam, const int32_t* frame_index, int F,
                            int B, int Hf, int Wf, int dsize, float* out, cudaStream_t stream) {
    using namespace kpf;
    KPF_REQUIRE(B >= 0 && F >= 0 && Hf >= 1 && Wf >= 1 && dsize >= 8 && (frame_index != nullptr || F == B));
    if (B == 0) return 0;
    crop_rgb_kernel<<<B, 256, 0, stream>>>((const uint8_t*)rgb_u8, center, cube, cam, frame_index, F, Hf, Wf, dsize, out);
    KPF_CHECK_LAUNCH();
    return 0;
}
