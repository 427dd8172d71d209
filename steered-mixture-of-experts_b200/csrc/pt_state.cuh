// Point-state layout and helpers shared by the point sweeps (points.cu: forward, cotangent, backward, coordinate
// gradient; jacobian.cu: the spatial Jacobian).
#pragma once
#include "smoe_common.cuh"
#include "fwd_records.cuh"

namespace smoe {

constexpr int PP_QTHR = 0, PP_GR = 1, PP_G = 2;                      // then C planes g_c, then d planes x'_l
__host__ __device__ constexpr int pp_x(int C) { return PP_G + C; }
__host__ __device__ constexpr int pt_stride(int d, int C) { return (2 + C + d) * SMOE_TPIX; }
constexpr int kTB = 8;                                                 // tile_box floats per tile
constexpr float kLn2 = 0.69314718055994530942f;

// tile-centred logit of one point, Horner: T + D FFMA
template <int D, int C>
__device__ __forceinline__ float point_logit(const float* __restrict__ f, const float (&x)[D]) {
    using R = Rec<D, C>;
    float q = f[R::OC];
#pragma unroll
    for (int l = 0; l < D; ++l) {
        float t = f[R::OL + l];
#pragma unroll
        for (int m = l; m < D; ++m) t = fmaf(f[R::OQ + ut(D, l, m)], x[m], t);
        q = fmaf(t, x[l], q);
    }
    return q;
}

// shared memory of the pixel-stationary point sweeps: two raw chunks, the compute records, barriers, `red`,
// `scratch` and the chunk list
template <int D, int C>
static size_t pt_sweep_smem_bytes(int max_chunks) {
    return (size_t)(2 * kChunk * pstride(D, C) + kChunk * Rec<D, C>::RC) * 4 + 2 * 8 + 32 * 4 + 8 * 4 +
           (size_t)max_chunks * 4 + 64;
}

static int pt_tiles(int n) { return (int)(((long long)n + SMOE_TPIX - 1) / SMOE_TPIX); }
static int pt_sms() {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

}  // namespace smoe
