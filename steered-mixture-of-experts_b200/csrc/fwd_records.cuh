// Kernel records of the pixel-stationary sweeps (smoe_forward, smoe_point_forward, smoe_point_xgrad): the packed
// record re-expressed in tile-centred coordinates, the ordered CTA compaction and the near / far rule of sweep A.
#pragma once
#include "smoe_common.cuh"

namespace smoe {

template <int D, int C>
struct Rec {
    static constexpr int T = tri(D);
    static constexpr int GN = T + D + 1;          // qq (upper-tri, off-diagonals doubled) | ql | qc
    static constexpr int EN = C + D * C;          // nu' | gamma
    static constexpr int RC0 = (GN + EN + 1 + 3) / 4 * 4;  // + the kernel's ORIGINAL index
    // an ODD number of float4 per record: the 8 threads of a quarter-warp then store their records' float4 to 8
    // different 16-byte bank groups (stride 80 / 48 / 112 B), so the per-thread record writes are conflict-free
    static constexpr int RC = (RC0 / 4) % 2 == 0 ? RC0 + 4 : RC0;
    static constexpr int NG4 = (GN + 3) / 4;      // float4 loads that cover the geometry part
    static constexpr int OQ = 0, OL = T, OC = T + D, ONU = GN, OGA = GN + C, OK = GN + EN;
};

// raw packed record + tile centre -> tile-centred compute record
template <int D, int C>
__device__ __forceinline__ void transform_record(const float* __restrict__ raw, const float (&mu)[D],
                                                 const float (&ctr)[3], int korig, float* __restrict__ dst) {
    using R = Rec<D, C>;
    float out[R::RC];
    float Qm[D][D], v[D];
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
        for (int m = l; m < D; ++m) Qm[l][m] = Qm[m][l] = raw[off_A(D, C) + ut(D, l, m)];
    float qc = raw[off_pi(D, C)];
#pragma unroll
    for (int l = 0; l < D; ++l) {
        v[l] = 0.f;
#pragma unroll
        for (int m = 0; m < D; ++m) v[l] = fmaf(Qm[l][m], mu[m], v[l]);
    }
#pragma unroll
    for (int l = 0; l < D; ++l) qc = fmaf(-mu[l], v[l], qc);
#pragma unroll
    for (int l = 0; l < D; ++l) {
        out[R::OL + l] = 2.f * v[l];
#pragma unroll
        for (int m = l; m < D; ++m) out[R::OQ + ut(D, l, m)] = (l == m) ? -Qm[l][m] : -2.f * Qm[l][m];
    }
    out[R::OC] = qc;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        float nu = raw[off_nu(D, C) + c];
#pragma unroll
        for (int l = 0; l < D; ++l) {
            float g = raw[off_ga(D, C) + l * C + c];
            nu = fmaf(g, ctr[l], nu);
            out[R::OGA + l * C + c] = g;
        }
        out[R::ONU + c] = nu;
    }
    out[R::OK] = __int_as_float(korig);
#pragma unroll
    for (int j = R::OK + 1; j < R::RC; ++j) out[j] = 0.f;
    float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int j = 0; j < R::RC / 4; ++j) d4[j] = make_float4(out[4 * j], out[4 * j + 1], out[4 * j + 2], out[4 * j + 3]);
}

// Ordered compaction helper for a 128-thread CTA: returns this thread's output slot (valid when flag) and the
// total through *total.  `scratch` holds 2 x 4 ints used alternately (`par` flips on every call), so ONE
// __syncthreads per call is enough: a thread can reach the call after next -- and overwrite this half -- only
// after every thread has passed the next call's barrier, i.e. has finished reading this half.
__device__ __forceinline__ int cta_compact(bool flag, int* scratch, int& par, int* total) {
    const unsigned bal = __ballot_sync(0xffffffffu, flag);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int* sc = scratch + 4 * par;
    par ^= 1;
    if (lane == 0) sc[w] = __popc(bal);
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int j = 0; j < kThreadsF / 32; ++j) {
        const int cnt = sc[j];
        off += (j < w) ? cnt : 0;
        tot += cnt;
    }
    *total = tot;
    return off + __popc(bal & ((1u << lane) - 1u));
}

// resident CTAs per SM of the d = 2 pixel-stationary sweeps (their __launch_bounds__); 4 for d = 3
#ifndef SMOE_FWD_CTAS_2D
#define SMOE_FWD_CTAS_2D 6
#endif
#ifndef SMOE_FWD_NEARCUT
#define SMOE_FWD_NEARCUT 8.0f
#endif
constexpr float kNearCut = SMOE_FWD_NEARCUT;      // sweep A, part 1: see build_chunk_list

}  // namespace smoe
