// Arguments of the point kernels and the planning pre-pass of the kernel-stationary point sweeps (points.cu:
// smoe_point_backward; gn_diag.cu: smoe_point_gn_diag).
#pragma once
#include "pt_state.cuh"

namespace smoe {

struct PtArgs {
    smoe_cfg cfg;
    const float* packed;
    const int32_t* counts;
    const float* chunk_bounds;
    const float* pts;          // [n][d] in tile order
    float* rout;               // [n][C]
    float* state;              // [ntiles][pt_stride]
    float* tile_box;           // [ntiles][kTB]
    float* xgrad;              // [n][d]
    float* raw_part;           // [num_splits][K_cap][P]
    int32_t* plan_cnt;
    uint32_t* plan_bits;
    int n, ntiles, nwords, K_cap, num_splits, max_list, max_chunks;
    float ltau;
};

// ---- parameter backward: planning pre-pass ---------------------------------------------------------------------
// One CTA per group of kGroup packed kernels: the group's bounding box (as bwd_plan_kernel) against EVERY tile box
// with the exact-zero criterion; one thread per tile, one ballot per 32 tiles, so the tile boxes are read coalesced.
// Same plan layout as smoe_backward: [groups] reachable-tile counts | [groups][nwords] bitmasks.
template <int D, int C>
__global__ void __launch_bounds__(128) point_plan_kernel(const PtArgs a) {
    constexpr int P = nparam(D, C), PK = pstride(D, C);
    __shared__ float sred[4][kCB];
    __shared__ int s_cnt[4];
    const int tid = threadIdx.x, g = blockIdx.x;
    const int K = a.counts[0];
    if (g * kGroup >= K) {
        if (tid == 0) a.plan_cnt[g] = 0;
        return;
    }
    const bool cull = a.cfg.dense_exec == 0;
    float v[kCB];
    {
        const int k = g * kGroup + tid;
        const bool on = tid < kGroup && k < K;
        const float* rec = a.packed + (size_t)(on ? k : 0) * PK;
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            const float m = (l < D && on) ? rec[off_mu(D, C) + l] : 0.f;
            v[l] = (l < D && on) ? m : INFINITY;
            v[3 + l] = (l < D && on) ? -m : INFINITY;
            v[8 + l] = (l < D && on) ? rec[P + 1 + l] : INFINITY;
        }
        v[6] = on ? rec[P] : INFINITY;
        const float c0 = on ? rec[off_pi(D, C)] : -INFINITY;
        v[7] = (c0 == c0) ? -c0 : -INFINITY;          // NaN c0: never cull
        v[11] = 0.f;
#pragma unroll
        for (int q = 0; q < kCB; ++q)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[q] = fminf(v[q], __shfl_xor_sync(0xffffffffu, v[q], o));
        if ((tid & 31) == 0)
#pragma unroll
            for (int q = 0; q < kCB; ++q) sred[tid >> 5][q] = v[q];
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kCB; ++q) v[q] = fminf(fminf(sred[0][q], sred[1][q]), fminf(sred[2][q], sred[3][q]));
    }
    const float blam = v[6], bc0 = -v[7];
    const float zcut_tile = -126.5f;
    uint32_t* bits = a.plan_bits + (size_t)g * a.nwords;
    int n = 0;
    for (int base = 0; base < a.nwords * 32; base += 128) {
        const int t = base + tid;
        bool need = t < a.ntiles;
        if (need && cull && blam >= 0.f) {
            const float* tb = a.tile_box + (size_t)t * kTB;
            float d2 = 0.f, kd = 0.f;
#pragma unroll
            for (int l = 0; l < D; ++l) {
                const float mn = v[l] - tb[l], mx = -v[3 + l] - tb[l];
                const float gap = fmaxf(fmaxf(mn - tb[3 + l], -tb[3 + l] - mx), 0.f);
                d2 = fmaf(gap, gap, d2);
                kd = fmaxf(kd, v[8 + l] * gap * gap);
            }
            const float ub = bc0 - fmaxf(blam * d2, kd) - tb[6];      // tb[6] is NaN for a NaN box: kept
            need = !(ub < zcut_tile);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, need);
        if ((tid & 31) == 0) {
            bits[t >> 5] = bal;
            n += __popc(bal);
        }
    }
    if ((tid & 31) == 0) s_cnt[tid >> 5] = n;
    __syncthreads();
    if (tid == 0) a.plan_cnt[g] = s_cnt[0] + s_cnt[1] + s_cnt[2] + s_cnt[3];
}

}  // namespace smoe
