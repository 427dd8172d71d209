// Planning pre-pass of the kernel-stationary grid sweeps (backward.cu: smoe_backward; gn_diag.cu: smoe_gn_diag) and
// the tile geometry they share.
#pragma once
#include "smoe_common.cuh"

namespace smoe {

struct BwdArgs {
    smoe_cfg cfg;
    smoe_batch b;
    const float* packed;
    const int32_t* counts;
    const float* pix;
    const float* tile_qmin;
    const float* ax[3];
    float* raw_part;
    unsigned long long* pair_counts;
    int32_t* plan_cnt;      // [groups] reachable tiles of each group of kGroup packed kernels
    uint32_t* plan_bits;    // [groups][nwords] bit t: tile t is reachable
    int K_cap, num_splits, ntiles, nt1, nt2, nwords, max_list;
    float tau, ltau;
    float zero_cut;         // gates below 2^zero_cut of the normaliser are skipped: -126 (exactly +0), or -eps_bits
};

// tile geometry (as the forward derives it)
template <int D>
__device__ __forceinline__ void tile_box_of(const BwdArgs& a, int tile, float (&ctr)[3], float (&half)[3]) {
    int tt[3];
    tt[2] = tile % a.nt2;
    tt[1] = (tile / a.nt2) % a.nt1;
    tt[0] = tile / (a.nt2 * a.nt1);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int lo = a.b.origin[i] + tt[i] * a.b.tile[i];
        const int hi = min(lo + a.b.tile[i], a.b.origin[i] + a.b.extent[i]) - 1;
        const float x0 = (i < D) ? a.ax[i][lo] : 0.f, x1 = (i < D) ? a.ax[i][hi] : 0.f;
        ctr[i] = 0.5f * (x0 + x1);
        half[i] = 0.5f * (x1 - x0) * 1.0001f + 1e-7f;
    }
}

// Planning pre-pass: one CTA per group of kGroup consecutive packed kernels.  The group's bounding box (box of
// the centres, smallest eigenvalue / per-axis bounds, largest c0) is tested against every tile of the batch with
// the exact-zero criterion (w = 2^(q - qthr) is exactly 0 when q - min qthr < -126, or below the eps cut); the
// reachable tiles are left as a bitmask.  dense_exec != 0: every tile.
template <int D, int C>
__global__ void __launch_bounds__(128) bwd_plan_kernel(const BwdArgs a) {
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
        __syncthreads();
    }
    const float blam = v[6], bc0 = -v[7];
    const float zcut_tile = a.zero_cut - 0.5f;
    uint32_t* bits = a.plan_bits + (size_t)g * a.nwords;
    extern __shared__ uint32_t s_bits[];                      // [nwords]
    for (int w = tid; w < a.nwords; w += 128) s_bits[w] = (cull && blam >= 0.f) ? 0u : 0xffffffffu;
    __syncthreads();
    int n = 0;
    if (cull && blam >= 0.f) {
        // Conservative tile rectangle: a tile further than r_l = sqrt((c0_max - cut - qthr_min) / kap_l) from the group's
        // box along axis l cannot pass the test below, and qthr >= log2(1e-11) > -36.6 everywhere (smoe.py:821).  Only the
        // tiles inside the rectangle are tested -- a few dozen instead of every tile of the batch.
        int tlo[3] = {0, 0, 0}, tn[3] = {1, 1, 1};
        const int ntile[3] = {(a.ntiles / (a.nt1 * a.nt2)), a.nt1, a.nt2};
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            tn[l] = ntile[l];
            if (l < D) {
                const int o = a.b.origin[l], e = a.b.extent[l];
                const float x0 = a.ax[l][o], dx = e > 1 ? (a.ax[l][o + e - 1] - x0) / (float)(e - 1) : 1.f;
                const float kap = v[8 + l];
                if (kap > 0.f && dx > 0.f) {
                    const float r = sqrtf(fmaxf(bc0 - zcut_tile + 36.6f, 0.f) / kap) * 1.001f + dx;
                    const float plo = (v[l] - r - x0) / dx, phi = (-v[3 + l] + r - x0) / dx;       // pixel range, batch-relative
                    int lo_t = (int)floorf(fmaxf(plo, 0.f)) / a.b.tile[l] - 1;
                    int hi_t = (int)ceilf(fminf(fmaxf(phi, 0.f), (float)(e - 1))) / a.b.tile[l] + 1;
                    lo_t = max(lo_t, 0);
                    hi_t = min(hi_t, ntile[l] - 1);
                    if (!(plo <= (float)e) || !(phi >= 0.f)) hi_t = lo_t - 1;                       // misses the batch
                    tlo[l] = lo_t;
                    tn[l] = max(hi_t - lo_t + 1, 0);
                }
            }
        }
        const int ncand = tn[0] * tn[1] * tn[2];
        for (int it = tid; it < ncand; it += 128) {
            const int c2 = it % tn[2], c1 = (it / tn[2]) % tn[1], c0i = it / (tn[2] * tn[1]);
            const int tile = ((tlo[0] + c0i) * a.nt1 + (tlo[1] + c1)) * a.nt2 + (tlo[2] + c2);
            float ctr[3], half[3];
            tile_box_of<D>(a, tile, ctr, half);
            float d2 = 0.f, kd = 0.f;
#pragma unroll
            for (int l = 0; l < D; ++l) {
                const float mn = v[l] - ctr[l], mx = -v[3 + l] - ctr[l];
                const float gap = fmaxf(fmaxf(mn - half[l], -half[l] - mx), 0.f);
                d2 = fmaf(gap, gap, d2);
                kd = fmaxf(kd, v[8 + l] * gap * gap);
            }
            const float ub = bc0 - fmaxf(blam * d2, kd) - a.tile_qmin[tile];
            if (!(ub < zcut_tile)) atomicOr(&s_bits[tile >> 5], 1u << (tile & 31));
        }
        __syncthreads();
    }
    for (int w = tid; w < a.nwords; w += 128) {
        uint32_t b = s_bits[w];
        const int base = w * 32;
        if (base + 32 > a.ntiles) b &= (base < a.ntiles) ? ((1u << (a.ntiles - base)) - 1u) : 0u;     // no bits beyond the batch
        bits[w] = b;
        n += __popc(b);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_down_sync(0xffffffffu, n, o);
    // fixed-order sum over the 4 warps
    if ((tid & 31) == 0) s_cnt[tid >> 5] = n;
    __syncthreads();
    n = s_cnt[0] + s_cnt[1] + s_cnt[2] + s_cnt[3];
    if (tid == 0) a.plan_cnt[g] = n;
}

}  // namespace smoe
