// SMoE evaluation at arbitrary points, differentiable in the parameters and in the coordinates:
// smoe_point_forward, smoe_point_cotangent, smoe_point_backward, smoe_point_xgrad.
//
// The grid kernels (forward.cu, backward.cu) take their tile geometry from a uniform grid.  Here the caller hands
// over points already in tile order (the Python layer sorts them along a Hilbert curve): a point tile is a run of
// SMOE_TPIX = 512 consecutive points, the last one possibly partial.  Its box (centre and rounded-out half extent
// per axis) is reduced from its points by the forward and kept in `tile_box` for the backward and the coordinate
// gradient; everything that culls -- chunk bounds, per-kernel bounds, the backward's plan -- only needs that box.
//
// Evaluation differs from the grid in one place: the 4 points of a thread share no coordinate, so the logit is the
// full tile-centred quadratic, by Horner  q = qc + sum_l x'_l (ql_l + sum_{m>=l} qq_lm x'_m):  T + d FFMA per
// (point, kernel), 5 for d = 2 and 9 for d = 3 (the grid's parabola costs 2).  Sweeps A and B, their near / far
// split, the half-ulp cut of sweep A, the log-domain tau test and the un-renormalised gates are the grid forward's.
//
// Point state (with grad), per tile: planes [qthr | gr | g_c | x'_l][512] -- qthr = log2 max(S, 1e-11) (+inf on the
// slots past the last point), gr = sum_c g_c r_c (before smoe_point_cotangent: the flag S > 1e-11), g_c = dL/dr_c,
// x'_l the tile-centred coordinates -- and tile_box[tile] = ctr[3] | half[3] | min qthr | 0.
//
// Every mode (cfg.dense_exec 0, 1, 2) returns the same bits: the culling and skip tests only drop terms that are
// exactly zero (or absorbed, sweep A part 2), and every sum runs in a fixed order.  No float atomics anywhere.
// A box with a NaN coordinate culls nothing: its thresholds become -inf (forward) and its min qthr NaN (backward,
// coordinate gradient), and every culling comparison is written as !(bound < threshold).
#include "pt_plan.cuh"

namespace smoe {

constexpr int kPtMaxSplits = 256;

// Box of the CTA's 512 points (first kThreadsF * PPT slots of the tile); x is made tile-centred in place.  `red`
// holds 32 floats.  Returns true when some coordinate is NaN: the centre is then that of the other points (fminf /
// fmaxf skip NaN, so they keep their values) and the half extents are NaN.
template <int D, int PPT>
__device__ __forceinline__ bool tile_box_from_points(float (&x)[PPT][D], unsigned okmask, float* red, float (&ctr)[3],
                                                     float (&half)[3]) {
    const int tid = threadIdx.x;
    float lo[D], nhi[D];
    bool nan = false;
#pragma unroll
    for (int l = 0; l < D; ++l) lo[l] = nhi[l] = INFINITY;
#pragma unroll
    for (int p = 0; p < PPT; ++p)
        if ((okmask >> p) & 1u)
#pragma unroll
            for (int l = 0; l < D; ++l) {
                lo[l] = fminf(lo[l], x[p][l]);
                nhi[l] = fminf(nhi[l], -x[p][l]);
                nan |= x[p][l] != x[p][l];
            }
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[l] = fminf(lo[l], __shfl_xor_sync(0xffffffffu, lo[l], o));
            nhi[l] = fminf(nhi[l], __shfl_xor_sync(0xffffffffu, nhi[l], o));
        }
    if ((tid & 31) == 0)
#pragma unroll
        for (int l = 0; l < D; ++l) {
            red[(tid >> 5) * 8 + l] = lo[l];
            red[(tid >> 5) * 8 + 3 + l] = nhi[l];
        }
    nan = __syncthreads_or(nan);
#pragma unroll
    for (int i = 0; i < 3; ++i) ctr[i] = half[i] = 0.f;
#pragma unroll
    for (int l = 0; l < D; ++l) {
        float a = INFINITY, b = INFINITY;
#pragma unroll
        for (int w = 0; w < kThreadsF / 32; ++w) {
            a = fminf(a, red[w * 8 + l]);
            b = fminf(b, red[w * 8 + 3 + l]);
        }
        const float c0 = a, c1 = -b;
        ctr[l] = 0.5f * (c0 + c1);
        // rounded outwards: the 1e-4 relative term covers the rounding of c1 - c0, the last one that of the centre
        half[l] = 0.5f * (c1 - c0) * 1.0001f + 1e-7f + 2.4e-7f * fmaxf(fabsf(c0), fabsf(c1));
        if (nan) half[l] = NAN;
    }
    __syncthreads();                                     // `red` is reused by the caller
#pragma unroll
    for (int p = 0; p < PPT; ++p)
#pragma unroll
        for (int l = 0; l < D; ++l) x[p][l] = ((okmask >> p) & 1u) ? x[p][l] - ctr[l] : 0.f;
    return nan;
}

// ---- forward: r per point; with `state`, the point state and tile_box ---------------------------------------
template <int D, int C, bool STATE>
__global__ void __launch_bounds__(kThreadsF, (D == 2) ? SMOE_FWD_CTAS_2D : 4) point_forward_kernel(const PtArgs a) {
    using R = Rec<D, C>;
    constexpr int PK = pstride(D, C);
    constexpr int PPT = kPixPerThread;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* raw0 = reinterpret_cast<float*>(smem_raw);
    float* raw1 = raw0 + kChunk * PK;
    float* crec = raw1 + kChunk * PK;
    uint64_t* bar = reinterpret_cast<uint64_t*>(crec + kChunk * R::RC);
    float* red = reinterpret_cast<float*>(bar + 2);          // [4 warps][8]
    int* scratch = reinterpret_cast<int*>(red + 32);         // [2][4]
    int* clist = scratch + 8;                                // [max_chunks]

    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int nchunks = (K + kChunk - 1) / kChunk;
    const int mode = a.cfg.dense_exec;                       // 0 cull+skip, 1 dense, 2 skip only
    const bool cull = mode == 0, skip = mode != 1;
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        fence_barrier_init();
    }
    __syncthreads();
    uint32_t phase0 = 0, phase1 = 0;
    int par = 0;

    auto issue = [&](int ci, int buf) {
        int nk = min(kChunk, K - ci * kChunk);
        uint32_t bytes = (uint32_t)nk * PK * 4u;
        fence_proxy_async();
        mbar_expect_tx(&bar[buf], bytes);
        tma_load_1d(buf ? raw1 : raw0, a.packed + (size_t)ci * kChunk * PK, bytes, &bar[buf]);
    };

    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        // ---- the tile's points (slot j = p * 128 + tid) and their box --------------------------------------------
        float x[PPT][D];
        unsigned okmask = 0;
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int g = tile * SMOE_TPIX + p * kThreadsF + tid;
            const bool ok = g < a.n;
            if (ok) okmask |= 1u << p;
#pragma unroll
            for (int l = 0; l < D; ++l) x[p][l] = ok ? a.pts[(size_t)g * D + l] : 0.f;
        }
        float ctr[3], half[3];
        const bool nanbox = tile_box_from_points<D, PPT>(x, okmask, red, ctr, half);
        auto cut = [&](float thr) { return nanbox ? -INFINITY : thr; };     // a NaN box culls nothing

        // chunk-level culling and the near / far parts of sweep A: csrc/forward.cu, build_chunk_list
        auto build_chunk_list = [&](float thr, int part) -> int {
            int n = 0;
            for (int base = 0; base < nchunks; base += kThreadsF) {
                const int ci = base + tid;
                bool need = false;
                if (ci < nchunks) {
                    const float* cb = a.chunk_bounds + (size_t)ci * kCB;
                    float d2 = 0.f, kd = 0.f;
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float mn = cb[l] - ctr[l], mx = cb[3 + l] - ctr[l];
                        const float gap = fmaxf(fmaxf(mn - half[l], -half[l] - mx), 0.f);
                        d2 = fmaf(gap, gap, d2);
                        kd = fmaxf(kd, cb[8 + l] * gap * gap);
                    }
                    const float lam = cb[6], drop = fmaxf(lam * d2, kd);
                    need = part != 1 || !(lam >= 0.f) || !(drop > kNearCut);
                    if (cull && need) need = !(lam >= 0.f) || !(cb[7] - drop < thr);
                }
                int tot;
                const int pos = cta_compact(need, scratch, par, &tot);
                if (need) clist[n + pos] = ci;
                n += tot;
            }
            __syncthreads();
            return n;
        };

        auto sweep = [&](int nlist, float thr, int part, auto&& body) {
            if (tid == 0 && nlist > 0) {
                issue(clist[0], 0);
                if (nlist > 1) issue(clist[1], 1);
            }
            for (int li = 0; li < nlist; ++li) {
                const int buf = li & 1;
                const int ci = clist[li];
                const int nk = min(kChunk, K - ci * kChunk);
                if (buf) { mbar_wait(&bar[1], phase1); phase1 ^= 1; } else { mbar_wait(&bar[0], phase0); phase0 ^= 1; }
                const float* raw = (buf ? raw1 : raw0) + tid * PK;
                bool need = tid < nk;
                float mu[D];
#pragma unroll
                for (int l = 0; l < D; ++l) mu[l] = need ? raw[off_mu(D, C) + l] - ctr[l] : 0.f;
                if (need && (cull || part != 0)) {
                    float d2 = 0.f, kd = 0.f;
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float gap = fmaxf(fabsf(mu[l]) - half[l], 0.f);
                        d2 = fmaf(gap, gap, d2);
                        kd = fmaxf(kd, raw[nparam(D, C) + 1 + l] * gap * gap);
                    }
                    const float lam = raw[nparam(D, C)], drop = fmaxf(lam * d2, kd);
                    if (part != 0) need = (part == 1) == (!(lam >= 0.f) || !(drop > kNearCut));
                    if (need && cull) need = !(lam >= 0.f) || !(raw[off_pi(D, C)] - drop < thr);
                }
                int nneed;
                const int pos = cta_compact(need, scratch, par, &nneed);
                if (need) transform_record<D, C>(raw, mu, ctr, 0, crec + pos * R::RC);
                __syncthreads();
                if (tid == 0 && li + 2 < nlist) issue(clist[li + 2], buf);
#pragma unroll 2
                for (int kk = 0; kk < nneed; ++kk) body(crec + kk * R::RC);
            }
            __syncthreads();
        };

        // ---- sweep A: normaliser (part 1 near kernels, part 2 the rest against the half-ulp cut) ------------------
        float S[PPT];
#pragma unroll
        for (int p = 0; p < PPT; ++p) S[p] = 0.f;
        const float cutA = -126.5f;
        float skipA = cutA + 0.5f;
        auto bodyA = [&](const float* rec) {
            float f[4 * R::NG4];
            const float4* r4 = reinterpret_cast<const float4*>(rec);
#pragma unroll
            for (int j = 0; j < R::NG4; ++j) {
                float4 v = r4[j];
                f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
            }
            float q[PPT];
            float qmax = -INFINITY;
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                q[p] = point_logit<D, C>(f, x[p]);
                qmax = fmaxf(qmax, q[p]);
            }
            if (__builtin_expect(!skip || __any_sync(0xffffffffu, qmax >= skipA), 0)) {
#pragma unroll
                for (int p = 0; p < PPT; ++p) S[p] += ex2f(q[p]);
            }
        };
        sweep(build_chunk_list(cut(cutA), 1), cut(cutA), 1, bodyA);
        {
            float Lt = INFINITY;
#pragma unroll
            for (int p = 0; p < PPT; ++p)
                if ((okmask >> p) & 1u) Lt = fminf(Lt, log2f(S[p]));
            float Lmin = Lt;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) Lmin = fminf(Lmin, __shfl_xor_sync(0xffffffffu, Lmin, o));
            if ((tid & 31) == 0) red[tid >> 5] = Lmin;
            __syncthreads();
            Lmin = fminf(fminf(red[0], red[1]), fminf(red[2], red[3]));
            __syncthreads();
            float cut2 = cutA;
            if (skip && Lmin == Lmin) {
                cut2 = fmaxf(cutA, Lmin - 25.5f);
                if (Lt == Lt) skipA = fmaxf(skipA, Lt - 25.25f);
            }
            sweep(build_chunk_list(cut(cut2), 2), cut(cut2), 2, bodyA);
        }

        // ---- sweep B: thresholded gates, experts ---------------------------------------------------------------
        float qthr[PPT], r[PPT][C];
        float qmin = INFINITY;
        unsigned live_mask = 0;
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            if (S[p] > kSFloor) live_mask |= 1u << p;
            qthr[p] = ((okmask >> p) & 1u) ? log2f(fmaxf(S[p], kSFloor)) : INFINITY;
            qmin = fminf(qmin, qthr[p]);
#pragma unroll
            for (int c = 0; c < C; ++c) r[p][c] = 0.f;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) qmin = fminf(qmin, __shfl_xor_sync(0xffffffffu, qmin, o));
        if ((tid & 31) == 0) red[tid >> 5] = qmin;
        __syncthreads();
        qmin = fminf(fminf(red[0], red[1]), fminf(red[2], red[3]));
        __syncthreads();
        {
            const float ltau = a.ltau;
            const float thrB = cut(qmin + ltau - 0.01f);
            sweep(build_chunk_list(thrB, 0), thrB, 0, [&](const float* rec) {
                float f[R::RC];
                const float4* r4 = reinterpret_cast<const float4*>(rec);
#pragma unroll
                for (int j = 0; j < R::NG4; ++j) {
                    float4 v = r4[j];
                    f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
                }
                float q[PPT];            // gate logit relative to the point's normaliser: q - log2 S
                bool any = false;
#pragma unroll
                for (int p = 0; p < PPT; ++p) {
                    q[p] = point_logit<D, C>(f, x[p]) - qthr[p];
                    any |= (q[p] > ltau);
                }
                if (__builtin_expect(!skip || __any_sync(0xffffffffu, any), 0)) {
#pragma unroll
                    for (int j = R::NG4; j < (R::OK + 4) / 4; ++j) {
                        float4 v = r4[j];
                        f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
                    }
#pragma unroll
                    for (int p = 0; p < PPT; ++p) {
                        const float w = ex2f(q[p]);
                        const float wm = q[p] > ltau ? w : 0.f;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            // expert E_c(x) = nu'_c + gamma_c . x' (nu' re-centred on the tile)
                            float E = f[R::ONU + c];
#pragma unroll
                            for (int l = 0; l < D; ++l) E = fmaf(f[R::OGA + l * C + c], x[p][l], E);
                            r[p][c] = fmaf(wm, E, r[p][c]);
                        }
                    }
                }
            });
        }

        // ---- epilogue --------------------------------------------------------------------------------------------
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int j = p * kThreadsF + tid;
            const int g = tile * SMOE_TPIX + j;
            const bool ok = (okmask >> p) & 1u;
            if (ok)
#pragma unroll
                for (int c = 0; c < C; ++c) a.rout[(size_t)g * C + c] = r[p][c];
            if (STATE) {
                float* tp = a.state + (size_t)tile * pt_stride(D, C);
                tp[PP_QTHR * SMOE_TPIX + j] = qthr[p];                          // +inf past the last point: w = 0
                tp[PP_GR * SMOE_TPIX + j] = (ok && ((live_mask >> p) & 1u)) ? 1.f : 0.f;
#pragma unroll
                for (int l = 0; l < D; ++l) tp[(pp_x(C) + l) * SMOE_TPIX + j] = x[p][l];
            }
        }
        if (STATE && tid == 0) {
            float4* tb = reinterpret_cast<float4*>(a.tile_box + (size_t)tile * kTB);
            tb[0] = make_float4(ctr[0], ctr[1], ctr[2], half[0]);
            tb[1] = make_float4(half[1], half[2], nanbox ? NAN : qmin, 0.f);
        }
    }
}

// ---- cotangent: dL/dr into the point state ---------------------------------------------------------------------
// g_c = grad_r (0 past the last point) and gr = sum_c g_c r_c (fmaf in channel order from 0, as loss_kernel) where
// S > 1e-11, else 0.  One thread per slot; elementwise, no reduction.
template <int C>
__global__ void __launch_bounds__(256) point_cotangent_kernel(const float* __restrict__ rbuf,
                                                              const float* __restrict__ grad_r, float* __restrict__ state,
                                                              int n, int nslots, int stride) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= nslots) return;
    float* tp = state + (size_t)(i / SMOE_TPIX) * stride;
    const int j = i % SMOE_TPIX;
    float g[C], gr = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) g[c] = 0.f;
    if (i < n) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
            g[c] = grad_r[(size_t)i * C + c];
            gr = fmaf(g[c], rbuf[(size_t)i * C + c], gr);
        }
    }
    const bool live = tp[PP_GR * SMOE_TPIX + j] != 0.f;
    tp[PP_GR * SMOE_TPIX + j] = live ? gr : 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) tp[(PP_G + c) * SMOE_TPIX + j] = g[c];
}

// ---- parameter backward: kernel-stationary sweep ---------------------------------------------------------------
// The CTA shape, thread <-> kernel mapping (kHalves lanes per kernel, alternate groups of 4 points), tile splits and
// the buffer hand-over of backward_kernel; the statistics are accumulated per point instead of per row and folded
// into kernel-centred moments at the end of each tile, into the raw_part layout smoe_grad_finalize reads.
template <int D, int C, bool DENSE>
__global__ void __launch_bounds__(kThreads, 512 / kThreads) point_backward_kernel(const PtArgs a) {
    using R = Rec<D, C>;
    constexpr int T = tri(D);
    constexpr int P = nparam(D, C), PK = pstride(D, C);
    constexpr int GRP = 4;
    constexpr int tstride = pt_stride(D, C);
    constexpr uint32_t kTileBytes = (uint32_t)tstride * 4u;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* buf0 = reinterpret_cast<float*>(smem_raw);
    float* buf1 = buf0 + tstride;
    uint64_t* bar = reinterpret_cast<uint64_t*>(buf1 + tstride);
    int* scratch = reinterpret_cast<int*>(bar + 2);                 // [16]
    int* tlist = scratch + 16;                                      // [max_list]

    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int k = blockIdx.x * kGroup + tid / kHalves;
    const int hsel = tid % kHalves;
    if ((int)blockIdx.x * kGroup >= K) return;
    if (a.plan_cnt[blockIdx.x] == 0) return;
    const bool active = k < K;
    const int split = blockIdx.y;
    const float zcut = -126.f, zcut_tile = -126.5f;
    const bool cull = !DENSE && a.cfg.dense_exec == 0;
    constexpr bool skip = !DENSE;
    const float ltau = a.ltau;

    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        fence_barrier_init();
    }
    __syncthreads();
    uint32_t phase0 = 0, phase1 = 0;
    auto issue = [&](int tile, int buf) {
        fence_proxy_async();
        mbar_expect_tx(&bar[buf], kTileBytes);
        tma_load_1d(buf ? buf1 : buf0, a.state + (size_t)tile * tstride, kTileBytes, &bar[buf]);
    };
    const float* rec = a.packed + (size_t)(active ? k : 0) * PK;

    int nlist = 0;
    {
        const uint32_t* bits = a.plan_bits + (size_t)blockIdx.x * a.nwords;
        const int my_tiles = (a.ntiles - split + a.num_splits - 1) / a.num_splits;
        for (int base = 0; base < my_tiles; base += kThreads) {
            const int it = base + tid;
            const int tile = split + it * a.num_splits;
            const bool need = it < my_tiles && ((bits[tile >> 5] >> (tile & 31)) & 1u);
            const unsigned bal = __ballot_sync(0xffffffffu, need);
            const int lane = tid & 31, w = tid >> 5;
            if (lane == 0) scratch[w] = __popc(bal);
            __syncthreads();
            int off = 0, tot = 0;
#pragma unroll
            for (int j = 0; j < kThreads / 32; ++j) {
                const int cnt = scratch[j];
                off += (j < w) ? cnt : 0;
                tot += cnt;
            }
            if (need) tlist[nlist + off + __popc(bal & ((1u << lane) - 1u))] = tile;
            nlist += tot;
            __syncthreads();
        }
    }

    float G0 = 0.f, G1[D], G2[T], GNu[C], GGa[D][C];
#pragma unroll
    for (int l = 0; l < D; ++l) G1[l] = 0.f;
#pragma unroll
    for (int q = 0; q < T; ++q) G2[q] = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        GNu[c] = 0.f;
#pragma unroll
        for (int l = 0; l < D; ++l) GGa[l][c] = 0.f;
    }

    int* done = scratch + 8;
    if (tid == 0) {
        done[0] = done[1] = 0;
        if (nlist > 0) issue(tlist[0], 0);
        if (nlist > 1) issue(tlist[1], 1);
    }
    __syncthreads();
    for (int li = 0; li < nlist; ++li) {
        const int buf = li & 1;
        const int tile = tlist[li];
        const float* tb = a.tile_box + (size_t)tile * kTB;
        float ctr[3], half[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) { ctr[i] = tb[i]; half[i] = tb[3 + i]; }
        float mup[D];
#pragma unroll
        for (int l = 0; l < D; ++l) mup[l] = __ldg(rec + off_mu(D, C) + l) - ctr[l];
        const float c0 = active ? __ldg(rec + off_pi(D, C)) : -INFINITY;
        bool need = active;
        if (cull && need) {
            const float lam = __ldg(rec + P);
            float d2 = 0.f, kd = 0.f;
#pragma unroll
            for (int l = 0; l < D; ++l) {
                const float gap = fmaxf(fabsf(mup[l]) - half[l], 0.f);
                d2 = fmaf(gap, gap, d2);
                kd = fmaxf(kd, __ldg(rec + P + 1 + l) * gap * gap);
            }
            const float ub = c0 - fmaxf(lam * d2, kd) - tb[6];
            need = !(lam >= 0.f) || !(ub < zcut_tile);
        }
        const bool warp_need = __any_sync(0xffffffffu, need);

        if (buf) { mbar_wait(&bar[1], phase1); phase1 ^= 1; } else { mbar_wait(&bar[0], phase0); phase0 ^= 1; }
        if (warp_need) {
            float f[R::GN + R::EN];
            {
                float Qm[D][D];
#pragma unroll
                for (int l = 0; l < D; ++l)
#pragma unroll
                    for (int m = l; m < D; ++m) Qm[l][m] = Qm[m][l] = __ldg(rec + off_A(D, C) + ut(D, l, m));
                float v[D];
                float qc = c0;
#pragma unroll
                for (int l = 0; l < D; ++l) {
                    v[l] = 0.f;
#pragma unroll
                    for (int m = 0; m < D; ++m) v[l] = fmaf(Qm[l][m], mup[m], v[l]);
                }
#pragma unroll
                for (int l = 0; l < D; ++l) qc = fmaf(-mup[l], v[l], qc);
#pragma unroll
                for (int l = 0; l < D; ++l) {
                    f[R::OL + l] = 2.f * v[l];
#pragma unroll
                    for (int m = l; m < D; ++m) f[R::OQ + ut(D, l, m)] = (l == m) ? -Qm[l][m] : -2.f * Qm[l][m];
                }
                f[R::OC] = qc;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    float nn = __ldg(rec + off_nu(D, C) + c);
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float gg = __ldg(rec + off_ga(D, C) + l * C + c);
                        nn = fmaf(gg, ctr[l], nn);
                        f[R::OGA + l * C + c] = gg;
                    }
                    f[R::ONU + c] = nn;
                }
            }
            float M0 = 0.f, M1[D], M2[T], N0[C], N1[D][C];
#pragma unroll
            for (int l = 0; l < D; ++l) M1[l] = 0.f;
#pragma unroll
            for (int q = 0; q < T; ++q) M2[q] = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                N0[c] = 0.f;
#pragma unroll
                for (int l = 0; l < D; ++l) N1[l][c] = 0.f;
            }
            const float* pl = buf ? buf1 : buf0;
            auto moments = [&](float t, const float (&xp)[D]) {
                M0 += t;
#pragma unroll
                for (int l = 0; l < D; ++l) {
                    const float tx = t * xp[l];
                    M1[l] += tx;
#pragma unroll
                    for (int m = l; m < D; ++m) M2[ut(D, l, m)] = fmaf(tx, xp[m], M2[ut(D, l, m)]);
                }
            };
            for (int gi = hsel; gi < SMOE_TPIX / GRP; gi += kHalves) {
                const int j0 = gi * GRP;
                float xg[GRP][D], dq[GRP];
                {
                    const float4 tv = *reinterpret_cast<const float4*>(pl + PP_QTHR * SMOE_TPIX + j0);
                    const float t4[GRP] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float4 xv = *reinterpret_cast<const float4*>(pl + (pp_x(C) + l) * SMOE_TPIX + j0);
                        xg[0][l] = xv.x; xg[1][l] = xv.y; xg[2][l] = xv.z; xg[3][l] = xv.w;
                    }
#pragma unroll
                    for (int u = 0; u < GRP; ++u) dq[u] = point_logit<D, C>(f, xg[u]) - t4[u];
                }
                float dmax = -INFINITY;
#pragma unroll
                for (int u = 0; u < GRP; ++u) dmax = fmaxf(dmax, dq[u]);
                const bool any_gate = !skip || __any_sync(0xffffffffu, dmax >= zcut);
                const bool any_pass = !skip || __any_sync(0xffffffffu, dmax > ltau);
                if (!any_gate) continue;
                const float4 gv = *reinterpret_cast<const float4*>(pl + PP_GR * SMOE_TPIX + j0);
                const float gr4[GRP] = {gv.x, gv.y, gv.z, gv.w};
                if (!any_pass) {
#pragma unroll
                    for (int u = 0; u < GRP; ++u) moments(-ex2f(dq[u]) * gr4[u], xg[u]);
                } else {
                    float g4[C][GRP];
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const float4 cv = *reinterpret_cast<const float4*>(pl + (PP_G + c) * SMOE_TPIX + j0);
                        g4[c][0] = cv.x; g4[c][1] = cv.y; g4[c][2] = cv.z; g4[c][3] = cv.w;
                    }
#pragma unroll
                    for (int u = 0; u < GRP; ++u) {
                        const float w = ex2f(dq[u]);
                        const float wm = dq[u] > ltau ? w : 0.f;     // w > tau; 0 * g is exact, as in backward_kernel
                        float gE = 0.f;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            float E = f[R::ONU + c];
#pragma unroll
                            for (int l = 0; l < D; ++l) E = fmaf(f[R::OGA + l * C + c], xg[u][l], E);
                            gE = fmaf(g4[c][u], E, gE);
                            const float vc = wm * g4[c][u];
                            N0[c] += vc;
#pragma unroll
                            for (int l = 0; l < D; ++l) N1[l][c] = fmaf(vc, xg[u][l], N1[l][c]);
                        }
                        moments(fmaf(wm, gE, -w * gr4[u]), xg[u]);
                    }
                }
            }
            // fold tile-centred statistics into kernel-centred ones (as backward_kernel)
            G0 += M0;
#pragma unroll
            for (int l = 0; l < D; ++l) G1[l] += fmaf(-mup[l], M0, M1[l]);
#pragma unroll
            for (int l = 0; l < D; ++l)
#pragma unroll
                for (int m = l; m < D; ++m) {
                    float dd = M2[ut(D, l, m)];
                    dd = fmaf(-mup[l], M1[m], dd);
                    dd = fmaf(-mup[m], M1[l], dd);
                    dd = fmaf(mup[l] * mup[m], M0, dd);
                    G2[ut(D, l, m)] += dd;
                }
#pragma unroll
            for (int c = 0; c < C; ++c) {
                GNu[c] += N0[c];
#pragma unroll
                for (int l = 0; l < D; ++l) GGa[l][c] += fmaf(ctr[l], N0[c], N1[l][c]);
            }
        }
        __syncwarp();
        if ((tid & 31) == 0) {
            __threadfence_block();
            const int old = atomicAdd(&done[buf], 1);
            if (old == kThreads / 32 - 1) {
                done[buf] = 0;
                __threadfence_block();
                if (li + 2 < nlist) issue(tlist[li + 2], buf);
            }
        }
    }

    {
        auto pair_sum = [&](float& v) {
#pragma unroll
            for (int o = 1; o < kHalves; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        };
        pair_sum(G0);
#pragma unroll
        for (int l = 0; l < D; ++l) pair_sum(G1[l]);
#pragma unroll
        for (int q = 0; q < T; ++q) pair_sum(G2[q]);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            pair_sum(GNu[c]);
#pragma unroll
            for (int l = 0; l < D; ++l) pair_sum(GGa[l][c]);
        }
    }
    if (active && hsel == 0) {
        float* out = a.raw_part + ((size_t)split * a.K_cap + k) * P;
#pragma unroll
        for (int l = 0; l < D; ++l) out[off_mu(D, C) + l] = G1[l];
#pragma unroll
        for (int q = 0; q < T; ++q) out[off_A(D, C) + q] = G2[q];
        out[off_pi(D, C)] = G0;
#pragma unroll
        for (int c = 0; c < C; ++c) out[off_nu(D, C) + c] = GNu[c];
#pragma unroll
        for (int l = 0; l < D; ++l)
#pragma unroll
            for (int c = 0; c < C; ++c) out[off_ga(D, C) + l * C + c] = GGa[l][c];
    }
}

// ---- coordinate gradient ---------------------------------------------------------------------------------------
// Pixel-stationary, the chunk staging of the forward.  With t_k = w_k (m_k gE_k - gr) (the backward's t):
//     dL/dx = sum_k [ m_k w_k sum_c g_c gamma_k[:, c] + t_k ln2 grad_x q_k(x) ]
// (the second term is d(w_k)/dx summed against m_k gE_k, through the normaliser too).  A kernel with
// q - qthr < -126 contributes exactly 0 (ex2.approx.ftz), so chunks and kernels are culled against min qthr - 126.5
// and a warp skips a kernel whose gates are all below -126 -- not tau: sub-threshold kernels still enter through
// the normaliser.  One accumulator per (point, axis), kernels added in packed order in every mode.
template <int D, int C>
__global__ void __launch_bounds__(kThreadsF, 4) point_xgrad_kernel(const PtArgs a) {
    using R = Rec<D, C>;
    constexpr int PK = pstride(D, C);
    constexpr int PPT = kPixPerThread;
    constexpr int tstride = pt_stride(D, C);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* raw0 = reinterpret_cast<float*>(smem_raw);
    float* raw1 = raw0 + kChunk * PK;
    float* crec = raw1 + kChunk * PK;
    uint64_t* bar = reinterpret_cast<uint64_t*>(crec + kChunk * R::RC);
    float* red = reinterpret_cast<float*>(bar + 2);
    int* scratch = reinterpret_cast<int*>(red + 32);
    int* clist = scratch + 8;

    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int nchunks = (K + kChunk - 1) / kChunk;
    const int mode = a.cfg.dense_exec;
    const bool cull = mode == 0, skip = mode != 1;
    const float ltau = a.ltau;
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        fence_barrier_init();
    }
    __syncthreads();
    uint32_t phase0 = 0, phase1 = 0;
    int par = 0;
    auto issue = [&](int ci, int buf) {
        int nk = min(kChunk, K - ci * kChunk);
        uint32_t bytes = (uint32_t)nk * PK * 4u;
        fence_proxy_async();
        mbar_expect_tx(&bar[buf], bytes);
        tma_load_1d(buf ? raw1 : raw0, a.packed + (size_t)ci * kChunk * PK, bytes, &bar[buf]);
    };

    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        const float* tb = a.tile_box + (size_t)tile * kTB;
        float ctr[3], half[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) { ctr[i] = tb[i]; half[i] = tb[3 + i]; }
        const float thr = tb[6] - 126.5f;                     // NaN for a NaN box: nothing is culled
        const float* tp = a.state + (size_t)tile * tstride;
        float x[PPT][D], qthr[PPT], gr[PPT], g[PPT][C], dx[PPT][D];
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int j = p * kThreadsF + tid;
            qthr[p] = tp[PP_QTHR * SMOE_TPIX + j];
            gr[p] = tp[PP_GR * SMOE_TPIX + j];
#pragma unroll
            for (int c = 0; c < C; ++c) g[p][c] = tp[(PP_G + c) * SMOE_TPIX + j];
#pragma unroll
            for (int l = 0; l < D; ++l) {
                x[p][l] = tp[(pp_x(C) + l) * SMOE_TPIX + j];
                dx[p][l] = 0.f;
            }
        }

        int nlist = 0;
        for (int base = 0; base < nchunks; base += kThreadsF) {
            const int ci = base + tid;
            bool need = ci < nchunks;
            if (need && cull) {
                const float* cb = a.chunk_bounds + (size_t)ci * kCB;
                float d2 = 0.f, kd = 0.f;
#pragma unroll
                for (int l = 0; l < D; ++l) {
                    const float mn = cb[l] - ctr[l], mx = cb[3 + l] - ctr[l];
                    const float gap = fmaxf(fmaxf(mn - half[l], -half[l] - mx), 0.f);
                    d2 = fmaf(gap, gap, d2);
                    kd = fmaxf(kd, cb[8 + l] * gap * gap);
                }
                const float lam = cb[6];
                need = !(lam >= 0.f) || !(cb[7] - fmaxf(lam * d2, kd) < thr);
            }
            int tot;
            const int pos = cta_compact(need, scratch, par, &tot);
            if (need) clist[nlist + pos] = ci;
            nlist += tot;
        }
        __syncthreads();

        if (tid == 0 && nlist > 0) {
            issue(clist[0], 0);
            if (nlist > 1) issue(clist[1], 1);
        }
        for (int li = 0; li < nlist; ++li) {
            const int buf = li & 1;
            const int ci = clist[li];
            const int nk = min(kChunk, K - ci * kChunk);
            if (buf) { mbar_wait(&bar[1], phase1); phase1 ^= 1; } else { mbar_wait(&bar[0], phase0); phase0 ^= 1; }
            const float* raw = (buf ? raw1 : raw0) + tid * PK;
            bool need = tid < nk;
            float mu[D];
#pragma unroll
            for (int l = 0; l < D; ++l) mu[l] = need ? raw[off_mu(D, C) + l] - ctr[l] : 0.f;
            if (need && cull) {
                float d2 = 0.f, kd = 0.f;
#pragma unroll
                for (int l = 0; l < D; ++l) {
                    const float gap = fmaxf(fabsf(mu[l]) - half[l], 0.f);
                    d2 = fmaf(gap, gap, d2);
                    kd = fmaxf(kd, raw[nparam(D, C) + 1 + l] * gap * gap);
                }
                const float lam = raw[nparam(D, C)];
                need = !(lam >= 0.f) || !(raw[off_pi(D, C)] - fmaxf(lam * d2, kd) < thr);
            }
            int nneed;
            const int pos = cta_compact(need, scratch, par, &nneed);
            if (need) transform_record<D, C>(raw, mu, ctr, 0, crec + pos * R::RC);
            __syncthreads();
            if (tid == 0 && li + 2 < nlist) issue(clist[li + 2], buf);
            for (int kk = 0; kk < nneed; ++kk) {
                const float* rc = crec + kk * R::RC;
                float f[R::RC];
                const float4* r4 = reinterpret_cast<const float4*>(rc);
#pragma unroll
                for (int j = 0; j < R::NG4; ++j) {
                    float4 v = r4[j];
                    f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
                }
                float dq[PPT];
                float dmax = -INFINITY;
#pragma unroll
                for (int p = 0; p < PPT; ++p) {
                    dq[p] = point_logit<D, C>(f, x[p]) - qthr[p];
                    dmax = fmaxf(dmax, dq[p]);
                }
                if (skip && !__any_sync(0xffffffffu, dmax >= -126.f)) continue;
#pragma unroll
                for (int j = R::NG4; j < (R::OK + 4) / 4; ++j) {
                    float4 v = r4[j];
                    f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
                }
#pragma unroll
                for (int p = 0; p < PPT; ++p) {
                    const float w = ex2f(dq[p]);
                    const float wm = dq[p] > ltau ? w : 0.f;
                    float gE = 0.f, gg[D];
#pragma unroll
                    for (int l = 0; l < D; ++l) gg[l] = 0.f;
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        float E = f[R::ONU + c];
#pragma unroll
                        for (int l = 0; l < D; ++l) {
                            E = fmaf(f[R::OGA + l * C + c], x[p][l], E);
                            gg[l] = fmaf(g[p][c], f[R::OGA + l * C + c], gg[l]);
                        }
                        gE = fmaf(g[p][c], E, gE);
                    }
                    const float tl = fmaf(wm, gE, -w * gr[p]) * kLn2;
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        // d q / d x'_l = ql_l + 2 qq_ll x'_l + sum_{m != l} qq_lm x'_m (off-diagonals stored doubled)
                        float gq = fmaf(2.f * f[R::OQ + ut(D, l, l)], x[p][l], f[R::OL + l]);
#pragma unroll
                        for (int m = 0; m < D; ++m)
                            if (m != l) gq = fmaf(f[R::OQ + (m > l ? ut(D, l, m) : ut(D, m, l))], x[p][m], gq);
                        dx[p][l] += fmaf(tl, gq, wm * gg[l]);
                    }
                }
            }
        }
        __syncthreads();          // the next tile rebuilds `clist` and re-uses `crec`
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int gi = tile * SMOE_TPIX + p * kThreadsF + tid;
            if (gi < a.n)
#pragma unroll
                for (int l = 0; l < D; ++l) a.xgrad[(size_t)gi * D + l] = dx[p][l];
        }
    }
}

static int pt_nwords(int ntiles) { return (ntiles + 127) / 128 * 4; }

}  // namespace smoe

using namespace smoe;

extern "C" {

int smoe_point_tiles(int n_points) { return n_points > 0 ? pt_tiles(n_points) : 0; }

int smoe_point_stride(int d, int C) { return pt_stride(d, C); }

size_t smoe_point_plan_bytes(int K_cap, int n_points) {
    const size_t groups = (size_t)(K_cap + kGroup - 1) / kGroup;
    return (groups + groups * (size_t)pt_nwords(pt_tiles(n_points))) * sizeof(int32_t);
}

int smoe_point_splits(int K_cap, int n_points) {
    // a few waves of 8 backward CTAs per SM of a B200 (148 SMs), at most kPtMaxSplits slabs for smoe_grad_finalize to
    // add, and at least enough splits to keep a split's tile list within 32 KB of shared memory.  N and K only.
    const int ntiles = pt_tiles(n_points > 0 ? n_points : 1);
    const int groups = ((K_cap > 64 ? K_cap : 64) + kGroup - 1) / kGroup;
    int s = (4 * 148 * 8 + groups - 1) / groups;
    if (s > kPtMaxSplits) s = kPtMaxSplits;
    const int need = (ntiles + 8191) / 8192;
    if (s < need) s = need;
    if (s > ntiles) s = ntiles;
    return s < 1 ? 1 : s;
}

int smoe_point_forward(const smoe_cfg* cfg, const float* packed, const int32_t* counts, const float* chunk_bounds,
                       int K_cap, const float* points, int n_points, float* r, float* state, float* tile_box,
                       void* stream) {
    SMOE_REQUIRE(cfg && packed && counts && chunk_bounds && points && r, "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    SMOE_REQUIRE(!state == !tile_box, "state and tile_box go together");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the point kernels");
    PtArgs a = {};
    a.cfg = *cfg;
    a.packed = packed; a.counts = counts; a.chunk_bounds = chunk_bounds;
    a.pts = points; a.rout = r; a.state = state; a.tile_box = tile_box;
    a.n = n_points;
    a.ntiles = pt_tiles(n_points);
    a.max_chunks = (K_cap + kChunk - 1) / kChunk;
    a.ltau = -(float)(cfg->precision + 1);
    const int per_sm = cfg->d == 2 ? SMOE_FWD_CTAS_2D : 4;
    const int cap = per_sm * pt_sms();
    const int grid = a.ntiles < cap ? a.ntiles : cap;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(D, C, ST)                                                                                             \
    {                                                                                                                \
        size_t sm = pt_sweep_smem_bytes<D, C>(a.max_chunks);                                                         \
        SMOE_REQUIRE(sm <= 200 * 1024, "too many kernel chunks for the shared-memory chunk list");                   \
        cudaFuncSetAttribute(point_forward_kernel<D, C, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);  \
        point_forward_kernel<D, C, ST><<<grid, kThreadsF, sm, st>>>(a);                                              \
    }
#define CALL(D, C) if (state) LAUNCH(D, C, true) else LAUNCH(D, C, false)
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
#undef LAUNCH
    return check_launch("smoe_point_forward");
}

int smoe_point_cotangent(const smoe_cfg* cfg, int n_points, const float* r, const float* grad_r, float* state,
                         void* stream) {
    SMOE_REQUIRE(cfg && r && grad_r && state, "null argument");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    const int nslots = pt_tiles(n_points) * SMOE_TPIX;
    const int stride = pt_stride(cfg->d, cfg->C);
    const int nb = (nslots + 255) / 256;
    cudaStream_t st = (cudaStream_t)stream;
    if (cfg->C == 1) point_cotangent_kernel<1><<<nb, 256, 0, st>>>(r, grad_r, state, n_points, nslots, stride);
    else point_cotangent_kernel<3><<<nb, 256, 0, st>>>(r, grad_r, state, n_points, nslots, stride);
    return check_launch("smoe_point_cotangent");
}

int smoe_point_backward(const smoe_cfg* cfg, const float* packed, const int32_t* counts, int K_cap, int n_points,
                        const float* state, const float* tile_box, int num_splits, float* raw_part, int32_t* plan,
                        void* stream) {
    SMOE_REQUIRE(cfg && packed && counts && state && tile_box && raw_part && plan, "null argument");
    SMOE_REQUIRE(K_cap > 0 && num_splits > 0 && num_splits <= 65535, "bad K_cap / num_splits");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the point kernels");
    PtArgs a = {};
    a.cfg = *cfg;
    a.packed = packed; a.counts = counts; a.state = const_cast<float*>(state);
    a.tile_box = const_cast<float*>(tile_box);
    a.raw_part = raw_part;
    a.n = n_points;
    a.ntiles = pt_tiles(n_points);
    a.nwords = pt_nwords(a.ntiles);
    a.K_cap = K_cap;
    a.num_splits = num_splits;
    a.max_list = (a.ntiles + num_splits - 1) / num_splits;
    a.ltau = -(float)(cfg->precision + 1);
    const int groups = (K_cap + kGroup - 1) / kGroup;
    a.plan_cnt = plan;
    a.plan_bits = reinterpret_cast<uint32_t*>(plan + groups);
    const dim3 grid(groups, num_splits);
    const size_t sm = 2 * (size_t)pt_stride(cfg->d, cfg->C) * 4 + 16 + 16 * 4 + (size_t)a.max_list * 4 + 64;
    SMOE_REQUIRE(sm <= 100 * 1024, "too many tiles per split for the shared-memory tile list: raise num_splits");
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(D, C, DN)                                                                                             \
    {                                                                                                                \
        point_plan_kernel<D, C><<<groups, 128, 0, st>>>(a);                                                          \
        cudaFuncSetAttribute(point_backward_kernel<D, C, DN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        point_backward_kernel<D, C, DN><<<grid, kThreads, sm, st>>>(a);                                              \
    }
#define CALL(D, C) if (cfg->dense_exec == 1) LAUNCH(D, C, true) else LAUNCH(D, C, false)
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
#undef LAUNCH
    return check_launch("smoe_point_backward");
}

int smoe_point_xgrad(const smoe_cfg* cfg, const float* packed, const int32_t* counts, const float* chunk_bounds,
                     int K_cap, int n_points, const float* state, const float* tile_box, float* grad_points,
                     void* stream) {
    SMOE_REQUIRE(cfg && packed && counts && chunk_bounds && state && tile_box && grad_points, "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the point kernels");
    PtArgs a = {};
    a.cfg = *cfg;
    a.packed = packed; a.counts = counts; a.chunk_bounds = chunk_bounds;
    a.state = const_cast<float*>(state);
    a.tile_box = const_cast<float*>(tile_box);
    a.xgrad = grad_points;
    a.n = n_points;
    a.ntiles = pt_tiles(n_points);
    a.max_chunks = (K_cap + kChunk - 1) / kChunk;
    a.ltau = -(float)(cfg->precision + 1);
    const int cap = 4 * pt_sms();
    const int grid = a.ntiles < cap ? a.ntiles : cap;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C)                                                                                              \
    {                                                                                                           \
        size_t sm = pt_sweep_smem_bytes<D, C>(a.max_chunks);                                                    \
        SMOE_REQUIRE(sm <= 200 * 1024, "too many kernel chunks for the shared-memory chunk list");              \
        cudaFuncSetAttribute(point_xgrad_kernel<D, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);   \
        point_xgrad_kernel<D, C><<<grid, kThreadsF, sm, st>>>(a);                                               \
    }
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_point_xgrad");
}

}  // extern "C"
