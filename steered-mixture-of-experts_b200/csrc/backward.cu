// Fused SMoE backward (smoe_backward, smoe_reduce_splits, smoe_grad_finalize, smoe_adam_step).
// Replaces tf.gradients(loss_op, variables) + assign_add + ApplyAdam (smoe.py:1148-1150, 1173-1193).
//
// Kernel-stationary: a thread owns ONE kernel (its record and 2*P accumulators live in
// registers), a CTA owns 64 consecutive packed kernels -- spatial neighbours, because smoe_pack
// writes the records in Hilbert order of their centres -- and a 1/num_splits share of the pixel tiles
// (split s owns tiles s, s+NS, ...: a geometry-fixed rule, so the partial sums group the same way in
// every execution mode).  Which of its tiles a CTA must visit comes from a planning pre-pass
// (bwd_plan_kernel: one CTA per group tests every tile of the batch against the group's bounding box and
// leaves a bitmask), so a CTA spends no time on geometry, and the CTAs of a group that cannot reach the
// batch at all -- most groups, when the batch is one rank's pixel block -- leave after one load.
// Pixel state written by the forward (per tile: planes z, log2 S, gr, g_c of 512 floats + row constants)
// arrives by TMA bulk copies (12 KB per tile for d=2, C=3; double buffered) and is broadcast to all threads
// from shared memory, so the per-kernel reductions over pixels happen in registers with no
// shuffles and no atomics.  Per (pixel, kernel): recompute the gate (T+d FFMA + ex2), then
//     t = w (m gE - gr)            [SURVEY 8a-8: dL/dlog(n_w)]
// and accumulate the sufficient statistics  sum t, sum t x', sum t x' x'^T, sum m w g_c,
// sum m w g_c x'  in tile-centred coordinates; at the end of each tile they are folded into
// kernel-centred moments (sum t delta, sum t delta delta^T) so that no cancellation against
// the absolute position builds up.  The chain rule to (mu, A, pi, nu, gamma) is applied once
// per kernel in smoe_grad_finalize from these P numbers -- for both maha forms.
// Exact-zero skipping (bit-identical to cfg.dense_exec = 1): the gate is w = tau * 2^(q - qthr)
// with the plane qthr = log2 S from the forward (w = 2^(q - log2 S), w > tau <=> q - log2 S > log2 tau); a group of 4 pixels is skipped after its logits when
// all 32 kernels of the warp have q - qthr < -126 (ex2.approx.ftz gives exactly +0 there), and
// the expert part (gE, sum m w g ...) runs only when some kernel of the warp passes the threshold.
#include "smoe_common.cuh"
#include "exchange.cuh"

namespace smoe {

template <int D, int C>
struct BRec {
    static constexpr int T = tri(D);
    static constexpr int GN = T + D + 1;
    static constexpr int EN = C + D * C;
    static constexpr int RC = GN + EN;
    static constexpr int OQ = 0, OL = T, OC = T + D, ONU = GN, OGA = GN + C;
};

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

// DENSE: the dense_exec = 1 instantiation (every pair executed in full) carries none of the skip tests.
template <int D, int C, bool COUNT, bool DENSE>
__global__ void __launch_bounds__(kThreads, 512 / kThreads) backward_kernel(const BwdArgs a) {
    using R = BRec<D, C>;
    constexpr int T = tri(D);
    constexpr int P = nparam(D, C), PK = pstride(D, C);
    const int RL = a.b.tile[D - 1];          // pixels per row of the tile (run along the last axis)
    const int NR = SMOE_TPIX / RL;           // rows per tile (a power of two: RL divides 128, smoe_forward checks it)
    const int tstride = pix_stride(D, C, RL);
    const uint32_t kTileBytes = (uint32_t)tstride * 4u;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* buf0 = reinterpret_cast<float*>(smem_raw);
    float* buf1 = buf0 + tstride;
    uint64_t* bar = reinterpret_cast<uint64_t*>(buf1 + tstride);
    int* scratch = reinterpret_cast<int*>(bar + 2);                 // [16]
    int* tlist = scratch + 16;                                      // [max_list]

    const int tid = threadIdx.x;
    const int K = a.counts[0];
    // kHalves = 2 adjacent lanes share one kernel and take alternate rows of every tile (their partial sums are
    // added at the end, fixed order): a warp then covers 16 neighbouring kernels x 2 rows instead of 32 kernels,
    // which tightens the warp-level skip tests, and a group of kernels gets twice the threads -- what a rank's
    // small pixel block, reached by a hundred groups only, needs to fill the GPU.
    const int k = blockIdx.x * kGroup + tid / kHalves;   // packed row (Hilbert order of the centres)
    const int hsel = tid % kHalves;
    if ((int)blockIdx.x * kGroup >= K) return;
    if (a.plan_cnt[blockIdx.x] == 0) return;             // the group reaches no tile of this batch
    const bool active = k < K;
    const int split = blockIdx.y;
    const float zcut = a.zero_cut, zcut_tile = a.zero_cut - 0.5f;
    unsigned cnt_vis = 0, cnt_gate = 0, cnt_exp = 0;      // COUNT only: warp-level group counters (lane 0)
    const int mode = a.cfg.dense_exec;                   // 0 cull+skip, 1 dense, 2 skip only
    const bool cull = !DENSE && mode == 0;
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
        tma_load_1d(buf ? buf1 : buf0, a.pix + (size_t)tile * tstride, kTileBytes, &bar[buf]);
    };

    // own kernel record: read again at every tile (the CTA's kGroup records stay in L1) rather than held in registers
    // across the tile loop -- the registers go to the look-ahead of the pixel loop below
    const float* rec = a.packed + (size_t)(active ? k : 0) * PK;

    // ordered list of this split's tiles (s, s + NS, ...) that the group can reach, from the plan's bitmask
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

    int* done = scratch + 8;                 // per-buffer count of warps that finished the current tile
    if (tid == 0) {
        done[0] = done[1] = 0;
        if (nlist > 0) issue(tlist[0], 0);
        if (nlist > 1) issue(tlist[1], 1);
    }
    __syncthreads();
    for (int li = 0; li < nlist; ++li) {
        const int buf = li & 1;
        const int tile = tlist[li];
        float ctr[3], half[3];
        tile_box_of<D>(a, tile, ctr, half);
        float mup[D];
#pragma unroll
        for (int l = 0; l < D; ++l) mup[l] = __ldg(rec + off_mu(D, C) + l) - ctr[l];
        const float c0 = active ? __ldg(rec + off_pi(D, C)) : -INFINITY;
        // own kernel vs this tile, then the warp's 32 kernels together
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
            const float ub = c0 - fmaxf(lam * d2, kd) - a.tile_qmin[tile];
            need = !(lam >= 0.f) || !(ub < zcut_tile);
        }
        const bool warp_need = __any_sync(0xffffffffu, need);

        if (buf) { mbar_wait(&bar[1], phase1); phase1 ^= 1; } else { mbar_wait(&bar[0], phase0); phase0 ^= 1; }
        if (warp_need) {
            // tile-centred record in registers
            float f[R::RC];
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
                    float n = __ldg(rec + off_nu(D, C) + c);
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float g = __ldg(rec + off_ga(D, C) + l * C + c);
                        n = fmaf(g, ctr[l], n);
                        f[R::OGA + l * C + c] = g;
                    }
                    f[R::ONU + c] = n;
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

            // pixel state: planes [z | qthr | gr | g_c][512] + the row-constant coordinates (smoe_common.cuh)
            const float* pl = buf ? buf1 : buf0;
            constexpr int GRP = 4;                               // pixels tested together for the exact-zero skip
            constexpr int NGRP = SMOE_TPIX / (GRP * kHalves);    // groups a lane visits per tile: every kHalves-th row
            const int gpr = RL / GRP;                            // groups per row
            // the pixels of a row differ only in their LAST coordinate z: q = cr + (br + qz z) z
            const float qz = f[R::OQ + ut(D, D - 1, D - 1)];
            auto row_coords = [&](int row, float (&x)[3]) {
                x[0] = x[1] = x[2] = 0.f;
#pragma unroll
                for (int l = 0; l < D - 1; ++l) x[l] = pl[pix_rowc_offset(C) + l * NR + row];
            };
            auto row_logit = [&](const float (&x)[3], float& cr, float& br) {
                cr = f[R::OC];
#pragma unroll
                for (int l = 0; l < D - 1; ++l) {
                    float tq = f[R::OL + l];
#pragma unroll
                    for (int m = l; m < D - 1; ++m) tq = fmaf(f[R::OQ + ut(D, l, m)], x[m], tq);
                    cr = fmaf(tq, x[l], cr);
                }
                br = f[R::OL + D - 1];
#pragma unroll
                for (int l = 0; l < D - 1; ++l) br = fmaf(f[R::OQ + ut(D, l, D - 1)], x[l], br);
            };
            // experts along the row: E_c = Er_c + gamma_{d-1,c} z
            auto row_experts = [&](const float (&x)[3], float (&Er)[C]) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    Er[c] = f[R::ONU + c];
#pragma unroll
                    for (int l = 0; l < D - 1; ++l) Er[c] = fmaf(f[R::OGA + l * C + c], x[l], Er[c]);
                }
            };
            // z, gr and the gate logits relative to the pixel's normaliser, dq = q - log2 S, of the group at pixel j
            auto load_group = [&](int j, float cr, float br, float (&z)[GRP], float (&g)[GRP], float (&dq)[GRP]) {
                const float4 zv = *reinterpret_cast<const float4*>(pl + PL_Z * SMOE_TPIX + j);
                const float4 tv = *reinterpret_cast<const float4*>(pl + PL_QTHR * SMOE_TPIX + j);
                const float4 gv = *reinterpret_cast<const float4*>(pl + PL_GR * SMOE_TPIX + j);
                z[0] = zv.x; z[1] = zv.y; z[2] = zv.z; z[3] = zv.w;
                g[0] = gv.x; g[1] = gv.y; g[2] = gv.z; g[3] = gv.w;
                const float t[GRP] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
                for (int u = 0; u < GRP; ++u) dq[u] = fmaf(fmaf(qz, z[u], br), z[u], cr) - t[u];
            };

            // Software pipeline over the lane's groups, across row boundaries: while group i is tested and
            // accumulated, the loads and logits of group i+1 (in the next row, after the last group of a row) are
            // already issued, so the two warp votes of a group never wait on a shared-memory round trip.
            // (the row coordinates are read again where they are needed, instead of being held across the row)
            int row = hsel;                                      // row of the look-ahead group
            float cr, br, Er[C];
            {
                float x[3];
                row_coords(row, x);
                row_logit(x, cr, br);                            // (cr, br): row of the look-ahead group
                row_experts(x, Er);
            }
            float zn[GRP], gn[GRP], dqn[GRP];                    // the look-ahead group
            load_group(row * RL, cr, br, zn, gn, dqn);
            int jn = row * RL, col = 0;
            // row sums: along a row only z varies, so sum t, sum t z, sum t z^2 (and sum v_c, sum v_c z) carry every
            // moment of the row; they are folded once per row and reset
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, nv[C], nz[C];
#pragma unroll
            for (int c = 0; c < C; ++c) nv[c] = nz[c] = 0.f;
            bool row_active = false;
            // (the two lanes of a kernel read rows RL floats apart, i.e. the same banks when RL = 32: a 2-way conflict
            // on these broadcast loads; measured, walking the second row rotated by half a row costs more
            // instructions than the conflicts cost LSU cycles -- the LSU pipe is at 16 %)
            // (unrolled twice, so that the registers of the current and the look-ahead group alternate instead of
            // being copied at every step)
#pragma unroll 2
            for (int gi = 0; gi < NGRP; ++gi) {
                float z4[GRP], gr4[GRP], dq[GRP];
#pragma unroll
                for (int u = 0; u < GRP; ++u) { z4[u] = zn[u]; gr4[u] = gn[u]; dq[u] = dqn[u]; }
                const int j0 = jn;
                // look ahead: the next group of this row, or the first of the lane's next row (after the last row,
                // the first row again -- loaded and never used)
                const bool row_end = ++col == gpr;
                const int rc = row;                              // the current row
                if (row_end) {
                    row = (row + kHalves) & (NR - 1);
                    float x[3];
                    row_coords(row, x);
                    row_logit(x, cr, br);
                    jn = row * RL;
                } else {
                    jn += GRP;
                }
                load_group(jn, cr, br, zn, gn, dqn);

                // both warp decisions of the group, with no load between them:
                //   some gate of the warp is nonzero -- w = 2^dq is exactly +0 for dq < -126 (ex2.approx.ftz);
                //   some gate passes the threshold (w > tau) -- most groups with a nonzero gate only carry
                //   sub-threshold ones: they need neither the g_c planes nor the expert part, only t = -w gr.
                float dmax = -INFINITY;
#pragma unroll
                for (int u = 0; u < GRP; ++u) dmax = fmaxf(dmax, dq[u]);
                const bool any_gate = !skip || __any_sync(0xffffffffu, dmax >= zcut);
                const bool any_pass = !skip || __any_sync(0xffffffffu, dmax > ltau);
                if (COUNT) cnt_vis += 1;
                if (__builtin_expect(any_gate, 0)) {
                    if (COUNT) cnt_gate += 1;
                    row_active = true;
                    if (!any_pass) {
#pragma unroll
                        for (int u = 0; u < GRP; ++u) {
                            const float w = ex2f(dq[u]);             // e / S: the plane holds log2 S
                            const float t = -w * gr4[u];
                            const float uz = t * z4[u];
                            s0 += t;
                            s1 += uz;
                            s2 = fmaf(uz, z4[u], s2);
                        }
                    } else {
                        float g4[C][GRP];
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            const float4 gv = *reinterpret_cast<const float4*>(pl + (PL_G + c) * SMOE_TPIX + j0);
                            g4[c][0] = gv.x; g4[c][1] = gv.y; g4[c][2] = gv.z; g4[c][3] = gv.w;
                        }
                        // the expert part runs for all 4 pixels, with wm = 0 on those whose gate does not pass: adding
                        // 0 * g is exact, so this is the dense instantiation's arithmetic, without a vote per pixel
                        if (COUNT) cnt_exp += GRP;
#pragma unroll
                        for (int u = 0; u < GRP; ++u) {
                            const float w = ex2f(dq[u]);             // e / S: the plane holds log2 S
                            const float wm = dq[u] > ltau ? w : 0.f; // w > tau
                            float gE = 0.f;
#pragma unroll
                            for (int c = 0; c < C; ++c) {
                                const float E = fmaf(f[R::OGA + (D - 1) * C + c], z4[u], Er[c]);
                                gE = fmaf(g4[c][u], E, gE);
                                const float vc = wm * g4[c][u];
                                nv[c] += vc;
                                nz[c] = fmaf(vc, z4[u], nz[c]);
                            }
                            const float t = fmaf(wm, gE, -w * gr4[u]);
                            const float uz = t * z4[u];
                            s0 += t;
                            s1 += uz;
                            s2 = fmaf(uz, z4[u], s2);
                        }
                    }
                }
                if (row_end) {
                    float xr[3];
                    if (row_active) {
                        // fold the row: x_l = xr[l] for l < D-1, x_{D-1} = z
                        row_coords(rc, xr);
                        M0 += s0;
#pragma unroll
                        for (int l = 0; l < D - 1; ++l) {
                            const float a0 = xr[l] * s0;
                            M1[l] += a0;
#pragma unroll
                            for (int m = l; m < D - 1; ++m) M2[ut(D, l, m)] = fmaf(a0, xr[m], M2[ut(D, l, m)]);
                            M2[ut(D, l, D - 1)] = fmaf(xr[l], s1, M2[ut(D, l, D - 1)]);
                        }
                        M1[D - 1] += s1;
                        M2[ut(D, D - 1, D - 1)] += s2;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            N0[c] += nv[c];
#pragma unroll
                            for (int l = 0; l < D - 1; ++l) N1[l][c] = fmaf(xr[l], nv[c], N1[l][c]);
                            N1[D - 1][c] += nz[c];
                            nv[c] = nz[c] = 0.f;
                        }
                        s0 = s1 = s2 = 0.f;
                        row_active = false;
                    }
                    row_coords(row, xr);
                    row_experts(xr, Er);
                    col = 0;
                }
            }
            // fold tile-centred statistics into kernel-centred ones
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
        // Release the buffer without a CTA barrier: the warp that finishes this tile LAST refills the buffer
        // with tile li+2, so a warp never waits for a slower sibling (only for the TMA of its next tile).
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

    if (COUNT && (tid & 31) == 0) {
        // groups of 4 pixels x 32 lanes (vis, gate) and single pixels x 32 lanes (expert part), as issued
        atomicAdd(&a.pair_counts[4], (unsigned long long)cnt_vis * 128ull);
        atomicAdd(&a.pair_counts[5], (unsigned long long)cnt_gate * 128ull);
        atomicAdd(&a.pair_counts[6], (unsigned long long)cnt_exp * 32ull);
    }
    // the kHalves lanes of a kernel are adjacent: add their partial sums (commutative: both lanes get the same bits)
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
        for (int q = 0; q < T; ++q) out[off_A(D, C) + q] = G2[q];     // upper-tri order of the symmetric D
        out[off_pi(D, C)] = G0;
#pragma unroll
        for (int c = 0; c < C; ++c) out[off_nu(D, C) + c] = GNu[c];
#pragma unroll
        for (int l = 0; l < D; ++l)
#pragma unroll
            for (int c = 0; c < C; ++c) out[off_ga(D, C) + l * C + c] = GGa[l][c];
    }
}

// raw[k][j] = sum_s raw_part[s][k][j], fixed order
__global__ void __launch_bounds__(256) reduce_splits_kernel(const int32_t* __restrict__ counts, int K_cap, int P,
                                                            int num_splits, const float* __restrict__ part,
                                                            const int32_t* __restrict__ plan_cnt,
                                                            float* __restrict__ raw) {
    size_t n = (size_t)counts[0] * P;
    size_t stride = (size_t)K_cap * P;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int used = plan_cnt ? segments_used(plan_cnt[(i / P) / kGroup], num_splits) : num_splits;
        raw[i] = slab_sum(part + i, stride, used);
    }
}


// statistics -> variable gradients, one thread per active kernel.
// PEERS (pixel-sharded step): the statistics are the sum over the R ranks' published windows, read straight from
// peer memory in fixed rank order after the flag barrier (exchange.cuh) -- the all-reduce of SURVEY.md 8e fused
// into its consumer; the same launch reduces the loss scalars and the influence flags.
template <int D, int C, bool PEERS>
__global__ void __launch_bounds__(256) grad_finalize_kernel(smoe_cfg cfg, const float* __restrict__ raw, int num_splits,
                                                            int K_cap, const float* __restrict__ theta,
                                                            const int32_t* __restrict__ indices,
                                                            const int32_t* __restrict__ counts, float pis_l1,
                                                            float l1_norm, float u_l1, QuantSet qs_in,
                                                            const QuantDyn* __restrict__ qdyn,
                                                            float* __restrict__ grads, smoe_peers pr,
                                                            float* __restrict__ scalars, uint8_t* __restrict__ infl,
                                                            const int32_t* __restrict__ plan_cnt) {
    constexpr int T = tri(D);
    constexpr int P = nparam(D, C);
    __shared__ float s_stats[kFin * P];
    const int k = blockIdx.x * kFin + threadIdx.x;
    const int K = counts[0];
    const int k0 = blockIdx.x * kFin;
    int epoch = 0;
    if (PEERS) {
        epoch = peer_barrier(pr);
        if (k0 < K) gather_stats<P>(pr, epoch, K_cap, k0, min(kFin, K - k0), s_stats);
        reduce_tail(pr, epoch, K_cap, P, scalars, infl);
        peer_epoch_end(pr, epoch);
    } else if (k0 < K) {
        // sum of the pixel-split slabs of this block's kFin kernels, fixed split order; the block's rows are one
        // contiguous range of every slab, read with coalesced loads (element e of the range by thread e % 256)
        const int n = min(kFin, K - k0) * P;
        const size_t beg = (size_t)k0 * P, stride = (size_t)K_cap * P;
        for (int e = threadIdx.x; e < n; e += 256) {
            // slabs of a group of kernels that reaches no tile were never written (and are not read)
            const int used = plan_cnt ? segments_used(plan_cnt[(k0 + e / P) / kGroup], num_splits) : num_splits;
            s_stats[e] = slab_sum(raw + beg + e, stride, used);
        }
        __syncthreads();
    }
    if (threadIdx.x >= kFin || k >= K) return;
    float s[P];
#pragma unroll
    for (int j = 0; j < P; ++j) s[j] = s_stats[threadIdx.x * P + j];
    const int row = indices[k];
    const float* th = theta + (size_t)row * P;
    float* gr = grads + (size_t)row * P;
    const QuantSet qs = qs_in.mode == 3 ? qdyn->qs : qs_in;
    const bool fq = qs.mode >= 2;
    const float l1 = pis_l1 / (cfg.kernel_count_as_norm_l1 ? (float)counts[1] : l1_norm);     // smoe.py:1022-1027
    float A[D][D], steA[D][D];
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
        for (int m = 0; m < D; ++m) {
            float v = (m <= l) ? th[off_A(D, C) + lt(l, m)] : 0.f;
            steA[l][m] = (fq && m <= l) ? ste_mask(v, qs.g[m == l ? QG_AD : QG_AC]) : 1.f;
            if (fq && m <= l) v = fake_quant(v, qs.g[m == l ? QG_AD : QG_AC]);
            A[l][m] = v;
        }
    float V[D], Dm[D][D];
#pragma unroll
    for (int l = 0; l < D; ++l) V[l] = s[off_mu(D, C) + l];
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
        for (int m = l; m < D; ++m) Dm[l][m] = Dm[m][l] = s[off_A(D, C) + ut(D, l, m)];
    const float M0 = s[off_pi(D, C)];
    // pi
    float pi = th[off_pi(D, C)];
    float ste = 1.f;
    if (cfg.quantize_pis) {
        ste = ste_mask(pi, qs.g[QG_PI]);
        pi = fake_quant(pi, qs.g[QG_PI]);
    }
    gr[off_pi(D, C)] += (M0 / pi + l1) * ste;
    // mu and A
    float gmu[D], gA[D][D];
    if (cfg.train_inverse_cov) {
        // maha = delta^T As delta, As = diag + L + L^T
#pragma unroll
        for (int l = 0; l < D; ++l) {
            float acc = 0.f;
#pragma unroll
            for (int m = 0; m < D; ++m) acc = fmaf((m <= l) ? A[l][m] : A[m][l], V[m], acc);
            gmu[l] = acc;
        }
#pragma unroll
        for (int l = 0; l < D; ++l)
#pragma unroll
            for (int m = 0; m <= l; ++m) gA[l][m] = (l == m) ? -0.5f * Dm[l][l] : -Dm[l][m];
    } else {
        // maha = |A^T delta|^2 : dmu = A (A^T V), dA = -(D A) on the lower triangle
        float AtV[D];
#pragma unroll
        for (int m = 0; m < D; ++m) {
            float acc = 0.f;
#pragma unroll
            for (int l = m; l < D; ++l) acc = fmaf(A[l][m], V[l], acc);
            AtV[m] = acc;
        }
#pragma unroll
        for (int l = 0; l < D; ++l) {
            float acc = 0.f;
#pragma unroll
            for (int m = 0; m <= l; ++m) acc = fmaf(A[l][m], AtV[m], acc);
            gmu[l] = acc;
        }
#pragma unroll
        for (int l = 0; l < D; ++l)
#pragma unroll
            for (int m = 0; m <= l; ++m) {
                float acc = 0.f;
#pragma unroll
                for (int j = m; j < D; ++j) acc = fmaf(Dm[l][j], A[j][m], acc);
                gA[l][m] = -acc;
            }
    }
#pragma unroll
    for (int l = 0; l < D; ++l) {
        gA[l][l] += u_l1;                                               // smoe.py:1044
        if (cfg.use_determinant) gA[l][l] += M0 / A[l][l];              // smoe.py:810
    }
    if (cfg.radial_as) {        // one scalar a per kernel, A = a * I (smoe.py:429-434, 714-721): d/da = sum_l d/dA_ll
        float gs = 0.f;
#pragma unroll
        for (int l = 0; l < D; ++l) gs += gA[l][l];
#pragma unroll
        for (int l = 0; l < D; ++l)
#pragma unroll
            for (int m = 0; m <= l; ++m) gA[l][m] = (l == m) ? gs : 0.f;      // A_corr is not trainable
    }
#pragma unroll
    for (int l = 0; l < D; ++l) {
        gr[off_mu(D, C) + l] += fq ? gmu[l] * ste_mask(th[off_mu(D, C) + l], qs.g[QG_MU]) : gmu[l];
#pragma unroll
        for (int m = 0; m <= l; ++m) gr[off_A(D, C) + lt(l, m)] += gA[l][m] * steA[l][m];
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
        gr[off_nu(D, C) + c] += fq ? s[off_nu(D, C) + c] * ste_mask(th[off_nu(D, C) + c], qs.g[QG_NU]) : s[off_nu(D, C) + c];
#pragma unroll
        for (int l = 0; l < D; ++l) {
            float gv = s[off_ga(D, C) + l * C + c];
            if (!cfg.train_gammas) gv = 0.f;
            if (cfg.use_yuv && cfg.only_y_gamma && c > 0) gv = 0.f;
            if (fq) gv *= ste_mask(th[off_ga(D, C) + l * C + c], qs.g[QG_GA]);
            gr[off_ga(D, C) + l * C + c] += gv;
        }
    }
}

// TF1 ApplyAdam: m += (g-m)(1-b1); v += (g^2-v)(1-b2); var -= alpha*m/(sqrt(v)+eps)
template <int D, int C>
__global__ void __launch_bounds__(256) adam_kernel(smoe_adam hp, const float* __restrict__ alpha_dev,
                                                   float* __restrict__ theta, const float* __restrict__ grads,
                                                   float* __restrict__ am, float* __restrict__ av, size_t n,
                                                   const uint8_t* __restrict__ infl, uint8_t* __restrict__ klist) {
    constexpr int P = nparam(D, C);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(i % P);
        if (klist && j == 0) klist[i / P] = infl[i / P] ? 1 : 0;      // kernel_list <- influential kernels (smoe.py:1763-1766)
        int grp;
        bool on = true;
        if (j < off_A(D, C)) { grp = 0; on = hp.train_musx != 0; }
        else if (j < off_pi(D, C)) grp = 2;
        else if (j == off_pi(D, C)) grp = 1;
        else if (j < off_ga(D, C)) grp = 0;
        else { grp = 0; on = hp.train_gammas != 0; }
        const float alpha = alpha_dev ? alpha_dev[grp] : hp.alpha[grp];
        if (!on || alpha == 0.f) continue;
        float g = grads[i];
        if (hp.grad_clip > 0.f) g = fminf(fmaxf(g, -hp.grad_clip), hp.grad_clip);
        float m = am[i], v = av[i];
        m = __fadd_rn(m, __fmul_rn(__fsub_rn(g, m), 1.f - hp.beta1[grp]));
        v = __fadd_rn(v, __fmul_rn(__fsub_rn(__fmul_rn(g, g), v), 1.f - hp.beta2[grp]));
        am[i] = m;
        av[i] = v;
        theta[i] = __fsub_rn(theta[i], __fdiv_rn(__fmul_rn(m, alpha), __fadd_rn(__fsqrt_rn(v), hp.epsilon[grp])));
    }
}

}  // namespace smoe

using namespace smoe;

extern "C" {

size_t smoe_backward_workspace_bytes(const smoe_cfg* cfg, int K_cap, int num_splits) {
    return (size_t)num_splits * K_cap * nparam(cfg->d, cfg->C) * sizeof(float);
}

size_t smoe_backward_plan_bytes(int K_cap, const smoe_batch* batch) {
    const size_t groups = (size_t)(K_cap + kGroup - 1) / kGroup;
    const size_t nwords = ((size_t)smoe_num_tiles(batch) + 127) / 128 * 4;       // whole 128-tile rounds of the plan CTA
    return (groups + groups * nwords) * sizeof(int32_t);
}

int smoe_backward(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const int32_t* counts, int K_cap,
                  const float* pix, const float* tile_qmin, const float* ax0, const float* ax1, const float* ax2,
                  int num_splits, float* raw_part, int32_t* plan, unsigned long long* pair_counts, void* stream) {
    SMOE_REQUIRE(cfg && batch && packed && counts && pix && tile_qmin && ax0 && ax1 && raw_part && plan, "null argument");
    SMOE_REQUIRE(K_cap > 0 && num_splits > 0 && num_splits <= 65535, "bad K_cap / num_splits");
    SMOE_REQUIRE(cfg->eps_bits == 0 || (cfg->eps_bits >= 24 && cfg->eps_bits <= 126 && cfg->dense_exec == 0),
                 "eps_bits must be 0 or in [24, 126], with dense_exec == 0");
    BwdArgs a;
    a.cfg = *cfg;
    a.b = *batch;
    a.packed = packed; a.counts = counts; a.pix = pix; a.tile_qmin = tile_qmin;
    a.raw_part = raw_part;
    a.pair_counts = pair_counts;
    a.ax[0] = ax0; a.ax[1] = ax1; a.ax[2] = ax2 ? ax2 : ax0;
    a.K_cap = K_cap;
    a.num_splits = num_splits;
    a.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    a.ntiles = smoe_num_tiles(batch);
    a.tau = 0.5f / (float)(1 << cfg->precision);
    a.ltau = -(float)(cfg->precision + 1);              // log2(tau), exact
    a.zero_cut = cfg->eps_bits > 0 ? -(float)cfg->eps_bits : -126.0f;
    const int groups = (K_cap + kGroup - 1) / kGroup;
    a.plan_cnt = plan;
    a.plan_bits = reinterpret_cast<uint32_t*>(plan + groups);
    a.nwords = (a.ntiles + 127) / 128 * 4;
    a.max_list = (a.ntiles + num_splits - 1) / num_splits;
    dim3 grid(groups, num_splits);
    size_t sm = 2 * (size_t)pix_stride(cfg->d, cfg->C, batch->tile[cfg->d - 1]) * 4 + 16 + 16 * 4 + (size_t)a.max_list * 4 + 64;
    SMOE_REQUIRE(sm <= 100 * 1024, "too many tiles per split for the shared-memory tile list: raise num_splits");
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(D, C, CNT, DN)                                                                                       \
    {                                                                                                               \
        bwd_plan_kernel<D, C><<<groups, 128, (size_t)a.nwords * 4, st>>>(a);                                        \
        cudaFuncSetAttribute(backward_kernel<D, C, CNT, DN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        backward_kernel<D, C, CNT, DN><<<grid, kThreads, sm, st>>>(a);                                              \
    }
#define CALL(D, C)                                                                                        \
    if (cfg->dense_exec == 1) { if (pair_counts) LAUNCH(D, C, true, true) else LAUNCH(D, C, false, true) } \
    else { if (pair_counts) LAUNCH(D, C, true, false) else LAUNCH(D, C, false, false) }
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
#undef LAUNCH
    return check_launch("smoe_backward");
}

int smoe_reduce_splits(const smoe_cfg* cfg, const int32_t* counts, int K_cap, int num_splits, const float* raw_part,
                       const int32_t* plan, float* raw, void* stream) {
    SMOE_REQUIRE(cfg && counts && raw_part && raw && K_cap > 0 && num_splits > 0, "bad argument");
    int P = nparam(cfg->d, cfg->C);
    size_t n = (size_t)K_cap * P;
    int nb = (int)((n + 255) / 256);
    if (nb > 148 * 16) nb = 148 * 16;
    reduce_splits_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(counts, K_cap, P, num_splits, raw_part, plan, raw);
    return check_launch("smoe_reduce_splits");
}

int smoe_grad_finalize(const smoe_cfg* cfg, const float* raw, int num_splits, const int32_t* plan, int K_cap,
                       const float* theta, const void* quant_ranges, const int32_t* indices, const int32_t* counts,
                       float pis_l1, float l1_norm, float u_l1, float* grads, void* stream) {
    SMOE_REQUIRE(cfg && raw && theta && indices && counts && grads && K_cap > 0 && num_splits > 0, "bad argument");
    SMOE_REQUIRE(cfg->quantization_mode != 3 || quant_ranges, "quantization_mode 3 needs quant_ranges");
    SMOE_REQUIRE(cfg->kernel_count_as_norm_l1 || l1_norm > 0.f, "l1_norm must be positive");
    const QuantSet qs = make_quantset(cfg);
    int nb = (K_cap + kFin - 1) / kFin;
    cudaStream_t st = (cudaStream_t)stream;
    smoe_peers none = {};
#define CALL(D, C)                                                                                                     \
    grad_finalize_kernel<D, C, false><<<nb, 256, 0, st>>>(*cfg, raw, num_splits, K_cap, theta, indices, counts, pis_l1, \
                                                          l1_norm, u_l1, qs, (const QuantDyn*)quant_ranges, grads,     \
                                                          none, nullptr, nullptr, plan);
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_grad_finalize");
}

int smoe_grad_finalize_peers(const smoe_cfg* cfg, const smoe_peers* peers, int K_cap, const float* theta,
                             const void* quant_ranges, const int32_t* indices, const int32_t* counts, float pis_l1,
                             float l1_norm, float u_l1, float* grads, float* scalars, uint8_t* infl, void* stream) {
    SMOE_REQUIRE(cfg && peers && theta && indices && counts && grads && scalars && infl && K_cap > 0, "bad argument");
    SMOE_REQUIRE(peers->world >= 1 && peers->world <= SMOE_MAX_PEERS && peers->rank >= 0 && peers->rank < peers->world,
                 "bad peer set");
    for (int r = 0; r < peers->world; ++r) SMOE_REQUIRE(peers->win[r], "null peer window");
    SMOE_REQUIRE(cfg->quantization_mode != 3 || quant_ranges, "quantization_mode 3 needs quant_ranges");
    SMOE_REQUIRE(cfg->kernel_count_as_norm_l1 || l1_norm > 0.f, "l1_norm must be positive");
    const QuantSet qs = make_quantset(cfg);
    int nb = (K_cap + kFin - 1) / kFin;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C)                                                                                                     \
    grad_finalize_kernel<D, C, true><<<nb, 256, 0, st>>>(*cfg, nullptr, 1, K_cap, theta, indices, counts, pis_l1,       \
                                                         l1_norm, u_l1, qs, (const QuantDyn*)quant_ranges, grads,      \
                                                         *peers, scalars, infl, nullptr);
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_grad_finalize_peers");
}

int smoe_adam_step(const smoe_cfg* cfg, const smoe_adam* hp, const float* alpha_dev, float* theta, const float* grads,
                   float* adam_m, float* adam_v, int K_all, const uint8_t* infl, uint8_t* kernel_list, void* stream) {
    SMOE_REQUIRE(cfg && hp && theta && grads && adam_m && adam_v && K_all > 0, "bad argument");
    SMOE_REQUIRE((infl == nullptr) == (kernel_list == nullptr), "infl and kernel_list go together");
    size_t n = (size_t)K_all * nparam(cfg->d, cfg->C);
    int nb = (int)((n + 255) / 256);
    if (nb > 148 * 8) nb = 148 * 8;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C) adam_kernel<D, C><<<nb, 256, 0, st>>>(*hp, alpha_dev, theta, grads, adam_m, adam_v, n, infl, kernel_list);
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_adam_step");
}

}  // extern "C"
