// Gauss-Newton diagonal of an SMoE: smoe_gn_state / smoe_gn_diag (uniform grid), smoe_point_gn_state /
// smoe_point_gn_diag (points), smoe_gn_diag_scatter.
//
// D = diag(J^T diag(h) J) for J = d r / d theta (r before clip) and a per-sample, per-channel weight h >= 0 (h = 1:
// diag(J^T J); h = l'' of a loss sum l(r): the generalised Gauss-Newton diagonal).  With jvp.cu's notation (gates
// w_k = 2^(q_k - qthr), m_k = [w_k > tau], f the flag S > 1e-11, experts E_kc = nu_kc + gamma_k[:, c] . x), a gate
// parameter theta_i of kernel k enters r_c only through q_k, and an expert parameter only through E_kc, so
//     D[gate theta_i]  = sum_n ln2^2 w_k^2 (dq_k / dtheta_i)^2 sum_c h_c (m_k E_kc - f r_c)^2
//     D[nu_kc]         = sum_n h_c m_k w_k^2
//     D[gamma_k[l, c]] = sum_n h_c m_k w_k^2 x_l^2
// -- P non-negative sums per kernel, the shape of the parameter backward.  dq / dtheta_i is the tangent logit that
// smoe_pack_tangent gives the one-hot tangent e_i (log2 units, delta = x - mu):
//     mu_l:   2 (Qm delta)_l
//     A_lm:   -kHalfLog2e delta^T dQm delta + [l == m] [use_determinant] log2(e) / A_ll
//             (dQm of A_lm: e_l e_m^T + e_m e_l^T halved on the diagonal under train_inverse_cov, else
//             e_l e_m^T A^T + A e_m e_l^T; so delta^T dQm delta = (2 - [l == m]) delta_l delta_m, or 2 delta_l (A^T delta)_m)
//     pi:     log2(e) / pi
// with dc0 = 0 for a kernel whose A_ll is 0 under use_determinant (no gate anywhere), as in smoe_pack_tangent.
//
// The state stage (gn_state_kernel / point_gn_state_kernel, elementwise, the launch geometry of the cotangent stages)
// copies what the sweep needs into one tile-major buffer that a single bulk copy per tile brings in: qthr, h_c and
// f r_c, and the coordinates.  The sweep (gn_diag_kernel) is backward_kernel's kernel-stationary CTA: 64 consecutive
// packed kernels (2 lanes each, alternate groups of 4 samples) over a 1/num_splits share of the tiles that the
// planning pre-pass (bwd_plan_kernel / point_plan_kernel) left reachable, tiles double buffered by TMA, partial sums in
// registers, one slab per split in the theta column layout (mu | A lower-tri | pi | nu | gamma) for smoe_reduce_splits.
// Every term carries w^2, evaluated as ex2(2 (q - qthr)): exactly +0 below q - qthr < -63 (ex2.approx.ftz), so the
// grid plan, the per-kernel tile test and the warp's group skip all cut at -63 instead of -126 (the point plan keeps
// its -126: it reads no cut).  Skipped terms are exact zeros, and every sum runs in a fixed order, so cfg.dense_exec
// 0, 1 and 2 give the same bits.  No float atomics, no host synchronisation.
#include "bwd_plan.cuh"
#include "pt_plan.cuh"

namespace smoe {

constexpr float kGnCut = -63.f;
constexpr float kLog2e = 1.44269504088896340736f;

// Grid state, per tile: planes [z | qthr | h_c | f r_c][SMOE_TPIX], then the row coordinates of the pix state.
constexpr int GP_Z = 0, GP_QTHR = 1, GP_H = 2;
__host__ __device__ constexpr int gp_fr(int C) { return GP_H + C; }
__host__ __device__ constexpr int gp_rowc_offset(int C) { return (2 + 2 * C) * SMOE_TPIX; }
__host__ __device__ inline int gp_rowc_floats(int d, int RL) { return ((d - 1) * (SMOE_TPIX / RL) + 3) / 4 * 4; }
__host__ __device__ inline int gp_stride(int d, int C, int RL) { return gp_rowc_offset(C) + gp_rowc_floats(d, RL); }
// Point state, per tile: planes [qthr | h_c | f r_c | x'_l][SMOE_TPIX].
constexpr int GQ_QTHR = 0, GQ_H = 1;
__host__ __device__ constexpr int gq_fr(int C) { return GQ_H + C; }
__host__ __device__ constexpr int gq_x(int C) { return GQ_H + 2 * C; }
__host__ __device__ constexpr int gq_stride(int d, int C) { return (1 + 2 * C + d) * SMOE_TPIX; }

struct GnStateArgs {
    smoe_batch b;
    const float* src;          // pix (grid) / point state, as the forward left them
    const float* r;            // rbuf (grid) / r in tile order (points)
    const float* h;            // weight, or NULL: h = 1
    const int64_t* order;      // points: the caller's row of tile slot i (read with a weight)
    long long hs_n, hs_c;      // element strides of the weight per sample and per channel
    float* gstate;
    int nt1, nt2, src_stride, dst_stride, rowc_floats, n, nslots;
};

// Grid: one CTA per tile, the geometry and slot numbering of cotangent_kernel.
template <int C>
__global__ void __launch_bounds__(256) gn_state_kernel(const GnStateArgs a) {
    const int tid = threadIdx.x;
    const int e1 = a.b.tile[1], e2 = a.b.tile[2];
    int tt[3], lo[3], hi[3];
    tt[0] = blockIdx.y;
    tt[1] = a.nt2 == 1 ? (int)blockIdx.x : (int)blockIdx.x / a.nt2;
    tt[2] = a.nt2 == 1 ? 0 : (int)blockIdx.x % a.nt2;
    const int tile = (tt[0] * a.nt1 + tt[1]) * a.nt2 + tt[2];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        lo[i] = a.b.origin[i] + tt[i] * a.b.tile[i];
        hi[i] = min(lo[i] + a.b.tile[i], a.b.origin[i] + a.b.extent[i]) - 1;
    }
    const float* sp = a.src + (size_t)tile * a.src_stride;
    float* dp = a.gstate + (size_t)tile * a.dst_stride;
    const int i2 = tid % e2, i1 = (tid / e2) % e1;
    const int g1 = lo[1] + i1, g2 = lo[2] + i2;
    const bool in12 = g1 <= hi[1] && g2 <= hi[2];
    const int rows_per_pass = 256 / (e1 * e2);
    int g0 = lo[0] + tid / (e1 * e2);
    for (int j = tid; j < SMOE_TPIX; j += 256, g0 += rows_per_pass) {
        const bool inb = in12 && g0 <= hi[0];
        const size_t gpix = inb ? ((size_t)g0 * a.b.dims[1] + g1) * a.b.dims[2] + g2 : 0;
        const bool live = inb && sp[PL_GR * SMOE_TPIX + j] != 0.f;          // the flag S > 1e-11
        dp[GP_Z * SMOE_TPIX + j] = sp[PL_Z * SMOE_TPIX + j];
        dp[GP_QTHR * SMOE_TPIX + j] = sp[PL_QTHR * SMOE_TPIX + j];       // +inf outside the batch: w = 0
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float h = !inb ? 0.f : a.h ? a.h[(long long)gpix * a.hs_n + c * a.hs_c] : 1.f;
            dp[(GP_H + c) * SMOE_TPIX + j] = h;
            dp[(gp_fr(C) + c) * SMOE_TPIX + j] = live ? a.r[gpix * C + c] : 0.f;
        }
    }
    for (int j = tid; j < a.rowc_floats; j += 256) dp[gp_rowc_offset(C) + j] = sp[pix_rowc_offset(C) + j];
}

// Points: one thread per slot, as point_cotangent_kernel.
template <int D, int C>
__global__ void __launch_bounds__(256) point_gn_state_kernel(const GnStateArgs a) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= a.nslots) return;
    const float* sp = a.src + (size_t)(i / SMOE_TPIX) * pt_stride(D, C);
    float* dp = a.gstate + (size_t)(i / SMOE_TPIX) * gq_stride(D, C);
    const int j = i % SMOE_TPIX;
    const bool ok = i < a.n;
    const bool live = sp[PP_GR * SMOE_TPIX + j] != 0.f;                    // the flag; 0 past the last point
    const long long row = (ok && a.h) ? a.order[i] : 0;
    dp[GQ_QTHR * SMOE_TPIX + j] = sp[PP_QTHR * SMOE_TPIX + j];             // +inf past the last point: w = 0
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const float h = !ok ? 0.f : a.h ? a.h[row * a.hs_n + c * a.hs_c] : 1.f;
        dp[(GQ_H + c) * SMOE_TPIX + j] = h;
        dp[(gq_fr(C) + c) * SMOE_TPIX + j] = live ? a.r[(size_t)i * C + c] : 0.f;
    }
#pragma unroll
    for (int l = 0; l < D; ++l) dp[(gq_x(C) + l) * SMOE_TPIX + j] = sp[(pp_x(C) + l) * SMOE_TPIX + j];
}

struct GnArgs {
    BwdArgs g;                 // grid geometry (tile_box_of), counts, packed record, plan, splits
    const float* theta;        // [K_all][P] rows, read through indices: pi and the raw A
    const int32_t* indices;
    const float* gstate;
    const float* tile_box;     // points: [tiles][kTB]
    int tstride;
};

// PTS: point tiles (else grid tiles); DENSE: the dense_exec = 1 instantiation, with none of the skip tests.
template <int D, int C, bool PTS, bool DENSE>
__global__ void __launch_bounds__(kThreads, 512 / kThreads) gn_diag_kernel(const GnArgs ga) {
    constexpr int T = tri(D);
    constexpr int P = nparam(D, C), PK = pstride(D, C);
    constexpr int GRP = 4;
    const BwdArgs& a = ga.g;
    const int tstride = ga.tstride;
    const uint32_t kTileBytes = (uint32_t)tstride * 4u;
    const int RL = PTS ? 1 : a.b.tile[D - 1];
    const int NR = SMOE_TPIX / RL;
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
    if (a.plan_cnt[blockIdx.x] == 0) return;             // the group reaches no tile of this batch
    const bool active = k < K;
    const int split = blockIdx.y;
    const float zcut_tile = kGnCut - 0.5f;
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
        tma_load_1d(buf ? buf1 : buf0, ga.gstate + (size_t)tile * tstride, kTileBytes, &bar[buf]);
    };
    const float* rec = a.packed + (size_t)(active ? k : 0) * PK;
    const float* th = ga.theta + (size_t)(active ? ga.indices[k] : 0) * P;

    // ordered list of this split's reachable tiles (s, s + NS, ...), as backward_kernel builds it
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

    float G[P];
#pragma unroll
    for (int j = 0; j < P; ++j) G[j] = 0.f;

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
        float ctr[3], half[3], qmin;
        if (PTS) {
            const float* tb = ga.tile_box + (size_t)tile * kTB;
#pragma unroll
            for (int i = 0; i < 3; ++i) { ctr[i] = tb[i]; half[i] = tb[3 + i]; }
            qmin = tb[6];
        } else {
            tile_box_of<D>(a, tile, ctr, half);
            qmin = a.tile_qmin[tile];
        }
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
            const float ub = c0 - fmaxf(lam * d2, kd) - qmin;
            need = !(lam >= 0.f) || !(ub < zcut_tile);
        }
        const bool warp_need = __any_sync(0xffffffffu, need);

        if (buf) { mbar_wait(&bar[1], phase1); phase1 ^= 1; } else { mbar_wait(&bar[0], phase0); phase0 ^= 1; }
        if (warp_need) {
            // the kernel: Qm (packed, log2 units), the matrix By with y = By^T delta (identity under train_inverse_cov,
            // else the raw lower-triangular A), dc0 / dA_ll, the experts re-centred on the tile
            float Q[D][D], By[D][D], dc[D], nuc[C], gam[D][C];
            const bool inv = a.cfg.train_inverse_cov != 0;
#pragma unroll
            for (int l = 0; l < D; ++l)
#pragma unroll
                for (int m = l; m < D; ++m) Q[l][m] = Q[m][l] = __ldg(rec + off_A(D, C) + ut(D, l, m));
            bool dead = false;
#pragma unroll
            for (int l = 0; l < D; ++l) {
#pragma unroll
                for (int m = 0; m <= l; ++m) By[l][m] = inv ? (l == m ? 1.f : 0.f) : __ldg(th + off_A(D, C) + lt(l, m));
                const float all = __ldg(th + off_A(D, C) + lt(l, l));
                dc[l] = a.cfg.use_determinant ? kLog2e / all : 0.f;
                dead |= a.cfg.use_determinant && all == 0.f;
            }
#pragma unroll
            for (int l = 0; l < D; ++l) dc[l] = dead ? 0.f : dc[l];
            const float sdiag = inv ? -kHalfLog2e : -2.f * kHalfLog2e, soff = -2.f * kHalfLog2e;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                float nn = __ldg(rec + off_nu(D, C) + c);
#pragma unroll
                for (int l = 0; l < D; ++l) {
                    gam[l][c] = __ldg(rec + off_ga(D, C) + l * C + c);
                    nn = fmaf(gam[l][c], ctr[l], nn);
                }
                nuc[c] = nn;
            }
            const float* pl = buf ? buf1 : buf0;
            const int hoff = PTS ? GQ_H : GP_H, froff = PTS ? gq_fr(C) : gp_fr(C);
            for (int gi = hsel; gi < SMOE_TPIX / GRP; gi += kHalves) {
                const int j0 = gi * GRP;
                float xg[GRP][D], dq[GRP];
                {
                    const float4 tv = *reinterpret_cast<const float4*>(pl + (PTS ? GQ_QTHR : GP_QTHR) * SMOE_TPIX + j0);
                    const float t4[GRP] = {tv.x, tv.y, tv.z, tv.w};
                    if (PTS) {
#pragma unroll
                        for (int l = 0; l < D; ++l) {
                            const float4 xv = *reinterpret_cast<const float4*>(pl + (gq_x(C) + l) * SMOE_TPIX + j0);
                            xg[0][l] = xv.x; xg[1][l] = xv.y; xg[2][l] = xv.z; xg[3][l] = xv.w;
                        }
                    } else {
                        // a group of 4 lies in one row (RL % 4 == 0): the other coordinates are the row's
                        const int row = j0 / RL;
#pragma unroll
                        for (int l = 0; l < D - 1; ++l) {
                            const float xr = pl[gp_rowc_offset(C) + l * NR + row];
#pragma unroll
                            for (int u = 0; u < GRP; ++u) xg[u][l] = xr;
                        }
                        const float4 zv = *reinterpret_cast<const float4*>(pl + GP_Z * SMOE_TPIX + j0);
                        xg[0][D - 1] = zv.x; xg[1][D - 1] = zv.y; xg[2][D - 1] = zv.z; xg[3][D - 1] = zv.w;
                    }
#pragma unroll
                    for (int u = 0; u < GRP; ++u) {
                        float q = c0;
#pragma unroll
                        for (int l = 0; l < D; ++l) {
                            const float dl = xg[u][l] - mup[l];
                            float v = 0.f;
#pragma unroll
                            for (int m = 0; m < D; ++m) v = fmaf(Q[l][m], xg[u][m] - mup[m], v);
                            q = fmaf(-dl, v, q);
                        }
                        dq[u] = q - t4[u];
                    }
                }
                float dmax = -INFINITY;
#pragma unroll
                for (int u = 0; u < GRP; ++u) dmax = fmaxf(dmax, dq[u]);
                if (skip && !__any_sync(0xffffffffu, dmax >= kGnCut)) continue;
#pragma unroll
                for (int u = 0; u < GRP; ++u) {
                    const float w2 = ex2f(2.f * dq[u]);                   // w^2; exactly +0 below -63
                    const float w2m = dq[u] > ltau ? w2 : 0.f;            // m w^2
                    float del[D], v[D], y[D];
#pragma unroll
                    for (int l = 0; l < D; ++l) del[l] = xg[u][l] - mup[l];
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        v[l] = 0.f;
#pragma unroll
                        for (int m = 0; m < D; ++m) v[l] = fmaf(Q[l][m], del[m], v[l]);
                        y[l] = 0.f;
#pragma unroll
                        for (int j = l; j < D; ++j) y[l] = fmaf(By[j][l], del[j], y[l]);
                    }
                    // gate weight sum_c h_c (m E_c - f r_c)^2 w^2 (ln2^2 is applied once, at the end)
                    float s = 0.f;
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        float E = nuc[c];
#pragma unroll
                        for (int l = 0; l < D; ++l) E = fmaf(gam[l][c], xg[u][l], E);
                        // h_c and f r_c of the sample, read where they are used (registers go to the accumulators)
                        const float hc = pl[(hoff + c) * SMOE_TPIX + j0 + u];
                        const float e = (dq[u] > ltau ? E : 0.f) - pl[(froff + c) * SMOE_TPIX + j0 + u];
                        s = fmaf(hc * e, e, s);
                        const float ew = w2m * hc;
                        G[off_nu(D, C) + c] += ew;
#pragma unroll
                        for (int l = 0; l < D; ++l) {
                            const float xa = xg[u][l] + ctr[l];
                            G[off_ga(D, C) + l * C + c] = fmaf(ew * xa, xa, G[off_ga(D, C) + l * C + c]);
                        }
                    }
                    const float t = w2 * s;
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float g = 2.f * v[l];
                        G[off_mu(D, C) + l] = fmaf(t * g, g, G[off_mu(D, C) + l]);
#pragma unroll
                        for (int m = 0; m <= l; ++m) {
                            const float ga = (l == m) ? fmaf(sdiag * del[l], y[m], dc[l]) : soff * del[l] * y[m];
                            G[off_A(D, C) + lt(l, m)] = fmaf(t * ga, ga, G[off_A(D, C) + lt(l, m)]);
                        }
                    }
                    G[off_pi(D, C)] += t;                                 // times (dq / dpi)^2, a constant, at the end
                }
            }
        }
        // the buffer hand-over of backward_kernel: the warp that finishes the tile last refills its buffer
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

#pragma unroll
    for (int j = 0; j < P; ++j)
#pragma unroll
        for (int o = 1; o < kHalves; o <<= 1) G[j] += __shfl_xor_sync(0xffffffffu, G[j], o);
    if (active && hsel == 0) {
        constexpr float kLn2sq = kLn2 * kLn2;
        bool dead = false;
        if (a.cfg.use_determinant)
#pragma unroll
            for (int l = 0; l < D; ++l) dead |= __ldg(th + off_A(D, C) + lt(l, l)) == 0.f;
        const float dpi = dead ? 0.f : kLog2e / __ldg(th + off_pi(D, C));
        float* out = a.raw_part + ((size_t)split * a.K_cap + k) * P;
#pragma unroll
        for (int j = 0; j < off_pi(D, C); ++j) out[j] = G[j] * kLn2sq;
        out[off_pi(D, C)] = G[off_pi(D, C)] * kLn2sq * (dpi * dpi);
#pragma unroll
        for (int j = off_nu(D, C); j < P; ++j) out[j] = G[j];
    }
}

// diag[indices[k]][j] = raw[k][j] for the counts[0] packed rows; the rows of dropped kernels keep the caller's zeros
__global__ void __launch_bounds__(256) gn_scatter_kernel(const int32_t* __restrict__ counts, int P,
                                                         const float* __restrict__ raw,
                                                         const int32_t* __restrict__ indices, float* __restrict__ diag) {
    const size_t n = (size_t)counts[0] * P;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        diag[(size_t)indices[i / P] * P + i % P] = raw[i];
}

static int gn_check_cfg(const smoe_cfg* cfg) {
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the Gauss-Newton diagonal");
    SMOE_REQUIRE(cfg->quantization_mode == 0 && !cfg->quantize_pis && !cfg->use_diff_center && !cfg->radial_as,
                 "the diagonal of fake-quantised, diff-centre or radial parameters is not supported");
    SMOE_REQUIRE(cfg->train_gammas && !(cfg->use_yuv && cfg->only_y_gamma), "every gamma must be trained");
    return 0;
}

static int gn_check_batch(const smoe_cfg* cfg, const smoe_batch* batch) {
    SMOE_REQUIRE(batch->tile[0] * batch->tile[1] * batch->tile[2] == SMOE_TPIX, "tile product must be SMOE_TPIX");
    SMOE_REQUIRE(kThreadsF % (batch->tile[1] * batch->tile[2]) == 0 && batch->tile[cfg->d - 1] % 4 == 0,
                 "tile[1]*tile[2] must divide 128 and the last tile extent must be a multiple of 4");
    SMOE_REQUIRE(batch->halo == 0, "the Gauss-Newton diagonal needs a batch without halo");
    for (int i = 0; i < 3; ++i)
        SMOE_REQUIRE(batch->extent[i] > 0 && batch->origin[i] >= 0 && batch->origin[i] + batch->extent[i] <= batch->dims[i],
                     "batch rectangle outside the image");
    SMOE_REQUIRE(cfg->d == 3 || (batch->dims[2] == 1 && batch->tile[2] == 1), "d == 2 needs dims[2] == tile[2] == 1");
    SMOE_REQUIRE((long long)batch->dims[0] * batch->dims[1] * batch->dims[2] < (1ll << 31), "more than 2^31 pixels");
    return 0;
}

}  // namespace smoe

using namespace smoe;

extern "C" {

int smoe_gn_state_stride(int d, int C, const smoe_batch* batch) {
    if (!batch || (d != 2 && d != 3) || batch->tile[d - 1] <= 0) return 0;
    return gp_stride(d, C, batch->tile[d - 1]);
}

int smoe_point_gn_state_stride(int d, int C) { return gq_stride(d, C); }

int smoe_gn_state(const smoe_cfg* cfg, const smoe_batch* batch, const float* pix, const float* rbuf,
                  const float* weight, long long weight_stride_sample, long long weight_stride_channel, float* gstate,
                  void* stream) {
    SMOE_REQUIRE(cfg && batch && pix && rbuf && gstate, "null argument");
    if (int rc = gn_check_cfg(cfg)) return rc;
    if (int rc = gn_check_batch(cfg, batch)) return rc;
    SMOE_REQUIRE(weight_stride_sample >= 0 && weight_stride_channel >= 0, "negative weight stride");
    GnStateArgs a = {};
    a.b = *batch;
    a.src = pix; a.r = rbuf; a.h = weight;
    a.hs_n = weight_stride_sample; a.hs_c = weight_stride_channel;
    a.gstate = gstate;
    a.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    const int RL = batch->tile[cfg->d - 1];
    a.src_stride = pix_stride(cfg->d, cfg->C, RL);
    a.dst_stride = gp_stride(cfg->d, cfg->C, RL);
    a.rowc_floats = gp_rowc_floats(cfg->d, RL);
    const int nt0 = smoe_num_tiles(batch) / (a.nt1 * a.nt2);
    SMOE_REQUIRE(nt0 <= 65535, "too many tiles along the first axis");
    const dim3 grid(a.nt1 * a.nt2, nt0);
    if (cfg->C == 1) gn_state_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    else gn_state_kernel<3><<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("smoe_gn_state");
}

int smoe_point_gn_state(const smoe_cfg* cfg, int n_points, const float* state, const float* r, const float* weight,
                        const int64_t* order, long long weight_stride_sample, long long weight_stride_channel,
                        float* gstate, void* stream) {
    SMOE_REQUIRE(cfg && state && r && gstate, "null argument");
    SMOE_REQUIRE(!weight || order, "a weight needs the point order");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    if (int rc = gn_check_cfg(cfg)) return rc;
    SMOE_REQUIRE(weight_stride_sample >= 0 && weight_stride_channel >= 0, "negative weight stride");
    GnStateArgs a = {};
    a.src = state; a.r = r; a.h = weight; a.order = order;
    a.hs_n = weight_stride_sample; a.hs_c = weight_stride_channel;
    a.gstate = gstate;
    a.n = n_points;
    a.nslots = pt_tiles(n_points) * SMOE_TPIX;
    const int nb = (a.nslots + 255) / 256;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C) point_gn_state_kernel<D, C><<<nb, 256, 0, st>>>(a);
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_point_gn_state");
}

int smoe_gn_diag(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const float* theta,
                 const int32_t* indices, const int32_t* counts, int K_cap, const float* gstate, const float* tile_qmin,
                 const float* ax0, const float* ax1, const float* ax2, int num_splits, float* raw_part, int32_t* plan,
                 void* stream) {
    SMOE_REQUIRE(cfg && batch && packed && theta && indices && counts && gstate && tile_qmin && ax0 && ax1 && raw_part &&
                     plan,
                 "null argument");
    SMOE_REQUIRE(K_cap > 0 && num_splits > 0 && num_splits <= 65535, "bad K_cap / num_splits");
    if (int rc = gn_check_cfg(cfg)) return rc;
    SMOE_REQUIRE(cfg->d == 2 || ax2, "ax2 required for d == 3");
    if (int rc = gn_check_batch(cfg, batch)) return rc;
    GnArgs ga = {};
    BwdArgs& a = ga.g;
    a.cfg = *cfg;
    a.b = *batch;
    a.packed = packed; a.counts = counts; a.tile_qmin = tile_qmin;
    a.raw_part = raw_part;
    a.ax[0] = ax0; a.ax[1] = ax1; a.ax[2] = ax2 ? ax2 : ax0;
    a.K_cap = K_cap;
    a.num_splits = num_splits;
    a.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    a.ntiles = smoe_num_tiles(batch);
    a.ltau = -(float)(cfg->precision + 1);
    a.zero_cut = kGnCut;
    const int groups = (K_cap + kGroup - 1) / kGroup;
    a.plan_cnt = plan;
    a.plan_bits = reinterpret_cast<uint32_t*>(plan + groups);
    a.nwords = (a.ntiles + 127) / 128 * 4;
    a.max_list = (a.ntiles + num_splits - 1) / num_splits;
    ga.theta = theta; ga.indices = indices; ga.gstate = gstate;
    ga.tstride = gp_stride(cfg->d, cfg->C, batch->tile[cfg->d - 1]);
    const dim3 grid(groups, num_splits);
    const size_t sm = 2 * (size_t)ga.tstride * 4 + 16 + 16 * 4 + (size_t)a.max_list * 4 + 64;
    SMOE_REQUIRE(sm <= 100 * 1024, "too many tiles per split for the shared-memory tile list: raise num_splits");
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(D, C, DN)                                                                                            \
    {                                                                                                               \
        bwd_plan_kernel<D, C><<<groups, 128, (size_t)a.nwords * 4, st>>>(a);                                        \
        cudaFuncSetAttribute(gn_diag_kernel<D, C, false, DN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        gn_diag_kernel<D, C, false, DN><<<grid, kThreads, sm, st>>>(ga);                                            \
    }
#define CALL(D, C) if (cfg->dense_exec == 1) LAUNCH(D, C, true) else LAUNCH(D, C, false)
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
#undef LAUNCH
    return check_launch("smoe_gn_diag");
}

int smoe_point_gn_diag(const smoe_cfg* cfg, const float* packed, const float* theta, const int32_t* indices,
                       const int32_t* counts, int K_cap, int n_points, const float* gstate, const float* tile_box,
                       int num_splits, float* raw_part, int32_t* plan, void* stream) {
    SMOE_REQUIRE(cfg && packed && theta && indices && counts && gstate && tile_box && raw_part && plan, "null argument");
    SMOE_REQUIRE(K_cap > 0 && num_splits > 0 && num_splits <= 65535, "bad K_cap / num_splits");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    if (int rc = gn_check_cfg(cfg)) return rc;
    const int groups = (K_cap + kGroup - 1) / kGroup;
    const int ntiles = pt_tiles(n_points), nwords = (ntiles + 127) / 128 * 4;
    PtArgs p = {};
    p.cfg = *cfg;
    p.packed = packed; p.counts = counts; p.tile_box = const_cast<float*>(tile_box);
    p.ntiles = ntiles; p.nwords = nwords;
    p.plan_cnt = plan;
    p.plan_bits = reinterpret_cast<uint32_t*>(plan + groups);
    GnArgs ga = {};
    BwdArgs& a = ga.g;
    a.cfg = *cfg;
    a.packed = packed; a.counts = counts;
    a.raw_part = raw_part;
    a.K_cap = K_cap;
    a.num_splits = num_splits;
    a.ntiles = ntiles;
    a.nwords = nwords;
    a.ltau = -(float)(cfg->precision + 1);
    a.zero_cut = kGnCut;
    a.plan_cnt = p.plan_cnt;
    a.plan_bits = p.plan_bits;
    a.max_list = (ntiles + num_splits - 1) / num_splits;
    ga.theta = theta; ga.indices = indices; ga.gstate = gstate; ga.tile_box = tile_box;
    ga.tstride = gq_stride(cfg->d, cfg->C);
    const dim3 grid(groups, num_splits);
    const size_t sm = 2 * (size_t)ga.tstride * 4 + 16 + 16 * 4 + (size_t)a.max_list * 4 + 64;
    SMOE_REQUIRE(sm <= 100 * 1024, "too many tiles per split for the shared-memory tile list: raise num_splits");
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(D, C, DN)                                                                                           \
    {                                                                                                              \
        point_plan_kernel<D, C><<<groups, 128, 0, st>>>(p);                                                        \
        cudaFuncSetAttribute(gn_diag_kernel<D, C, true, DN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        gn_diag_kernel<D, C, true, DN><<<grid, kThreads, sm, st>>>(ga);                                            \
    }
#define CALL(D, C) if (cfg->dense_exec == 1) LAUNCH(D, C, true) else LAUNCH(D, C, false)
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
#undef LAUNCH
    return check_launch("smoe_point_gn_diag");
}

int smoe_gn_diag_scatter(const smoe_cfg* cfg, const float* raw, const int32_t* indices, const int32_t* counts,
                         int K_cap, float* diag, void* stream) {
    SMOE_REQUIRE(cfg && raw && indices && counts && diag, "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    const int P = nparam(cfg->d, cfg->C);
    int nb = (int)(((size_t)K_cap * P + 255) / 256);
    if (nb > 148 * 16) nb = 148 * 16;
    gn_scatter_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(counts, P, raw, indices, diag);
    return check_launch("smoe_gn_diag_scatter");
}

}  // extern "C"
