// Spatial Jacobian of an SMoE at arbitrary points and on a uniform grid: smoe_point_jacobian, smoe_jacobian.
//
// J[c][l] = d r_c / d x_l at every point, from the state smoe_point_forward keeps (qthr, the flag S > 1e-11 in the gr
// plane, the tile-centred x'_l, tile_box) and the forward's r, in one pixel-stationary sweep.  With the gates
// w_k = 2^(q_k - qthr), m_k = [w_k > tau], the experts E_kc = nu'_kc + gamma_k[:, c] . x' and f the flag,
//     J[c][l] = sum_k  m_k w_k gamma_k[l, c]  +  ln2 (m_k w_k E_kc - w_k f r_c) d q_k / d x_l
// -- smoe_point_xgrad's sum with the cotangent g replaced by each unit vector e_c.  Like dL/dx it is the derivative
// of r before clip and has no term for the 0/1 gate decision w > tau (a step).
//
// Chunk staging, culling and skipping are smoe_point_xgrad's: a kernel with q - qthr < -126 contributes exactly 0
// (ex2.approx.ftz), so chunks and kernels are culled against min qthr - 126.5 and a warp skips a kernel whose gates
// are all below -126.  The cut is the exact zero, not tau: sub-threshold kernels still act through the normaliser.
// Per (point, kernel) the gate, ln2 * grad q (d FFMA chains) and E_c are shared by the C x d accumulators, which are
// added in packed-kernel order in every mode (cfg.dense_exec 0, 1, 2 give the same bits).  No float atomics.  A
// tile with a NaN coordinate has a NaN min qthr, so nothing is culled.
//
// smoe_jacobian is the same sweep over a uniform grid, from smoe_forward's pixel state (qthr, the live flag) and
// tile_qmin and its rbuf; the tile geometry and coordinates are recomputed from the batch and the axes exactly as the
// forward computes them.  A thread's 4 pixels differ only in x'_0, so the logit is the forward's parabola, the
// gradient along x'_0 is b + 2 qq00 x'_0 and along every other axis it is affine in x'_0: the parts that do not
// depend on x'_0 are computed once per (thread, kernel).
#include "pt_state.cuh"

namespace smoe {

// resident CTAs per SM: 4 (128 registers a thread) except at (3, 3), whose 36 accumulators, 12 coordinates, 12
// f * r_c and 28-float record need 3 (168 registers)
__host__ __device__ constexpr int jac_ctas(int d, int C) { return (d == 3 && C == 3) ? 3 : 4; }

struct JacArgs {
    smoe_cfg cfg;
    smoe_batch b;              // smoe_jacobian only
    const float* packed;
    const int32_t* counts;
    const float* chunk_bounds;
    const float* state;        // smoe_point_jacobian: [ntiles][pt_stride], as smoe_point_forward left it;
                               // smoe_jacobian: pix [ntiles][pix_stride], as smoe_forward left it
    const float* tile_box;     // smoe_point_jacobian: [ntiles][kTB]; smoe_jacobian: tile_qmin [ntiles]
    const float* ax[3];        // smoe_jacobian only
    const float* r;            // [n][C]: tile order (points) or the grid's rbuf
    float* jac;                // [n][C][d], the layout of r
    int n, ntiles, nt1, nt2;
    float ltau;
};

// Shared memory of a Jacobian sweep: two raw chunks, the compute records, barriers, `red`, `scratch`, chunk list.
struct JacSmem {
    float *raw0, *raw1, *crec;
    uint64_t* bar;
    int *scratch, *clist;
    uint32_t phase0, phase1;
    int par;
};

template <int D, int C>
__device__ __forceinline__ JacSmem jac_smem_init() {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    JacSmem s;
    s.raw0 = reinterpret_cast<float*>(smem_raw);
    s.raw1 = s.raw0 + kChunk * pstride(D, C);
    s.crec = s.raw1 + kChunk * pstride(D, C);
    s.bar = reinterpret_cast<uint64_t*>(s.crec + kChunk * Rec<D, C>::RC);
    s.scratch = reinterpret_cast<int*>(reinterpret_cast<float*>(s.bar + 2) + 32);
    s.clist = s.scratch + 8;
    if (threadIdx.x == 0) {
        mbar_init(&s.bar[0], 1);
        mbar_init(&s.bar[1], 1);
        fence_barrier_init();
    }
    __syncthreads();
    s.phase0 = s.phase1 = 0;
    s.par = 0;
    return s;
}

// One tile's sweep, smoe_point_xgrad's staging and culling: the ordered list of chunks whose bound over the box
// (ctr, half) reaches `thr`, TMA double buffering, per-kernel culling and ordered compaction; body(rec) is called for
// every kernel that can matter, in packed order, with its tile-centred record.  Ends with a CTA barrier.
template <int D, int C, class Body>
__device__ __forceinline__ void jac_sweep(const JacArgs& a, JacSmem& s, int K, bool cull, const float (&ctr)[3],
                                          const float (&half)[3], float thr, Body&& body) {
    using R = Rec<D, C>;
    constexpr int PK = pstride(D, C);
    const int tid = threadIdx.x;
    const int nchunks = (K + kChunk - 1) / kChunk;
    auto issue = [&](int ci, int buf) {
        int nk = min(kChunk, K - ci * kChunk);
        uint32_t bytes = (uint32_t)nk * PK * 4u;
        fence_proxy_async();
        mbar_expect_tx(&s.bar[buf], bytes);
        tma_load_1d(buf ? s.raw1 : s.raw0, a.packed + (size_t)ci * kChunk * PK, bytes, &s.bar[buf]);
    };
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
        const int pos = cta_compact(need, s.scratch, s.par, &tot);
        if (need) s.clist[nlist + pos] = ci;
        nlist += tot;
    }
    __syncthreads();

    if (tid == 0 && nlist > 0) {
        issue(s.clist[0], 0);
        if (nlist > 1) issue(s.clist[1], 1);
    }
    for (int li = 0; li < nlist; ++li) {
        const int buf = li & 1;
        const int ci = s.clist[li];
        const int nk = min(kChunk, K - ci * kChunk);
        if (buf) { mbar_wait(&s.bar[1], s.phase1); s.phase1 ^= 1; } else { mbar_wait(&s.bar[0], s.phase0); s.phase0 ^= 1; }
        const float* raw = (buf ? s.raw1 : s.raw0) + tid * PK;
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
        const int pos = cta_compact(need, s.scratch, s.par, &nneed);
        if (need) transform_record<D, C>(raw, mu, ctr, 0, s.crec + pos * R::RC);
        __syncthreads();
        if (tid == 0 && li + 2 < nlist) issue(s.clist[li + 2], buf);
        for (int kk = 0; kk < nneed; ++kk) body(s.crec + kk * R::RC);
    }
    __syncthreads();          // the next tile rebuilds `clist` and re-uses `crec`
}

// record -> registers: the geometry part (NG4 float4), or the rest up to the original index
template <int D, int C>
__device__ __forceinline__ void load_rec(const float* rc, float (&f)[Rec<D, C>::RC], int from, int to) {
    const float4* r4 = reinterpret_cast<const float4*>(rc);
#pragma unroll
    for (int j = from; j < to; ++j) {
        float4 v = r4[j];
        f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
    }
}

template <int D, int C>
__global__ void __launch_bounds__(kThreadsF, jac_ctas(D, C)) point_jacobian_kernel(const JacArgs a) {
    using R = Rec<D, C>;
    constexpr int PPT = kPixPerThread;
    constexpr int tstride = pt_stride(D, C);
    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int mode = a.cfg.dense_exec;
    const bool cull = mode == 0, skip = mode != 1;
    const float ltau = a.ltau;
    JacSmem s = jac_smem_init<D, C>();

    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        const float* tb = a.tile_box + (size_t)tile * kTB;
        float ctr[3], half[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) { ctr[i] = tb[i]; half[i] = tb[3 + i]; }
        const float thr = tb[6] - 126.5f;                     // NaN for a NaN box: nothing is culled
        const float* tp = a.state + (size_t)tile * tstride;
        float x[PPT][D], qthr[PPT], fr[PPT][C], jac[PPT][C][D];
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int j = p * kThreadsF + tid;
            const int gi = tile * SMOE_TPIX + j;
            qthr[p] = tp[PP_QTHR * SMOE_TPIX + j];
            const bool live = tp[PP_GR * SMOE_TPIX + j] != 0.f;        // 0 past the last point too
#pragma unroll
            for (int c = 0; c < C; ++c) {
                fr[p][c] = live ? a.r[(size_t)gi * C + c] : 0.f;
#pragma unroll
                for (int l = 0; l < D; ++l) jac[p][c][l] = 0.f;
            }
#pragma unroll
            for (int l = 0; l < D; ++l) x[p][l] = tp[(pp_x(C) + l) * SMOE_TPIX + j];
        }

        jac_sweep<D, C>(a, s, K, cull, ctr, half, thr, [&](const float* rc) {
            float f[R::RC];
            load_rec<D, C>(rc, f, 0, R::NG4);
            float dq[PPT];
            float dmax = -INFINITY;
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                dq[p] = point_logit<D, C>(f, x[p]) - qthr[p];
                dmax = fmaxf(dmax, dq[p]);
            }
            if (skip && !__any_sync(0xffffffffu, dmax >= -126.f)) return;
            load_rec<D, C>(rc, f, R::NG4, (R::OK + 4) / 4);
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                const float w = ex2f(dq[p]);
                const float wm = dq[p] > ltau ? w : 0.f;
                float gq[D];
#pragma unroll
                for (int l = 0; l < D; ++l) {
                    // d q / d x'_l = ql_l + 2 qq_ll x'_l + sum_{m != l} qq_lm x'_m (off-diagonals stored doubled)
                    float g = fmaf(2.f * f[R::OQ + ut(D, l, l)], x[p][l], f[R::OL + l]);
#pragma unroll
                    for (int m = 0; m < D; ++m)
                        if (m != l) g = fmaf(f[R::OQ + (m > l ? ut(D, l, m) : ut(D, m, l))], x[p][m], g);
                    gq[l] = g * kLn2;
                }
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    float E = f[R::ONU + c];
#pragma unroll
                    for (int l = 0; l < D; ++l) E = fmaf(f[R::OGA + l * C + c], x[p][l], E);
                    const float t = fmaf(wm, E, -w * fr[p][c]);
#pragma unroll
                    for (int l = 0; l < D; ++l) jac[p][c][l] += fmaf(t, gq[l], wm * f[R::OGA + l * C + c]);
                }
            }
        });
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int gi = tile * SMOE_TPIX + p * kThreadsF + tid;
            if (gi < a.n)
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int l = 0; l < D; ++l) a.jac[((size_t)gi * C + c) * D + l] = jac[p][c][l];
        }
    }
}

// The grid sweep: tile geometry, pixel coordinates and the logit as forward_kernel computes them.
template <int D, int C>
__global__ void __launch_bounds__(kThreadsF, jac_ctas(D, C)) grid_jacobian_kernel(const JacArgs a) {
    using R = Rec<D, C>;
    constexpr int PPT = kPixPerThread;
    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int mode = a.cfg.dense_exec;
    const bool cull = mode == 0, skip = mode != 1;
    const float ltau = a.ltau;
    const int e1 = a.b.tile[1], e2 = a.b.tile[2];
    const int tstride = pix_stride(D, C, a.b.tile[D - 1]);
    JacSmem s = jac_smem_init<D, C>();

    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        int tt[3];
        tt[2] = tile % a.nt2;
        tt[1] = (tile / a.nt2) % a.nt1;
        tt[0] = tile / (a.nt2 * a.nt1);
        int lo[3], hi[3];
        float ctr[3], half[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            lo[i] = a.b.origin[i] + tt[i] * a.b.tile[i];
            hi[i] = min(lo[i] + a.b.tile[i], a.b.origin[i] + a.b.extent[i]) - 1;
            const float c0 = (i < D) ? a.ax[i][lo[i]] : 0.f, c1 = (i < D) ? a.ax[i][hi[i]] : 0.f;
            ctr[i] = 0.5f * (c0 + c1);
            half[i] = 0.5f * (c1 - c0) * 1.0001f + 1e-7f;
        }
        const float thr = a.tile_box[tile] - 126.5f;          // tile_qmin
        const float* tp = a.state + (size_t)tile * tstride;
        const int i2 = tid % e2, i1 = (tid / e2) % e1;
        const int g1 = lo[1] + i1, g2 = lo[2] + i2;
        float x0[PPT], xs[3] = {0.f, 0.f, 0.f}, qthr[PPT], fr[PPT][C], jac[PPT][C][D];
        int gpix[PPT];
        unsigned okmask = 0;
        if (D > 1) xs[1] = a.ax[1][min(g1, hi[1])] - ctr[1];
        if (D > 2) xs[2] = a.ax[2][min(g2, hi[2])] - ctr[2];
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int j = p * kThreadsF + tid;
            const int g0 = lo[0] + j / (e2 * e1);
            const bool ok = g0 <= hi[0] && g1 <= hi[1] && g2 <= hi[2];
            if (ok) okmask |= 1u << p;
            gpix[p] = ok ? (g0 * a.b.dims[1] + g1) * a.b.dims[2] + g2 : 0;
            x0[p] = a.ax[0][min(g0, hi[0])] - ctr[0];
            qthr[p] = tp[PL_QTHR * SMOE_TPIX + j];                     // +inf outside the batch: w = 0
            const bool live = ok && tp[PL_GR * SMOE_TPIX + j] != 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                fr[p][c] = live ? a.r[(size_t)gpix[p] * C + c] : 0.f;
#pragma unroll
                for (int l = 0; l < D; ++l) jac[p][c][l] = 0.f;
            }
        }

        jac_sweep<D, C>(a, s, K, cull, ctr, half, thr, [&](const float* rc) {
            float f[R::RC];
            load_rec<D, C>(rc, f, 0, R::NG4);
            // q = c + (b + qq00 x'_0) x'_0 with c, b from the row coordinates (forward.cu, parabola)
            float cq = f[R::OC];
#pragma unroll
            for (int l = 1; l < D; ++l) {
                float t = f[R::OL + l];
#pragma unroll
                for (int m = l; m < D; ++m) t = fmaf(f[R::OQ + ut(D, l, m)], xs[m], t);
                cq = fmaf(t, xs[l], cq);
            }
            float bq = f[R::OL + 0];
#pragma unroll
            for (int m = 1; m < D; ++m) bq = fmaf(f[R::OQ + ut(D, 0, m)], xs[m], bq);
            float dq[PPT];
            float dmax = -INFINITY;
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                dq[p] = fmaf(fmaf(f[R::OQ], x0[p], bq), x0[p], cq) - qthr[p];
                dmax = fmaxf(dmax, dq[p]);
            }
            if (skip && !__any_sync(0xffffffffu, dmax >= -126.f)) return;
            load_rec<D, C>(rc, f, R::NG4, (R::OK + 4) / 4);
            // d q / d x'_l for l >= 1: a_l + qq_0l x'_0 (qq_0l stored doubled); d q / d x'_0 = b + 2 qq00 x'_0
            float ga[D];
#pragma unroll
            for (int l = 1; l < D; ++l) {
                float g = fmaf(2.f * f[R::OQ + ut(D, l, l)], xs[l], f[R::OL + l]);
#pragma unroll
                for (int m = 1; m < D; ++m)
                    if (m != l) g = fmaf(f[R::OQ + (m > l ? ut(D, l, m) : ut(D, m, l))], xs[m], g);
                ga[l] = g;
            }
            float Eb[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                Eb[c] = f[R::ONU + c];
#pragma unroll
                for (int l = 1; l < D; ++l) Eb[c] = fmaf(f[R::OGA + l * C + c], xs[l], Eb[c]);
            }
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                const float w = ex2f(dq[p]);
                const float wm = dq[p] > ltau ? w : 0.f;
                float gq[D];
                gq[0] = fmaf(2.f * f[R::OQ], x0[p], bq) * kLn2;
#pragma unroll
                for (int l = 1; l < D; ++l) gq[l] = fmaf(f[R::OQ + ut(D, 0, l)], x0[p], ga[l]) * kLn2;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float E = fmaf(f[R::OGA + c], x0[p], Eb[c]);
                    const float t = fmaf(wm, E, -w * fr[p][c]);
#pragma unroll
                    for (int l = 0; l < D; ++l) jac[p][c][l] += fmaf(t, gq[l], wm * f[R::OGA + l * C + c]);
                }
            }
        });
#pragma unroll
        for (int p = 0; p < PPT; ++p)
            if ((okmask >> p) & 1u)
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int l = 0; l < D; ++l) a.jac[((size_t)gpix[p] * C + c) * D + l] = jac[p][c][l];
    }
}

}  // namespace smoe

using namespace smoe;

extern "C" {

int smoe_point_jacobian(const smoe_cfg* cfg, const float* packed, const int32_t* counts, const float* chunk_bounds,
                        int K_cap, int n_points, const float* state, const float* tile_box, const float* r, float* jac,
                        void* stream) {
    SMOE_REQUIRE(cfg && packed && counts && chunk_bounds && state && tile_box && r && jac, "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the point kernels");
    JacArgs a = {};
    a.cfg = *cfg;
    a.packed = packed; a.counts = counts; a.chunk_bounds = chunk_bounds;
    a.state = state; a.tile_box = tile_box; a.r = r; a.jac = jac;
    a.n = n_points;
    a.ntiles = pt_tiles(n_points);
    a.ltau = -(float)(cfg->precision + 1);
    const int max_chunks = (K_cap + kChunk - 1) / kChunk;
    const int cap = jac_ctas(cfg->d, cfg->C) * pt_sms();
    const int grid = a.ntiles < cap ? a.ntiles : cap;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C)                                                                                              \
    {                                                                                                           \
        size_t sm = pt_sweep_smem_bytes<D, C>(max_chunks);                                                      \
        SMOE_REQUIRE(sm <= 200 * 1024, "too many kernel chunks for the shared-memory chunk list");              \
        cudaFuncSetAttribute(point_jacobian_kernel<D, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        point_jacobian_kernel<D, C><<<grid, kThreadsF, sm, st>>>(a);                                            \
    }
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_point_jacobian");
}

int smoe_jacobian(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const int32_t* counts,
                  const float* chunk_bounds, int K_cap, const float* pix, const float* tile_qmin, const float* ax0,
                  const float* ax1, const float* ax2, const float* rbuf, float* jac, void* stream) {
    SMOE_REQUIRE(cfg && batch && packed && counts && chunk_bounds && pix && tile_qmin && ax0 && ax1 && rbuf && jac,
                 "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    SMOE_REQUIRE(cfg->d == 2 || ax2, "ax2 required for d == 3");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the Jacobian");
    SMOE_REQUIRE(batch->tile[0] * batch->tile[1] * batch->tile[2] == SMOE_TPIX, "tile product must be SMOE_TPIX");
    SMOE_REQUIRE(kThreadsF % (batch->tile[1] * batch->tile[2]) == 0 && batch->tile[cfg->d - 1] % 4 == 0,
                 "tile[1]*tile[2] must divide 128 and the last tile extent must be a multiple of 4");
    SMOE_REQUIRE(batch->halo == 0, "the Jacobian needs a batch without halo");
    for (int i = 0; i < 3; ++i)
        SMOE_REQUIRE(batch->extent[i] > 0 && batch->origin[i] >= 0 && batch->origin[i] + batch->extent[i] <= batch->dims[i],
                     "batch rectangle outside the image");
    SMOE_REQUIRE(cfg->d == 3 || (batch->dims[2] == 1 && batch->tile[2] == 1), "d == 2 needs dims[2] == tile[2] == 1");
    SMOE_REQUIRE((long long)batch->dims[0] * batch->dims[1] * batch->dims[2] < (1ll << 31), "more than 2^31 pixels");
    JacArgs a = {};
    a.cfg = *cfg;
    a.b = *batch;
    a.packed = packed; a.counts = counts; a.chunk_bounds = chunk_bounds;
    a.state = pix; a.tile_box = tile_qmin; a.r = rbuf; a.jac = jac;
    a.ax[0] = ax0; a.ax[1] = ax1; a.ax[2] = ax2 ? ax2 : ax0;
    a.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    a.ntiles = smoe_num_tiles(batch);
    a.ltau = -(float)(cfg->precision + 1);
    const int max_chunks = (K_cap + kChunk - 1) / kChunk;
    const int cap = jac_ctas(cfg->d, cfg->C) * pt_sms();
    const int grid = a.ntiles < cap ? a.ntiles : cap;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C)                                                                                              \
    {                                                                                                           \
        size_t sm = pt_sweep_smem_bytes<D, C>(max_chunks);                                                      \
        SMOE_REQUIRE(sm <= 200 * 1024, "too many kernel chunks for the shared-memory chunk list");              \
        cudaFuncSetAttribute(grid_jacobian_kernel<D, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        grid_jacobian_kernel<D, C><<<grid, kThreadsF, sm, st>>>(a);                                            \
    }
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_jacobian");
}

}  // extern "C"
