// Forward-mode derivatives of an SMoE: smoe_pack_tangent, smoe_jvp (uniform grid), smoe_point_jvp (points).
//
// For a tangent (v, xdot) of the parameters and the points, dr = (d r / d theta) v + (d r / d x) xdot, the derivative
// of r before clip.  With jacobian.cu's notation (gates w_k = 2^(q_k - qthr), m_k = [w_k > tau], experts
// E_kc = nu'_kc + gamma_k[:, c] . x', f the flag S > 1e-11 the forward leaves in the gr plane), a tangent logit dq_k
// (log2 units) and tangent experts dE_kc per (point, kernel) give
//     dr_c = sum_k  m_k w_k dE_kc  +  ln2 dq_k (m_k w_k E_kc - w_k f r_c)
// -- the Jacobian's sum with grad q replaced by dq and gamma by dE: C accumulators per point, not C x d.
//   parameter tangents: smoe_pack_tangent writes one raw tangent record per packed row (d mu, d Qm, d c0, d nu,
//     d gamma); the sweep stages it next to the primal chunk and re-centres it per tile (transform_tangent), so dq is
//     the tile-centred quadratic of the tangent record and dE_c = dnu'_c + dgamma_c . x'.
//   point tangents (points only): dq += grad q . xdot and dE_c += gamma_c . xdot, inside the same per-pair terms.
// Kernels dropped by smoe_pack (pi <= 0) have no record, so their tangents have no effect; the 0/1 decision w > tau
// contributes no term.  Staging, culling and skipping are the Jacobian's (jac_sweep): the exact-zero cut on the primal
// gates, where a pair contributes exactly 0, and a fixed packed-kernel order, so cfg.dense_exec 0, 1 and 2 give the
// same bits.  No float atomics, no host synchronisation.
#include "jac_sweep.cuh"

namespace smoe {

// Resident CTAs per SM.  With parameter tangents the sweep also holds two raw tangent chunks and their re-centred
// records in shared memory (jvp_smem_bytes): 37 / 57 / 57 / 81 KB at (2,1) / (2,3) / (3,1) / (3,3) for up to 32K
// kernels, so 4 / 3 / 3 / 2 CTAs fit the 228 KB of an SM.  With point tangents alone the sweep has the Jacobian's
// shared memory and fewer accumulators: 4 CTAs.
__host__ __device__ constexpr int jvp_ctas(int d, int C, bool pt) {
    return !pt ? 4 : (d == 2 && C == 1) ? 4 : (d == 3 && C == 3) ? 2 : 3;
}

template <int D, int C>
__host__ __device__ constexpr int jvp_tan_floats() { return 2 * kChunk * tan_stride(D, C) + kChunk * Rec<D, C>::RC; }

template <int D, int C>
static size_t jvp_smem_bytes(int max_chunks, bool pt) {
    return pt_sweep_smem_bytes<D, C>(max_chunks) + (pt ? (size_t)jvp_tan_floats<D, C>() * 4 : 0);
}

struct JvpArgs {
    JacArgs j;                 // primal state, as for the Jacobian (j.jac unused)
    const float* tangent;      // [K_cap][tan_stride] packed order, or NULL
    const float* dx;           // [n][d] tile order, or NULL (points only)
    float* dr;                 // [n][C] in the layout of r
};

template <int D, int C, bool PT>
__device__ __forceinline__ JacSmem jvp_smem_init(const float* tangent) {
    JacSmem s = jac_smem_init<D, C, PT ? jvp_tan_floats<D, C>() : 0>();
    if (PT) {
        s.tangent = tangent;
        s.traw0 = s.crec + kChunk * Rec<D, C>::RC;
        s.traw1 = s.traw0 + kChunk * tan_stride(D, C);
        s.trec = s.traw1 + kChunk * tan_stride(D, C);
    }
    return s;
}

// ---- smoe_pack_tangent: one raw tangent record per packed row ---------------------------------------------------
template <int D, int C>
__global__ void __launch_bounds__(256) pack_tangent_kernel(smoe_cfg cfg, const float* __restrict__ theta,
                                                           const float* __restrict__ dtheta,
                                                           const int32_t* __restrict__ indices,
                                                           const int32_t* __restrict__ counts, float* __restrict__ tangent) {
    constexpr int P = nparam(D, C), TS = tan_stride(D, C);
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= counts[0]) return;
    const size_t i = (size_t)indices[j];
    const float* row = theta + i * P;
    const float* drow = dtheta + i * P;
    float out[TS];
    float A[D][D], dA[D][D];
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
        for (int m = 0; m < D; ++m) {
            const bool lo = m <= l || cfg.train_inverse_cov;       // stage_record: lower part, symmetric for Qm = A
            const int src = off_A(D, C) + (m <= l ? lt(l, m) : lt(m, l));
            A[l][m] = lo ? row[src] : 0.f;
            dA[l][m] = lo ? drow[src] : 0.f;
        }
#pragma unroll
    for (int l = 0; l < D; ++l) out[off_mu(D, C) + l] = drow[off_mu(D, C) + l];
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
        for (int m = l; m < D; ++m) {
            float dq;
            if (cfg.train_inverse_cov) {
                dq = 0.5f * (dA[l][m] + dA[m][l]);
            } else {
                dq = 0.f;
#pragma unroll
                for (int k = 0; k < D; ++k) dq = fmaf(dA[l][k], A[m][k], fmaf(A[l][k], dA[m][k], dq));   // d (A A^T)
            }
            out[off_A(D, C) + ut(D, l, m)] = kHalfLog2e * dq;
        }
    // c0 = log2 |pi det(A) / sqrt(2 pi)^D|: d c0 = (dpi / pi + sum_l dA_ll / A_ll) / ln2, for either sign of A_ll.  A
    // kernel with a zero A_ll has c0 = -inf and no gate anywhere: its d c0 is 0 rather than inf
    float dc = drow[off_pi(D, C)] / row[off_pi(D, C)];
    bool dead = false;
    if (cfg.use_determinant) {
#pragma unroll
        for (int l = 0; l < D; ++l) {
            dc += dA[l][l] / A[l][l];
            dead |= A[l][l] == 0.f;
        }
    }
    out[off_pi(D, C)] = dead ? 0.f : dc * 1.44269504088896340736f;
#pragma unroll
    for (int c = 0; c < C; ++c) out[off_nu(D, C) + c] = drow[off_nu(D, C) + c];
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            float g = drow[off_ga(D, C) + l * C + c];
            if (!cfg.train_gammas) g = 0.f;
            if (cfg.use_yuv && cfg.train_gammas && cfg.only_y_gamma && c > 0) g = 0.f;
            out[off_ga(D, C) + l * C + c] = g;
        }
#pragma unroll
    for (int q = P; q < TS; ++q) out[q] = 0.f;
    float4* d4 = reinterpret_cast<float4*>(tangent + (size_t)j * TS);
#pragma unroll
    for (int q = 0; q < TS / 4; ++q) d4[q] = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
}

// ---- the point sweep ------------------------------------------------------------------------------------------
// PT: parameter tangents; XT: point tangents (at least one)
template <int D, int C, bool PT, bool XT>
__global__ void __launch_bounds__(kThreadsF, jvp_ctas(D, C, PT)) point_jvp_kernel(const JvpArgs ja) {
    using R = Rec<D, C>;
    constexpr int PPT = kPixPerThread;
    constexpr int tstride = pt_stride(D, C);
    const JacArgs& a = ja.j;
    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int mode = a.cfg.dense_exec;
    const bool cull = mode == 0, skip = mode != 1;
    const float ltau = a.ltau;
    JacSmem s = jvp_smem_init<D, C, PT>(ja.tangent);

    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        const float* tb = a.tile_box + (size_t)tile * kTB;
        float ctr[3], half[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) { ctr[i] = tb[i]; half[i] = tb[3 + i]; }
        const float thr = tb[6] - 126.5f;                     // NaN for a NaN box: nothing is culled
        const float* tp = a.state + (size_t)tile * tstride;
        float x[PPT][D], xd[PPT][D], qthr[PPT], fr[PPT][C], acc[PPT][C];
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int j = p * kThreadsF + tid;
            const int gi = tile * SMOE_TPIX + j;
            qthr[p] = tp[PP_QTHR * SMOE_TPIX + j];
            const bool live = tp[PP_GR * SMOE_TPIX + j] != 0.f;        // 0 past the last point too
#pragma unroll
            for (int c = 0; c < C; ++c) {
                fr[p][c] = live ? a.r[(size_t)gi * C + c] : 0.f;
                acc[p][c] = 0.f;
            }
#pragma unroll
            for (int l = 0; l < D; ++l) {
                x[p][l] = tp[(pp_x(C) + l) * SMOE_TPIX + j];
                xd[p][l] = (XT && gi < a.n) ? ja.dx[(size_t)gi * D + l] : 0.f;
            }
        }

        auto pair_terms = [&](const float* rc, const float* tr) {
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
            float t[R::RC];
            if (PT) load_rec<D, C>(tr, t, 0, (R::OK + 4) / 4);
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                const float w = ex2f(dq[p]);
                const float wm = dq[p] > ltau ? w : 0.f;
                float tq = PT ? point_logit<D, C>(t, x[p]) : 0.f;
                if (XT) {
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        float g = fmaf(2.f * f[R::OQ + ut(D, l, l)], x[p][l], f[R::OL + l]);
#pragma unroll
                        for (int m = 0; m < D; ++m)
                            if (m != l) g = fmaf(f[R::OQ + (m > l ? ut(D, l, m) : ut(D, m, l))], x[p][m], g);
                        tq = fmaf(g, xd[p][l], tq);
                    }
                }
                tq *= kLn2;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    float E = f[R::ONU + c], dE = PT ? t[R::ONU + c] : 0.f;
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        E = fmaf(f[R::OGA + l * C + c], x[p][l], E);
                        if (PT) dE = fmaf(t[R::OGA + l * C + c], x[p][l], dE);
                        if (XT) dE = fmaf(f[R::OGA + l * C + c], xd[p][l], dE);
                    }
                    const float u = fmaf(wm, E, -w * fr[p][c]);
                    acc[p][c] += fmaf(u, tq, wm * dE);
                }
            }
        };
        if constexpr (PT)
            jac_sweep<D, C, true>(a, s, K, cull, ctr, half, thr, pair_terms);
        else
            jac_sweep<D, C>(a, s, K, cull, ctr, half, thr, [&](const float* rc) { pair_terms(rc, rc); });
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int gi = tile * SMOE_TPIX + p * kThreadsF + tid;
            if (gi < a.n)
#pragma unroll
                for (int c = 0; c < C; ++c) ja.dr[(size_t)gi * C + c] = acc[p][c];
        }
    }
}

// ---- the grid sweep (parameter tangents): tile geometry, coordinates and logit as forward_kernel computes them ----
template <int D, int C>
__global__ void __launch_bounds__(kThreadsF, jvp_ctas(D, C, true)) grid_jvp_kernel(const JvpArgs ja) {
    using R = Rec<D, C>;
    constexpr int PPT = kPixPerThread;
    const JacArgs& a = ja.j;
    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int mode = a.cfg.dense_exec;
    const bool cull = mode == 0, skip = mode != 1;
    const float ltau = a.ltau;
    const int e1 = a.b.tile[1], e2 = a.b.tile[2];
    const int tstride = pix_stride(D, C, a.b.tile[D - 1]);
    JacSmem s = jvp_smem_init<D, C, true>(ja.tangent);

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
        float x0[PPT], xs[3] = {0.f, 0.f, 0.f}, qthr[PPT], fr[PPT][C], acc[PPT][C];
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
                acc[p][c] = 0.f;
            }
        }

        jac_sweep<D, C, true>(a, s, K, cull, ctr, half, thr, [&](const float* rc, const float* tr) {
            float f[R::RC];
            load_rec<D, C>(rc, f, 0, R::NG4);
            // q = c + (b + qq00 x'_0) x'_0 with c, b from the row coordinates (forward.cu, parabola); dq likewise
            float cq = f[R::OC];
#pragma unroll
            for (int l = 1; l < D; ++l) {
                float u = f[R::OL + l];
#pragma unroll
                for (int m = l; m < D; ++m) u = fmaf(f[R::OQ + ut(D, l, m)], xs[m], u);
                cq = fmaf(u, xs[l], cq);
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
            float t[R::RC];
            load_rec<D, C>(tr, t, 0, (R::OK + 4) / 4);
            float tc = t[R::OC];
#pragma unroll
            for (int l = 1; l < D; ++l) {
                float u = t[R::OL + l];
#pragma unroll
                for (int m = l; m < D; ++m) u = fmaf(t[R::OQ + ut(D, l, m)], xs[m], u);
                tc = fmaf(u, xs[l], tc);
            }
            float tb = t[R::OL + 0];
#pragma unroll
            for (int m = 1; m < D; ++m) tb = fmaf(t[R::OQ + ut(D, 0, m)], xs[m], tb);
            float Eb[C], dEb[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                Eb[c] = f[R::ONU + c];
                dEb[c] = t[R::ONU + c];
#pragma unroll
                for (int l = 1; l < D; ++l) {
                    Eb[c] = fmaf(f[R::OGA + l * C + c], xs[l], Eb[c]);
                    dEb[c] = fmaf(t[R::OGA + l * C + c], xs[l], dEb[c]);
                }
            }
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                const float w = ex2f(dq[p]);
                const float wm = dq[p] > ltau ? w : 0.f;
                const float tq = fmaf(fmaf(t[R::OQ], x0[p], tb), x0[p], tc) * kLn2;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float E = fmaf(f[R::OGA + c], x0[p], Eb[c]);
                    const float dE = fmaf(t[R::OGA + c], x0[p], dEb[c]);
                    const float u = fmaf(wm, E, -w * fr[p][c]);
                    acc[p][c] += fmaf(u, tq, wm * dE);
                }
            }
        });
#pragma unroll
        for (int p = 0; p < PPT; ++p)
            if ((okmask >> p) & 1u)
#pragma unroll
                for (int c = 0; c < C; ++c) ja.dr[(size_t)gpix[p] * C + c] = acc[p][c];
    }
}

}  // namespace smoe

using namespace smoe;

extern "C" {

int smoe_tangent_stride(int d, int C) { return tan_stride(d, C); }

int smoe_pack_tangent(const smoe_cfg* cfg, const float* theta, const float* dtheta, const int32_t* indices,
                      const int32_t* counts, int K_cap, float* tangent, void* stream) {
    SMOE_REQUIRE(cfg && theta && dtheta && indices && counts && tangent, "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the JVP");
    SMOE_REQUIRE(cfg->quantization_mode == 0 && !cfg->quantize_pis && !cfg->use_diff_center,
                 "the tangent of fake-quantised or diff-centre parameters is not supported");
    const int blocks = (K_cap + 255) / 256;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C) pack_tangent_kernel<D, C><<<blocks, 256, 0, st>>>(*cfg, theta, dtheta, indices, counts, tangent);
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_pack_tangent");
}

int smoe_point_jvp(const smoe_cfg* cfg, const float* packed, const float* tangent, const int32_t* counts,
                   const float* chunk_bounds, int K_cap, int n_points, const float* state, const float* tile_box,
                   const float* r, const float* dpoints, float* dr, void* stream) {
    SMOE_REQUIRE(cfg && packed && counts && chunk_bounds && state && tile_box && r && dr, "null argument");
    SMOE_REQUIRE(tangent || dpoints, "at least one of the parameter and point tangents is needed");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE(n_points > 0 && n_points <= SMOE_POINT_MAX, "n_points must be in [1, SMOE_POINT_MAX]");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the point kernels");
    JvpArgs a = {};
    a.j.cfg = *cfg;
    a.j.packed = packed; a.j.counts = counts; a.j.chunk_bounds = chunk_bounds;
    a.j.state = state; a.j.tile_box = tile_box; a.j.r = r;
    a.j.n = n_points;
    a.j.ntiles = pt_tiles(n_points);
    a.j.ltau = -(float)(cfg->precision + 1);
    a.tangent = tangent; a.dx = dpoints; a.dr = dr;
    const int max_chunks = (K_cap + kChunk - 1) / kChunk;
    const bool pt = tangent != nullptr, xt = dpoints != nullptr;
    const int cap = jvp_ctas(cfg->d, cfg->C, pt) * pt_sms();
    const int grid = a.j.ntiles < cap ? a.j.ntiles : cap;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(D, C, PT, XT)                                                                                       \
    {                                                                                                              \
        size_t sm = jvp_smem_bytes<D, C>(max_chunks, PT);                                                          \
        SMOE_REQUIRE(sm <= 200 * 1024, "too many kernel chunks for the shared-memory chunk list");                 \
        cudaFuncSetAttribute(point_jvp_kernel<D, C, PT, XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        point_jvp_kernel<D, C, PT, XT><<<grid, kThreadsF, sm, st>>>(a);                                            \
    }
#define CALL(D, C)                              \
    if (pt && xt) LAUNCH(D, C, true, true)      \
    else if (pt) LAUNCH(D, C, true, false)      \
    else LAUNCH(D, C, false, true)
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
#undef LAUNCH
    return check_launch("smoe_point_jvp");
}

int smoe_jvp(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const float* tangent,
             const int32_t* counts, const float* chunk_bounds, int K_cap, const float* pix, const float* tile_qmin,
             const float* ax0, const float* ax1, const float* ax2, const float* rbuf, float* dr, void* stream) {
    SMOE_REQUIRE(cfg && batch && packed && tangent && counts && chunk_bounds && pix && tile_qmin && ax0 && ax1 &&
                     rbuf && dr,
                 "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    SMOE_REQUIRE(cfg->d == 2 || ax2, "ax2 required for d == 3");
    SMOE_REQUIRE(cfg->eps_bits == 0, "eps_bits is not supported by the JVP");
    SMOE_REQUIRE(batch->tile[0] * batch->tile[1] * batch->tile[2] == SMOE_TPIX, "tile product must be SMOE_TPIX");
    SMOE_REQUIRE(kThreadsF % (batch->tile[1] * batch->tile[2]) == 0 && batch->tile[cfg->d - 1] % 4 == 0,
                 "tile[1]*tile[2] must divide 128 and the last tile extent must be a multiple of 4");
    SMOE_REQUIRE(batch->halo == 0, "the JVP needs a batch without halo");
    for (int i = 0; i < 3; ++i)
        SMOE_REQUIRE(batch->extent[i] > 0 && batch->origin[i] >= 0 && batch->origin[i] + batch->extent[i] <= batch->dims[i],
                     "batch rectangle outside the image");
    SMOE_REQUIRE(cfg->d == 3 || (batch->dims[2] == 1 && batch->tile[2] == 1), "d == 2 needs dims[2] == tile[2] == 1");
    SMOE_REQUIRE((long long)batch->dims[0] * batch->dims[1] * batch->dims[2] < (1ll << 31), "more than 2^31 pixels");
    JvpArgs a = {};
    a.j.cfg = *cfg;
    a.j.b = *batch;
    a.j.packed = packed; a.j.counts = counts; a.j.chunk_bounds = chunk_bounds;
    a.j.state = pix; a.j.tile_box = tile_qmin; a.j.r = rbuf;
    a.j.ax[0] = ax0; a.j.ax[1] = ax1; a.j.ax[2] = ax2 ? ax2 : ax0;
    a.j.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.j.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    a.j.ntiles = smoe_num_tiles(batch);
    a.j.ltau = -(float)(cfg->precision + 1);
    a.tangent = tangent; a.dr = dr;
    const int max_chunks = (K_cap + kChunk - 1) / kChunk;
    const int cap = jvp_ctas(cfg->d, cfg->C, true) * pt_sms();
    const int grid = a.j.ntiles < cap ? a.j.ntiles : cap;
    cudaStream_t st = (cudaStream_t)stream;
#define CALL(D, C)                                                                                         \
    {                                                                                                      \
        size_t sm = jvp_smem_bytes<D, C>(max_chunks, true);                                                \
        SMOE_REQUIRE(sm <= 200 * 1024, "too many kernel chunks for the shared-memory chunk list");         \
        cudaFuncSetAttribute(grid_jvp_kernel<D, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        grid_jvp_kernel<D, C><<<grid, kThreadsF, sm, st>>>(a);                                            \
    }
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
    return check_launch("smoe_jvp");
}

}  // extern "C"
