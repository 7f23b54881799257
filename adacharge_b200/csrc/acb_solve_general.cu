// General ("streaming") solve path for instances that do not fit on one SM (e.g. the
// 1000-EVSE site of BASELINE config 5): the same ADMM split and the same rigorous
// duality-gap stopping rule as acb_solve_kernel.cuh, with the state in HBM/L2 and one
// kernel per phase over the whole batch:
//   k_rows  block per (group of electrically identical EVSEs, instance): x, over-relaxed v,
//           box ∩ energy projection (warp per row, Newton on the multiplier), group sums; the rate
//           bounds come straight from the session table (nothing but v is streamed)
//   k_cols_it  block per (32-period tile, instance): the Woodbury solve in factored, rank-reduced form
//           b = C sa - (d/rho) g,  h = -(b/(d/rho) + Ur diag(1/(d/rho+lam) - 1/(d/rho)) Ur' b),  Kx = (g - h)/rho,
//           hg = C'h - c as four shared-memory blocked products, then the coupling-row v update for the tile
//   k_level one warp per instance: peak-epigraph level of the aggregate-power row
// and, every check_every iterations, k_rows<2/3> / k_cols_check / k_decide for P (candidate objective), D
// (Lagrangian bound), violation, stopping flags and the rho balance.
// Replaces the same reference code as the on-chip kernel (aco.py:220-321, 363-408).
// Differences from the on-chip path: no running average / restarts; scalar reductions use
// float64 atomics (summation order, hence the exact stopping iteration, may vary run to run).
#include <algorithm>
#include "acb_common.cuh"

namespace {

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double wsumd(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }
__device__ __forceinline__ void proj_disc(float a, float b, float lim, float& za, float& zb) {
    float n2 = a * a + b * b;
    float f = (n2 > lim * lim) ? lim * rsqrtf(n2) : 1.0f;
    za = a * f;
    zb = b * f;
}
__device__ __forceinline__ void atomic_max_pos(float* addr, float v) {  // v >= 0
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
}

// per-instance scalars
enum { GS_RHO = 0, GS_PLEVEL, GS_CS, GS_QD, GS_GAMMA, GS_PKW, GS_PKP0, GS_E1, GS_E2, GS_XMAX, GS_YMAX, GS_VIOL, GS_UMAX, GS_ZUMAX, GS_GAP, GS_RP, GS_RD,
       GS_STALL, GS_NRESCUE, GS_NFEAS, GS_BESTVIOL, GS_VSTALL, GS_N };
enum { GD_P = 0, GD_D, GD_UQ, GD_DBEST, GD_PMAX, GD_BESTGAP, GD_N };

struct GenWork {
    float *V, *VC, *KX, *SG, *SGZ, *HG, *MU, *AL, *BE;  // AL/BE: cost-scaled alpha, beta [B][Tp]
    float* scal;     // [B][GS_N]
    double* dacc;    // [B][GD_N]
    int* status;     // [B] -1 = running
    int* row_first;  // [B][N] first session of the row
    int* row_cnt;    // [B][N]
    int* ndone;      // [1]
    int* iters;      // [B]
};

struct GenDims {
    int N, R, NG, Tp, Tt /*tiles*/, S_max, nDisc, nLin, has_pl, has_u, rPL, rU, lin_two_sided;
};

// ---------------------------------------------------------------------------- setup
__global__ void k_setup(SiteDev S, acb_batch B, acb_options opt, GenWork W, GenDims D) {
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const int nS = B.n_sessions[b], Tb = B.T[b], Tp = D.Tp;
    __shared__ float red[32];
    // (warm_shift / warm_had: see the on-chip kernel)
    const int wsh = B.warm_shift;
    const bool hadW = !B.warm_had || B.warm_had[b] != 0;
    for (int i = tid; i < D.N; i += blockDim.x) { W.row_first[(size_t)b * D.N + i] = 0; W.row_cnt[(size_t)b * D.N + i] = 0; }
    __syncthreads();
    // per-row session runs (sessions are sorted by row)
    for (int s = tid; s < nS; s += blockDim.x) {
        const int* rows = B.sess_row + (size_t)b * B.S_max;
        int row = rows[s];
        if (s == 0 || rows[s - 1] != row) {
            int c = 1;
            while (s + c < nS && rows[s + c] == row) ++c;
            W.row_first[(size_t)b * D.N + row] = s;
            W.row_cnt[(size_t)b * D.N + row] = c;
        }
        W.MU[(size_t)b * B.S_max + s] = (B.warm_mu && hadW) ? B.warm_mu[(size_t)b * B.S_max + s] : 0.f;
    }
    // cost scale and scaled cost vectors
    float m = 0.f;
    for (int i = tid; i < D.NG * Tp; i += blockDim.x) {
        int g = i / Tp, t = i - g * Tp;
        if (t < Tb) m = fmaxf(m, fabsf(B.alpha[(size_t)b * Tp + t] + S.kg[g] * B.beta[(size_t)b * Tp + t]));
    }
    m = wmax(m);
    if (lane == 0) red[warp] = m;
    __syncthreads();
    if (tid == 0) {
        float mm = 0.f;
        for (int w = 0; w < nw; ++w) mm = fmaxf(mm, red[w]);
        red[0] = (mm > 1e-20f) ? 1.f / mm : 1.f;
    }
    __syncthreads();
    const float cs = red[0];
    for (int t = tid; t < Tp; t += blockDim.x) {
        bool ok = t < Tb;
        W.AL[(size_t)b * Tp + t] = ok ? B.alpha[(size_t)b * Tp + t] * cs : 0.f;
        W.BE[(size_t)b * Tp + t] = ok ? B.beta[(size_t)b * Tp + t] * cs : 0.f;
    }
    // (row-level infeasibility, the initial v and the box maximum of the objective are row work: k_rows<Q, 6>)
    __shared__ double redd[32];
    {
        // soft energy rows: their part of the box maximum of the objective (see the on-chip kernel), in scaled units
        double pq = 0.0;
        if (B.sess_quad)
            for (int s2 = tid; s2 < nS; s2 += blockDim.x) {
                const double Eb = (double)B.sess_energy[(size_t)b * B.S_max + s2];
                pq += (double)(B.sess_quad[(size_t)b * B.S_max + s2] * cs) * Eb * Eb;
            }
        pq = wsumd(pq);
        if (lane == 0) redd[warp] = pq;
        __syncthreads();
    }
    if (tid == 0) {
        float* sc = W.scal + (size_t)b * GS_N;
        {
            double tot = 0.0;
            for (int w = 0; w < nw; ++w) tot += redd[w];
            W.dacc[(size_t)b * GD_N + GD_PMAX] = tot;  // k_rows<Q, 6> and k_setup_agg add the rest
        }
        // cold start: rho0, raised to the curvature of the aggregate quadratic seen through the scaled aggregate row
        // (2 Gamma u^2 with u = su * (Khat r)_u): at rho ~ Gamma su^2 the row's prox is balanced; a 1000-EVSE
        // load-flattening instance goes from > 1000 iterations at rho0 to the first check
        const float su0 = D.has_u ? S.row_scale[D.rU] : 0.f;
        sc[GS_RHO] = (B.warm_scal && hadW && B.warm_scal[b * 2] > 0.f) ? B.warm_scal[b * 2] : fmaxf(opt.rho0, opt.rho_curv * B.gamma[b] * cs * su0 * su0);
        sc[GS_PLEVEL] = (B.warm_scal && hadW) ? fmaxf(B.warm_scal[b * 2 + 1], B.peak_p0[b]) : B.peak_p0[b];
        sc[GS_CS] = cs;
        sc[GS_QD] = B.qd[b] * cs; sc[GS_GAMMA] = B.gamma[b] * cs; sc[GS_PKW] = B.peak_w[b] * cs; sc[GS_PKP0] = B.peak_p0[b];
        sc[GS_E1] = sc[GS_E2] = sc[GS_XMAX] = sc[GS_YMAX] = sc[GS_VIOL] = sc[GS_UMAX] = sc[GS_ZUMAX] = sc[GS_GAP] = sc[GS_RP] = sc[GS_RD] = 0.f;
        double* da = W.dacc + (size_t)b * GD_N;
        da[GD_P] = da[GD_D] = da[GD_UQ] = 0.0;
        da[GD_DBEST] = -1.0e300;
        da[GD_BESTGAP] = 1.0e300;
        sc[GS_STALL] = 0.f; sc[GS_NRESCUE] = 0.f; sc[GS_NFEAS] = 0.f; sc[GS_BESTVIOL] = 3.0e38f; sc[GS_VSTALL] = 0.f;
        W.status[b] = -1;
        W.iters[b] = 0;
    }
    // state of the coupling rows (the EVSE rows' v: k_rows<Q, 6>)
    for (int i = tid; i < D.R * Tp; i += blockDim.x) {
        size_t k = (size_t)b * D.R * Tp + i;
        const int t = i % Tp;
        W.VC[k] = (B.warm_vc && hadW && t + wsh < Tp) ? B.warm_vc[k + wsh] : 0.f;
        W.KX[k] = 0.f;
    }
}

// per instance, after k_rows<Q, 6 / 7>: the aggregate-power terms of the box maximum of the objective from the group sums
// of the bounds (SG: upper, SGZ: lower or absent)
__global__ void k_setup_agg(SiteDev S, acb_batch B, GenWork W, GenDims D, int have_lb) {
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const float* sc = W.scal + (size_t)b * GS_N;
    const float gam_s = sc[GS_GAMMA], pkw_s = sc[GS_PKW];
    if (!D.has_u || !(gam_s > 0.f || pkw_s > 0.f)) return;
    const int Tp = D.Tp, Tb = B.T[b];
    __shared__ double redd[32];
    __shared__ float redu[32];
    double pm = 0.0;
    float cmax = 0.f;
    for (int t = tid; t < Tb; t += blockDim.x) {
        float umax = 0.f, umin = 0.f;
        for (int g = 0; g < D.NG; ++g) {
            umax += S.kg[g] * W.SG[((size_t)b * D.NG + g) * Tp + t];
            if (have_lb) umin += S.kg[g] * W.SGZ[((size_t)b * D.NG + g) * Tp + t];
        }
        const float e = B.ext ? B.ext[(size_t)b * Tp + t] : 0.f;
        pm += (double)gam_s * (double)fmaxf((umax + e) * (umax + e), (umin + e) * (umin + e));
        cmax = fmaxf(cmax, umax);
    }
    pm = wsumd(pm); cmax = wmax(cmax);
    if (lane == 0) { redd[warp] = pm; redu[warp] = cmax; }
    __syncthreads();
    if (tid == 0) {
        double tot = 0.0;
        float um = 0.f;
        for (int w = 0; w < nw; ++w) { tot += redd[w]; um = fmaxf(um, redu[w]); }
        W.dacc[(size_t)b * GD_N + GD_PMAX] += tot + (double)pkw_s * (double)fmaxf(um, sc[GS_PKP0]);
    }
}

// multiplier of the session covering period t
__device__ __forceinline__ float mu_at(const float* MU, const int* SA, const int* SL, int sf, int sc, int t) {
    float m = 0.f;
    for (int s = sf; s < sf + sc; ++s)
        if (t >= SA[s] && t < SA[s] + SL[s]) m = MU[s];
    return m;
}

// MODE 0: iteration (x, v update, projection, SG <- sums of q);  MODE 1: init (SG <- sums of q from V);
// MODE 2: check (SGZ <- sums of z, P_lin);  MODE 3: check (Lagrangian inner terms with HG = C'y);
// MODE 4: write the schedule;  MODE 5: rescale V for a new rho (scal[GS_E1] holds rho_old/rho_new);
// MODE 8: iteration without the residual maxima (they are read at checks only: every iteration of a burst but the last);
// MODE 6: setup (initial v, row-level infeasibility, the rows' part of the box maximum of the objective, SG <- group sums
//         of the upper bounds);  MODE 7: setup (SGZ <- group sums of the lower bounds; only when some minimum rate is not 0)
//
// Q > 0: padded horizon 32*Q known at compile time, a row lives in registers (Q values per lane).
// Q = 0: any horizon that is a multiple of 32 (the offline algorithm, sessions longer than a day; reference
//        aco.py:243-245 puts no limit on T): a row is staged in the warp's slice of dynamic shared memory instead
//        (v, lb, ub and the partial group sums: 4 Tp floats per warp), everything else is the same code.
template <int Q>
struct RowStore {
    float v[Q > 0 ? Q : 1], lb[Q > 0 ? Q : 1], ub[Q > 0 ? Q : 1];
    __device__ __forceinline__ RowStore(float*, int, int) {}
    __device__ __forceinline__ float& V(int q) { return v[q]; }
    __device__ __forceinline__ float& LB(int q) { return lb[q]; }
    __device__ __forceinline__ float& UB(int q) { return ub[q]; }
};
template <>
struct RowStore<0> {
    float *v, *lb, *ub;
    __device__ __forceinline__ RowStore(float* base, int Tp, int lane) : v(base + lane), lb(base + Tp + lane), ub(base + 2 * Tp + lane) {}
    __device__ __forceinline__ float& V(int q) { return v[32 * q]; }
    __device__ __forceinline__ float& LB(int q) { return lb[32 * q]; }
    __device__ __forceinline__ float& UB(int q) { return ub[32 * q]; }
};

template <int Q, int MODE>
__global__ void __launch_bounds__(Q > 0 ? 128 : 256, Q > 0 ? 5 : 1) k_rows(SiteDev S, acb_batch B, acb_options opt, GenWork W, GenDims D, const int* grp_off) {
    constexpr bool SETUP = (MODE == 6 || MODE == 7), ITER = (MODE == 0 || MODE == 8), TRACK = (MODE == 0);
    const int g = blockIdx.x, b = blockIdx.y;
    if (W.status[b] >= 0 && MODE != 4 && !SETUP) return;
    constexpr bool DYN = (Q == 0);
    const int Tp = DYN ? D.Tp : 32 * Q, nq = DYN ? D.Tp / 32 : Q;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    extern __shared__ float dsm[];                      // DYN: [nw][4][Tp] (v, lb, ub, partial sums); else [nw][Tp] partial sums
    float* part = DYN ? dsm + (size_t)warp * 4 * Tp + 3 * Tp : dsm + (size_t)warp * Tp;
    const int part_stride = DYN ? 4 * Tp : Tp;
    const float* sc = W.scal + (size_t)b * GS_N;
    const float rho = sc[GS_RHO], rho1 = opt.kappa * rho, qd = sc[GS_QD], dd = 2.f * qd + rho1, inv_d = 1.f / dd, alpha = opt.alpha;
    const float kgc = S.kg[g];
    const float* AL = W.AL + (size_t)b * Tp;
    const float* BE = W.BE + (size_t)b * Tp;
    const int* SA = B.sess_start + (size_t)b * B.S_max;
    const int* SL = B.sess_len + (size_t)b * B.S_max;
    float* MU = W.MU + (size_t)b * B.S_max;
    float acc[Q > 0 ? Q : 1];  // Q > 0: the warp's partial group sums stay in registers until the end
#pragma unroll
    for (int q = 0; q < nq; ++q) { if constexpr (DYN) part[lane + 32 * q] = 0.f; else acc[q] = 0.f; }
    auto add_part = [&](int q, float val) { if constexpr (DYN) part[lane + 32 * q] += val; else acc[q] += val; };
    float e1 = 0.f, e2 = 0.f, xm = 0.f, ym = 0.f;
    double dsum = 0.0;
    const float rescale = (MODE == 5) ? sc[GS_E1] : 1.f;
    if (MODE == 5 && rescale == 1.f) return;
    RowStore<Q> rs(DYN ? dsm + (size_t)warp * 4 * Tp : nullptr, Tp, lane);
    const int* SO = B.sess_rate_off + (size_t)b * B.S_max;
    // the group's row of the column pass (K'h - c), the same for every EVSE of the group
    const float* HGg = W.HG + ((size_t)b * D.NG + g) * Tp;
    float hgq[Q > 0 ? Q : 1];
    if constexpr (!DYN) {
        if (ITER || MODE == 3) {
#pragma unroll
            for (int q = 0; q < Q; ++q) hgq[q] = HGg[lane + 32 * q];
        }
    }
    auto hg_at = [&](int q) -> float { if constexpr (DYN) return HGg[lane + 32 * q]; else return hgq[q]; };
    // The warp's rows are walked in chunks of 32: lane j first fetches the table entries of the chunk's j-th row (row index,
    // session run and, for a single session with constant limits — the usual case — its window, limits, energy and
    // multiplier), so the chain of dependent loads is paid once per chunk instead of once per row; the row loop then takes
    // them by shuffle.  Register path: the next row's v is requested before the current row's multiplier search starts.
    const int kend = grp_off[g + 1];
    float vnx[Q > 0 ? Q : 1];
    for (int kc = grp_off[g] + warp; kc < kend; kc += 32 * nw) {
    int m_row = 0, m_sf = 0, m_scn = 0, m_a = 0, m_len = 0, m_off = 0;
    float m_lo = 0.f, m_hi = 0.f, m_mu = 0.f;
    if (kc + lane * nw < kend) {
        m_row = S.slot_row[kc + lane * nw];
        m_sf = W.row_first[(size_t)b * D.N + m_row];
        m_scn = W.row_cnt[(size_t)b * D.N + m_row];
        if (m_scn == 1) {
            m_a = SA[m_sf]; m_len = SL[m_sf]; m_off = SO[m_sf];
            m_mu = MU[m_sf];
            if (m_off < 0) { m_lo = B.min_rates[-(m_off + 1)]; m_hi = fmaxf(B.max_rates[-(m_off + 1)], m_lo); }
        }
    }
    if constexpr (!DYN && !SETUP) {
        const size_t bn = ((size_t)b * D.N + __shfl_sync(0xffffffffu, m_row, 0)) * Tp + lane;
#pragma unroll
        for (int q = 0; q < Q; ++q) vnx[q] = W.V[bn + 32 * q];
    }
    for (int jr = 0; jr < 32 && kc + jr * nw < kend; ++jr) {
        const int row = __shfl_sync(0xffffffffu, m_row, jr), sf = __shfl_sync(0xffffffffu, m_sf, jr), scn = __shfl_sync(0xffffffffu, m_scn, jr);
        const int s_a = __shfl_sync(0xffffffffu, m_a, jr), s_len = __shfl_sync(0xffffffffu, m_len, jr), s_off = __shfl_sync(0xffffffffu, m_off, jr);
        const float s_lo = __shfl_sync(0xffffffffu, m_lo, jr), s_hi = __shfl_sync(0xffffffffu, m_hi, jr), s_mu = __shfl_sync(0xffffffffu, m_mu, jr);
        const size_t base = ((size_t)b * D.N + row) * Tp + lane;
        if constexpr (SETUP) {
        } else if constexpr (DYN) {
            for (int q = 0; q < nq; ++q) rs.V(q) = W.V[base + 32 * q];
        } else {
#pragma unroll
            for (int q = 0; q < Q; ++q) rs.V(q) = vnx[q];
            if (jr + 1 < 32 && kc + (jr + 1) * nw < kend) {
                const size_t bn = ((size_t)b * D.N + __shfl_sync(0xffffffffu, m_row, jr + 1)) * Tp + lane;
#pragma unroll
                for (int q = 0; q < Q; ++q) vnx[q] = W.V[bn + 32 * q];
            }
        }
        // rate bounds straight from the session table (charging_rate_bounds, aco.py:61-79: zero outside the session windows,
        // ub := lb where ub < lb)
        if (scn == 1 && s_off < 0) {
#pragma unroll
            for (int q = 0; q < nq; ++q) {
                const bool in = (unsigned)(lane + 32 * q - s_a) < (unsigned)s_len;
                rs.LB(q) = in ? s_lo : 0.f; rs.UB(q) = in ? s_hi : 0.f;
            }
        } else {
#pragma unroll
            for (int q = 0; q < nq; ++q) { rs.LB(q) = 0.f; rs.UB(q) = 0.f; }
            for (int s = sf; s < sf + scn; ++s) {
                const int a = SA[s], len = SL[s], off = SO[s];
#pragma unroll
                for (int q = 0; q < nq; ++q) {
                    const int j = lane + 32 * q - a;
                    if (j >= 0 && j < len) {
                        const int ri = off >= 0 ? off + j : -(off + 1);
                        const float lo = B.min_rates[ri];
                        rs.LB(q) = lo; rs.UB(q) = fmaxf(B.max_rates[ri], lo);
                    }
                }
            }
        }
        if (SETUP) {
            if (MODE == 6) {
                // (warm_shift / warm_had: see the on-chip kernel)
                const int wsh = B.warm_shift;
                const bool hadW = !B.warm_had || B.warm_had[b] != 0;
#pragma unroll
                for (int q = 0; q < nq; ++q) {
                    const int t = lane + 32 * q;
                    const float lo = rs.LB(q), hi = rs.UB(q);
                    W.V[base + 32 * q] = (B.warm_v1 && hadW) ? ((t + wsh < Tp) ? B.warm_v1[base + 32 * q + wsh] : 0.f) : clampf(0.f, lo, hi);
                    const float c = AL[t] + kgc * BE[t];
                    dsum += (double)fmaxf(c * lo, c * hi) + (double)qd * (double)fmaxf(lo * lo, hi * hi);
                    add_part(q, hi);
                }
                // row-level infeasibility (same rule as the on-chip kernel)
                for (int s = sf; s < sf + scn; ++s) {
                    const int a = SA[s], e = min(a + SL[s], Tp);
                    float slo = 0.f, shi = 0.f;
#pragma unroll
                    for (int q = 0; q < nq; ++q) {
                        const int t = lane + 32 * q;
                        if (t >= a && t < e) { slo += rs.LB(q); shi += rs.UB(q); }
                    }
                    slo = wsum(slo); shi = wsum(shi);
                    const float Eb = B.sess_energy[(size_t)b * B.S_max + s], tol = 1e-5f * (fabsf(Eb) + 1.f);
                    if (lane == 0 && (slo > Eb + tol || (opt.equality && shi < Eb - tol)) && atomicCAS(W.status + b, -1, (int)ACB_INFEASIBLE) == -1)
                        atomicAdd(W.ndone, 1);
                }
            } else {
#pragma unroll
                for (int q = 0; q < nq; ++q) add_part(q, rs.LB(q));
            }
        } else if (ITER) {
            float zo[Q > 0 ? Q : 1];  // previous z for the dual residual (register path only; long horizons report r_dual = 0)
            // one session on the row (the usual case): the bounds are zero outside its window, so clamp(v - mu, lb, ub) is
            // already 0 there and neither the multiplier lookup nor the window tests are needed
            const bool one = (scn == 1);
            float mu1 = s_mu;
#pragma unroll
            for (int q = 0; q < nq; ++q) {
                const int t = lane + 32 * q;
                const float vq = rs.V(q);
                float z = clampf(vq - (one ? mu1 : mu_at(MU, SA, SL, sf, scn, t)), rs.LB(q), rs.UB(q));
                float x = (rho1 * (2.f * z - vq) + hg_at(q)) * inv_d;
                rs.V(q) = vq + alpha * (x - z);
                if constexpr (TRACK) {
                    if constexpr (!DYN) zo[q] = z;
                    e1 = fmaxf(e1, fabsf(x - z));
                    xm = fmaxf(xm, fabsf(x));
                }
            }
            for (int s = sf; s < sf + scn; ++s) {
                const int a = SA[s], e = a + SL[s];
                const float Eb = B.sess_energy[(size_t)b * B.S_max + s];
                const float tol = 2e-6f * (Eb + 1.f);
                float mu = one ? s_mu : MU[s];
                // quadratic shortfall term cq (Eb - E)^2 (non_completion_penalty, norm 2): see newton_mu in acb_solve_kernel.cuh
                const float cq = B.sess_quad ? B.sess_quad[(size_t)b * B.S_max + s] * sc[GS_CS] : 0.f;
                const bool soft = cq > 0.f && !opt.equality, freeMu = opt.equality || soft;
                const float ikq = soft ? rho1 / (2.f * cq) : 0.f;
                float lo = freeMu ? -3.0e38f : -1.f, hi = 3.0e38f;
                if (!freeMu) mu = fmaxf(mu, 0.f);
                for (int step = 0; step < 16; ++step) {
                    float E = 0.f;
                    int nf = 0;
                    if (one) {
#pragma unroll
                        for (int q = 0; q < nq; ++q) {
                            const float w = rs.V(q) - mu;
                            E += clampf(w, rs.LB(q), rs.UB(q));
                            nf += (w > rs.LB(q) && w < rs.UB(q)) ? 1 : 0;
                        }
                    } else {
#pragma unroll
                        for (int q = 0; q < nq; ++q) {
                            const int t = lane + 32 * q;
                            if (t >= a && t < e) {
                                float w = rs.V(q) - mu;
                                E += clampf(w, rs.LB(q), rs.UB(q));
                                nf += (w > rs.LB(q) && w < rs.UB(q)) ? 1 : 0;
                            }
                        }
                    }
                    E = wsum(E);
                    nf = __reduce_add_sync(0xffffffffu, nf);
                    float rr = E - Eb - ((soft && mu < 0.f) ? mu * ikq : 0.f);
                    const float slope = (float)nf + ((soft && mu < 0.f) ? ikq : 0.f);
                    if (fabsf(rr) <= tol) break;
                    if (!freeMu && mu <= 0.f && rr < 0.f) { mu = 0.f; break; }
                    if (rr > 0.f) lo = mu; else hi = mu;
                    float mun = (slope > 0.f) ? mu + rr / slope : (rr > 0.f ? 3.0e38f : -3.0e38f);
                    if (!freeMu) mun = fmaxf(mun, 0.f);
                    if (!(mun > lo && mun < hi)) {
                        if (hi < 1.0e38f && lo > -1.0e38f) mun = 0.5f * (fmaxf(lo, freeMu ? lo : 0.f) + hi);
                        else if (rr > 0.f) mun = mu + fmaxf(1.f, 2.f * fabsf(mu));
                        else mun = mu - fmaxf(1.f, 2.f * fabsf(mu));
                        if (!freeMu) mun = fmaxf(mun, 0.f);
                    }
                    mu = mun;
                }
                if (lane == 0) MU[s] = mu;
                mu1 = mu;
                __syncwarp();
            }
#pragma unroll
            for (int q = 0; q < nq; ++q) {
                const int t = lane + 32 * q;
                const float vq = rs.V(q);
                float zn = clampf(vq - (one ? mu1 : mu_at(MU, SA, SL, sf, scn, t)), rs.LB(q), rs.UB(q));
                add_part(q, 2.f * zn - vq);
                W.V[base + 32 * q] = vq;
                if constexpr (TRACK) {
                    if constexpr (!DYN) e2 = fmaxf(e2, fabsf(zn - zo[q]));
                    ym = fmaxf(ym, fabsf(rho1 * (vq - zn)));
                }
            }
        } else {
#pragma unroll
            for (int q = 0; q < nq; ++q) {
                const int t = lane + 32 * q;
                const float mu = mu_at(MU, SA, SL, sf, scn, t);
                const float vq = rs.V(q), lbq = rs.LB(q), ubq = rs.UB(q);
                const float z = clampf(vq - mu, lbq, ubq);
                if (MODE == 1) add_part(q, 2.f * z - vq);
                if (MODE == 2) {
                    add_part(q, z);
                    float c = AL[t] + kgc * BE[t];
                    dsum += (double)(c * z + qd * z * z);
                }
                if (MODE == 3) {
                    float rt = AL[t] + kgc * BE[t] + hg_at(q) + rho1 * mu;
                    float phi;
                    if (qd > 0.f) { float xs = clampf(-rt / (2.f * qd), lbq, ubq); phi = qd * xs * xs + rt * xs; }
                    else phi = fminf(lbq * rt, ubq * rt);
                    dsum += (double)phi;
                }
                if (MODE == 4) {
                    B.rates[base + 32 * q] = z;
                    if (B.pilots) {  // fused project_into_continuous_feasible_pilots, same selects as k_project_continuous
                        double pv = (double)z;
                        const double mp = S.max_pilot[row];
                        pv = (mp < pv) ? mp : pv;
                        B.pilots[base + 32 * q] = (pv > 0.0) ? pv : 0.0;
                    }
                }
                if (MODE == 5) W.V[base + 32 * q] = z + rescale * (vq - z);
                if (MODE == 4 && B.out_v1) B.out_v1[base + 32 * q] = vq;
            }
            if (MODE == 3 && lane == 0)
                for (int s = sf; s < sf + scn; ++s) {
                    const double m = (double)(rho1 * MU[s]);
                    dsum -= m * (double)B.sess_energy[(size_t)b * B.S_max + s];
                    const float cq = B.sess_quad ? B.sess_quad[(size_t)b * B.S_max + s] * sc[GS_CS] : 0.f;
                    if (m < 0.0 && cq > 0.f) dsum -= m * m / (4.0 * (double)cq);  // conjugate of the quadratic shortfall term
                }
            if (MODE == 2 && B.sess_quad) {
                // objective term cq (Eb - E)^2 of the candidate, E = planned amp-periods inside the session window
                for (int s = sf; s < sf + scn; ++s) {
                    const float cq = B.sess_quad[(size_t)b * B.S_max + s] * sc[GS_CS];
                    if (!(cq > 0.f)) continue;
                    const int a = SA[s], e = a + SL[s];
                    float Es = 0.f;
#pragma unroll
                    for (int q = 0; q < nq; ++q) {
                        const int t = lane + 32 * q;
                        if (t >= a && t < e) Es += clampf(rs.V(q) - MU[s], rs.LB(q), rs.UB(q));
                    }
                    Es = wsum(Es);
                    const float Eb = B.sess_energy[(size_t)b * B.S_max + s];
                    if (lane == 0) dsum += (double)cq * (double)(Eb - Es) * (double)(Eb - Es);
                }
            }
        }
    }
    }
    if (MODE <= 2 || SETUP || MODE == 8) {
        if constexpr (!DYN) {
#pragma unroll
            for (int q = 0; q < nq; ++q) part[lane + 32 * q] = acc[q];
        }
        __syncthreads();
        float* out = ((MODE == 2 || MODE == 7) ? W.SGZ : W.SG) + ((size_t)b * D.NG + g) * Tp;
        const float* p0 = DYN ? dsm + 3 * Tp : dsm;
        for (int t = tid; t < Tp; t += blockDim.x) {
            float s = 0.f;
            for (int w = 0; w < nw; ++w) s += p0[(size_t)w * part_stride + t];
            out[t] = s;
        }
    }
    if (MODE == 0) {
        e1 = wmax(e1); e2 = wmax(e2); xm = wmax(xm); ym = wmax(ym);
        if (lane == 0) {
            float* s = W.scal + (size_t)b * GS_N;
            atomic_max_pos(s + GS_E1, e1); atomic_max_pos(s + GS_E2, e2); atomic_max_pos(s + GS_XMAX, xm); atomic_max_pos(s + GS_YMAX, ym);
        }
    }
    if (MODE == 2 || MODE == 3 || MODE == 6) {
        dsum = wsumd(dsum);
        if (lane == 0) atomicAdd(W.dacc + (size_t)b * GD_N + (MODE == 2 ? GD_P : MODE == 3 ? GD_D : GD_PMAX), dsum);
    }
}

// ---------------------------------------------------------------------------- iteration column pass as a blocked product
// One stage of the Woodbury chain for a tile of 32 periods: out[m][c] = epi(sum_k MatT[k][m] * in[k][c]), m < M, c < 32.
// MatT is the k-major operand in global memory (row stride ldm, a multiple of 4, zero padded; shared by every instance of
// the site), staged through `mbuf` in chunks of 32 k-rows with the next chunk's global loads in flight while the current one
// is multiplied.  256 threads; thread (tr, tc) = (tid / 8, tid % 8) owns rows RPT*tr .. +RPT-1 and periods 4*tc .. +3 of a
// 32*RPT-row block: per k one 16-byte (RPT = 4) shared-memory load of the matrix, one of the input vector, 4*RPT FMAs
// (both loads are one wavefront: 4 distinct row quads and 8 distinct period quads per warp).
constexpr int MM_KC = 32;
template <int RPT, class Epi>
__device__ __forceinline__ void mm_stage(const float* __restrict__ MatT, int ldm, int K, int M, const float* __restrict__ in,
                                         float* __restrict__ mbuf, Epi epi) {
    constexpr int MB = 32 * RPT, NV = MM_KC * MB / 4 / 256;  // float4 per thread and chunk
    const int tid = threadIdx.x, tr = tid >> 3, tc = tid & 7;
    for (int m0 = 0; m0 < M; m0 += MB) {
        float acc[RPT][4];
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        float4 pre[NV];
        auto fetch = [&](int k0) {
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const int j = tid + 256 * i, kk = j / (MB / 4), c4 = j - kk * (MB / 4);
                const int k = k0 + kk, m = m0 + 4 * c4;
                pre[i] = (k < K && m < ldm) ? __ldg(reinterpret_cast<const float4*>(MatT + (size_t)k * ldm + m)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        fetch(0);
        for (int k0 = 0; k0 < K; k0 += MM_KC) {
            __syncthreads();  // the previous chunk (and the previous stage's output) is no longer being read / is complete
#pragma unroll
            for (int i = 0; i < NV; ++i) reinterpret_cast<float4*>(mbuf)[tid + 256 * i] = pre[i];
            __syncthreads();
            if (k0 + MM_KC < K) fetch(k0 + MM_KC);
            const int kmax = min(MM_KC, K - k0);
            const float* inp = in + (size_t)k0 * 32 + 4 * tc;
            const float* mp = mbuf + RPT * tr;
#pragma unroll 4
            for (int kk = 0; kk < kmax; ++kk) {
                const float4 bq = *reinterpret_cast<const float4*>(inp + kk * 32);
                float a[RPT];
                if constexpr (RPT == 4) {
                    const float4 aq = *reinterpret_cast<const float4*>(mp + kk * MB);
                    a[0] = aq.x; a[1] = aq.y; a[2] = aq.z; a[3] = aq.w;
                } else {
                    const float2 aq = *reinterpret_cast<const float2*>(mp + kk * MB);
                    a[0] = aq.x; a[1] = aq.y;
                }
#pragma unroll
                for (int i = 0; i < RPT; ++i) {
                    acc[i][0] = fmaf(a[i], bq.x, acc[i][0]); acc[i][1] = fmaf(a[i], bq.y, acc[i][1]);
                    acc[i][2] = fmaf(a[i], bq.z, acc[i][2]); acc[i][3] = fmaf(a[i], bq.w, acc[i][3]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
            const int m = m0 + RPT * tr + i;
            if (m < M) epi(m, 4 * tc, acc[i]);
        }
    }
}

// Check column pass, block per (tile of 32 periods, instance): evaluation of the candidate (violation, aggregate-power
// part of P, conjugate terms of D, HG <- C'y).  Runs once per check_every iterations; the iteration's column pass is
// k_cols_it below.
#define ACB_CPL 1  // columns per lane
__global__ void __launch_bounds__(256) k_cols_check(SiteDev S, acb_batch B, acb_options opt, GenWork W, GenDims D) {
    constexpr int CHECK = 1, CPL = ACB_CPL, TW = 32 * CPL;
    const int tile = blockIdx.x, b = blockIdx.y;
    if (W.status[b] >= 0) return;
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const int R = D.R, NG = D.NG, Tp = D.Tp, t0 = tile * TW + lane, Tb = B.T[b];
    float* sa = sm;                 // [NG][TW]   group inputs / group sums of z
    float* gg = sa + NG * TW;       // [R][TW]    g (iteration) or y (check)
    const int Rp = S.Rp;            // R rounded up to a multiple of 4
    float* bv = gg + R * TW;        // [Rp][TW]  K z
    float* mbuf = bv + Rp * TW;     // [MM_KC][128] matrix chunk of mm_stage
    const float* sc = W.scal + (size_t)b * GS_N;
    const float rho = sc[GS_RHO], rho1 = opt.kappa * rho, qd = sc[GS_QD], dd = 2.f * qd + rho1, dr = dd / rho;
    const float Gamma = sc[GS_GAMMA], pk_w = sc[GS_PKW], pk_p0 = sc[GS_PKP0], plevel = sc[GS_PLEVEL];
    const float su = D.has_u ? S.row_scale[D.rU] : 1.f;
    const float linLo = D.lin_two_sided ? -1.f : -3.0e38f;
    const float* AL = W.AL + (size_t)b * Tp;
    const float* BE = W.BE + (size_t)b * Tp;
    const float* ext = B.ext ? B.ext + (size_t)b * Tp : nullptr;
    float* VC = W.VC + (size_t)b * R * Tp;
    float* KX = W.KX + (size_t)b * R * Tp;
    auto ebar = [&](int tt) -> float { return (ext && tt < Tb) ? ext[tt] : 0.f; };
    auto plim = [&](int tt) -> float { return (B.peak_limit && tt < Tb) ? B.peak_limit[(size_t)b * Tp + tt] / S.row_scale[D.rPL] : 3.0e38f; };
    auto agg_a = [&](float v, int tt) -> float { float rp = rho / (su * su); return (rp * (v * su) - 2.f * Gamma * ebar(tt)) / (rp + 2.f * Gamma); };
    // z of coupling row r (disc rows are handled pairwise by the caller)
    auto proj_row = [&](int r, float v, int tt) -> float {
        if (r < 2 * D.nDisc + D.nLin) return clampf(v, (linLo < -1.0e30f) ? linLo : linLo * S.lim[r], S.lim[r]);
        if (D.has_pl && r == D.rPL) return fminf(v, plim(tt));
        float a = agg_a(v, tt);
        return ((pk_w > 0.f) ? fminf(a, plevel) : a) / su;
    };
    double dconj = 0.0, duq = 0.0;
    float viol = -1.f, umax = 0.f, zumax = 0.f;
    // (excess allowed on a row of L amperes: min(viol_tol L, viol_abs); see eval_columns of the on-chip kernel)
    auto vfac = [&](float lim_amps) -> float { return (opt.viol_abs > 0.f) ? fmaxf(1.f, lim_amps * opt.viol_tol / opt.viol_abs) : 1.f; };
    // ---- stage 1: inputs (columns beyond Tp read as zero and are never written back)
    for (int g = warp; g < NG; g += nw) {
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const int t = t0 + 32 * c;
            float val = 0.f;
            if (t < Tp) {
                float s = (CHECK ? W.SGZ : W.SG)[((size_t)b * NG + g) * Tp + t];
                val = CHECK ? s : rho1 * s - S.ngrp[g] * (AL[t] + S.kg[g] * BE[t]);
            }
            sa[g * TW + 32 * c + lane] = val;
        }
    }
    for (int r = warp; r < R; r += nw) {
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const int t = t0 + 32 * c;
            if (t >= Tp) { gg[r * TW + 32 * c + lane] = 0.f; continue; }
            float z;
            if (r < 2 * D.nDisc) {
                int r0 = r & ~1;
                float a = VC[r0 * Tp + t], bb = VC[(r0 + 1) * Tp + t], za, zb;
                proj_disc(a, bb, S.lim[r0], za, zb);
                z = (r & 1) ? zb : za;
            } else z = proj_row(r, VC[r * Tp + t], t);
            float v = VC[r * Tp + t];
            gg[r * TW + 32 * c + lane] = CHECK ? rho * (v - z) : rho * (2.f * z - v);
            if (CHECK) {
                float y = rho * (v - z);
                if (r < 2 * D.nDisc) {
                    // support function of the disc: after the barrier, from both components
                } else if (r < 2 * D.nDisc + D.nLin + D.has_pl) {
                    float cap = (D.has_pl && r == D.rPL) ? plim(t) : S.lim[r];
                    if (y != 0.f && cap < 1.0e30f) dconj -= (double)(cap * fabsf(y));
                } else {
                    // aggregate-power row: Fenchel equality -g*(y) = g(z) - <y, z>; the max term is added in k_decide
                    float zk = z * su;
                    if (t < Tb) { dconj += (double)Gamma * (double)(zk + ebar(t)) * (double)(zk + ebar(t)); zumax = fmaxf(zumax, zk); }
                    dconj -= (double)y * (double)z;
                }
            }
        }
    }
    __syncthreads();
    if (CHECK) {
        // disc support functions need both components
        for (int j = warp; j < D.nDisc; j += nw)
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                float ya = gg[(2 * j) * TW + 32 * c + lane], yb = gg[(2 * j + 1) * TW + 32 * c + lane];
                dconj -= (double)(S.lim[2 * j] * sqrtf(ya * ya + yb * yb));
            }
        // Kz rows: violation and aggregate power of the candidate
        mm_stage<4>(S.Ct, Rp, NG, R, sa, mbuf, [&](int m, int c, const float* a) {
            *reinterpret_cast<float4*>(bv + m * TW + c) = make_float4(a[0], a[1], a[2], a[3]);
        });
        __syncthreads();
        for (int j = warp; j < D.nDisc; j += nw)
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                float ka = bv[(2 * j) * TW + 32 * c + lane], kb = bv[(2 * j + 1) * TW + 32 * c + lane];
                if (S.lim[2 * j] > 0.f) viol = fmaxf(viol, (sqrtf(ka * ka + kb * kb) / S.lim[2 * j] - 1.f) * vfac(S.lim[2 * j] * S.row_scale[2 * j]));
                else viol = fmaxf(viol, sqrtf(ka * ka + kb * kb) * S.row_scale[2 * j]);  // limit 0: the current itself, in amperes
            }
        for (int r = 2 * D.nDisc + warp; r < 2 * D.nDisc + D.nLin + D.has_pl; r += nw)
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const int t = t0 + 32 * c;
                float ka = bv[r * TW + 32 * c + lane];
                float cap = (D.has_pl && r == D.rPL) ? plim(t) : S.lim[r];
                if (r < 2 * D.nDisc + D.nLin && D.lin_two_sided) ka = fabsf(ka);
                if (cap > 0.f && cap < 1.0e30f) viol = fmaxf(viol, (ka / cap - 1.f) * vfac(cap * S.row_scale[r]));
                else if (cap <= 0.f) viol = fmaxf(viol, fmaxf(ka, 0.f) * S.row_scale[r]);
            }
        if (D.has_u && warp == 0)
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const int t = t0 + 32 * c;
                if (t < Tb) {
                    float u = bv[D.rU * TW + 32 * c + lane] * su;
                    umax = fmaxf(umax, u);
                    duq += (double)(u + ebar(t)) * (double)(u + ebar(t));
                }
            }
        // HG <- C'y
        {
            auto hg_out = [&](int m, int c, const float* a) {
                *reinterpret_cast<float4*>(W.HG + ((size_t)b * NG + m) * Tp + tile * TW + c) = make_float4(a[0], a[1], a[2], a[3]);
            };
            if (NG <= 64) mm_stage<2>(S.Cp, S.NGp, R, NG, gg, mbuf, hg_out);
            else mm_stage<4>(S.Cp, S.NGp, R, NG, gg, mbuf, hg_out);
        }
        viol = wmax(viol); umax = wmax(umax); zumax = wmax(zumax);
        dconj = wsumd(dconj); duq = wsumd(duq);
        if (lane == 0) {
            float* s = W.scal + (size_t)b * GS_N;
            atomic_max_pos(s + GS_VIOL, viol + 4.f);
            atomic_max_pos(s + GS_UMAX, fmaxf(umax, 0.f));
            atomic_max_pos(s + GS_ZUMAX, fmaxf(zumax, 0.f));
            atomicAdd(W.dacc + (size_t)b * GD_N + GD_D, dconj);
            atomicAdd(W.dacc + (size_t)b * GD_N + GD_UQ, duq);
        }
        return;
    }
}

// Iteration column pass: block per (tile of 32 periods, instance), 256 threads.
//   b = C sa - (d/rho) g,  h = -U diag(1/(d/rho+lam)) U' b (rank-reduced, SiteDev::nEig),  hg = C' h - c,  Kx = (g - h)/rho,  v_c += alpha (Kx - z_c)
// The four products are mm_stage calls (shared-memory blocked, FMA bound); everything else is one pass over the tile.
__global__ void __launch_bounds__(256, 4) k_cols_it(SiteDev S, acb_batch B, acb_options opt, GenWork W, GenDims D) {
    constexpr int TW = 32;
    const int tile = blockIdx.x, b = blockIdx.y;
    if (W.status[b] >= 0) return;
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const int R = D.R, NG = D.NG, Tp = D.Tp, t = tile * TW + lane, Tb = B.T[b], Rp = S.Rp;
    float* mbuf = sm;                               // [MM_KC][128] matrix chunk
    float* sa = mbuf + MM_KC * 128;                 // [max(NG, nEigp)][TW]  group inputs, later y1
    float* gg = sa + (size_t)max(NG, S.nEigp) * TW; // [R][TW]   rho (2 z_c - v_c)
    float* bv = gg + (size_t)R * TW;                // [Rp][TW]  b, later h
    float* y1 = sa;
    const float* sc = W.scal + (size_t)b * GS_N;
    const float rho = sc[GS_RHO], rho1 = opt.kappa * rho, qd = sc[GS_QD], dd = 2.f * qd + rho1, dr = dd / rho;
    const float Gamma = sc[GS_GAMMA], pk_w = sc[GS_PKW], plevel = sc[GS_PLEVEL];
    const float su = D.has_u ? S.row_scale[D.rU] : 1.f;
    const float linLo = D.lin_two_sided ? -1.f : -3.0e38f;
    const float* AL = W.AL + (size_t)b * Tp;
    const float* BE = W.BE + (size_t)b * Tp;
    const float* ext = B.ext ? B.ext + (size_t)b * Tp : nullptr;
    float* VC = W.VC + (size_t)b * R * Tp;
    float* KX = W.KX + (size_t)b * R * Tp;
    // ---- inputs.  The tile of the coupling rows' v is staged through `bv` (free until the first product's epilogue) and the
    // group sums go straight into `sa`: every thread issues its (up to four) 16-byte loads before it uses any of them, so
    // the tile costs one memory round trip instead of one per row.
    const int t4 = tile * TW;
    {
        const int n = R * 8;
        for (int i0 = 0; i0 < n; i0 += 1024) {
            float4 tmp[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + tid + 256 * u;
                if (i < n) tmp[u] = *reinterpret_cast<const float4*>(VC + (size_t)(i >> 3) * Tp + t4 + 4 * (i & 7));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + tid + 256 * u;
                if (i < n) reinterpret_cast<float4*>(bv)[i] = tmp[u];
            }
        }
        const int ng8 = NG * 8;
        const float* SGb = W.SG + (size_t)b * NG * Tp;
        for (int i0 = 0; i0 < ng8; i0 += 1024) {
            float4 tmp[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + tid + 256 * u;
                if (i < ng8) tmp[u] = *reinterpret_cast<const float4*>(SGb + (size_t)(i >> 3) * Tp + t4 + 4 * (i & 7));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + tid + 256 * u;
                if (i < ng8) {
                    const int g = i >> 3, c = 4 * (i & 7);
                    const float4 al4 = *reinterpret_cast<const float4*>(AL + t4 + c), be4 = *reinterpret_cast<const float4*>(BE + t4 + c);
                    const float ng = S.ngrp[g], k = S.kg[g];
                    reinterpret_cast<float4*>(sa)[i] = make_float4(rho1 * tmp[u].x - ng * (al4.x + k * be4.x), rho1 * tmp[u].y - ng * (al4.y + k * be4.y),
                                                                   rho1 * tmp[u].z - ng * (al4.z + k * be4.z), rho1 * tmp[u].w - ng * (al4.w + k * be4.w));
                }
            }
        }
    }
    __syncthreads();
    for (int r = warp; r < R; r += nw) {
        const float v = bv[r * TW + lane];
        float z;
        if (r < 2 * D.nDisc) {
            const int r0 = r & ~1;
            float za, zb;
            proj_disc(bv[r0 * TW + lane], bv[(r0 + 1) * TW + lane], S.lim[r0], za, zb);
            z = (r & 1) ? zb : za;
        } else if (r < 2 * D.nDisc + D.nLin) z = clampf(v, (linLo < -1.0e30f) ? linLo : linLo * S.lim[r], S.lim[r]);
        else if (D.has_pl && r == D.rPL) z = fminf(v, (B.peak_limit && t < Tb) ? B.peak_limit[(size_t)b * Tp + t] / S.row_scale[D.rPL] : 3.0e38f);
        else {
            const float rp = rho / (su * su), a = (rp * (v * su) - 2.f * Gamma * ((ext && t < Tb) ? ext[t] : 0.f)) / (rp + 2.f * Gamma);
            z = ((pk_w > 0.f) ? fminf(a, plevel) : a) / su;
        }
        gg[r * TW + lane] = rho * (2.f * z - v);
    }
    // (mm_stage starts with a barrier)
    mm_stage<4>(S.Ct, Rp, NG, R, sa, mbuf, [&](int m, int c, const float* a) {
        const float4 g4 = *reinterpret_cast<const float4*>(gg + m * TW + c);
        *reinterpret_cast<float4*>(bv + m * TW + c) = make_float4(a[0] - dr * g4.x, a[1] - dr * g4.y, a[2] - dr * g4.z, a[3] - dr * g4.w);
    });
    // y1 = diag(1/(d/rho+lam) - 1/(d/rho)) Ur' b over the nEig non-null eigenvectors, then h = -(b/(d/rho) + Ur y1) in place
    const float inv_dr = 1.f / dr;
    const int nE = S.nEig;
    auto y_out = [&](int m, int c, const float* a) {
        const float w = 1.f / (dr + S.lamr[m]) - inv_dr;
        *reinterpret_cast<float4*>(y1 + m * TW + c) = make_float4(a[0] * w, a[1] * w, a[2] * w, a[3] * w);
    };
    if (nE <= 64) mm_stage<2>(S.Urp, S.nEigp, R, nE, bv, mbuf, y_out);
    else mm_stage<4>(S.Urp, S.nEigp, R, nE, bv, mbuf, y_out);
    mm_stage<4>(S.Urt, Rp, nE, R, y1, mbuf, [&](int m, int c, const float* a) {
        float4* o = reinterpret_cast<float4*>(bv + m * TW + c);
        const float4 b4 = *o;
        *o = make_float4(-(b4.x * inv_dr + a[0]), -(b4.y * inv_dr + a[1]), -(b4.z * inv_dr + a[2]), -(b4.w * inv_dr + a[3]));
    });
    auto hg_out = [&](int m, int c, const float* a) {
        const int tt = tile * TW + c;
        const float4 al4 = *reinterpret_cast<const float4*>(AL + tt), be4 = *reinterpret_cast<const float4*>(BE + tt);
        const float k = S.kg[m];
        *reinterpret_cast<float4*>(W.HG + ((size_t)b * NG + m) * Tp + tt) =
            make_float4(a[0] - (al4.x + k * be4.x), a[1] - (al4.y + k * be4.y), a[2] - (al4.z + k * be4.z), a[3] - (al4.w + k * be4.w));
    };
    if (NG <= 64) mm_stage<2>(S.Cp, S.NGp, R, NG, bv, mbuf, hg_out);
    else mm_stage<4>(S.Cp, S.NGp, R, NG, bv, mbuf, hg_out);
    // bv (h) was complete before the last stage's first barrier.  Kx and the over-relaxed v of the coupling rows, 16 bytes
    // per thread and row segment, loads first:
    {
        const int n = R * 8;
        const float inv_rho = 1.f / rho, alpha = opt.alpha;
        for (int i0 = 0; i0 < n; i0 += 1024) {
            float4 tmp[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + tid + 256 * u;
                if (i < n) tmp[u] = *reinterpret_cast<const float4*>(VC + (size_t)(i >> 3) * Tp + t4 + 4 * (i & 7));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + tid + 256 * u;
                if (i < n) {
                    const float4 g4 = reinterpret_cast<const float4*>(gg)[i], h4 = reinterpret_cast<const float4*>(bv)[i], v4 = tmp[u];
                    const size_t o = (size_t)(i >> 3) * Tp + t4 + 4 * (i & 7);
                    // g = rho (2z - v):  z = (g/rho + v)/2
                    const float4 kx = make_float4((g4.x - h4.x) * inv_rho, (g4.y - h4.y) * inv_rho, (g4.z - h4.z) * inv_rho, (g4.w - h4.w) * inv_rho);
                    *reinterpret_cast<float4*>(KX + o) = kx;
                    *reinterpret_cast<float4*>(VC + o) = make_float4(v4.x + alpha * (kx.x - 0.5f * (g4.x * inv_rho + v4.x)), v4.y + alpha * (kx.y - 0.5f * (g4.y * inv_rho + v4.y)),
                                                                     v4.z + alpha * (kx.z - 0.5f * (g4.z * inv_rho + v4.z)), v4.w + alpha * (kx.w - 0.5f * (g4.w * inv_rho + v4.w)));
                }
            }
        }
    }
}

// one warp per instance: peak-epigraph level of the aggregate-power row
__global__ void k_level(SiteDev S, acb_batch B, GenWork W, GenDims D) {
    const int b = blockIdx.x, lane = threadIdx.x;
    if (W.status[b] >= 0 || !D.has_u) return;
    float* sc = W.scal + (size_t)b * GS_N;
    const float rho = sc[GS_RHO], Gamma = sc[GS_GAMMA], pk_w = sc[GS_PKW], pk_p0 = sc[GS_PKP0];
    const float su = S.row_scale[D.rU], rp = rho / (su * su), cur = rp + 2.f * Gamma;
    const int Tb = B.T[b], Tp = D.Tp;
    const float* vu = W.VC + ((size_t)b * D.R + D.rU) * Tp;
    const float* ext = B.ext ? B.ext + (size_t)b * Tp : nullptr;
    auto a_of = [&](int t) -> float { return (rp * (vu[t] * su) - 2.f * Gamma * (ext ? ext[t] : 0.f)) / cur; };
    float amax = -3.0e38f;
    for (int t = lane; t < Tb; t += 32) amax = fmaxf(amax, a_of(t));
    amax = wmax(amax);
    float pl = fmaxf(amax, pk_p0);
    if (pk_w > 0.f && amax > pk_p0) {
        float F0 = 0.f;
        for (int t = lane; t < Tb; t += 32) F0 += fmaxf(a_of(t) - pk_p0, 0.f);
        F0 = wsum(F0) * cur;
        if (F0 <= pk_w) pl = pk_p0;
        else {
            float p = fminf(fmaxf(sc[GS_PLEVEL], pk_p0), amax), lo = pk_p0, hi = amax;
            for (int step = 0; step < 24; ++step) {
                float F = 0.f;
                int na = 0;
                for (int t = lane; t < Tb; t += 32) { float a = a_of(t); if (a > p) { F += a - p; ++na; } }
                F = wsum(F) * cur - pk_w;
                na = __reduce_add_sync(0xffffffffu, na);
                if (fabsf(F) <= 1e-6f * pk_w) break;
                if (F > 0.f) lo = p; else hi = p;
                float pn = (na > 0) ? p + F / (cur * (float)na) : 0.5f * (lo + hi);
                if (!(pn > lo && pn < hi)) pn = 0.5f * (lo + hi);
                p = pn;
            }
            pl = p;
        }
    }
    if (lane == 0) sc[GS_PLEVEL] = pl;
}

// per instance: combine the check reductions, decide
__global__ void k_decide(acb_batch B, acb_options opt, GenWork W, GenDims D, int it, int last, int minor) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B.B || W.status[b] >= 0) return;
    float* sc = W.scal + (size_t)b * GS_N;
    double* da = W.dacc + (size_t)b * GD_N;
    const float rho = sc[GS_RHO], rho1 = opt.kappa * rho;
    double P = da[GD_P], Dv = da[GD_D];
    double mag = fabs(P);  // magnitude of the objective's terms (see the on-chip kernel: the terms can cancel)
    if (D.has_u) {
        const double gterm = (double)sc[GS_GAMMA] * da[GD_UQ] + (double)sc[GS_PKW] * (double)fmaxf(sc[GS_UMAX], sc[GS_PKP0]);
        P += gterm; mag += fabs(gterm);
        Dv += (double)sc[GS_PKW] * (double)fmaxf(sc[GS_ZUMAX], sc[GS_PKP0]);
    }
    mag = fmax(fabs(P), (double)opt.term_floor * mag);
    double Dbest = da[GD_DBEST];
    if (Dv == Dv && Dv > Dbest) Dbest = Dv;
    const double gap = P - Dbest, tol = (double)opt.eps_abs + (double)opt.eps_rel * fmax(mag, fabs(Dbest));
    const float viol = sc[GS_VIOL] - 4.f;
    const float rp = sc[GS_E1] + sc[GS_E2], rd = rho1 * (fabsf(opt.alpha - 1.f) * sc[GS_E1] + sc[GS_E2]);
    const float rp_rel = rp / fmaxf(sc[GS_XMAX], 1e-6f), rd_rel = rd / fmaxf(1.f, sc[GS_YMAX]);
    sc[GS_GAP] = (float)(gap / fmax(fmax(mag, fabs(Dbest)), 1e-30));
    sc[GS_RP] = rp_rel; sc[GS_RD] = rd_rel;
    const float viol_out = viol;
    int st = -1;
    float ratio_out = 1.f;
    if (!(P == P)) st = ACB_NUMERICAL;
    else if (Dbest > da[GD_PMAX] + 1e-3 * (fabs(da[GD_PMAX]) + 1.0)) st = ACB_INFEASIBLE;  // dual bound above the box maximum
    // (a slightly negative gap is rounding noise and passes.  A minor check may stop an instance only when it has no per-EVSE
    // quadratic term: with one the optimum is unique in the rates and callers compare rates, which the major-only schedule
    // had converged further than the gap alone demands)
    else if (gap <= tol && viol <= opt.viol_tol && !(minor && sc[GS_QD] > 0.f)) st = ACB_SOLVED;
    else if (last) st = ACB_MAX_ITER;
    else if (minor) {
        // stopping test only: rescues and the rho balance keep the time scale of the major checks
    } else if (opt.stall_checks > 0 && sc[GS_NRESCUE] < (float)(opt.max_rescues > 0 ? 1 : 0) &&
             ((fmax(gap, 0.1 * tol) < 0.9 * da[GD_BESTGAP]) ? (da[GD_BESTGAP] = fmax(gap, 0.1 * tol), sc[GS_STALL] = 0.f, false)
                                                          : ((sc[GS_STALL] += 1.f) >= (float)opt.stall_checks))) {
        // stagnation rescue as in the on-chip kernel: the gap has not improved by 10 % over stall_checks checks -> one
        // stiffer penalty, v and the multipliers rescaled so that y is kept
        const float rn = fminf(fmaxf(rho * 3.f, 1e-4f), 1e4f);
        ratio_out = rho / rn;
        sc[GS_RHO] = rn;
        sc[GS_NRESCUE] += 1.f;
        sc[GS_STALL] = 0.f;
        da[GD_BESTGAP] = 1.0e300;
    } else if (gap <= tol && opt.stall_checks > 0 && sc[GS_NFEAS] < 3.f &&
               ((viol < 0.9f * sc[GS_BESTVIOL]) ? (sc[GS_BESTVIOL] = viol, sc[GS_VSTALL] = 0.f, false) : ((sc[GS_VSTALL] += 1.f) >= (float)opt.stall_checks))) {
        // feasibility rescue: gap certified, violation no longer shrinking -> stiffer penalty (up to three times)
        const float rn = fminf(fmaxf(rho * 3.f, 1e-4f), 1e4f);
        ratio_out = rho / rn;
        sc[GS_RHO] = rn;
        sc[GS_NFEAS] += 1.f;
        sc[GS_VSTALL] = 0.f; sc[GS_BESTVIOL] = 3.0e38f; sc[GS_STALL] = 0.f;
        da[GD_BESTGAP] = 1.0e300;
    } else if (opt.adapt_rho) {
        float ratio = sqrtf(fmaxf(rp_rel, 1e-12f) / fmaxf(rd_rel, 1e-12f));
        if (ratio > 5.f || ratio < 0.2f) {
            float rn = fminf(fmaxf(rho * ratio, 1e-4f), 1e4f);
            ratio_out = rho / rn;
            sc[GS_RHO] = rn;
        }
    }
    W.iters[b] = it;
    // reset the accumulators for the next check; GS_E1 carries the v rescale factor to k_rows<5>/k_rescale_vc
    da[GD_P] = da[GD_D] = da[GD_UQ] = 0.0;
    if (!(minor && sc[GS_QD] > 0.f)) da[GD_DBEST] = Dbest;  // (such an instance sees the major checks only, bound included)
    sc[GS_E2] = sc[GS_XMAX] = sc[GS_YMAX] = sc[GS_UMAX] = sc[GS_ZUMAX] = 0.f;
    sc[GS_VIOL] = viol_out;  // kept for the stats; k_clear_viol resets it before the next check
    sc[GS_E1] = ratio_out;
    if (st >= 0) { W.status[b] = st; atomicAdd(W.ndone, 1); }
}

// coupling rows: v <- z + f (v - z) after a rho change (f in GS_E1, rho already new: z uses the OLD rho = rho_new * f... see below)
__global__ void k_rescale_vc(SiteDev S, acb_batch B, GenWork W, GenDims D) {
    const int b = blockIdx.y;
    if (W.status[b] >= 0) return;
    float* sc = W.scal + (size_t)b * GS_N;
    const float f = sc[GS_E1];
    if (f == 1.f) return;
    const int Tp = D.Tp, R = D.R, t = blockIdx.x * blockDim.x + threadIdx.x, Tb = B.T[b];
    // mu = (energy-row dual) / rho1 scales with the penalty like v - z does (k_rows<5> ran before this kernel)
    if (blockIdx.x == 0)
        for (int s2 = threadIdx.x; s2 < B.S_max; s2 += blockDim.x) W.MU[(size_t)b * B.S_max + s2] *= f;
    if (t >= Tp) return;
    const float rho_old = sc[GS_RHO] * f;  // GS_RHO already holds the new value
    const float Gamma = sc[GS_GAMMA], pk_w = sc[GS_PKW], plevel = sc[GS_PLEVEL];
    const float su = D.has_u ? S.row_scale[D.rU] : 1.f;
    const float linLo = D.lin_two_sided ? -1.f : -3.0e38f;
    float* VC = W.VC + (size_t)b * R * Tp;
    int r = 0;
    for (int j = 0; j < D.nDisc; ++j, r += 2) {
        float a = VC[r * Tp + t], bb = VC[(r + 1) * Tp + t], za, zb;
        proj_disc(a, bb, S.lim[r], za, zb);
        VC[r * Tp + t] = za + f * (a - za); VC[(r + 1) * Tp + t] = zb + f * (bb - zb);
    }
    for (int j = 0; j < D.nLin; ++j, ++r) {
        float v = VC[r * Tp + t], z = clampf(v, (linLo < -1.0e30f) ? linLo : linLo * S.lim[r], S.lim[r]);
        VC[r * Tp + t] = z + f * (v - z);
    }
    if (D.has_pl) {
        float cap = (B.peak_limit && t < Tb) ? B.peak_limit[(size_t)b * Tp + t] / S.row_scale[D.rPL] : 3.0e38f;
        float v = VC[r * Tp + t], z = fminf(v, cap);
        VC[r * Tp + t] = z + f * (v - z);
        ++r;
    }
    if (D.has_u) {
        float rp = rho_old / (su * su);
        float e = (B.ext && t < Tb) ? B.ext[(size_t)b * Tp + t] : 0.f;
        float v = VC[r * Tp + t], a = (rp * (v * su) - 2.f * Gamma * e) / (rp + 2.f * Gamma);
        float z = ((pk_w > 0.f) ? fminf(a, plevel) : a) / su;
        VC[r * Tp + t] = z + f * (v - z);
    }
}

__global__ void k_clear_check(GenWork W, int B_) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B_ || W.status[b] >= 0) return;  // a finished instance keeps its last violation for the stats
    float* sc = W.scal + (size_t)b * GS_N;
    sc[GS_VIOL] = 0.f;  // encoded as viol + 4 by the atomic max
    sc[GS_E1] = sc[GS_E2] = sc[GS_XMAX] = sc[GS_YMAX] = 0.f;
}

__global__ void k_finish(acb_batch B, GenWork W, GenDims D) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B.B) return;
    const float* sc = W.scal + (size_t)b * GS_N;
    int st = W.status[b];
    B.status[b] = st < 0 ? ACB_MAX_ITER : st;
    B.iters[b] = W.iters[b];
    float* o = B.stats + (size_t)b * ACB_NSTATS;
    o[0] = sc[GS_RP]; o[1] = sc[GS_RD]; o[2] = sc[GS_GAP]; o[3] = sc[GS_VIOL]; o[4] = sc[GS_RHO]; o[5] = sc[GS_CS]; o[6] = 0.f; o[7] = 0.f;
    if (B.out_scal) { B.out_scal[b * 2] = sc[GS_RHO]; B.out_scal[b * 2 + 1] = sc[GS_PLEVEL]; }
    if (B.out_mu)  // (empty session slots: 0, as on chip; k_setup leaves their W.MU unset)
        for (int s = 0; s < B.S_max; ++s) B.out_mu[(size_t)b * B.S_max + s] = s < B.n_sessions[b] ? W.MU[(size_t)b * B.S_max + s] : 0.f;
}

template <int Q>
int run_general(acb_site* site, const acb_batch* batch, const acb_options& opt, cudaStream_t st) {
    const SiteDev& d = site->d;
    const int B = batch->B, Tp = batch->Tp, N = d.N, R = d.R, NG = d.NG;
    GenDims D{N, R, NG, Tp, Tp / 32, batch->S_max, d.nDisc, d.nLin, d.has_pl, d.has_u, 2 * d.nDisc + d.nLin, 2 * d.nDisc + d.nLin + d.has_pl, d.lin_two_sided};
    // workspace
    const size_t nNT = (size_t)B * N * Tp, nRT = (size_t)B * std::max(R, 1) * Tp, nGT = (size_t)B * NG * Tp;
    const size_t floats = nNT + 2 * nRT + 3 * nGT + (size_t)B * batch->S_max + 2 * (size_t)B * Tp + (size_t)B * GS_N;
    const size_t bytes = floats * sizeof(float) + (size_t)B * GD_N * sizeof(double) + ((size_t)B * (2 + 2 * N) + 4) * sizeof(int) + 256;
    {
        // keep the stream-ordered pool's memory across calls (the default threshold of 0 gives it back at every sync)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, site->device) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    char* base = nullptr;
    ACB_CUDA(cudaMallocAsync((void**)&base, bytes, st));
    GenWork W;
    char* p = base;
    auto take = [&](size_t n, size_t sz) { void* r = p; p += ((n * sz + 15) / 16) * 16; return r; };
    W.dacc = (double*)take((size_t)B * GD_N, 8);
    W.V = (float*)take(nNT, 4);
    W.VC = (float*)take(nRT, 4); W.KX = (float*)take(nRT, 4);
    W.SG = (float*)take(nGT, 4); W.SGZ = (float*)take(nGT, 4); W.HG = (float*)take(nGT, 4);
    W.MU = (float*)take((size_t)B * batch->S_max, 4);
    W.AL = (float*)take((size_t)B * Tp, 4); W.BE = (float*)take((size_t)B * Tp, 4);
    W.scal = (float*)take((size_t)B * GS_N, 4);
    W.status = (int*)take(B, 4); W.iters = (int*)take(B, 4);
    W.row_first = (int*)take((size_t)B * N, 4); W.row_cnt = (int*)take((size_t)B * N, 4);
    W.ndone = (int*)take(1, 4);
    ACB_CUDA(cudaMemsetAsync(W.ndone, 0, sizeof(int), st));
    ACB_CUDA(cudaMemsetAsync(W.HG, 0, nGT * sizeof(float), st));
    // row kernels: registers (Q > 0: 8 warps, Tp floats of partial sums each) or shared-memory staging (Q = 0: as many
    // warps as fit, 4 Tp floats each)
    // (register path: 2 warps per block, measured: 4 warps 134 us, 2 warps 128 us, 1 warp 138 us per launch on the 1000-EVSE site —
    // a warp pays its chain of dependent table loads once, so more rows per warp amortise it; one warp alone hides too little)
    int row_threads = 64;
    size_t row_smem = (size_t)2 * Tp * sizeof(float);
    if (Q == 0) {
        const int nw = (int)std::max<size_t>(1, std::min<size_t>(8, (size_t)232448 / ((size_t)16 * Tp)));
        row_threads = 32 * nw;
        row_smem = (size_t)nw * 4 * Tp * sizeof(float);
        if (row_smem > 232448) { acb_set_error("acb_solve_batch (general path): horizon too long for the shared-memory row staging"); cudaFreeAsync(base, st); return ACB_E_TOO_LARGE; }
    }
    if (row_smem > 48 * 1024) {
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
        ACB_CUDA(cudaFuncSetAttribute(k_rows<Q, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem));
    }
#define ROWS(MODE) k_rows<Q, MODE><<<grow, row_threads, row_smem, st>>>(d, *batch, opt, W, D, site->grp_off_dev)
    const dim3 grow(NG, B), gcol((Tp + 32 * ACB_CPL - 1) / (32 * ACB_CPL), B);
    k_setup<<<B, 256, 0, st>>>(d, *batch, opt, W, D);
    ROWS(6);
    if (!batch->lb_zero) ROWS(7);
    k_setup_agg<<<B, 256, 0, st>>>(d, *batch, W, D, batch->lb_zero ? 0 : 1);
    const size_t smem_cols = ((size_t)(NG + std::max(R, 1) + std::max(d.Rp, 4)) * 32 * ACB_CPL + (size_t)MM_KC * 128) * sizeof(float);
    const size_t smem_it = ((size_t)MM_KC * 128 + (size_t)(std::max(NG, std::max(d.nEigp, 4)) + std::max(R, 1) + std::max(d.Rp, 4)) * 32) * sizeof(float);
    if (smem_it > 48 * 1024) ACB_CUDA(cudaFuncSetAttribute(k_cols_it, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_it));
    if (smem_cols > 48 * 1024) {
        ACB_CUDA(cudaFuncSetAttribute(k_cols_check, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cols));
    }
    ROWS(1);
    // Check schedule.  "Major" checks (stopping test, rescues, rho balance) at ACB_FIRST_CHECK and then every check_every
    // iterations, as on chip.  Between them, while the iteration count is still small, "minor" checks that only ask whether
    // the certified gap already allows the instance to stop (at it + max(5, it/4); instances without a per-EVSE quadratic
    // term only, see k_decide): they change nothing in the iteration, so the trajectory is the one of the major-only
    // schedule, an instance just leaves earlier (config 5 certifies at iteration 20 instead of 35: 9.6 -> 6.5 ms per 128
    // instances); from iteration ~100 on only the major checks remain.
    int h_done = 0, it = 0, next_major = std::min(ACB_FIRST_CHECK, opt.check_every);
    while (it < opt.max_iter) {
        int target = (it == 0) ? next_major : std::min(next_major, it + std::max(5, it / 4));
        target = std::min(target, opt.max_iter);
        const bool major = (target >= next_major) || (target >= opt.max_iter);
        const int burst = target - it;
        for (int k = 0; k < burst; ++k) {
            k_cols_it<<<gcol, 256, smem_it, st>>>(d, *batch, opt, W, D);
            k_level<<<B, 32, 0, st>>>(d, *batch, W, D);
            if (k == burst - 1) {
                k_clear_check<<<(B + 127) / 128, 128, 0, st>>>(W, B);
                ROWS(0);
            } else
                ROWS(8);
        }
        it = target;
        // check
        ROWS(2);
        k_cols_check<<<gcol, 256, smem_cols, st>>>(d, *batch, opt, W, D);
        ROWS(3);
        k_decide<<<(B + 127) / 128, 128, 0, st>>>(*batch, opt, W, D, it, it >= opt.max_iter ? 1 : 0, major ? 0 : 1);
        if (major) {
            ROWS(5);
            k_rescale_vc<<<dim3((Tp + 127) / 128, B), 128, 0, st>>>(d, *batch, W, D);
            ROWS(1);  // SG for the next column pass
            if (target >= next_major) next_major += opt.check_every;
        }
        // (a minor check leaves v, the multipliers and SG as the last iteration wrote them; HG is rebuilt by the next column pass)
        ACB_CUDA(cudaMemcpyAsync(&h_done, W.ndone, sizeof(int), cudaMemcpyDeviceToHost, st));
        ACB_CUDA(cudaStreamSynchronize(st));
        if (h_done >= B) break;
    }
    ROWS(4);
    k_finish<<<(B + 127) / 128, 128, 0, st>>>(*batch, W, D);
    if (batch->out_vc) ACB_CUDA(cudaMemcpyAsync(batch->out_vc, W.VC, nRT * sizeof(float), cudaMemcpyDeviceToDevice, st));
    ACB_CUDA(cudaGetLastError());
    ACB_CUDA(cudaFreeAsync(base, st));
    return ACB_OK;
#undef ROWS
}

}  // namespace

int acb_solve_general(acb_site* site, const acb_batch* batch, const acb_options& opt, cudaStream_t st) {
    const int Q = batch->Tp / 32;
    if (Q == 2) return run_general<2>(site, batch, opt, st);
    if (Q == 4) return run_general<4>(site, batch, opt, st);
    if (Q == 5) return run_general<5>(site, batch, opt, st);
    if (Q == 9) return run_general<9>(site, batch, opt, st);
    return run_general<0>(site, batch, opt, st);  // any other multiple of 32: rows staged in shared memory
}
