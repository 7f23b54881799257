// Site construction: turns the InfrastructureInfo arrays into the constants the kernels
// use (scaled coupling matrix, electrically-distinct EVSE groups, row -> warp slots,
// eigen-decomposition of Khat Khat', float64 postprocessing rows).
// Replaces the per-call Python work of reference
// adacharge/adaptive_charging_optimization.py:152-172 and adacharge/utils.py:6-8.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include "acb_common.cuh"

static thread_local std::string g_err;
void acb_set_error(const std::string& s) { g_err = s; }
extern "C" const char* acb_last_error(void) { return g_err.c_str(); }
extern "C" int acb_version(void) { return ACB_VERSION; }

extern "C" void acb_default_options(acb_options* o) {
    o->eps_abs = 1e-5f;
    o->eps_rel = 1e-4f;
    o->viol_tol = 1e-5f;
    o->viol_abs = 1e-3f;
    o->rho0 = 0.07f;
    o->kappa = 0.7f;
    o->alpha = 1.8f;
    o->max_iter = 20000;
    o->check_every = 25;
    o->equality = 0;
    o->adapt_rho = 0;  // residual balancing measured worse than the fixed penalty + stagnation rescue on every workload tried
    o->restart = 1;
    o->avg_every = 5;
    o->stall_checks = 2;
    o->max_rescues = 1;  // a 2nd rescue (cold reset of a warm-started solve) measured worse on the 1024-site replay
    o->stall_exit = 0;
    o->dual_refine = 1;
    o->term_floor = 0.05f;
    o->rho_curv = 1.0f;
    o->path = 0;
    o->rate_tol = 3e-4f;
    o->polish_min_qd = 5e-4f;
    o->newton_rel = 0.25f;
    o->phase_iters = 0;
}

// cyclic Jacobi eigen-decomposition of a symmetric n x n matrix (row-major), double.
static void jacobi_eigh(std::vector<double>& A, int n, std::vector<double>& V, std::vector<double>& w) {
    V.assign((size_t)n * n, 0.0);
    for (int i = 0; i < n; ++i) V[(size_t)i * n + i] = 1.0;
    for (int sweep = 0; sweep < 100; ++sweep) {
        double off = 0;
        for (int p = 0; p < n; ++p)
            for (int q = p + 1; q < n; ++q) off += A[(size_t)p * n + q] * A[(size_t)p * n + q];
        if (off < 1e-30) break;
        for (int p = 0; p < n; ++p)
            for (int q = p + 1; q < n; ++q) {
                double apq = A[(size_t)p * n + q];
                if (std::fabs(apq) < 1e-300) continue;
                double app = A[(size_t)p * n + p], aqq = A[(size_t)q * n + q];
                double theta = (aqq - app) / (2 * apq);
                double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1));
                double c = 1 / std::sqrt(t * t + 1), s = t * c;
                for (int k = 0; k < n; ++k) {
                    double akp = A[(size_t)k * n + p], akq = A[(size_t)k * n + q];
                    A[(size_t)k * n + p] = c * akp - s * akq;
                    A[(size_t)k * n + q] = s * akp + c * akq;
                }
                for (int k = 0; k < n; ++k) {
                    double apk = A[(size_t)p * n + k], aqk = A[(size_t)q * n + k];
                    A[(size_t)p * n + k] = c * apk - s * aqk;
                    A[(size_t)q * n + k] = s * apk + c * aqk;
                }
                for (int k = 0; k < n; ++k) {
                    double vkp = V[(size_t)k * n + p], vkq = V[(size_t)k * n + q];
                    V[(size_t)k * n + p] = c * vkp - s * vkq;
                    V[(size_t)k * n + q] = s * vkp + c * vkq;
                }
            }
    }
    w.resize(n);
    for (int i = 0; i < n; ++i) w[i] = std::max(0.0, A[(size_t)i * n + i]);
}

template <typename T>
static int upload(acb_site* s, const std::vector<T>& h, const T** dptr) {
    void* p = nullptr;
    size_t bytes = std::max<size_t>(1, h.size()) * sizeof(T);
    ACB_CUDA(cudaMalloc(&p, bytes));
    s->allocs.push_back(p);
    if (!h.empty()) ACB_CUDA(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    *dptr = (const T*)p;
    return ACB_OK;
}

extern "C" int acb_site_create(acb_site** out, int device, int N, int M, const double* cm,
                               const double* phases_deg, const double* limits, const double* voltages,
                               int constraint_type, int use_peak_row, int use_agg_row,
                               const double* max_pilot, const int32_t* allow_off, const double* allow_vals) {
    if (!out || N <= 0 || M < 0 || !voltages || (M > 0 && (!cm || !limits))) {
        acb_set_error("acb_site_create: bad arguments");
        return ACB_E_INVALID;
    }
    if (constraint_type != ACB_SOC && constraint_type != ACB_LINEAR) {
        acb_set_error("acb_site_create: constraint_type must be ACB_SOC or ACB_LINEAR");
        return ACB_E_INVALID;
    }
    if (M > 0 && constraint_type == ACB_SOC && !phases_deg) {
        acb_set_error("phases is required when using SOC infrastructure constraints.");
        return ACB_E_INVALID;
    }
    ACB_CUDA(cudaSetDevice(device));
    acb_site* s = new acb_site();
    s->device = device;
    s->constraint_type = constraint_type;
    SiteDev& d = s->d;
    memset(&d, 0, sizeof(d));
    d.N = N;
    d.M = M;
    d.has_pl = use_peak_row ? 1 : 0;
    d.has_u = use_agg_row ? 1 : 0;

    // float64 rows exactly as the reference forms them (utils.py:6-8)
    std::vector<double> acos_((size_t)M * N, 0.0), asin_((size_t)M * N, 0.0);
    if (M > 0 && phases_deg) {
        for (int j = 0; j < M; ++j)
            for (int i = 0; i < N; ++i) {
                double rad = phases_deg[i] * (M_PI / 180.0);
                acos_[(size_t)j * N + i] = cm[(size_t)j * N + i] * std::cos(rad);
                asin_[(size_t)j * N + i] = cm[(size_t)j * N + i] * std::sin(rad);
            }
    }
    // SOC rows whose EVSEs all share one phase angle have colinear components:
    // ||(c s, s' s)|| = |s| with s = sum_i A_ji r_i, i.e. an exact two-sided linear row.  They are
    // kept as single rows (half the coupling rows on the Caltech site).
    std::vector<int> discRows, absRows;
    if (constraint_type == ACB_SOC) {
        for (int j = 0; j < M; ++j) {
            bool same = true, any = false;
            double ph0 = 0;
            for (int i = 0; i < N; ++i)
                if (cm[(size_t)j * N + i] != 0.0) {
                    if (!any) { ph0 = phases_deg[i]; any = true; }
                    else if (phases_deg[i] != ph0) same = false;
                }
            if (same) absRows.push_back(j); else discRows.push_back(j);
        }
    }
    d.nDisc = (int)discRows.size();
    d.nLin = (constraint_type == ACB_LINEAR) ? M : (int)absRows.size();
    d.lin_two_sided = (constraint_type == ACB_SOC) ? 1 : 0;
    const int R = 2 * d.nDisc + d.nLin + d.has_pl + d.has_u;
    d.R = R;
    // scaled coupling matrix
    std::vector<double> K((size_t)R * N, 0.0), scale(R, 1.0), lim(R, 0.0), kv(N);
    for (int i = 0; i < N; ++i) kv[i] = voltages[i] / 1e3;
    int r = 0;
    for (int jj = 0; jj < d.nDisc; ++jj, r += 2) {
        const int j = discRows[jj];
        double ss = 0;
        for (int i = 0; i < N; ++i)
            ss += acos_[(size_t)j * N + i] * acos_[(size_t)j * N + i] + asin_[(size_t)j * N + i] * asin_[(size_t)j * N + i];
        double sc = std::sqrt(ss / 2);
        if (!(sc > 0)) sc = 1;
        for (int i = 0; i < N; ++i) {
            K[(size_t)r * N + i] = acos_[(size_t)j * N + i] / sc;
            K[(size_t)(r + 1) * N + i] = asin_[(size_t)j * N + i] / sc;
        }
        scale[r] = scale[r + 1] = sc;
        lim[r] = lim[r + 1] = limits[j] / sc;
    }
    for (int jj = 0; jj < d.nLin; ++jj, ++r) {
        const int j = (constraint_type == ACB_LINEAR) ? jj : absRows[jj];
        double ss = 0;
        for (int i = 0; i < N; ++i) ss += cm[(size_t)j * N + i] * cm[(size_t)j * N + i];
        double sc = std::sqrt(ss);
        if (!(sc > 0)) sc = 1;
        for (int i = 0; i < N; ++i)
            K[(size_t)r * N + i] = ((constraint_type == ACB_LINEAR) ? std::fabs(cm[(size_t)j * N + i]) : cm[(size_t)j * N + i]) / sc;
        scale[r] = sc;
        lim[r] = limits[j] / sc;
    }
    if (d.has_pl) {
        double sc = std::sqrt((double)N);
        for (int i = 0; i < N; ++i) K[(size_t)r * N + i] = 1.0 / sc;
        scale[r] = sc;
        ++r;
    }
    if (d.has_u) {
        double ss = 0;
        for (int i = 0; i < N; ++i) ss += kv[i] * kv[i];
        double sc = std::sqrt(ss);
        for (int i = 0; i < N; ++i) K[(size_t)r * N + i] = kv[i] / sc;
        scale[r] = sc;
        ++r;
    }
    // electrically distinct groups: identical Khat column and identical kW/A
    std::map<std::vector<double>, int> gmap;
    std::vector<int> grp(N), gfirst;
    for (int i = 0; i < N; ++i) {
        std::vector<double> key(R + 1);
        for (int q = 0; q < R; ++q) key[q] = K[(size_t)q * N + i];
        key[R] = kv[i];
        auto it = gmap.find(key);
        if (it == gmap.end()) {
            int g = (int)gfirst.size();
            gmap[key] = g;
            gfirst.push_back(i);
            grp[i] = g;
        } else
            grp[i] = it->second;
    }
    const int NG = (int)gfirst.size();
    d.NG = NG;
    // slots: EVSEs ordered by group, TPW per warp
    int TPW = 3;  // EVSE rows per warp of the on-chip kernel (3 rows, 768-thread blocks, 80 registers: fastest of 2/3/4 measured)
    while ((N + TPW - 1) / TPW > ACB_MAX_WARPS) ++TPW;
    d.TPW = TPW;
    d.nRowWarps = (N + TPW - 1) / TPW;
    d.nSlots = d.nRowWarps * TPW;
    std::vector<int> order(N);
    for (int i = 0; i < N; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return grp[a] < grp[b]; });
    std::vector<int> slot_row(d.nSlots, -1), slot_grp(d.nSlots, 0), slot_prow(d.nSlots, 0), slot_first(d.nSlots, 0);
    std::vector<int> pg_off(NG + 1, 0);
    int np = 0;
    for (int sl = 0; sl < d.nSlots; ++sl) {
        if (sl >= N) continue;
        int i = order[sl], g = grp[i];
        slot_row[sl] = i;
        slot_grp[sl] = g;
        bool newp = (sl % TPW == 0) || slot_grp[sl - 1] != g;
        if (newp) {
            slot_first[sl] = 1;
            slot_prow[sl] = np++;
            pg_off[g + 1]++;
        } else
            slot_prow[sl] = slot_prow[sl - 1];
    }
    for (int g = 0; g < NG; ++g) pg_off[g + 1] += pg_off[g];
    d.NP = np;
    std::vector<float> ngrp(NG, 0.f), kg(NG), Cf((size_t)R * NG), Uf((size_t)R * R), lamf(R), scf(R), limf(R);
    for (int i = 0; i < N; ++i) ngrp[grp[i]] += 1.f;
    for (int g = 0; g < NG; ++g) {
        kg[g] = (float)kv[gfirst[g]];
        for (int q = 0; q < R; ++q) Cf[(size_t)q * NG + g] = (float)K[(size_t)q * N + gfirst[g]];
    }
    std::vector<double> KKt((size_t)R * R, 0.0), V, w;
    for (int a = 0; a < R; ++a)
        for (int b = 0; b < R; ++b) {
            double acc = 0;
            for (int i = 0; i < N; ++i) acc += K[(size_t)a * N + i] * K[(size_t)b * N + i];
            KKt[(size_t)a * R + b] = acc;
        }
    jacobi_eigh(KKt, R, V, w);
    for (int a = 0; a < R; ++a) {
        lamf[a] = (float)w[a];
        scf[a] = (float)scale[a];
        limf[a] = (float)lim[a];
        for (int b = 0; b < R; ++b) Uf[(size_t)a * R + b] = (float)V[(size_t)a * R + b];
    }
    std::vector<double> lim64(limits, limits + M), mp(N, 0.0);
    if (max_pilot) mp.assign(max_pilot, max_pilot + N);
    std::vector<int> aoff(N + 1, 0);
    std::vector<double> avals;
    if (allow_off && allow_vals) {
        aoff.assign(allow_off, allow_off + N + 1);
        avals.assign(allow_vals, allow_vals + allow_off[N]);
    }
    d.nAllow = (int)avals.size();
    int rc = ACB_OK;
#define UP(vec, field) if ((rc = upload(s, vec, &d.field)) != ACB_OK) { acb_site_destroy(s); return rc; }
    UP(slot_row, slot_row) UP(slot_grp, slot_grp) UP(slot_prow, slot_prow) UP(slot_first, slot_first)
    UP(pg_off, pg_off) UP(ngrp, ngrp) UP(kg, kg) UP(Cf, C) UP(Uf, U) UP(lamf, lam) UP(scf, row_scale) UP(limf, lim)
    {
        std::vector<int> goff(NG + 1, 0);
        for (int g = 0; g < NG; ++g) goff[g + 1] = goff[g] + (int)ngrp[g];
        if ((rc = upload(s, goff, &s->grp_off_dev)) != ACB_OK) { acb_site_destroy(s); return rc; }
    }
    {
        const int Rp = (R + 3) & ~3;
        d.Rp = Rp;
        std::vector<float> up((size_t)std::max(R, 1) * std::max(Rp, 4), 0.f), ut((size_t)std::max(R, 1) * std::max(Rp, 4), 0.f);
        for (int a = 0; a < R; ++a)
            for (int b2 = 0; b2 < R; ++b2) { up[(size_t)a * Rp + b2] = Uf[(size_t)a * R + b2]; ut[(size_t)a * Rp + b2] = Uf[(size_t)b2 * R + a]; }
        if ((rc = upload(s, up, &d.Up)) != ACB_OK) { acb_site_destroy(s); return rc; }
        if ((rc = upload(s, ut, &d.Ut)) != ACB_OK) { acb_site_destroy(s); return rc; }
        const int NGp = (NG + 3) & ~3;
        d.NGp = NGp;
        std::vector<float> cp((size_t)std::max(R, 1) * NGp, 0.f), ct((size_t)NG * std::max(Rp, 4), 0.f);
        for (int a = 0; a < R; ++a)
            for (int g = 0; g < NG; ++g) { cp[(size_t)a * NGp + g] = Cf[(size_t)a * NG + g]; ct[(size_t)g * Rp + a] = Cf[(size_t)a * NG + g]; }
        if ((rc = upload(s, cp, &d.Cp)) != ACB_OK) { acb_site_destroy(s); return rc; }
        if ((rc = upload(s, ct, &d.Ct)) != ACB_OK) { acb_site_destroy(s); return rc; }
        // eigenvectors with a non-zero eigenvalue (the others are null directions of Khat Khat': rank <= NG)
        double wmax = 0.0;
        for (int e = 0; e < R; ++e) wmax = std::max(wmax, w[e]);
        std::vector<int> nz;
        for (int e = 0; e < R; ++e)
            if (w[e] > 1e-9 * wmax) nz.push_back(e);
        const int nE = (int)nz.size(), nEp = (nE + 3) & ~3;
        d.nEig = nE;
        d.nEigp = nEp;
        std::vector<float> urp((size_t)std::max(R, 1) * std::max(nEp, 4), 0.f), urt((size_t)std::max(nE, 1) * std::max(Rp, 4), 0.f), lamr(std::max(nE, 1), 0.f);
        for (int j = 0; j < nE; ++j) {
            lamr[j] = lamf[nz[j]];
            for (int a = 0; a < R; ++a) { urp[(size_t)a * nEp + j] = Uf[(size_t)a * R + nz[j]]; urt[(size_t)j * Rp + a] = Uf[(size_t)a * R + nz[j]]; }
        }
        if ((rc = upload(s, urp, &d.Urp)) != ACB_OK) { acb_site_destroy(s); return rc; }
        if ((rc = upload(s, urt, &d.Urt)) != ACB_OK) { acb_site_destroy(s); return rc; }
        if ((rc = upload(s, lamr, &d.lamr)) != ACB_OK) { acb_site_destroy(s); return rc; }
    }
    UP(acos_, a_cos) UP(asin_, a_sin) UP(lim64, limits) UP(mp, max_pilot) UP(aoff, allow_off) UP(avals, allow_vals)
    {
        // CSR of the nonzero entries of the SOC rows, by row (columns ascending) and by EVSE (rows ascending)
        std::vector<int> rc_off(M + 1, 0), rc_col, er_cnt(N + 1, 0), er_off(N + 1, 0), er_rows;
        std::vector<double> rc_cos, rc_sin;
        for (int j = 0; j < M; ++j) {
            for (int i = 0; i < N; ++i) {
                const double c = acos_[(size_t)j * N + i], sn = asin_[(size_t)j * N + i];
                if (c != 0.0 || sn != 0.0) { rc_col.push_back(i); rc_cos.push_back(c); rc_sin.push_back(sn); ++er_cnt[i + 1]; }
            }
            rc_off[j + 1] = (int)rc_col.size();
        }
        for (int i = 0; i < N; ++i) er_off[i + 1] = er_off[i] + er_cnt[i + 1];
        er_rows.resize(rc_col.size());
        std::vector<int> fill(er_off.begin(), er_off.end() - 1);
        for (int j = 0; j < M; ++j)
            for (int p = rc_off[j]; p < rc_off[j + 1]; ++p) er_rows[fill[rc_col[p]]++] = j;
        UP(er_off, evse_row_off) UP(er_rows, evse_rows) UP(rc_off, row_col_off) UP(rc_col, row_cols) UP(rc_cos, row_cos) UP(rc_sin, row_sin)
    }
    {
        std::vector<double> volt64(voltages, voltages + N);
        UP(volt64, volt)
    }
#undef UP
    // second slot layout, two EVSE rows per warp, for the FAST on-chip variant (v in shared memory, 1024-thread blocks:
    // with no per-element state in registers more, smaller warps hide the latencies better)
    s->has_d2 = 0;
    if ((N + 1) / 2 <= ACB_MAX_WARPS) {
        SiteDev& e = s->d2;
        e = d;
        e.TPW = 2;
        e.nRowWarps = (N + 1) / 2;
        e.nSlots = e.nRowWarps * 2;
        std::vector<int> s_row(e.nSlots, -1), s_grp(e.nSlots, 0), s_prow(e.nSlots, 0), s_first(e.nSlots, 0), p_off(NG + 1, 0);
        int np2 = 0;
        for (int sl = 0; sl < e.nSlots && sl < N; ++sl) {
            const int i = order[sl], g = grp[i];
            s_row[sl] = i;
            s_grp[sl] = g;
            const bool newp = (sl % 2 == 0) || s_grp[sl - 1] != g;
            if (newp) { s_first[sl] = 1; s_prow[sl] = np2++; p_off[g + 1]++; }
            else s_prow[sl] = s_prow[sl - 1];
        }
        for (int g = 0; g < NG; ++g) p_off[g + 1] += p_off[g];
        e.NP = np2;
        if ((rc = upload(s, s_row, &e.slot_row)) != ACB_OK || (rc = upload(s, s_grp, &e.slot_grp)) != ACB_OK ||
            (rc = upload(s, s_prow, &e.slot_prow)) != ACB_OK || (rc = upload(s, s_first, &e.slot_first)) != ACB_OK ||
            (rc = upload(s, p_off, &e.pg_off)) != ACB_OK) { acb_site_destroy(s); return rc; }
        s->has_d2 = 1;
    }
    *out = s;
    return ACB_OK;
}

extern "C" void acb_site_destroy(acb_site* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    for (void* p : s->allocs) cudaFree(p);
    delete s;
}

extern "C" int acb_site_dims(const acb_site* s, int* N, int* M, int* R, int* NG, int* NP) {
    if (!s) return ACB_E_INVALID;
    if (N) *N = s->d.N;
    if (M) *M = s->d.M;
    if (R) *R = s->d.R;
    if (NG) *NG = s->d.NG;
    if (NP) *NP = s->d.NP;
    return ACB_OK;
}

extern "C" int acb_site_max_horizon(const acb_site* s) {
    if (!s) return 0;
    int best = 0;
    for (int Tp = 32; Tp <= 288; Tp += 32)
        if (acb_solve_smem_bytes(s->d, Tp, 64, 32) <= 232448) best = Tp;
    return best;
}
