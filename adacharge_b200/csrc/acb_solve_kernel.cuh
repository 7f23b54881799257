// Batched MPC solve (kernel template; instantiated per horizon in acb_solve_q*.cu): one thread block per instance, all solver state on chip.
//
// Replaces AdaptiveChargingOptimization.build_problem + solve (reference
// adacharge/adaptive_charging_optimization.py:220-321, i.e. cvxpy canonicalisation and
// the ECOS interior-point solve) and the objective library (:363-408) by an
// over-relaxed, restarted ADMM on the split
//     minimise  c'r + qd|r|^2 + g(Khat r_t)   s.t.  r in B,
// B = charging-rate box (aco.py:61-79) intersected with the per-session energy rows
// (aco.py:105-123), Khat = scaled [A cos(phi); A sin(phi)] / |A| rows (aco.py:156-172),
// the peak-limit row (aco.py:196-197) and the aggregate-power row used by
// peak / demand_charge / load_flattening (aco.py:387-408).
//
// Per iteration (DESIGN.md "solve kernel"):
//   column pass  : per period t, group sums of q = 2 z - v over electrically identical
//                  EVSEs, then ONE (NG+R) x (NG+R) matrix apply that yields both
//                  Khat'h (per group) and Khat x (per coupling row).
//   row pass     : per EVSE row (one warp, lanes over t): x, over-relaxed v update,
//                  projection onto box ∩ energy row by a warm-started safeguarded
//                  Newton on the multiplier (warp reductions);
//                  per coupling row: v update; disc / half-line projections; peak
//                  epigraph level by Newton.
//   every check_every iterations: a rigorous duality gap.  P = objective of a candidate
//   schedule that satisfies box and energy rows exactly; D = Lagrangian lower bound that
//   dualises only the coupling and energy rows (the box keeps the inner minimum finite, so
//   ANY multipliers give a valid bound).  Candidates: the current z and the projection of
//   the running average of v; when the averaged candidate's gap has halved the iteration
//   restarts from the average (restarted averaging gives linear convergence on the
//   LP-like instances).  Stop when P - D <= eps_abs + eps_rel max(|P|,|D|) and the
//   candidate's relative coupling violation <= viol_tol.
// State: v (N x Tp) in registers, coupling v (R x Tp), bounds and partial sums in
// shared memory; HBM is touched at load/store and for the running average only.
#pragma once
#include <cfloat>
#include <type_traits>
#include "acb_common.cuh"

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

// projection of (a, b) onto the disc of radius lim: (a, b) * disc_scale(a, b, lim)
__device__ __forceinline__ float disc_scale(float a, float b, float lim) {
    float n2 = a * a + b * b;
    return (n2 > lim * lim) ? lim * rsqrtf(n2) : 1.0f;
}
__device__ __forceinline__ void proj_disc(float a, float b, float lim, float& za, float& zb) {
    const float f = disc_scale(a, b, lim);
    za = a * f;
    zb = b * f;
}

// shared-memory layout (in floats), computed identically on host and device
struct SmemLayout {
    int LB, UB, PART, VC, VOUT, GIN, HG, THC, THA, ALPHA, BETA, PLIM, EBAR, MFT, CS, SESS_A, SESS_B, SESS_E, SESS_MU, SESS_MU2, SESS_NF, SESS_Q, ROWHI,
        SLOT, PGOFF, NGRP, KG, LIM, SCALE, REDF, REDD, SCAL, SCALD, total;
    int OP;  // padded output count of MFT
};
__host__ __device__ inline SmemLayout make_layout(int N, int R, int NG, int NP, int nSlots, int Tp, int S_max, int nwarps) {
    SmemLayout L;
    int o = 0;
    auto take = [&](int n) { int p = o; o += (n + 3) & ~3; return p; };
    L.OP = ((NG + R + ACB_OHT - 1) / ACB_OHT) * ACB_OHT;  // one or two column-pass threads per period, ACB_OHT outputs each
    L.LB = take(N * Tp);
    L.UB = take(N * Tp);
    // PART doubles as scratch for Sinv (R*R) and X (R*NG) while the column matrix is rebuilt
    const int scratch = R * R + R * NG + 8;
    L.PART = take(NP * Tp > scratch ? NP * Tp : scratch);
    L.VC = take(R * Tp);
    L.GIN = take(R * Tp);  // rho (2 z - v) of the coupling rows: written where v is updated, read by the column pass
    L.HG = take(NG * Tp);  // HG and VOUT are one (NG + R) x Tp output block of the column pass: keep them adjacent
    L.VOUT = take(R * Tp);
    L.THC = take(Tp);  // per-period restoration factors of the current / averaged candidate
    L.THA = take(Tp);
    L.ALPHA = take(Tp);
    L.BETA = take(Tp);
    L.PLIM = take(Tp);
    L.EBAR = take(Tp);
    L.MFT = take((NG + R + 2) * L.OP);  // inputs: NG group sums, R coupling inputs, alpha_t, beta_t
    L.CS = take(R * NG);
    L.SESS_A = take(S_max);
    L.SESS_B = take(S_max);
    L.SESS_E = take(S_max);
    L.SESS_MU = take(S_max);
    L.SESS_MU2 = take(S_max);
    L.SESS_Q = take(S_max);    // per-session quadratic weight cq (cost-scaled): objective term cq (Ebar_s - sum_window r)^2
    L.SESS_NF = take(S_max);   // slope estimate (number of free elements) of each session's energy equation, 0 = unknown
    L.ROWHI = take(nSlots);    // the row's upper bound inside its window when that is one constant, else -1
    L.SLOT = take(nSlots * 6);  // row, grp, prow, first, sess_first, sess_cnt
    L.PGOFF = take(NG + 1);
    L.NGRP = take(NG);
    L.KG = take(NG);
    L.LIM = take(R);
    L.SCALE = take(R);
    L.REDF = take(nwarps * ACB_NRED);
    L.REDD = take(nwarps * ACB_NRED * 2);  // doubles
    L.SCAL = take(32);
    L.SCALD = take(32);  // 16 doubles
    L.total = o;
    return L;
}

// float scalars
enum { SC_RHO = 0, SC_PLEVEL, SC_FLAG, SC_NEWRHO, SC_CS, SC_RP, SC_RD, SC_GAP, SC_VIOL, SC_NSUM, SC_NREST, SC_USEDAVG, SC_LBPOS, SC_STALL, SC_NRESCUE,
       SC_RHOSTART, SC_DZ, SC_KAP, SC_NDZ, SC_RATE_EST, SC_UBVAR, SC_NFEAS, SC_BESTVIOL, SC_VSTALL, SC_RATEM, SC_RATECNT, SC_NRATEOK };
// double scalars
enum { SD_DBEST = 0, SD_GAPRESTART, SD_BESTGAP, SD_PMAX };
// per-warp float reduction slots (max-type)
enum { RF_E1 = 0, RF_E2, RF_XMAX, RF_ZMAX, RF_YMAX, RF_NAN, RF_VIOLC, RF_VIOLA, RF_UMAXC, RF_UMAXA, RF_DZ };
// per-warp double reduction slots (sum-type)
enum { RD_PC = 0, RD_PA, RD_D, RD_UQC, RD_UQA, RD_PLC, RD_PLA };

// One launch of a (possibly multi-launch) solve.  A batch can be solved in phases: a launch leaves the iteration loop
// after iteration `it_stop` and parks the complete solver state of every unfinished instance (status ACB_RUNNING);
// a later launch with `resume` continues those instances exactly where they stopped (the straggler tail of a batch
// is then rescheduled longest-expected-first, see acb_solve.cu).
#define ACB_RUNNING (-1)
#define ACB_NSTATE 64  // floats of parked scalar state per instance: SCAL (32) + SCALD (16 doubles)
struct SolvePhase {
    int it_stop;       // park unfinished instances after this iteration (>= max_iter: never)
    int resume;        // 1: continue from the parked state
    const int* list;   // instance of block i (NULL: i); blocks >= *count exit
    const int* count;
    float* st_v1;      // parked state: [B][N][Tp], [B][R][Tp], [B][2 S_max] (multipliers, slope estimates), [B][ACB_NSTATE]
    float* st_vc;
    float* st_mu;
    float* st_scal;
    float* zprev;      // [B][N][Tp] schedule at the previous check (rate polish) or NULL
};

#ifdef ACB_TRACE
// development build only (tools/trace_solve.py): per-warp clock64() stamps of block 0 at the phase boundaries
#ifndef ACB_TR_IT0
#define ACB_TR_IT0 111
#endif
#define ACB_TR_NIT 16
#define ACB_TR_SLOTS 16
__device__ long long g_acb_trace[ACB_TR_NIT * 32 * ACB_TR_SLOTS];
__device__ __forceinline__ long long acb_clock() { long long c; asm volatile("mov.u64 %0, %%clock64;" : "=l"(c) :: "memory"); return c; }
#define ACB_TR(k) do { if (b == 0 && it >= ACB_TR_IT0 && it < ACB_TR_IT0 + ACB_TR_NIT && lane == 0) g_acb_trace[((it - ACB_TR_IT0) * 32 + warp) * ACB_TR_SLOTS + (k)] = acb_clock(); } while (0)
// (stamp that waits for a value: the float operand orders the clock read after the instructions producing it)
__device__ __forceinline__ long long acb_clock_after(float v) { long long c; asm volatile("mov.u64 %0, %%clock64;" : "=l"(c) : "f"(v) : "memory"); return c; }
#define ACB_TRV(k, v) do { if (b == 0 && it >= ACB_TR_IT0 && it < ACB_TR_IT0 + ACB_TR_NIT) { long long c_ = acb_clock_after(v); if (lane == 0) g_acb_trace[((it - ACB_TR_IT0) * 32 + warp) * ACB_TR_SLOTS + (k)] = c_; } } while (0)
#else
#define ACB_TR(k) do { } while (0)
#define ACB_TRV(k, v) do { } while (0)
#endif

// FAST: the caller declared every minimum rate 0 (acb_batch.lb_zero) and rows hold one session.  The lower-bound
// array is then not needed and its shared memory holds v instead of registers: the hot loop keeps no per-element state
// in registers (no spills under the 80-register cap, loop constants stay resident).
template <int Q, int TPW, bool MULTI, bool FAST>
__global__ void __launch_bounds__(TPW == 2 ? 1024 : (FAST ? ACB_FAST_THREADS : 768), 1) acb_solve_kernel(const SiteDev S, const acb_batch B, const acb_options opt, const SmemLayout L, const SolvePhase P) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nthreads = blockDim.x, nwarps = nthreads >> 5;
    constexpr int Tp = 32 * Q;  // the host pads every batch to an instantiated horizon
    // paired fp32 ops (FFMA2 / FADD2 / FMUL2: each half rounds as the scalar op) in the column pass and the hot row pass.
    // Only where v lives in shared memory with three rows per warp: there the aligned register pairs fit; in the other
    // variants they raise the spills (v in registers, or 64 registers per thread)
    constexpr bool PAIR = FAST && TPW == 3;
    const int N = S.N, R = S.R, NG = S.NG, NP = S.NP;
    float* LB = sm + L.LB; float* UB = sm + L.UB; float* PART = sm + L.PART; float* VC = sm + L.VC;
    float* VOUT = sm + L.VOUT; float* GIN = sm + L.GIN; float* HG = sm + L.HG; float* THC = sm + L.THC; float* THA = sm + L.THA; float* ALPHA = sm + L.ALPHA; float* BETA = sm + L.BETA;
    float* PLIM = sm + L.PLIM; float* EBAR = sm + L.EBAR; float* MFT = sm + L.MFT; float* CS = sm + L.CS;
    float* SINV = PART; float* XS = PART + R * R;
    int* SESS_A = (int*)(sm + L.SESS_A); int* SESS_B = (int*)(sm + L.SESS_B);
    float* SESS_E = sm + L.SESS_E; float* SESS_MU = sm + L.SESS_MU; float* SESS_MU2 = sm + L.SESS_MU2;
    float* SESS_NF = sm + L.SESS_NF; float* ROWHI = sm + L.ROWHI; float* SESS_Q = sm + L.SESS_Q;
    int* SLOT = (int*)(sm + L.SLOT); int* PGOFF = (int*)(sm + L.PGOFF);
    float* NGRP = sm + L.NGRP; float* KG = sm + L.KG; float* LIM = sm + L.LIM; float* SCALE = sm + L.SCALE;
    float* REDF = sm + L.REDF; double* REDD = (double*)(sm + L.REDD); float* SCAL = sm + L.SCAL;
    double* SCALD = (double*)(sm + L.SCALD);
    const int OP = L.OP, NIN = NG + R;

    if (P.count && (int)blockIdx.x >= *P.count) return;
    const int b = P.list ? P.list[blockIdx.x] : blockIdx.x;
    const int Tb = B.T[b];
    const int nS = B.n_sessions[b];
    const int nDisc = S.nDisc, nLin = S.nLin;
    const int rPL = 2 * nDisc + nLin, rU = rPL + S.has_pl;
    const int nCT = nDisc + nLin + S.has_pl + S.has_u;  // coupling tasks
    const float linLo = S.lin_two_sided ? -1.f : -3.0e38f;  // lower end of a linear row as a multiple of its limit
    // coupling rows run on the warps that own no EVSE rows (if any): the disc / linear / peak-limit tasks are cut into
    // 32-period chunks and dealt round-robin to those warps; the aggregate-power row, which carries the peak-level
    // root find over the whole horizon, gets the last warp (to itself when two or more warps are free)
    const int nCT1 = nDisc + nLin + S.has_pl;
    int cwIdx = -1, nCW = 1;
    bool doAgg = false;
    {
        const int nFree = nwarps - S.nRowWarps;
        if (nFree <= 0) { cwIdx = warp; nCW = nwarps; }
        else if (S.has_u && nFree >= 2) { nCW = nFree - 1; if (warp >= S.nRowWarps && warp < nwarps - 1) cwIdx = warp - S.nRowWarps; }
        else { nCW = nFree; if (warp >= S.nRowWarps) cwIdx = warp - S.nRowWarps; }
        doAgg = S.has_u && warp == nwarps - 1;
    }
    // balance: a coupling warp carries about 16 chunk items; what exceeds that rides on the row warps (blocks with few
    // spare warps: the FAST variant runs 640 threads for 96 registers per thread)
    const int rowShare = (nwarps > S.nRowWarps) ? max(0, (nCT1 * Q - 16 * nCW + S.nRowWarps - 1) / S.nRowWarps) : 0;
    float* VSUM = B.work ? B.work + (size_t)b * (N + R) * Tp : nullptr;  // running sum of v (rows, then coupling rows)
    const bool useAvg = opt.restart && VSUM != nullptr;

    float* Vs = LB;  // FAST: v lives where the lower bounds would be
    // bounds of element (row, t)
    auto lbv = [&](int row, int t) -> float { if constexpr (FAST) return 0.f; else return LB[row * Tp + t]; };
    auto ubv = [&](int row, int t) -> float { return UB[row * Tp + t]; };
    // the lane's Q elements of a row (t = lane + 32 q)
    auto load_bounds = [&](int row, float (&lb)[Q], float (&ub)[Q]) {
        const float* lbp = LB + row * Tp + lane;
        const float* ubp = UB + row * Tp + lane;
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            if constexpr (FAST) lb[q] = 0.f; else lb[q] = lbp[32 * q];
            ub[q] = ubp[32 * q];
        }
    };

    // ------------------------------------------------------------------ prologue
    for (int i = tid; i < 2 * N * Tp; i += nthreads) LB[i] = 0.f;  // LB (FAST: v) and UB are contiguous
    // warm start of a closed-loop replay: the previous step's state is read `warm_shift` columns ahead (column t of this
    // problem was column t + 1 of the previous one), and instances whose site was idle before start cold (warm_had = 0:
    // no warm array is read, the same start as a solve without warm arrays)
    const int wsh = B.warm_shift;
    const bool hadW = !B.warm_had || B.warm_had[b] != 0;
    const float* warm_v1 = hadW ? B.warm_v1 : nullptr;
    for (int i = tid; i < R * Tp; i += nthreads) {
        const int t = i % Tp;
        VC[i] = (B.warm_vc && hadW && t + wsh < Tp) ? B.warm_vc[(size_t)b * R * Tp + i + wsh] : 0.f;
        VOUT[i] = 0.f;
    }
    for (int i = tid; i < R * NG; i += nthreads) CS[i] = S.C[i];
    for (int i = tid; i < R; i += nthreads) { LIM[i] = S.lim[i]; SCALE[i] = S.row_scale[i]; }
    for (int i = tid; i <= NG; i += nthreads) PGOFF[i] = S.pg_off[i];
    for (int i = tid; i < NG; i += nthreads) { NGRP[i] = S.ngrp[i]; KG[i] = S.kg[i]; }
    for (int i = tid; i < S.nSlots; i += nthreads) {
        SLOT[i * 6 + 0] = S.slot_row[i]; SLOT[i * 6 + 1] = S.slot_grp[i];
        SLOT[i * 6 + 2] = S.slot_prow[i]; SLOT[i * 6 + 3] = S.slot_first[i];
        SLOT[i * 6 + 4] = 0; SLOT[i * 6 + 5] = 0;
    }
    for (int i = tid; i < B.S_max; i += nthreads) {
        bool ok = i < nS;
        size_t k = (size_t)b * B.S_max + i;
        SESS_A[i] = ok ? B.sess_start[k] : 0;
        SESS_B[i] = ok ? B.sess_start[k] + B.sess_len[k] : 0;
        SESS_E[i] = ok ? B.sess_energy[k] : 0.f;
        SESS_MU[i] = (ok && B.warm_mu && hadW) ? B.warm_mu[k] : 0.f;
        SESS_MU2[i] = 0.f;
        SESS_NF[i] = 0.f;
        SESS_Q[i] = (ok && B.sess_quad) ? B.sess_quad[k] : 0.f;  // (scaled by the cost scale below)
    }
    if (tid == 0) { SCAL[SC_FLAG] = 0.f; SCAL[SC_LBPOS] = 0.f; SCAL[SC_UBVAR] = 0.f; }
    for (int t = tid; t < Tp; t += nthreads) {
        bool ok = t < Tb;
        ALPHA[t] = ok ? B.alpha[(size_t)b * Tp + t] : 0.f;
        BETA[t] = ok ? B.beta[(size_t)b * Tp + t] : 0.f;
        EBAR[t] = (ok && B.ext) ? B.ext[(size_t)b * Tp + t] : 0.f;
        PLIM[t] = (ok && B.peak_limit && S.has_pl) ? B.peak_limit[(size_t)b * Tp + t] / S.row_scale[rPL] : 3.0e38f;
    }
    __syncthreads();
    // sessions -> bounds (charging_rate_bounds incl. the ub<lb patch) and per-slot session lists.
    // Sessions arrive sorted by EVSE row (host packer), so each row's sessions are contiguous.
    for (int s = warp; s < nS; s += nwarps) {
        size_t k = (size_t)b * B.S_max + s;
        int row = B.sess_row[k], a = SESS_A[s], len = SESS_B[s] - a, off = B.sess_rate_off[k];
        for (int j = lane; j < len; j += 32) {
            const int ri = off >= 0 ? off + j : -(off + 1);  // off < 0: one (min, max) pair for the whole session
            float lo = B.min_rates[ri], hi = B.max_rates[ri];
            if (a + j < Tp) {
                if constexpr (FAST) { if (lo != 0.f) SCAL[SC_LBPOS] = 1.f; }  // the caller's lb_zero promise is broken: flagged below
                else LB[row * Tp + a + j] = lo;
                UB[row * Tp + a + j] = fmaxf(hi, lo);
            }
        }
    }
    if (tid < S.nSlots) {
        int row = SLOT[tid * 6 + 0], first = -1, cnt = 0;
        if (row >= 0)
            for (int s = 0; s < nS; ++s)
                if (B.sess_row[(size_t)b * B.S_max + s] == row) { if (first < 0) first = s; ++cnt; }
        SLOT[tid * 6 + 4] = first < 0 ? 0 : first;
        SLOT[tid * 6 + 5] = cnt;
    }
    for (int t = tid; t < Tp; t += nthreads) { THC[t] = 1.f; THA[t] = 1.f; }
    __syncthreads();
    if constexpr (!FAST) {
        bool pos = false;
        for (int i = tid; i < N * Tp; i += nthreads) pos |= (LB[i] != 0.f);
        if (pos) SCAL[SC_LBPOS] = 1.f;  // benign race: every writer stores the same value
    }
    // rows whose upper bound is one constant inside the window (the usual case): the hot row pass clips with a
    // saturating multiply on the FMA pipe instead of min/max pairs on the half-rate ALU pipe
    if (warp < S.nRowWarps) {
        for (int k = 0; k < S.TPW; ++k) {
            const int sl = warp * S.TPW + k, row = SLOT[sl * 6];
            float m = 0.f;
            if (row >= 0) for (int t = lane; t < Tp; t += 32) m = fmaxf(m, UB[row * Tp + t]);
            m = warp_max(m);
            bool uni = true;
            if (row >= 0) for (int t = lane; t < Tp; t += 32) { const float u = UB[row * Tp + t]; uni &= (u == 0.f || u == m); }
            uni = __all_sync(0xffffffffu, uni);
            if (lane == 0) { ROWHI[sl] = uni ? m : -1.f; if (!uni) SCAL[SC_UBVAR] = 1.f; }
        }
    }
    // row-level infeasibility: a session whose window cannot hold its energy equality, or whose
    // minimum rates already exceed its energy cap (the reference would get INFEASIBLE from ECOS)
    for (int s = warp; s < nS; s += nwarps) {
        int row = B.sess_row[(size_t)b * B.S_max + s];
        float slo = 0.f, shi = 0.f;
        for (int t = SESS_A[s] + lane; t < min(SESS_B[s], Tp); t += 32) { slo += lbv(row, t); shi += ubv(row, t); }
        slo = warp_sum(slo); shi = warp_sum(shi);
        const float Eb = SESS_E[s], tol = 1e-5f * (fabsf(Eb) + 1.f);
        if (lane == 0 && (slo > Eb + tol || (opt.equality && shi < Eb - tol))) SCAL[SC_FLAG] = 1.f;
    }
    __syncthreads();
    const bool badHint = FAST && SCAL[SC_LBPOS] != 0.f;  // lb_zero was declared but a minimum rate is positive
    if (SCAL[SC_FLAG] != 0.f || badHint) {
        for (int i = tid; i < N * Tp; i += nthreads) B.rates[(size_t)b * N * Tp + i] = 0.f;
        if (tid == 0) {
            B.status[b] = badHint ? ACB_INVALID : ACB_INFEASIBLE;
            B.iters[b] = 0;
            for (int k = 0; k < ACB_NSTATS; ++k) B.stats[(size_t)b * ACB_NSTATS + k] = 0.f;
        }
        return;
    }
    // cost scale = 1 / max |alpha_t + k_g beta_t|
    {
        float m = 0.f;
        for (int i = tid; i < NG * Tp; i += nthreads) {
            int g = i / Tp, t = i - g * Tp;
            m = fmaxf(m, fabsf(ALPHA[t] + KG[g] * BETA[t]));
        }
        m = warp_max(m);
        if (lane == 0) REDF[warp * ACB_NRED] = m;
    }
    __syncthreads();
    if (tid == 0) {
        float m = 0.f;
        for (int w = 0; w < nwarps; ++w) m = fmaxf(m, REDF[w * ACB_NRED]);
        SCAL[SC_CS] = (m > 1e-20f) ? 1.0f / m : 1.0f;
        // cold start: rho0, raised to the curvature of the aggregate quadratic seen through the scaled aggregate row
        // (see acb_solve_general.cu: k_setup)
        const float su0 = S.has_u ? S.row_scale[rU] : 0.f;
        SCAL[SC_RHO] = (B.warm_scal && hadW && B.warm_scal[b * 2] > 0.f) ? B.warm_scal[b * 2]
                                                                           : fmaxf(opt.rho0, opt.rho_curv * B.gamma[b] * SCAL[SC_CS] * su0 * su0);
        SCAL[SC_PLEVEL] = (B.warm_scal && hadW) ? fmaxf(B.warm_scal[b * 2 + 1], B.peak_p0[b]) : B.peak_p0[b];
        SCAL[SC_FLAG] = 0.f;
        SCAL[SC_NSUM] = 0.f;
        SCAL[SC_NREST] = 0.f;
        SCAL[SC_USEDAVG] = 0.f;
        SCAL[SC_RP] = SCAL[SC_RD] = SCAL[SC_GAP] = SCAL[SC_VIOL] = 0.f;
        SCALD[SD_DBEST] = -1.0e300;
        SCALD[SD_GAPRESTART] = 1.0e300;
        SCALD[SD_BESTGAP] = 1.0e300;
        SCAL[SC_STALL] = 0.f;
        SCAL[SC_NRESCUE] = 0.f;
        SCAL[SC_RHOSTART] = SCAL[SC_RHO];
        SCAL[SC_DZ] = 0.f; SCAL[SC_KAP] = 1.f; SCAL[SC_RATEM] = 1.f; SCAL[SC_RATECNT] = 0.f; SCAL[SC_NRATEOK] = 0.f; SCAL[SC_NDZ] = 0.f; SCAL[SC_RATE_EST] = -1.f;
        SCAL[SC_NFEAS] = 0.f; SCAL[SC_BESTVIOL] = 3.0e38f; SCAL[SC_VSTALL] = 0.f;
    }
    __syncthreads();
    const float cs = SCAL[SC_CS];
    for (int t = tid; t < Tp; t += nthreads) { ALPHA[t] *= cs; BETA[t] *= cs; }
    bool hasQuad = false;  // some session carries a quadratic shortfall term (non_completion_penalty, norm 2)
    if (B.sess_quad) {
        for (int i = 0; i < nS; ++i) hasQuad |= SESS_Q[i] > 0.f;
        __syncthreads();  // everybody has read the unscaled weights
        for (int i = tid; i < B.S_max; i += nthreads) SESS_Q[i] *= cs;
    }
    const float qd = B.qd[b] * cs, Gamma = B.gamma[b] * cs, pk_w = B.peak_w[b] * cs, pk_p0 = B.peak_p0[b];
    const float alpha = opt.alpha, kappa = opt.kappa;
    // Feasibility restoration of a candidate: r_t <- theta_t r_t with theta_t = 1 / max(1, worst current/limit at t).
    // With lb = 0, no quadratic term and inequality energy rows the scaled schedule satisfies box, energy caps and
    // every coupling row exactly, and its objective follows from the per-group column sums.
    // (a quadratic weight below 1e-9 of the largest cost coefficient -- the reference's 1e-12 tie-breaker -- changes the
    // objective of the scaled candidate by less than float32 resolves and does not block the restoration)
    const bool canRestore = (SCAL[SC_LBPOS] == 0.f) && (qd <= 1e-9f) && !opt.equality && !hasQuad;
    // rate polish (strictly convex objective, unique optimum): besides the certified gap the stop also asks that the
    // schedule has stopped moving -- estimated distance to the fixed point <= rate_tol amperes (see the check path)
    float* ZPREV = P.zprev ? P.zprev + (size_t)b * N * Tp : nullptr;
    const bool polish = opt.rate_tol > 0.f && qd >= opt.polish_min_qd && ZPREV != nullptr;
    const float su = S.has_u ? S.row_scale[rU] : 1.f;
    // resume of a parked instance: the scalar state replaces the cold / warm-start values set above
    int it0 = 0;
    if (P.resume) {
        __syncthreads();
        const float* stp = P.st_scal + (size_t)b * ACB_NSTATE;
        if (tid < 32) SCAL[tid] = stp[tid];
        else if (tid < 64) sm[L.SCALD + tid - 32] = stp[tid];
        __syncthreads();
        it0 = B.iters[b];
    }
    float rho = SCAL[SC_RHO];
    const float rho_start = SCAL[SC_RHOSTART];  // what a warm start of the next solve inherits (a stagnation rescue is not carried over)
    float rho1 = kappa * rho, dd = 2.f * qd + rho1, inv_d = 1.f / dd;

    // Infeasibility certificate: the Lagrangian bound D is a lower bound of the optimal value over the feasible set, and
    // no feasible point can cost more than the maximum of the objective over the box.  D > that maximum => infeasible
    // (the duals of an infeasible instance diverge, so D gets there quickly).  PMAX = that maximum, in scaled units.
    {
        __syncthreads();  // scaled ALPHA / BETA
        double pm = 0.0;
        float cmax = 0.f;
        for (int i = tid; i < S.nSlots * Tp; i += nthreads) {
            const int s = i / Tp, t = i - s * Tp, row = SLOT[s * 6];
            if (row < 0) continue;
            const float c = ALPHA[t] + KG[SLOT[s * 6 + 1]] * BETA[t], lo = lbv(row, t), hi = ubv(row, t);
            pm += (double)fmaxf(c * lo, c * hi) + (double)qd * (double)fmaxf(lo * lo, hi * hi);
        }
        if (S.has_u && (Gamma > 0.f || pk_w > 0.f)) {
            for (int t = tid; t < Tb; t += nthreads) {
                float umax = 0.f, umin = 0.f;
                for (int s = 0; s < S.nSlots; ++s) {
                    const int row = SLOT[s * 6];
                    if (row < 0) continue;
                    const float k = KG[SLOT[s * 6 + 1]];
                    umax += k * ubv(row, t); umin += k * lbv(row, t);
                }
                const float e = EBAR[t];
                pm += (double)Gamma * (double)fmaxf((umax + e) * (umax + e), (umin + e) * (umin + e));
                cmax = fmaxf(cmax, umax);
            }
        }
        pm = warp_sum(pm); cmax = warp_max(cmax);
        if (lane == 0) { REDD[warp * ACB_NRED] = pm; REDF[warp * ACB_NRED] = cmax; }
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            float um = 0.f;
            for (int w = 0; w < nwarps; ++w) { tot += REDD[w * ACB_NRED]; um = fmaxf(um, REDF[w * ACB_NRED]); }
            if (hasQuad)  // the planned energy stays in [0, Eb] under the cap: (Eb - E)^2 <= Eb^2
                for (int i = 0; i < nS; ++i) tot += (double)SESS_Q[i] * (double)SESS_E[i] * (double)SESS_E[i];
            SCALD[SD_PMAX] = tot + (double)pk_w * (double)fmaxf(um, pk_p0);
        }
        __syncthreads();
    }

    // per-lane state: v for this warp's EVSE rows
    float v1[FAST ? 1 : TPW][FAST ? 1 : Q];
    auto vget = [&](int k, int q, int row) -> float {
        if constexpr (FAST) return Vs[row * Tp + lane + 32 * q]; else return v1[k][q];
    };
    auto vset = [&](int k, int q, int row, float val) {
        if constexpr (FAST) Vs[row * Tp + lane + 32 * q] = val; else v1[k][q] = val;
    };
    const bool rowWarp = warp < S.nRowWarps;
#pragma unroll
    for (int k = 0; k < TPW; ++k) {
        int row = rowWarp ? SLOT[(warp * TPW + k) * 6] : -1;
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            int t = lane + 32 * q;
            float v = 0.f;
            if (row >= 0) {
                if (P.resume) v = P.st_v1[((size_t)b * N + row) * Tp + t];
                else if (warm_v1) v = (t + wsh < Tp) ? warm_v1[((size_t)b * N + row) * Tp + t + wsh] : 0.f;
                else v = clampf(0.f, lbv(row, t), ubv(row, t));
                vset(k, q, row, v);
            }
        }
    }

    // ---- helpers --------------------------------------------------------------
    // multiplier of the session covering period t of a row (rows with a single session use
    // its multiplier everywhere: outside the window lb = ub = 0)
    auto mu_at = [&](const float* MU, int sfirst, int scnt, int t) -> float {
        float m = 0.f;
        for (int s = sfirst; s < sfirst + scnt; ++s)
            if (t >= SESS_A[s] && t < SESS_B[s]) m = MU[s];
        return m;
    };
#define MU_ELEM(MU, sf, scn, mu0, t) (MULTI ? mu_at(MU, sf, scn, t) : (mu0))
    // multiplier mu with sum_{t in [a,e)} clip(vv_t - mu, lb_t, ub_t) = Eb (or <= Eb with mu >= 0):
    // safeguarded Newton on a piecewise-linear monotone function, warm-started at mu
    // `single`: the row has one session, so outside its window lb = ub = 0 and no mask is needed.
    // `max_evals` = 1 gives one Newton step from the warm start without re-evaluation (used on
    // non-check iterations: the projection is then inexact by an active-set change at most).
    // `cq` > 0 (inequality rows only): the row also carries the objective term cq (Eb - E)^2 (non_completion_penalty,
    // norm 2), so this is a prox rather than a projection: the multiplier may go negative, mu = kq (E(mu) - Eb) with
    // kq = 2 cq / rho1 while the cap is inactive; in residual form E(mu) - Eb - min(mu, 0) / kq = 0, still monotone.
    auto newton_mu = [&](const float (&vv)[Q], const float (&lb)[Q], const float (&ub)[Q], int a, int e, float Eb, float mu,
                         bool single, int max_evals, float cq = 0.f) -> float {
        const float tol = 2e-6f * (Eb + 1.f);
        const bool soft = cq > 0.f && !opt.equality;
        const float ikq = soft ? rho1 / (2.f * cq) : 0.f;
        const bool freeMu = opt.equality || soft;
        // inequality rows: lo = -1 marks "mu = 0 not evaluated yet" (mu itself stays >= 0)
        float lo = freeMu ? -3.0e38f : -1.f, hi = 3.0e38f;
        if (!freeMu) mu = fmaxf(mu, 0.f);
        for (int step = 0; step < 16; ++step) {
            float E = 0.f;
            int nf = 0;
            if (single) {
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    float w = vv[q] - mu;
                    E += clampf(w, lb[q], ub[q]);
                    nf += (w > lb[q] && w < ub[q]) ? 1 : 0;
                }
            } else {
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    int t = lane + 32 * q;
                    if (t >= a && t < e) {
                        float w = vv[q] - mu;
                        E += clampf(w, lb[q], ub[q]);
                        nf += (w > lb[q] && w < ub[q]) ? 1 : 0;
                    }
                }
            }
            E = warp_sum(E);
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
            if (step + 1 >= max_evals && slope > 0.f) break;
        }
        return mu;
    };
    // Best energy-row multiplier for the dual bound: the maximiser over lam (>= 0 for inequality rows) of
    //   -lam Eb + sum_{t in [a,e)} min_{lb <= r <= ub} (aa_t + lam) r + qd r^2,
    // a concave function of lam whose slope is sum_t r_t(lam) - Eb: bracket around lam0, then bisect.  Any lam
    // gives a valid bound; the iterate's own multiplier drifts along degenerate dual faces (a site sitting at its
    // previous peak), this one does not.
    auto dual_lambda = [&](const float (&aa)[Q], const float (&lb)[Q], const float (&ub)[Q], int a, int e, float Eb, float lam0,
                           bool single) -> float {
        auto total = [&](float lam) -> float {
            float Ssum = 0.f;
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                const int t = lane + 32 * q;
                if (single || (t >= a && t < e)) {
                    const float rt = aa[q] + lam;
                    Ssum += (qd > 0.f) ? clampf(-rt / (2.f * qd), lb[q], ub[q]) : (rt < 0.f ? ub[q] : lb[q]);
                }
            }
            return warp_sum(Ssum);
        };
        const bool ineq = !opt.equality;
        const float l0 = ineq ? fmaxf(lam0, 0.f) : lam0;
        float step = 1e-3f * (1.f + fabsf(l0)), lo, hi;
        if (total(l0) > Eb) {
            lo = l0; hi = l0 + step;
            for (int i = 0; i < 14 && total(hi) > Eb; ++i) { lo = hi; step *= 8.f; hi = lo + step; }
        } else {
            if (ineq && l0 <= 0.f) return 0.f;
            hi = l0; lo = l0 - step;
            for (int i = 0; i < 14; ++i) {
                if (ineq && lo <= 0.f) {
                    lo = 0.f;
                    if (total(0.f) <= Eb) return 0.f;
                    break;
                }
                if (total(lo) > Eb) break;
                hi = lo; step *= 8.f; lo = hi - step;
            }
        }
        for (int i = 0; i < 20; ++i) {
            const float mid = 0.5f * (lo + hi);
            if (total(mid) > Eb) lo = mid; else hi = mid;
        }
        return hi;
    };
    // (NG+R)^2 matrix of the column pass for the current rho (see DESIGN.md):
    //   Sinv = U diag(1/(d/rho + lam)) U',  X = Sinv C,
    //   hg = -C'X sa + (d/rho) X' g,   v = X sa + (I - (d/rho) Sinv) g
    // (PART is scratch here: callers rewrite it afterwards)
    auto build_matrix = [&]() {
        const float dr = dd / rho;
        for (int i = tid; i < R * R; i += nthreads) {
            int r = i / R, c = i - r * R;
            float acc = 0.f;
            for (int e = 0; e < R; ++e) acc += __ldg(S.U + r * R + e) * __ldg(S.U + c * R + e) / (dr + __ldg(S.lam + e));
            SINV[i] = acc;
        }
        __syncthreads();
        for (int i = tid; i < R * NG; i += nthreads) {
            int r = i / NG, g = i - r * NG;
            float acc = 0.f;
            for (int c = 0; c < R; ++c) acc += SINV[r * R + c] * CS[c * NG + g];
            XS[i] = acc;
        }
        __syncthreads();
        // base element M(c, o) of the (NG+R) x (NG+R) column matrix
        auto melem = [&](int c, int o) -> float {
            float m = 0.f;
            if (o < NG && c < NG) {
                for (int r = 0; r < R; ++r) m -= CS[r * NG + o] * XS[r * NG + c];
            } else if (o < NG) {
                m = dr * XS[(c - NG) * NG + o];
            } else if (c < NG) {
                m = XS[(o - NG) * NG + c];
            } else {
                int r = o - NG, j = c - NG;
                m = (r == j ? 1.f : 0.f) - dr * SINV[r * R + j];
            }
            return m;
        };
        // folded form used by the column pass: inputs are the RAW group sums of q, the coupling inputs GIN and the two
        // cost coefficients of the period; outputs are HG = Khat'h - c (rows < NG) and Khat x (rows >= NG, the 1/rho
        // included).  With in_g = rho1 sum_g - n_g (alpha + k_g beta):
        //   row g       : rho1 M(g, o)
        //   row NG + r  : M(NG + r, o)
        //   row alpha   : -sum_g n_g M(g, o) - [o < NG]
        //   row beta    : -sum_g n_g k_g M(g, o) - [o < NG] k_o
        for (int i = tid; i < (NIN + 2) * OP; i += nthreads) {
            int c = i / OP, o = i - c * OP;
            float m = 0.f;
            if (o < NIN) {
                const float so = (o < NG) ? 1.f : 1.f / rho;
                if (c < NG) m = rho1 * melem(c, o);
                else if (c < NIN) m = melem(c, o);
                else {
                    for (int g = 0; g < NG; ++g) m -= NGRP[g] * (c == NIN ? 1.f : KG[g]) * melem(g, o);
                    if (o < NG) m -= (c == NIN) ? 1.f : KG[o];
                }
                m *= so;
            }
            MFT[i] = m;
        }
        __syncthreads();
    };
    // unconstrained minimiser of the aggregate-power prox (kW) given the stored v of that row
    float aggA = 0.f, aggB = 0.f;  // a = aggA v - aggB ext_t; follow rho
    auto set_agg = [&]() {
        const float rp = rho / (su * su), den = 1.f / (rp + 2.f * Gamma);
        aggA = rp * su * den;
        aggB = 2.f * Gamma * den;
    };
    set_agg();
    auto agg_a = [&](float v, int t) -> float { return aggA * v - aggB * EBAR[t]; };
    // peak-epigraph level for the aggregate-power row stored in VC (called by one warp):
    // minimise pk_w*max(p,p0) + cur/2 sum (a_t - p)_+^2 over p
    auto peak_level = [&](float guess) -> float {
        const int r = rU;
        const float rp = rho / (su * su), cur = rp + 2.f * Gamma;
        float av[Q];
        float amax = -3.0e38f;
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            int t = lane + 32 * q;
            av[q] = (t < Tb) ? agg_a(VC[r * Tp + t], t) : -3.0e38f;
            amax = fmaxf(amax, av[q]);
        }
        amax = warp_max(amax);
        float pl = fmaxf(amax, pk_p0);
        if (pk_w > 0.f && amax > pk_p0) {
            float F0 = 0.f;
#pragma unroll
            for (int q = 0; q < Q; ++q) F0 += fmaxf(av[q] - pk_p0, 0.f);
            F0 = warp_sum(F0) * cur;
            if (F0 <= pk_w) pl = pk_p0;
            else {
                float p = fminf(fmaxf(guess, pk_p0), amax), lo = pk_p0, hi = amax;
                for (int step = 0; step < 24; ++step) {
                    float F = 0.f;
                    int na = 0;
#pragma unroll
                    for (int q = 0; q < Q; ++q)
                        if (av[q] > p) { F += av[q] - p; ++na; }
                    F = warp_sum(F) * cur - pk_w;
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
        return pl;
    };
    // write partial sums of q = 2z - v for this warp's rows (z from the stored v and multipliers)
    auto write_part_q = [&]() {
        if (!rowWarp) return;
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            const int* sl = SLOT + (warp * TPW + k) * 6;
            int row = sl[0];
            if (row < 0) continue;
            int prow = sl[2], first = sl[3], sf = sl[4], scn = sl[5];
            const float mu0 = scn ? SESS_MU[sf] : 0.f;
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                int t = lane + 32 * q;
                if (t >= Tp) continue;
                const float vq = vget(k, q, row);
                float z = clampf(vq - MU_ELEM(SESS_MU, sf, scn, mu0, t), lbv(row, t), ubv(row, t));
                float val = 2.f * z - vq;
                if (first) PART[prow * Tp + t] = val; else PART[prow * Tp + t] += val;
            }
        }
    };
    // GIN <- rho (2 z(v) - v) for every coupling row from the stored v (start, restart, penalty change)
    auto write_gin = [&]() {
        const float pl = SCAL[SC_PLEVEL];
        for (int t = tid; t < Tp; t += nthreads) {
            int r = 0;
            for (int j = 0; j < nDisc; ++j, r += 2) {
                float a = VC[r * Tp + t], bb = VC[(r + 1) * Tp + t], za, zb;
                proj_disc(a, bb, LIM[r], za, zb);
                GIN[r * Tp + t] = rho * (2.f * za - a); GIN[(r + 1) * Tp + t] = rho * (2.f * zb - bb);
            }
            for (int j = 0; j < nLin; ++j, ++r) {
                float v = VC[r * Tp + t], z = clampf(v, (linLo < -1.0e30f) ? linLo : linLo * LIM[r], LIM[r]);
                GIN[r * Tp + t] = rho * (2.f * z - v);
            }
            if (S.has_pl) { float v = VC[r * Tp + t], z = fminf(v, PLIM[t]); GIN[r * Tp + t] = rho * (2.f * z - v); ++r; }
            if (S.has_u) {
                float v = VC[r * Tp + t], a = agg_a(v, t);
                float z = ((pk_w > 0.f) ? fminf(a, pl) : a) / su;
                GIN[r * Tp + t] = rho * (2.f * z - v);
            }
        }
    };
    // column evaluation of a candidate whose group partial sums are in PART: relative coupling
    // violation, max and quadratic part of the aggregate power; optionally HG <- C' yc (yc in VOUT)
    // a row whose limit is 0 (a de-rated line, a curtailment period) has no relative violation: any current above 1e-5 A
    // counts.  With restoration the whole period is scaled to (numerically) zero; without it the violation is the
    // current in amperes, measured against viol_tol like the relative ones.
    auto zero_limit = [&](float amps) -> float { return canRestore ? (amps > 1e-5f ? 1.0e30f : 0.f) : 1.f + amps; };
    // Two adjacent lanes share a period: the group sums, the coupling rows and the C'y outputs are dealt to them by parity
    // (the pass is a chain of dependent shared-memory loads; one thread per period left 9 of the block's warps to do it).
    auto eval_columns = [&](bool with_hy, float* TH, float& viol, float& umax, double& uq, double& plin) {
        viol = -1.f; umax = -3.0e38f; uq = 0.0; plin = 0.0;
        const int h = tid & 1, half = nthreads >> 1;
        // a row with limit L amperes may exceed it by min(viol_tol L, viol_abs): the relative excess is scaled up where
        // viol_abs (1e-3 A, the bar of the reference's own tests) is the tighter of the two
        auto vfac = [&](float lim_amps) -> float { return (opt.viol_abs > 0.f) ? fmaxf(1.f, lim_amps * opt.viol_tol / opt.viol_abs) : 1.f; };
        for (int base = 0; base < Tp; base += half) {
            const int t = base + (tid >> 1);
            if (t >= Tp) continue;  // (whole warps: Tp and half are multiples of 16)
            float pcol = 0.f;
            for (int g = h; g < NG; g += 2) {
                float sz = 0.f;
                for (int p = PGOFF[g]; p < PGOFF[g + 1]; ++p) sz += PART[p * Tp + t];
                HG[g * Tp + t] = sz;
                pcol += (ALPHA[t] + KG[g] * BETA[t]) * sz;  // linear cost of the period (same coefficient within a group)
            }
            __syncwarp();  // the partner's group sums
            float worst = 0.f;  // worst current / limit of the period
            float vmax = -1.f;  // worst excess in units of the row's tolerance: relative, tightened to viol_abs amperes on large limits
            for (int j = h; j < nDisc; j += 2) {
                const int r = 2 * j;
                float ka = 0.f, kb = 0.f;
                for (int g = 0; g < NG; ++g) { float sz = HG[g * Tp + t]; ka += CS[r * NG + g] * sz; kb += CS[(r + 1) * NG + g] * sz; }
                const float cur = sqrtf(ka * ka + kb * kb);
                float ratio;
                if (LIM[r] > 0.f) { ratio = cur / LIM[r]; vmax = fmaxf(vmax, (ratio - 1.f) * vfac(LIM[r] * SCALE[r])); }
                else { ratio = zero_limit(cur * SCALE[r]); vmax = fmaxf(vmax, ratio - 1.f); }
                worst = fmaxf(worst, ratio);
            }
            for (int j = h; j < nLin + S.has_pl; j += 2) {
                const int r = 2 * nDisc + j;
                float ka = 0.f;
                for (int g = 0; g < NG; ++g) ka += CS[r * NG + g] * HG[g * Tp + t];
                float cap = (j == nLin) ? PLIM[t] : LIM[r];
                if (j < nLin && S.lin_two_sided) ka = fabsf(ka);
                if (cap > 0.f && cap < 1.0e30f) { const float ratio = ka / cap; worst = fmaxf(worst, ratio); vmax = fmaxf(vmax, (ratio - 1.f) * vfac(cap * SCALE[r])); }
                else if (cap <= 0.f) { const float ratio = zero_limit(fmaxf(ka, 0.f) * SCALE[r]); worst = fmaxf(worst, ratio); vmax = fmaxf(vmax, ratio - 1.f); }
            }
            worst = fmaxf(worst, __shfl_xor_sync(0xffffffffu, worst, 1));
            vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, 1));
            const float th = (canRestore && worst > 1.f) ? 1.f / (worst * (1.f + 2e-7f)) : 1.f;
            if (h == 0) TH[t] = th;
            viol = fmaxf(viol, th < 1.f ? worst * th - 1.f : vmax);
            plin += (double)(th * pcol);  // (each lane its own groups: the block sum adds them)
            if (S.has_u && t < Tb && h == 1) {
                float ka = 0.f;
                for (int g = 0; g < NG; ++g) ka += CS[rU * NG + g] * HG[g * Tp + t];
                float u = ka * su * th;
                umax = fmaxf(umax, u);
                uq += (double)(u + EBAR[t]) * (double)(u + EBAR[t]);
            }
            if (with_hy) {
                __syncwarp();  // both lanes are done with the group sums
                for (int g = h; g < NG; g += 2) {
                    float acc = 0.f;
                    for (int rr = 0; rr < R; ++rr) acc += CS[rr * NG + g] * VOUT[rr * Tp + t];
                    HG[g * Tp + t] = acc;
                }
            }
        }
    };

    // the running sums are accumulated with fire-and-forget reductions, so they start from zero
    auto zero_sums = [&]() {
        if (useAvg) for (int i = tid; i < (N + R) * Tp; i += nthreads) VSUM[i] = 0.f;
    };
    if (P.resume) {
        // (the prologue filled VC / SESS_MU from the warm-start arrays; the PMAX block above ended with a barrier)
        for (int i = tid; i < R * Tp; i += nthreads) VC[i] = P.st_vc[(size_t)b * R * Tp + i];
        for (int i = tid; i < B.S_max; i += nthreads) {
            SESS_MU[i] = P.st_mu[(size_t)b * 2 * B.S_max + i];
            SESS_NF[i] = P.st_mu[(size_t)b * 2 * B.S_max + B.S_max + i];
        }
        __syncthreads();
    } else zero_sums();
    build_matrix();
    write_part_q();
    write_gin();
    __syncthreads();
    // hot row pass: every minimum rate is 0, one session per row, constant upper bound inside each window
    const bool fastRows = !MULTI && SCAL[SC_LBPOS] == 0.f && SCAL[SC_UBVAR] == 0.f && !hasQuad;  // (FAST implies the first two)

    int it = 0, status = ACB_MAX_ITER;
    bool parked = false;
    const int nParts = (NIN + ACB_OHT - 1) / ACB_OHT;
    const int avgEvery = max(1, opt.avg_every);
    for (it = it0 + 1; it <= opt.max_iter; ++it) {
        if (it > P.it_stop) { parked = true; break; }
        const float plevel = SCAL[SC_PLEVEL];
        ACB_TR(0);
        // ------------------------------------------------------------ column pass
        // work item = (period t, block of ACB_OHT outputs): one or two threads per period.  Inputs of a period: the NG
        // group sums of q = 2z - v (summed here from the row warps' partial rows) and the R coupling inputs
        // rho (2z - v), which the coupling warps left in GIN when they updated v.
        for (int wk = tid; wk < nParts * Tp; wk += nthreads) {
            const int part = wk / Tp, t = wk - part * Tp;
            const int obase = part * ACB_OHT;
            float2 out[ACB_OHT / 2];  // outputs (2i, 2i + 1)
#pragma unroll
            for (int k = 0; k < ACB_OHT / 2; ++k) out[k] = make_float2(0.f, 0.f);
            auto accum = [&](int c, float in) {
                const float4* mrow = reinterpret_cast<const float4*>(MFT + c * OP + obase);
#pragma unroll
                for (int h = 0; h < ACB_OHT / 4; ++h) {
                    const float4 m = mrow[h];
                    if constexpr (PAIR) {
                        out[2 * h] = __ffma2_rn(make_float2(m.x, m.y), make_float2(in, in), out[2 * h]);
                        out[2 * h + 1] = __ffma2_rn(make_float2(m.z, m.w), make_float2(in, in), out[2 * h + 1]);
                    } else {
                        out[2 * h].x += m.x * in; out[2 * h].y += m.y * in; out[2 * h + 1].x += m.z * in; out[2 * h + 1].y += m.w * in;
                    }
                }
            };
            for (int g = 0; g < NG; ++g) {
                float acc = 0.f;
                const int p1 = PGOFF[g + 1];
#pragma unroll 4
                for (int p = PGOFF[g]; p < p1; ++p) acc += PART[p * Tp + t];
                accum(g, acc);
            }
            const float* gin = GIN + t;
#pragma unroll 4
            for (int r = 0; r < R; ++r) accum(NG + r, gin[r * Tp]);
            accum(NIN, ALPHA[t]);
            accum(NIN + 1, BETA[t]);
            float* ob = HG + obase * Tp + t;  // (HG, VOUT) output block
#pragma unroll
            for (int k = 0; k < ACB_OHT; ++k)
                if (obase + k < NIN) ob[k * Tp] = (k & 1) ? out[k / 2].y : out[k / 2].x;
        }
        ACB_TR(1);
        __syncthreads();
        ACB_TR(2);
#ifdef ACB_NOCHECK  // experiment: compile the check path out of the loop (the caller never lets a check iteration happen)
        constexpr bool chk = false;
#else
        const bool chk = (it % opt.check_every == 0) || (it == opt.max_iter) || (it == ACB_FIRST_CHECK);  // easy / warm-started instances stop early
#endif
        const bool doAvg = useAvg && (it % avgEvery == 0);
        // rate polish: this check measures the movement of the schedule (every check, or every fourth once the iteration
        // has turned out to contract slowly; see the check path)
        const bool rateTick = polish && chk && SCAL[SC_RATECNT] + 1.f >= SCAL[SC_RATEM];
        const bool avgFirst = SCAL[SC_NSUM] == 0.f;
        float rE1 = 0.f, rE2 = 0.f, rXm = 0.f, rZm = 0.f, rYm = 0.f, rNan = 0.f, rDz = 0.f;
        double dPc = 0.0, dD = 0.0;  // primal (linear + diagonal part) of the current candidate; dual pieces
        // --------------------------------------------------------------- row pass
        // (two instantiations: the hot non-check version keeps fewer values live)
        auto row_pass = [&](auto chk_tag) {
            constexpr bool CHK = decltype(chk_tag)::value;
#pragma unroll
            for (int k = 0; k < TPW; ++k) {
                const int* sl = SLOT + (warp * TPW + k) * 6;
                const int row = sl[0];
                if (row < 0) continue;
                const int g = sl[1], prow = sl[2], first = sl[3], sf = sl[4], scn = sl[5];
                const float mu0 = scn ? SESS_MU[sf] : 0.f;
                const float* hgp = HG + g * Tp + lane;
                float lb[Q], ub[Q], zo[CHK ? Q : 1], xs[CHK ? Q : 1];
                load_bounds(row, lb, ub);
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    float vo = vget(k, q, row);
                    float z = clampf(vo - MU_ELEM(SESS_MU, sf, scn, mu0, lane + 32 * q), lb[q], ub[q]);
                    float x = (rho1 * (2.f * z - vo) + hgp[32 * q]) * inv_d;
                    vset(k, q, row, vo + alpha * (x - z));
                    if (CHK) { zo[q] = z; xs[q] = x; rXm = fmaxf(rXm, fabsf(x)); }
                }
                // projection onto box ∩ energy rows: one multiplier per session
                float vrow[Q];
#pragma unroll
                for (int q = 0; q < Q; ++q) vrow[q] = vget(k, q, row);
                for (int s = sf; s < sf + scn; ++s) {
                    float mu = newton_mu(vrow, lb, ub, SESS_A[s], SESS_B[s], SESS_E[s], SESS_MU[s], !MULTI, 16, SESS_Q[s]);
                    if (lane == 0) SESS_MU[s] = mu;
                    __syncwarp();
                }
                const float mu1 = scn ? SESS_MU[sf] : 0.f;
                float* pp = PART + prow * Tp + lane;
                const float kgc = KG[g];
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    const int t = lane + 32 * q;
                    float vn = vrow[q];
                    float zn = clampf(vn - MU_ELEM(SESS_MU, sf, scn, mu1, t), lb[q], ub[q]);
                    float val = CHK ? zn : 2.f * zn - vn;
                    if (first) pp[32 * q] = val; else pp[32 * q] += val;
                    if (doAvg) {
                        float* vs = VSUM + (size_t)row * Tp + t;
                        atomicAdd(vs, vn);  // result unused -> RED: no load latency on the hot path
                    }
                    if (CHK) {
                        float c = ALPHA[t] + kgc * BETA[t];
                        dPc += (double)(c * zn + qd * zn * zn);
                        rE1 = fmaxf(rE1, fabsf(xs[q] - zn));  // primal residual x - z
                        rE2 = fmaxf(rE2, fabsf(zn - zo[q]));  // dual residual / rho1
                        rZm = fmaxf(rZm, fabsf(zn));
                        rYm = fmaxf(rYm, fabsf(rho1 * (vn - zn)));
                        if (!(fabsf(vn) < 1.0e30f)) rNan = 1.f;
                        if (rateTick) {  // movement of the schedule since the previous measurement
                            float* zp = ZPREV + (size_t)row * Tp + t;
                            rDz = fmaxf(rDz, fabsf(zn - *zp));
                            *zp = zn;
                        }
                    }
                }
                if (CHK && hasQuad) {
                    // objective term cq (Eb - E)^2 of each session of the row, E = planned amp-periods inside its window
                    for (int s = sf; s < sf + scn; ++s) {
                        if (!(SESS_Q[s] > 0.f)) continue;
                        float Es = 0.f;
#pragma unroll
                        for (int q = 0; q < Q; ++q) {
                            const int t = lane + 32 * q;
                            if (MULTI && !(t >= SESS_A[s] && t < SESS_B[s])) continue;
                            Es += clampf(vrow[q] - MU_ELEM(SESS_MU, sf, scn, mu1, t), lb[q], ub[q]);
                        }
                        Es = warp_sum(Es);
                        if (lane == 0) dPc += (double)SESS_Q[s] * (double)(SESS_E[s] - Es) * (double)(SESS_E[s] - Es);
                    }
                }
            }
        };
        // Hot row pass (every minimum rate 0, one session per row, constant upper bound inside each window).  The warp's
        // TPW rows advance together so that their warp reductions overlap.  Clipping is ub * sat((v - mu) / hi) on the
        // FMA pipe; x is never formed (v' = c1 v + c2 z + c3 hg).  The multiplier takes ONE Newton step with the slope
        // remembered from the previous iterations (secant update), and the pass that produces z and the partial sums
        // also verifies the energy equation; only a row that fails the verification (its active set changed) runs the
        // exact safeguarded Newton search.
        auto row_pass_fast = [&]() {
            const float nrel = opt.newton_rel;
            const bool eq = opt.equality != 0;
            const float c1 = 1.f - alpha * rho1 * inv_d, c2 = alpha * (2.f * rho1 * inv_d - 1.f), c3 = alpha * inv_d;
            float mu[TPW], Eb[TPW], E[TPW], E1[TPW], ih[TPW];
            int rowk[TPW], sfk[TPW];
            unsigned verify = 0, exact = 0;  // bit k: row k took a step to be verified / needs the exact search
#pragma unroll
            for (int k = 0; k < TPW; ++k) {
                const int* sl = SLOT + (warp * TPW + k) * 6;
                const int row = sl[0];
                rowk[k] = row; E[k] = 0.f; E1[k] = 0.f; mu[k] = 0.f; Eb[k] = 0.f; ih[k] = 0.f; sfk[k] = -1;
                if (row < 0) continue;
                const int g = sl[1], sf = sl[4], scn = sl[5];
                const float mu0 = scn ? SESS_MU[sf] : 0.f;
                mu[k] = eq ? mu0 : fmaxf(mu0, 0.f);
                Eb[k] = scn ? SESS_E[sf] : 0.f;
                sfk[k] = scn ? sf : -1;
                const float hi_ = ROWHI[warp * TPW + k];
                ih[k] = hi_ > 0.f ? 1.f / hi_ : 0.f;  // rows without any capacity: sat(0 * w) = 0
                const float* hgp = HG + g * Tp + lane;
                const float* ubp = UB + row * Tp + lane;
                float e = 0.f;
#pragma unroll
                for (int q = 0; q < Q; q += PAIR ? 2 : 1) {
                    if (PAIR && q + 1 < Q) {  // elements (q, q + 1) in paired ops; the saturating multiplies and the sum e stay scalar
                        const float2 ub = make_float2(ubp[32 * q], ubp[32 * q + 32]), vo = make_float2(vget(k, q, row), vget(k, q + 1, row));
                        const float2 d = __fadd2_rn(vo, make_float2(-mu0, -mu0));
                        const float2 z = __fmul2_rn(ub, make_float2(__saturatef(d.x * ih[k]), __saturatef(d.y * ih[k])));
                        const float2 vn = __ffma2_rn(make_float2(c3, c3), make_float2(hgp[32 * q], hgp[32 * q + 32]),
                                                     __ffma2_rn(make_float2(c2, c2), z, __fmul2_rn(make_float2(c1, c1), vo)));
                        vset(k, q, row, vn.x); vset(k, q + 1, row, vn.y);
                        const float2 d1 = __fadd2_rn(vn, make_float2(-mu[k], -mu[k]));
                        e = fmaf(ub.x, __saturatef(d1.x * ih[k]), e);
                        e = fmaf(ub.y, __saturatef(d1.y * ih[k]), e);
                    } else {
                        const float ub = ubp[32 * q], vo = vget(k, q, row);
                        const float z = ub * __saturatef((vo - mu0) * ih[k]);
                        const float vn = fmaf(c3, hgp[32 * q], fmaf(c2, z, c1 * vo));
                        vset(k, q, row, vn);
                        e = fmaf(ub, __saturatef((vn - mu[k]) * ih[k]), e);
                    }
                }
                E[k] = e;
            }
            if (doAvg) {
#pragma unroll
                for (int k = 0; k < TPW; ++k) {
                    if (rowk[k] < 0) continue;
                    float* vs = VSUM + (size_t)rowk[k] * Tp + lane;
#pragma unroll
                    for (int q = 0; q < Q; ++q) atomicAdd(vs + 32 * q, vget(k, q, rowk[k]));  // result unused -> RED
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int k = 0; k < TPW; ++k) E[k] += __shfl_xor_sync(0xffffffffu, E[k], o);
            }
            float mun[TPW];
#pragma unroll
            for (int k = 0; k < TPW; ++k) {
                mun[k] = mu[k];
                if (sfk[k] < 0) continue;
                const float rr = E[k] - Eb[k];
                if (fabsf(rr) <= 2e-6f * (Eb[k] + 1.f)) continue;            // still exact
                if (!eq && mu[k] <= 0.f && rr < 0.f) { mun[k] = 0.f; continue; }  // energy cap inactive
                const float nfe = SESS_NF[sfk[k]];
                if (nfe > 0.f) {
                    float m1 = mu[k] + rr / nfe;
                    if (!eq) m1 = fmaxf(m1, 0.f);
                    mun[k] = m1;
                    verify |= 1u << k;
                } else exact |= 1u << k;
            }
            // z and the partial sums of 2z - v with the stepped multipliers (verifying them on the way); the pass is
            // repeated once, without verification, if some row had to run the exact search
            for (int round = 0; round < 2; ++round) {
                float2 acc[(Q + 1) / 2];  // elements (q, q + 1) of the partial row in acc[q / 2] (odd Q: the last .y is unused)
#pragma unroll
                for (int k = 0; k < TPW; ++k) {
                    const int row = rowk[k];
                    if (row < 0) continue;
                    const int* sl = SLOT + (warp * TPW + k) * 6;
                    const bool first = sl[3] != 0;
                    const float* ubp = UB + row * Tp + lane;
                    float e = 0.f;
#pragma unroll
                    for (int q = 0; q < Q; q += PAIR ? 2 : 1) {
                        if (PAIR && q + 1 < Q) {
                            const float2 vn = make_float2(vget(k, q, row), vget(k, q + 1, row));
                            const float2 d = __fadd2_rn(vn, make_float2(-mun[k], -mun[k]));
                            const float2 zn = __fmul2_rn(make_float2(ubp[32 * q], ubp[32 * q + 32]),
                                                         make_float2(__saturatef(d.x * ih[k]), __saturatef(d.y * ih[k])));
                            const float2 val = __ffma2_rn(make_float2(2.f, 2.f), zn, make_float2(-vn.x, -vn.y));
                            acc[q / 2] = first ? val : __fadd2_rn(acc[q / 2], val);
                            e += zn.x;
                            e += zn.y;
                        } else {
                            const float vn = vget(k, q, row);
                            const float zn = ubp[32 * q] * __saturatef((vn - mun[k]) * ih[k]);
                            const float val = fmaf(2.f, zn, -vn);
                            float& a = (q & 1) ? acc[q / 2].y : acc[q / 2].x;
                            a = first ? val : a + val;
                            e += zn;
                        }
                    }
                    E1[k] = e;
                    const bool last = (k == TPW - 1) || rowk[k + 1 < TPW ? k + 1 : k] < 0 || SLOT[(warp * TPW + k + 1) * 6 + 3] != 0;
                    if (last) {
                        float* pp = PART + sl[2] * Tp + lane;
#pragma unroll
                        for (int q = 0; q < Q; ++q) pp[32 * q] = (q & 1) ? acc[q / 2].y : acc[q / 2].x;
                    }
                }
                if (round == 1 || (verify | exact) == 0) break;
                if (verify) {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                        for (int k = 0; k < TPW; ++k) E1[k] += __shfl_xor_sync(0xffffffffu, E1[k], o);
                    }
#pragma unroll
                    for (int k = 0; k < TPW; ++k) {
                        if (!(verify >> k & 1)) continue;
                        const float rr1 = E1[k] - Eb[k], dmu = mun[k] - mu[k];
                        // (between checks the projection may be inexact by a fraction of the step it just took: the
                        // multiplier is warm-started every iteration and the check iterations project exactly)
                        const bool ok = fabsf(rr1) <= 2e-6f * (Eb[k] + 1.f) + nrel * fabsf(E[k] - Eb[k]) || (!eq && mun[k] <= 0.f && rr1 < 0.f);
                        // secant slope of the energy equation between the two evaluations = free elements on the way
                        const float sec = (dmu != 0.f) ? (E[k] - E1[k]) / dmu : 0.f;
                        if (lane == 0) SESS_NF[sfk[k]] = (ok && sec >= 0.5f) ? sec : 0.f;
                        if (!ok) exact |= 1u << k;
                    }
                }
                if (!exact) break;
                // exact search for the rows that need it (first visit, or the active set changed under the step)
#pragma unroll
                for (int k = 0; k < TPW; ++k) {
                    if (!(exact >> k & 1)) continue;
                    float lb[Q], ub[Q], vrow[Q];
                    load_bounds(rowk[k], lb, ub);
#pragma unroll
                    for (int q = 0; q < Q; ++q) vrow[q] = vget(k, q, rowk[k]);
                    const float m0 = mu[k];
                    mun[k] = newton_mu(vrow, lb, ub, 0, Tp, Eb[k], m0, true, 16);
                    // slope at the solution for the next iterations
                    int nf = 0;
#pragma unroll
                    for (int q = 0; q < Q; ++q) { const float w = vrow[q] - mun[k]; nf += (w > 0.f && w < ub[q]) ? 1 : 0; }
                    nf = __reduce_add_sync(0xffffffffu, nf);
                    if (lane == 0) SESS_NF[sfk[k]] = (float)nf;
                }
            }
            if (lane == 0) {
#pragma unroll
                for (int k = 0; k < TPW; ++k)
                    if (sfk[k] >= 0) SESS_MU[sfk[k]] = mun[k];
            }
        };
        // ---------------------------------------------------------- coupling rows
        // v update and GIN <- rho (2 z(v) - v) for the next column pass; on check iterations VOUT <- y = rho (v - z)
        // and the conjugate terms of D.  Work item = (task, 32-period chunk), dealt round-robin to the coupling warps.
        // (templated on the check flag like the row pass: the accumulators of the dual bound must not be live, i.e. spilled,
        // across the hot iterations)
        auto couple_item = [&](int item, auto chk_tag) {
            constexpr bool CHK = decltype(chk_tag)::value;
            {
                const int c = item / Q, t = (item - c * Q) * 32 + lane;
                if (c < nDisc) {
                    const int r = 2 * c;
                    const float lim = LIM[r];
                    // the (a, b) components in paired ops; v + alpha (k - f v) keeps k - f v as one FMA (f v is not rounded)
                    const float2 v = make_float2(VC[r * Tp + t], VC[(r + 1) * Tp + t]);
                    const float f = disc_scale(v.x, v.y, lim);
                    const float2 kv = make_float2(VOUT[r * Tp + t], VOUT[(r + 1) * Tp + t]);
                    const float2 vn = __ffma2_rn(__ffma2_rn(v, make_float2(-f, -f), kv), make_float2(alpha, alpha), v);
                    const float an = vn.x, bn = vn.y;
                    VC[r * Tp + t] = an; VC[(r + 1) * Tp + t] = bn;
                    const float fn = disc_scale(an, bn, lim);
                    const float2 zn = __fmul2_rn(vn, make_float2(fn, fn));
                    const float2 gin = __fmul2_rn(make_float2(rho, rho), __fadd2_rn(__fadd2_rn(zn, zn), make_float2(-an, -bn)));  // rho (2 z - v)
                    GIN[r * Tp + t] = gin.x; GIN[(r + 1) * Tp + t] = gin.y;
                    if (doAvg) {
                        float* vs = VSUM + (size_t)(N + r) * Tp + t;
                        atomicAdd(vs, an); atomicAdd(vs + Tp, bn);
                    }
                    if (CHK) {
                        const float zan = zn.x, zbn = zn.y;
                        float ya = rho * (an - zan), yb = rho * (bn - zbn);
                        VOUT[r * Tp + t] = ya; VOUT[(r + 1) * Tp + t] = yb;
                        dD -= (double)(lim * sqrtf(ya * ya + yb * yb));  // support function of the disc
                    }
                } else {
                    const int r = 2 * nDisc + (c - nDisc);
                    const bool isPL = (c == nDisc + nLin);
                    const float lo = isPL ? -3.0e38f : linLo;
                    float cap = isPL ? PLIM[t] : LIM[r];
                    float capLo = (lo < -1.0e30f) ? lo : lo * cap;
                    float v = VC[r * Tp + t], z = clampf(v, capLo, cap), kx = VOUT[r * Tp + t];
                    float vn = v + alpha * (kx - z);
                    VC[r * Tp + t] = vn;
                    float zn = clampf(vn, capLo, cap);
                    GIN[r * Tp + t] = rho * (2.f * zn - vn);
                    if (doAvg) { atomicAdd(VSUM + (size_t)(N + r) * Tp + t, vn); }
                    if (CHK) {
                        float y = rho * (vn - zn);
                        VOUT[r * Tp + t] = y;
                        if (y != 0.f) dD -= (double)(cap * fabsf(y));  // support function of the half line / interval
                    }
                }
            }
        };
        // the first rowShare * nRowWarps items ride on the row warps (after their own rows), the rest is dealt
        // round-robin to the coupling warps
        auto couple_all = [&](auto chk_tag) {
        constexpr bool CHK = decltype(chk_tag)::value;
        if (rowWarp) {
            for (int j = 0; j < rowShare; ++j) couple_item(warp * rowShare + j, chk_tag);
        }
        if (cwIdx >= 0) {
            for (int item = rowShare * S.nRowWarps + cwIdx; item < nCT1 * Q; item += nCW) couple_item(item, chk_tag);
        }
        if (doAgg) {
            // aggregate-power row: quadratic (load flattening) + peak epigraph
            const int r = rU;
            for (int t = lane; t < Tp; t += 32) {
                float v = VC[r * Tp + t], a = agg_a(v, t);
                float z = ((pk_w > 0.f) ? fminf(a, plevel) : a) / su;
                float vn = v + alpha * (VOUT[r * Tp + t] - z);
                VC[r * Tp + t] = vn;
                if (doAvg) { atomicAdd(VSUM + (size_t)(N + r) * Tp + t, vn); }
            }
            __syncwarp();
            const float pl = peak_level(plevel);
            if (lane == 0) SCAL[SC_PLEVEL] = pl;
            float zmax = -3.0e38f;
            double acc = 0.0;
            for (int t = lane; t < Tp; t += 32) {
                float vn = VC[r * Tp + t], an = agg_a(vn, t);
                float zk = (pk_w > 0.f) ? fminf(an, pl) : an;  // kW
                float zn = zk / su;
                GIN[r * Tp + t] = rho * (2.f * zn - vn);
                if (CHK) {
                    // Fenchel equality for y in dg(z): -g*(y) = g(z) - <y, z>
                    float y = rho * (vn - zn);
                    VOUT[r * Tp + t] = y;
                    if (t < Tb) { zmax = fmaxf(zmax, zk); acc += (double)Gamma * (double)(zk + EBAR[t]) * (double)(zk + EBAR[t]); }
                    acc -= (double)y * (double)zn;
                }
            }
            if (CHK) {
                zmax = warp_max(zmax);
                dD += acc;
                if (lane == 0) dD += (double)pk_w * (double)fmaxf(zmax, pk_p0);
            }
        }
        };
        if (!chk) {
            if (rowWarp) {
                if (fastRows) row_pass_fast();
                else row_pass(std::false_type{});
            }
            couple_all(std::false_type{});
            ACB_TR(3);
            __syncthreads();
            ACB_TR(4);
            if (doAvg && tid == 0) SCAL[SC_NSUM] = avgFirst ? 1.f : SCAL[SC_NSUM] + 1.f;  // next read is after the next barrier
            continue;
        }
#ifndef ACB_NOCHECK

        // ============================================================= check path
        // (a check-iteration variant of the fast pass was measured slower: its exact mode ends in the full search)
        if (rowWarp) row_pass(std::true_type{});
        couple_all(std::true_type{});
        ACB_TR(3);
        __syncthreads();  // PART = group sums of z, VOUT = y
        if (doAvg && tid == 0) SCAL[SC_NSUM] = avgFirst ? 1.f : SCAL[SC_NSUM] + 1.f;
        float violC, umaxC; double uqC, plC;
        eval_columns(true, THC, violC, umaxC, uqC, plC);  // HG <- C'y afterwards
        __syncthreads();
        ACB_TR(4);
        // Lagrangian inner minimum over the box and energy-row terms; averaged candidate
        const float nsum = SCAL[SC_NSUM];
        const bool haveAvg = useAvg && nsum >= 2.f;
        const float inv_nsum = 1.f / fmaxf(nsum, 1.f);
        const bool refineDual = opt.dual_refine > 1 || (opt.dual_refine == 1 && SCAL[SC_STALL] >= 1.f);
        double dPa = 0.0;
        if (rowWarp) {
#pragma unroll
            for (int k = 0; k < TPW; ++k) {
                const int* sl = SLOT + (warp * TPW + k) * 6;
                const int row = sl[0];
                if (row < 0) continue;
                const int g = sl[1], prow = sl[2], first = sl[3], sf = sl[4], scn = sl[5];
                const float kgc = KG[g];
                const float mu0 = scn ? SESS_MU[sf] : 0.f;
                float lb[Q], ub[Q], va[Q];
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    int t = lane + 32 * q;
                    bool in = t < Tp;
                    lb[q] = in ? lbv(row, t) : 0.f;
                    ub[q] = in ? ubv(row, t) : 0.f;
                    va[q] = (in && haveAvg) ? VSUM[(size_t)row * Tp + t] : 0.f;  // (all loads in flight together: a division
                    // per load would wait for each in turn)
                }
#pragma unroll
                for (int q = 0; q < Q; ++q) va[q] *= inv_nsum;
#ifdef ACB_TRACE
                if (k == 0) { float sv_ = 0.f; for (int q = 0; q < Q; ++q) sv_ += va[q]; ACB_TRV(12, sv_); }
#endif
                // energy-row multipliers of the dual bound: the iterate's (rho1 * mu_s), or the maximiser given y
                if (refineDual) {
                    float aa[Q];
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        int t = lane + 32 * q;
                        aa[q] = (t < Tp) ? ALPHA[t] + kgc * BETA[t] + HG[g * Tp + t] : 0.f;
                    }
                    for (int s = sf; s < sf + scn; ++s) {
                        // (rows with a quadratic shortfall term keep the iterate's multiplier: any value gives a valid bound)
                        float lam = (SESS_Q[s] > 0.f) ? rho1 * SESS_MU[s] : dual_lambda(aa, lb, ub, SESS_A[s], SESS_B[s], SESS_E[s], rho1 * SESS_MU[s], !MULTI);
                        if (lane == 0) SESS_MU2[s] = lam;
                    }
                } else if (lane == 0) {
                    for (int s = sf; s < sf + scn; ++s) SESS_MU2[s] = rho1 * SESS_MU[s];
                }
                __syncwarp();
                {
                    const float lam0 = scn ? SESS_MU2[sf] : 0.f;
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        int t = lane + 32 * q;
                        if (t >= Tp) continue;
                        // reduced cost: c + (Khat' y) + lambda_s on the session window
                        float rt = ALPHA[t] + kgc * BETA[t] + HG[g * Tp + t] + MU_ELEM(SESS_MU2, sf, scn, lam0, t);
                        float phi;
                        if (qd > 0.f) { float xs = clampf(-rt / (2.f * qd), lb[q], ub[q]); phi = qd * xs * xs + rt * xs; }
                        else phi = fminf(lb[q] * rt, ub[q] * rt);
                        dD += (double)phi;
                    }
                }
                if (lane == 0)
                    for (int s = sf; s < sf + scn; ++s) {
                        const double m = (double)SESS_MU2[s];
                        dD -= m * (double)SESS_E[s];
                        // cq (Eb - E)^2 >= nu (Eb - E) - nu^2 / (4 cq): a negative multiplier m is nu = -m of that bound
                        if (m < 0.0 && SESS_Q[s] > 0.f) dD -= m * m / (4.0 * (double)SESS_Q[s]);
                    }
                __syncwarp();  // SESS_MU2 is reused for the averaged candidate below
                if (k == 0) ACB_TRV(13, (float)dD);
                if (haveAvg) {
                    for (int s = sf; s < sf + scn; ++s) {
                        float mu = newton_mu(va, lb, ub, SESS_A[s], SESS_B[s], SESS_E[s], SESS_MU[s], !MULTI, 16, SESS_Q[s]);
                        if (lane == 0) SESS_MU2[s] = mu;
                        __syncwarp();
                        if (k == 0) ACB_TRV(14, mu);
                    }
                    const float mu2 = scn ? SESS_MU2[sf] : 0.f;
                    if (hasQuad) {
                        for (int s = sf; s < sf + scn; ++s) {
                            if (!(SESS_Q[s] > 0.f)) continue;
                            float Es = 0.f;
#pragma unroll
                            for (int q = 0; q < Q; ++q) {
                                const int t = lane + 32 * q;
                                if (MULTI && !(t >= SESS_A[s] && t < SESS_B[s])) continue;
                                Es += clampf(va[q] - MU_ELEM(SESS_MU2, sf, scn, mu2, t), lb[q], ub[q]);
                            }
                            Es = warp_sum(Es);
                            if (lane == 0) dPa += (double)SESS_Q[s] * (double)(SESS_E[s] - Es) * (double)(SESS_E[s] - Es);
                        }
                    }
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        int t = lane + 32 * q;
                        if (t >= Tp) continue;
                        float zn = clampf(va[q] - MU_ELEM(SESS_MU2, sf, scn, mu2, t), lb[q], ub[q]);
                        if (first) PART[prow * Tp + t] = zn; else PART[prow * Tp + t] += zn;
                        float c = ALPHA[t] + kgc * BETA[t];
                        dPa += (double)(c * zn + qd * zn * zn);
                    }
                }
            }
        }
        ACB_TR(5);
        __syncthreads();  // PART = group sums of the averaged candidate
        float violA = 3.0e38f, umaxA = -3.0e38f; double uqA = 0.0, plA = 0.0;
        if (haveAvg) eval_columns(false, THA, violA, umaxA, uqA, plA);
        ACB_TR(6);
        // block reductions
        rE1 = warp_max(rE1); rE2 = warp_max(rE2); rXm = warp_max(rXm); rZm = warp_max(rZm); rYm = warp_max(rYm); rNan = warp_max(rNan); rDz = warp_max(rDz);
        violC = warp_max(violC); umaxC = warp_max(umaxC);
        violA = warp_max(violA); umaxA = warp_max(umaxA);
        dPc = warp_sum(dPc); dPa = warp_sum(dPa); dD = warp_sum(dD); uqC = warp_sum(uqC); uqA = warp_sum(uqA);
        plC = warp_sum(plC); plA = warp_sum(plA);
        if (lane == 0) {
            float* rf = REDF + warp * ACB_NRED;
            rf[RF_E1] = rE1; rf[RF_E2] = rE2; rf[RF_XMAX] = rXm; rf[RF_ZMAX] = rZm; rf[RF_YMAX] = rYm; rf[RF_NAN] = rNan;
            rf[RF_VIOLC] = violC; rf[RF_VIOLA] = violA; rf[RF_UMAXC] = umaxC; rf[RF_UMAXA] = umaxA; rf[RF_DZ] = rDz;
            double* rd = REDD + warp * ACB_NRED;
            rd[RD_PC] = dPc; rd[RD_PA] = dPa; rd[RD_D] = dD; rd[RD_UQC] = uqC; rd[RD_UQA] = uqA; rd[RD_PLC] = plC; rd[RD_PLA] = plA;
        }
        __syncthreads();
        ACB_TR(7);
        if (tid == 0) {
            float e1 = 0, e2 = 0, xm = 0, zm = 0, ym = 0, nn = 0, vC = -1.f, vA = -1.f, uC = -3.0e38f, uA = -3.0e38f, dz = 0.f;
            double Pc = 0, Pa = 0, D = 0, qC = 0, qA = 0, lC = 0, lA = 0;
            for (int w = 0; w < nwarps; ++w) {
                const float* rf = REDF + w * ACB_NRED;
                e1 = fmaxf(e1, rf[RF_E1]); e2 = fmaxf(e2, rf[RF_E2]); xm = fmaxf(xm, rf[RF_XMAX]); zm = fmaxf(zm, rf[RF_ZMAX]);
                ym = fmaxf(ym, rf[RF_YMAX]); nn = fmaxf(nn, rf[RF_NAN]); vC = fmaxf(vC, rf[RF_VIOLC]);
                if (haveAvg) vA = fmaxf(vA, rf[RF_VIOLA]);
                uC = fmaxf(uC, rf[RF_UMAXC]); uA = fmaxf(uA, rf[RF_UMAXA]); dz = fmaxf(dz, rf[RF_DZ]);
                const double* rd = REDD + w * ACB_NRED;
                Pc += rd[RD_PC]; Pa += rd[RD_PA]; D += rd[RD_D]; qC += rd[RD_UQC]; qA += rd[RD_UQA]; lC += rd[RD_PLC]; lA += rd[RD_PLA];
            }
            if (canRestore) { Pc = lC; Pa = lA; }  // objective of the restored (scaled) candidates, from the column sums
            // The tolerance scale is max(|P|, |D|, opt.term_floor * sum of the |objective terms|): with a demand charge
            // the sunk peak cost w*p0 and the energy revenue can cancel to ~0 (closed-loop replay sitting at the
            // previous peak), and a gap relative to that difference alone would ask for more digits than the terms have.
            double magC = fabs(Pc), magA = fabs(Pa);
            if (S.has_u) {
                const double gC = (double)Gamma * qC + (double)pk_w * (double)fmaxf(uC, pk_p0);
                const double gA = (double)Gamma * qA + (double)pk_w * (double)fmaxf(uA, pk_p0);
                Pc += gC; Pa += gA;
                magC += fabs(gC); magA += fabs(gA);
            }
            magC = fmax(fabs(Pc), (double)opt.term_floor * magC);
            magA = fmax(fabs(Pa), (double)opt.term_floor * magA);
            double Dbest = SCALD[SD_DBEST];
            if (D == D && D > Dbest) Dbest = D;
            SCALD[SD_DBEST] = Dbest;
            const double gapC = Pc - Dbest, gapA = Pa - Dbest;
            const double tolC = (double)opt.eps_abs + (double)opt.eps_rel * fmax(magC, fabs(Dbest));
            const double tolA = (double)opt.eps_abs + (double)opt.eps_rel * fmax(magA, fabs(Dbest));
            // residual estimates (only used to balance rho)
            float rp = e1, rd_ = rho1 * e2;
            float rp_rel = rp / fmaxf(fmaxf(xm, zm), 1e-6f), rd_rel = rd_ / fmaxf(1.0f, ym);
            float flag = 0.f;
            // a (slightly) negative gap is rounding noise around a converged pair and passes; negative tolerances
            // therefore mean "never stop on the gap" (run the whole iteration budget)
            // rate polish: with a linearly converging iteration the movement dz between two measurements and the ratio
            // kap of two consecutive movements give the remaining distance dz kap / (1 - kap).  The extrapolation is only
            // trusted while the contraction per measurement is strong (ratios <= 0.5: factor <= 1).  On nearly flat
            // objectives the schedule contracts by ~0.9 per check period, the movement per period at 1e-3 A from the
            // optimum (~1e-4 A) is as large as the float32 noise of the iteration, and single ratios are meaningless:
            // the measurements then switch to every FOURTH check (contraction ~0.7, four times the signal).  There the
            // stop is est <= rate_tol with the ratio capped at 0.9, or a movement below rate_tol at two consecutive
            // measurements: the float32 floor of the schedule on such objectives is 1e-4 .. 5e-4 A, where the ratios carry
            // no information any more (the maximum over 15 k elements is biased upwards by the noise, so the movement is
            // not underestimated; polish_min_qd keeps flatter objectives, which contract slower than ~0.7 per hundred
            // iterations, out of the polish).
            bool okRate = true;
            if (polish) {
                okRate = false;
                if (rateTick) {
                    const float dzp = SCAL[SC_DZ], nd = SCAL[SC_NDZ], m = SCAL[SC_RATEM];
                    const float kap = (nd >= 1.f && dzp > 0.f) ? dz / dzp : 1.f;
                    const float kprev = (nd >= 2.f) ? SCAL[SC_KAP] : (m > 1.f ? 0.f : 1.f);
                    const float ku = fminf(fmaxf(kap, kprev), m > 1.f ? 0.9f : 0.98f);
                    float est = 3.0e38f, nok = 0.f;
                    bool slow = false;
                    if (m <= 1.f) {
                        if (nd >= 2.f) {
                            est = dz * ku / (1.f - ku);
                            // (a movement at the float32 noise floor of the rates counts as converged whatever the ratio says)
                            okRate = (ku <= 0.5f && est <= opt.rate_tol) || dz <= 1e-5f;
                            slow = !okRate && ku > 0.5f;
                        }
                    } else if (nd >= 1.f) {
                        est = dz * ku / (1.f - ku);
                        nok = (dz <= opt.rate_tol) ? SCAL[SC_NRATEOK] + 1.f : 0.f;
                        okRate = est <= opt.rate_tol || nok >= 2.f;
                        if (okRate && est > opt.rate_tol) est = dz;  // at the floor: nothing below the movement itself is resolved
                    }
                    SCAL[SC_RATE_EST] = est;
                    SCAL[SC_NRATEOK] = nok;
                    if (slow) {  // start over on the long baseline (the snapshot was just refreshed)
                        SCAL[SC_RATEM] = 4.f; SCAL[SC_NDZ] = 0.f; SCAL[SC_DZ] = 0.f; SCAL[SC_KAP] = 0.f;
                    } else {
                        SCAL[SC_KAP] = (nd >= 1.f) ? kap : 0.f;
                        SCAL[SC_DZ] = dz;
                        SCAL[SC_NDZ] = nd + 1.f;
                    }
                    SCAL[SC_RATECNT] = 0.f;
                } else SCAL[SC_RATECNT] += 1.f;
            }
            const bool certC = gapC <= tolC && vC <= opt.viol_tol;  // gap and violation certified; the polish may still be running
            const bool okC = certC && okRate;
            const bool okA = haveAvg && !polish && gapA <= tolA && vA <= opt.viol_tol;
            if (nn > 0.f || !(Pc == Pc)) flag = 3.f;
            else if (Dbest > SCALD[SD_PMAX] + 1e-3 * (fabs(SCALD[SD_PMAX]) + 1.0)) flag = 6.f;  // infeasibility certificate
            else if (okC && (!okA || gapC <= gapA)) flag = 1.f;
            else if (okA) flag = 4.f;
            else if (certC) {
                // only the rate polish is pending: no restarts, rescues or penalty changes (each would reset its history)
            } else {
                // (once the averaged gap is inside the tolerance only the violation is pending: restarting on the noise of
                // a converged gap would keep resetting the stall counter and block the penalty rescue)
                if (haveAvg && gapA <= 0.5 * SCALD[SD_GAPRESTART] && SCALD[SD_GAPRESTART] > tolA && vA <= fmaxf(vC, opt.viol_tol) + 1e-3f) {
                    SCALD[SD_GAPRESTART] = gapA;
                    flag = 5.f;
                }
                // stagnation rescue: the best gap has not improved by 10 % over `stall_checks` checks ->
                // change the penalty once to 3x and, if that stalls too, once to 1/3 of the start value
                {
                    // (a gap below a tenth of the tolerance has nothing left to gain: its rounding noise must not keep
                    // resetting the stall counter while only the violation is pending)
                    const double gbest = fmax(fmin(gapC, haveAvg ? gapA : gapC), 0.1 * tolC);
                    if (gbest < 0.9 * SCALD[SD_BESTGAP]) { SCALD[SD_BESTGAP] = gbest; SCAL[SC_STALL] = 0.f; }
                    else SCAL[SC_STALL] += 1.f;
                    // 1st rescue: a stiffer penalty (x3).  2nd, only for warm-started solves: drop the inherited state and
                    // start over cold, keeping the best dual bound.  (A second penalty change on cold-started solves
                    // measured worse than none.)
                    const int nresc = (int)SCAL[SC_NRESCUE];
                    const bool canRescue = nresc < opt.max_rescues && (nresc == 0 || (nresc == 1 && B.warm_v1 != nullptr && (!B.warm_had || B.warm_had[b] != 0)));
                    if (flag == 0.f && opt.stall_checks > 0 && SCAL[SC_STALL] >= (float)opt.stall_checks && canRescue) {
                        const bool cold = nresc > 0;
                        SCAL[SC_NEWRHO] = cold ? opt.rho0 : fminf(fmaxf(rho * 3.f, 1e-4f), 1e4f);
                        SCAL[SC_NRESCUE] = (float)(nresc + 1);
                        SCAL[SC_STALL] = 0.f;
                        SCALD[SD_BESTGAP] = 1.0e300;
                        SCALD[SD_GAPRESTART] = 1.0e300;
                        flag = cold ? 11.f : 10.f;
                    } else if (flag == 0.f && gapC <= tolC && opt.stall_checks > 0 && SCAL[SC_NFEAS] < 3.f &&
                               ((vC < 0.9f * SCAL[SC_BESTVIOL]) ? (SCAL[SC_BESTVIOL] = vC, SCAL[SC_VSTALL] = 0.f, false)
                                                               : ((SCAL[SC_VSTALL] += 1.f) >= (float)opt.stall_checks))) {
                        // feasibility rescue: the gap is certified but the coupling violation of a candidate that cannot be
                        // restored by scaling (minimum rates, quadratic terms, equality rows) no longer shrinks: a stiffer
                        // penalty drives the primal residual down (up to three times)
                        SCAL[SC_NEWRHO] = fminf(fmaxf(rho * 3.f, 1e-4f), 1e4f);
                        SCAL[SC_NFEAS] += 1.f;
                        SCAL[SC_VSTALL] = 0.f; SCAL[SC_BESTVIOL] = 3.0e38f; SCAL[SC_STALL] = 0.f;
                        SCALD[SD_BESTGAP] = 1.0e300;
                        SCALD[SD_GAPRESTART] = 1.0e300;
                        flag = 10.f;
                    } else if (flag == 0.f && opt.stall_exit > 0 && SCAL[SC_STALL] >= (float)opt.stall_exit && !canRescue) {
                        flag = 2.f;  // stalled for good: stop with the best certified gap so far (status ACB_MAX_ITER)
                    }
                }
                if (opt.adapt_rho && flag < 10.f && flag != 2.f) {
                    const float opt_ratio = (opt.adapt_rho > 1) ? 0.1f * (float)opt.adapt_rho : 5.f;  // adapt_rho = 10 x threshold, 1 = default 5
                    float ratio = sqrtf(fmaxf(rp_rel, 1e-12f) / fmaxf(rd_rel, 1e-12f));
                    if (ratio > opt_ratio || ratio < 1.f / opt_ratio) {
                        SCAL[SC_NEWRHO] = fminf(fmaxf(rho * ratio, 0.1f * rho_start), 10.f * rho_start);  // stay within a decade of the start value
                        flag += 10.f;  // combined with a restart: 15
                    }
                }
            }
            if (flag == 5.f || flag >= 10.f) { SCAL[SC_NDZ] = 0.f; SCAL[SC_NRATEOK] = 0.f; }  // the iterate jumps: the movement history starts over
            SCAL[SC_FLAG] = flag;
            SCAL[SC_RP] = rp_rel; SCAL[SC_RD] = rd_rel;
            const bool useA = (flag == 4.f);
            SCAL[SC_GAP] = (float)((useA ? gapA : gapC) / fmax(fmax(useA ? magA : magC, fabs(Dbest)), 1e-30));
            SCAL[SC_VIOL] = useA ? vA : vC;
        }
        __syncthreads();
        ACB_TR(8);
        const float flag = SCAL[SC_FLAG];
#ifdef ACB_TRACE
        if (b == 0 && it >= ACB_TR_IT0 && it < ACB_TR_IT0 + ACB_TR_NIT && tid == 0) g_acb_trace[((it - ACB_TR_IT0) * 32 + 31) * ACB_TR_SLOTS + 15] = (long long)flag;
#endif
        if (flag == 1.f) { status = ACB_SOLVED; break; }
        if (flag == 3.f) { status = ACB_NUMERICAL; break; }
        if (flag == 6.f) { status = ACB_INFEASIBLE; break; }
        if (flag == 2.f) break;  // status stays ACB_MAX_ITER
        // (not on the last iteration: the returned schedule and its reported gap / violation must be the current candidate's)
        const bool toAvg = (flag == 4.f) || ((flag == 5.f || flag == 15.f) && it < opt.max_iter);
        if (toAvg) {
            // adopt the averaged state: v <- mean v, multipliers of its projection, mean coupling v
            if (rowWarp) {
#pragma unroll
                for (int k = 0; k < TPW; ++k) {
                    const int* sl = SLOT + (warp * TPW + k) * 6;
                    int row = sl[0];
                    if (row < 0) continue;
                    float* vs = VSUM + (size_t)row * Tp + lane;
                    float sv[Q];
#pragma unroll
                    for (int q = 0; q < Q; ++q) sv[q] = vs[32 * q];
#pragma unroll
                    for (int q = 0; q < Q; ++q) { vset(k, q, row, sv[q] * inv_nsum); vs[32 * q] = 0.f; }
                }
            }
            // (the running sums restart from zero: every element is zeroed by the thread that just read it; rows without
            // a session never receive a contribution)
            for (int i = tid; i < B.S_max; i += nthreads) SESS_MU[i] = SESS_MU2[i];
            for (int i = tid; i < R * Tp; i += nthreads) { float* vs = VSUM + (size_t)N * Tp + i; VC[i] = *vs * inv_nsum; *vs = 0.f; }
            __syncthreads();
            if (S.has_u && warp == nwarps - 1) {
                float pl = peak_level(SCAL[SC_PLEVEL]);
                if (lane == 0) SCAL[SC_PLEVEL] = pl;
            }
            if (tid == 0) { SCAL[SC_NSUM] = 0.f; SCAL[SC_NREST] += 1.f; }
            __syncthreads();
            if (flag == 4.f) { status = ACB_SOLVED; if (tid == 0) SCAL[SC_USEDAVG] = 1.f; break; }
        }
        if (it == opt.max_iter) break;
        if (flag >= 10.f) {
            // keep y: v <- z + (rho/rho_new)(v - z), then rebuild the column matrix
            const float rn = SCAL[SC_NEWRHO], f = rho / rn;
            if (flag == 11.f) {
                // cold reset: the state a solve without warm start begins with
                if (rowWarp) {
#pragma unroll
                    for (int k = 0; k < TPW; ++k) {
                        int row = SLOT[(warp * TPW + k) * 6];
                        if (row < 0) continue;
#pragma unroll
                        for (int q = 0; q < Q; ++q) {
                            int t = lane + 32 * q;
                            if (t < Tp) vset(k, q, row, clampf(0.f, lbv(row, t), ubv(row, t)));
                        }
                    }
                }
                for (int i = tid; i < B.S_max; i += nthreads) SESS_MU[i] = 0.f;
                for (int i = tid; i < R * Tp; i += nthreads) VC[i] = 0.f;
                if (tid == 0) SCAL[SC_PLEVEL] = pk_p0;
            } else {
            if (rowWarp) {
#pragma unroll
                for (int k = 0; k < TPW; ++k) {
                    const int* sl = SLOT + (warp * TPW + k) * 6;
                    int row = sl[0];
                    if (row < 0) continue;
                    const float mu0 = sl[5] ? SESS_MU[sl[4]] : 0.f;
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        int t = lane + 32 * q;
                        if (t >= Tp) continue;
                        const float vq = vget(k, q, row);
                        float z = clampf(vq - MU_ELEM(SESS_MU, sl[4], sl[5], mu0, t), lbv(row, t), ubv(row, t));
                        vset(k, q, row, z + f * (vq - z));
                    }
                }
            }
            __syncthreads();  // every row warp has used the old multipliers
            // mu = (energy-row dual) / rho1 scales with the penalty like v - z does
            for (int i = tid; i < B.S_max; i += nthreads) SESS_MU[i] *= f;
            const float pl = SCAL[SC_PLEVEL];
            for (int t = tid; t < Tp; t += nthreads) {
                int r = 0;
                for (int j = 0; j < nDisc; ++j, r += 2) {
                    float a = VC[r * Tp + t], bb = VC[(r + 1) * Tp + t], za, zb;
                    proj_disc(a, bb, LIM[r], za, zb);
                    VC[r * Tp + t] = za + f * (a - za); VC[(r + 1) * Tp + t] = zb + f * (bb - zb);
                }
                for (int j = 0; j < nLin; ++j, ++r) { float v = VC[r * Tp + t], z = clampf(v, (linLo < -1.0e30f) ? linLo : linLo * LIM[r], LIM[r]); VC[r * Tp + t] = z + f * (v - z); }
                if (S.has_pl) { float v = VC[r * Tp + t], z = fminf(v, PLIM[t]); VC[r * Tp + t] = z + f * (v - z); ++r; }
                if (S.has_u) {
                    float v = VC[r * Tp + t], a = agg_a(v, t);
                    float z = ((pk_w > 0.f) ? fminf(a, pl) : a) / su;
                    VC[r * Tp + t] = z + f * (v - z);
                }
            }
            }
            __syncthreads();
            rho = rn; rho1 = kappa * rho; dd = 2.f * qd + rho1; inv_d = 1.f / dd;
            set_agg();
            zero_sums();
            if (tid == 0) { SCAL[SC_RHO] = rho; SCAL[SC_NSUM] = 0.f; }  // the average restarts with the new metric
            build_matrix();
        }
        ACB_TR(9);
        write_part_q();
        ACB_TR(10);
        if (toAvg || flag >= 10.f) write_gin();  // (otherwise the coupling pass of this iteration left GIN current)
        __syncthreads();
        ACB_TR(11);
#endif
    }
    if (it > opt.max_iter) it = opt.max_iter;
    if (parked) {
        // park the complete state; PART / VOUT / MFT are rebuilt from it on resume, the running sums stay in B.work
        --it;
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            const int row = rowWarp ? SLOT[(warp * TPW + k) * 6] : -1;
            if (row < 0) continue;
#pragma unroll
            for (int q = 0; q < Q; ++q) P.st_v1[((size_t)b * N + row) * Tp + lane + 32 * q] = vget(k, q, row);
        }
        for (int i = tid; i < R * Tp; i += nthreads) P.st_vc[(size_t)b * R * Tp + i] = VC[i];
        for (int i = tid; i < B.S_max; i += nthreads) {
            P.st_mu[(size_t)b * 2 * B.S_max + i] = SESS_MU[i];
            P.st_mu[(size_t)b * 2 * B.S_max + B.S_max + i] = SESS_NF[i];
        }
        float* stp = P.st_scal + (size_t)b * ACB_NSTATE;
        if (tid < 32) stp[tid] = SCAL[tid];
        else if (tid < 64) stp[tid] = sm[L.SCALD + tid - 32];
        if (tid == 0) {
            B.status[b] = ACB_RUNNING;
            B.iters[b] = it;
            float* st = B.stats + (size_t)b * ACB_NSTATS;  // the scheduler between the launches ranks by the gap of the last check
            st[2] = SCAL[SC_GAP]; st[3] = SCAL[SC_VIOL];
        }
        return;
    }

    // ------------------------------------------------------------------ epilogue
    __syncthreads();  // SC_USEDAVG (written by thread 0 just before leaving the loop) must be visible
    const float* THX = (SCAL[SC_USEDAVG] != 0.f) ? THA : THC;  // restoration factors of the returned candidate
    if (rowWarp) {
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            const int* sl = SLOT + (warp * TPW + k) * 6;
            int row = sl[0];
            if (row < 0) continue;
            const float mu0 = sl[5] ? SESS_MU[sl[4]] : 0.f;
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                int t = lane + 32 * q;
                if (t >= Tp) continue;
                const float vq = vget(k, q, row);
                float z = clampf(vq - MU_ELEM(SESS_MU, sl[4], sl[5], mu0, t), lbv(row, t), ubv(row, t));
                const float rt = z * THX[t];
                B.rates[((size_t)b * N + row) * Tp + t] = rt;
                // fused project_into_continuous_feasible_pilots (postprocessing.py:77-94) + the final max(., 0) of schedule()
                if (B.pilots) {  // same selects as k_project_continuous (acb_post.cu)
                    double pv = (double)rt;
                    const double mp = S.max_pilot[row];
                    pv = (mp < pv) ? mp : pv;
                    B.pilots[((size_t)b * N + row) * Tp + t] = (pv > 0.0) ? pv : 0.0;
                }
                if (B.out_v1) B.out_v1[((size_t)b * N + row) * Tp + t] = vq;
            }
        }
    }
    if (B.out_vc) for (int i = tid; i < R * Tp; i += nthreads) B.out_vc[(size_t)b * R * Tp + i] = VC[i];
    if (B.out_mu) for (int i = tid; i < B.S_max; i += nthreads) B.out_mu[(size_t)b * B.S_max + i] = SESS_MU[i];
    if (tid == 0) {
        if (B.out_scal) { B.out_scal[b * 2] = (SCAL[SC_NRESCUE] > 0.f) ? rho_start : rho; B.out_scal[b * 2 + 1] = SCAL[SC_PLEVEL]; }
        if (B.rate_est) B.rate_est[b] = SCAL[SC_RATE_EST];
        B.status[b] = status;
        B.iters[b] = it;
        float* st = B.stats + (size_t)b * ACB_NSTATS;
        st[0] = SCAL[SC_RP]; st[1] = SCAL[SC_RD]; st[2] = SCAL[SC_GAP]; st[3] = SCAL[SC_VIOL]; st[4] = rho; st[5] = cs;
        st[6] = SCAL[SC_NREST]; st[7] = SCAL[SC_USEDAVG];
    }
}


// explicit launch helper used by the per-horizon translation units
template <int Q, int TPW, bool MULTI, bool FAST>
int acb_launch_solve_t(const acb_site* site, const acb_batch* batch, const acb_options* opt, const SolvePhase* ph, int nthreads, size_t smem, cudaStream_t st) {
    auto kern = acb_solve_kernel<Q, TPW, MULTI, FAST>;
    ACB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const SiteDev& d = (TPW == 2) ? site->d2 : site->d;
    SmemLayout L = make_layout(d.N, d.R, d.NG, d.NP, d.nSlots, 32 * Q, batch->S_max, nthreads / 32);
    kern<<<batch->B, nthreads, smem, st>>>(d, *batch, *opt, L, *ph);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}
#define ACB_INSTANTIATE_Q(QQ)                                                                                              \
    int acb_launch_solve_q##QQ(const acb_site* site, const acb_batch* batch, const acb_options* opt, const SolvePhase* ph, \
                               int nthreads, size_t smem, cudaStream_t st, bool multi, int fast) {                         \
        if (multi) return acb_launch_solve_t<QQ, 3, true, false>(site, batch, opt, ph, nthreads, smem, st);                 \
        if (fast == 2) return acb_launch_solve_t<QQ, 2, false, true>(site, batch, opt, ph, nthreads, smem, st);             \
        if (fast) return acb_launch_solve_t<QQ, 3, false, true>(site, batch, opt, ph, nthreads, smem, st);                  \
        return acb_launch_solve_t<QQ, 3, false, false>(site, batch, opt, ph, nthreads, smem, st);                           \
    }
