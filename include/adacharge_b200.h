/* adacharge_b200 — C ABI of the B200-native MPC solve + postprocessing path.
 *
 * The reference (caltech-netlab/adacharge) is pure Python; it has no FFI of its own.
 * These entry points are what a binding for its hot path would call; each one names
 * the reference function(s) it replaces (paths relative to the reference repo):
 *
 *   acb_site_create / acb_site_destroy
 *       the per-site constants every reference call rebuilds from InfrastructureInfo:
 *       a_j = [v cos(phi); v sin(phi)] rows   adacharge/adaptive_charging_optimization.py:152-164
 *       |v| rows (LINEAR)                       adacharge/adaptive_charging_optimization.py:165-172
 *       voltages -> kW per A                    adacharge/adaptive_charging_optimization.py:336-339
 *       max_pilot / allowable_pilots            adacharge/postprocessing.py:92,114,176
 *   acb_charging_rate_bounds
 *       AdaptiveChargingOptimization.charging_rate_bounds        ...optimization.py:45-79
 *   acb_solve_batch / acb_solve_batch_masked
 *       build_problem + solve (cvxpy canonicalisation + ECOS)    ...optimization.py:220-321
 *       objective library quick_charge ... load_flattening        ...optimization.py:363-408
 *   acb_project_continuous      project_into_continuous_feasible_pilots   postprocessing.py:77-94
 *   acb_project_discrete        project_into_discrete_feasible_pilots     postprocessing.py:97-118
 *   acb_reallocate              index_based_reallocation / diff_based_reallocation
 *                                                                 postprocessing.py:121-258
 *   acb_quantize_pilots         project_into_discrete_feasible_pilots / diff_based_reallocation for a solved batch
 *                                                                 postprocessing.py:97-118, 189-258
 *   acb_constraints_feasible    infrastructure_constraints_feasible       utils.py:5-12
 *   acb_pack_sessions           the host work before the solver: horizon, energy rows, build_objective
 *                                                                 ...optimization.py:114-122, 200-218, 243-245, 363-408
 *   acb_preprocess_sessions / acb_min_rate_admission
 *                               acnportal preprocessing called at      adacharge/adacharge.py:141-150
 *   acb_fleet_sessions / acb_fleet_apply (_ev: with batteries and the rampdown estimate)
 *                               the simulator side of a closed-loop step  adacharge/adacharge.py:18-39, 135-193
 *
 * Conventions: plain C, no exceptions; every function returns 0 on success or a
 * negative ACB_E_* code (acb_last_error() gives text).  Unless a parameter is marked
 * "host", data pointers are DEVICE pointers on the site's device; work is enqueued on
 * the given cudaStream_t (passed as void*) and is asynchronous.  Re-entrant per
 * (site, stream); no global mutable state except the last-error string.
 */
#ifndef ADACHARGE_B200_H
#define ADACHARGE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACB_OK 0
#define ACB_E_INVALID -1   /* bad argument */
#define ACB_E_CUDA -2      /* CUDA runtime error */
#define ACB_E_TOO_LARGE -3 /* instance does not fit the on-chip solve path */

#define ACB_SOC 0
#define ACB_LINEAR 1

/* per-instance solve status written to acb_batch.status */
#define ACB_SOLVED 0
#define ACB_MAX_ITER 1   /* iteration limit hit; residuals are in stats */
#define ACB_INFEASIBLE 2 /* primal infeasibility detected */
#define ACB_NUMERICAL 3  /* non-finite iterate */
#define ACB_INVALID 4    /* the instance breaks a property the caller declared (acb_batch.lb_zero) */

#define ACB_NSTATS 8 /* stats row: r_prim, r_dual, rel. gap, violation, rho, cost_scale, restarts, 1 if the averaged candidate was returned */

typedef struct acb_site acb_site;

/* Site constants (all pointers host).  constraint_matrix is M x N row-major and may be
 * NULL when M == 0.  allow_off (N+1) / allow_vals is a CSR list of each EVSE's sorted
 * allowable pilots (may be NULL if discrete postprocessing is not used).
 * use_peak_row: the solve has a peak_limit (sum_i rates <= P_t).  use_agg_row: the
 * objective uses aggregate power (peak / demand_charge / load_flattening). */
int acb_site_create(acb_site** out, int device, int N, int M, const double* constraint_matrix,
                    const double* phases_deg, const double* limits, const double* voltages,
                    int constraint_type, int use_peak_row, int use_agg_row,
                    const double* max_pilot, const int32_t* allow_off, const double* allow_vals);
void acb_site_destroy(acb_site* site);
/* R = coupling rows, NG = electrically distinct EVSE groups, NP = partial rows. */
int acb_site_dims(const acb_site* site, int* N, int* M, int* R, int* NG, int* NP);
/* Largest padded horizon (multiple of 32) that fits on chip for this site, 0 if none. */
int acb_site_max_horizon(const acb_site* site);

typedef struct acb_options {
    float eps_abs;      /* absolute gap tolerance in cost-scaled units (largest |cost coefficient| = 1) */
    float eps_rel;      /* relative duality-gap tolerance: P - D <= eps_abs + eps_rel * max(|P|, |D|, term_floor * terms), where
                           P is the objective of the returned schedule and D a Lagrangian lower bound (DESIGN.md); negative
                           tolerances never pass: the solve runs its whole iteration budget (status ACB_MAX_ITER) */
    float viol_tol;     /* max relative infrastructure / peak violation of the returned schedule */
    float viol_abs;     /* ... and at most this many amperes over any limit (default 1e-3 A, the bar of the reference's own tests,
                           tests/test_adaptive_charging_optimization.py:82; it is the tighter one for limits above 100 A); 0 = off.
                           stats[3] reports the excess in units of the tighter tolerance (<= viol_tol means both hold) */
    float rho0;         /* initial penalty */
    float kappa;        /* identity-block penalty = kappa * rho */
    float alpha;        /* over-relaxation in (0, 2) */
    int32_t max_iter;
    int32_t check_every; /* convergence-check period in iterations (the first check is at iteration 10) */
    int32_t equality;    /* enforce_energy_equality */
    int32_t adapt_rho;   /* 0 = off, 1 = residual balancing with threshold 5, n > 1 = threshold n/10 */
    int32_t restart;     /* 1 = average the state and restart from the average when its gap halves */
    int32_t avg_every;   /* state is added to the average every avg_every iterations */
    int32_t stall_checks; /* change rho when the best gap has not improved by 10 % over this many checks (0 = never) */
    int32_t max_rescues;  /* at most this many stagnation rescues (1st: rho x3; 2nd, warm-started solves only: restart cold) */
    int32_t path;        /* 0 = on-chip kernel when the instance fits, else the general path; 1 = on-chip only; 2 = general only */
    int32_t stall_exit;  /* with all rescues used: stop (ACB_MAX_ITER, stats[2] = certified gap) after this many checks without a 10 % better gap; 0 = never */
    int32_t dual_refine; /* dual bound uses the best energy-row multipliers given y: 0 = never, 1 = when the gap stalled at the last check, 2 = at every check */
    float term_floor;    /* the gap tolerance is eps_abs + eps_rel * max(|P|, |D|, term_floor * sum of |objective terms|); default 0.05.
                          * 1 = relative to the terms' magnitude (closed-loop replay: the sunk demand charge w*p0 is a constant
                          * that can cancel the energy term), 0 = relative to |P| alone */
    float rho_curv;      /* cold start: rho = max(rho0, rho_curv * Gamma * s_u^2), the curvature of the aggregate quadratic seen
                          * through the scaled aggregate-power row (default 1; 0 = plain rho0) */
    float rate_tol;      /* rate polish (on-chip path): when the objective is strictly convex in the rates (equal_share with a
                          * cost-scaled coefficient >= polish_min_qd) the optimum is unique and the solve additionally runs until
                          * the estimated distance of the schedule to its limit point is <= rate_tol amperes (default 3e-4; 0 = off) */
    float polish_min_qd; /* smallest cost-scaled quadratic coefficient for which the rate polish is applied (default 5e-4: the
                          * reference's 1e-12 tie-breaker does not trigger it, a 1e-3 equal_share weight does) */
    float newton_rel;    /* on-chip hot row pass: between convergence checks a row's energy-row multiplier takes one Newton step per
                          * iteration and is accepted if the remaining energy mismatch is at most newton_rel times the mismatch
                          * before the step (else the exact safeguarded search runs); 0 = always exact; check iterations are exact */
    int32_t phase_iters; /* on-chip path, batches larger than one wave of SMs: first launch stops every instance after this many
                          * iterations, parks the unfinished ones and relaunches them longest-expected-first (default 100;
                          * 0 = one launch) */
} acb_options;

void acb_default_options(acb_options* o);

/* One batch of independent MPC instances on one site.  Horizon arrays are padded to
 * Tp (64, 128, 160 or 288, >= every T[b]); session arrays to S_max.  Objective in
 * minimisation form per instance:
 *   sum_it (alpha_t + k_i beta_t) r_it + qd sum r_it^2 + gamma sum_t (u_t + ext_t)^2
 *   + peak_w * max(max_t u_t, peak_p0) + sum_s sess_quad_s (sess_energy_s - sum_{t in window_s} r_it)^2,   u_t = sum_i k_i r_it  (kW)
 */
typedef struct acb_batch {
    int32_t B, Tp, S_max;
    int32_t multi_session;       /* 1 if any EVSE has more than one session in some instance of the batch */
    int32_t lb_zero;             /* 1 = the caller guarantees that every minimum rate of the batch is 0 (the usual case): the on-chip
                                  * kernel then keeps no lower-bound array and runs its fastest variant; an instance that breaks the
                                  * promise gets status ACB_INVALID.  0 = no promise */
    const int32_t* T;            /* [B] horizon (reference: aco.py:243-245) */
    const int32_t* n_sessions;   /* [B] */
    const int32_t* sess_row;     /* [B*S_max] EVSE index */
    const int32_t* sess_start;   /* [B*S_max] arrival_offset */
    const int32_t* sess_len;     /* [B*S_max] remaining_time */
    const float* sess_energy;    /* [B*S_max] remaining_demand in A*periods */
    const int32_t* sess_rate_off;/* [B*S_max] offset o into min_rates/max_rates; o < 0: constant limits, the pair at index -(o+1) */
    const float* min_rates;      /* flat, per session remaining_time entries */
    const float* max_rates;
    const float* alpha;          /* [B*Tp] */
    const float* beta;           /* [B*Tp] */
    const float* qd;             /* [B] */
    const float* gamma;          /* [B] */
    const float* ext;            /* [B*Tp] or NULL */
    const float* peak_w;         /* [B] */
    const float* peak_p0;        /* [B] */
    const float* peak_limit;     /* [B*Tp] or NULL (required iff use_peak_row) */
    const float* sess_quad;      /* [B*S_max] or NULL: per-session weight cq of the objective term cq (energy_s - sum_window r)^2 in
                                  * (A*periods)^2 (non_completion_penalty with norm 2: coefficient * (kWh per A*period)^2) */
    /* warm start (all optional, NULL = cold).  Layout: v1 [B][N][Tp], vc [B][R][Tp],
     * mu [B][S_max], scal [B][2] = {rho, peak level}. */
    float* work;                 /* scratch [B][N+R][Tp] for the averaged state; NULL disables restarts */
    const float* warm_v1; const float* warm_vc; const float* warm_mu; const float* warm_scal;
    int32_t warm_shift;          /* closed-loop replay: warm_v1 / warm_vc are read this many columns ahead (1 = the previous control
                                  * step's state: its column t + 1 is this problem's column t), zero beyond the horizon */
    const int32_t* warm_had;     /* optional [B]: 0 = this instance starts cold although warm arrays are given (site idle before): no
                                  * warm array is read for it and it is solved bit for bit as without warm arrays (also in
                                  * the choice of stagnation rescues) */
    float* out_v1; float* out_vc; float* out_mu; float* out_scal;
    /* results */
    float* rates;                /* [B][N][Tp] */
    double* pilots;              /* optional [B][N][Tp]: max(min(rates, max_pilot), 0) in float64, i.e. the solve's epilogue also does
                                  * project_into_continuous_feasible_pilots (postprocessing.py:77-94); NULL = skip (quantised pilots:
                                  * acb_quantize_pilots after the solve) */
    float* rate_est;             /* optional [B]: estimated distance (A) of the schedule to its limit point when the rate polish ran, else -1 */
    int32_t* status;             /* [B] */
    int32_t* iters;              /* [B] */
    float* stats;                /* [B][ACB_NSTATS] */
    /* first-period limits (uninterrupted charging, acb_admit_sessions), NULL = none: the pair replaces min_rates /
     * max_rates of session k at its first column sess_start[k] only (the bound there is max(sess_max0, sess_min0)) */
    const float* sess_min0;      /* [B*S_max] */
    const float* sess_max0;      /* [B*S_max] */
} acb_batch;

int acb_solve_batch(acb_site* site, const acb_batch* batch, const acb_options* opt, void* stream);
/* Event-driven recompute (closed-loop replays that re-solve a site only at events or every max_recompute steps):
 * acb_solve_batch with two optional [B] device arrays (acb_solve_batch = both NULL; acb_batch keeps its layout).
 *  solve_mask   NULL = solve every instance.  An instance with solve_mask[b] == 0 is not solved and none of its outputs is
 *               written (rates, pilots, rate_est, status, iters, stats), except that with both warm_* and out_* given its
 *               out_v1 / out_vc / out_mu / out_scal receive an unshifted copy of its warm_v1 / warm_vc / warm_mu / warm_scal
 *               (a replay that alternates two state sets keeps the state of a site it skips).
 *  warm_shifts  NULL = batch->warm_shift for every instance; else instance b reads its warm arrays warm_shifts[b] columns
 *               ahead (zero beyond the horizon). */
int acb_solve_batch_masked(acb_site* site, const acb_batch* batch, const int32_t* solve_mask, const int32_t* warm_shifts,
                           const acb_options* opt, void* stream);

/* ---- packing on the device: raw session tables + interface quantities -> the acb_batch input fields ----
 * What the reference does on the host before every solve (T = max(arrival_offset + remaining_time) aco.py:243-245,
 * energy rows aco.py:114-122, build_objective over the ObjectiveComponent list aco.py:200-218 with the objective
 * library aco.py:363-408), for a whole batch, so that a caller only ships the raw arrays.  float64 inputs, the
 * reference's order of operations, one rounding to float32: bit-identical to the host packer. */
#define ACB_OBJ_QUICK_CHARGE 0
#define ACB_OBJ_EQUAL_SHARE 1
#define ACB_OBJ_TOU_ENERGY_COST 2
#define ACB_OBJ_TOTAL_ENERGY 3
#define ACB_OBJ_PEAK 4              /* only with a negative coefficient (concavity) */
#define ACB_OBJ_DEMAND_CHARGE 5
#define ACB_OBJ_LOAD_FLATTENING 6
#define ACB_OBJ_NON_COMPLETION_L1 7 /* build-defined (absent from the reference): -sum_s |remaining_demand_s - E_s| */
#define ACB_OBJ_NON_COMPLETION_L2 8 /* -sum_s (remaining_demand_s - E_s)^2 (kWh^2); needs batch->sess_quad */
#define ACB_MAX_COMPONENTS 16

typedef struct acb_sessions {      /* [B][S_max] tables, any order within an instance; station < 0 marks an empty slot */
    int32_t B, S_max;
    const int32_t* station;         /* EVSE index (InfrastructureInfo.get_station_index) */
    const int32_t* arrival_offset;  /* SessionInfo.arrival_offset */
    const int32_t* remaining_time;  /* SessionInfo.remaining_time */
    const double* remaining_demand; /* SessionInfo.remaining_demand, kWh */
    const double* min_rate;         /* constant per session (time-varying limits go through the host packer) */
    const double* max_rate;
    const int32_t* arrival;         /* absolute arrival period (SessionInfo.arrival); read by acb_admit_sessions only */
    const double* min_rate0;        /* first-period limits (written by acb_admit_sessions); NULL = min_rate / max_rate */
    const double* max_rate0;
} acb_sessions;

typedef struct acb_objective {     /* the ObjectiveComponent list, in order: sum_c coef[c] * f_kind[c](rates) is maximised */
    int32_t n;
    int32_t kind[ACB_MAX_COMPONENTS];
    double coef[ACB_MAX_COMPONENTS];
    double param[ACB_MAX_COMPONENTS]; /* baseline_peak of peak / demand_charge components, else unused */
    double period;                    /* interface.period, minutes */
    const double* prices;             /* [B][prices_stride >= Tp] $/kWh, interface.get_prices; required by tou_energy_cost */
    int32_t prices_stride;
    const double* prev_peak;          /* [B] A, interface.get_prev_peak; NULL = 0 */
    const double* demand_charge;      /* [B] $/kW, interface.get_demand_charge; NULL = demand_charge_scalar */
    double demand_charge_scalar;
    const double* external_signal;    /* [B][ext_stride >= Tp] kW for load_flattening; NULL = zeros */
    int32_t ext_stride;
    const double* peak_limit;         /* [B][pl_stride]: pl_stride 1 = scalar per instance, else per period; required iff use_peak_row */
    int32_t pl_stride;
} acb_objective;

/* Fills batch->{T, n_sessions, sess_*, min_rates, max_rates ([B*S_max] each), alpha, beta, qd, gamma, ext, peak_w, peak_p0,
 * peak_limit} (device buffers owned by the caller; B, Tp, S_max, multi_session set by the caller).  flags (device, one
 * int32, zeroed by the caller) receives bit 0 if an EVSE holds two sessions although multi_session is 0, bit 1 if a
 * session ends beyond Tp. */
int acb_pack_sessions(acb_site* site, const acb_sessions* sessions, const acb_objective* objective, const acb_batch* batch,
                      int32_t* flags, void* stream);

/* lb/ub [B][N][Tp] from the session tables of a batch (only the session fields, B, Tp,
 * S_max, T and n_sessions are read). */
int acb_charging_rate_bounds(acb_site* site, const acb_batch* batch, float* lb, float* ub, void* stream);

/* Postprocessing, float64 like the reference.  rates_* are [B][N][T] row-major. */
int acb_project_continuous(acb_site* site, const double* rates_in, double* rates_out, int B, int T, void* stream);
int acb_project_discrete(acb_site* site, const double* rates_in, double* rates_out, int B, int T, void* stream);

/* Greedy first-period reallocation.  mode 0 = index based (rates modified in place,
 * order[] given by the caller, peak_limit[b] given); mode 1 = diff based (rates_in is
 * the continuous schedule, rates_out receives the rounded + reallocated schedule, order
 * and peak limit are derived on device).  Per-session arrays are [B][S_max]:
 * sess_row, sess_start (arrival_offset), sess_ramp (interface.remaining_amp_periods),
 * sess_max0 (max_rates[0]); order [B][S_max] holds session indices (mode 0 only). */
int acb_reallocate(acb_site* site, int mode, const double* rates_in, double* rates_out, int B, int T,
                   int S_max, const int32_t* n_sessions, const int32_t* sess_row, const int32_t* sess_start,
                   const double* sess_ramp, const double* sess_max0, const int32_t* order,
                   const double* peak_limit, void* stream);

/* Quantised pilots of a solved batch, in one launch: what AdaptiveSchedulingAlgorithm(quantize=True[, reallocate=True])
 * does after the solve (adacharge/adacharge.py:177-190), for every instance.  Reads batch->rates (float32 [B][N][Tp]),
 * batch->T, batch->n_sessions (an instance without sessions gets all-zero pilots) and, for ACB_PILOTS_REALLOCATE, the raw session tables (after acb_preprocess_sessions, if used); writes
 * pilots [B][N][Tp] float64, bit-identical to the reference applied to rates[:, :T] in float64 and then np.maximum(., 0).
 * Columns >= T[b] are 0.  The reallocation takes the sessions in slot order (empty slots, station < 0, skipped) and their
 * ramp as interface.remaining_amp_periods: remaining_demand * 1000 / voltage * (60 / period), and max_rates[0] from
 * sessions->max_rate0 when given (acb_admit_sessions), else max_rate.  The site needs
 * allowable_pilots; sessions->B must equal batch->B.  acb_quantize_pilots_masked: an instance with solve_mask[b] == 0 (the
 * mask of acb_solve_batch_masked; NULL = none) keeps its pilots. */
#define ACB_PILOTS_DISCRETE 1   /* project_into_discrete_feasible_pilots   postprocessing.py:97-118 */
#define ACB_PILOTS_REALLOCATE 2 /* diff_based_reallocation                 postprocessing.py:189-258 */
int acb_quantize_pilots(acb_site* site, int mode, const acb_sessions* sessions, double period, const acb_batch* batch,
                        double* pilots, void* stream);
int acb_quantize_pilots_masked(acb_site* site, int mode, const acb_sessions* sessions, double period, const acb_batch* batch,
                               const int32_t* solve_mask, double* pilots, void* stream);

/* feasible[b] = 1 iff every SOC line current of column `col` is <= limit + 1e-7. */
int acb_constraints_feasible(acb_site* site, const double* rates, int B, int T, int col, int32_t* feasible, void* stream);

/* Preprocessing before the solve (reference adacharge/adacharge.py:149-150 -> acnportal's
 * apply_minimum_charging_rate): per instance, sessions are offered in the caller's order ([B][S_max] arrays,
 * the reference sorts by arrival); session s asks for try_rate[s] (= min(min_pilot, override)) on EVSE
 * sess_row[s]; admitted[s] = 1 if the network stays feasible (same check as acb_constraints_feasible) together
 * with everything admitted before it, else 0 and that EVSE goes back to 0 A. */
int acb_min_rate_admission(acb_site* site, int B, int S_max, const int32_t* n_sessions, const int32_t* sess_row,
                           const double* try_rate, int32_t* admitted, void* stream);

/* Batched preprocessing of the raw session tables, in place (reference adacharge/adacharge.py:141-146 -> acnportal's
 * enforce_pilot_limit and apply_upper_bound_estimate): max_rate <- min(max_rate, max_pilot[EVSE]) if enforce_pilot_limit;
 * if upper_bound ([B][S_max], device) is given, max_rate <- min(max_rate, upper_bound) and then max_rate <- min_rate where
 * it fell below the minimum rate. */
int acb_preprocess_sessions(acb_site* site, const acb_sessions* sessions, int enforce_pilot_limit, const double* upper_bound, void* stream);

/* Uninterrupted charging (reference adacharge/adacharge.py:149-150 -> acnportal's apply_minimum_charging_rate with
 * override), batched, in place, one block per instance:
 *  1. the raw tables (station, arrival_offset, remaining_time, remaining_demand, min_rate, max_rate, arrival) are
 *     permuted into the stable (arrival, slot) order, empty slots last: the order of the reference's sorted(sessions,
 *     key=arrival), which every later step (the packer's (EVSE, slot) sort, acb_quantize_pilots' tie order) then sees;
 *  2. the sessions are offered try = min(min_pilot[EVSE], override) in that order (acb_min_rate_admission's greedy);
 *  3. min_rate0 / max_rate0 receive the first-period limits: admitted max(try, min_rate) and max(max_rate, that);
 *     refused 0 and 0.
 * skip_unabsorbable = 1 (closed-loop replays): a session whose remaining_amp_periods (remaining_demand * 1000 / voltage
 * * (60 / period)) is below its try rate is not offered the minimum and keeps min_rate / max_rate (the reference would
 * declare the instance infeasible).  min_pilot: [N] device.  sessions needs arrival, min_rate0 and max_rate0. */
int acb_admit_sessions(acb_site* site, const acb_sessions* sessions, const double* min_pilot, double override, double period,
                       int32_t skip_unabsorbable, void* stream);

/* ---- closed-loop replay on the device (the simulator side of a control step for a fleet of sites) ----
 * The loop acnportal's Simulator drives around AdaptiveSchedulingAlgorithm.schedule (adacharge/adacharge.py:18-39 active
 * sessions in, :135-193 pilots out; tests/test_integration.py:115-118), as two kernels around acb_pack_sessions +
 * acb_solve_batch.  All pointers device.  The EV table is sorted by (day, site, station); day_site_off[(day, site)] is
 * the first EV of that site-day (length days * n_sites + 1). */
typedef struct acb_fleet {
    int32_t n_sites, n_ev, days, steps_per_day;
    const int32_t* ev_station;   /* [n_ev] EVSE index */
    const int32_t* ev_arr;       /* [n_ev] arrival period (absolute) */
    const int32_t* ev_dep;       /* [n_ev] departure period (absolute) */
    const double* ev_req;        /* [n_ev] requested energy, kWh */
    const double* ev_max;        /* [n_ev] maximum rate, A */
    double* ev_dlv;              /* [n_ev] state: energy delivered so far, kWh */
    float* ev_mu;                /* [n_ev] state: energy-row multiplier of the EV's last solve (warm start) */
    const int32_t* day_site_off; /* [days * n_sites + 1] */
    double* prev_peak;           /* [n_sites] state: largest aggregate first-period current so far, A (interface.get_prev_peak) */
    int32_t* had;                /* [n_sites] state: 1 if the site had sessions at its last solve */
    /* event-driven recompute (acnportal's Simulator re-solves a site only at a plug-in or unplug there, or when max_recompute
     * periods have passed since its last solve; in between each EVSE gets the next column of the last schedule) */
    int32_t max_recompute;       /* 0 = at events only (max_recompute None); k >= 1 = also at least every k steps */
    int32_t* last_solve;         /* [n_sites] state: step of the site's last solve, -1 = none yet; NULL = every site solves every step */
    int32_t* recompute;          /* [n_sites] written by acb_fleet_sessions (with last_solve): 1 = solve this step (acb_solve_batch_masked's solve_mask) */
    int32_t* shift;              /* [n_sites] written by acb_fleet_sessions (with last_solve): t - last_solve (its warm_shifts) */
} acb_fleet;

/* Step t: the active sessions of every site (plugged in, energy still owed) into the raw tables acb_pack_sessions takes
 * (arrival_offset 0, remaining_time = departure - t, remaining_demand = requested - delivered, arrival = ev_arr if
 * sessions->arrival is given), plus the EV behind each slot (sess_ev [n_sites][S_max], -1 = empty) and its warm-start
 * multiplier (warm_mu [n_sites][S_max]).  Slots are in station order; sess_ev and warm_mu keep that order after
 * acb_admit_sessions, which is the packed order of a single-session site.  With last_solve: recompute[b] = 1 if the site has
 * never solved, an EV plugs in or unplugs there at t (ev_arr == t or ev_dep == t; an EV that has its energy but is still
 * plugged in is no event), or max_recompute > 0 and t - last_solve[b] >= max_recompute; shift[b] = t - last_solve[b]. */
int acb_fleet_sessions(acb_site* site, const acb_fleet* fleet, int t, const acb_sessions* sessions, int32_t* sess_ev, float* warm_mu,
                       void* stream);
/* After the solve of step t: the first-period pilots (batch->pilots) charge every plugged-in EV (delivered energy capped at
 * the request), prev_peak and had are updated, the session multipliers (batch->out_mu) go back to their EVs.  first_pilots
 * (optional [n_sites][N]) receives the applied pilots; stats (optional, 3 doubles) accumulates site-steps solved, iterations,
 * uncertified solves.  With last_solve: a site that solved (recompute[b]) applies column 0 and sets last_solve[b] = t; any
 * other site applies column c = t - last_solve[b] of the pilots its last solve left in batch->pilots (0 for c >= Tp), and
 * only sites that solved update had, their EVs' multipliers and stats. */
int acb_fleet_apply(acb_site* site, const acb_fleet* fleet, int t, double period, const acb_batch* batch, const int32_t* sess_ev,
                    double* first_pilots, double* stats, void* stream);

/* Per-EV batteries and the rampdown max-rate estimate of a fleet replay (acb_fleet keeps its layout: these are a struct of
 * their own, passed to the _ev entry points).  All pointers device.
 * Battery (acnportal's stepwise Linear2StageBattery without noise, in amperes; this library's statement: DESIGN.md §8): a
 * plugged-in EV e under pilot p on an EVSE of w kWh per A*period takes the current
 *   a = 0 if p == 0, else min(p, ev_max) below transition_soc and min(p, (1 - soc) / (1 - transition_soc) * ev_max) from it
 *   on (soc = charge / cap), cut to (cap - charge) / w where charge + a * w would pass cap, and at least 0;
 * it receives de = max(min(a * w, requested - delivered), 0), added to ev_dlv and ev_charge.  float64, no contraction.
 * Rampdown estimate (acnportal's SimpleRampdown): after every applied step where e is plugged in, if p - a > down_threshold
 * then ev_ub[e] = a + up_increment.  acb_fleet_sessions_ev writes each slot's ev_ub into upper_bound, the table
 * acb_preprocess_sessions takes. */
typedef struct acb_fleet_ev {
    const double* ev_cap;        /* [n_ev] battery capacity, kWh; NULL = ideal batteries (a = p) */
    double* ev_charge;           /* [n_ev] state: battery charge, kWh (required with ev_cap) */
    double transition_soc;       /* state of charge where the taper starts, in (0, 1) */
    double* ev_ub;               /* [n_ev] state: estimated maximum rate, A; NULL = no estimate */
    double up_increment;         /* A, > 0 */
    double down_threshold;       /* A, >= 0 */
    double* upper_bound;         /* [n_sites][S_max] written by acb_fleet_sessions_ev (with ev_ub): the slot's ev_ub, 0 in empty slots */
    double* rates;               /* [n_sites][N] written by acb_fleet_apply_ev: each EVSE's current a, 0 where no EV is plugged in;
                                  * required with ev_cap (prev_peak is then the largest sum of these) */
} acb_fleet_ev;

/* acb_fleet_sessions / acb_fleet_apply with batteries and the rampdown estimate; ev NULL = the plain entry points. */
int acb_fleet_sessions_ev(acb_site* site, const acb_fleet* fleet, const acb_fleet_ev* ev, int t, const acb_sessions* sessions,
                          int32_t* sess_ev, float* warm_mu, void* stream);
int acb_fleet_apply_ev(acb_site* site, const acb_fleet* fleet, const acb_fleet_ev* ev, int t, double period, const acb_batch* batch,
                       const int32_t* sess_ev, double* first_pilots, double* stats, void* stream);

const char* acb_last_error(void);
int acb_version(void);

#ifdef __cplusplus
}
#endif
#endif
