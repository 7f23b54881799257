// Closed-loop replay on the device (SURVEY.md 8(f) N1): the simulator side of one control step for a fleet of sites.
//
// The reference is driven by acnportal's Simulator, which at every period hands the algorithm the active sessions
// (adacharge/adacharge.py:18-39 get_active_sessions: plugged in, energy still owed) and applies the first-period pilots
// it returns (call pattern adacharge/adacharge.py:135-193; loop shape exercised by tests/test_integration.py:115-118).
// For a fleet replay that loop is two kernels around the solve, with the EV table, the energy delivered so far, the
// previous peak and the per-EV warm-start multipliers resident on the device:
//   acb_fleet_sessions   step t -> the raw [sites][S_max] session tables acb_pack_sessions consumes (+ the EV behind each
//                        slot and its warm-start multiplier)
//   acb_fleet_apply      first-period pilots -> energy delivered, previous peak, per-EV multipliers, step statistics
// The EV table is sorted by (day, site, station), so a site's active sessions come out ordered by EVSE row.
// With acb_fleet.last_solve the step is event-driven, as acnportal's Simulator loop is (this library's reading of it:
// DESIGN.md §8): acb_fleet_sessions decides which sites re-solve (a plug-in or unplug there, max_recompute steps since the
// last solve, or no solve yet) and that decision is acb_solve_batch_masked's solve_mask; every other site keeps its last schedule and
// acb_fleet_apply charges its EVs with the schedule's next column.
// With an acb_fleet_ev (the _ev entry points) the EVs have two-stage batteries and the rampdown estimate of their maximum
// rate (DESIGN.md §8): acb_fleet_apply charges each battery with the current it takes under its pilot and updates the
// estimate, acb_fleet_sessions hands the estimate to acb_preprocess_sessions.  Both kernels are templated on it: the
// instantiations without it are the plain entry points' kernels.
#include "acb_common.cuh"

// The current (A) a two-stage battery takes under pilot p (stepwise Linear2StageBattery without noise, in amperes):
// float64, the stated order of operations, no contraction (the host replay computes the same bits with numpy).
__device__ __forceinline__ double battery_current(double p, double w, double amax, double cap, double charge, double theta) {
    if (p == 0.0) return 0.0;
    const double soc = __ddiv_rn(charge, cap);
    const double lim = soc < theta ? amax : __dmul_rn(__ddiv_rn(__dsub_rn(1.0, soc), __dsub_rn(1.0, theta)), amax);
    double a = (lim < p) ? lim : p;
    if (__dadd_rn(charge, __dmul_rn(a, w)) > cap) a = __ddiv_rn(__dsub_rn(cap, charge), w);
    return (a > 0.0) ? a : 0.0;
}

template <bool EV>
__global__ void acb_fleet_sessions_kernel(acb_fleet F, int t, acb_sessions X, int32_t* sess_ev, float* warm_mu, acb_fleet_ev E) {
    const int b = blockIdx.x, lane = threadIdx.x;  // one warp per site
    const int day = min(t / F.steps_per_day, F.days - 1);
    const int lo = F.day_site_off[(size_t)day * F.n_sites + b], hi = F.day_site_off[(size_t)day * F.n_sites + b + 1];
    const size_t base = (size_t)b * X.S_max;
    int32_t* station = const_cast<int32_t*>(X.station) + base;
    int32_t* arr = const_cast<int32_t*>(X.arrival_offset) + base;
    int32_t* rem_t = const_cast<int32_t*>(X.remaining_time) + base;
    double* dem = const_cast<double*>(X.remaining_demand) + base;
    double* mn = const_cast<double*>(X.min_rate) + base;
    double* mx = const_cast<double*>(X.max_rate) + base;
    int32_t* ev_arr = X.arrival ? const_cast<int32_t*>(X.arrival) + base : nullptr;  // (uninterrupted charging)
    const bool had = F.had[b] != 0;
    int n = 0;
    bool event = false;  // an EV plugs in or unplugs at this site now
    for (int e0 = lo; e0 < hi; e0 += 32) {
        const int e = e0 + lane;
        bool act = false;
        double owed = 0.0;
        if (e < hi) {
            owed = F.ev_req[e] - F.ev_dlv[e];
            const int a = F.ev_arr[e], d = F.ev_dep[e];
            act = a <= t && t < d && owed > 1e-6;  // plugged in and energy still owed
            event |= a == t || d == t;
        }
        const unsigned m = __ballot_sync(0xffffffffu, act);
        const int j = n + __popc(m & ((1u << lane) - 1u));
        if (act && j < X.S_max) {
            station[j] = F.ev_station[e];
            arr[j] = 0;
            rem_t[j] = F.ev_dep[e] - t;
            dem[j] = owed;
            mn[j] = 0.0;
            mx[j] = F.ev_max[e];
            if (ev_arr) ev_arr[j] = F.ev_arr[e];
            sess_ev[base + j] = e;
            warm_mu[base + j] = had ? F.ev_mu[e] : 0.f;
            if (EV && E.ev_ub) E.upper_bound[base + j] = E.ev_ub[e];
        }
        n += __popc(m);
    }
    n = min(n, X.S_max);
    for (int j = n + lane; j < X.S_max; j += 32) {
        station[j] = -1; arr[j] = 0; rem_t[j] = 0; dem[j] = 0.0; mn[j] = 0.0; mx[j] = 0.0;
        if (ev_arr) ev_arr[j] = 0;
        sess_ev[base + j] = -1;
        warm_mu[base + j] = 0.f;
        if (EV && E.ev_ub) E.upper_bound[base + j] = 0.0;
    }
    if (F.last_solve) {
        // the unplug of a previous-day EV at a day boundary (t = d * steps_per_day) is in day d - 1's slice
        const int d = t / F.steps_per_day;
        if (t % F.steps_per_day == 0 && d >= 1 && d <= F.days) {
            const int lo1 = F.day_site_off[(size_t)(d - 1) * F.n_sites + b], hi1 = F.day_site_off[(size_t)(d - 1) * F.n_sites + b + 1];
            for (int e = lo1 + lane; e < hi1; e += 32) event |= F.ev_dep[e] == t;
        }
        event = __any_sync(0xffffffffu, event);
        if (lane == 0) {
            const int last = F.last_solve[b];
            F.recompute[b] = (last < 0 || event || (F.max_recompute > 0 && t - last >= F.max_recompute)) ? 1 : 0;
            F.shift[b] = t - last;
        }
    }
}

template <bool EV>
__global__ void acb_fleet_apply_kernel(SiteDev S, acb_fleet F, int t, double period, const double* pilots, int Tp, const int32_t* n_sessions,
                                       const int32_t* sess_ev, int S_max, const float* out_mu, const int32_t* status, const int32_t* iters,
                                       double* first_out, double* stats, acb_fleet_ev E) {
    const int b = blockIdx.x, lane = threadIdx.x;  // one warp per site
    const int N = S.N;
    const int day = min(t / F.steps_per_day, F.days - 1);
    const int lo = F.day_site_off[(size_t)day * F.n_sites + b], hi = F.day_site_off[(size_t)day * F.n_sites + b + 1];
    // a site that solved now applies column 0 of its schedule, any other site column c = t - last_solve of the schedule its
    // last solve left in `pilots`.  Columns from that solve's horizon to Tp hold 0 (the rate bounds are 0 outside every
    // session window); c >= Tp (a site idle overnight without max_recompute) is 0 and never loaded.  (The horizon is not
    // batch->T: the packer rewrites T and the session tables of every site at every step.)
    const bool solved = !F.last_solve || F.recompute[b] != 0;
    const int c = solved ? 0 : t - F.last_solve[b];
    const bool live = c < Tp;
    const double* p0 = pilots + (size_t)b * N * Tp + (live ? c : 0);  // pilots[b][i][c] = p0[i * Tp]
    auto pil = [&](int i) -> double { return live ? p0[(size_t)i * Tp] : 0.0; };
    double* rates = EV && E.rates ? E.rates + (size_t)b * N : nullptr;  // each EVSE's current, 0 where no EV is plugged in
    if (EV && rates) {
        for (int i = lane; i < N; i += 32) rates[i] = 0.0;
        __syncwarp();
    }
    // the simulator side: the applied pilots charge every EV that is plugged in (also those that owe nothing)
    for (int e = lo + lane; e < hi; e += 32) {
        if (F.ev_arr[e] <= t && t < F.ev_dep[e]) {
            const int i = F.ev_station[e];
            const double w = S.volt[i] * period / 1e3 / 60;  // kWh per A*period
            const double owed = F.ev_req[e] - F.ev_dlv[e];
            if (EV) {
                // the battery takes a <= p; the estimate follows the gap between pilot and current
                const double p = pil(i);
                const double charge = E.ev_cap ? E.ev_charge[e] : 0.0;
                const double a = E.ev_cap ? battery_current(p, w, F.ev_max[e], E.ev_cap[e], charge, E.transition_soc) : p;
                double de = __dmul_rn(a, w);
                de = (owed < de) ? owed : de;
                de = (de > 0.0) ? de : 0.0;
                F.ev_dlv[e] = __dadd_rn(F.ev_dlv[e], de);
                if (E.ev_cap) E.ev_charge[e] = __dadd_rn(charge, de);
                if (E.ev_ub && __dsub_rn(p, a) > E.down_threshold) E.ev_ub[e] = __dadd_rn(a, E.up_increment);
                if (rates) rates[i] = a;
            } else {
                double de = pil(i) * w;
                de = (owed < de) ? owed : de;
                F.ev_dlv[e] += (de > 0.0) ? de : 0.0;
            }
        }
    }
    const int n = n_sessions[b];  // (this step's sessions: those of the solve when the site solved)
    if (solved)
        for (int j = lane; j < n; j += 32) {
            const int e = sess_ev[(size_t)b * S_max + j];
            if (e >= 0) F.ev_mu[e] = out_mu[(size_t)b * S_max + j];
        }
    if (first_out)
        for (int i = lane; i < N; i += 32) first_out[(size_t)b * N + i] = pil(i);
    __syncwarp();  // every lane has read last_solve[b] (and written its EVSEs' currents)
    if (lane == 0) {
        // aggregate applied current, summed in numpy's pairwise order (the host replay takes first.sum(axis=1)); with
        // batteries the currents the EVs took (rates.sum(axis=1))
        auto cur = [&](int i) -> double { return (EV && E.ev_cap) ? rates[i] : pil(i); };
        double tot;
        if (N < 8) {
            tot = 0.0;
            for (int i = 0; i < N; ++i) tot = __dadd_rn(tot, cur(i));
        } else {
            double r[8];
            for (int j = 0; j < 8; ++j) r[j] = cur(j);
            int i;
            for (i = 8; i < N - (N % 8); i += 8)
                for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], cur(i + j));
            tot = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
            for (; i < N; ++i) tot = __dadd_rn(tot, cur(i));
        }
        if (tot > F.prev_peak[b]) F.prev_peak[b] = tot;
        if (solved) {
            F.had[b] = n > 0 ? 1 : 0;
            if (F.last_solve) F.last_solve[b] = t;
            if (stats && n > 0) {
                atomicAdd(stats + 0, 1.0);                                  // site-steps solved
                atomicAdd(stats + 1, (double)iters[b]);                     // iterations
                if (status[b] != ACB_SOLVED) atomicAdd(stats + 2, 1.0);     // not certified
            }
        }
    }
}

// an acb_fleet_ev as the kernels take it: NULL = all NULL (the EV = false instantiations never read it)
static int fleet_ev_check(const acb_fleet_ev* ev, const char* who) {
    if (!ev) return ACB_OK;
    const bool bad = (ev->ev_cap && (!ev->ev_charge || !ev->rates || !(ev->transition_soc > 0.0 && ev->transition_soc < 1.0))) ||
                     (ev->ev_ub && (!ev->upper_bound || !(ev->up_increment > 0.0) || !(ev->down_threshold >= 0.0)));
    if (bad) {
        acb_set_error(std::string(who) + ": ev_cap needs ev_charge, rates and 0 < transition_soc < 1; ev_ub needs upper_bound, "
                      "up_increment > 0 and down_threshold >= 0");
        return ACB_E_INVALID;
    }
    return ACB_OK;
}

extern "C" int acb_fleet_sessions_ev(acb_site* site, const acb_fleet* fleet, const acb_fleet_ev* ev, int t, const acb_sessions* sessions,
                                     int32_t* sess_ev, float* warm_mu, void* stream) {
    if (!site || !fleet || !sessions || !sess_ev || !warm_mu || sessions->B != fleet->n_sites || t < 0) {
        acb_set_error("acb_fleet_sessions: bad arguments (one instance per site)");
        return ACB_E_INVALID;
    }
    if (fleet->last_solve && (!fleet->recompute || !fleet->shift || fleet->max_recompute < 0)) {
        acb_set_error("acb_fleet_sessions: last_solve needs recompute, shift and max_recompute >= 0");
        return ACB_E_INVALID;
    }
    if (fleet_ev_check(ev, "acb_fleet_sessions_ev") != ACB_OK) return ACB_E_INVALID;
    ACB_CUDA(cudaSetDevice(site->device));
    if (ev && ev->ev_ub)
        acb_fleet_sessions_kernel<true><<<fleet->n_sites, 32, 0, (cudaStream_t)stream>>>(*fleet, t, *sessions, sess_ev, warm_mu, *ev);
    else
        acb_fleet_sessions_kernel<false><<<fleet->n_sites, 32, 0, (cudaStream_t)stream>>>(*fleet, t, *sessions, sess_ev, warm_mu, acb_fleet_ev{});
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

extern "C" int acb_fleet_sessions(acb_site* site, const acb_fleet* fleet, int t, const acb_sessions* sessions, int32_t* sess_ev, float* warm_mu,
                                  void* stream) {
    return acb_fleet_sessions_ev(site, fleet, nullptr, t, sessions, sess_ev, warm_mu, stream);
}

extern "C" int acb_fleet_apply_ev(acb_site* site, const acb_fleet* fleet, const acb_fleet_ev* ev, int t, double period, const acb_batch* batch,
                                  const int32_t* sess_ev, double* first_pilots, double* stats, void* stream) {
    if (!site || !fleet || !batch || !batch->pilots || !batch->out_mu || !sess_ev || batch->B != fleet->n_sites) {
        acb_set_error("acb_fleet_apply: bad arguments (the batch needs pilots and out_mu)");
        return ACB_E_INVALID;
    }
    if (fleet->last_solve && !fleet->recompute) {
        acb_set_error("acb_fleet_apply: last_solve needs recompute");
        return ACB_E_INVALID;
    }
    if (fleet_ev_check(ev, "acb_fleet_apply_ev") != ACB_OK) return ACB_E_INVALID;
    ACB_CUDA(cudaSetDevice(site->device));
    const cudaStream_t st = (cudaStream_t)stream;
    if (ev && (ev->ev_cap || ev->ev_ub || ev->rates))
        acb_fleet_apply_kernel<true><<<fleet->n_sites, 32, 0, st>>>(site->d, *fleet, t, period, batch->pilots, batch->Tp, batch->n_sessions, sess_ev,
                                                                    batch->S_max, batch->out_mu, batch->status, batch->iters, first_pilots, stats, *ev);
    else
        acb_fleet_apply_kernel<false><<<fleet->n_sites, 32, 0, st>>>(site->d, *fleet, t, period, batch->pilots, batch->Tp, batch->n_sessions, sess_ev,
                                                                     batch->S_max, batch->out_mu, batch->status, batch->iters, first_pilots, stats,
                                                                     acb_fleet_ev{});
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

extern "C" int acb_fleet_apply(acb_site* site, const acb_fleet* fleet, int t, double period, const acb_batch* batch, const int32_t* sess_ev,
                               double* first_pilots, double* stats, void* stream) {
    return acb_fleet_apply_ev(site, fleet, nullptr, t, period, batch, sess_ev, first_pilots, stats, stream);
}
