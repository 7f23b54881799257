// Device-side packing: raw per-instance session tables + interface quantities -> the acb_batch fields the solve reads.
//
// Replaces, for a whole batch at once, the host work the reference does per call before the solver runs:
//   T = max(arrival_offset + remaining_time)                        adacharge/adaptive_charging_optimization.py:243-245
//   energy rows in A*periods: remaining_demand / (V_i period / 1e3 / 60)                                   ...:114-122
//   build_objective: sum_c coefficient_c * f_c over the ObjectiveComponent list                            ...:200-218
//   quick_charge / equal_share / tou_energy_cost / total_energy / peak / demand_charge / load_flattening   ...:363-408
// so that a caller (the batched API, the closed-loop replay) only moves the raw session arrays to the device.
// All arithmetic is float64 in the reference's order of operations and rounded to float32 once, which makes the result
// bit-identical to the host packer (engine.PackedBatch / pack_objective); tests/test_gpu_batched.py checks that.
// One block per instance; sessions are rank-sorted by (EVSE row, slot) as the solve kernels expect.
#include <algorithm>
#include "acb_common.cuh"

__global__ void acb_pack_kernel(SiteDev S, acb_sessions X, acb_objective O, acb_batch B, int32_t* flags) {
    const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const int Sm = X.S_max, Tp = B.Tp;
    extern __shared__ int sh[];
    int* key = sh;            // [Sm] row * Sm + slot, or INT_MAX for an empty slot
    __shared__ int s_T, s_n, s_dup;
    if (tid == 0) { s_T = 1; s_n = 0; s_dup = 0; }
    __syncthreads();
    const size_t base = (size_t)b * Sm;
    int tmax = 1, cnt = 0;
    for (int s = tid; s < Sm; s += nt) {
        const int row = X.station[base + s];
        const bool ok = row >= 0 && row < S.N;
        key[s] = ok ? row * Sm + s : 0x7fffffff;
        if (ok) { tmax = max(tmax, X.arrival_offset[base + s] + X.remaining_time[base + s]); ++cnt; }
    }
    atomicMax(&s_T, tmax);
    atomicAdd(&s_n, cnt);
    __syncthreads();
    const int T = min(s_T, Tp), n = s_n;
    if (s_T > Tp && tid == 0) atomicOr(flags, 2);  // a session ends beyond the padded horizon
    // rank sort (S_max is small: one EVSE rarely holds more than a few sessions per horizon)
    int32_t* o_row = const_cast<int32_t*>(B.sess_row) + base;
    int32_t* o_start = const_cast<int32_t*>(B.sess_start) + base;
    int32_t* o_len = const_cast<int32_t*>(B.sess_len) + base;
    float* o_en = const_cast<float*>(B.sess_energy) + base;
    int32_t* o_off = const_cast<int32_t*>(B.sess_rate_off) + base;
    float* o_min = const_cast<float*>(B.min_rates) + base;
    float* o_max = const_cast<float*>(B.max_rates) + base;
    float* o_sq = B.sess_quad ? const_cast<float*>(B.sess_quad) + base : nullptr;
    float* o_min0 = B.sess_min0 ? const_cast<float*>(B.sess_min0) + base : nullptr;
    float* o_max0 = B.sess_max0 ? const_cast<float*>(B.sess_max0) + base : nullptr;
    for (int s = tid; s < Sm; s += nt) {
        const int k = key[s];
        if (k == 0x7fffffff) continue;
        int rank = 0, same = 0;
        const int row = k / Sm, klo = row * Sm, khi = klo + Sm;  // keys of the same EVSE row lie in [klo, khi)
        for (int j = 0; j < Sm; ++j) { const int kj = key[j]; rank += (kj < k) ? 1 : 0; same += (kj >= klo && kj < khi) ? 1 : 0; }
        if (same > 1) s_dup = 1;  // (the session itself counts once)
        o_row[rank] = row;
        o_start[rank] = X.arrival_offset[base + s];
        o_len[rank] = X.remaining_time[base + s];
        // aco.py:114-122: remaining_demand / (voltage * period / 1e3 / 60)
        const double w = S.volt[row] * O.period / 1e3 / 60;
        o_en[rank] = (float)(X.remaining_demand[base + s] / w);
        o_off[rank] = -(int)(base + rank + 1);
        o_min[rank] = (float)X.min_rate[base + s];
        o_max[rank] = (float)fmin(X.max_rate[base + s], 3.0e38);
        if (o_min0) {  // first-period limits (uninterrupted charging), rounded like min_rates / max_rates
            o_min0[rank] = (float)(X.min_rate0 ? X.min_rate0[base + s] : X.min_rate[base + s]);
            o_max0[rank] = (float)fmin(X.max_rate0 ? X.max_rate0[base + s] : X.max_rate[base + s], 3.0e38);
        }
        if (o_sq) {  // non_completion_penalty, norm 2: coefficient * (kWh per A*period)^2 per session
            double c2 = 0.0;
            for (int c = 0; c < O.n; ++c)
                if (O.kind[c] == ACB_OBJ_NON_COMPLETION_L2) c2 += O.coef[c] * 1.0;
            o_sq[rank] = (float)(c2 * w * w);
        }
    }
    for (int s = n + tid; s < Sm; s += nt) { o_row[s] = 0; o_start[s] = 0; o_len[s] = 0; o_en[s] = 0.f; o_off[s] = -(int)(base + s + 1); o_min[s] = 0.f; o_max[s] = 0.f; if (o_sq) o_sq[s] = 0.f; if (o_min0) { o_min0[s] = 0.f; o_max0[s] = 0.f; } }
    __syncthreads();
    if (tid == 0) {
        const_cast<int32_t*>(B.T)[b] = T;
        const_cast<int32_t*>(B.n_sessions)[b] = n;
        if (s_dup && !B.multi_session) atomicOr(flags, 1);  // an EVSE holds two sessions but the batch was declared single-session
        // scalar objective pieces, accumulated in component order like pack_objective
        double qd = 0.0, gamma = 0.0, pw = 0.0, p0 = 0.0;
        bool havePeak = false;
        for (int c = 0; c < O.n; ++c) {
            const double coef = O.coef[c];
            switch (O.kind[c]) {
                case ACB_OBJ_EQUAL_SHARE: qd += coef * 1.0; break;
                case ACB_OBJ_LOAD_FLATTENING: gamma += coef * 1.0; break;
                case ACB_OBJ_PEAK:
                case ACB_OBJ_DEMAND_CHARGE: {
                    // aco.py:387-400: max(peak, baseline_peak if > 0, prev_peak * V_0 / 1000)
                    const double prev = (O.prev_peak ? O.prev_peak[b] : 0.0) * S.volt[0] / 1000;
                    const double bl = O.param[c];
                    const double base0 = (bl > 0) ? fmax(prev, bl) : prev;
                    const double w = (O.kind[c] == ACB_OBJ_PEAK) ? coef * -1.0 : coef * (O.demand_charge ? O.demand_charge[b] : O.demand_charge_scalar);
                    pw += w;
                    p0 = havePeak ? fmax(p0, base0) : base0;  // cp.maximum over all terms' baselines
                    havePeak = true;
                    break;
                }
                default: break;
            }
        }
        const_cast<float*>(B.qd)[b] = (float)qd;
        const_cast<float*>(B.gamma)[b] = (float)gamma;
        const_cast<float*>(B.peak_w)[b] = (float)pw;
        const_cast<float*>(B.peak_p0)[b] = (float)p0;
    }
    // per-period cost vectors
    float* o_al = const_cast<float*>(B.alpha) + (size_t)b * Tp;
    float* o_be = const_cast<float*>(B.beta) + (size_t)b * Tp;
    float* o_ext = B.ext ? const_cast<float*>(B.ext) + (size_t)b * Tp : nullptr;
    float* o_pl = B.peak_limit ? const_cast<float*>(B.peak_limit) + (size_t)b * Tp : nullptr;
    for (int t = tid; t < Tp; t += nt) {
        double al = 0.0, be = 0.0, ex = 0.0, gam = 0.0;
        if (t < T) {
            for (int c = 0; c < O.n; ++c) {
                const double coef = O.coef[c];
                switch (O.kind[c]) {
                    case ACB_OBJ_QUICK_CHARGE: al += coef * -((double)(T - t) / (double)T); break;           // aco.py:363-371
                    case ACB_OBJ_TOU_ENERGY_COST: be += coef * (O.prices[(size_t)b * O.prices_stride + t] * (O.period / 60)); break;  // aco.py:378-380
                    case ACB_OBJ_TOTAL_ENERGY:                                                                  // aco.py:383-384
                    case ACB_OBJ_NON_COMPLETION_L1: be += coef * -(O.period / 60); break;
                    case ACB_OBJ_LOAD_FLATTENING: {                                                            // aco.py:403-408
                        const double g = coef * 1.0;
                        gam += g;
                        ex += g * (O.external_signal ? O.external_signal[(size_t)b * O.ext_stride + t] : 0.0);
                        break;
                    }
                    default: break;
                }
            }
        }
        o_al[t] = (float)al;
        o_be[t] = (float)be;
        if (o_ext) o_ext[t] = (gam > 0.0) ? (float)(ex / gam) : 0.f;
        if (o_pl) o_pl[t] = (t < T && O.peak_limit) ? (float)O.peak_limit[(size_t)b * O.pl_stride + (O.pl_stride > 1 ? t : 0)] : 3.0e38f;
    }
}

extern "C" int acb_pack_sessions(acb_site* site, const acb_sessions* sessions, const acb_objective* objective, const acb_batch* batch,
                                 int32_t* flags, void* stream) {
    if (!site || !sessions || !objective || !batch || !flags || sessions->S_max <= 0 || sessions->S_max != batch->S_max || sessions->B != batch->B) {
        acb_set_error("acb_pack_sessions: bad arguments (sessions and batch must agree on B and S_max)");
        return ACB_E_INVALID;
    }
    if (objective->n < 0 || objective->n > ACB_MAX_COMPONENTS) { acb_set_error("acb_pack_sessions: too many objective components"); return ACB_E_INVALID; }
    for (int c = 0; c < objective->n; ++c) {
        const int k = objective->kind[c];
        if (k == ACB_OBJ_TOU_ENERGY_COST && !objective->prices) { acb_set_error("acb_pack_sessions: tou_energy_cost needs prices"); return ACB_E_INVALID; }
        if (k == ACB_OBJ_EQUAL_SHARE || k == ACB_OBJ_LOAD_FLATTENING) {
            if (objective->coef[c] < 0) { acb_set_error("acb_pack_sessions: equal_share / load_flattening with a negative coefficient is not concave"); return ACB_E_INVALID; }
        }
        if (k == ACB_OBJ_NON_COMPLETION_L2 && (!batch->sess_quad || objective->coef[c] < 0)) {
            acb_set_error("acb_pack_sessions: non_completion_penalty (norm 2) needs batch.sess_quad and a non-negative coefficient");
            return ACB_E_INVALID;
        }
        if ((k == ACB_OBJ_PEAK && objective->coef[c] > 0) || (k == ACB_OBJ_DEMAND_CHARGE && objective->coef[c] < 0)) {
            acb_set_error("acb_pack_sessions: peak / demand_charge with this sign is not concave (cvxpy would raise a DCP error)");
            return ACB_E_INVALID;
        }
    }
    if (site->d.has_pl && !batch->peak_limit) { acb_set_error("acb_pack_sessions: the site has a peak-limit row but batch.peak_limit is NULL"); return ACB_E_INVALID; }
    ACB_CUDA(cudaSetDevice(site->device));
    const size_t smem = (size_t)sessions->S_max * sizeof(int);
    if (smem > 48 * 1024) { acb_set_error("acb_pack_sessions: S_max too large"); return ACB_E_TOO_LARGE; }
    // the rank sort is S_max^2 comparisons per instance: one thread per session slot up to 1024 (a 1000-session instance took
    // 0.8 ms on 128 threads, 7 % of a config-5 step)
    const int threads = std::min(1024, std::max(128, (sessions->S_max + 31) / 32 * 32));
    acb_pack_kernel<<<batch->B, threads, smem, (cudaStream_t)stream>>>(site->d, *sessions, *objective, *batch, flags);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

// ---- batched preprocessing of the raw session tables (SURVEY.md 8(f) N2) ----------------------------------------
// What AdaptiveSchedulingAlgorithm.schedule applies to the sessions before every solve (reference
// adacharge/adacharge.py:141-146, acnportal's helpers):
//   enforce_pilot_limit          max_rate <- min(max_rate, max_pilot of the session's EVSE)
//   apply_upper_bound_estimate   max_rate <- min(max_rate, estimator's upper bound), then max_rate <- min_rate
//                                where it fell below the minimum rate
// element-wise over the [B][S_max] tables, in place.
__global__ void acb_preprocess_kernel(SiteDev S, acb_sessions X, int do_pilot_limit, const double* upper) {
    const size_t n = (size_t)X.B * X.S_max;
    double* mx = const_cast<double*>(X.max_rate);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int row = X.station[i];
        if (row < 0 || row >= S.N) continue;
        double m = mx[i];
        if (do_pilot_limit) { const double p = S.max_pilot[row]; m = (p < m) ? p : m; }  // np.minimum
        if (upper) {
            const double u = upper[i];
            m = (u < m) ? u : m;
            const double lo = X.min_rate[i];
            if (m < lo) m = lo;  // reconcile: the minimum rate wins
        }
        mx[i] = m;
    }
}

extern "C" int acb_preprocess_sessions(acb_site* site, const acb_sessions* sessions, int enforce_pilot_limit, const double* upper_bound, void* stream) {
    if (!site || !sessions || sessions->B <= 0 || sessions->S_max <= 0 || !sessions->station || !sessions->max_rate || !sessions->min_rate) {
        acb_set_error("acb_preprocess_sessions: bad arguments");
        return ACB_E_INVALID;
    }
    ACB_CUDA(cudaSetDevice(site->device));
    const size_t n = (size_t)sessions->B * sessions->S_max;
    const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 8);
    acb_preprocess_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(site->d, *sessions, enforce_pilot_limit, upper_bound);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}
