// Postprocessing kernels, float64 like the reference (numpy defaults), written so that
// the results are bit-identical to reference adacharge/postprocessing.py given the same
// continuous schedule:
//   acb_project_continuous  <- project_into_continuous_feasible_pilots  pp.py:77-94
//   acb_project_discrete    <- project_into_discrete_feasible_pilots    pp.py:97-118
//                              (floor_to_set pp.py:10-31, eps = 0.05)
//   acb_reallocate          <- index_based_reallocation pp.py:121-186 (mode 0),
//                              diff_based_reallocation  pp.py:189-258 (mode 1)
//                              (increment_in_set pp.py:58-74)
//   acb_quantize_pilots     <- the same two projections for a solved batch (acb_batch.rates, float32), sessions
//                              from the raw tables; both reallocation modes share one greedy (realloc_greedy)
//   acb_constraints_feasible<- infrastructure_constraints_feasible      utils.py:5-12
// Arithmetic notes: sums that the reference takes with np.sum follow numpy's pairwise
// summation order; products/sums are issued without FMA contraction.
#include <algorithm>
#include "acb_common.cuh"

__device__ __forceinline__ int bisect_left(const double* a, int n, double x) {
    int lo = 0, hi = n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (a[mid] < x) lo = mid + 1; else hi = mid; }
    return lo;
}
__device__ __forceinline__ int bisect_right(const double* a, int n, double x) {
    int lo = 0, hi = n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (x < a[mid]) hi = mid; else lo = mid + 1; }
    return lo;
}
__device__ __forceinline__ double floor_to_set(double x, const double* set, int n, double eps) {
    int pos = bisect_left(set, n, __dadd_rn(x, eps));
    if (pos < n && x == set[pos]) return x;
    if (pos == 0) return set[0];
    if (pos == n) return set[n - 1];
    return set[pos - 1];
}
__device__ __forceinline__ double increment_in_set(double x, const double* set, int n) {
    int pos = bisect_right(set, n, x);
    if (pos == 0) return set[0];
    if (pos == n) return set[n - 1];
    return set[pos];
}

__global__ void k_project_continuous(SiteDev S, const double* in, double* out, int B, int T) {
    size_t total = (size_t)B * S.N * T;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        int row = (int)((i / T) % S.N);
        double v = in[i];
        double mp = S.max_pilot[row];
        v = (mp < v) ? mp : v;          // np.minimum
        out[i] = (v > 0.0) ? v : 0.0;   // np.maximum(., 0)
    }
}

__global__ void k_project_discrete(SiteDev S, const double* in, double* out, int B, int T) {
    size_t total = (size_t)B * S.N * T;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        int row = (int)((i / T) % S.N);
        int o = S.allow_off[row], n = S.allow_off[row + 1] - o;
        double v = floor_to_set(in[i], S.allow_vals + o, n, 0.05);
        out[i] = (v > 0.0) ? v : 0.0;
    }
}

// numpy's pairwise sum of n float64 values (numpy/core/src/umath/loops_utils.h.src
// pairwise_sum: blocks of 128, 8 accumulators) so that `np.sum(col) <= peak_limit`
// compares the same number.  np_pairwise_leaf is one block (n <= 128) of that recursion,
// with a[sub] read as sub_val (sub < 0: none).
__device__ double np_pairwise_leaf(const double* a, int n, int sub, double sub_val) {
#define ACB_AT(k) ((k) == sub ? sub_val : a[k])
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, ACB_AT(i));
        return res;
    }
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = ACB_AT(j);
    int i;
    for (i = 8; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], ACB_AT(i + j));
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, ACB_AT(i));
    return res;
#undef ACB_AT
}

__device__ double np_pairwise_sum(const double* a, int n) {
    if (n <= 128) return np_pairwise_leaf(a, n, -1, 0.0);
    int n2 = n / 2;
    n2 -= n2 % 8;
    return __dadd_rn(np_pairwise_sum(a, n2), np_pairwise_sum(a + n2, n - n2));
}

// The same sum over a[o, o + n) with the leaf sums cached in leaf[] (leaf[q] = sum of the leaf block that starts at q).
// fill: compute and store every leaf sum.  Otherwise a[i] reads as v: only the leaf holding i is summed again (its sum
// and start go to *leaf_v / *leaf_o, the cache is left alone) and the others come from the cache, so a trial that
// changes one entry costs one block of <= 128 additions plus the path up the tree.
__device__ double np_pairwise_cached(const double* a, int o, int n, double* leaf, bool fill, int i, double v, double* leaf_v,
                                     int* leaf_o) {
    if (n <= 128) {
        if (fill) return leaf[o] = np_pairwise_leaf(a + o, n, -1, 0.0);
        if (i < o || i >= o + n) return leaf[o];
        *leaf_o = o;
        return *leaf_v = np_pairwise_leaf(a + o, n, i - o, v);
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    const double lo = np_pairwise_cached(a, o, n2, leaf, fill, i, v, leaf_v, leaf_o);
    return __dadd_rn(lo, np_pairwise_cached(a, o + n2, n - n2, leaf, fill, i, v, leaf_v, leaf_o));
}

// all SOC line currents of `col` (length N) within limit + 1e-7; warp-cooperative,
// each lane takes constraint rows j = lane, lane+32, ...
__device__ bool warp_feasible(const SiteDev& S, const double* col, int lane) {
    bool ok = true;
    for (int j = lane; j < S.M; j += 32) {
        double x = 0.0, y = 0.0;
        const double* ac = S.a_cos + (size_t)j * S.N;
        const double* as = S.a_sin + (size_t)j * S.N;
        for (int i = 0; i < S.N; ++i) {
            x = __dadd_rn(x, __dmul_rn(ac[i], col[i]));
            y = __dadd_rn(y, __dmul_rn(as[i], col[i]));
        }
        double cur = __dsqrt_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
        if (!(cur <= __dadd_rn(S.limits[j], 1e-7))) ok = false;
    }
    return __all_sync(0xffffffffu, ok);
}

// Row j of the SOC constraints for the column `col` with col[i] read as v (i < 0: none): the test of
// infrastructure_constraints_feasible (utils.py:5-12), sqrt(x^2 + y^2) <= limit + 1e-7.  The sums run over the row's
// nonzero entries only, in ascending column order, and give the same bits as warp_feasible's dense sums over all N
// columns: a zero coefficient times a finite rate is +-0; adding +-0 to a nonzero partial sum leaves it unchanged, and
// adding it to a zero partial sum can at most flip that zero's sign, which the next nonzero term or the squaring erases.
__device__ bool row_within_limit(const SiteDev& S, int j, const double* col, int i, double v) {
    double x = 0.0, y = 0.0;
    for (int p = S.row_col_off[j]; p < S.row_col_off[j + 1]; ++p) {
        const int q = S.row_cols[p];
        const double r = (q == i) ? v : col[q];
        x = __dadd_rn(x, __dmul_rn(S.row_cos[p], r));
        y = __dadd_rn(y, __dmul_rn(S.row_sin[p], r));
    }
    const double cur = __dsqrt_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
    return cur <= __dadd_rn(S.limits[j], 1e-7);
}

// Shared memory of the reallocation greedy of one instance.
struct GreedySmem {
    double* col;   // [N] rounded first column in, reallocated first column out
    double* init;  // [N] continuous first column (diff based)
    double* ub;    // [N] first-period cap of each EVSE
    double* leaf;  // [N] leaf sums of the pairwise sum of col
    double* key;   // [S_max] rounding loss of each candidate (diff based)
    int* cand;     // [S_max] sessions in the caller's order whose EVSE takes part
    int* order;    // [S_max] EVSE of each candidate, in greedy order
    int* active;   // [N]
    int* rowok;    // [M] row j of col is within its limit
};

static __host__ __device__ size_t greedy_smem_bytes(int N, int M, int S_max) {
    return (size_t)(4 * N + S_max) * sizeof(double) + (size_t)(3 * S_max + N + M) * sizeof(int);
}

__device__ GreedySmem greedy_carve(unsigned char* p, int N, int M, int S_max) {
    GreedySmem g;
    double* d = reinterpret_cast<double*>(p);
    g.col = d; g.init = d + N; g.ub = d + 2 * N; g.leaf = d + 3 * N; g.key = d + 4 * N;
    int* q = reinterpret_cast<int*>(g.key + S_max);
    g.cand = q; g.order = q + S_max; g.active = q + 2 * S_max; g.rowok = q + 2 * S_max + N;
    (void)M;
    return g;
}

// Greedy first-period reallocation of one instance (index based pp.py:152-185, mode 0; diff based pp.py:209-257,
// mode 1), run by one full warp.  Sessions s < nS in list order: s_row (EVSE), s_start (arrival_offset), s_ramp
// (interface.remaining_amp_periods), s_max0 (max_rates[0]); order_in (mode 0) lists session indices in the caller's
// sort order, peak_limit is the mode-0 limit.  On entry g.col holds the rounded first column and g.init (mode 1) the
// continuous one; on exit g.col holds the reallocated column.
__device__ void realloc_greedy(const SiteDev& S, int mode, int nS, const int32_t* s_row, const int32_t* s_start, const double* s_ramp,
                               const double* s_max0, const int32_t* order_in, double peak_limit, const GreedySmem& g, int lane) {
    const unsigned FULL = 0xffffffffu;
    const int N = S.N;
    for (int i = lane; i < N; i += 32) { g.active[i] = 0; g.ub[i] = 0.0; }
    __syncwarp();
    int nC = 0;
    if (lane == 0) {
        if (mode == 1) peak_limit = np_pairwise_sum(g.init, N);  // pp.py:209-211
        for (int s = 0; s < nS; ++s) {
            if (s_start[s] != 0) continue;  // pp.py:154-164 / 226-236 (a later session of the same EVSE wins)
            const int i = s_row[s];
            double u = s_ramp[s];
            if (s_max0[s] < u) u = s_max0[s];
            if (S.max_pilot[i] < u) u = S.max_pilot[i];
            g.active[i] = 1;
            g.ub[i] = u;
        }
        // only sessions whose EVSE starts active take part: every pass of the round robin skips the others, so dropping
        // them (keeping the order) leaves the sequence of trials unchanged
        for (int k = 0; k < nS; ++k) {
            const int s = (mode == 1) ? k : order_in[k];
            const int i = s_row[s];
            if (!g.active[i]) continue;
            g.cand[nC] = s;
            if (mode == 1) g.key[nC] = -(g.init[i] - g.col[i]);  // pp.py:214-216
            ++nC;
        }
    }
    nC = __shfl_sync(FULL, nC, 0);
    peak_limit = __shfl_sync(FULL, peak_limit, 0);
    __syncwarp();
    // mode 1: stable sort by rounding loss (Python sorted() is stable), as a rank sort
    for (int c = lane; c < nC; c += 32) {
        int r = c;
        if (mode == 1) {
            const double m = g.key[c];
            r = 0;
            for (int d = 0; d < nC; ++d) r += (g.key[d] < m || (g.key[d] == m && d < c)) ? 1 : 0;
        }
        g.order[r] = s_row[g.cand[c]];
    }
    // state of the starting column: which rows are within their limit, leaf sums of its pairwise sum
    int bad = 0, n_active = 0;
    for (int j = lane; j < S.M; j += 32) {
        const bool ok = row_within_limit(S, j, g.col, -1, 0.0);
        g.rowok[j] = ok ? 1 : 0;
        bad += ok ? 0 : 1;
    }
    int n_bad = __reduce_add_sync(FULL, bad);
    for (int i = lane; i < N; i += 32) n_active += g.active[i];
    n_active = __reduce_add_sync(FULL, n_active);
    if (lane == 0) np_pairwise_cached(g.col, 0, N, g.leaf, true, -1, 0.0, nullptr, nullptr);
    __syncwarp();
    // for i in cycle(sorted_indexes)
    int ptr = 0, skipped = 0;
    while (nC > 0 && n_active > 0) {
        const int i = g.order[ptr];
        ptr = (ptr + 1 == nC) ? 0 : ptr + 1;
        if (!g.active[i]) {
            if (++skipped >= nC) break;
            continue;
        }
        skipped = 0;
        const double cur = g.col[i], u = g.ub[i];
        bool accept = false;
        if (!(cur >= u)) {
            const int o = S.allow_off[i];
            const double nv = increment_in_set(cur, S.allow_vals + o, S.allow_off[i + 1] - o);
            // accept is the AND of four tests (pp.py:175-181): the O(1) ones first, then the peak, then the network.
            // nv == cur cannot make progress (the reference would spin forever here): stop this EVSE
            accept = (nv <= u) && (nv != cur);
            double leaf_v = 0.0;
            int leaf_o = 0;
            if (accept) {
                double sum = 0.0;
                if (lane == 0) sum = np_pairwise_cached(g.col, 0, N, g.leaf, false, i, nv, &leaf_v, &leaf_o);
                accept = __shfl_sync(FULL, sum, 0) <= peak_limit;
            }
            if (accept) {
                // the rows without EVSE i keep their state: only the rows of i are summed again
                bool ok = true;
                int was_bad = 0;
                for (int k = S.evse_row_off[i] + lane; k < S.evse_row_off[i + 1]; k += 32) {
                    const int j = S.evse_rows[k];
                    ok = row_within_limit(S, j, g.col, i, nv) && ok;
                    was_bad += g.rowok[j] ? 0 : 1;
                }
                accept = __all_sync(FULL, ok) && __reduce_add_sync(FULL, was_bad) == n_bad;
            }
            if (accept) {
                if (lane == 0) { g.col[i] = nv; g.leaf[leaf_o] = leaf_v; }
                if (n_bad > 0) {  // the accepted column is feasible: every row is within its limit from now on
                    for (int j = lane; j < S.M; j += 32) g.rowok[j] = 1;
                    n_bad = 0;
                }
            }
        }
        if (!accept) { if (lane == 0) g.active[i] = 0; --n_active; }
        __syncwarp();
    }
}

// one warp per instance
__global__ void k_reallocate(SiteDev S, int mode, const double* rates_in, double* rates, int B, int T, int S_max,
                             const int32_t* n_sessions, const int32_t* sess_row, const int32_t* sess_start,
                             const double* sess_ramp, const double* sess_max0, const int32_t* order_in,
                             const double* peak_limit_in) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int b = blockIdx.x, lane = threadIdx.x, N = S.N;
    const GreedySmem g = greedy_carve(smraw, N, S.M, S_max);
    double* R = rates + (size_t)b * N * T;
    const double* Rin = rates_in + (size_t)b * N * T;
    // init_rates / peak limit come from the *continuous* schedule (pp.py:209-211)
    for (int i = lane; i < N; i += 32) { g.init[i] = Rin[(size_t)i * T]; g.col[i] = R[(size_t)i * T]; }
    __syncwarp();
    const size_t k = (size_t)b * S_max;
    realloc_greedy(S, mode, n_sessions[b], sess_row + k, sess_start + k, sess_ramp + k, sess_max0 + k,
                   mode == 0 ? order_in + k : nullptr, mode == 0 ? peak_limit_in[b] : 0.0, g, lane);
    __syncwarp();
    for (int i = lane; i < N; i += 32) R[(size_t)i * T] = g.col[i];
}

// acb_quantize_pilots: one block per instance.  The projection (pp.py:97-118, then np.maximum(., 0)) covers the live
// columns t < T[b]; padded columns are written as 0 without projecting them (a set without 0 would turn them into
// set[0]).  An instance without sessions has nothing to schedule (the reference's schedule() returns no pilots) and
// is written as 0 as a whole, although the packer gives it a one-period horizon.  With the reallocation, warp 0 owns column 0: it lays out the sessions, runs the greedy and writes the
// column, while the other warps project the rest.
#define ACB_QP_THREADS 256
__global__ void __launch_bounds__(ACB_QP_THREADS) k_quantize_pilots(SiteDev S, int mode, acb_sessions X, double period, const float* rates,
                                                                    const int32_t* Tv, const int32_t* n_sessions, int Tp, double* pilots) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int b = blockIdx.x, tid = threadIdx.x, N = S.N, T = (n_sessions[b] > 0) ? Tv[b] : 0;
    const float* Rb = rates + (size_t)b * N * Tp;
    double* Pb = pilots + (size_t)b * N * Tp;
    const bool realloc = (mode == ACB_PILOTS_REALLOCATE);
    const int first = realloc ? 32 : 0;
    if (tid >= first) {
        for (int idx = tid - first; idx < N * Tp; idx += blockDim.x - first) {
            const int i = idx / Tp, t = idx - i * Tp;
            if (realloc && t == 0) continue;
            double v = 0.0;
            if (t < T) {
                const int o = S.allow_off[i];
                v = floor_to_set((double)Rb[idx], S.allow_vals + o, S.allow_off[i + 1] - o, 0.05);
                v = (v > 0.0) ? v : 0.0;
            }
            Pb[idx] = v;
        }
        return;
    }
    // warp 0, reallocation: the session arrays in the caller's slot order, empty slots skipped
    const unsigned FULL = 0xffffffffu;
    const int lane = tid, Sm = X.S_max;
    const GreedySmem g = greedy_carve(smraw, N, S.M, Sm);
    double* s_ramp = reinterpret_cast<double*>(smraw + ((greedy_smem_bytes(N, S.M, Sm) + 7) & ~(size_t)7));
    double* s_max0 = s_ramp + Sm;
    int32_t* s_row = reinterpret_cast<int32_t*>(s_max0 + Sm);
    int32_t* s_start = s_row + Sm;
    const size_t base = (size_t)b * Sm;
    const double per_period = __ddiv_rn(60.0, period);
    int n = 0;
    for (int s0 = 0; s0 < Sm; s0 += 32) {
        const int s = s0 + lane;
        const int row = (s < Sm) ? X.station[base + s] : -1;
        const bool ok = row >= 0 && row < N;
        const unsigned m = __ballot_sync(FULL, ok);
        if (ok) {
            const int j = n + __popc(m & ((1u << lane) - 1u));
            s_row[j] = row;
            s_start[j] = X.arrival_offset[base + s];
            // interface.remaining_amp_periods: remaining_demand * 1000 / voltage * (60 / period), in this order
            s_ramp[j] = __dmul_rn(__ddiv_rn(__dmul_rn(X.remaining_demand[base + s], 1000.0), S.volt[row]), per_period);
            s_max0[j] = X.max_rate[base + s];
        }
        n += __popc(m);
    }
    for (int i = lane; i < N; i += 32) {
        const double r = (double)Rb[(size_t)i * Tp];
        const int o = S.allow_off[i];
        const double v = floor_to_set(r, S.allow_vals + o, S.allow_off[i + 1] - o, 0.05);
        g.init[i] = r;
        g.col[i] = (v > 0.0) ? v : 0.0;
    }
    __syncwarp();
    if (T > 0) realloc_greedy(S, 1, n, s_row, s_start, s_ramp, s_max0, nullptr, 0.0, g, lane);
    __syncwarp();
    for (int i = lane; i < N; i += 32) {
        const double v = g.col[i];
        Pb[(size_t)i * Tp] = (T > 0 && v > 0.0) ? v : 0.0;
    }
}

static size_t quantize_smem_bytes(const SiteDev& d, int S_max) {
    return ((greedy_smem_bytes(d.N, d.M, S_max) + 7) & ~(size_t)7) + (size_t)S_max * (2 * sizeof(double) + 2 * sizeof(int32_t));
}

__global__ void k_feasible(SiteDev S, const double* rates, int B, int T, int colidx, int32_t* feasible) {
    extern __shared__ __align__(16) unsigned char smraw[];
    double* col = reinterpret_cast<double*>(smraw);
    const int b = blockIdx.x, lane = threadIdx.x;
    for (int i = lane; i < S.N; i += 32) col[i] = rates[((size_t)b * S.N + i) * T + colidx];
    __syncwarp();
    bool ok = warp_feasible(S, col, lane);
    if (lane == 0) feasible[b] = ok ? 1 : 0;
}

// Preprocessing greedy of apply_minimum_charging_rate (acnportal, called at adacharge.py:149-150): sessions are
// offered in the caller's order; a session keeps its minimum rate if the network stays feasible with everything
// admitted before it.  One warp per instance.
__global__ void k_min_rate_admission(SiteDev S, int B, int S_max, const int32_t* n_sessions, const int32_t* sess_row,
                                     const double* try_rate, int32_t* admitted) {
    extern __shared__ __align__(16) unsigned char smraw[];
    double* col = reinterpret_cast<double*>(smraw);
    const int b = blockIdx.x, lane = threadIdx.x;
    for (int i = lane; i < S.N; i += 32) col[i] = 0.0;
    __syncwarp();
    const int nS = n_sessions[b];
    for (int s = 0; s < nS; ++s) {
        const size_t k = (size_t)b * S_max + s;
        const int i = sess_row[k];
        if (lane == 0) col[i] = try_rate[k];
        __syncwarp();
        const bool ok = warp_feasible(S, col, lane);
        if (lane == 0) {
            if (!ok) col[i] = 0.0;
            admitted[k] = ok ? 1 : 0;
        }
        __syncwarp();
    }
}

#define ACB_MAX_SMEM 232448  // opt-in shared memory per block (sm_100)
static int grid_for(size_t total) { return (int)std::min<size_t>((total + 255) / 256, 148 * 16); }

extern "C" int acb_project_continuous(acb_site* site, const double* in, double* out, int B, int T, void* stream) {
    if (!site || !in || !out || B <= 0 || T <= 0) { acb_set_error("acb_project_continuous: bad arguments"); return ACB_E_INVALID; }
    ACB_CUDA(cudaSetDevice(site->device));
    k_project_continuous<<<grid_for((size_t)B * site->d.N * T), 256, 0, (cudaStream_t)stream>>>(site->d, in, out, B, T);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

extern "C" int acb_project_discrete(acb_site* site, const double* in, double* out, int B, int T, void* stream) {
    if (!site || !in || !out || B <= 0 || T <= 0) { acb_set_error("acb_project_discrete: bad arguments"); return ACB_E_INVALID; }
    if (site->d.nAllow == 0) { acb_set_error("acb_project_discrete: site has no allowable_pilots"); return ACB_E_INVALID; }
    ACB_CUDA(cudaSetDevice(site->device));
    k_project_discrete<<<grid_for((size_t)B * site->d.N * T), 256, 0, (cudaStream_t)stream>>>(site->d, in, out, B, T);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

extern "C" int acb_reallocate(acb_site* site, int mode, const double* rates_in, double* rates_out, int B, int T,
                              int S_max, const int32_t* n_sessions, const int32_t* sess_row, const int32_t* sess_start,
                              const double* sess_ramp, const double* sess_max0, const int32_t* order,
                              const double* peak_limit, void* stream) {
    if (!site || !rates_in || !rates_out || B <= 0 || T <= 0 || S_max <= 0 || (mode != 0 && mode != 1) ||
        (mode == 0 && (!order || !peak_limit))) {
        acb_set_error("acb_reallocate: bad arguments");
        return ACB_E_INVALID;
    }
    if (site->d.nAllow == 0) { acb_set_error("acb_reallocate: site has no allowable_pilots"); return ACB_E_INVALID; }
    ACB_CUDA(cudaSetDevice(site->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t total = (size_t)B * site->d.N * T;
    if (mode == 1) {
        k_project_discrete<<<grid_for(total), 256, 0, st>>>(site->d, rates_in, rates_out, B, T);
        ACB_CUDA(cudaGetLastError());
    } else if (rates_in != rates_out) {
        ACB_CUDA(cudaMemcpyAsync(rates_out, rates_in, total * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    const size_t smem = greedy_smem_bytes(site->d.N, site->d.M, S_max);
    if (smem > 48 * 1024) ACB_CUDA(cudaFuncSetAttribute(k_reallocate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_reallocate<<<B, 32, smem, st>>>(site->d, mode, rates_in, rates_out, B, T, S_max, n_sessions, sess_row, sess_start,
                                      sess_ramp, sess_max0, order, peak_limit);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

extern "C" int acb_quantize_pilots(acb_site* site, int mode, const acb_sessions* sessions, double period, const acb_batch* batch,
                                   double* pilots, void* stream) {
    if (!site || !sessions || !batch || !pilots || !batch->rates || !batch->T || !batch->n_sessions || batch->B <= 0 || batch->Tp <= 0 ||
        (mode != ACB_PILOTS_DISCRETE && mode != ACB_PILOTS_REALLOCATE) || sessions->B != batch->B) {
        acb_set_error("acb_quantize_pilots: bad arguments");
        return ACB_E_INVALID;
    }
    if (mode == ACB_PILOTS_REALLOCATE && (sessions->S_max <= 0 || !sessions->station || !sessions->arrival_offset ||
                                          !sessions->remaining_demand || !sessions->max_rate || !(period > 0))) {
        acb_set_error("acb_quantize_pilots: the reallocation needs the session tables and period > 0");
        return ACB_E_INVALID;
    }
    if (site->d.nAllow == 0) { acb_set_error("acb_quantize_pilots: site has no allowable_pilots"); return ACB_E_INVALID; }
    const size_t smem = (mode == ACB_PILOTS_REALLOCATE) ? quantize_smem_bytes(site->d, sessions->S_max) : 0;
    if (smem > ACB_MAX_SMEM) { acb_set_error("acb_quantize_pilots: site and S_max need more shared memory than a block has"); return ACB_E_TOO_LARGE; }
    ACB_CUDA(cudaSetDevice(site->device));
    if (smem > 48 * 1024) ACB_CUDA(cudaFuncSetAttribute(k_quantize_pilots, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_quantize_pilots<<<batch->B, ACB_QP_THREADS, smem, (cudaStream_t)stream>>>(site->d, mode, *sessions, period, batch->rates, batch->T,
                                                                                batch->n_sessions, batch->Tp, pilots);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

extern "C" int acb_constraints_feasible(acb_site* site, const double* rates, int B, int T, int col, int32_t* feasible, void* stream) {
    if (!site || !rates || !feasible || B <= 0 || col < 0 || col >= T) { acb_set_error("acb_constraints_feasible: bad arguments"); return ACB_E_INVALID; }
    ACB_CUDA(cudaSetDevice(site->device));
    k_feasible<<<B, 32, site->d.N * sizeof(double), (cudaStream_t)stream>>>(site->d, rates, B, T, col, feasible);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

extern "C" int acb_min_rate_admission(acb_site* site, int B, int S_max, const int32_t* n_sessions, const int32_t* sess_row,
                                      const double* try_rate, int32_t* admitted, void* stream) {
    if (!site || !n_sessions || !sess_row || !try_rate || !admitted || B <= 0 || S_max <= 0) {
        acb_set_error("acb_min_rate_admission: bad arguments");
        return ACB_E_INVALID;
    }
    ACB_CUDA(cudaSetDevice(site->device));
    k_min_rate_admission<<<B, 32, site->d.N * sizeof(double), (cudaStream_t)stream>>>(site->d, B, S_max, n_sessions, sess_row, try_rate, admitted);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}
