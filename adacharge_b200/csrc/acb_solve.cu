// Host side of the batched solve: argument checks, launch configuration, dispatch to the
// per-horizon kernel instantiations (acb_solve_q5.cu, acb_solve_q9.cu), and the standalone
// charging_rate_bounds kernel.
#include <algorithm>
#include "acb_solve_kernel.cuh"

size_t acb_solve_smem_bytes(const SiteDev& s, int Tp, int S_max, int nwarps) {
    return (size_t)make_layout(s.N, s.R, s.NG, s.NP, s.nSlots, Tp, S_max, nwarps).total * sizeof(float);
}

// charging_rate_bounds as a standalone kernel (parity tests; the solve kernel fuses it)
__global__ void acb_bounds_kernel(SiteDev S, acb_batch B, float* lb, float* ub) {
    const int b = blockIdx.x, N = S.N, Tp = B.Tp;
    const int nS = B.n_sessions[b];
    float* lbb = lb + (size_t)b * N * Tp;
    float* ubb = ub + (size_t)b * N * Tp;
    for (int i = threadIdx.x; i < N * Tp; i += blockDim.x) { lbb[i] = 0.f; ubb[i] = 0.f; }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int s = warp; s < nS; s += nwarps) {
        size_t k = (size_t)b * B.S_max + s;
        int row = B.sess_row[k], a = B.sess_start[k], len = B.sess_len[k], off = B.sess_rate_off[k];
        for (int j = lane; j < len; j += 32) {
            const int ri = off >= 0 ? off + j : -(off + 1);  // off < 0: one (min, max) pair for the whole session
            const bool f0 = j == 0 && B.sess_min0;  // first-period limits (uninterrupted charging)
            float lo = f0 ? B.sess_min0[k] : B.min_rates[ri], hi = f0 ? B.sess_max0[k] : B.max_rates[ri];
            if (a + j < Tp) { lbb[row * Tp + a + j] = lo; ubb[row * Tp + a + j] = fmaxf(hi, lo); }
        }
    }
}

int acb_launch_solve_q2(const acb_site*, const acb_batch*, const acb_options*, const SolvePhase*, int, size_t, cudaStream_t, bool, int);
int acb_launch_solve_q4(const acb_site*, const acb_batch*, const acb_options*, const SolvePhase*, int, size_t, cudaStream_t, bool, int);
int acb_launch_solve_q5(const acb_site*, const acb_batch*, const acb_options*, const SolvePhase*, int, size_t, cudaStream_t, bool, int);
int acb_launch_solve_q9(const acb_site*, const acb_batch*, const acb_options*, const SolvePhase*, int, size_t, cudaStream_t, bool, int);

// Between the launches of a phased solve: the parked (still running) instances, ordered by the relative gap of their
// last convergence check, largest first (a counting sort over 256 logarithmic buckets; one block).  The gap after the
// first phase is the best available predictor of the iterations an instance still needs, so the relaunch approximates
// longest-processing-time-first scheduling and the longest instances no longer start last.  An instance the solve skips
// (mask) is never listed: its status is still the previous solve's.
__global__ void acb_phase_list_kernel(const int32_t* status, const float* stats, const int32_t* mask, int B, int* list, int* count) {
    __shared__ int hist[256], base[256];
    const int tid = threadIdx.x;
    for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    auto bucket = [&](int b) -> int {
        const float g = stats[(size_t)b * ACB_NSTATS + 2];
        int key = (g > 0.f) ? (int)((log2f(g) + 24.f) * 8.f) : 0;  // 2^-24 .. 2^8 in steps of 2^(1/8)
        key = min(max(key, 0), 255);
        return 255 - key;
    };
    for (int b = tid; b < B; b += blockDim.x)
        if (status[b] == ACB_RUNNING && (!mask || mask[b])) atomicAdd(&hist[bucket(b)], 1);
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int i = 0; i < 256; ++i) { base[i] = acc; acc += hist[i]; }
        *count = acc;
    }
    __syncthreads();
    for (int b = tid; b < B; b += blockDim.x)
        if (status[b] == ACB_RUNNING && (!mask || mask[b])) list[atomicAdd(&base[bucket(b)], 1)] = b;
}

extern "C" int acb_solve_batch(acb_site* site, const acb_batch* batch, const acb_options* opt, void* stream) {
    return acb_solve_batch_masked(site, batch, nullptr, nullptr, opt, stream);
}

extern "C" int acb_solve_batch_masked(acb_site* site, const acb_batch* batch, const int32_t* solve_mask, const int32_t* warm_shifts,
                                      const acb_options* opt_in, void* stream) {
    if (!site || !batch || batch->B <= 0 || batch->Tp <= 0 || batch->Tp % 32 != 0) {
        acb_set_error("acb_solve_batch: bad arguments (Tp must be a positive multiple of 32)");
        return ACB_E_INVALID;
    }
    if ((site->d.has_pl && !batch->peak_limit)) {
        acb_set_error("acb_solve_batch: site was created with use_peak_row but batch.peak_limit is NULL");
        return ACB_E_INVALID;
    }
    acb_options opt;
    if (opt_in) opt = *opt_in; else acb_default_options(&opt);
    ACB_CUDA(cudaSetDevice(site->device));
    const SiteDev& d = site->d;
    const int nCT_ = d.nDisc + d.nLin + d.has_pl + d.has_u;
    const int nCT = nCT_;
    const int Q = batch->Tp / 32;
    const bool chipQ = (Q == 2 || Q == 4 || Q == 5 || Q == 9);  // horizons the on-chip kernel is instantiated for
    cudaStream_t st = (cudaStream_t)stream;
    const int NIN = d.NG + d.R;
    const int nParts = (NIN + ACB_OHT - 1) / ACB_OHT;  // column-pass threads per period
    // threads: warps for the EVSE rows plus room for the coupling rows, and one column-pass sweep if possible
    int want = std::max(d.nRowWarps * 32 + nCT * 16, std::min(1024, nParts * batch->Tp));
    // (registers are allocated in groups of four warps: round up to a multiple of 128 threads, the extra warps take coupling work)
    int nthreads = std::min(768, ((want + 127) / 128) * 128);
    size_t smem = acb_solve_smem_bytes(d, batch->Tp, batch->S_max, nthreads / 32);
    const bool fits = chipQ && d.TPW == 3 && NIN <= 2 * ACB_OHT && nthreads <= 768 && d.nRowWarps * 32 <= nthreads && smem <= 232448;
    if (opt.path == 2 || (!fits && opt.path == 0)) return acb_solve_general(site, batch, solve_mask, warm_shifts, opt, st);
    if (!fits) {
        acb_set_error("acb_solve_batch: instance does not fit the on-chip path (Tp in {64, 128, 160, 288}, N <= ~66 EVSEs, <= 32 coupling tasks, " +
                      std::to_string(smem) + " B of shared memory needed, 232448 available)");
        return ACB_E_TOO_LARGE;
    }
    const bool multi = batch->multi_session != 0;
    // every minimum rate declared 0: v in shared memory instead of the lower bounds.  opt.path 4 (experimental) runs that
    // variant with two rows per warp in 1024-thread blocks (measured 3-4 % slower than three rows in 768 threads)
    int fast = (!multi && batch->lb_zero != 0) ? 1 : 0;
    if (fast == 1 && opt.path != 4) {
        // FAST, three rows per warp: cap the block at ACB_FAST_THREADS (more registers per thread); the coupling items that
        // the fewer spare warps cannot carry ride on the row warps
        const int ntf = std::min(nthreads, std::max(ACB_FAST_THREADS, ((d.nRowWarps * 32 + 64 + 127) / 128) * 128));
        if (ntf <= ACB_FAST_THREADS && d.nRowWarps * 32 + 32 <= ntf) {
            nthreads = ntf;
            smem = acb_solve_smem_bytes(d, batch->Tp, batch->S_max, nthreads / 32);
        } else fast = 0;  // more than 19 row warps: the register-state kernel with its 768-thread bound
    }
    if (fast && site->has_d2 && opt.path == 4) {
        const SiteDev& e = site->d2;
        const int nt2 = std::min(1024, ((std::max(e.nRowWarps * 32 + nCT * 16, std::min(1024, nParts * batch->Tp)) + 127) / 128) * 128);
        const size_t sm2 = (size_t)make_layout(e.N, e.R, e.NG, e.NP, e.nSlots, batch->Tp, batch->S_max, nt2 / 32).total * sizeof(float);
        if (e.nRowWarps * 32 <= nt2 && sm2 <= 232448) { fast = 2; nthreads = nt2; smem = sm2; }
    }
    auto launch = [&](const SolvePhase& ph) -> int {
        if (Q == 2) return acb_launch_solve_q2(site, batch, &opt, &ph, nthreads, smem, st, multi, fast);
        if (Q == 4) return acb_launch_solve_q4(site, batch, &opt, &ph, nthreads, smem, st, multi, fast);
        if (Q == 5) return acb_launch_solve_q5(site, batch, &opt, &ph, nthreads, smem, st, multi, fast);
        return acb_launch_solve_q9(site, batch, &opt, &ph, nthreads, smem, st, multi, fast);
    };
    // scratch from the stream-ordered pool: the schedule of the previous check (rate polish) and the parked state
    int nSM = 148;
    cudaDeviceGetAttribute(&nSM, cudaDevAttrMultiProcessorCount, site->device);
    const int B = batch->B, N = d.N, Tp = batch->Tp, R1 = std::max(d.R, 1);
    const bool phased = opt.phase_iters > 0 && opt.phase_iters < opt.max_iter && B > nSM;
    const bool wantZ = opt.rate_tol > 0.f;
    const size_t nNT = (size_t)B * N * Tp;
    size_t bytes = 256;
    if (wantZ) bytes += nNT * 4;
    if (phased) bytes += nNT * 4 + ((size_t)B * R1 * Tp + (size_t)B * 2 * batch->S_max + (size_t)B * ACB_NSTATE + B + 64) * 4 + 1024;
    char* base = nullptr;
    SolvePhase ph{};
    ph.it_stop = opt.max_iter;
    ph.solve_mask = solve_mask;
    ph.warm_shifts = warm_shifts;
    if (wantZ || phased) {
        acb_keep_pool(site->device);
        ACB_CUDA(cudaMallocAsync((void**)&base, bytes, st));
        char* p = base;
        auto take = [&](size_t n) { void* r = p; p += ((n * 4 + 255) / 256) * 256; return r; };
        if (wantZ) ph.zprev = (float*)take(nNT);
        if (phased) {
            ph.st_v1 = (float*)take(nNT);
            ph.st_vc = (float*)take((size_t)B * R1 * Tp);
            ph.st_mu = (float*)take((size_t)B * 2 * batch->S_max);
            ph.st_scal = (float*)take((size_t)B * ACB_NSTATE);
        }
    }
    int rc;
    if (!phased) rc = launch(ph);
    else {
        int* list = (int*)(base + bytes - ((size_t)B + 64) * 4);
        int* count = list + B;
        ph.it_stop = opt.phase_iters;
        rc = launch(ph);
        if (rc == ACB_OK) {
            acb_phase_list_kernel<<<1, 1024, 0, st>>>(batch->status, batch->stats, solve_mask, B, list, count);
            ph.it_stop = opt.max_iter; ph.resume = 1; ph.list = list; ph.count = count;
            rc = launch(ph);
        }
    }
    if (base) ACB_CUDA(cudaFreeAsync(base, st));
    return rc;
}

extern "C" int acb_charging_rate_bounds(acb_site* site, const acb_batch* batch, float* lb, float* ub, void* stream) {
    if (!site || !batch || !lb || !ub) { acb_set_error("acb_charging_rate_bounds: bad arguments"); return ACB_E_INVALID; }
    ACB_CUDA(cudaSetDevice(site->device));
    acb_bounds_kernel<<<batch->B, 256, 0, (cudaStream_t)stream>>>(site->d, *batch, lb, ub);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}
