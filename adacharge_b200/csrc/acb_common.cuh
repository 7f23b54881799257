// Shared definitions of the adacharge_b200 native library (see include/adacharge_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/adacharge_b200.h"

#define ACB_VERSION 100
#ifndef ACB_FAST_THREADS
#define ACB_FAST_THREADS 640  // block size cap of the FAST variant (v in shared memory): 20 warps -> 96 registers per thread, no spills in the hot loop
#endif
#define ACB_OHT 12         // outputs per column-pass thread (one or two threads per period: at most 24 column inputs on chip)
#define ACB_NRED 16        // floats per warp in the reduction scratch
#define ACB_MAX_WARPS 32
#define ACB_FIRST_CHECK 10  // iteration of the first convergence check (then every check_every)

// Device view of a site (all pointers device).  Row layout of the scaled coupling
// matrix Khat (R x N): 2*nDisc SOC rows (cos, sin pairs) for rows that mix phases, nLin
// linear rows (LINEAR mode: |A| rows; SOC mode: single-phase rows, two-sided), then the
// optional peak-limit row (1/sqrt(N)) and the optional aggregate-power row (k/|k|).
struct SiteDev {
    int N, M, R, NG, NP, nDisc, nLin, has_pl, has_u;
    int lin_two_sided;  // linear rows are |.| <= limit (single-phase SOC rows) instead of . <= limit (LINEAR mode)
    int TPW;        // EVSE rows per warp
    int nRowWarps;  // warps that own EVSE rows
    int nSlots;     // nRowWarps * TPW
    int nAllow;     // total allowable pilots
    const int* slot_row;    // [nSlots] EVSE index or -1
    const int* slot_grp;    // [nSlots]
    const int* slot_prow;   // [nSlots] partial-row id
    const int* slot_first;  // [nSlots] 1 = first contributor to its partial row
    const int* pg_off;      // [NG+1] partial rows of group g
    const float* ngrp;      // [NG] EVSEs per group
    const float* kg;        // [NG] kW per A
    const float* C;         // [R*NG] distinct scaled columns of Khat
    const float* U;         // [R*R] eigenvectors of Khat Khat' (U[r*R+e])
    const float* Up;        // [R*Rp] U with rows padded to Rp = roundup(R, 4) (general path, float4 loads)
    const float* Ut;        // [R*Rp] U' padded the same way
    int Rp;
    const float* Cp;        // [R*NGp] C with rows padded to NGp = roundup(NG, 4) (general path: k-major operand of hg = C'h)
    const float* Ct;        // [NG*Rp] C' padded the same way (k-major operand of b = C sa)
    int NGp;
    // rank-reduced form of the Woodbury solve (general path): Khat = C G has rank <= NG, so most eigenvalues of
    // Khat Khat' are exactly 0 and S^-1 = I/(d/rho) + Ur diag(1/(d/rho+lam) - 1/(d/rho)) Ur' over the nEig others
    int nEig, nEigp;        // nEigp = roundup(nEig, 4)
    const float* Urp;       // [R*nEigp]  Urp[r][j] = U[r][e_j]
    const float* Urt;       // [nEig*Rp]  Urt[j][r] = U[r][e_j]
    const float* lamr;      // [nEig]
    const float* lam;       // [R] eigenvalues
    const float* row_scale; // [R]
    const float* lim;       // [R] limit / row_scale (disc rows: both entries; 0 for pl/u rows)
    // float64 postprocessing constants (unscaled)
    const double* a_cos;    // [M*N] A_ji cos(phi_i)
    const double* a_sin;    // [M*N]
    const double* limits;   // [M]
    const double* max_pilot;// [N]
    const double* volt;     // [N] voltages (V), float64 for the device packer
    const int* allow_off;   // [N+1]
    const double* allow_vals;
    // sparsity of the SOC rows (entries where a_cos or a_sin is nonzero), for the reallocation greedy
    const int* evse_row_off;  // [N+1] rows with a nonzero coefficient at EVSE i: evse_rows[evse_row_off[i] ..]
    const int* evse_rows;
    const int* row_col_off;   // [M+1] nonzero columns of row j, ascending: row_cols[row_col_off[j] ..]
    const int* row_cols;
    const double* row_cos;    // a_cos / a_sin at those entries
    const double* row_sin;
};

struct acb_site {
    int device;
    SiteDev d;
    SiteDev d2;          // same site with 2 EVSE rows per warp (slot tables only differ): the FAST variant's 1024-thread blocks
    int has_d2;
    std::vector<void*> allocs;
    int constraint_type;
    const int* grp_off_dev;  // [NG+1] offsets of each group's rows in the (group-sorted) slot list
    size_t smem_fixed;   // bytes of shared memory independent of Tp
    size_t smem_per_col; // bytes per padded column
};

void acb_set_error(const std::string& s);
#define ACB_CUDA(x)                                                                   \
    do {                                                                              \
        cudaError_t e_ = (x);                                                         \
        if (e_ != cudaSuccess) {                                                      \
            acb_set_error(std::string(#x) + ": " + cudaGetErrorString(e_));          \
            return ACB_E_CUDA;                                                        \
        }                                                                             \
    } while (0)

// keep the stream-ordered pool's memory across calls (the default release threshold of 0 gives it back at every sync)
inline void acb_keep_pool(int device) {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
}
size_t acb_solve_smem_bytes(const SiteDev& s, int Tp, int S_max, int nwarps);
int acb_solve_general(acb_site* site, const acb_batch* batch, const acb_options& opt, cudaStream_t st);
