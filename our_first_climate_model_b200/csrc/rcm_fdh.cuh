// rcm_fdh.cuh - declarations of the adjusted-forcing call's kernels (rcm_fdh_kernels.cuh, rcm_adjusted_forcing).
#ifndef RCM_FDH_CUH
#define RCM_FDH_CUH

#include "rcm_fjac.cuh"

constexpr int FDH_MAXM = NLAY - 1;  // at most 19 stratospheric layers: the tropopause is level 0 .. 19
constexpr int FDH_ACTIVE = -2;      // iters[c] of a column that still iterates; frozen: the updates applied, or -1

// One chunk of columns whose tile blocks rcm_split_col_kernel (prep) has written into a scratch buffer and
// rcm_diag_scale_kernel has scaled.  Every array is [ncol][...] of the chunk.
struct FdhArgs {
    int ncol;
    int iter, max_iter;           // the evaluation being checked: iter Newton updates applied so far
    double tol;                   // convergence: max_{l < ntrop} |dE_l - dE0_l| <= tol (W m-2)
    double T_floor;
    unsigned char* tile;          // [ceil(ncol / 16)][TILE_BYTES]
    const double* Tb;             // [20] the sorted profile prep radiates (its Planck source)
    const double* Ttau;           // [20] the profile prep interpolated tau at: at step 0 the unsorted copy, otherwise Tb
    double* Tp;                   // [20] Tb + dT, the Planck profile of FjacArgs::T
    double* dT;                   // [20] the adjustment, exactly 0.0 at l >= ntrop
    const int* ntrop;             // stratospheric layers 0 .. ntrop - 1
    const double *Ed0, *Eu0, *dE0;  // [21], [21], [20] the base state (unscaled, dT = 0)
    const double *Ed, *Eu, *dE;     // [21], [21], [20] the evaluation at the current iterate
    const double* dE_jac;         // [20][41] rcm_fjac_kernel at the current iterate
    int* iters;                   // FDH_ACTIVE, or the column's result (updates applied, -1: not converged)
    double* F;                    // [4] IRF at TOA and tropopause, SARF at TOA and tropopause
    double *Ed_out, *Eu_out;      // [21] fluxes of the evaluation a column froze at
    int* nactive;                 // [1] columns still active after the check
};

cudaError_t rcm_launch_fdh_retemper(const FdhArgs& a, cudaStream_t st);
cudaError_t rcm_launch_fdh_check(const FdhArgs& a, cudaStream_t st);
cudaError_t rcm_launch_fdh_newton(const FdhArgs& a, cudaStream_t st);

#endif
