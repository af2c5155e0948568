// rcm_fjac.cuh - declarations of the flux-Jacobian call's kernel (rcm_fjac_kernels.cuh, rcm_flux_jacobian).
#ifndef RCM_FJAC_CUH
#define RCM_FJAC_CUH

#include "rcm_jac.cuh"

constexpr int FJAC_NJ = 2 * NLEV * JAC_NE;  // J of one column: [2][21][41], E_down rows then E_up rows
constexpr int FJAC_NH = NLAY * JAC_NE;      // dE_jac of one column: [20][41]

// One chunk of columns whose tile blocks rcm_split_col_kernel (prep) has written into a scratch buffer.
struct FjacArgs {
    int ncol, clampk;
    double tau_clamp, T_floor;
    double wtau;                      // 2 pi dmu, as JacArgs
    const double* __restrict__ coef;  // the split path's rows (SplitArgs::coef)
    const double* __restrict__ planck_c;
    const double* __restrict__ planck_k;
    const double* __restrict__ exp_tab;
    const unsigned char* tile;        // [ceil(ncol / 16)][TILE_BYTES]
    const double* T;                  // [ncol][20] the sorted profile the Planck source is evaluated at (prep's output)
    const double* Ts;                 // [ncol] surface temperature
    double* J;                        // [ncol][2][21][41]
    double* dE_jac;                   // [ncol][20][41]
};

cudaError_t rcm_launch_fjac(const FjacArgs& a, cudaStream_t st);
int rcm_fjac_ctas_per_sm();

#endif
