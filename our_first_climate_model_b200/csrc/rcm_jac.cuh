// rcm_jac.cuh - declarations of the radiative-kernel call's kernels (rcm_jac_kernels.cuh, rcm_radiative_kernels).
#ifndef RCM_JAC_CUH
#define RCM_JAC_CUH

#include "rcm_diag.cuh"

constexpr int JAC_NE = 2 * NLAY + 1;  // entries per output: dF/dT_l (20), dF/dT_surf, dF/dln q_l (20)
constexpr int JAC_NK = 2 * JAC_NE;    // [2][41]: output 0 = E_up[0] (OLR), output 1 = E_down[20] (surface downward flux)

// One chunk of columns whose tile blocks rcm_split_col_kernel (prep) has written into a scratch buffer.
struct JacArgs {
    int ncol, ntiles;                 // columns of the chunk; tiles of 16 columns
    int nsplit, ipu, nitem, nunits;   // as SplitArgs: (tile, split) units of ipu wavelength rounds
    int clampk;
    double tau_clamp, T_floor;
    double wtau;                      // 2 pi dmu: the quadrature weight 2 pi mu dmu of every angle over its mu
    const double* __restrict__ coef;  // the split path's rows (SplitArgs::coef)
    const double* __restrict__ planck_c;
    const double* __restrict__ planck_k;
    const double* __restrict__ exp_tab;
    const unsigned char* tile;        // [ntiles][TILE_BYTES]
    const double* T;                  // [ncol][20] the sorted profile the Planck source is evaluated at (prep's output)
    const double* Ts;                 // [ncol] surface temperature
    double* K_spec;                   // [ncol][nwvl][2][41] every wavelength alone
    double* K;                        // [ncol][2][41] sums over the wavelengths in index order
};

cudaError_t rcm_launch_jac_rt(const JacArgs& a, int grid, cudaStream_t st);
cudaError_t rcm_launch_jac_sum(const JacArgs& a, cudaStream_t st);
int rcm_jac_ctas_per_sm();

#endif
