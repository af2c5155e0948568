// rcm_grad.cuh - declarations of the flux-gradient calls' kernels (rcm_grad_kernels.cuh, rcm_lbl_grad_kernels.cuh;
// rcm_flux_gradient, rcm_lbl_flux_gradient).
#ifndef RCM_GRAD_CUH
#define RCM_GRAD_CUH

#include "rcm_species.cuh"

constexpr int GRAD_NE = NLEV + SPJ_NE;  // entries per column: T_l (20), T_surf, ln x_{s,l} (100) at 21 + 20 s + l
constexpr int GRAD_NCO = 2 * NLEV;      // level cotangents per column: b_k on E_down[k] (21), then a_k on E_up[k] (21)
constexpr int GRAD_LBL_SPAN = 1024;     // LBL wavelengths per partial sum (a multiple of the kernel's 4 wavelength groups)

// One chunk of columns whose tile blocks rcm_split_col_kernel (prep) has written into a scratch buffer, as JacArgs.
struct GradArgs {
    int ncol, ntiles;                 // columns of the chunk; tiles of 16 columns
    int nsplit, ipu, nitem, nunits;   // as SplitArgs: (tile, split) units of ipu wavelength rounds
    int clampk;
    double tau_clamp, T_floor;
    double wtau;                      // 2 pi dmu, as JacArgs
    const double* __restrict__ coef;  // the split path's rows (SplitArgs::coef)
    const double* __restrict__ planck_c;
    const double* __restrict__ planck_k;
    const double* __restrict__ exp_tab;
    const unsigned char* tile;        // [ntiles][TILE_BYTES]
    const double* T;                  // [ncol][20] the sorted profile the Planck source is evaluated at (prep's output)
    const double* Ts;                 // [ncol] surface temperature
    const double* co;                 // [ncol][42] level cotangents, w_dE folded in (b_0..b_20, a_0..a_20)
    double* part;                     // [ncol][nsplit][121] the sum of each split's wavelengths
};

cudaError_t rcm_launch_grad_rt(const GradArgs& a, int grid, cudaStream_t st);
int rcm_grad_ctas_per_sm();

// Line-by-line: the LblArgs of a prepared chunk (as rcm_launch_lbl_species_fjac: wtau, raw and the factors f_co2x, f_ch4,
// f_n2o), the chunk's level cotangents co [ncol][42] and the partial sums part [ncol][ceil(nwvl / GRAD_LBL_SPAN)][121].
cudaError_t rcm_launch_lbl_grad(const LblArgs& a, double wtau, const double* raw, double f_co2x, double f_ch4, double f_n2o,
                                const double* co, double* part, cudaStream_t st);

// grad [ncol][121] = sum of part [ncol][npart][121] over the parts in index order, from 0.0
cudaError_t rcm_launch_grad_sum(int ncol, int npart, const double* part, double* grad, cudaStream_t st);

#endif
