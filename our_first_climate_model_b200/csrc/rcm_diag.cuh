// rcm_diag.cuh - declarations of the diagnostic radiation call's kernels (rcm_diag_kernels.cuh, rcm_diagnose_fluxes).
#ifndef RCM_DIAG_CUH
#define RCM_DIAG_CUH

#include "rcm_kernels.cuh"

// One chunk of columns whose tile blocks rcm_split_col_kernel (prep) has written into a scratch buffer.
struct DiagArgs {
    int ncol, ntiles;                 // columns of the chunk; tiles of 16 columns
    int nsplit, ipu, nitem, nunits;   // as SplitArgs: (tile, split) units of ipu wavelength rounds
    int clampk;
    double tau_clamp;
    const double* __restrict__ coef;  // the split path's rows (SplitArgs::coef)
    const double* __restrict__ planck_c;
    const double* __restrict__ planck_k;
    const double* __restrict__ exp_tab;
    const unsigned char* tile;        // [ntiles][TILE_BYTES]
    double* spec_dn;                  // [ncol][nwvl][21] E_down of every wavelength alone (level 0 = 0)
    double* spec_up;                  // [ncol][nwvl][21] E_up
    double* E_down;                   // [ncol][21] sums over the wavelengths in index order
    double* E_up;                     // [ncol][21]
    double* dE;                       // [ncol][20] main.cpp:337-341 from them
    const double* solar_col;          // [ncol] or NULL (rcm_params::solar_irr)
};
struct DiagScale { double f[5]; };  // factors on the five active species' VMR rows of the tile blocks

cudaError_t rcm_launch_diag_scale(unsigned char* tile, int ntiles, const DiagScale& sc, cudaStream_t st);
cudaError_t rcm_launch_diag_rt(const DiagArgs& a, int grid, cudaStream_t st);
cudaError_t rcm_launch_diag_sum(const DiagArgs& a, cudaStream_t st);

#endif
