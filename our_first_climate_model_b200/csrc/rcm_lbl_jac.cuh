// rcm_lbl_jac.cuh - launches of the line-by-line radiative-kernel call's kernels (rcm_lbl_jac_kernels.cuh,
// rcm_lbl_radiative_kernels).
#ifndef RCM_LBL_JAC_CUH
#define RCM_LBL_JAC_CUH

#include "rcm_jac.cuh"

// Arguments: the LblArgs of a prepared chunk (rcm_lbl_prep_kernel, and rcm_lbl_scale_kernel with factors; a.tau3 the composed
// planes with CO2, CH4 or N2O scaled), wtau = 2 pi / nangle (JacArgs::wtau), and the staging K_spec [ncol][nwvl][2][41]:
// every (column, wavelength)'s derivatives of the OLR and the surface downward flux (entries as rcm_radiative_kernels).
size_t rcm_lbl_jac_smem_bytes();
cudaError_t rcm_launch_lbl_jac(const LblArgs& a, double wtau, double* K_spec, cudaStream_t st);
// K_band [ncol][nband][2][41]: band b the sum of K_spec's rows [band_start[b], band_start[b + 1]) in index order, from 0.0
// (band_start [nband + 1] on the device)
cudaError_t rcm_launch_lbl_jac_band_sum(int ncol, int nwvl, int nband, const int* band_start, const double* K_spec, double* K_band,
                                        cudaStream_t st);

#endif
