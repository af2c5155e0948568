// rcm_lbl_diag.cuh - launches of the LBL step's kernels one at a time and of the line-by-line diagnostic call's kernels
// (rcm_lbl_diag_kernels.cuh, rcm_lbl_diagnose_fluxes).
#ifndef RCM_LBL_DIAG_CUH
#define RCM_LBL_DIAG_CUH

#include "rcm_kernels.cuh"

// the step's three kernels one at a time (rcm_lbl_diagnose_fluxes runs them on scratch copies)
cudaError_t rcm_launch_lbl_prep(const LblArgs& a, cudaStream_t st);
cudaError_t rcm_launch_lbl_rt(const LblArgs& a, cudaStream_t st, cudaEvent_t ev0, cudaEvent_t ev1);
cudaError_t rcm_launch_lbl_finish(const LblArgs& a, cudaStream_t st);
// sH / sO of the prep from a.vmr with one factor on H2O and O3; the column-independent plane from raw [3][n] (CO2, CH4, N2O)
cudaError_t rcm_launch_lbl_scale(const LblArgs& a, double f_h2o, double f_o3, cudaStream_t st);
cudaError_t rcm_launch_lbl_plane(const double* raw, size_t n, double f_co2x, double f_ch4, double f_n2o, double* out, cudaStream_t st);
// every (column, wavelength)'s fluxes into spec_dn / spec_up [ncol][nwvl][21]; bands of them summed in index order into
// band_dn / band_up [ncol][nband][21] (band_start [nband + 1] on the device)
size_t rcm_lbl_band_smem_bytes();
cudaError_t rcm_launch_lbl_band(const LblArgs& a, double* spec_dn, double* spec_up, cudaStream_t st);
cudaError_t rcm_launch_lbl_band_sum(int ncol, int nwvl, int nband, const int* band_start, const double* spec_dn,
                                    const double* spec_up, double* band_dn, double* band_up, cudaStream_t st);

#endif
