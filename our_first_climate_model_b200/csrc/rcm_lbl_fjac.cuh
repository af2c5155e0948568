// rcm_lbl_fjac.cuh - launches of the line-by-line flux-Jacobian and adjusted-forcing calls' kernels (rcm_lbl_fjac_kernels.cuh,
// rcm_lbl_flux_jacobian, rcm_lbl_adjusted_forcing).
#ifndef RCM_LBL_FJAC_CUH
#define RCM_LBL_FJAC_CUH

#include "rcm_fdh.cuh"

// Arguments: the LblArgs of a prepared chunk (rcm_lbl_prep_kernel, and rcm_lbl_scale_kernel with factors; a.tau3 the composed
// planes with CO2, CH4 or N2O scaled; a.Tlayer, a.Tsurf the profile the Planck source is evaluated at), wtau = 2 pi / nangle,
// and the outputs J [ncol][2][21][41] and dE_jac [ncol][20][41] (entries as rcm_flux_jacobian).
cudaError_t rcm_launch_lbl_fjac(const LblArgs& a, double wtau, double* J, double* dE_jac, cudaStream_t st);
// Before each evaluation of rcm_lbl_adjusted_forcing: T [ncol][20] = f.Tb + dT and f.Tp the same (dT = 0 and every column
// active at f.iter 0), Ts [ncol] = Ts0, *f.nactive = 0.  Every column's copy is rewritten: the finish kernel moved it.
cudaError_t rcm_launch_lbl_fdh_retemper(const FdhArgs& f, double* T, double* Ts, const double* Ts0, cudaStream_t st);

#endif
