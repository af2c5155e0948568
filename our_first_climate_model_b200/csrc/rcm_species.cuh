// rcm_species.cuh - declarations of the species-Jacobian calls' kernels (rcm_species_kernels.cuh, rcm_lbl_species_kernels.cuh;
// rcm_species_jacobian, rcm_lbl_species_jacobian).
#ifndef RCM_SPECIES_CUH
#define RCM_SPECIES_CUH

#include "rcm_fjac.cuh"

constexpr int SPJ_NS = 5;                   // species: H2O, CO2, O3, N2O, CH4 (ascending species index, the order of vmr_scale)
constexpr int SPJ_NE = SPJ_NS * NLAY;       // entries e = 20 s + l: d/dln x_{s,l}
constexpr int SPJ_NJ = 2 * NLEV * SPJ_NE;   // J of one column: [2][21][100], E_down rows then E_up rows
constexpr int SPJ_NH = NLAY * SPJ_NE;       // dE_jac of one column: [20][100]

// One chunk of columns whose tile blocks rcm_split_col_kernel (prep) has written into a scratch buffer (FjacArgs without the
// Planck-derivative inputs: no entry moves T).
struct SpjacArgs {
    int ncol, clampk;
    double tau_clamp;
    double wtau;                      // 2 pi dmu, as JacArgs
    const double* __restrict__ coef;  // the split path's rows (SplitArgs::coef)
    const double* __restrict__ planck_c;
    const double* __restrict__ planck_k;
    const double* __restrict__ exp_tab;
    const unsigned char* tile;        // [ceil(ncol / 16)][TILE_BYTES]
    double* J;                        // [ncol][2][21][100]
    double* dE_jac;                   // [ncol][20][100]
};

cudaError_t rcm_launch_species_fjac(const SpjacArgs& a, cudaStream_t st);

// Line-by-line: the LblArgs of a prepared chunk (as rcm_launch_lbl_fjac), wtau = 2 pi / nangle, raw = the tables' raw CO2, CH4
// and N2O planes [3][nwvl][20] and their factors f_co2x = f_CO2 x co2_factor, f_ch4, f_n2o (those rcm_lbl_plane_kernel composes
// with), and the outputs J [ncol][2][21][100], dE_jac [ncol][20][100].
cudaError_t rcm_launch_lbl_species_fjac(const LblArgs& a, double wtau, const double* raw, double f_co2x, double f_ch4,
                                        double f_n2o, double* J, double* dE_jac, cudaStream_t st);

#endif
