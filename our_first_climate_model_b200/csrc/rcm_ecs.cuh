// rcm_ecs.cuh - declarations of the climate-response call's kernels (rcm_ecs_kernels.cuh, rcm_climate_response,
// rcm_lbl_climate_response).
#ifndef RCM_ECS_CUH
#define RCM_ECS_CUH

#include "rcm_fdh.cuh"

constexpr int ECS_MAXM = NLAY;  // unknowns: at most 19 stratospheric layers and the tropospheric increment

// One chunk of columns: the adjusted-forcing call's evaluation copies (tile blocks on repwvl, the LBL copies on line-by-line)
// and the base evaluation.  Unknowns of a column: dT_l of the stratospheric layers l < ntrop and dTs, the uniform
// potential-temperature increment of the troposphere and the surface (dT_l = dTs / conv_l for l >= ntrop).  Every array is
// [ncol][...] of the chunk.
struct EcsArgs {
    int ncol;
    int iter, max_iter;           // the evaluation being checked: iter Newton updates applied so far
    int fixed_rh;                 // H2O re-evaluated at T + dT by the water-vapour feedback (else every VMR stays fixed)
    double tol;                   // convergence: max over the ntrop + 1 residuals <= tol (W m-2)
    double T_floor;
    double f_h2o;                 // the H2O factor of vmr_scale (1 when unscaled)
    unsigned char* tile;          // repwvl: [ceil(ncol / 16)][TILE_BYTES]
    const double* Tb;             // [20] the sorted profile prep radiates (its Planck source)
    const double* Ttau;           // [20] repwvl: the profile prep interpolated tau at (at step 0 the unsorted copy, else Tb)
    const double* Ts0;            // [1] surface temperature the base state radiates
    const double* rel_hum;        // [20] relative humidity of the feedback
    double* Tp;                   // [20] Tb + dT: the Planck profile of the Jacobian
    double* Tsp;                  // [1] Ts0 + dTs: the surface temperature of the Jacobian
    double* dT;                   // [20] the response profile
    double* dTs;                  // [1] the surface (and tropospheric potential-temperature) response
    double *T, *Ts, *sH;          // line-by-line: the copies the step's kernels radiate (rewritten at every iterate)
    const double* h2o_ref;        // line-by-line: [20] the H2O reference profile of s_H2O
    const int* ntrop;             // stratospheric layers 0 .. ntrop - 1
    const double *Ed0, *Eu0, *dE0;  // [21], [21], [20] the base state (unscaled, dT = 0)
    const double *Ed, *Eu, *dE;     // [21], [21], [20] the evaluation at the current iterate
    const double* J;              // [2][21][41] the flux Jacobian at the current iterate
    const double* dE_jac;         // [20][41]
    int* iters;                   // FDH_ACTIVE, or the column's result (updates applied, -1: not converged)
    double* F;                    // [2] IRF at TOA and tropopause (iterate 0)
    double *Ed_out, *Eu_out;      // [21] fluxes of the evaluation a column froze at
    int* nactive;                 // [1] columns still active after the check
};

cudaError_t rcm_launch_ecs_retemper(const EcsArgs& a, cudaStream_t st);
cudaError_t rcm_launch_lbl_ecs_retemper(const EcsArgs& a, cudaStream_t st);
cudaError_t rcm_launch_ecs_check(const EcsArgs& a, cudaStream_t st);
cudaError_t rcm_launch_ecs_newton(const EcsArgs& a, cudaStream_t st);
// the adjoint of the converged response (rcm_ecs_adj_kernels.cuh): dF [ncol][21] = dTs / d(forcing term of equation i) and
// co [ncol][42], the level cotangents of the gradient sweep that give dTs / dp
cudaError_t rcm_launch_ecs_adjoint(const EcsArgs& a, double* dF, double* co, cudaStream_t st);

#endif
