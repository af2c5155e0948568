// rcm_ecs_adj_kernels.cuh - the adjoint of the converged climate response (rcm_climate_response_gradient,
// rcm_lbl_climate_response_gradient).  Included by rcm_kernels.cu inside its anonymous namespace, after rcm_ecs_kernels.cuh
// (ecs_h2o, ECS_NEWTON_NT) and rcm_grad_kernels.cuh.
//
//   rcm_ecs_adjoint_kernel   one warp per column: the Newton matrix A at the solution, assembled as rcm_ecs_newton_kernel does,
//                            the transpose solve A^T lambda = e_m by its elimination, s = -lambda into dTs_dF, and s folded into
//                            the level cotangents of rcm_grad_rt_kernel / rcm_lbl_grad_kernel
// Every value is a function of its column alone.
#pragma once

// The column's m = ntrop + 1 equations R(y) in y = (dT_0 .. dT_{ntrop-1}, dTs) at the solution: A = dR/dy from J and dE_jac
// at the solution (rcm_ecs_newton_kernel's D_i, gamma_l and conv_l in its index order), stored transposed, with e_m as the
// right-hand side.  The elimination is rcm_ecs_newton_kernel's: lane r owns row r, partial pivoting, the lowest row on ties,
// NaN counts as infinite so that it is chosen and refused.  A zero or non-finite pivot, a non-finite lambda, or iters == -1
// (the response did not converge) give a row of quiet NaN in dF and zero cotangents.  Otherwise, with s = -lambda:
//   dF [21]: s_i for i < ntrop, s_m at 20, 0.0 elsewhere;
//   co [42]: w_dE[i] = s_i (i < ntrop), w_E_down[ntrop] = s_m, w_E_up[ntrop] = -s_m, every other cotangent 0.0, folded with
//            grad_fold's expressions in its order: b_k = (w_Ed[k] + w_dE[k]) - w_dE[k-1], a_k = (w_Eu[k] - w_dE[k]) + w_dE[k-1].
__global__ void __launch_bounds__(ECS_NEWTON_NT) rcm_ecs_adjoint_kernel(const EcsArgs a, double* dF, double* co) {
    __shared__ double sA[ECS_NEWTON_WARPS][ECS_MAXM][ECS_MAXM + 1];  // [row][column] of A^T, column m = right-hand side
    __shared__ double sg[ECS_NEWTON_WARPS][NLAY];                   // gamma_l
    __shared__ int sok[ECS_NEWTON_WARPS];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int col = blockIdx.x * ECS_NEWTON_WARPS + wp;
    if (col >= a.ncol) return;  // (whole warps)
    double(*A)[ECS_MAXM + 1] = sA[wp];
    double* const g = sg[wp];
    const int nt = a.ntrop[col], m = nt + 1;
    bool ok = a.iters[col] != -1;  // (warp-uniform)
    if (ok) {
        const double* H = a.dE_jac + (size_t)col * NLAY * JAC_NE;
        const double* Jd = a.J + ((size_t)col * 2 * NLEV + nt) * JAC_NE;
        const double* Ju = Jd + NLEV * JAC_NE;
        if (lane < NLAY) {
            double v = 0.0;
            if (a.fixed_rh) {
                const double x = a.Tp[(size_t)col * NLAY + lane] - 273.15 + 243.04;
                v = 17.625 * 243.04 / (x * x);
            }
            g[lane] = v;
        }
        __syncwarp();
        auto D = [&](int r, int e) { return r < nt ? H[r * JAC_NE + e] : Jd[e] - Ju[e]; };
        for (int i = lane; i < m * (m + 1); i += 32) {
            const int r = i / (m + 1), j = i % (m + 1);
            if (j < nt) {
                A[j][r] = D(r, j) + g[j] * D(r, NLAY + 1 + j);
            } else if (j == nt) {
                double v = D(r, NLAY);
                for (int l = nt; l < NLAY; ++l) v = v + (D(r, l) + g[l] * D(r, NLAY + 1 + l)) / cst.conv[l];
                A[j][r] = v;
            } else {
                A[r][m] = r == nt ? 1.0 : 0.0;
            }
        }
        __syncwarp();
        for (int k = 0; k < m; ++k) {
            double v = -1.0;
            int p = k;
            if (lane >= k && lane < m) {
                const double x = A[lane][k];
                v = isnan(x) ? INFINITY : fabs(x);
                p = lane;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {  // a total order on (v, p): every lane ends with the same pivot
                const double v2 = __shfl_xor_sync(0xffffffffu, v, off);
                const int p2 = __shfl_xor_sync(0xffffffffu, p, off);
                if (v2 > v || (v2 == v && p2 < p)) {
                    v = v2;
                    p = p2;
                }
            }
            const double piv = A[p][k];
            if (!(piv != 0.0 && isfinite(piv))) {  // (warp-uniform)
                ok = false;
                break;
            }
            __syncwarp();
            if (p != k && lane >= k && lane <= m) {
                const double t = A[k][lane];
                A[k][lane] = A[p][lane];
                A[p][lane] = t;
            }
            __syncwarp();
            if (lane > k && lane < m) {
                const double f = A[lane][k] / A[k][k];
                for (int j = k + 1; j <= m; ++j) A[lane][j] = A[lane][j] - f * A[k][j];
            }
            __syncwarp();
        }
        if (ok && lane == 0) {
            bool finite = true;
            for (int r = m - 1; r >= 0; --r) {  // back substitution; lambda_r replaces the right-hand side in A[r][m]
                double v = A[r][m];
                for (int j = r + 1; j < m; ++j) v = v - A[r][j] * A[j][m];
                A[r][m] = v / A[r][r];
                finite = finite && isfinite(A[r][m]);
            }
            sok[wp] = finite;
        }
        __syncwarp();
        ok = ok && sok[wp];
    }
    if (lane >= NLEV) return;
    const int k = lane;
    auto w = [&](int i) { return ok && i < nt ? -A[i][m] : 0.0; };  // w_dE[i] = s_i
    const double sm = ok ? -A[nt][m] : 0.0;
    double f = 0.0;
    if (!ok) f = __longlong_as_double(0x7ff8000000000000LL);
    else if (k < nt) f = w(k);
    else if (k == NLAY) f = sm;
    dF[(size_t)col * NLEV + k] = f;
    double bk = k == nt ? sm : 0.0, ak = k == nt ? -sm : 0.0;
    if (k < NLAY) {
        bk = bk + w(k);
        ak = ak - w(k);
    }
    if (k >= 1 && k < NLAY) {
        bk = bk - w(k - 1);
        ak = ak + w(k - 1);
    }
    co[(size_t)col * 2 * NLEV + k] = bk;
    co[(size_t)col * 2 * NLEV + NLEV + k] = ak;
}
