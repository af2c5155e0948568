// rcm_ecs_kernels.cuh - the equilibrium climate response (rcm_climate_response, rcm_lbl_climate_response): Newton on the
// stratospheric heating rates and the net flux at the tropopause, in the unknowns dT_l (l < ntrop) and dTs, the uniform
// potential-temperature increment of the troposphere and the surface, with the water-vapour feedback re-applied at every
// iterate.  The evaluation and the Jacobian are the adjusted-forcing call's (rcm_diag_rt_kernel / rcm_diag_sum_kernel and
// rcm_fjac_kernel; the LBL step's rt and finish kernels and rcm_lbl_fjac_kernel), reused unchanged.  Included by
// rcm_kernels.cu inside its anonymous namespace, after rcm_split_kernels.cuh (tile block layout) and rcm_fdh_kernels.cuh.
//
//   rcm_ecs_retemper_kernel      one thread per (column, layer): the temperature-dependent fields of the tile block at T + dT,
//                                the surface's at Ts + dTs, with fixed RH the H2O row
//   rcm_lbl_ecs_retemper_kernel  the same for the LBL copies: T_B + dT, T_surf + dTs and s_H2O
//   rcm_ecs_check_kernel         one thread per column: the ntrop + 1 residuals, outputs, freeze, count
//   rcm_ecs_newton_kernel        one warp per column: the (ntrop + 1)-square Newton matrix from J and dE_jac, Gaussian
//                                elimination with partial pivoting, the update
// Every value is a function of its column alone; the atomic add only counts the columns still active.
#pragma once

// the water-vapour feedback of the step (main.cpp:281-289), with the prep's expression: H2O VMR of layer l at T
__device__ __forceinline__ double ecs_h2o(double T, double rel_hum, int l) {
    const double Tc = T - 273.15;
    const double e_sat = 6.1094 * exp(17.625 * Tc / (Tc + 243.04));
    return rel_hum * e_sat / cst.player[l];
}

// rcm_fdh_retemper_kernel's fields at T + dT, TB_INVTS and Tsp at Ts + dTs, and with fixed RH the H2O row of the tile block:
// the feedback at T + dT times the H2O factor, as rcm_diag_scale_kernel multiplies it.  With prep's expressions, so that at
// dT = dTs = 0 the block is bit-identical to what rcm_split_col_kernel and rcm_diag_scale_kernel wrote.
__global__ void __launch_bounds__(256) rcm_ecs_retemper_kernel(const EcsArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *a.nactive = 0;  // the check kernel that follows on this stream counts into it
    if (i >= a.ncol * NLAY) return;
    const int col = i / NLAY, l = i % NLAY;
    if (a.iter == 0) {
        if (l == 0) {
            a.iters[col] = FDH_ACTIVE;
            a.dTs[col] = 0.0;
        }
        a.dT[i] = 0.0;
    } else if (a.iters[col] != FDH_ACTIVE) {
        return;
    }
    const double d = a.iter == 0 ? 0.0 : a.dT[i];
    const int cc = col % SPLIT_C, r = prow(l);
    double* const tb = reinterpret_cast<double*>(a.tile + (size_t)(col / SPLIT_C) * TILE_BYTES);
    int* const tbi = reinterpret_cast<int*>(tb + TB_DOUBLES);
    const double midT = a.Ttau[i] + d, tref = cst.tref_ip[r];
    const int it = lowerpos_t(tref, midT, cst.n_tpert);
    const double t0 = tref + cst.t_pert[it], t1 = tref + cst.t_pert[it + 1];
    tbi[TBI_IT + tbix(r, cc)] = it;
    const double w = (midT - t0) / (t1 - t0);
    tb[TB_DELT + tbd(r, cc)] = w;
    tb[TB_DTDP + tbd(r, cc)] = __dmul_rn(w, cst.delP[r]);
    const double T = a.Tb[i] + d;
    a.Tp[i] = T;
    tb[TB_INVT + tbd(r, cc)] = (1.0 / fmax(T, a.T_floor)) * L2E64;
    if (a.fixed_rh) tb[TB_VMR + tbd(r, cc)] = __dmul_rn(ecs_h2o(T, a.rel_hum[i], l), a.f_h2o);  // (H2O: slot 0)
    if (l == 0) {
        const double Ts = a.Ts0[col] + (a.iter == 0 ? 0.0 : a.dTs[col]);
        a.Tsp[col] = Ts;
        tb[TB_INVTS + cc] = (1.0 / fmax(Ts, a.T_floor)) * L2E64;
    }
}

// The LBL evaluation: the step's rt and finish kernels run on the chunk's copies, and the finish moves their T and T_surf in
// place.  Before each evaluation every column's copy is rewritten: T = T_B + dT, T_surf = T_surf,B + dTs, and with fixed RH
// s_H2O = (f_H2O x h2o(T)) / h2o_ref, rcm_lbl_scale_kernel's expression on the feedback at T.  The Jacobian gets the same
// values in Tp and Tsp.  LBL tau depends on T only through s_H2O.
__global__ void __launch_bounds__(256) rcm_lbl_ecs_retemper_kernel(const EcsArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *a.nactive = 0;
    if (i >= a.ncol * NLAY) return;
    const int col = i / NLAY, l = i % NLAY;
    if (a.iter == 0) {
        if (l == 0) {
            a.iters[col] = FDH_ACTIVE;
            a.dTs[col] = 0.0;
        }
        a.dT[i] = 0.0;
    }
    const double T = a.Tb[i] + (a.iter == 0 ? 0.0 : a.dT[i]);
    a.T[i] = T;
    a.Tp[i] = T;
    if (a.fixed_rh) a.sH[i] = __dmul_rn(a.f_h2o, ecs_h2o(T, a.rel_hum[i], l)) / a.h2o_ref[l];
    if (l == 0) {
        const double Ts = a.Ts0[col] + (a.iter == 0 ? 0.0 : a.dTs[col]);
        a.Ts[col] = Ts;
        a.Tsp[col] = Ts;
    }
}

// residual r of equation e of column col: e < ntrop the heating rate of layer e, e = ntrop the net flux at level ntrop,
// N = E_down - E_up, formed as (Ed[k] - Eu[k]) - (Ed0[k] - Eu0[k])
__device__ __forceinline__ double ecs_residual(const EcsArgs& a, int col, int nt, int e) {
    if (e < nt) return a.dE[(size_t)col * NLAY + e] - a.dE0[(size_t)col * NLAY + e];
    const size_t k = (size_t)col * NLEV + nt;
    return (a.Ed[k] - a.Eu[k]) - (a.Ed0[k] - a.Eu0[k]);
}

// After the evaluation of iterate iter: a column converges when the largest |residual| of its ntrop + 1 equations is <= tol.
// An active column writes its outputs at every evaluation, so that a frozen column keeps those of the evaluation it froze at
// (met the test, hit max_iter, residual not finite, or - frozen by the Newton kernel - a failed solve).  F is that of
// iterate 0: the IRF at TOA and at the tropopause.
__global__ void __launch_bounds__(FDH_CHECK_NT) rcm_ecs_check_kernel(const EcsArgs a) {
    const int col = blockIdx.x * FDH_CHECK_NT + threadIdx.x;
    bool active = false;
    if (col < a.ncol && a.iters[col] == FDH_ACTIVE) {
        const int nt = a.ntrop[col];
        double res = 0.0;
        bool finite = true;
        for (int e = 0; e <= nt; ++e) {
            const double r = ecs_residual(a, col, nt, e);
            finite = finite && isfinite(r);
            res = fmax(res, fabs(r));
        }
        const double* Ed = a.Ed + (size_t)col * NLEV;
        const double* Eu = a.Eu + (size_t)col * NLEV;
        if (a.iter == 0) {
            const double* Ed0 = a.Ed0 + (size_t)col * NLEV;
            const double* Eu0 = a.Eu0 + (size_t)col * NLEV;
            a.F[(size_t)col * 2] = (Ed[0] - Eu[0]) - (Ed0[0] - Eu0[0]);
            a.F[(size_t)col * 2 + 1] = (Ed[nt] - Eu[nt]) - (Ed0[nt] - Eu0[nt]);
        }
        for (int k = 0; k < NLEV; ++k) {
            a.Ed_out[(size_t)col * NLEV + k] = Ed[k];
            a.Eu_out[(size_t)col * NLEV + k] = Eu[k];
        }
        if (!finite) a.iters[col] = -1;
        else if (res <= a.tol) a.iters[col] = a.iter;
        else if (a.iter == a.max_iter) a.iters[col] = -1;
        else active = true;
    }
    const int n = __syncthreads_count(active);
    if (threadIdx.x == 0 && n) atomicAdd(a.nactive, n);
}

constexpr int ECS_NEWTON_NT = 128, ECS_NEWTON_WARPS = ECS_NEWTON_NT / 32;

// Newton step of an active column, m = ntrop + 1 unknowns (dT_0 .. dT_{ntrop-1}, dTs).  D_i, the 41 entries of equation i, is
// row i of dE_jac for i < ntrop and J_down[ntrop] - J_up[ntrop] for i = ntrop; gamma_l = d ln q_l / dT_l of the feedback at
// T_l = T_B,l + dT_l (0 with fixed q).  Then A[i][j] = D_i[j] + gamma_j D_i[21 + j] for j < ntrop, and A[i][ntrop] =
// D_i[20] + sum_{l = ntrop}^{19} (D_i[l] + gamma_l D_i[21 + l]) / conv_l in index order; A delta = -residual.  The elimination
// is rcm_fdh_newton_kernel's: lane r owns row r; the pivot of column k is the largest |A[r][k]|, r >= k, the lowest row on
// ties (NaN counts as infinite, so that it is chosen and refused).  A zero or non-finite pivot, or a non-finite delta, freezes
// the column at -1 with dT and dTs unchanged.  Otherwise dT_l += delta_l (l < ntrop), dTs += delta_ntrop and dT_l = dTs /
// conv_l for l >= ntrop.
__global__ void __launch_bounds__(ECS_NEWTON_NT) rcm_ecs_newton_kernel(const EcsArgs a) {
    __shared__ double sA[ECS_NEWTON_WARPS][ECS_MAXM][ECS_MAXM + 1];  // [row][column], column m = right-hand side
    __shared__ double sg[ECS_NEWTON_WARPS][NLAY];                   // gamma_l
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int col = blockIdx.x * ECS_NEWTON_WARPS + wp;
    if (col >= a.ncol || a.iters[col] != FDH_ACTIVE) return;  // (whole warps)
    double(*A)[ECS_MAXM + 1] = sA[wp];
    double* const g = sg[wp];
    const int nt = a.ntrop[col], m = nt + 1;
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
        double v;
        if (j < nt) {
            v = D(r, j) + g[j] * D(r, NLAY + 1 + j);
        } else if (j == nt) {
            v = D(r, NLAY);
            for (int l = nt; l < NLAY; ++l) v = v + (D(r, l) + g[l] * D(r, NLAY + 1 + l)) / cst.conv[l];
        } else {
            v = -ecs_residual(a, col, nt, r);
        }
        A[r][j] = v;
    }
    __syncwarp();
    bool ok = true;
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
    if (lane != 0) return;
    bool finite = ok;
    if (ok) {
        for (int r = m - 1; r >= 0; --r) {  // back substitution; delta_r replaces the right-hand side in A[r][m]
            double v = A[r][m];
            for (int j = r + 1; j < m; ++j) v = v - A[r][j] * A[j][m];
            A[r][m] = v / A[r][r];
            finite = finite && isfinite(A[r][m]);
        }
    }
    if (!finite) {
        a.iters[col] = -1;
        return;
    }
    double* const dT = a.dT + (size_t)col * NLAY;
    for (int l = 0; l < nt; ++l) dT[l] += A[l][m];
    const double th = a.dTs[col] + A[nt][m];
    a.dTs[col] = th;
    for (int l = nt; l < NLAY; ++l) dT[l] = th / cst.conv[l];
}
