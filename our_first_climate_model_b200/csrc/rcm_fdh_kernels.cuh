// rcm_fdh_kernels.cuh - stratosphere-adjusted forcing by fixed dynamical heating (rcm_adjusted_forcing): Newton on the
// stratospheric heating rates, with rcm_diag_rt_kernel / rcm_diag_sum_kernel as the evaluation and rcm_fjac_kernel as the
// Jacobian, both reused unchanged.  Included by rcm_kernels.cu inside its anonymous namespace, after rcm_split_kernels.cuh
// (tile block layout) and rcm_fjac_kernels.cuh.
//
//   rcm_fdh_retemper_kernel  one thread per (column, layer): the temperature-dependent fields of the tile block at T + dT
//   rcm_fdh_check_kernel     one thread per column: residual against the base heating rates, outputs, freeze, count
//   rcm_fdh_newton_kernel    one warp per column: Gaussian elimination with partial pivoting on the ntrop x ntrop block
// Every value is a function of its column alone; the atomic add only counts the columns still active.
#pragma once

// The fields of the tile block that depend on the temperature, with prep's expressions (split_col_body: indices() and the
// TB_INVT loop): at dT = 0 the block is bit-identical to what rcm_split_col_kernel wrote.  The global-memory K1 of
// rcm_diag_rt_kernel and rcm_fjac_kernel reads only these, the VMR rows, the cloud and TB_INVTS; the row-staging plan
// (TBI_ROWSEL, TBI_ROWOFF, TBI_OUTSIDE) belongs to the step's unit kernel and stays as prep left it.
__global__ void __launch_bounds__(256) rcm_fdh_retemper_kernel(const FdhArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *a.nactive = 0;  // the check kernel that follows on this stream counts into it
    if (i >= a.ncol * NLAY) return;
    const int col = i / NLAY, l = i % NLAY;
    if (a.iter == 0) {
        if (l == 0) a.iters[col] = FDH_ACTIVE;
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
}

constexpr int FDH_CHECK_NT = 128;

// After the evaluation of iterate iter: a column converges when max_{l < ntrop} |dE_l - dE0_l| <= tol.  An active column
// writes its outputs at every evaluation, so that a frozen column keeps those of the evaluation it froze at (met the test,
// hit max_iter, residual not finite, or - frozen by the Newton kernel - a failed solve).  The IRF is that of iterate 0.
__global__ void __launch_bounds__(FDH_CHECK_NT) rcm_fdh_check_kernel(const FdhArgs a) {
    const int col = blockIdx.x * FDH_CHECK_NT + threadIdx.x;
    bool active = false;
    if (col < a.ncol && a.iters[col] == FDH_ACTIVE) {
        const int m = a.ntrop[col];
        const double* dE = a.dE + (size_t)col * NLAY;
        const double* dE0 = a.dE0 + (size_t)col * NLAY;
        double res = 0.0;
        bool finite = true;
        for (int l = 0; l < m; ++l) {
            const double r = dE[l] - dE0[l];
            finite = finite && isfinite(r);
            res = fmax(res, fabs(r));
        }
        const double* Ed = a.Ed + (size_t)col * NLEV;
        const double* Eu = a.Eu + (size_t)col * NLEV;
        const double* Ed0 = a.Ed0 + (size_t)col * NLEV;
        const double* Eu0 = a.Eu0 + (size_t)col * NLEV;
        double* F = a.F + (size_t)col * 4;
        const double toa = (Ed[0] - Eu[0]) - (Ed0[0] - Eu0[0]), trop = (Ed[m] - Eu[m]) - (Ed0[m] - Eu0[m]);
        if (a.iter == 0) {
            F[0] = toa;
            F[1] = trop;
        }
        F[2] = toa;
        F[3] = trop;
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

constexpr int FDH_NEWTON_NT = 128, FDH_NEWTON_WARPS = FDH_NEWTON_NT / 32;

// Newton step of an active column: solve dE_jac[0..m)[0..m) delta = -(dE - dE0)[0..m), then dT += delta.  Lane r owns row r
// during the elimination; the pivot of column k is the largest |A[r][k]|, r >= k, the lowest row on ties (NaN counts as
// infinite, so that it is chosen and refused).  A zero or non-finite pivot, or a non-finite delta, freezes the column at
// -1 with dT unchanged: its outputs are those of the evaluation just checked.
__global__ void __launch_bounds__(FDH_NEWTON_NT) rcm_fdh_newton_kernel(const FdhArgs a) {
    __shared__ double sA[FDH_NEWTON_WARPS][FDH_MAXM][FDH_MAXM + 1];  // [row][column], column m = right-hand side
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int col = blockIdx.x * FDH_NEWTON_WARPS + wp;
    if (col >= a.ncol || a.iters[col] != FDH_ACTIVE) return;  // (whole warps)
    double(*A)[FDH_MAXM + 1] = sA[wp];
    const int m = a.ntrop[col];  // >= 1: with no stratosphere a column converges at iterate 0
    const double* H = a.dE_jac + (size_t)col * NLAY * JAC_NE;
    for (int i = lane; i < m * (m + 1); i += 32) {
        const int r = i / (m + 1), j = i % (m + 1);
        A[r][j] = j < m ? H[r * JAC_NE + j] : -(a.dE[(size_t)col * NLAY + r] - a.dE0[(size_t)col * NLAY + r]);
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
    for (int l = 0; l < m; ++l) a.dT[(size_t)col * NLAY + l] += A[l][m];
}
