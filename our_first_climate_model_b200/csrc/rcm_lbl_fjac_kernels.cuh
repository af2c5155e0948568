// rcm_lbl_fjac_kernels.cuh - flux Jacobians of the line-by-line path (rcm_lbl_flux_jacobian): the analytic derivatives of every
// level's E_down and E_up, summed over the wavelengths, with respect to every layer's temperature, the surface temperature and
// every layer's ln(H2O VMR), of the state rcm_lbl_prep_kernel (and rcm_lbl_scale_kernel) prepared.  Included by rcm_kernels.cu
// inside its anonymous namespace, after rcm_lbl_kernels.cuh, rcm_fjac_kernels.cuh (the layout of J and dE_jac) and
// rcm_lbl_jac_kernels.cuh (cplkavg_narrow_dT).
//
//   rcm_lbl_fjac_kernel  rcm_fjac_kernel's layout on LBL tau and source: one warp per column, lane k owns level k and runs
//                        every wavelength in index order into per-lane slots, so the sum over the wavelengths is fixed by the
//                        table alone and nothing is staged per wavelength.
// LBL tau does not depend on T: d/dT_l acts through layer l's band Planck source alone (dB/dT of cplkavg_narrow_dT), and
// d/dln q_l through tau_H2O,l x s_H2O,l, 0 where the clamp acts.  Every value is a function of its column alone.
#pragma once

constexpr int LBL_FJAC_NT = 128, LBL_FJAC_WARPS = LBL_FJAC_NT / 32, LBL_FJAC_CTAS = 2;

// a warp's shared memory: FjacWarp without dtau/dT
struct LblFjacWarp {
    double t[NLAY], omt[NLAY];  // this angle's transmissions t_l and 1 - t_l
    double x[2][NLAY];          // [0][l] = D_l - B_l, [1][l] = U_{l+1} - B_l at this angle
    double B[NLEV];             // band Planck source of the layers, [20] = surface
    double dB[NLEV];            // its dB/dT
    double dtdq[NLAY];          // dtau/dln q (0 where a clamp acts on tau)
    double W[2][NLAY][32];      // [0][i][lane]: dF/dT_l, [1][i][lane]: dF/dln q_l of the lane's layer slot i
};
constexpr size_t LBL_FJAC_SMEM = (size_t)EXP_TAB * EXP_REP * 8 + LBL_FJAC_WARPS * sizeof(LblFjacWarp);

// ------------------------------------------------------------------------------------------
// Per wavelength, lane l < 20 evaluates its layer's tau as rcm_lbl_rt_kernel does (the two FMAs on tau3, the cloud, the clamp)
// and (B, dB/dT) at T_l; lane 20 (B, dB/dT) at T_surf.  The angles, the sweeps of lanes 0 and 1 and the slot walk are
// rcm_fjac_kernel's (see there): slot i < 20 - k is the up row's layer k + i, slot i >= 20 - k the down row's layer 19 - i.
// ------------------------------------------------------------------------------------------
template <bool CLAMPK>
__global__ void __launch_bounds__(LBL_FJAC_NT, LBL_FJAC_CTAS) rcm_lbl_fjac_kernel(const LblArgs a, double wtau, double* J,
                                                                                  double* dE_jac) {
    constexpr int NE = JAC_NE;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* const s_exp = reinterpret_cast<double*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    LblFjacWarp& s = reinterpret_cast<LblFjacWarp*>(smem_raw + (size_t)EXP_TAB * EXP_REP * 8)[tid >> 5];
    load_exp_tab(s_exp, a.exp_tab, tid, LBL_FJAC_NT);
    __syncthreads();
    const int col = blockIdx.x * LBL_FJAC_WARPS + (tid >> 5);
    if (col >= a.ncol) return;  // (whole warps)
    const unsigned tab_lane = (unsigned)__cvta_generic_to_shared(s_exp + (lane & (EXP_REP - 1)));
    const int tau_clamp_hi = __double2hiint(a.tau_clamp);
    const int nwvl = a.nwvl;
    const size_t plane = (size_t)nwvl * NLAY;

    // the layer whose tau and source this lane evaluates (lane 20 the surface's source; lanes 21..31 repeat layer 19)
    const int l = min(lane, NLAY - 1);
    const bool sfc = lane == NLAY;
    const size_t gi = (size_t)col * NLAY + l;
    const double sH = a.sH[gi], sO = a.sO[gi];
    const double cw_l = cst.cloud_w[prow(l)];  // cloud weight of the layer (pair-order row, as the rt kernel)
    const double cl = a.cloud_col ? a.cloud_col[col] : cst.cloud_tau;
    const double Tsrc = sfc ? a.Tsurf[col] : a.Tlayer[gi];

    const int k = min(lane, NLAY), nu = NLAY - k;  // level of the lane; slots of its up row
    double Ws = 0.0;                               // sum over the wavelengths of dE_up[k]/dT_s
#pragma unroll
    for (int i = 0; i < NLAY; ++i) s.W[0][i][lane] = s.W[1][i][lane] = 0.0;

#pragma unroll 1
    for (int w = 0; w < nwvl; ++w) {
        const double* t3 = a.tau3 + (size_t)w * NLAY + l;
        double v = fma(__ldg(t3), sH, fma(__ldg(t3 + plane), sO, __ldg(t3 + 2 * plane)));
        v = fma(cw_l, cl, v);
        const double tau = CLAMPK ? v : clamp_hi(v, tau_clamp_hi);
        const double2 b = cplkavg_narrow_dT(__ldg(a.wvl_lo + w), __ldg(a.wvl_hi + w), __ldg(a.wn_hi + w), __ldg(a.wn_lo + w),
                                            __ldg(a.bin_ok + w) != 0, Tsrc, tab_lane);
        if (lane < NLAY) {
            s.B[lane] = b.x;
            s.dB[lane] = b.y;
            s.dtdq[lane] = (tau == v) ? __ldg(t3) * sH : 0.0;
        } else if (sfc) {
            s.B[NLAY] = b.x;
            s.dB[NLAY] = b.y;
        }
        __syncwarp();

        double aB[NLAY], aT[NLAY], aS = 0.0;
#pragma unroll
        for (int i = 0; i < NLAY; ++i) aB[i] = aT[i] = 0.0;
        auto sweep = [&](double tc, int slot) {
            const double cm = cst.cmu[slot], cw = (cm != 0.0) ? wtau : 0.0;
            if (lane < NLAY) {
                s.t[lane] = tc;
                s.omt[lane] = 1.0 - tc;
            }
            __syncwarp();
            if (lane < 2) {  // lane 0: D downwards from D_0 = 0; lane 1: U upwards from U_20 = B_s (sweep_item's expression)
                double X = lane ? s.B[NLAY] : 0.0;
#pragma unroll
                for (int i = 0; i < NLAY; ++i) {
                    const int m = lane ? NLAY - 1 - i : i;
                    const double d = X - s.B[m];
                    s.x[lane][m] = d;
                    X = fma(s.t[m], d, s.B[m]);
                }
            }
            __syncwarp();
            double P = 1.0;
#pragma unroll
            for (int i = 0; i < NLAY; ++i) {
                if (i == nu) {  // the up row is done: the surface term, then the down row from layer k - 1
                    aS = fma(cm, P, aS);
                    P = 1.0;
                }
                const int up = i < nu, m = up ? k + i : NLAY - 1 - i;
                const double t = s.t[m];
                aB[i] = fma(cm, P * s.omt[m], aB[i]);
                aT[i] = fma(cw, P * t * s.x[up][m], aT[i]);
                P = P * t;
            }
            if (nu == NLAY) aS = fma(cm, P, aS);
            __syncwarp();  // everybody is done with this angle's t and x
        };
        // the angle schedule of jac_sweep_item, one layer per lane
        int slot = 0;
        auto chain = [&](double& tc, double& tn, int len, double nim) {
#pragma unroll 1
            for (int j = 1; j < len; ++j) {
                sweep(tc, slot++);
                tc = tc * tc * tc;
            }
            tn = exp_scaled<CLAMPK>(tau, nim, tab_lane);
            sweep(tc, slot++);
        };
        const int nchain = cst.nchain, npair = cst.npair;
        double tA = exp_scaled<CLAMPK>(tau, npair ? cst.pair_nim[0] : cst.neg_inv_mu_l2e[0], tab_lane), tB;
#pragma unroll 1
        for (int p = 0; p < npair; ++p) {
            const int type = cst.pair_type[p];
            tB = tA * tA;
            tA = tA * tB;
            if (type == 1) tA = tA * tB;
            else if (type == 2) tB = tB * tB;
            tB = tB * tA;
            const int lenA = cst.pair_lenA[p], lenB = cst.pair_lenB[p];
#pragma unroll 1
            for (int j = 1; j < lenA; ++j) {
                sweep(tA, slot++);
                tA = tA * tA * tA;
            }
            sweep(tA, slot++);
            chain(tB, tA, lenB, cst.pair_nim[p + 1]);
        }
#pragma unroll 1
        for (int ic = 0; ic < nchain; ic += 2) {
            chain(tA, tB, cst.chain_len[ic], cst.neg_inv_mu_l2e[ic + 1]);
            chain(tB, tA, cst.chain_len[ic + 1], cst.neg_inv_mu_l2e[ic + 2]);
        }
        // chain rule to T (the source alone) and ln q (rcm_lbl_jac_kernel's expressions), summed over the wavelengths in
        // index order
#pragma unroll
        for (int i = 0; i < NLAY; ++i) {
            const int m = i < nu ? k + i : NLAY - 1 - i;
            s.W[0][i][lane] = s.W[0][i][lane] + aB[i] * s.dB[m];
            s.W[1][i][lane] = s.W[1][i][lane] + -aT[i] * s.dtdq[m];
        }
        Ws = Ws + aS * s.dB[NLAY];
        __syncwarp();  // the next wavelength rewrites B, dB, dtdq
    }

    // lane k's rows of J and, with lane k + 1's rows, row k of dE_jac: rcm_fjac_kernel's epilogue
    double* const Jd = J + ((size_t)col * 2 * NLEV + k) * NE;
    double* const Ju = Jd + NLEV * NE;
    double* const H = dE_jac + ((size_t)col * NLAY + k) * NE;
#pragma unroll 1
    for (int e = 0; e < NE; ++e) {
        const int m = e < NLAY ? e : e - NLAY - 1;  // layer of entry e (the surface: -1)
        const int i = m >= k ? m - k : NLAY - 1 - m;  // its slot
        const double v = (e == NLAY) ? Ws : s.W[e > NLAY][i < NLAY ? i : 0][lane];
        const double d = (e != NLAY && m < k) ? v : 0.0;
        const double u = (e == NLAY || m >= k) ? v : 0.0;
        const double d1 = __shfl_down_sync(0xffffffffu, d, 1), u1 = __shfl_down_sync(0xffffffffu, u, 1);
        if (lane <= NLAY) {
            Jd[e] = d;
            Ju[e] = u;
        }
        if (lane < NLAY) {
            double h = d - d1 + u1 - u;
            if (lane == NLAY - 1) h += d1 - u1;
            H[e] = h;
        }
    }
}

// ------------------------------------------------------------------------------------------
// rcm_lbl_adjusted_forcing's evaluation at T_B + dT: the step's rt and finish kernels run on the chunk's copies, and the finish
// moves their T and T_surf in place.  One thread per (column, layer) rewrites every column's copy before each evaluation,
// T = T_B + dT and T_surf as prepared, and hands the Jacobian the same T_B + dT in Tp.  LBL tau does not depend on T, so
// nothing else moves with dT.  At iter 0 it also starts every column (dT = 0, active), as rcm_fdh_retemper_kernel.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rcm_lbl_fdh_retemper_kernel(const FdhArgs a, double* T, double* Ts, const double* Ts0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *a.nactive = 0;  // the check kernel that follows on this stream counts into it
    if (i >= a.ncol * NLAY) return;
    const int col = i / NLAY, l = i % NLAY;
    if (a.iter == 0) {
        if (l == 0) a.iters[col] = FDH_ACTIVE;
        a.dT[i] = 0.0;
    }
    const double v = a.Tb[i] + (a.iter == 0 ? 0.0 : a.dT[i]);
    T[i] = v;
    a.Tp[i] = v;
    if (l == 0) Ts[col] = Ts0[col];
}
