// rcm_lbl_species_kernels.cuh - species Jacobians of the line-by-line path (rcm_lbl_species_jacobian): the analytic derivatives
// of every level's E_down and E_up, summed over the wavelengths, with respect to the ln VMR of each of the five species in each
// layer, of the state rcm_lbl_prep_kernel (and rcm_lbl_scale_kernel) prepared.  Included by rcm_kernels.cu inside its anonymous
// namespace, after rcm_lbl_kernels.cuh, rcm_lbl_fjac_kernels.cuh and rcm_species_kernels.cuh (SpjacWarp).
//
//   rcm_lbl_species_fjac_kernel  rcm_lbl_fjac_kernel's layout, tau and angle schedule: one warp per column, lane k owns level
//                                k and runs every wavelength in index order into per-lane slots; nothing is staged per
//                                wavelength.
// dtau_l/dln x_{s,l} is species s's share of tau_l as rcm_lbl_diagnose_fluxes composes it: tau_H2O,l x s_H2O,l,
// (f_CO2 x co2_factor) x tau_CO2,l, tau_O3,l x s_O3,l, f_N2O x tau_N2O,l, f_CH4 x tau_CH4,l, each one rounded product, 0 where
// the clamp acts.  The H2O share is rcm_lbl_fjac_kernel's dtau/dln q, so the H2O block equals its entries 21..40 bit for bit.
#pragma once

// ------------------------------------------------------------------------------------------
// Per wavelength lane l < 20 evaluates its layer's tau as rcm_lbl_rt_kernel does and its five shares, and (lanes 0..20) the
// band Planck source.  The sweeps, the angle schedule, the slot walk and the epilogue are rcm_species_fjac_kernel's (copies:
// see rcm_lbl_fjac_kernel for the originals on LBL tau).
// ------------------------------------------------------------------------------------------
template <bool CLAMPK>
__global__ void __launch_bounds__(SPJ_NT, SPJ_CTAS) rcm_lbl_species_fjac_kernel(const LblArgs a, double wtau,
                                                                              const double* __restrict__ raw, double f_co2x,
                                                                              double f_ch4, double f_n2o, double* J,
                                                                              double* dE_jac) {
    constexpr int NACT = SPJ_NS, NE = SPJ_NE;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* const s_exp = reinterpret_cast<double*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    SpjacWarp& s = reinterpret_cast<SpjacWarp*>(smem_raw + (size_t)EXP_TAB * EXP_REP * 8)[tid >> 5];
    load_exp_tab(s_exp, a.exp_tab, tid, SPJ_NT);
    __syncthreads();
    const int col = blockIdx.x * SPJ_WARPS + (tid >> 5);
    if (col >= a.ncol) return;  // (whole warps)
    const unsigned tab_lane = (unsigned)__cvta_generic_to_shared(s_exp + (lane & (EXP_REP - 1)));
    const int tau_clamp_hi = __double2hiint(a.tau_clamp);
    const int nwvl = a.nwvl;
    const size_t plane = (size_t)nwvl * NLAY;

    // the layer whose tau and source this lane evaluates (lane 20 the surface's source; lanes 21..31 repeat layer 19)
    const int l = min(lane, NLAY - 1);
    const bool sfc = lane == NLAY, keep = lane <= NLAY;
    const size_t gi = (size_t)col * NLAY + l;
    const double sH = a.sH[gi], sO = a.sO[gi];
    const double cw_l = cst.cloud_w[prow(l)];  // cloud weight of the layer (pair-order row, as the rt kernel)
    const double cl = a.cloud_col ? a.cloud_col[col] : cst.cloud_tau;
    const double Tsrc = sfc ? a.Tsurf[col] : a.Tlayer[gi];

    const int k = min(lane, NLAY), nu = NLAY - k;  // level of the lane; slots of its up row
    if (keep) {
#pragma unroll
        for (int q = 0; q < NACT; ++q)
#pragma unroll
            for (int i = 0; i < NLAY; ++i) s.W[q][i][lane] = 0.0;
    }

#pragma unroll 1
    for (int w = 0; w < nwvl; ++w) {
        const double* t3 = a.tau3 + (size_t)w * NLAY + l;
        double v = fma(__ldg(t3), sH, fma(__ldg(t3 + plane), sO, __ldg(t3 + 2 * plane)));
        v = fma(cw_l, cl, v);
        const double tau = CLAMPK ? v : clamp_hi(v, tau_clamp_hi);
        // rcm_lbl_fjac_kernel's source, its derivative stored as there (see SpjacWarp::dB)
        const double2 b = cplkavg_narrow_dT(__ldg(a.wvl_lo + w), __ldg(a.wvl_hi + w), __ldg(a.wn_hi + w), __ldg(a.wn_lo + w),
                                            __ldg(a.bin_ok + w) != 0, Tsrc, tab_lane);
        const double B = b.x;
        if (lane < NLAY) {
            s.B[lane] = B;
            s.dB[lane] = b.y;
            const bool on = tau == v;
            const double* rw = raw + (size_t)w * NLAY + l;  // CO2, CH4, N2O
            s.dts[0][lane] = on ? __ldg(t3) * sH : 0.0;
            s.dts[1][lane] = on ? __dmul_rn(f_co2x, __ldg(rw)) : 0.0;
            s.dts[2][lane] = on ? __ldg(t3 + plane) * sO : 0.0;
            s.dts[3][lane] = on ? __dmul_rn(f_n2o, __ldg(rw + 2 * plane)) : 0.0;
            s.dts[4][lane] = on ? __dmul_rn(f_ch4, __ldg(rw + plane)) : 0.0;
        } else if (sfc) {
            s.B[NLAY] = B;
            s.dB[NLAY] = b.y;
        }
        __syncwarp();

        double aT[NLAY];
#pragma unroll
        for (int i = 0; i < NLAY; ++i) aT[i] = 0.0;
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
                if (i == nu) P = 1.0;  // the up row is done: the down row from layer k - 1
                const int up = i < nu, m = up ? k + i : NLAY - 1 - i;
                const double t = s.t[m];
                aT[i] = fma(cw, P * t * s.x[up][m], aT[i]);
                P = P * t;
            }
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
        // chain rule to the five species (rcm_lbl_fjac_kernel's ln q expression), summed over the wavelengths in index order
        if (keep) {
#pragma unroll
            for (int i = 0; i < NLAY; ++i) {
                const int m = i < nu ? k + i : NLAY - 1 - i;
#pragma unroll
                for (int q = 0; q < NACT; ++q) s.W[q][i][lane] = s.W[q][i][lane] + -aT[i] * s.dts[q][m];
            }
        }
        __syncwarp();  // the next wavelength rewrites B and dts
    }

    // rcm_species_fjac_kernel's epilogue
    double* const Jd = J + ((size_t)col * 2 * NLEV + k) * NE;
    double* const Ju = Jd + NLEV * NE;
    double* const H = dE_jac + ((size_t)col * NLAY + k) * NE;
#pragma unroll 1
    for (int e = 0; e < NE; ++e) {
        const int q = e / NLAY, m = e - q * NLAY;     // species and layer of entry e
        const int i = m >= k ? m - k : NLAY - 1 - m;  // its slot
        const double v = keep ? s.W[q][i][lane] : 0.0;
        const double d = (m < k) ? v : 0.0;
        const double u = (m >= k) ? v : 0.0;
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
