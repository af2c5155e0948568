// rcm_fjac_kernels.cuh - flux Jacobians of the resident ensemble (rcm_flux_jacobian): the analytic derivatives of every
// level's E_down and E_up, summed over the wavelengths, with respect to every layer's temperature, the surface temperature
// and every layer's ln(H2O VMR), from tile blocks that the split path's prep (rcm_split_col_kernel) wrote into a scratch
// buffer.  Included by rcm_kernels.cu inside its anonymous namespace, after rcm_split_kernels.cuh (tile block layout,
// exp_scaled, div_fast) and rcm_jac_kernels.cuh.
//
//   rcm_fjac_kernel  one warp per column: lane k owns level k (lanes 21..31 only help with the source and the
//                    transmissions) and runs every wavelength in index order, so the sum over the wavelengths is fixed by
//                    the table alone; lane k stores rows E_down[k] and E_up[k] of J and, with its neighbour's rows, row k
//                    of dE_jac.
// Every value is a function of its column alone (K1 from global memory, no sum across columns).
#pragma once

constexpr int FJAC_NT = 128, FJAC_WARPS = FJAC_NT / 32, FJAC_CTAS = 2;

// a warp's shared memory: the per-angle exchange between the lanes, and every lane's sums over the wavelengths
struct FjacWarp {
    double t[NLAY], omt[NLAY];  // this angle's transmissions t_l and 1 - t_l
    double x[2][NLAY];          // [0][l] = D_l - B_l, [1][l] = U_{l+1} - B_l at this angle
    double B[NLEV];             // Planck source of the layers, [20] = surface
    double dB[NLEV];            // dB/dT (0 at or below T_floor)
    double dtdT[NLAY], dtdq[NLAY];  // dtau/dT and dtau/dln q (0 where a clamp acts on tau)
    double W[2][NLAY][32];      // [0][i][lane]: dF/dT_l, [1][i][lane]: dF/dln q_l of the lane's layer slot i
};
constexpr size_t FJAC_SMEM = (size_t)EXP_TAB * EXP_REP * 8 + FJAC_WARPS * sizeof(FjacWarp);

// ------------------------------------------------------------------------------------------
// Tangent of K3 for every level.  Per angle with transmissions t_l (D_0 = 0, D_{l+1} = t_l D_l + (1 - t_l) B_l;
// U_20 = B_s, U_l = t_l U_{l+1} + (1 - t_l) B_l):
//   up row of level k, layers l >= k:   dU_k/dB_l = P (1 - t_l),  dU_k/dt_l = P (U_{l+1} - B_l),  P = prod_{k<=m<l} t_m
//                                       dU_k/dB_s = prod_{k<=m<20} t_m
//   down row of level k, layers l < k:  dD_k/dB_l = S (1 - t_l),  dD_k/dt_l = S (D_l - B_l),      S = prod_{l<m<k} t_m
// and dt_l/dtau_l = -t_l / mu: with the weight c_mu = 2 pi mu dmu the tau derivatives carry 2 pi dmu (wtau).  The two rows
// of a level use disjoint layers, 20 in all, so lane k keeps one accumulator per layer slot i: slot i < 20 - k is the up
// row's layer k + i, slot i >= 20 - k the down row's layer 19 - i (k - 1 first).  Per angle every lane < 20 publishes its
// layer's transmission, lanes 0 and 1 run the down and up sweeps, and every lane walks its 20 slots.  The schedule of the
// transmissions (chains of cubes, pair units, pipelined chain heads) is sweep_item's, one layer per lane.
// ------------------------------------------------------------------------------------------
template <bool CLAMPK>
__global__ void __launch_bounds__(FJAC_NT, FJAC_CTAS) rcm_fjac_kernel(const FjacArgs a) {
    constexpr int NACT = 5, NE = JAC_NE;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* const s_exp = reinterpret_cast<double*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    FjacWarp& s = reinterpret_cast<FjacWarp*>(smem_raw + (size_t)EXP_TAB * EXP_REP * 8)[tid >> 5];
    load_exp_tab(s_exp, a.exp_tab, tid, FJAC_NT);
    __syncthreads();
    const int col = blockIdx.x * FJAC_WARPS + (tid >> 5);
    if (col >= a.ncol) return;  // (whole warps)
    const unsigned tab_lane = (unsigned)__cvta_generic_to_shared(s_exp + (lane & (EXP_REP - 1)));
    const int tau_clamp_hi = __double2hiint(a.tau_clamp);
    const int nwvl = cst.nwvl;

    // the layer whose tau and source this lane evaluates (lane 20 also the surface's source; lanes 21..31 repeat layer 19)
    const int l = min(lane, NLAY - 1), r = prow(l), cc = col % SPLIT_C;
    const bool sfc = lane == NLAY;
    const double* tb = reinterpret_cast<const double*>(a.tile + (size_t)(col / SPLIT_C) * TILE_BYTES);
    const int* tbi = reinterpret_cast<const int*>(tb + TB_DOUBLES);
    const int it = tbi[TBI_IT + tbix(r, cc)];
    const double dT = tb[TB_DELT + tbd(r, cc)], dTdP = tb[TB_DTDP + tbd(r, cc)];
    double vmr[NACT];
#pragma unroll
    for (int q = 0; q < NACT; ++q) vmr[q] = tb[TB_VMR + q * TBD_LEN + tbd(r, cc)];
    const double cl = tb[TB_CLOUD + cc];
    const double invT = sfc ? tb[TB_INVTS + cc] : tb[TB_INVT + tbd(r, cc)];
    const double Tsrc = sfc ? a.Ts[col] : a.T[(size_t)col * NLAY + l];
    const double tref = cst.tref_ip[r];
    const double span = (tref + cst.t_pert[it + 1]) - (tref + cst.t_pert[it]);
    const double2* rows = reinterpret_cast<const double2*>(a.coef) + (size_t)(cst.ipcell[r] + it) * nwvl * 8;

    const int k = min(lane, NLAY), nu = NLAY - k;  // level of the lane; slots of its up row
    double Ws = 0.0;                               // sum over the wavelengths of dE_up[k]/dT_s
#pragma unroll
    for (int i = 0; i < NLAY; ++i) s.W[0][i][lane] = s.W[1][i][lane] = 0.0;

#pragma unroll 1
    for (int w = 0; w < nwvl; ++w) {
        // K1: tau_k1's expression (a copy: the call changes this kernel's SASS), and the chain-rule factors of its layer
        double c[16];
#pragma unroll
        for (int q2 = 0; q2 < 8; ++q2) {
            const double2 v = rows[(size_t)w * 8 + q2];
            c[2 * q2] = v.x;
            c[2 * q2 + 1] = v.y;
        }
        double acc = 0.0, xT = 0.0;
#pragma unroll
        for (int q = 0; q < NACT; ++q) {
            double v = fma(c[3 * q + 1], dT, c[3 * q]);
            v = fma(c[3 * q + 2], dTdP, v);
            acc = fma(v, vmr[q], acc);
            xT = fma(fma(c[3 * q + 2], cst.delP[r], c[3 * q + 1]), vmr[q], xT);
        }
        acc = acc * cst.numDens[r];
        const double tv = fma(cst.cloud_w[r], cl, acc);
        const double tau = fmax(CLAMPK ? tv : clamp_hi(tv, tau_clamp_hi), TAU_FLOOR);
        const double xq = fma(c[2], dTdP, fma(c[1], dT, c[0])) * vmr[0];
        const double nd = (tau == tv) ? cst.numDens[r] : 0.0;
        // K2 (main.cpp:188-191) and dB/dT = B (1 + B/k) (c/T) / T for B = k / (exp(c/T) - 1)
        const double pc = __ldg(a.planck_c + w), pk = __ldg(a.planck_k + w);
        const double B = planck_b(pc, pk, invT, tab_lane);
        const double dB = (Tsrc > a.T_floor) ? B * (1.0 + B / pk) * (pc / Tsrc) / Tsrc : 0.0;
        if (lane < NLAY) {
            s.B[lane] = B;
            s.dB[lane] = dB;
            s.dtdT[lane] = nd * xT / span;
            s.dtdq[lane] = nd * xq;
        } else if (sfc) {
            s.B[NLAY] = B;
            s.dB[NLAY] = dB;
        }
        __syncwarp();

        double aB[NLAY], aT[NLAY], aS = 0.0;
#pragma unroll
        for (int i = 0; i < NLAY; ++i) aB[i] = aT[i] = 0.0;
        auto sweep = [&](double tc, int slot) {
            const double cm = cst.cmu[slot], cw = (cm != 0.0) ? a.wtau : 0.0;
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
        // chain rule to T and ln q (rcm_jac_rt_kernel's expressions), summed over the wavelengths in index order
#pragma unroll
        for (int i = 0; i < NLAY; ++i) {
            const int m = i < nu ? k + i : NLAY - 1 - i;
            s.W[0][i][lane] = s.W[0][i][lane] + fma(aB[i], s.dB[m], -aT[i] * s.dtdT[m]);
            s.W[1][i][lane] = s.W[1][i][lane] + -aT[i] * s.dtdq[m];
        }
        Ws = Ws + aS * s.dB[NLAY];
        __syncwarp();  // the next wavelength rewrites B, dB, dtdT, dtdq
    }

    // lane k's rows of J: entry e of E_down[k] and E_up[k] (0.0 where the row does not depend on x_e), and with lane
    // k + 1's rows, row k of dE_jac entry by entry as dE from E (main.cpp:337-341; the solar term is constant)
    double* const Jd = a.J + ((size_t)col * 2 * NLEV + k) * NE;
    double* const Ju = Jd + NLEV * NE;
    double* const H = a.dE_jac + ((size_t)col * NLAY + k) * NE;
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
