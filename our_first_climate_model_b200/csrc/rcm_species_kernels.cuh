// rcm_species_kernels.cuh - species Jacobians of the resident ensemble (rcm_species_jacobian): the analytic derivatives of every
// level's E_down and E_up, summed over the wavelengths, with respect to the ln VMR of each of the five species in each layer,
// from tile blocks that the split path's prep (rcm_split_col_kernel) wrote into a scratch buffer.  Included by rcm_kernels.cu
// inside its anonymous namespace, after rcm_split_kernels.cuh (tile block layout, exp_scaled) and rcm_fjac_kernels.cuh.
//
//   rcm_species_fjac_kernel  rcm_fjac_kernel's layout: one warp per column, lane k owns level k (lanes 21..31 only help with
//                            the source and the transmissions) and runs every wavelength in index order into per-lane slots,
//                            so the sum over the wavelengths is fixed by the table alone.
// Entry e = 20 s + l is d/dln x_{s,l} at fixed T: dtau_l/dln x_{s,l} is species s's own term of K1 at layer l times numDens_l,
// 0 where the clamp or the floor acts on tau.  For s = 0 it is rcm_fjac_kernel's dtau/dln q, so the H2O block equals that
// kernel's entries 21..40 bit for bit.  Every value is a function of its column alone.
#pragma once

constexpr int SPJ_NT = 128, SPJ_WARPS = SPJ_NT / 32, SPJ_CTAS = 2;

// A warp's shared memory: FjacWarp without the Planck derivative, with five species rows.  Lanes 21..31 keep no sums (their
// rows are never stored), so W holds 21 lanes: 16.8 KB of sums per warp, 82.5 KB per CTA with the exp table, two CTAs per SM.
struct SpjacWarp {
    double t[NLAY], omt[NLAY];  // this angle's transmissions t_l and 1 - t_l
    double x[2][NLAY];          // [0][l] = D_l - B_l, [1][l] = U_{l+1} - B_l at this angle
    double B[NLEV];             // Planck source of the layers, [20] = surface
    double dB[NLEV];            // line-by-line only: dB/dT, never read.  Stored so that B is evaluated as rcm_lbl_fjac_kernel
                                // evaluates it: with the derivative dead the compiler contracts B's expression differently
                                // and the H2O block no longer equals that kernel's bit for bit.
    double dts[SPJ_NS][NLAY];   // dtau_l/dln x_{s,l} (0 where a clamp acts on tau)
    double W[SPJ_NS][NLAY][NLEV];  // [s][i][lane]: dF/dln x_{s,m} of the lane's layer slot i (lanes 0..20)
};
constexpr size_t SPJ_SMEM = (size_t)EXP_TAB * EXP_REP * 8 + SPJ_WARPS * sizeof(SpjacWarp);

// ------------------------------------------------------------------------------------------
// The tau tangent of rcm_fjac_kernel (see there) without the source terms: per angle lane k accumulates
// aT[i] = sum_mu 2 pi dmu P t_m x_m for its slot i (slot i < 20 - k: the up row's layer k + i, slot i >= 20 - k: the down
// row's layer 19 - i), and per wavelength W[s][i] += -aT[i] dtau_m/dln x_{s,m} for the five species.  The K1 expression, the
// sweeps, the angle schedule and the epilogue are copies of rcm_fjac_kernel's (sharing them changes that kernel's SASS).
// ------------------------------------------------------------------------------------------
template <bool CLAMPK>
__global__ void __launch_bounds__(SPJ_NT, SPJ_CTAS) rcm_species_fjac_kernel(const SpjacArgs a) {
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
    const int nwvl = cst.nwvl;

    // the layer whose tau and source this lane evaluates (lane 20 also the surface's source; lanes 21..31 repeat layer 19)
    const int l = min(lane, NLAY - 1), r = prow(l), cc = col % SPLIT_C;
    const bool sfc = lane == NLAY, keep = lane <= NLAY;
    const double* tb = reinterpret_cast<const double*>(a.tile + (size_t)(col / SPLIT_C) * TILE_BYTES);
    const int* tbi = reinterpret_cast<const int*>(tb + TB_DOUBLES);
    const int it = tbi[TBI_IT + tbix(r, cc)];
    const double dT = tb[TB_DELT + tbd(r, cc)], dTdP = tb[TB_DTDP + tbd(r, cc)];
    double vmr[NACT];
#pragma unroll
    for (int q = 0; q < NACT; ++q) vmr[q] = tb[TB_VMR + q * TBD_LEN + tbd(r, cc)];
    const double cl = tb[TB_CLOUD + cc];
    const double invT = sfc ? tb[TB_INVTS + cc] : tb[TB_INVT + tbd(r, cc)];
    const double2* rows = reinterpret_cast<const double2*>(a.coef) + (size_t)(cst.ipcell[r] + it) * nwvl * 8;

    const int k = min(lane, NLAY), nu = NLAY - k;  // level of the lane; slots of its up row
    if (keep) {
#pragma unroll
        for (int q = 0; q < NACT; ++q)
#pragma unroll
            for (int i = 0; i < NLAY; ++i) s.W[q][i][lane] = 0.0;
    }

#pragma unroll 1
    for (int w = 0; w < nwvl; ++w) {
        // K1 (rcm_fjac_kernel's copy of tau_k1) and each species' own term of it
        double c[16];
#pragma unroll
        for (int q2 = 0; q2 < 8; ++q2) {
            const double2 v = rows[(size_t)w * 8 + q2];
            c[2 * q2] = v.x;
            c[2 * q2 + 1] = v.y;
        }
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < NACT; ++q) {
            double v = fma(c[3 * q + 1], dT, c[3 * q]);
            v = fma(c[3 * q + 2], dTdP, v);
            acc = fma(v, vmr[q], acc);
        }
        acc = acc * cst.numDens[r];
        const double tv = fma(cst.cloud_w[r], cl, acc);
        const double tau = fmax(CLAMPK ? tv : clamp_hi(tv, tau_clamp_hi), TAU_FLOOR);
        const double nd = (tau == tv) ? cst.numDens[r] : 0.0;
        const double B = planck_b(__ldg(a.planck_c + w), __ldg(a.planck_k + w), invT, tab_lane);  // K2 (main.cpp:188-191)
        if (lane < NLAY) {
            s.B[lane] = B;
#pragma unroll
            for (int q = 0; q < NACT; ++q) s.dts[q][lane] = nd * (fma(c[3 * q + 2], dTdP, fma(c[3 * q + 1], dT, c[3 * q])) * vmr[q]);
        } else if (sfc) {
            s.B[NLAY] = B;
        }
        __syncwarp();

        double aT[NLAY];
#pragma unroll
        for (int i = 0; i < NLAY; ++i) aT[i] = 0.0;
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
        // chain rule to the five species (rcm_fjac_kernel's ln q expression), summed over the wavelengths in index order
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

    // lane k's rows of J: entry e of E_down[k] and E_up[k] (0.0 where the row does not depend on x_e), and with lane
    // k + 1's rows, row k of dE_jac entry by entry as dE from E (main.cpp:337-341; the solar term is constant)
    double* const Jd = a.J + ((size_t)col * 2 * NLEV + k) * NE;
    double* const Ju = Jd + NLEV * NE;
    double* const H = a.dE_jac + ((size_t)col * NLAY + k) * NE;
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
