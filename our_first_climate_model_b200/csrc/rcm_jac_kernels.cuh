// rcm_jac_kernels.cuh - radiative kernels of the resident ensemble (rcm_radiative_kernels): the analytic derivatives of
// the OLR (E_up[0]) and the surface downward flux (E_down[20]) with respect to every layer's temperature, the surface
// temperature and every layer's ln(H2O VMR), per (column, wavelength), from tile blocks that the split path's prep
// (rcm_split_col_kernel) wrote into a scratch buffer.  Included by rcm_kernels.cu inside its anonymous namespace, after
// rcm_split_kernels.cuh (tile block layout, exp_scaled, div_fast) and rcm_diag_kernels.cuh.
//
//   rcm_jac_rt_kernel   (tile, split) units as the diagnostic call's rcm_diag_rt_kernel: K1 from global memory, the same
//                       Planck source, exp and angle schedule (cube chains and pair units), then the tangent sweep
//                       (jac_sweep_item) and the chain rule to T and ln q once per wavelength; the 82 values of each
//                       (column, wavelength) leave through shared memory as contiguous [col][w][2][41] rows
//   rcm_jac_sum_kernel  K = sum over the wavelengths in index order
// Every value is a function of its column alone (no staged table rows, no sum across columns).
#pragma once

constexpr int JAC_NT = SPLIT_NT, JAC_CTAS = 2;
constexpr int JAC_OUT = SPLIT_G * SPLIT_C * JAC_NK;  // doubles of one round's staged results [group][column][2][41]
constexpr size_t JAC_SMEM = (size_t)EXP_TAB * EXP_REP * 8 + TILE_BYTES + (size_t)JAC_OUT * 8;

// ------------------------------------------------------------------------------------------
// Tangent of K3 for one (column, wavelength, half), accumulated over the angles.  Per angle with transmissions t_l:
//   OLR:          U_20 = B_s, U_l = t_l U_{l+1} + (1 - t_l) B_l;  T_l = prod_{k<l} t_k
//                 dU_0/dB_l = T_l (1 - t_l),  dU_0/dB_s = T_20,  dU_0/dt_l = T_l (U_{l+1} - B_l)
//   surface down: D_0 = 0, D_{l+1} = t_l D_l + (1 - t_l) B_l;     S_l = prod_{k>l} t_k
//                 dD_20/dB_l = S_l (1 - t_l),                    dD_20/dt_l = S_l (D_l - B_l)
// and dt_l/dtau_l = -t_l / mu, so that with the weight c_mu = 2 pi mu dmu the tau derivatives carry c_mu / mu = 2 pi dmu
// (wtau; 0 on a padding slot).
// Lanes as in sweep_item: h = 0 owns layers 0..9 top-down, h = 1 layers 19..10 bottom-up, both as j = 0..9.  Phase A runs
// from the lane's outer boundary inward (h = 0: down from D_0 = 0, h = 1: up from U_20 = B_s) and records the radiance
// entering every owned layer (Xin) and the transmission product in front of it (Pout); the lanes swap radiance and total
// product at level 10, and phase B runs outward, with the partner's values, and accumulates:
//   set a = (Pout, Y):   h = 0 -> OLR,     h = 1 -> surface     (aB: d/dB_l, aT: d/dtau_l with the sign of -dt/dtau left out)
//   set b = (Q, Xin):    h = 0 -> surface, h = 1 -> OLR
// aS = sum c_mu T_20 (d OLR/dB_s).  The schedule (chains of cubes, pair units, pipelined chain heads) is sweep_item's.
// ------------------------------------------------------------------------------------------
template <bool CLAMPK>
__device__ __forceinline__ void jac_sweep_item(const double (&tau)[HALF], const double (&Bo)[HALF], double Bs, int h,
                                               unsigned tab_lane, double wtau, double (&aB)[HALF], double (&aT)[HALF],
                                               double (&bB)[HALF], double (&bT)[HALF], double& aS) {
    const double Xstart = h ? Bs : 0.0;
    auto sweep = [&](const double (&tc)[HALF], int slot) {
        const double cm = cst.cmu[slot], cw = (cm != 0.0) ? wtau : 0.0;
        double Xin[HALF], Pout[HALF];
        double X = Xstart, P = 1.0;
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            Xin[j] = X;
            Pout[j] = P;
            X = fma(tc[j], X - Bo[j], Bo[j]);
            P = P * tc[j];
        }
        double Y = __shfl_xor_sync(0xffffffffu, X, 1);
        double Q = __shfl_xor_sync(0xffffffffu, P, 1);
        aS = fma(cm, P * Q, aS);
#pragma unroll
        for (int j = HALF - 1; j >= 0; --j) {
            const double omt = 1.0 - tc[j];
            aB[j] = fma(cm, Pout[j] * omt, aB[j]);
            aT[j] = fma(cw, Pout[j] * tc[j] * (Y - Bo[j]), aT[j]);
            bB[j] = fma(cm, Q * omt, bB[j]);
            bT[j] = fma(cw, Q * tc[j] * (Xin[j] - Bo[j]), bT[j]);
            Y = fma(tc[j], Y - Bo[j], Bo[j]);
            Q = Q * tc[j];
        }
    };
    int slot = 0;
    auto chain = [&](double (&tc)[HALF], double (&tn)[HALF], int len, double nim) {
#pragma unroll 1
        for (int k = 1; k < len; ++k) {
            sweep(tc, slot++);
#pragma unroll
            for (int j = 0; j < HALF; ++j) tc[j] = tc[j] * tc[j] * tc[j];
        }
#pragma unroll
        for (int j = 0; j < HALF; ++j) tn[j] = exp_scaled<CLAMPK>(tau[j], nim, tab_lane);
        sweep(tc, slot++);
    };
    const int nchain = cst.nchain;
    const int npair = cst.npair;
    double tA[HALF], tB[HALF];
    {
        const double nim = npair ? cst.pair_nim[0] : cst.neg_inv_mu_l2e[0];
#pragma unroll
        for (int j = 0; j < HALF; ++j) tA[j] = exp_scaled<CLAMPK>(tau[j], nim, tab_lane);
    }
#pragma unroll 1
    for (int p = 0; p < npair; ++p) {
        const int type = cst.pair_type[p];
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            tB[j] = tA[j] * tA[j];
            tA[j] = tA[j] * tB[j];
        }
        if (type == 1) {
#pragma unroll
            for (int j = 0; j < HALF; ++j) tA[j] = tA[j] * tB[j];
        } else if (type == 2) {
#pragma unroll
            for (int j = 0; j < HALF; ++j) tB[j] = tB[j] * tB[j];
        }
#pragma unroll
        for (int j = 0; j < HALF; ++j) tB[j] = tB[j] * tA[j];
        const int lenA = cst.pair_lenA[p];
        const int lenB = cst.pair_lenB[p];
#pragma unroll 1
        for (int k = 1; k < lenA; ++k) {
            sweep(tA, slot++);
#pragma unroll
            for (int j = 0; j < HALF; ++j) tA[j] = tA[j] * tA[j] * tA[j];
        }
        sweep(tA, slot++);
        chain(tB, tA, lenB, cst.pair_nim[p + 1]);
    }
    for (int ic = 0; ic < nchain; ic += 2) {
        chain(tA, tB, cst.chain_len[ic], cst.neg_inv_mu_l2e[ic + 1]);
        chain(tB, tA, cst.chain_len[ic + 1], cst.neg_inv_mu_l2e[ic + 2]);
    }
}

template <bool CLAMPK>
__global__ void __launch_bounds__(JAC_NT, JAC_CTAS) rcm_jac_rt_kernel(const JacArgs a) {
    constexpr int C = SPLIT_C, NT = JAC_NT, G = SPLIT_G, NACT = 5;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* const s_exp = reinterpret_cast<double*>(smem_raw);
    double* const tb = reinterpret_cast<double*>(smem_raw + (size_t)EXP_TAB * EXP_REP * 8);
    const int* const tbi = reinterpret_cast<const int*>(tb + TB_DOUBLES);
    double* const s_out = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(tb) + TILE_BYTES);

    const int tid = threadIdx.x, lane = tid & 31;
    const int h = tid & 1, q = tid >> 1, c = q % C, g = q / C;  // as the unit kernel: one warp per wavelength group
    const int sb = tbd(h * HALF, c), sbi = tbix(h * HALF, c);
    const int nwvl = cst.nwvl;
    load_exp_tab(s_exp, a.exp_tab, tid, NT);
    const unsigned tab_lane = (unsigned)__cvta_generic_to_shared(s_exp + (lane & (EXP_REP - 1)));
    const int tau_clamp_hi = __double2hiint(a.tau_clamp);

    auto row_of = [&](int j, int w) {
        const int cell = cst.ipcell[h * HALF + j] + tbi[TBI_IT + sbi + j * C];
        return reinterpret_cast<const double2*>(a.coef) + (size_t)(cell * nwvl + w) * 8;
    };
    auto load_row = [&](const double2* cf, double (&cc)[16]) {
#pragma unroll
        for (int q2 = 0; q2 < 8; ++q2) {
            const double2 v = cf[q2];
            cc[2 * q2] = v.x;
            cc[2 * q2 + 1] = v.y;
        }
    };

    for (int unit = blockIdx.x; unit < a.nunits; unit += gridDim.x) {
        const int tile = unit / a.nsplit, split = unit - tile * a.nsplit;
        const int col0 = tile * C, ncl = min(C, a.ncol - col0);
        const int col = col0 + (c < ncl ? c : 0);  // padding columns of the last tile repeat its first column (prep)
        __syncthreads();  // the previous unit is done with the tile block
        load_tile(tb, a.tile + (size_t)tile * TILE_BYTES, tid, NT);
        __syncthreads();
        const int item0 = split * a.ipu, item1 = min(item0 + a.ipu, a.nitem);
#pragma unroll 1
        for (int item = item0; item < item1; ++item) {
            const int w_any = g + item * G;
            const bool real = w_any < nwvl;  // a group beyond the table runs the last wavelength with a zero source, unwritten
            const int w = real ? w_any : nwvl - 1;
            double tau[HALF], Bo[HALF];
            unsigned live = 0;  // bit j: no clamp acts on tau of owned layer j (else its derivatives are 0)
            const double cl = tb[TB_CLOUD + c];
#pragma unroll
            for (int j = 0; j < HALF; ++j) {
                const double v = tau_k1(tb, sb + j * C, h * HALF + j, row_of(j, w), cl);
                tau[j] = fmax(CLAMPK ? v : clamp_hi(v, tau_clamp_hi), TAU_FLOOR);
                live |= (tau[j] == v ? 1u : 0u) << j;
            }
            // K2 (main.cpp:188-191)
            const double pc = __ldg(a.planck_c + w);
            const double pk = real ? __ldg(a.planck_k + w) : 0.0;
#pragma unroll
            for (int j = 0; j < HALF; ++j) Bo[j] = planck_b(pc, pk, tb[TB_INVT + sb + j * C], tab_lane);
            const double Bs = planck_b(pc, pk, tb[TB_INVTS + c], tab_lane);
            double aB[HALF], aT[HALF], bB[HALF], bT[HALF], aS = 0.0;
#pragma unroll
            for (int j = 0; j < HALF; ++j) aB[j] = aT[j] = bB[j] = bT[j] = 0.0;
            jac_sweep_item<CLAMPK>(tau, Bo, Bs, h, tab_lane, a.wtau, aB, aT, bB, bT, aS);
            // chain rule.  dB/dT = B (1 + B/k) (c/T) / T for B = k / (exp(c/T) - 1), 0 at or below T_floor;
            // dtau/dT = numDens sum_k (cT_k + cPT_k delP) vmr_k / (T interval), dtau/dln q = numDens x_H2O q (H2O: slot 0
            // of the default five species)
            double* o = s_out + (size_t)(g * C + c) * JAC_NK;
            const int oa = h * JAC_NE, ob = (1 - h) * JAC_NE;
#pragma unroll
            for (int j = 0; j < HALF; ++j) {
                const int r = h * HALF + j, l = h ? (NLAY - 1 - j) : j;
                const int it = tbi[TBI_IT + sbi + j * C];
                const double tref = cst.tref_ip[r];
                const double span = (tref + cst.t_pert[it + 1]) - (tref + cst.t_pert[it]);
                double cc[16];
                load_row(row_of(j, w), cc);
                double xT = 0.0;
#pragma unroll
                for (int k = 0; k < NACT; ++k) xT = fma(fma(cc[3 * k + 2], cst.delP[r], cc[3 * k + 1]), tb[TB_VMR + k * TBD_LEN + sb + j * C], xT);
                const double dT = tb[TB_DELT + sb + j * C], dTdP = tb[TB_DTDP + sb + j * C];
                const double xq = fma(cc[2], dTdP, fma(cc[1], dT, cc[0])) * tb[TB_VMR + sb + j * C];
                const double nd = ((live >> j) & 1u) ? cst.numDens[r] : 0.0;
                const double dtdT = nd * xT / span, dtdq = nd * xq;
                const double T = a.T[(size_t)col * NLAY + l];
                const double dB = (real && T > a.T_floor) ? Bo[j] * (1.0 + Bo[j] / pk) * (pc / T) / T : 0.0;
                o[oa + l] = fma(aB[j], dB, -aT[j] * dtdT);
                o[oa + NLAY + 1 + l] = -aT[j] * dtdq;
                o[ob + l] = fma(bB[j], dB, -bT[j] * dtdT);
                o[ob + NLAY + 1 + l] = -bT[j] * dtdq;
            }
            if (h == 0) {
                const double T = a.Ts[col];
                const double dB = (real && T > a.T_floor) ? Bs * (1.0 + Bs / pk) * (pc / T) / T : 0.0;
                o[NLAY] = aS * dB;  // the OLR sees the surface through the whole atmosphere
            } else {
                o[JAC_NE + NLAY] = 0.0;  // a black surface: its temperature does not reach the downward flux
            }
            __syncthreads();
            // the round's wavelengths w0 .. w0 + nw - 1 are consecutive: per column one run of nw * 82 doubles
            const int w0 = item * G, nw = min(G, nwvl - w0), run = nw * JAC_NK;
            for (int i = tid; i < ncl * run; i += NT) {
                const int cc = i / run, k = i - cc * run, gg = k / JAC_NK, e = k - gg * JAC_NK;
                a.K_spec[((size_t)(col0 + cc) * nwvl + w0) * JAC_NK + k] = s_out[(size_t)(gg * C + cc) * JAC_NK + e];
            }
            __syncthreads();
        }
    }
}

// K[c][k] = sum_w K_spec[c][w][k], wavelengths in index order from 0.0 (numpy's acc = acc + K_spec[:, w], bit for bit)
__global__ void __launch_bounds__(256) rcm_jac_sum_kernel(const JacArgs a) {
    const int nwvl = cst.nwvl;
    const size_t n = (size_t)a.ncol * JAC_NK;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / JAC_NK, k = i - c * JAC_NK;
        const double* p = a.K_spec + c * nwvl * JAC_NK + k;
        double s = 0.0;
        for (int w = 0; w < nwvl; ++w) s += p[(size_t)w * JAC_NK];
        a.K[i] = s;
    }
}
