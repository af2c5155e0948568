// rcm_grad_kernels.cuh - adjoint flux gradients of the resident ensemble (rcm_flux_gradient): the derivatives of one weighted
// sum of a column's broadband fluxes and heating rates with respect to every layer's temperature, the surface temperature and
// every layer's ln VMR of the five species, by one reverse sweep per (column, wavelength, angle), from tile blocks that the
// split path's prep (rcm_split_col_kernel) wrote into a scratch buffer.  Included by rcm_kernels.cu inside its anonymous
// namespace, after rcm_jac_kernels.cuh and rcm_species_kernels.cuh.
//
//   rcm_grad_rt_kernel   rcm_jac_rt_kernel's (tile, split) units, K1, Planck source, exp and angle schedule, with
//                        grad_sweep_item in place of jac_sweep_item; the chain rule to the 121 entries once per wavelength,
//                        summed per thread in shared memory, then per unit over the 4 wavelength groups in group order
//   rcm_grad_sum_kernel  grad = the sum of the units' partials over the splits in split order, from 0.0
// Summation order of an entry: the wavelengths g, g + 4, ... of a split per group g, the groups 0..3, the splits 0..nsplit - 1:
// fixed by the table (nsplit = ceil(nitem / SPLIT_IPU)) and the angle schedule alone.  Every value is a function of its column.
#pragma once

constexpr int GRAD_NT = SPLIT_NT, GRAD_CTAS = 2;
constexpr int GRAD_ACC = SPLIT_G * SPLIT_C * GRAD_NE;  // doubles of a unit's per-thread sums [group][column][121]
constexpr size_t GRAD_SMEM = (size_t)EXP_TAB * EXP_REP * 8 + TILE_BYTES + (size_t)GRAD_ACC * 8;

// ------------------------------------------------------------------------------------------
// Adjoint of K3 for one (column, wavelength, half), accumulated over the angles.  Per angle with weight c = c_mu, tau weight
// cw = 2 pi dmu (0 on a padding slot), transmissions t_l and the level cotangents a_k (on E_up[k]) and b_k (on E_down[k]):
//   forward:  D_0 = 0, D_{l+1} = t_l D_l + (1 - t_l) B_l;          U_20 = B_s, U_l = t_l U_{l+1} + (1 - t_l) B_l
//   adjoint:  Ub_0 = a_0, Ub_{l+1} = a_{l+1} + t_l Ub_l;           Db_20 = b_20, Db_l = b_l + t_l Db_{l+1}
//   gB_l += c (Ub_l + Db_{l+1}) (1 - t_l)                           (d/dB_l)
//   gT_l += cw t_l [Ub_l (U_{l+1} - B_l) + Db_{l+1} (D_l - B_l)]    (d/dtau_l with the sign of -dt/dtau left out)
//   gS   += c Ub_20                                                 (d/dB_s; h = 1 only)
// Lanes as jac_sweep_item: h = 0 owns layers 0..9 and runs D and Ub down, h = 1 owns layers 19..10 and runs U and Db up, both
// as j = 0..9.  In the lane's frame cA[0..10] are the cotangents its phase A picks up (h = 0: a_0..a_10, h = 1: b_20..b_10)
// and cB[j] the one its phase B picks up leaving owned layer j (h = 0: b_j, h = 1: a_{20-j}).  Phase A records the radiance
// (Xin) and the adjoint (Gin) entering every owned layer from the lane's outer boundary; the lanes swap both at level 10, and
// phase B runs outward with the partner's radiance Y and adjoint H and accumulates.  The schedule is jac_sweep_item's.
// ------------------------------------------------------------------------------------------
template <bool CLAMPK>
__device__ __forceinline__ void grad_sweep_item(const double (&tau)[HALF], const double (&Bo)[HALF], double Bs, int h,
                                                unsigned tab_lane, double wtau, const double (&cA)[HALF + 1],
                                                const double (&cB)[HALF], double (&gB)[HALF], double (&gT)[HALF], double& gS) {
    const double Xstart = h ? Bs : 0.0;
    auto sweep = [&](const double (&tc)[HALF], int slot) {
        const double cm = cst.cmu[slot], cw = (cm != 0.0) ? wtau : 0.0;
        double Xin[HALF], Gin[HALF];
        double X = Xstart, G = cA[0];
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            Xin[j] = X;
            Gin[j] = G;
            X = fma(tc[j], X - Bo[j], Bo[j]);
            G = fma(tc[j], G, cA[j + 1]);
        }
        double Y = __shfl_xor_sync(0xffffffffu, X, 1);
        double H = __shfl_xor_sync(0xffffffffu, G, 1);
#pragma unroll
        for (int j = HALF - 1; j >= 0; --j) {
            const double omt = 1.0 - tc[j];
            gB[j] = fma(cm, (Gin[j] + H) * omt, gB[j]);
            gT[j] = fma(cw, tc[j] * fma(Gin[j], Y - Bo[j], H * (Xin[j] - Bo[j])), gT[j]);
            Y = fma(tc[j], Y - Bo[j], Bo[j]);
            H = fma(tc[j], H, cB[j]);
        }
        gS = fma(cm, H, gS);
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

// The lane's cotangents in its own frame (see grad_sweep_item) from the column's row co = {b_0..b_20, a_0..a_20}.
__device__ __forceinline__ void grad_load_co(const double* co, int h, double (&cA)[HALF + 1], double (&cB)[HALF]) {
#pragma unroll
    for (int j = 0; j <= HALF; ++j) cA[j] = h ? co[NLAY - j] : co[NLEV + j];
#pragma unroll
    for (int j = 0; j < HALF; ++j) cB[j] = h ? co[NLEV + NLAY - j] : co[j];
}

template <bool CLAMPK>
__global__ void __launch_bounds__(GRAD_NT, GRAD_CTAS) rcm_grad_rt_kernel(const GradArgs a) {
    constexpr int C = SPLIT_C, NT = GRAD_NT, G = SPLIT_G, NACT = SPJ_NS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* const s_exp = reinterpret_cast<double*>(smem_raw);
    double* const tb = reinterpret_cast<double*>(smem_raw + (size_t)EXP_TAB * EXP_REP * 8);
    const int* const tbi = reinterpret_cast<const int*>(tb + TB_DOUBLES);
    double* const s_acc = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(tb) + TILE_BYTES);

    const int tid = threadIdx.x, lane = tid & 31;
    const int h = tid & 1, q = tid >> 1, c = q % C, g = q / C;  // as the unit kernel: one warp per wavelength group
    const int sb = tbd(h * HALF, c), sbi = tbix(h * HALF, c);
    const int nwvl = cst.nwvl;
    load_exp_tab(s_exp, a.exp_tab, tid, NT);
    const unsigned tab_lane = (unsigned)__cvta_generic_to_shared(s_exp + (lane & (EXP_REP - 1)));
    const int tau_clamp_hi = __double2hiint(a.tau_clamp);
    double* const acc = s_acc + (size_t)(g * C + c) * GRAD_NE;  // this thread's sums (its own entries only)

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
        __syncthreads();  // the previous unit is done with the tile block and the sums
        load_tile(tb, a.tile + (size_t)tile * TILE_BYTES, tid, NT);
        for (int i = tid; i < GRAD_ACC; i += NT) s_acc[i] = 0.0;
        __syncthreads();
        double cA[HALF + 1], cB[HALF];
        grad_load_co(a.co + (size_t)col * GRAD_NCO, h, cA, cB);
        const int item0 = split * a.ipu, item1 = min(item0 + a.ipu, a.nitem);
#pragma unroll 1
        for (int item = item0; item < item1; ++item) {
            const int w_any = g + item * G;
            const bool real = w_any < nwvl;  // a group beyond the table runs the last wavelength with a zero source, unsummed
            const int w = real ? w_any : nwvl - 1;
            double tau[HALF], Bo[HALF];
            unsigned live = 0;  // bit j: no clamp acts on tau of owned layer j (else its tau derivatives are 0)
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
            double gB[HALF], gT[HALF], gS = 0.0;
#pragma unroll
            for (int j = 0; j < HALF; ++j) gB[j] = gT[j] = 0.0;
            grad_sweep_item<CLAMPK>(tau, Bo, Bs, h, tab_lane, a.wtau, cA, cB, gB, gT, gS);
            if (!real) continue;
            // chain rule as rcm_jac_rt_kernel (T) and rcm_species_fjac_kernel (the five species' own terms of K1)
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
                const double nd = ((live >> j) & 1u) ? cst.numDens[r] : 0.0;
                const double dtdT = nd * xT / span;
                const double T = a.T[(size_t)col * NLAY + l];
                const double dB = (T > a.T_floor) ? Bo[j] * (1.0 + Bo[j] / pk) * (pc / T) / T : 0.0;
                acc[l] = acc[l] + fma(gB[j], dB, -gT[j] * dtdT);
#pragma unroll
                for (int k = 0; k < NACT; ++k) {
                    const double dts = nd * (fma(cc[3 * k + 2], dTdP, fma(cc[3 * k + 1], dT, cc[3 * k])) * tb[TB_VMR + k * TBD_LEN + sb + j * C]);
                    acc[NLEV + k * NLAY + l] = acc[NLEV + k * NLAY + l] + -gT[j] * dts;
                }
            }
            if (h == 1) {  // the surface: Ub_20 lives in the bottom lane
                const double T = a.Ts[col];
                const double dB = (T > a.T_floor) ? Bs * (1.0 + Bs / pk) * (pc / T) / T : 0.0;
                acc[NLAY] = acc[NLAY] + gS * dB;
            }
        }
        __syncthreads();
        // the unit's partial: per column and entry the sum over the groups in group order, from 0.0
        for (int i = tid; i < ncl * GRAD_NE; i += NT) {
            const int cc = i / GRAD_NE, e = i - cc * GRAD_NE;
            double s = 0.0;
#pragma unroll
            for (int gg = 0; gg < G; ++gg) s += s_acc[(size_t)(gg * C + cc) * GRAD_NE + e];
            a.part[((size_t)(col0 + cc) * a.nsplit + split) * GRAD_NE + e] = s;
        }
    }
}

// grad[c][e] = sum_p part[c][p][e], parts in index order from 0.0
__global__ void __launch_bounds__(256) rcm_grad_sum_kernel(int ncol, int npart, const double* __restrict__ part, double* grad) {
    const size_t n = (size_t)ncol * GRAD_NE;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / GRAD_NE, e = i - c * GRAD_NE;
        const double* p = part + c * npart * GRAD_NE + e;
        double s = 0.0;
        for (int k = 0; k < npart; ++k) s += p[(size_t)k * GRAD_NE];
        grad[i] = s;
    }
}
