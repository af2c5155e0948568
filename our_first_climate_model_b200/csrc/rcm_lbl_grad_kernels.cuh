// rcm_lbl_grad_kernels.cuh - adjoint flux gradients of the line-by-line path (rcm_lbl_flux_gradient), of the state
// rcm_lbl_prep_kernel (and rcm_lbl_scale_kernel) prepared.  Included by rcm_kernels.cu inside its anonymous namespace, after
// rcm_lbl_jac_kernels.cuh (cplkavg_narrow_dT) and rcm_grad_kernels.cuh (grad_sweep_item, grad_load_co).
//
//   rcm_lbl_grad_kernel  rcm_lbl_jac_kernel's lanes, tau, clamp and rolled Planck loop on one CTA per (16-column tile,
//                        GRAD_LBL_SPAN-wavelength span), grad_sweep_item in place of jac_sweep_item, and the chain rule once
//                        per wavelength into per-thread sums in shared memory; the span's partial is the sum over the 4
//                        wavelength groups in group order.  rcm_grad_sum_kernel then sums the spans in index order.
// d/dT_l acts through layer l's Planck source alone (LBL tau does not depend on T); dtau_l/dln x_{s,l} is species s's share of
// tau_l as rcm_lbl_species_fjac_kernel takes it (one rounded product each), 0 where the clamp acts.  Summation order of an
// entry: the wavelengths g, g + 4, ... of a span per group g, the groups 0..3, the spans in index order: fixed by the table.
#pragma once

// ------------------------------------------------------------------------------------------
template <int C, int NT, bool CLAMPK>
__global__ void __launch_bounds__(NT, LBL_JAC_CTAS) rcm_lbl_grad_kernel(const LblArgs a, double wtau, const double* __restrict__ raw,
                                                                        double f_co2x, double f_ch4, double f_n2o,
                                                                        const double* __restrict__ co, double* part) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int G = NT / (2 * C);
    static_assert(GRAD_LBL_SPAN % G == 0, "a span is whole rounds of G wavelengths");
    double* p = reinterpret_cast<double*>(smem_raw);
    double* s_tab = p; p += EXP_TAB * EXP_REP;
    static_assert(C == 16, "tbd() is laid out for 16-column tiles");
    double* s_T = p;   p += TBD_LEN;
    double* s_sH = p;  p += TBD_LEN;
    double* s_sO = p;  p += TBD_LEN;
    double* s_Ts = p;  p += C;
    double* s_cl = p;  p += C;
    double* s_B = p;   p += (HALF + 1) * NT;  // [11][NT] B of the thread's ten layers, then of the surface
    double* s_dB = p;  p += (HALF + 1) * NT;  // [11][NT] their dB/dT
    double* s_acc = p;                        // [G][C][121] per-thread sums
    const int tid = threadIdx.x, lane = tid & 31;
    const int h = tid & 1, q = tid >> 1, c = q % C, g = q / C;
    const int sb = tbd(h * HALF, c);
    for (int i = tid; i < EXP_TAB * EXP_REP; i += NT) s_tab[i] = a.exp_tab[i / EXP_REP];
    const unsigned tab_lane = (unsigned)__cvta_generic_to_shared(s_tab + (lane & (EXP_REP - 1)));
    const int nspan = (a.nwvl + GRAD_LBL_SPAN - 1) / GRAD_LBL_SPAN;
    const int tile = blockIdx.x % a.ntiles, span = blockIdx.x / a.ntiles;
    const int col0 = tile * C, ncl = min(C, a.ncol - col0);
    for (int i = tid; i < NLAY * C; i += NT) {
        const int l = i / C, cc = i % C, r = tbd(prow(l), cc);
        const bool ok = cc < ncl;
        const size_t gi = (size_t)(col0 + cc) * NLAY + l;
        s_T[r] = ok ? a.Tlayer[gi] : 250.0;
        s_sH[r] = ok ? a.sH[gi] : 1.0;
        s_sO[r] = ok ? a.sO[gi] : 1.0;
    }
    if (tid < C) {
        s_Ts[tid] = (tid < ncl) ? a.Tsurf[col0 + tid] : 250.0;
        s_cl[tid] = a.cloud_col ? a.cloud_col[col0 + (tid < ncl ? tid : 0)] : cst.cloud_tau;
    }
    for (int i = tid; i < G * C * GRAD_NE; i += NT) s_acc[i] = 0.0;
    __syncthreads();
    double* const acc = s_acc + (size_t)(g * C + c) * GRAD_NE;  // this thread's sums (its own entries only)
    double cA[HALF + 1], cB[HALF];
    grad_load_co(co + (size_t)(col0 + (c < ncl ? c : 0)) * GRAD_NCO, h, cA, cB);

    const int w_lo = span * GRAD_LBL_SPAN;
    const int tau_clamp_hi = __double2hiint(a.tau_clamp);
    const size_t plane = (size_t)a.nwvl * NLAY;
#pragma unroll 1
    for (int item = 0; item < GRAD_LBL_SPAN / G; ++item) {
        const int w_any = w_lo + g + item * G;
        if (w_lo + item * G >= a.nwvl) break;  // (CTA-uniform) the last span's rounds beyond the table
        const bool real = w_any < a.nwvl;  // a group beyond the table runs the last wavelength with a zero source, unsummed
        const int w = real ? w_any : a.nwvl - 1;
        double tau[HALF], Bo[HALF];
        unsigned live = 0;  // bit j: no clamp acts on tau of owned layer j
        const double lo = __ldg(a.wvl_lo + w), hi = __ldg(a.wvl_hi + w);
        const double whi = __ldg(a.wn_hi + w), wlo = __ldg(a.wn_lo + w);
        const bool bin_ok = __ldg(a.bin_ok + w) != 0;
        const double* t3 = a.tau3 + (size_t)w * NLAY;
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            const int l = h ? (NLAY - 1 - j) : j;
            double v = fma(__ldg(t3 + l), s_sH[sb + j * C], fma(__ldg(t3 + plane + l), s_sO[sb + j * C], __ldg(t3 + 2 * plane + l)));
            v = fma(cst.cloud_w[h * HALF + j], s_cl[c], v);
            tau[j] = CLAMPK ? v : clamp_hi(v, tau_clamp_hi);
            live |= (tau[j] == v ? 1u : 0u) << j;
        }
#pragma unroll 1
        for (int j = 0; j <= HALF; ++j) {
            const double2 b = cplkavg_narrow_dT(lo, hi, whi, wlo, bin_ok, j < HALF ? s_T[sb + j * C] : s_Ts[c], tab_lane);
            s_B[j * NT + tid] = b.x;
            s_dB[j * NT + tid] = b.y;
        }
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            const double B = s_B[j * NT + tid];
            Bo[j] = real ? B : 0.0;
        }
        const double Bsurf = s_B[HALF * NT + tid];
        double gB[HALF], gT[HALF], gS = 0.0;
#pragma unroll
        for (int j = 0; j < HALF; ++j) gB[j] = gT[j] = 0.0;
        grad_sweep_item<CLAMPK>(tau, Bo, real ? Bsurf : 0.0, h, tab_lane, wtau, cA, cB, gB, gT, gS);
        if (!real) continue;
        const double* rw = raw + (size_t)w * NLAY;  // CO2, CH4, N2O
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            const int l = h ? (NLAY - 1 - j) : j;
            acc[l] = acc[l] + gB[j] * s_dB[j * NT + tid];
            if ((live >> j) & 1u) {
                double dts[SPJ_NS];
                dts[0] = __ldg(t3 + l) * s_sH[sb + j * C];
                dts[1] = __dmul_rn(f_co2x, __ldg(rw + l));
                dts[2] = __ldg(t3 + plane + l) * s_sO[sb + j * C];
                dts[3] = __dmul_rn(f_n2o, __ldg(rw + 2 * plane + l));
                dts[4] = __dmul_rn(f_ch4, __ldg(rw + plane + l));
#pragma unroll
                for (int k = 0; k < SPJ_NS; ++k) acc[NLEV + k * NLAY + l] = acc[NLEV + k * NLAY + l] + -gT[j] * dts[k];
            }
        }
        if (h == 1) acc[NLAY] = acc[NLAY] + gS * s_dB[HALF * NT + tid];  // the surface: Ub_20 lives in the bottom lane
    }
    __syncthreads();
    // the span's partial: per column and entry the sum over the groups in group order, from 0.0
    for (int i = tid; i < ncl * GRAD_NE; i += NT) {
        const int cc = i / GRAD_NE, e = i - cc * GRAD_NE;
        double s = 0.0;
#pragma unroll
        for (int gg = 0; gg < G; ++gg) s += s_acc[(size_t)(gg * C + cc) * GRAD_NE + e];
        part[((size_t)(col0 + cc) * nspan + span) * GRAD_NE + e] = s;
    }
}
