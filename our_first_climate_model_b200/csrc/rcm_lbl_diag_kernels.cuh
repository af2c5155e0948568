// rcm_lbl_diag_kernels.cuh - the diagnostic radiation call of the line-by-line path (rcm_lbl_diagnose_fluxes).
// Included by rcm_kernels.cu inside its anonymous namespace, after rcm_lbl_kernels.cuh (cplkavg_narrow, the LBL tile layout)
// and rcm_step_kernel.cuh (sweep_item).
#pragma once

// ------------------------------------------------------------------------------------------
// The broadband fluxes come from the three step kernels
// above on scratch copies of a chunk; the kernels below add the species factors and the band-resolved fluxes.
//   rcm_lbl_scale_kernel     sH / sO of the prep from the VMRs times a factor: (f x vmr) / ref, one rounded multiplication in
//                            front of the prep's division (f = 1 gives the prep's values bit for bit)
//   rcm_lbl_plane_kernel     the column-independent plane of rcm_set_lbl_tables with a factor on each of its species:
//                            ((f_CO2 x co2_factor) x CO2 + f_CH4 x CH4) + f_N2O x N2O, left to right, no contraction
//   rcm_lbl_band_kernel      the CTAs, tau, Planck source and sweeps of rcm_lbl_rt_kernel, but the accumulators start at zero
//                            for every wavelength and the 42 level values of each (column, wavelength) leave through shared
//                            memory as contiguous [col][w][21] rows of E_down and E_up
//   rcm_lbl_band_sum_kernel  a band = the sum of its wavelengths' rows in index order, from 0.0
// Every value is a function of its column alone.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rcm_lbl_scale_kernel(const LblArgs a, double f_h2o, double f_o3) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.ncol * NLAY) return;
    const int col = i / NLAY, l = i - col * NLAY;
    const double* v = a.vmr + (size_t)col * a.nact * NLAY + l;
    a.sH[i] = __dmul_rn(f_h2o, v[a.h2o_slot * NLAY]) / a.h2o_ref[l];
    a.sO[i] = a.o3_ref ? __dmul_rn(f_o3, v[a.o3_slot * NLAY]) / a.o3_ref[l] : f_o3;
}

// raw [3][n]: CO2, CH4, N2O; f_co2x = f_CO2 x co2_factor
__global__ void __launch_bounds__(256) rcm_lbl_plane_kernel(const double* __restrict__ raw, size_t n, double f_co2x, double f_ch4,
                                                            double f_n2o, double* __restrict__ out) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = __dadd_rn(__dadd_rn(__dmul_rn(f_co2x, raw[i]), __dmul_rn(f_ch4, raw[n + i])), __dmul_rn(f_n2o, raw[2 * n + i]));
}

template <int C, int NT, bool CLAMPK>
__global__ void __launch_bounds__(NT, 384 / NT) rcm_lbl_band_kernel(const LblArgs a, double* spec_dn, double* spec_up) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int G = NT / (2 * C);
    double* p = reinterpret_cast<double*>(smem_raw);
    double* s_tab = p; p += EXP_TAB * EXP_REP;
    static_assert(C == 16, "tbd() is laid out for 16-column tiles");
    double* s_T = p;   p += TBD_LEN;
    double* s_sH = p;  p += TBD_LEN;
    double* s_sO = p;  p += TBD_LEN;
    double* s_Ts = p;  p += C;
    double* s_cl = p;  p += C;
    double* s_B = p;   p += HALF * NT;
    double* s_out = p;  // [G][C][E_down 21 | E_up 21] of one round
    const int tid = threadIdx.x, lane = tid & 31;
    const int h = tid & 1, q = tid >> 1, c = q % C, g = q / C;
    const int sb = tbd(h * HALF, c);
    for (int i = tid; i < EXP_TAB * EXP_REP; i += NT) s_tab[i] = a.exp_tab[i / EXP_REP];
    const unsigned tab_lane = (unsigned)__cvta_generic_to_shared(s_tab + (lane & (EXP_REP - 1)));
    const int tile = blockIdx.x % a.ntiles, chunk = blockIdx.x / a.ntiles;
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
    __syncthreads();

    const int w_lo = chunk * a.chunk_len;
    const int tau_clamp_hi = __double2hiint(a.tau_clamp);
    const size_t plane = (size_t)a.nwvl * NLAY;
#pragma unroll 1
    for (int item = 0; item < a.chunk_len / G; ++item) {
        const int w_any = w_lo + g + item * G;
        const bool real = w_any < a.nwvl;  // a group beyond the table runs the last wavelength with a zero source, unwritten
        const int w = real ? w_any : a.nwvl - 1;
        double tau[HALF], Bo[HALF], E1[HALF], E2[HALF], Eu20 = 0.0;
#pragma unroll
        for (int j = 0; j < HALF; ++j) E1[j] = E2[j] = 0.0;
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
        }
#pragma unroll 1
        for (int j = 0; j < HALF; ++j) s_B[j * NT + tid] = cplkavg_narrow(lo, hi, whi, wlo, bin_ok, s_T[sb + j * C], tab_lane);
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            const double B = s_B[j * NT + tid];
            Bo[j] = real ? B : 0.0;
        }
        const double Bsurf = cplkavg_narrow(lo, hi, whi, wlo, bin_ok, s_Ts[c], tab_lane);
        sweep_item<CLAMPK>(tau, Bo, real ? Bsurf : 0.0, h, tab_lane, E1, E2, Eu20);
        // the pair's 42 values in level order: E_down[0..20], then E_up[0..20] (the rows rcm_lbl_rt_kernel writes to part)
        double* o = s_out + (size_t)(g * C + c) * 2 * NLEV;
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            const int l = h ? (NLAY - 1 - j) : j;
            o[l + 1] = h ? E2[j] : E1[j];
            o[NLEV + l] = h ? E1[j] : E2[j];
        }
        if (h) o[NLEV + NLAY] = Eu20;
        else o[0] = 0.0;
        __syncthreads();
        // the round's wavelengths w0 .. w0 + nw - 1 are consecutive: per column one run of nw * 21 doubles in each array
        const int w0 = w_lo + item * G, nw = min(G, a.nwvl - w0), run = nw * NLEV;
        for (int i = tid; i < ncl * run; i += NT) {
            const int cc = i / run, k = i - cc * run, gg = k / NLEV, lev = k - gg * NLEV;
            const double* so = s_out + (size_t)(gg * C + cc) * 2 * NLEV;
            const size_t gi = ((size_t)(col0 + cc) * a.nwvl + w0) * NLEV + k;
            spec_dn[gi] = so[lev];
            spec_up[gi] = so[NLEV + lev];
        }
        __syncthreads();
    }
}

// one thread per (column, band, level): out [ncol][nband][21]
__global__ void __launch_bounds__(256) rcm_lbl_band_sum_kernel(int ncol, int nwvl, int nband, const int* __restrict__ band_start,
                                                               const double* __restrict__ spec_dn, const double* __restrict__ spec_up,
                                                               double* band_dn, double* band_up) {
    const size_t n = (size_t)ncol * nband * NLEV;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int lev = (int)(i % NLEV);
        const size_t cb = i / NLEV;
        const int b = (int)(cb % nband);
        const size_t base = (cb / nband) * nwvl * NLEV + lev;
        double sd = 0.0, su = 0.0;
        for (int w = band_start[b]; w < band_start[b + 1]; ++w) {
            sd += spec_dn[base + (size_t)w * NLEV];
            su += spec_up[base + (size_t)w * NLEV];
        }
        band_dn[i] = sd;
        band_up[i] = su;
    }
}
