// rcm_lbl_jac_kernels.cuh - radiative kernels of the line-by-line path (rcm_lbl_radiative_kernels): the analytic derivatives
// of the OLR (E_up[0]) and the surface downward flux (E_down[20]) with respect to every layer's temperature, the surface
// temperature and every layer's ln(H2O VMR), per (column, wavelength).  Included by rcm_kernels.cu inside its anonymous
// namespace, after rcm_lbl_kernels.cuh (cplkavg_narrow, cplkavg_dev) and rcm_jac_kernels.cuh (jac_sweep_item).
//
// LBL optical depth does not depend on temperature (tables at fixed T): d/dT acts through the band Planck source alone, and
// d/dln q_l through tau_H2O,l x s_H2O,l.
//   cplkavg_narrow_dT            (B, dB/dT) of one bin: B bit for bit cplkavg_narrow's, dB/dT from the same exponentials
//   rcm_lbl_jac_kernel           the CTAs, tau and clamp of rcm_lbl_band_kernel, then the tangent sweep (jac_sweep_item) and
//                                the chain rule once per wavelength; the 82 values of each (column, wavelength) leave through
//                                shared memory as contiguous [col][w][2][41] rows
//   rcm_lbl_jac_band_sum_kernel  a band = the sum of its wavelengths' rows in index order, from 0.0 (the broadband K is the
//                                one band {0, nwvl})
// Every value is a function of its column alone.
#pragma once

constexpr int LBL_JAC_CTAS = 2;

// ------------------------------------------------------------------------------------------
// dB/dT of the band Planck source, K = sigma/pi x 15/pi^4, f(x) = x^3 / (e^x - 1), v = c2 nu / T:
//  * Simpson branch: B = K T^4 S_n[f] with abscissae x_k = c2 nu_k / T, so dx_k/dT = -x_k / T and, since x f'(x) = 3 f - g,
//      dB/dT = K T^3 S_n[g],   g(x) = x^4 e^x / (e^x - 1)^2 = f x e / (e - 1),
//    Simpson's rule on the same abscissae, exponentials and n at which B's convergence test stopped: the exact derivative of
//    the Simpson value B at fixed n (not of a different integral).
//  * every other branch (wide bins, the series of cplkavg_dev): B = K T^4 (integral of f from v0 to v1), so
//      dB/dT = 4 B / T - K T^3 (v1 f(v1) - v0 f(v0)), an overflowing exp giving a term of 0.
//  * T < 1e-4: B = 0 and dB/dT = 0.
// ------------------------------------------------------------------------------------------
__device__ __noinline__ double2 cplkavg_dev_dT(double wvllo, double wvlhi, double t) {
    const double B = cplkavg_dev(wvllo, wvlhi, t);
    if (t < 1.e-4) return make_double2(B, 0.0);
    const double c2 = 1.438786, sigma = 5.67032E-8, pi = 3.14159265358979323846;
    const double sigdpi = sigma / pi, conc = 15. / (pi * pi * pi * pi);
    const double whi = 1.0E7 / wvllo, wlo = 1.0E7 / wvlhi;
    const double v0 = c2 * wlo / t, v1 = c2 * whi / t;
    auto vf = [](double v) { return v > 0.0 ? (v * v) * (v * v) / expm1(v) : 0.0; };  // v f(v); exp overflow: v^4 / inf = 0
    return make_double2(B, 4.0 * B / t - sigdpi * (t * t * t) * conc * (vf(v1) - vf(v0)));
}

// cplkavg_narrow restated with g next to f: every operation of B is the one cplkavg_narrow performs, in the same order.
__device__ __forceinline__ double2 cplkavg_narrow_dT(double wvllo, double wvlhi, double whi, double wlo, bool bin_ok, double t,
                                                     unsigned tab_lane) {
    const double c2 = 1.438786, sigma = 5.67032E-8, pi = 3.14159265358979323846;
    const double vmax = 709.782712893384, sigdpi = sigma / pi, conc = 15. / (pi * pi * pi * pi);
    const double v0 = div_fast(c2 * wlo, t), v1 = div_fast(c2 * whi, t);
    if (!(bin_ok && t >= 1.e-4 && v0 > DBL_EPSILON && v1 < vmax)) return cplkavg_dev_dT(wvllo, wvlhi, t);
    // f(x) with e = exp(x), and g(x) = f x e / (e - 1) into gx
    auto fg = [&](double x, double e, double& gx) {
        const double fx = div_fast(x * x * x, e - 1.);
        gx = div_fast(fx * x * e, e - 1.);
        return fx;
    };
    auto f = [&](double x, double& gx) { return fg(x, exp_scaled<false>(x, L2E64, tab_lane), gx); };
    const double hh = v1 - v0;
    const double t4 = (t * t) * (t * t);
    const double del1 = hh * 0.5, del2 = hh * 0.25;
    const double x1 = v0 + del2, x2 = v0 + del1, x3 = v0 + 3.0 * del2;
    double fa, fb, fm, fq1, fq3, ga, gb, gm, gq1, gq3;
    if (v0 >= 0.25) {
        const double e0 = exp_scaled<false>(v0, L2E64, tab_lane), r = exp_scaled<false>(del2, L2E64, tab_lane);
        const double e1 = e0 * r, e2 = e1 * r, e3 = e2 * r, e4 = e3 * r;
        fa = fg(v0, e0, ga); fq1 = fg(x1, e1, gq1); fm = fg(x2, e2, gm); fq3 = fg(x3, e3, gq3); fb = fg(v1, e4, gb);
    } else {
        fa = f(v0, ga); fq1 = f(x1, gq1); fm = f(x2, gm); fq3 = f(x3, gq3); fb = f(v1, gb);
    }
    const double ends = fa + fb, gends = ga + gb;
    const double k3 = sigdpi * ((t * t) * t) * conc;
    double prev = (ends + 4.0 * fm) * (del1 * (1. / 3.));
    double val = (((ends + 4.0 * fq1) + 2.0 * fm) + 4.0 * fq3) * (del2 * (1. / 3.));
    double sg = (((gends + 4.0 * gq1) + 2.0 * gm) + 4.0 * gq3) * (del2 * (1. / 3.));
    if (fabs(val - prev) <= 1.e-6 * fabs(val)) return make_double2(sigdpi * t4 * conc * val, k3 * sg);
    prev = val;
    for (int n = 3; n <= 10; ++n) {
        const double del = hh / (2 * n);
        val = ends;
        sg = gends;
        for (int k = 1; k <= 2 * n - 1; ++k) {
            double gx;
            const double fx = f(v0 + (double)k * del, gx);
            val += (double)(2 * (1 + k % 2)) * fx;
            sg += (double)(2 * (1 + k % 2)) * gx;
        }
        val *= del * (1. / 3.);
        sg *= del * (1. / 3.);
        if (fabs((val - prev) / val) <= 1.e-6) break;
        prev = val;
    }
    return make_double2(sigdpi * t4 * conc * val, k3 * sg);
}

// ------------------------------------------------------------------------------------------
// One CTA per (16-column tile, 128-wavelength chunk), lanes as rcm_lbl_rt_kernel (h = 0: layers 0..9, h = 1: layers 19..10,
// G = 4 wavelength groups).  Per wavelength: tau as the step (the same FMAs on tau3, cloud and clamp), a live bit per owned
// layer (no clamp acted on its tau; else its ln q derivatives are 0), (B, dB/dT) of the ten layers and the surface in a
// ROLLED loop through shared memory (inlined eleven times the kernel's instruction fetch would stall, as the rt kernel's did),
// jac_sweep_item with wtau = 2 pi / nangle, then
//   o[oa + l] = aB_l dB_l,  o[oa + 21 + l] = -aT_l dtau_l/dln q_l,  o[ob + ...] likewise with bB, bT,
//   o[20] = aS dB_s (the OLR sees the surface through the whole atmosphere), o[41 + 20] = 0 (a black surface)
// with dtau_l/dln q_l = tau_H2O,l x s_H2O,l and oa / ob the output offsets of rcm_jac_rt_kernel.
// ------------------------------------------------------------------------------------------
template <int C, int NT, bool CLAMPK>
__global__ void __launch_bounds__(NT, LBL_JAC_CTAS) rcm_lbl_jac_kernel(const LblArgs a, double wtau, double* K_spec) {
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
    double* s_B = p;   p += (HALF + 1) * NT;  // [11][NT] B of the thread's ten layers, then of the surface
    double* s_dB = p;  p += (HALF + 1) * NT;  // [11][NT] their dB/dT
    double* s_out = p;                        // [G][C][2][41] of one round
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
        double aB[HALF], aT[HALF], bB[HALF], bT[HALF], aS = 0.0;
#pragma unroll
        for (int j = 0; j < HALF; ++j) aB[j] = aT[j] = bB[j] = bT[j] = 0.0;
        jac_sweep_item<CLAMPK>(tau, Bo, real ? Bsurf : 0.0, h, tab_lane, wtau, aB, aT, bB, bT, aS);
        double* o = s_out + (size_t)(g * C + c) * JAC_NK;
        const int oa = h * JAC_NE, ob = (1 - h) * JAC_NE;
#pragma unroll
        for (int j = 0; j < HALF; ++j) {
            const int l = h ? (NLAY - 1 - j) : j;
            const double dB = s_dB[j * NT + tid];
            const double dtdq = ((live >> j) & 1u) ? __ldg(t3 + l) * s_sH[sb + j * C] : 0.0;
            o[oa + l] = aB[j] * dB;
            o[oa + NLAY + 1 + l] = -aT[j] * dtdq;
            o[ob + l] = bB[j] * dB;
            o[ob + NLAY + 1 + l] = -bT[j] * dtdq;
        }
        if (h == 0) o[NLAY] = aS * s_dB[HALF * NT + tid];
        else o[JAC_NE + NLAY] = 0.0;
        __syncthreads();
        // the round's wavelengths w0 .. w0 + nw - 1 are consecutive: per column one run of nw * 82 doubles
        const int w0 = w_lo + item * G, nw = min(G, a.nwvl - w0), run = nw * JAC_NK;
        for (int i = tid; i < ncl * run; i += NT) {
            const int cc = i / run, k = i - cc * run, gg = k / JAC_NK, e = k - gg * JAC_NK;
            K_spec[((size_t)(col0 + cc) * a.nwvl + w0) * JAC_NK + k] = s_out[(size_t)(gg * C + cc) * JAC_NK + e];
        }
        __syncthreads();
    }
}

// one thread per (column, band, entry): K_band [ncol][nband][2][41]
__global__ void __launch_bounds__(256) rcm_lbl_jac_band_sum_kernel(int ncol, int nwvl, int nband, const int* __restrict__ band_start,
                                                                   const double* __restrict__ K_spec, double* K_band) {
    const size_t n = (size_t)ncol * nband * JAC_NK;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int e = (int)(i % JAC_NK);
        const size_t cb = i / JAC_NK;
        const int b = (int)(cb % nband);
        const double* row = K_spec + (cb / nband) * nwvl * JAC_NK + e;
        double sum = 0.0;
        for (int w = band_start[b]; w < band_start[b + 1]; ++w) sum += row[(size_t)w * JAC_NK];
        K_band[i] = sum;
    }
}
