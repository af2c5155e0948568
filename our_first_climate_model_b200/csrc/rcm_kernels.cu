// Hand-written sm_100a kernels of the radiative-convective column solver.
//
// One fused kernel does a complete reference time step (main.cpp:531-583) per column:
//   K5a  theta-sort adjustment + water-vapour feedback + table indices     (main.cpp:536-540, :281-289,
//                                                                          repwvl_thermal.cpp:226-240)
//   K1   optical depth tau[lambda][layer]                                  (repwvl_thermal.cpp:197-248,
//                                                                          main.cpp:266-274)
//   K2   Planck source per wavelength and layer                            (main.cpp:186-204)
//   K3   30-angle Schwarzschild down/up recurrences                        (main.cpp:291-318)
//   K4   spectral + angular reduction to E_down, E_up, heating dE          (main.cpp:326-341)
//   K5b  adaptive time step, temperature update, surface temperature       (main.cpp:156-176)
//
// Mapping.  A CTA owns a tile of C consecutive columns for all fused steps.  Its threads are
// C columns x 2 halves x G wavelength groups: the lane pair (c, g) walks wavelengths g, g+G, ... of
// column c, one lane per half of the atmosphere, so lanes of a warp hold the same wavelength for
// consecutive columns (table rows and Planck constants are warp-uniform, per-column scalars come from
// shared memory without bank conflicts).  The vertical problem of one (column, wavelength, half) lives in
// registers: tau[10], source differences[10], two sets of transmissions[10], 20 flux accumulators.
// The path is FP64-pipe bound (DESIGN.md): no tensor cores, HBM traffic ~1.6 KB per column-step.
#include <cfloat>
#include <cstdio>

#include "rcm_kernels.cuh"
#include "rcm_diag.cuh"
#include "rcm_jac.cuh"
#include "rcm_fjac.cuh"
#include "rcm_fdh.cuh"
#include "rcm_lbl_diag.cuh"
#include "rcm_lbl_jac.cuh"

__constant__ DevConst cst;

cudaError_t rcm_upload_const(const DevConst& c) { return cudaMemcpyToSymbol(cst, &c, sizeof(DevConst)); }

namespace {

#include "rcm_device_math.cuh"
#include "rcm_step_kernel.cuh"

// Bilinear coefficients per LAYER, temperature interval and active species, in the reference's operation order
// (repwvl_thermal.cpp:235-238):  coef[(r*(nt-1)+it)][w][k] = {c0, cT, cP * delP_r, cPT}, r = pair-order layer row.
// The layer's pressure interval ip and its weight delP come from the shared pressure grid (constant bank), so the
// product cP * delP - one rounding in the reference too - is taken here once instead of once per column and step.
// src is the file-order table xsec[it][species][w][ip].
__global__ void rcm_coef_kernel(const double* __restrict__ src, double* __restrict__ dst, int nt, int ns, int nw,
                                int np, int nact, const int* __restrict__ species) {
    const size_t n = (size_t)NLAY * (nt - 1) * nw * nact;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        size_t r = i;
        const int k = r % nact; r /= nact;
        const int w = r % nw; r /= nw;
        const int it = r % (nt - 1); r /= (nt - 1);
        const int row = (int)r;                             // pair-order layer row
        const int l = row < HALF ? row : 29 - row;          // top-down layer
        const int ip = cst.ip[l];
        const int sp = species[k];
        auto X = [&](int b, int cc) { return src[(((size_t)b * ns + sp) * nw + w) * np + cc]; };
        const double c0 = X(it, ip);
        const double cT = __dsub_rn(X(it + 1, ip), c0);
        const double cP = __dsub_rn(X(it, ip + 1), c0);
        const double cPT = __dsub_rn(__dsub_rn(__dsub_rn(X(it + 1, ip + 1), cP), cT), c0);
        dst[4 * i + 0] = c0;
        dst[4 * i + 1] = cT;
        dst[4 * i + 2] = __dmul_rn(cP, cst.delP[row]);
        dst[4 * i + 3] = cPT;
    }
}

// The split path's rows: per (layer row, temperature interval, wavelength) 16 doubles = 128 bytes,
//   {c0 + cP*delP, cT, cPT} for each of the five species, one pad.
// Its K1 evaluates x = (c0 + cP*delP) + cT*dT + cPT*(dT*dP) with three FMAs per species (contracted: within 4 ulp of the
// reference's operation order, which rcm_build_tau / rcm_step_kernel keep bit for bit).
__global__ void rcm_coef3_kernel(const double* __restrict__ coef4, double* __restrict__ dst, size_t nrows) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nrows * 5; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / 5;
        const int k = (int)(i % 5);
        const double* c = coef4 + (row * 5 + k) * 4;
        double* d = dst + row * 16 + 3 * k;
        d[0] = __dadd_rn(c[0], c[2]);
        d[1] = c[1];
        d[2] = c[3];
        if (k == 4) dst[row * 16 + 15] = 0.0;
    }
}

// ------------------------------------------------------------------------------------------
// Per-step ensemble scalars from the per-column diagnostics.  RED_BLOCKS CTAs per step reduce fixed slices
// of the columns with a fixed-order tree into partial[step][block][4]; the CTA that finishes last (ticket
// counter, reset for the next launch) folds the partials in block order.  The result does not depend on
// scheduling.  out[step] = {sum toa, max dT, #converged, max|dE|} (layout of rcm_step_scalars).
// ------------------------------------------------------------------------------------------
constexpr int RED_BLOCKS = 64, RED_THREADS = 256;

__device__ __forceinline__ void red4(double& sum, double& mx, double& cnt, double& mde, double (*sh)[RED_THREADS / 32]) {
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        mde = fmax(mde, __shfl_xor_sync(0xffffffffu, mde, o));
    }
    const int w = threadIdx.x >> 5, ln = threadIdx.x & 31;
    __syncthreads();
    if (ln == 0) {
        sh[0][w] = sum; sh[1][w] = mx; sh[2][w] = cnt; sh[3][w] = mde;
    }
    __syncthreads();
    constexpr int NW = RED_THREADS / 32;
    sum = ln < NW ? sh[0][ln] : 0.0;
    mx = ln < NW ? sh[1][ln] : 0.0;
    cnt = ln < NW ? sh[2][ln] : 0.0;
    mde = ln < NW ? sh[3][ln] : 0.0;
    for (int o = NW / 2; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        mde = fmax(mde, __shfl_xor_sync(0xffffffffu, mde, o));
    }
}

__global__ void __launch_bounds__(RED_THREADS) rcm_reduce_diag_kernel(const double* __restrict__ diag, int ncol,
                                                                      double dT_conv, double* __restrict__ partial,
                                                                      unsigned* __restrict__ ticket,
                                                                      double* __restrict__ out) {
    __shared__ double sh[4][RED_THREADS / 32];
    __shared__ bool last;
    const int step = blockIdx.y, b = blockIdx.x;
    const double* d = diag + (size_t)step * ncol * 4;
    const int per = (ncol + RED_BLOCKS - 1) / RED_BLOCKS, lo = b * per, hi = min(ncol, lo + per);
    double sum = 0.0, mx = 0.0, cnt = 0.0, mde = 0.0;
    for (int i = lo + threadIdx.x; i < hi; i += RED_THREADS) {
        const double4 v = *reinterpret_cast<const double4*>(d + (size_t)i * 4);
        sum += v.x;
        mx = fmax(mx, v.y);
        cnt += (v.y < dT_conv) ? 1.0 : 0.0;
        mde = fmax(mde, v.z);
    }
    red4(sum, mx, cnt, mde, sh);
    if (threadIdx.x == 0) {
        double* pp = partial + ((size_t)step * RED_BLOCKS + b) * 4;
        pp[0] = sum; pp[1] = mx; pp[2] = cnt; pp[3] = mde;
        __threadfence();
        last = (atomicAdd(ticket + step, 1u) == RED_BLOCKS - 1);
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    sum = mx = cnt = mde = 0.0;
    if (threadIdx.x < 32) {  // 64 partials, two per lane, folded in block order by the fixed tree
        for (int k = threadIdx.x; k < RED_BLOCKS; k += 32) {
            const double* pp = partial + ((size_t)step * RED_BLOCKS + k) * 4;
            sum += pp[0];
            mx = fmax(mx, pp[1]);
            cnt += pp[2];
            mde = fmax(mde, pp[3]);
        }
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            mde = fmax(mde, __shfl_xor_sync(0xffffffffu, mde, o));
        }
        if (threadIdx.x == 0) {
            out[step * 4 + 0] = sum; out[step * 4 + 1] = mx; out[step * 4 + 2] = cnt; out[step * 4 + 3] = mde;
            ticket[step] = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------
// FP64-pipe microbenchmarks: the measured denominators of the roofline (DESIGN.md).  Each
// thread runs `iters` rounds of 8 independent dependency chains.
// ------------------------------------------------------------------------------------------
template <int WHICH>
__global__ void __launch_bounds__(256) rcm_microbench_kernel(double* out, long iters, const double* tab) {
    __shared__ double stab[EXP_TAB * EXP_REP];
    for (int i = threadIdx.x; i < EXP_TAB * EXP_REP; i += blockDim.x) stab[i] = tab[i / EXP_REP];
    __syncthreads();
    const unsigned tl = (unsigned)__cvta_generic_to_shared(stab + (threadIdx.x & (EXP_REP - 1)));
    double v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = -1.0 - 0.001 * (threadIdx.x + k);
    const double a = 0.999999, b = -1e-7;
    for (long i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (WHICH == 0) v[k] = fma(v[k], a, b);
            if (WHICH == 1) v[k] = exp(v[k]) - 1.5;
            if (WHICH == 2) v[k] = -1.0 / v[k] - 1.7;
            if (WHICH == 3) v[k] = exp_scaled<false>(v[k], L2E64, tl) - 1.5;
        }
    }
    double sacc = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) sacc += v[k];
    out[blockIdx.x * (size_t)blockDim.x + threadIdx.x] = sacc;
}

#include "rcm_lbl_kernels.cuh"
#include "rcm_lbl_diag_kernels.cuh"
#include "rcm_split_kernels.cuh"
#include "rcm_diag_kernels.cuh"
#include "rcm_jac_kernels.cuh"
#include "rcm_fjac_kernels.cuh"
#include "rcm_fdh_kernels.cuh"
#include "rcm_lbl_jac_kernels.cuh"

// ------------------------------------------------------------------------------------------
// Solar setup per column (SURVEY section 8(f)3): doubling_adding + solar_radiative_transfer_setup
// (main.cpp:214-264) with per-column cloud optical depth, zenith cosine and surface albedo.  One thread per
// column, the reference's operation order, no FMA contraction (explicit round-to-nearest intrinsics, IEEE
// division); pow(2, doublings) is an exact power of two, pow(t_dir, 2) the correctly rounded square.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rcm_solar_kernel(const SolarArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const double tau_s = a.tau_s_col ? a.tau_s_col[i] : a.tau_s;
    const double mu_s = a.mu_s_col ? a.mu_s_col[i] : a.mu_s;
    const double albedo = a.albedo_col ? a.albedo_col[i] : a.albedo;
    auto mul = [](double x, double y) { return __dmul_rn(x, y); };
    auto add = [](double x, double y) { return __dadd_rn(x, y); };
    auto sub = [](double x, double y) { return __dsub_rn(x, y); };
    auto dvd = [](double x, double y) { return __ddiv_rn(x, y); };
    const double tau = mul(sub(1.0, a.g_asym), tau_s);                       // main.cpp:216
    const double dtau = dvd(tau, scalbn(1.0, a.doublings));                  // :217
    const double thin = dvd(dtau, mu_s);
    double r = mul(0.5, thin), t = sub(1.0, r);                              // :223-224
    double r_dir = mul(thin, 0.5), s_dir = r_dir, t_dir = sub(1.0, thin);    // :225-227
    for (int k = 0; k < a.doublings; ++k) {                                  // :232-250
        const double denom = sub(1.0, mul(r, r));
        const double r2 = add(r, dvd(mul(mul(r, t), t), denom));
        const double t2 = dvd(mul(t, t), denom);
        const double s2 = add(dvd(add(mul(t, s_dir), mul(mul(mul(t_dir, r_dir), r), t)), denom), mul(t_dir, s_dir));
        const double rd2 = add(dvd(add(mul(mul(t, s_dir), r), mul(mul(t, t_dir), r)), denom), r_dir);
        t_dir = mul(t_dir, t_dir);
        s_dir = s2;
        r_dir = rd2;
        r = r2;
        t = t2;
    }
    // solar_radiative_transfer_setup, main.cpp:258-260
    const double r_total = add(r_dir, mul(mul(dvd(add(t_dir, s_dir), sub(1.0, mul(albedo, r))), t), albedo));
    if (a.r_total) a.r_total[i] = r_total;
    if (a.solar_irr) a.solar_irr[i] = mul(mul(mul(a.daytime, a.E_0), mu_s), sub(1.0, r_total));
    if (a.cloud_tau) a.cloud_tau[i] = dvd(tau_s, 2.0);                       // main.cpp:267
}

__global__ void __launch_bounds__(256) rcm_cplkavg_kernel(int n, const double* lo, const double* hi, const double* t,
                                                          double* out, const double* tab, int narrow) {
    __shared__ double stab[EXP_TAB * EXP_REP];
    for (int i = threadIdx.x; i < EXP_TAB * EXP_REP; i += blockDim.x) stab[i] = tab[i / EXP_REP];
    __syncthreads();
    const unsigned tl = (unsigned)__cvta_generic_to_shared(stab + (threadIdx.x & (EXP_REP - 1)));
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const double whi = 1.0E7 / lo[i], wlo = 1.0E7 / hi[i];
        const bool bin_ok = whi > wlo && wlo >= 0. && (whi - wlo) / whi < 1.e-2;
        out[i] = narrow ? cplkavg_narrow(lo[i], hi[i], whi, wlo, bin_ok, t[i], tl) : cplkavg_dev(lo[i], hi[i], t[i]);
    }
}

}  // namespace

size_t rcm_step_smem_bytes(int C, int nactive, int nthreads) {
#define RCM_SHAPE(CC, TT) \
    if (C == CC && nthreads == TT) return nactive == 5 ? Smem<CC, TT, 5>::bytes(5) : Smem<CC, TT, 0>::bytes(nactive);
    RCM_SHAPE(16, 128)
    RCM_SHAPE(8, 128)
    RCM_SHAPE(4, 128)
    RCM_SHAPE(32, 192)
    RCM_SHAPE(16, 96)
#undef RCM_SHAPE
    return 0;
}

template <int MODE, int NACT, int C, int NT>
static cudaError_t launch_t(const StepArgs& a, int nactive, int grid, cudaStream_t st) {
    const size_t smem = Smem<C, NT, NACT>::bytes(nactive);
    auto kern = a.clampk ? rcm_step_kernel<MODE, NACT, C, NT, true> : rcm_step_kernel<MODE, NACT, C, NT, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, NT, smem, st>>>(a);
    return cudaGetLastError();
}

template <int MODE>
static cudaError_t launch_m(const StepArgs& a, int nactive, int grid, cudaStream_t st) {
    const bool five = (nactive == 5);
#define RCM_SHAPE(CC, TT)                  \
    if (a.C == CC && a.nthreads == TT)     \
        return five ? launch_t<MODE, 5, CC, TT>(a, nactive, grid, st) : launch_t<MODE, 0, CC, TT>(a, nactive, grid, st);
    RCM_SHAPE(16, 128)
    RCM_SHAPE(8, 128)
    RCM_SHAPE(4, 128)
    RCM_SHAPE(32, 192)
    RCM_SHAPE(16, 96)
#undef RCM_SHAPE
    return cudaErrorInvalidValue;
}

cudaError_t rcm_launch_step(int mode, const StepArgs& a, int nactive, int grid, cudaStream_t st) {
    switch (mode) {
        case MODE_STEP: return launch_m<MODE_STEP>(a, nactive, grid, st);
        case MODE_TAU: return launch_m<MODE_TAU>(a, nactive, grid, st);
        case MODE_RT: return launch_m<MODE_RT>(a, nactive, grid, st);
    }
    return cudaErrorInvalidValue;
}

size_t rcm_split_tile_bytes() { return TILE_BYTES; }
size_t rcm_split_part_doubles() { return SPLIT_PART; }
int rcm_split_ipu() { return SPLIT_IPU; }

cudaError_t rcm_launch_split_col(const SplitArgs& a, const SplitColFlags& f, cudaStream_t st) {
    rcm_split_col_kernel<<<a.ntiles, SPLIT_COL_NT, 0, st>>>(a, f);
    return cudaGetLastError();
}

cudaError_t rcm_launch_split_rt(const SplitArgs& a, int grid, cudaStream_t st) {
    auto kern = a.clampk ? rcm_split_rt_kernel<true> : rcm_split_rt_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPLIT_SMEM);
    if (e != cudaSuccess) return e;
    kern<<<grid, SPLIT_NT, SPLIT_SMEM, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_split_multi(const SplitArgs& a, const SplitMultiArgs& m, int grid, cudaStream_t st) {
    auto kern = a.clampk ? rcm_split_multi_kernel<true> : rcm_split_multi_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPLIT_SMEM);
    if (e != cudaSuccess) return e;
    kern<<<grid, SPLIT_NT, SPLIT_SMEM, st>>>(a, m);
    return cudaGetLastError();
}

size_t rcm_reduce_scratch_doubles(int nsteps) { return (size_t)nsteps * RED_BLOCKS * 4; }

// scratch: rcm_reduce_scratch_doubles(capacity) doubles; ticket: one counter per step of the CAPACITY the buffers were
// allocated for, zeroed once at allocation (every launch leaves its counters at zero again).  The counters have their
// own allocation: placed behind the partials of the current nsteps they aliased the partials of an earlier, longer call.
cudaError_t rcm_launch_reduce_diag(const double* diag, int nsteps, int ncol, double dT_converged, double* scratch,
                                   unsigned* ticket, double* scalars, cudaStream_t st) {
    rcm_reduce_diag_kernel<<<dim3(RED_BLOCKS, nsteps), RED_THREADS, 0, st>>>(diag, ncol, dT_converged, scratch, ticket, scalars);
    return cudaGetLastError();
}

cudaError_t rcm_launch_coef(const double* xsec_file, double* coef, int nt, int ns, int nw, int np, int nact,
                            const int* d_species, cudaStream_t st) {
    rcm_coef_kernel<<<296, 256, 0, st>>>(xsec_file, coef, nt, ns, nw, np, nact, d_species);
    return cudaGetLastError();
}

cudaError_t rcm_launch_coef3(const double* coef4, double* coef3, size_t nrows, cudaStream_t st) {
    rcm_coef3_kernel<<<296, 256, 0, st>>>(coef4, coef3, nrows);
    return cudaGetLastError();
}

cudaError_t rcm_launch_microbench(int which, double* out, const double* tab, long iters, int grid,
                                  cudaStream_t st) {
    switch (which) {
        case 0: rcm_microbench_kernel<0><<<grid, 256, 0, st>>>(out, iters, tab); break;
        case 1: rcm_microbench_kernel<1><<<grid, 256, 0, st>>>(out, iters, tab); break;
        case 2: rcm_microbench_kernel<2><<<grid, 256, 0, st>>>(out, iters, tab); break;
        case 3: rcm_microbench_kernel<3><<<grid, 256, 0, st>>>(out, iters, tab); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t rcm_launch_solar(const SolarArgs& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    rcm_solar_kernel<<<(a.n + 127) / 128, 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_cplkavg(int n, const double* lo, const double* hi, const double* t, double* out,
                               const double* exp_tab, int narrow, cudaStream_t st) {
    rcm_cplkavg_kernel<<<148, 256, 0, st>>>(n, lo, hi, t, out, exp_tab, narrow);
    return cudaGetLastError();
}

size_t rcm_lbl_smem_bytes(int C, int nthreads) {
    return ((size_t)EXP_TAB * EXP_REP + (size_t)TBD_LEN * 3 + 2 * C + (size_t)HALF * nthreads +
            (size_t)NLEV * (nthreads / 2)) * sizeof(double);
}

cudaError_t rcm_launch_lbl_prep(const LblArgs& a, cudaStream_t st) {
    rcm_lbl_prep_kernel<<<(a.ncol + 127) / 128, 128, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_lbl_rt(const LblArgs& a, cudaStream_t st, cudaEvent_t ev0, cudaEvent_t ev1) {
    constexpr int C = RCM_LBL_C, NT = RCM_LBL_NT;
    const size_t smem = rcm_lbl_smem_bytes(C, NT);
    auto kern = a.clampk ? rcm_lbl_rt_kernel<C, NT, true> : rcm_lbl_rt_kernel<C, NT, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (ev0) cudaEventRecord(ev0, st);
    kern<<<a.ntiles * a.nchunks, NT, smem, st>>>(a);
    if (ev1) cudaEventRecord(ev1, st);
    return cudaGetLastError();
}

cudaError_t rcm_launch_lbl_finish(const LblArgs& a, cudaStream_t st) {
    rcm_lbl_finish_kernel<<<a.ncol, LBL_FIN_NT, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_lbl_step(const LblArgs& a, cudaStream_t st, cudaEvent_t ev0, cudaEvent_t ev1) {
    cudaError_t e = rcm_launch_lbl_prep(a, st);
    if (e == cudaSuccess) e = rcm_launch_lbl_rt(a, st, ev0, ev1);
    if (e == cudaSuccess) e = rcm_launch_lbl_finish(a, st);
    return e;
}

cudaError_t rcm_launch_lbl_scale(const LblArgs& a, double f_h2o, double f_o3, cudaStream_t st) {
    rcm_lbl_scale_kernel<<<(a.ncol * NLAY + 127) / 128, 128, 0, st>>>(a, f_h2o, f_o3);
    return cudaGetLastError();
}

cudaError_t rcm_launch_lbl_plane(const double* raw, size_t n, double f_co2x, double f_ch4, double f_n2o, double* out, cudaStream_t st) {
    rcm_lbl_plane_kernel<<<296, 256, 0, st>>>(raw, n, f_co2x, f_ch4, f_n2o, out);
    return cudaGetLastError();
}

size_t rcm_lbl_band_smem_bytes() {
    return rcm_lbl_smem_bytes(RCM_LBL_C, RCM_LBL_NT) + (size_t)NLEV * (RCM_LBL_NT / 2) * sizeof(double);
}

cudaError_t rcm_launch_lbl_band(const LblArgs& a, double* spec_dn, double* spec_up, cudaStream_t st) {
    constexpr int C = RCM_LBL_C, NT = RCM_LBL_NT;
    const size_t smem = rcm_lbl_band_smem_bytes();
    auto kern = a.clampk ? rcm_lbl_band_kernel<C, NT, true> : rcm_lbl_band_kernel<C, NT, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<a.ntiles * a.nchunks, NT, smem, st>>>(a, spec_dn, spec_up);
    return cudaGetLastError();
}

cudaError_t rcm_launch_lbl_band_sum(int ncol, int nwvl, int nband, const int* band_start, const double* spec_dn,
                                    const double* spec_up, double* band_dn, double* band_up, cudaStream_t st) {
    const size_t blocks = ((size_t)ncol * nband * NLEV + 255) / 256;
    rcm_lbl_band_sum_kernel<<<blocks < 4096 ? (int)blocks : 4096, 256, 0, st>>>(ncol, nwvl, nband, band_start, spec_dn, spec_up,
                                                                                band_dn, band_up);
    return cudaGetLastError();
}

cudaError_t rcm_launch_diag_scale(unsigned char* tile, int ntiles, const DiagScale& sc, cudaStream_t st) {
    rcm_diag_scale_kernel<<<296, 256, 0, st>>>(tile, ntiles, sc);
    return cudaGetLastError();
}

cudaError_t rcm_launch_diag_rt(const DiagArgs& a, int grid, cudaStream_t st) {
    auto kern = a.clampk ? rcm_diag_rt_kernel<true> : rcm_diag_rt_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DIAG_SMEM);
    if (e != cudaSuccess) return e;
    kern<<<grid, DIAG_NT, DIAG_SMEM, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_diag_sum(const DiagArgs& a, cudaStream_t st) {
    rcm_diag_sum_kernel<<<(a.ncol + DIAG_SUM_COLS - 1) / DIAG_SUM_COLS, 128, 0, st>>>(a);
    return cudaGetLastError();
}

int rcm_jac_ctas_per_sm() { return JAC_CTAS; }

cudaError_t rcm_launch_jac_rt(const JacArgs& a, int grid, cudaStream_t st) {
    auto kern = a.clampk ? rcm_jac_rt_kernel<true> : rcm_jac_rt_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)JAC_SMEM);
    if (e != cudaSuccess) return e;
    kern<<<grid, JAC_NT, JAC_SMEM, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_jac_sum(const JacArgs& a, cudaStream_t st) {
    const size_t blocks = ((size_t)a.ncol * JAC_NK + 255) / 256;
    const int grid = blocks < 4096 ? (int)blocks : 4096;
    rcm_jac_sum_kernel<<<grid, 256, 0, st>>>(a);
    return cudaGetLastError();
}

int rcm_fjac_ctas_per_sm() { return FJAC_CTAS; }

cudaError_t rcm_launch_fjac(const FjacArgs& a, cudaStream_t st) {
    auto kern = a.clampk ? rcm_fjac_kernel<true> : rcm_fjac_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FJAC_SMEM);
    if (e != cudaSuccess) return e;
    kern<<<(a.ncol + FJAC_WARPS - 1) / FJAC_WARPS, FJAC_NT, FJAC_SMEM, st>>>(a);
    return cudaGetLastError();
}

size_t rcm_lbl_jac_smem_bytes() {
    constexpr int C = RCM_LBL_C, NT = RCM_LBL_NT;
    return ((size_t)EXP_TAB * EXP_REP + 3 * TBD_LEN + 2 * C + 2 * (HALF + 1) * NT + (size_t)(NT / (2 * C)) * C * JAC_NK) *
           sizeof(double);
}

cudaError_t rcm_launch_lbl_jac(const LblArgs& a, double wtau, double* K_spec, cudaStream_t st) {
    constexpr int C = RCM_LBL_C, NT = RCM_LBL_NT;
    const size_t smem = rcm_lbl_jac_smem_bytes();
    auto kern = a.clampk ? rcm_lbl_jac_kernel<C, NT, true> : rcm_lbl_jac_kernel<C, NT, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<a.ntiles * a.nchunks, NT, smem, st>>>(a, wtau, K_spec);
    return cudaGetLastError();
}

cudaError_t rcm_launch_lbl_jac_band_sum(int ncol, int nwvl, int nband, const int* band_start, const double* K_spec, double* K_band,
                                        cudaStream_t st) {
    const size_t blocks = ((size_t)ncol * nband * JAC_NK + 255) / 256;
    rcm_lbl_jac_band_sum_kernel<<<blocks < 4096 ? (int)blocks : 4096, 256, 0, st>>>(ncol, nwvl, nband, band_start, K_spec, K_band);
    return cudaGetLastError();
}

cudaError_t rcm_launch_fdh_retemper(const FdhArgs& a, cudaStream_t st) {
    rcm_fdh_retemper_kernel<<<(a.ncol * NLAY + 255) / 256, 256, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_fdh_check(const FdhArgs& a, cudaStream_t st) {
    rcm_fdh_check_kernel<<<(a.ncol + FDH_CHECK_NT - 1) / FDH_CHECK_NT, FDH_CHECK_NT, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t rcm_launch_fdh_newton(const FdhArgs& a, cudaStream_t st) {
    rcm_fdh_newton_kernel<<<(a.ncol + FDH_NEWTON_WARPS - 1) / FDH_NEWTON_WARPS, FDH_NEWTON_NT, 0, st>>>(a);
    return cudaGetLastError();
}
