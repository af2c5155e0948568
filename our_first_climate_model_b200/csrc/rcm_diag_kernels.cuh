// rcm_diag_kernels.cuh - the diagnostic radiation call (rcm_diagnose_fluxes): K1-K4 per (column, wavelength) from tile
// blocks that the split path's prep (rcm_split_col_kernel) wrote into a scratch buffer, with every wavelength's fluxes
// kept apart.  Included by rcm_kernels.cu inside its anonymous namespace, after rcm_split_kernels.cuh (tile block layout,
// sweep_item, exp_scaled, div_fast).
//
//   rcm_diag_scale_kernel  the VMR rows of the tile blocks times one factor per active species (forcing experiments)
//   rcm_diag_rt_kernel     (tile, split) units as the unit kernel's, but the accumulators start at zero for every
//                          wavelength and the 42 level values of each (column, wavelength) leave through shared memory as
//                          contiguous [col][w][21] rows of E_down and E_up
//   rcm_diag_sum_kernel    broadband E_down / E_up = sum over the wavelengths in index order, then dE (main.cpp:337-341)
// Every value is a function of its column alone: no staged table rows (their candidate plan depends on the tile's other
// columns), no sum across columns.
#pragma once

constexpr int DIAG_NT = SPLIT_NT;
constexpr int DIAG_OUT = SPLIT_G * SPLIT_C * 2 * NLEV;  // doubles of one round's staged fluxes [group][column][E_down | E_up]
constexpr size_t DIAG_SMEM = (size_t)EXP_TAB * EXP_REP * 8 + TILE_BYTES + (size_t)DIAG_OUT * 8;

__global__ void __launch_bounds__(256) rcm_diag_scale_kernel(unsigned char* tile, int ntiles, const DiagScale sc) {
    constexpr int PER_TILE = NLAY * SPLIT_C;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)ntiles * PER_TILE; i += (size_t)gridDim.x * blockDim.x) {
        const int t = (int)(i / PER_TILE), r = (int)(i % PER_TILE) / SPLIT_C, cc = (int)(i % SPLIT_C);
        double* v = reinterpret_cast<double*>(tile + (size_t)t * TILE_BYTES) + TB_VMR + tbd(r, cc);
#pragma unroll
        for (int sp = 0; sp < 5; ++sp) v[sp * TBD_LEN] = __dmul_rn(v[sp * TBD_LEN], sc.f[sp]);
    }
}

template <bool CLAMPK>
__global__ void __launch_bounds__(DIAG_NT, 3) rcm_diag_rt_kernel(const DiagArgs a) {
    constexpr int C = SPLIT_C, NT = DIAG_NT, G = SPLIT_G;
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

    for (int unit = blockIdx.x; unit < a.nunits; unit += gridDim.x) {
        const int tile = unit / a.nsplit, split = unit - tile * a.nsplit;
        const int col0 = tile * C, ncl = min(C, a.ncol - col0);
        __syncthreads();  // the previous unit is done with the tile block
        load_tile(tb, a.tile + (size_t)tile * TILE_BYTES, tid, NT);
        __syncthreads();
        const int item0 = split * a.ipu, item1 = min(item0 + a.ipu, a.nitem);
#pragma unroll 1
        for (int item = item0; item < item1; ++item) {
            const int w_any = g + item * G;
            const bool real = w_any < nwvl;  // a group beyond the table runs the last wavelength with a zero source, unwritten
            const int w = real ? w_any : nwvl - 1;
            double tau[HALF], Bo[HALF], E1[HALF], E2[HALF], Eu20 = 0.0;
#pragma unroll
            for (int j = 0; j < HALF; ++j) E1[j] = E2[j] = 0.0;
            const double cl = tb[TB_CLOUD + c];
#pragma unroll
            for (int j = 0; j < HALF; ++j) {
                const int cell = cst.ipcell[h * HALF + j] + tbi[TBI_IT + sbi + j * C];
                const double v = tau_k1(tb, sb + j * C, h * HALF + j,
                                        reinterpret_cast<const double2*>(a.coef) + (size_t)(cell * nwvl + w) * 8, cl);
                tau[j] = fmax(CLAMPK ? v : clamp_hi(v, tau_clamp_hi), TAU_FLOOR);
            }
            // K2 (main.cpp:188-191)
            const double pc = __ldg(a.planck_c + w);
            const double pk = real ? __ldg(a.planck_k + w) : 0.0;
#pragma unroll
            for (int j = 0; j < HALF; ++j) Bo[j] = planck_b(pc, pk, tb[TB_INVT + sb + j * C], tab_lane);
            const double Bs = planck_b(pc, pk, tb[TB_INVTS + c], tab_lane);
            sweep_item<CLAMPK>(tau, Bo, Bs, h, tab_lane, E1, E2, Eu20);
            // the pair's 42 values in level order: E_down[0..20], then E_up[0..20] (rows of the unit kernel's K4)
            double* o = s_out + (size_t)(g * C + c) * 2 * NLEV;
#pragma unroll
            for (int j = 0; j < HALF; ++j) {
                const int l = h ? (NLAY - 1 - j) : j;
                o[l + 1] = h ? E2[j] : E1[j];
                o[NLEV + l] = h ? E1[j] : E2[j];
            }
            if (h) o[NLEV + NLAY] = Eu20;
            else o[0] = 0.0;  // E_down at the top of the atmosphere (main.cpp:300)
            __syncthreads();
            // the round's wavelengths w0 .. w0 + nw - 1 are consecutive: per column one run of nw * 21 doubles in each array
            const int w0 = item * G, nw = min(G, nwvl - w0), run = nw * NLEV;
            for (int i = tid; i < ncl * run; i += NT) {
                const int cc = i / run, k = i - cc * run, gg = k / NLEV, lev = k - gg * NLEV;
                const double* so = s_out + (size_t)(gg * C + cc) * 2 * NLEV;
                const size_t gi = ((size_t)(col0 + cc) * nwvl + w0) * NLEV + k;
                a.spec_dn[gi] = so[lev];
                a.spec_up[gi] = so[NLEV + lev];
            }
            __syncthreads();
        }
    }
}

constexpr int DIAG_SUM_COLS = 6;  // columns per CTA of the sum kernel: 6 x 21 = 126 threads

__global__ void __launch_bounds__(128) rcm_diag_sum_kernel(const DiagArgs a) {
    __shared__ double sEd[DIAG_SUM_COLS * NLEV], sEu[DIAG_SUM_COLS * NLEV];
    const int nwvl = cst.nwvl;
    const int cb = blockIdx.x * DIAG_SUM_COLS, ncl = min(DIAG_SUM_COLS, a.ncol - cb);
    const int tid = threadIdx.x;
    if (tid < ncl * NLEV) {
        const int cc = tid / NLEV, lev = tid % NLEV;
        const size_t base = (size_t)(cb + cc) * nwvl * NLEV + lev;
        double sd = 0.0, su = 0.0;
        for (int w = 0; w < nwvl; ++w) {
            sd += a.spec_dn[base + (size_t)w * NLEV];
            su += a.spec_up[base + (size_t)w * NLEV];
        }
        sEd[tid] = sd;
        sEu[tid] = su;
        a.E_down[(size_t)cb * NLEV + tid] = sd;
        a.E_up[(size_t)cb * NLEV + tid] = su;
    }
    __syncthreads();
    if (tid < ncl * NLAY) {  // heating rates as split_col_body (main.cpp:337-341)
        const int cc = tid / NLAY, l = tid % NLAY;
        const double* Ed = sEd + cc * NLEV;
        const double* Eu = sEu + cc * NLEV;
        double d = Ed[l] - Ed[l + 1] + Eu[l + 1] - Eu[l];
        if (l == NLAY - 1) d += (a.solar_col ? a.solar_col[cb + cc] : cst.solar_irr) + Ed[NLAY] - Eu[NLAY];
        a.dE[(size_t)cb * NLAY + tid] = d;
    }
}
