// rcm_split_kernels.cuh - the repwvl time step as TWO kernels per step, the default path of rcm_advance.
// Included by rcm_kernels.cu inside its anonymous namespace (after rcm_step_kernel.cuh: sweep_item, Smem helpers).
//
// Why.  The fused tile kernel (rcm_step_kernel) gives a CTA 16 whole columns x all wavelengths: 25 wavelength
// rounds per tile.  With 8,192 columns per GPU (the 65,536-column ensemble on 8 GPUs) that is 512 tiles on 444
// resident CTAs - a second round that is 15 % full - and the only way out was another tile shape, i.e. another order
// of the spectral sum: results depended on how many columns a GPU happened to own.  Here the unit of work is
// (tile of 16 columns) x (SPLIT_IPU = 5 wavelength rounds): 5 units per tile for repwvl-100, handed out to persistent
// CTAs by an atomic counter, so 8,192 columns are 2,560 units = 5.8 rounds of 444.  The order of every floating-point
// addition is fixed by (column, wavelength) alone:
//     E = sum_split ( sum_group ( register sum over the unit's rounds and angles ) )         [both outer sums in index order]
// whatever the ensemble size, the shard, the GPU count or the CTA that happened to take the unit - an N-GPU run is
// bit-identical to the 1-GPU run (tests/test_gpu_split.py).
//
//   rcm_split_col_kernel  K5, one CTA per tile, all threads on (column, layer) elements:
//       finish of step n  : sum of the step's partial fluxes, dE, time step, T update       (main.cpp:337-341, :156-176)
//       prep of step n+1  : theta-sort, stationarity diagnostic, water-vapour feedback, table indices and
//                           interpolation weights in T, 1/T, row-staging plan                (main.cpp:536-540, :281-289,
//                                                                                            repwvl_thermal.cpp:226-240)
//       and leaves everything the unit kernel needs for the tile in ONE contiguous 24,192-byte block.
//   rcm_split_rt_kernel   K1-K4 for (tile, split) units: the tile block arrives by ONE TMA bulk copy
//       (cp.async.bulk + mbarrier), issued for the NEXT unit while the partial fluxes of the current one are reduced;
//       K1 rows are staged per warp by cp.async as in the fused kernel; partial fluxes leave as [42][16] per unit.
//   rcm_split_multi_kernel  the same unit code (rcm_split_unit_loop.inc) for a BLOCK of steps in one launch: (step, unit)
//       items, per-tile step flags instead of kernel boundaries, the K5 body run in place by the CTA that completes a
//       tile's step.  For small shards, where a step is only a few rounds per CTA (see the comment in front of it).
#pragma once

constexpr int SPLIT_C = 16, SPLIT_NT = 128, SPLIT_G = 4;
constexpr int SPLIT_IPU = 5;  // wavelength rounds (of SPLIT_G wavelengths) per unit - fixed: it defines the summation order
constexpr int SPLIT_COL_NT = 128;  // K5 kernel: 8 CTAs (tiles) per SM at 64 registers

// the tile block (doubles, then ints); per-layer rows in pair order r = prow(l)
// A [20][16] array of the block keeps its rows 10..19 - the ones the h = 1 lanes read - half a bank row further on (8 doubles
// resp. 16 ints of padding after row 9): the two lanes of a pair read rows j and 10 + j of the same column in the same
// instruction, and at a distance of exactly 10 rows (1280 bytes) they would hit the same bank every time.
// (tbd / tbix / TBD_LEN / TBI_LEN: rcm_step_kernel.cuh, shared with the LBL kernel)
constexpr int TB_INVT = 0;                               // [20][16]  EXP_L2E / T (sorted profile): Planck exponent factor
constexpr int TB_DELT = TB_INVT + TBD_LEN;               // [20][16]  interpolation weight in T
constexpr int TB_DTDP = TB_DELT + TBD_LEN;               // [20][16]  that weight times the layer's weight in p (rounded once)
constexpr int TB_VMR = TB_DTDP + TBD_LEN;                // [5][20][16]
constexpr int TB_INVTS = TB_VMR + 5 * TBD_LEN;           // [16]      EXP_L2E / T_surface
constexpr int TB_CLOUD = TB_INVTS + SPLIT_C;             // [16]
constexpr int TB_DOUBLES = TB_CLOUD + SPLIT_C;
constexpr int TBI_IT = 0;                                // [20][16]  temperature interval (LowerPos)
constexpr int TBI_ROWSEL = TBI_IT + TBI_LEN;             // [20][16]  byte offset of the (layer, column)'s row in a warp's row buffer
constexpr int TBI_ROWOFF = TBI_ROWSEL + TBI_LEN;         // [20][NCAND] first table row of every candidate
constexpr int TBI_OUTSIDE = TBI_ROWOFF + NLAY * NCAND;   // some column needs a row beyond the candidates: global-memory K1
constexpr int TB_INTS = (TBI_OUTSIDE + 1 + 3) / 4 * 4;
constexpr int TILE_BYTES = TB_DOUBLES * 8 + TB_INTS * 4;
static_assert(TILE_BYTES % 16 == 0, "bulk copies move multiples of 16 bytes");
constexpr int ROWB3 = 16 * 8;                   // bytes of one row of the split path's table: 5 species x {c0', cT, cPT} + pad
// In shared memory the rows are 144 bytes apart: at 128 every row starts at bank 0, and the two lanes of a pair - always
// on different rows (layers j and 19-j) at the same offset - collide on every LDS.128 (measured: the kernel 14 % slower).
constexpr int ROWS3 = ROWB3 + 16;
constexpr int ROWBUF3 = NLAY * NCAND * ROWS3;   // per warp: 60 rows, 8,640 bytes
constexpr int SPLIT_PART = 2 * NLEV * SPLIT_C;  // doubles of one unit's partial fluxes: rows 0..19 E_down[l+1], 20 unused, 21..41 E_up[l]

// ------------------------------------------------------------------------------------------
// K5 for one tile (one CTA, threads on (column, layer) elements): finish of a step and / or preparation of the next.
// Everything the CTA will read from global memory is requested up front in one batch (one memory latency instead of
// one per phase - with a load in front of every phase the kernel took 260 us per 65,536 columns, latency-bound at four
// CTAs per SM); the phases then run out of shared memory and results leave as contiguous tile rows.
// ------------------------------------------------------------------------------------------
struct SplitColSmem {
    double sT[NLAY * SPLIT_C], sTh[NLAY * SPLIT_C], sPrev[NLAY * SPLIT_C], sRh[NLAY * SPLIT_C], sEd[NLEV * SPLIT_C],
        sEu[NLEV * SPLIT_C], sdE[NLAY * SPLIT_C], sdt[SPLIT_C], sTs[SPLIT_C], sSol[SPLIT_C], sStat[SPLIT_C];
    int sit[NLAY * SPLIT_C], sitmin[NLAY], sout[NLAY + 1];
};

// The body for one tile, by the 128 threads of a CTA: the K5 kernel's (STANDALONE), and the multi-step unit kernel's, where
// the CTA that finishes a tile's last unit of a step runs it in place.  State written by an earlier call of this function
// may come from another SM: everything mutable is loaded past L1 (__ldcg).
template <bool STANDALONE>
__device__ __forceinline__ void split_col_body(const SplitArgs& a, const SplitColFlags f, const int tile, SplitColSmem& cs) {
    constexpr int C = SPLIT_C, NT = SPLIT_COL_NT, LC = NLAY * C;
    double* const sT = cs.sT; double* const sTh = cs.sTh; double* const sPrev = cs.sPrev; double* const sRh = cs.sRh;
    double* const sEd = cs.sEd; double* const sEu = cs.sEu; double* const sdE = cs.sdE; double* const sdt = cs.sdt;
    double* const sTs = cs.sTs; double* const sSol = cs.sSol; double* const sStat = cs.sStat;
    int* const sit = cs.sit; int* const sitmin = cs.sitmin; int* const sout = cs.sout;
    int extrap = 0;  // some temperature of the tile lies outside the table's nodes: cross sections are extrapolated
    const int tid = threadIdx.x;
    const int col0 = tile * C, ncl = min(C, a.ncol - col0);
    const int nact = cst.nactive, nwvl = cst.nwvl;
    if (STANDALONE && tile == 0 && tid == 0 && a.counter) *a.counter = 0u;  // work counter of the unit kernel that follows on this stream
    double* const tb = reinterpret_cast<double*>(a.tile + (size_t)tile * TILE_BYTES);
    int* const tbi = reinterpret_cast<int*>(tb + TB_DOUBLES);
    const bool feedback = f.prep && !f.first && a.h2o_slot >= 0;
    // ---- one batch of loads: the tile's [16][20] blocks are contiguous; natural layer order in shared memory
    // (s[l * C + cc]); padding columns of the last tile repeat its first column -----------------------------------
    for (int i = tid; i < LC; i += NT) {
        const int cc = i / NLAY, l = i % NLAY;
        const size_t gi = (size_t)(col0 + (cc < ncl ? cc : 0)) * NLAY + l;
        sT[l * C + cc] = __ldcg(a.Tlayer + gi);
        if (f.prep) sPrev[l * C + cc] = __ldcg(a.Tprev + gi);
        if (feedback) sRh[l * C + cc] = a.rel_hum[gi];
    }
    if (tid < C) {
        const int col = col0 + (tid < ncl ? tid : 0);
        sTs[tid] = __ldcg(a.Tsurf + col);
        sSol[tid] = a.solar_col ? a.solar_col[col] : cst.solar_irr;
        if (f.finish) sStat[tid] = __ldcg(a.dTstat + col);
    }
    if (f.finish) {
        // K4 tail: the step's partial fluxes, summed over the splits in index order
        const double* part = a.part + (size_t)tile * a.nsplit * SPLIT_PART;
        for (int i = tid; i < SPLIT_PART; i += NT) {
            const int row = i / C;
            double sum = 0.0;
            if (row != NLAY)
                for (int sp = 0; sp < a.nsplit; ++sp) sum += __ldcg(part + (size_t)sp * SPLIT_PART + i);
            if (row < NLAY) sEd[i + C] = sum;
            else if (row == NLAY) sEd[i % C] = 0.0;  // E_down at the top of the atmosphere stays 0 (main.cpp:300)
            else sEu[i - NLEV * C] = sum;
        }
    }
    __syncthreads();

    if (f.finish) {
        for (int i = tid; i < LC; i += NT) {  // heating rates (main.cpp:337-341)
            const int l = i / C, cc = i % C;
            double d = sEd[l * C + cc] - sEd[(l + 1) * C + cc] + sEu[(l + 1) * C + cc] - sEu[l * C + cc];
            if (l == NLAY - 1) d += sSol[cc] + sEd[NLAY * C + cc] - sEu[NLAY * C + cc];
            sdE[i] = d;
        }
        __syncthreads();
        if (tid < C) {  // time step of the column (main.cpp:156-162) and its diagnostics
            double mx = sdE[tid], mabs = 0.0;
#pragma unroll
            for (int l = 0; l < NLAY; ++l) {
                const double d = sdE[l * C + tid];
                if (mx < d) mx = d;
                mabs = fmax(mabs, fabs(d));
            }
            double dt = (double)(float)cst.max_dT / mx * (1004.0 * cst.dp * 100.0) / 9.80665;
            if (dt > cst.dt_cap) dt = cst.dt_cap;
            sdt[tid] = dt;
            if (tid < ncl) {
                const int col = col0 + tid;
                a.time_h[col] = __ldcg(a.time_h + col) + (float)dt / 3600;  // main.cpp:581
                if (a.diag) {
                    double* dg = a.diag + ((size_t)f.diag_step * a.diag_ncol + col) * 4;
                    dg[0] = sSol[tid] - sEu[tid];
                    dg[1] = sStat[tid];
                    dg[2] = mabs;
                    dg[3] = dt;
                }
                if (f.write_out) a.dt[col] = dt;
            }
        }
        __syncthreads();
        for (int i = tid; i < LC; i += NT) {  // thermodynamics (main.cpp:164-176)
            const int l = i / C, cc = i % C;
            const double Tn = sT[i] + sdE[i] * sdt[cc] * 9.80665 / (1004.0 * cst.dp * 100.0);
            sT[i] = Tn;
            if (l == NLAY - 1) {
                const double ts = Tn * cst.conv[NLAY - 1];  // main.cpp:173
                sTs[cc] = ts;
                if (cc < ncl) a.Tsurf[col0 + cc] = ts;
            }
        }
        if (f.write_out) {
            for (int i = tid; i < NLEV * ncl; i += NT) {
                const int cc = i / NLEV, l = i % NLEV;
                a.E_down[(size_t)col0 * NLEV + i] = sEd[l * C + cc];
                a.E_up[(size_t)col0 * NLEV + i] = sEu[l * C + cc];
            }
            for (int i = tid; i < NLAY * ncl; i += NT) a.dE[(size_t)col0 * NLAY + i] = sdE[(i % NLAY) * C + i / NLAY];
        }
        __syncthreads();
        if (!f.prep) {
            for (int i = tid; i < NLAY * ncl; i += NT) a.Tlayer[(size_t)col0 * NLAY + i] = sT[(i % NLAY) * C + i / NLAY];
            return;
        }
    }

    // table indices and interpolation weights in T from the profile currently in sT (repwvl_thermal.cpp:229-239)
    auto indices = [&] {
        for (int i = tid; i < LC; i += NT) {
            const int l = i / C, cc = i % C, r = prow(l);
            const double midT = sT[i], tref = cst.tref_ip[r];
            const int it = lowerpos_t(tref, midT, cst.n_tpert);
            const double t0 = tref + cst.t_pert[it], t1 = tref + cst.t_pert[it + 1];
            extrap |= (midT < tref + cst.t_pert[0]) | (midT > tref + cst.t_pert[cst.n_tpert - 1]);
            sit[r * C + cc] = it;
            tbi[TBI_IT + tbix(r, cc)] = it;
            const double dT = (midT - t0) / (t1 - t0);
            tb[TB_DELT + tbd(r, cc)] = dT;
            tb[TB_DTDP + tbd(r, cc)] = __dmul_rn(dT, cst.delP[r]);
        }
    };
    if (f.first) indices();  // tau of the initial profile is built BEFORE the first sort (main.cpp:500-504)
    // theta-sort (main.cpp:536-540) by ranking: element (l, c) goes to layer #{l' : theta[l'] > theta[l], or equal and l' < l}
    for (int i = tid; i < LC; i += NT) sTh[i] = sT[i] * cst.conv[i / C];
    __syncthreads();
    for (int i = tid; i < LC; i += NT) {
        const int l = i / C, cc = i % C;
        const double my = sTh[i];
        int rank = 0;
#pragma unroll
        for (int l2 = 0; l2 < NLAY; ++l2) {
            const double v = sTh[l2 * C + cc];
            rank += (v > my || (v == my && l2 < l)) ? 1 : 0;
        }
        const double Tn = my / cst.conv[rank];
        sT[rank * C + cc] = Tn;
        sdE[rank * C + cc] = fabs(Tn - sPrev[rank * C + cc]);  // stationarity diagnostic of the step being prepared
    }
    __syncthreads();
    // the sorted profile: what the finish of this step updates, and the next step's "previous" profile
    for (int i = tid; i < NLAY * ncl; i += NT) {
        const double v = sT[(i % NLAY) * C + i / NLAY];
        a.Tlayer[(size_t)col0 * NLAY + i] = v;
        a.Tprev[(size_t)col0 * NLAY + i] = v;
    }
    if (tid < ncl) {
        double dmax = 0.0;
#pragma unroll
        for (int l = 0; l < NLAY; ++l) dmax = fmax(dmax, sdE[l * C + tid]);
        a.dTstat[col0 + tid] = dmax;
    }
    // volume mixing ratios of the tile: H2O from the water-vapour feedback (main.cpp:281-289, from the second
    // iteration on), the others only when the columns were (re)loaded
    for (int i = tid; i < nact * LC; i += NT) {
        const int cc = i % C, l = (i / C) % NLAY, sp = i / LC;
        const bool h2o = (sp == a.h2o_slot) && !f.first;
        if (!h2o && !f.write_all_vmr) continue;
        double v = 0.0;
        if (cc < ncl) {
            const size_t gi = ((size_t)(col0 + cc) * nact + sp) * NLAY + l;
            if (h2o) {
                const double Tc = sT[l * C + cc] - 273.15;
                const double e_sat = 6.1094 * exp(17.625 * Tc / (Tc + 243.04));
                v = sRh[l * C + cc] * e_sat / cst.player[l];
                a.vmr[gi] = v;
            } else {
                v = a.vmr[gi];
            }
        }
        tb[TB_VMR + sp * TBD_LEN + tbd(prow(l), cc)] = v;
    }
    if (!f.first) indices();
    // (T_floor: a column colder than ~5 K would take the fast exp's exponent out of range - its source is 0 either way)
    for (int i = tid; i < LC; i += NT) tb[TB_INVT + tbd(prow(i / C), i % C)] = (1.0 / fmax(sT[i], a.T_floor)) * L2E64;
    if (tid < C) {
        tb[TB_INVTS + tid] = (1.0 / fmax(sTs[tid], a.T_floor)) * L2E64;
        tb[TB_CLOUD + tid] = a.cloud_col ? a.cloud_col[col0 + (tid < ncl ? tid : 0)] : cst.cloud_tau;
    }
    const int any_extrap = __syncthreads_or(extrap);
    // the candidate rows of every layer: temperature intervals it_min .. it_min + NCAND - 1 of the tile's columns
    if (tid < NLAY) {
        int mn = sit[tid * C], mx = mn;
        for (int cc = 1; cc < C; ++cc) {
            mn = min(mn, sit[tid * C + cc]);
            mx = max(mx, sit[tid * C + cc]);
        }
        sitmin[tid] = mn;
        sout[tid] = (mx - mn >= NCAND);
        // (byte offset of the candidate's first row in the table: 32 bits are plenty - 20 layers x 8 intervals x nwvl x 128 B)
        for (int k = 0; k < NCAND; ++k) tbi[TBI_ROWOFF + NCAND * tid + k] = (cst.ipcell[tid] + min(mn + k, cst.n_tpert - 2)) * nwvl * ROWB3;
    }
    __syncthreads();
    for (int i = tid; i < LC; i += NT) {
        const int r = i / C;
        tbi[TBI_ROWSEL + tbix(r, i % C)] = (NCAND * r + min(sit[i] - sitmin[r], NCAND - 1)) * ROWS3;
    }
    if (tid == 0) {
        // extrapolated cross sections can come out negative: such a tile also takes the global-memory K1, which clamps
        // tau from below so that the transmissions' exp stays in range (the staged K1 of ordinary tiles pays nothing)
        int any = any_extrap;
        for (int r = 0; r < NLAY; ++r) any |= sout[r];
        tbi[TBI_OUTSIDE] = any;
    }
}

// for the multi-step unit kernel: a real call, so that the body's registers and code stay out of the unit loop's allocation
// and scheduling (inlined, ptxas arranged the angle loop differently and the units ran 15 % slower)
__device__ __noinline__ void split_col_body_call(const SplitArgs& a, const SplitColFlags f, const int tile, SplitColSmem& cs) {
    split_col_body<false>(a, f, tile, cs);
}

__global__ void __launch_bounds__(SPLIT_COL_NT, 8) rcm_split_col_kernel(const SplitArgs a, const SplitColFlags f) {
    __shared__ SplitColSmem cs;
    split_col_body<true>(a, f, blockIdx.x, cs);
}

// ---- per-tile step flags of the multi-step kernel (gpu scope) ----
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned* p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// A real call: inlined at the top of the unit loop, this spin loop made ptxas arrange the angle loop differently (units 15 %
// slower).  A step flag that never comes is a bug: fail loudly after seconds instead of hanging the GPU.
__device__ __noinline__ void wait_tile_ready(const unsigned* flag, unsigned step) {
    unsigned spins = 0;
    while (ld_acquire_gpu(flag) < step) {
        __nanosleep(128);
        if (++spins > (1u << 23)) __trap();
    }
    asm volatile("fence.proxy.async;" ::: "memory");  // the block was written through the generic proxy (another SM)
}

// ---- TMA bulk copy + mbarrier (one elected thread issues, everybody waits on the phase) -------------------------
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_1d(unsigned dst, const void* src, unsigned bytes, unsigned mbar) {
    // the buffer was last touched through the generic proxy (loads of the previous unit, ordered by the CTA barrier)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(mbar)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned phase) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(mbar),
        "r"(phase)
        : "memory");
}

// ------------------------------------------------------------------------------------------
// K1, K2 and the shared-memory fills of the unit kernels, also used by the diagnostic kernels (rcm_diag_kernels.cuh,
// rcm_jac_kernels.cuh): one definition, so that every kernel evaluates the same expression on the same numbers, bit for bit.
// ------------------------------------------------------------------------------------------
// K1 for the layer of tile-block row r whose doubles start at offset s (tbd(r, column)), from the row at cf: the bilinear
// (p, T) interpolation of repwvl_thermal.cpp:235-246,
//   x = c0 + cT*dT + cP*dP + cPT*dT*dP,   tau = numDens * sum_k x_k * vmr_k,
// contracted to three FMAs per species on {c0 + cP*dP, cT, cPT} and dT, dT*dP (17 instead of 42 FP64 instructions per
// layer and wavelength; within a few ulp of the reference's operation order - the bit-exact form is rcm_build_tau's).
__device__ __forceinline__ double tau_k1(const double* tb, int s, int r, const double2* cf, double cl) {
    const double dT = tb[TB_DELT + s], dTdP = tb[TB_DTDP + s];
    double c[16];
#pragma unroll
    for (int q2 = 0; q2 < 8; ++q2) {
        const double2 v = cf[q2];
        c[2 * q2] = v.x;
        c[2 * q2 + 1] = v.y;
    }
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        double v = fma(c[3 * k + 1], dT, c[3 * k]);
        v = fma(c[3 * k + 2], dTdP, v);
        acc = fma(v, tb[TB_VMR + k * TBD_LEN + s], acc);
    }
    acc = acc * cst.numDens[r];
    return fma(cst.cloud_w[r], cl, acc);  // main.cpp:270: + cl on the cloud layer, + 0 * cl (exact) elsewhere
}

// K2: Planck source B = k_w / (exp(c_w / T) - 1) (main.cpp:188-191, wavelength-only factors from the host) at
// invT = EXP_L2E / T
__device__ __forceinline__ double planck_b(double pc, double pk, double invT, unsigned tab_lane) {
    return div_fast(pk, exp_scaled<false>(pc, invT, tab_lane) - 1.0);
}

// the exp table into shared memory, EXP_REP copies of every entry side by side (exp_scaled), by the nt threads of a CTA
__device__ __forceinline__ void load_exp_tab(double* s_exp, const double* tab, int tid, int nt) {
    for (int i = tid; i < EXP_TAB * EXP_REP; i += nt) s_exp[i] = tab[i / EXP_REP];
}

// a tile block into shared memory, 16 bytes per copy, by the nt threads of a CTA
__device__ __forceinline__ void load_tile(double* tb, const unsigned char* tile, int tid, int nt) {
    const uint4* src = reinterpret_cast<const uint4*>(tile);
    uint4* dst = reinterpret_cast<uint4*>(tb);
    for (int i = tid; i < TILE_BYTES / 16; i += nt) dst[i] = src[i];
}

// ------------------------------------------------------------------------------------------
// K1-K4 for (tile, split) units.  Persistent CTAs (3 per SM, 168 registers), units by atomic counter.
// Shared memory: exp table 8 KB | four row buffers 4 x 7,680 B (after the wavelength loop: the groups' partial fluxes)
// | tile block 23,552 B | Planck factors 2 KB | mbarrier, next unit.
// ------------------------------------------------------------------------------------------
constexpr size_t SPLIT_SMEM = (size_t)EXP_TAB * EXP_REP * 8 + (size_t)SPLIT_G * ROWBUF3 + TILE_BYTES + 2 * PLK_MAX * 8 + 48;  // + mbarrier (8) + s_next[8]
static_assert(SPLIT_PART * 8 <= ROWBUF3, "a warp's row buffer carries its partial fluxes after the wavelength loop");

static_assert(sizeof(SplitColSmem) <= (size_t)SPLIT_G * ROWBUF3, "the K5 body of the multi-step kernel works in the row buffers");
static_assert(SPLIT_COL_NT == SPLIT_NT, "the multi-step kernel runs the K5 body with its own CTA");

// MULTI: one launch runs m.nsteps steps.  Work items are (step, unit) in step-major order from the same counter; a unit of
// step n waits for ready[tile] >= n, and the CTA that completes a tile's last unit of step n runs the K5 body for it (finish
// n, prep n + 1) and publishes ready[tile] = n + 1.  Dependencies point to lower item numbers only and every handed-out item
// is held by a running CTA, so the smallest unfinished item can always proceed: no deadlock whatever the grid.  The order of
// every addition is that of the one-step kernels - results are bit-identical - but there is no kernel boundary per step: no
// partial last round per step (8,192 columns: 5.77 rounds), K5 off the critical path.
template <bool CLAMPK>
__global__ void __launch_bounds__(SPLIT_NT, 3) rcm_split_rt_kernel(const SplitArgs a) {
#define RCM_SPLIT_MULTI 0
#include "rcm_split_unit_loop.inc"
#undef RCM_SPLIT_MULTI
}

template <bool CLAMPK>
__global__ void __launch_bounds__(SPLIT_NT, 3) rcm_split_multi_kernel(const __grid_constant__ SplitArgs a, const __grid_constant__ SplitMultiArgs m) {
#define RCM_SPLIT_MULTI 1
#include "rcm_split_unit_loop.inc"
#undef RCM_SPLIT_MULTI
}
