// rcm_rce - the RCE driver for ensembles, host C++ over the C ABI (include/rcm_b200.h).
//
// The reference's driver is main() of main.cpp: one hard-coded column (main.cpp:396-430), hard-coded table
// (main.cpp:500), a fixed number of iterations (main.cpp:531) and rows appended to output.txt (main.cpp:102-114).
// This is the same run for an ensemble of columns on one GPU: read the .atm file, build ncol perturbed members
// (member 0 is the file's own column), solar setup, upload, iterate until every column is stationary or
// max_steps is reached, write the profiles in the reference's row format and, optionally, a checkpoint.
//
//   rcm_rce --atm test.atm --table Reduced100Forcing.nc [--ncol N] [--seed S] [--max-steps M] [--check-every K]
//           [--dT 1e-3] [--device D] [--out output.txt] [--checkpoint file] [--resume file] [--steps-exact]
//           [--spectral-out spectrum.csv] [--kernels-out kernels.csv] [--jacobian-out jacobian.csv]
//           [--forcing-out forcing.csv [--forcing-scale 1,2,1,1,1] [--trop-layers 4]]
//   rcm_rce --atm fpda.lbl.atm --lbl DIR [--co2-factor F] ...     line-by-line: DIR/lbl.{h2o,co2,o3,ch4,n2o}.asc
//           [--lbl-bands-out bands.csv [--band-size 100] [--forcing-scale 1,2,1,1,1]] [--lbl-kernels-out kernels.csv]
//           [--lbl-jacobian-out jacobian.csv] [--lbl-forcing-out forcing.csv [--forcing-scale 1,2,1,1,1] [--trop-layers 4]]
//           [--response-out response.csv [--forcing-scale 1,2,1,1,1] [--trop-layers 4] [--fixed-q]]
//           [--species-jacobian-out species.csv] [--lbl-species-jacobian-out species.csv]
//           [--lbl-response-out response.csv [--forcing-scale 1,2,1,1,1] [--trop-layers 4] [--fixed-q]]
//   rcm_rce ... --gpus N                                          the same ensemble sharded over N GPUs of this node
//
// --gpus N (N > 1): one process, one host thread and one solver per GPU, contiguous blocks of columns per GPU (tables
// replicated), NCCL directly: after every block of --check-every fused iterations ONE pair of ncclAllReduce calls (sum,
// max) over the block's four scalars per step decides - identically on every GPU - whether the whole ensemble is
// stationary.  Nothing else crosses GPUs.  Per-column results do not depend on N (the solver's order of additions is
// fixed per column): the profile rows of an N-GPU run are byte-identical to the 1-GPU run's.
//
// The line-by-line form reads the five tables with the drop-in of ASCII_file2xy2D (lbl.arts/testlblarts.cpp:24-26 is the
// reference's only call of that reader); a six-column .atm (lbl.arts/README:1-3) gets the well-mixed CO2 / CH4 / N2O of
// lbl.arts/README:13-16.  The tables hold the optical depths of the file's own column: member 0's H2O and O3.
//
// --spectral-out FILE (repwvl tables only): after the run, the radiation the next step would see (rcm_diagnose_fluxes) per
// wavelength - header "wvl_nm,weight,olr,surface_down", then one row per wavelength with the ensemble means of the TOA upward
// and the surface downward flux of that wavelength (W/m2, its spectral weight included), summed in column order: the file is
// byte-identical for any --gpus N.
//
// --kernels-out FILE (repwvl tables only): after the run, the radiative kernels of the next step (rcm_radiative_kernels) -
// header "layer,p_layer,dOLR_dT,dOLR_dlnq,dSFC_dT,dSFC_dlnq", then one row per layer (top-down; p_layer in hPa) with the
// ensemble means of the derivatives of the OLR and of the surface downward flux with respect to the layer's temperature
// (W/m2/K) and ln(H2O VMR) (W/m2), then the row "surface" with the surface pressure and the derivatives with respect to the
// surface temperature (the ln q fields 0).  Summed in column order: the file is byte-identical for any --gpus N.
//
// --jacobian-out FILE (repwvl tables only): after the run, the derivatives of the next step's heating rates
// (rcm_flux_jacobian's dE_jac) - header "layer,p_layer,dT_0..dT_19,dT_surf,dlnq_0..dlnq_19", then one row per layer l
// (top-down; p_layer in hPa) with the ensemble means of d dE_l/dx_e (W/m2 per K resp. per unit ln q) for the 41 entries x_e.
// Summed in column order: the file is byte-identical for any --gpus N.
//
// --forcing-out FILE (repwvl tables only): after the run, the stratosphere-adjusted forcing of the next step's state by fixed
// dynamical heating (rcm_adjusted_forcing, tol 1e-6 W/m2, at most 20 Newton updates) for the factors --forcing-scale on the
// five active species' VMRs (H2O, CO2, O3, N2O, CH4; default 1,2,1,1,1: doubled CO2) with the --trop-layers top layers
// (default 4) as the stratosphere - header "layer,p_layer,dT_adj", then one row per layer (top-down; p_layer in hPa) with the
// ensemble-mean adjustment (K), then the rows "IRF_toa,,v", "IRF_trop,,v", "SARF_toa,,v", "SARF_trop,,v" with the ensemble
// means (W/m2) and "unconverged,,n" with the number of columns that did not converge.  Summed in column order: the file is
// byte-identical for any --gpus N.
//
// --lbl-bands-out FILE (line-by-line tables only): after the run, the fluxes the next step would see
// (rcm_lbl_diagnose_fluxes) in bands of --band-size K consecutive wavelengths (default 100; the last band is shorter),
// unscaled and with the factors --forcing-scale (H2O, CO2, O3, N2O, CH4; default 1,2,1,1,1) - header
// "wvl_lo_nm,wvl_hi_nm,olr,surface_down,olr_scaled,surface_down_scaled", then one row per band with its edges (the midpoint
// bins of rcm_set_lbl_tables) and the ensemble means of its TOA upward and surface downward flux (W/m2), unscaled and scaled.
// Summed in column order: the file is byte-identical for any --gpus N.
//
// --lbl-kernels-out FILE (line-by-line tables only): after the run, the radiative kernels of the next LBL step
// (rcm_lbl_radiative_kernels, summed over all wavelengths) in the format of --kernels-out.  Summed in column order: the file
// is byte-identical for any --gpus N.
//
// --lbl-jacobian-out FILE (line-by-line tables only): after the run, the derivatives of the next LBL step's heating rates
// (rcm_lbl_flux_jacobian's dE_jac) in the format of --jacobian-out.  Summed in column order: the file is byte-identical for any
// --gpus N.
//
// --lbl-forcing-out FILE (line-by-line tables only): after the run, the stratosphere-adjusted forcing of the next LBL step's
// state (rcm_lbl_adjusted_forcing, tol 1e-6 W/m2, at most 20 Newton updates) for the factors --forcing-scale with the
// --trop-layers top layers as the stratosphere, in the format of --forcing-out.  Summed in column order: the file is
// byte-identical for any --gpus N.
//
// --response-out FILE (repwvl tables only): after the run, the equilibrium climate response of the next step's state
// (rcm_climate_response, tol 1e-6 W/m2, at most 20 Newton updates) to the factors --forcing-scale with the --trop-layers top
// layers as the stratosphere, at fixed relative humidity (--fixed-q: at fixed absolute humidity) - header "layer,p_layer,dT",
// then one row per layer (top-down; p_layer in hPa) with the ensemble-mean response (K), then the rows "dTs,,v", "IRF_toa,,v",
// "IRF_trop,,v" with the ensemble means (K, W/m2) and "unconverged,,n".  Summed in column order: the file is byte-identical for
// any --gpus N.
//
// --lbl-response-out FILE (line-by-line tables only): the same from rcm_lbl_climate_response, in the format of --response-out.
//
// --species-jacobian-out FILE (repwvl tables only): after the run, the layer-resolved species kernels of the next step
// (rcm_species_jacobian) - header "species,layer,p_layer,dOLR_dlnx,dSFC_dlnx,dHeat_dlnx", then one row per species (h2o, co2,
// o3, n2o, ch4) and layer (top-down; p_layer in hPa) with the ensemble means of the derivatives of the OLR, of the surface
// downward flux and of the layer's own heating rate dE_l with respect to ln of the species' VMR in that layer (W/m2).  Summed
// in column order: the file is byte-identical for any --gpus N.
//
// --lbl-species-jacobian-out FILE (line-by-line tables only): the same from rcm_lbl_species_jacobian.
//
// --steps-exact runs exactly max_steps iterations (the reference's n_steps semantics, main.cpp:83) instead of
// stopping at stationarity.  Exit code 0, or 1 with the library's error text on stderr.  No CPU fallback.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime_api.h>
#include <nccl.h>

#include "rcm_b200.h"

namespace {

int die(const char* what, int st, const rcm_solver* s) {
    std::fprintf(stderr, "rcm_rce: %s: %s%s%s\n", what, rcm_status_string(st), s ? " - " : "", s ? rcm_last_error(s) : "");
    return 1;
}

// ---- N GPUs: one thread per GPU, columns [lo, hi) each ---------------------------------------------------------
struct Shard {
    int dev = 0, lo = 0, hi = 0;
    rcm_solver* s = nullptr;
    cudaStream_t stream = nullptr;
    ncclComm_t comm = nullptr;
    double *d_sum = nullptr, *d_max = nullptr;  // [check_every][4] reduced scalars of a block
    long done = 0;
    rcm_step_scalars last{};
    double loop_s = 0.0;  // wall time of the time loop (first launch to last block decided)
    std::string err;
};

struct Job {  // what every shard needs; host arrays cover the WHOLE ensemble
    const rcm_params* p;
    const rcm_table* table;  // repwvl, or NULL
    const std::vector<double>*wvl, *tau5;
    int lbl_nwvl;
    double co2_factor;
    const double *plevel, *Tlayer, *Tsurf, *vmr9, *rel_hum;
    int ncol;
    long max_steps;
    int check_every, steps_exact;
    std::string resume, ckpt;
    double *T_out, *Ts_out, *Eu_out;
    float* time_out;
    int spec_nwvl;            // > 0: --spectral-out, rows [ncol][spec_nwvl] of olr / sfc
    double *olr_out, *sfc_out;
    int kernels;              // --kernels-out / --lbl-kernels-out: rows [ncol][2][41] of rcm_radiative_kernels (repwvl) or
                              // rcm_lbl_radiative_kernels (line-by-line) into K_out
    double* K_out;
    int jacobian;             // --jacobian-out / --lbl-jacobian-out: rows [ncol][20][41] of rcm_flux_jacobian's (repwvl) or
                              // rcm_lbl_flux_jacobian's (line-by-line) dE_jac into H_out
    double* H_out;
    int forcing;              // --forcing-out / --lbl-forcing-out: rcm_adjusted_forcing's (repwvl) or rcm_lbl_adjusted_forcing's
                              // (line-by-line) F [ncol][4], dT_adj [ncol][20], iters [ncol]
    const double* forcing_scale;
    const int* ntrop;         // [ncol]
    double *F_out, *dTadj_out;
    int* iters_out;
    int lbl_nband;            // > 0: --lbl-bands-out, rows [ncol][nband][4] (olr, sfc, olr scaled, sfc scaled) into B_out
    const int* lbl_bstart;    // [nband + 1]
    double* B_out;
    int response;             // --response-out / --lbl-response-out: rcm_climate_response's (repwvl) or
                              // rcm_lbl_climate_response's (line-by-line) F [ncol][2], dT [ncol][20], dTs [ncol], iters [ncol]
    int fixed_rh;
    double *RF_out, *RdT_out, *RdTs_out;
    int* Riters_out;
    int species;              // --species-jacobian-out / --lbl-species-jacobian-out: rows [ncol][3][100] of species_rows into S_out
    double* S_out;
};

std::atomic<int> g_failed{0};

// TOA E_up and surface E_down of every (column, wavelength) of the n columns of s: olr / sfc [n][nwvl]
int diagnose_spectrum(rcm_solver* s, int n, int nwvl, double* olr, double* sfc) {
    constexpr int NLEV = RCM_NLEVEL, CHUNK = 4096;
    std::vector<double> dn((size_t)std::min(n, CHUNK) * nwvl * NLEV), up(dn.size());
    for (int c0 = 0; c0 < n; c0 += CHUNK) {
        const int m = std::min(CHUNK, n - c0);
        const int st = rcm_diagnose_fluxes(s, c0, m, nullptr, dn.data(), up.data(), nullptr, nullptr, nullptr);
        if (st != RCM_OK) return st;
        for (size_t c = 0; c < (size_t)m; ++c)
            for (size_t w = 0; w < (size_t)nwvl; ++w) {
                olr[(c0 + c) * nwvl + w] = up[(c * nwvl + w) * NLEV];
                sfc[(c0 + c) * nwvl + w] = dn[(c * nwvl + w) * NLEV + NLEV - 1];
            }
    }
    return RCM_OK;
}

// ensemble means per wavelength, summed in column order
int write_spectrum(const std::string& path, int ncol, int nwvl, const double* wvl, const double* weight, const double* olr,
                   const double* sfc) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) {
        std::fprintf(stderr, "rcm_rce: cannot write %s\n", path.c_str());
        return 1;
    }
    std::fprintf(f, "wvl_nm,weight,olr,surface_down\n");
    for (int w = 0; w < nwvl; ++w) {
        double so = 0.0, ss = 0.0;
        for (size_t c = 0; c < (size_t)ncol; ++c) {
            so += olr[c * nwvl + w];
            ss += sfc[c * nwvl + w];
        }
        std::fprintf(f, "%.17g,%.17g,%.17g,%.17g\n", wvl[w], weight[w], so / ncol, ss / ncol);
    }
    if (std::fclose(f) != 0) {
        std::fprintf(stderr, "rcm_rce: short write to %s\n", path.c_str());
        return 1;
    }
    return 0;
}

constexpr int KERN_NE = 2 * RCM_NLAYER + 1, KERN_NK = 2 * KERN_NE;  // rcm_radiative_kernels: [2][41] per column

// ensemble means of the radiative kernels, summed in column order
int write_kernels(const std::string& path, int ncol, const double* player, double p_surface, const double* K) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) {
        std::fprintf(stderr, "rcm_rce: cannot write %s\n", path.c_str());
        return 1;
    }
    auto mean = [&](int o, int e) {
        double sum = 0.0;
        for (size_t c = 0; c < (size_t)ncol; ++c) sum += K[c * KERN_NK + o * KERN_NE + e];
        return sum / ncol;
    };
    constexpr int NLAY = RCM_NLAYER;
    std::fprintf(f, "layer,p_layer,dOLR_dT,dOLR_dlnq,dSFC_dT,dSFC_dlnq\n");
    for (int l = 0; l < NLAY; ++l)
        std::fprintf(f, "%d,%.17g,%.17g,%.17g,%.17g,%.17g\n", l, player[l], mean(0, l), mean(0, NLAY + 1 + l), mean(1, l),
                     mean(1, NLAY + 1 + l));
    std::fprintf(f, "surface,%.17g,%.17g,0,%.17g,0\n", p_surface, mean(0, NLAY), mean(1, NLAY));
    if (std::fclose(f) != 0) {
        std::fprintf(stderr, "rcm_rce: short write to %s\n", path.c_str());
        return 1;
    }
    return 0;
}

constexpr int JAC_NH = RCM_NLAYER * KERN_NE;  // rcm_flux_jacobian: dE_jac [20][41] per column

// ensemble means of the heating-rate Jacobians, summed in column order
int write_jacobian(const std::string& path, int ncol, const double* player, const double* H) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) {
        std::fprintf(stderr, "rcm_rce: cannot write %s\n", path.c_str());
        return 1;
    }
    constexpr int NLAY = RCM_NLAYER;
    std::fprintf(f, "layer,p_layer");
    for (int l = 0; l < NLAY; ++l) std::fprintf(f, ",dT_%d", l);
    std::fprintf(f, ",dT_surf");
    for (int l = 0; l < NLAY; ++l) std::fprintf(f, ",dlnq_%d", l);
    std::fprintf(f, "\n");
    for (int l = 0; l < NLAY; ++l) {
        std::fprintf(f, "%d,%.17g", l, player[l]);
        for (int e = 0; e < KERN_NE; ++e) {
            double sum = 0.0;
            for (size_t c = 0; c < (size_t)ncol; ++c) sum += H[c * JAC_NH + l * KERN_NE + e];
            std::fprintf(f, ",%.17g", sum / ncol);
        }
        std::fprintf(f, "\n");
    }
    if (std::fclose(f) != 0) {
        std::fprintf(stderr, "rcm_rce: short write to %s\n", path.c_str());
        return 1;
    }
    return 0;
}

constexpr int SPJ_NE = 5 * RCM_NLAYER, SPJ_NJ = 2 * RCM_NLEVEL * SPJ_NE, SPJ_NH = RCM_NLAYER * SPJ_NE;  // rcm_species_jacobian

// rows [n][3][100] of the n columns of s from rcm_species_jacobian (repwvl) or rcm_lbl_species_jacobian (line-by-line): per entry
// e = 20 s + l, dE_up[0]/dx_e, dE_down[20]/dx_e and d dE_l/dx_e, the layer's own heating rate
int species_rows(rcm_solver* s, bool lbl, int n, double* R) {
    constexpr int NLAY = RCM_NLAYER, NLEV = RCM_NLEVEL, CHUNK = 1024;
    std::vector<double> J((size_t)std::min(n, CHUNK) * SPJ_NJ), H((size_t)std::min(n, CHUNK) * SPJ_NH);
    for (int c0 = 0; c0 < n; c0 += CHUNK) {
        const int m = std::min(CHUNK, n - c0);
        const int st = (lbl ? rcm_lbl_species_jacobian : rcm_species_jacobian)(s, c0, m, nullptr, J.data(), H.data());
        if (st != RCM_OK) return st;
        for (size_t c = 0; c < (size_t)m; ++c)
            for (int e = 0; e < SPJ_NE; ++e) {
                double* r = R + (c0 + c) * 3 * SPJ_NE + e;
                r[0] = J[c * SPJ_NJ + (size_t)(NLEV + 0) * SPJ_NE + e];     // E_up[0]
                r[SPJ_NE] = J[c * SPJ_NJ + (size_t)(NLEV - 1) * SPJ_NE + e];  // E_down[20]
                r[2 * SPJ_NE] = H[c * SPJ_NH + (size_t)(e % NLAY) * SPJ_NE + e];
            }
    }
    return RCM_OK;
}

// ensemble means of the species rows, summed in column order
int write_species(const std::string& path, int ncol, const double* player, const double* R) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) {
        std::fprintf(stderr, "rcm_rce: cannot write %s\n", path.c_str());
        return 1;
    }
    constexpr int NLAY = RCM_NLAYER;
    const char* names[5] = {"h2o", "co2", "o3", "n2o", "ch4"};  // ascending species index, the entries' order
    std::fprintf(f, "species,layer,p_layer,dOLR_dlnx,dSFC_dlnx,dHeat_dlnx\n");
    for (int e = 0; e < SPJ_NE; ++e) {
        std::fprintf(f, "%s,%d,%.17g", names[e / NLAY], e % NLAY, player[e % NLAY]);
        for (int o = 0; o < 3; ++o) {
            double sum = 0.0;
            for (size_t c = 0; c < (size_t)ncol; ++c) sum += R[(c * 3 + o) * SPJ_NE + e];
            std::fprintf(f, ",%.17g", sum / ncol);
        }
        std::fprintf(f, "\n");
    }
    if (std::fclose(f) != 0) {
        std::fprintf(stderr, "rcm_rce: short write to %s\n", path.c_str());
        return 1;
    }
    return 0;
}

constexpr int FORCING_MAX_ITER = 20;
constexpr double FORCING_TOL = 1e-6;

// ensemble means of the climate response, summed in column order
int write_response(const std::string& path, int ncol, const double* player, const double* F, const double* dT, const double* dTs,
                   const int* iters) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) {
        std::fprintf(stderr, "rcm_rce: cannot write %s\n", path.c_str());
        return 1;
    }
    constexpr int NLAY = RCM_NLAYER;
    std::fprintf(f, "layer,p_layer,dT\n");
    for (int l = 0; l < NLAY; ++l) {
        double sum = 0.0;
        for (size_t c = 0; c < (size_t)ncol; ++c) sum += dT[c * NLAY + l];
        std::fprintf(f, "%d,%.17g,%.17g\n", l, player[l], sum / ncol);
    }
    double sum = 0.0;
    for (size_t c = 0; c < (size_t)ncol; ++c) sum += dTs[c];
    std::fprintf(f, "dTs,,%.17g\n", sum / ncol);
    const char* names[2] = {"IRF_toa", "IRF_trop"};
    for (int k = 0; k < 2; ++k) {
        double sk = 0.0;
        for (size_t c = 0; c < (size_t)ncol; ++c) sk += F[c * 2 + k];
        std::fprintf(f, "%s,,%.17g\n", names[k], sk / ncol);
    }
    int bad = 0;
    for (size_t c = 0; c < (size_t)ncol; ++c) bad += iters[c] < 0;
    std::fprintf(f, "unconverged,,%d\n", bad);
    if (std::fclose(f) != 0) {
        std::fprintf(stderr, "rcm_rce: short write to %s\n", path.c_str());
        return 1;
    }
    return 0;
}

// ensemble means of the adjusted forcing, summed in column order
int write_forcing(const std::string& path, int ncol, const double* player, const double* F, const double* dT, const int* iters) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) {
        std::fprintf(stderr, "rcm_rce: cannot write %s\n", path.c_str());
        return 1;
    }
    constexpr int NLAY = RCM_NLAYER;
    std::fprintf(f, "layer,p_layer,dT_adj\n");
    for (int l = 0; l < NLAY; ++l) {
        double sum = 0.0;
        for (size_t c = 0; c < (size_t)ncol; ++c) sum += dT[c * NLAY + l];
        std::fprintf(f, "%d,%.17g,%.17g\n", l, player[l], sum / ncol);
    }
    const char* names[4] = {"IRF_toa", "IRF_trop", "SARF_toa", "SARF_trop"};
    for (int k = 0; k < 4; ++k) {
        double sum = 0.0;
        for (size_t c = 0; c < (size_t)ncol; ++c) sum += F[c * 4 + k];
        std::fprintf(f, "%s,,%.17g\n", names[k], sum / ncol);
    }
    int bad = 0;
    for (size_t c = 0; c < (size_t)ncol; ++c) bad += iters[c] < 0;
    std::fprintf(f, "unconverged,,%d\n", bad);
    if (std::fclose(f) != 0) {
        std::fprintf(stderr, "rcm_rce: short write to %s\n", path.c_str());
        return 1;
    }
    return 0;
}

// TOA E_up and surface E_down of every (column, band) of the n columns of s, unscaled and with the factors scale:
// out [n][nband][4] = olr, sfc, olr scaled, sfc scaled
int diagnose_lbl_bands(rcm_solver* s, int n, int nband, const int* bstart, const double* scale, double* out) {
    constexpr int NLEV = RCM_NLEVEL, CHUNK = 1024;
    std::vector<double> dn((size_t)std::min(n, CHUNK) * nband * NLEV), up(dn.size());
    for (int pass = 0; pass < 2; ++pass)
        for (int c0 = 0; c0 < n; c0 += CHUNK) {
            const int m = std::min(CHUNK, n - c0);
            const int st = rcm_lbl_diagnose_fluxes(s, c0, m, pass ? scale : nullptr, nband, bstart, dn.data(), up.data(), nullptr,
                                                   nullptr, nullptr);
            if (st != RCM_OK) return st;
            for (size_t c = 0; c < (size_t)m; ++c)
                for (size_t b = 0; b < (size_t)nband; ++b) {
                    double* o = out + (((size_t)c0 + c) * nband + b) * 4 + 2 * pass;
                    o[0] = up[(c * nband + b) * NLEV];
                    o[1] = dn[(c * nband + b) * NLEV + NLEV - 1];
                }
        }
    return RCM_OK;
}

// band starts of K consecutive wavelengths: [nband + 1]
std::vector<int> lbl_band_starts(int nwvl, int K) {
    std::vector<int> b;
    for (int w = 0; w < nwvl; w += K) b.push_back(w);
    b.push_back(nwvl);
    return b;
}

// ensemble means per band, summed in column order; edges as rcm_set_lbl_tables' bins
int write_lbl_bands(const std::string& path, int ncol, const std::vector<double>& wvl, const std::vector<int>& bstart, const double* B) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) {
        std::fprintf(stderr, "rcm_rce: cannot write %s\n", path.c_str());
        return 1;
    }
    const int nwvl = (int)wvl.size(), nband = (int)bstart.size() - 1;
    std::fprintf(f, "wvl_lo_nm,wvl_hi_nm,olr,surface_down,olr_scaled,surface_down_scaled\n");
    for (int b = 0; b < nband; ++b) {
        const int i = bstart[b], k = bstart[b + 1] - 1;
        const double dl = (i > 0) ? (wvl[i] - wvl[i - 1]) : (wvl[1] - wvl[0]);
        const double dh = (k < nwvl - 1) ? (wvl[k + 1] - wvl[k]) : (wvl[k] - wvl[k - 1]);
        double sum[4] = {0.0, 0.0, 0.0, 0.0};
        for (size_t c = 0; c < (size_t)ncol; ++c)
            for (int q = 0; q < 4; ++q) sum[q] += B[(c * nband + b) * 4 + q];
        std::fprintf(f, "%.17g,%.17g,%.17g,%.17g,%.17g,%.17g\n", wvl[i] - dl / 2.0, wvl[k] + dh / 2.0, sum[0] / ncol, sum[1] / ncol,
                     sum[2] / ncol, sum[3] / ncol);
    }
    if (std::fclose(f) != 0) {
        std::fprintf(stderr, "rcm_rce: short write to %s\n", path.c_str());
        return 1;
    }
    return 0;
}

void run_shard(Shard* sh, const Job* j) {
    auto fail = [&](const char* what, int st) {
        sh->err = std::string(what) + ": " + rcm_status_string(st) + (sh->s ? std::string(" - ") + rcm_last_error(sh->s) : "");
        g_failed.store(1);
    };
    constexpr int NLAY = RCM_NLAYER, NLEV = RCM_NLEVEL;
    const size_t lo = (size_t)sh->lo, n = (size_t)(sh->hi - sh->lo);
    int st = rcm_create(sh->dev, j->p, &sh->s);
    if (st != RCM_OK) return fail("rcm_create", st);
    if (cudaSetDevice(sh->dev) != cudaSuccess || cudaStreamCreateWithFlags(&sh->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaMalloc((void**)&sh->d_sum, (size_t)j->check_every * 4 * sizeof(double)) != cudaSuccess ||
        cudaMalloc((void**)&sh->d_max, (size_t)j->check_every * 4 * sizeof(double)) != cudaSuccess)
        return fail("cuda setup", RCM_ERR_CUDA);
    rcm_set_stream(sh->s, sh->stream);  // the solver's kernels and the NCCL calls share one stream: ordered without events
    st = j->table ? rcm_set_repwvl_table_from(sh->s, j->table)
                  : rcm_set_lbl_tables(sh->s, j->wvl->data(), j->tau5->data(), j->lbl_nwvl, j->vmr9 + 0 * NLAY, j->vmr9 + 2 * NLAY,
                                       j->co2_factor);
    if (st != RCM_OK) return fail("tables", st);
    if (!j->resume.empty()) {
        st = rcm_load_checkpoint(sh->s, (j->resume + ".gpu" + std::to_string(sh->dev)).c_str());
        if (st == RCM_OK && rcm_column_count(sh->s) != (int)n) st = RCM_ERR_STATE;
    } else {
        st = rcm_set_columns(sh->s, (int)n, j->plevel, j->Tlayer + lo * NLAY, j->Tsurf + lo, j->vmr9 + lo * RCM_NSPECIES * NLAY,
                             j->rel_hum + lo * NLAY);
    }
    if (st != RCM_OK) return fail("columns", st);
    // ---- the time loop (main.cpp:531-583) in blocks; one allreduce pair per block ------------------------------
    std::vector<double> hs(4), hm(4);
    // warm-up outside the clock: the first launch loads the kernels, the first collective builds NCCL's channels; the
    // ensemble then restarts from its initial state (a resumed run keeps its state: only the collective is warmed up)
    if (j->resume.empty()) {
        st = rcm_advance(sh->s, 1, nullptr);
        if (st == RCM_OK)
            st = rcm_set_columns(sh->s, (int)n, j->plevel, j->Tlayer + lo * NLAY, j->Tsurf + lo, j->vmr9 + lo * RCM_NSPECIES * NLAY,
                                 j->rel_hum + lo * NLAY);
        if (st != RCM_OK) return fail("warm-up", st);
    }
    cudaMemsetAsync(sh->d_sum, 0, 4 * sizeof(double), sh->stream);
    if (ncclAllReduce(sh->d_sum, sh->d_max, 4, ncclDouble, ncclSum, sh->comm, sh->stream) != ncclSuccess)
        return fail("ncclAllReduce (warm-up)", RCM_ERR_CUDA);
    cudaStreamSynchronize(sh->stream);
    const auto t0 = std::chrono::steady_clock::now();
    while (sh->done < j->max_steps && !g_failed.load()) {
        const int k = (int)((j->max_steps - sh->done < j->check_every) ? (j->max_steps - sh->done) : j->check_every);
        double* d_sc = nullptr;
        st = rcm_advance_async(sh->s, k, &d_sc);
        if (st != RCM_OK) return fail("rcm_advance_async", st);
        if (ncclAllReduce(d_sc, sh->d_sum, (size_t)k * 4, ncclDouble, ncclSum, sh->comm, sh->stream) != ncclSuccess ||
            ncclAllReduce(d_sc, sh->d_max, (size_t)k * 4, ncclDouble, ncclMax, sh->comm, sh->stream) != ncclSuccess)
            return fail("ncclAllReduce", RCM_ERR_CUDA);
        cudaMemcpyAsync(hs.data(), sh->d_sum + (size_t)(k - 1) * 4, 4 * sizeof(double), cudaMemcpyDeviceToHost, sh->stream);
        cudaMemcpyAsync(hm.data(), sh->d_max + (size_t)(k - 1) * 4, 4 * sizeof(double), cudaMemcpyDeviceToHost, sh->stream);
        if (cudaStreamSynchronize(sh->stream) != cudaSuccess) return fail("block", RCM_ERR_CUDA);
        sh->done += k;
        sh->last = {hs[0], hm[1], hs[2], hm[3]};  // sums: TOA net, converged count; maxima: dT, |dE|
        if (!j->steps_exact && sh->last.n_converged >= (double)j->ncol) break;  // the same numbers on every GPU
    }
    sh->loop_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (g_failed.load()) return;
    st = rcm_get_state(sh->s, j->T_out + lo * NLAY, j->Ts_out + lo, nullptr, j->time_out + lo, nullptr, j->Eu_out + lo * NLEV, nullptr,
                       nullptr);
    if (st != RCM_OK) return fail("rcm_get_state", st);
    if (!j->ckpt.empty()) {
        st = rcm_save_checkpoint(sh->s, (j->ckpt + ".gpu" + std::to_string(sh->dev)).c_str());
        if (st != RCM_OK) return fail("rcm_save_checkpoint", st);
    }
    if (j->spec_nwvl > 0) {
        st = diagnose_spectrum(sh->s, (int)n, j->spec_nwvl, j->olr_out + lo * j->spec_nwvl, j->sfc_out + lo * j->spec_nwvl);
        if (st != RCM_OK) return fail("rcm_diagnose_fluxes", st);
    }
    if (j->kernels) {
        st = j->table ? rcm_radiative_kernels(sh->s, 0, (int)n, nullptr, nullptr, j->K_out + lo * KERN_NK)
                      : rcm_lbl_radiative_kernels(sh->s, 0, (int)n, nullptr, 0, nullptr, nullptr, j->K_out + lo * KERN_NK);
        if (st != RCM_OK) return fail(j->table ? "rcm_radiative_kernels" : "rcm_lbl_radiative_kernels", st);
    }
    if (j->jacobian) {
        st = (j->table ? rcm_flux_jacobian : rcm_lbl_flux_jacobian)(sh->s, 0, (int)n, nullptr, nullptr, j->H_out + lo * JAC_NH);
        if (st != RCM_OK) return fail(j->table ? "rcm_flux_jacobian" : "rcm_lbl_flux_jacobian", st);
    }
    if (j->forcing) {
        st = (j->table ? rcm_adjusted_forcing : rcm_lbl_adjusted_forcing)(sh->s, 0, (int)n, j->forcing_scale, j->ntrop + lo, FORCING_TOL,
                                                                         FORCING_MAX_ITER, j->F_out + lo * 4, j->dTadj_out + lo * NLAY,
                                                                         nullptr, nullptr, j->iters_out + lo);
        if (st != RCM_OK) return fail(j->table ? "rcm_adjusted_forcing" : "rcm_lbl_adjusted_forcing", st);
    }
    if (j->response) {
        st = (j->table ? rcm_climate_response : rcm_lbl_climate_response)(sh->s, 0, (int)n, j->forcing_scale, j->ntrop + lo, j->fixed_rh,
                                                                         FORCING_TOL, FORCING_MAX_ITER, j->RF_out + lo * 2,
                                                                         j->RdT_out + lo * NLAY, j->RdTs_out + lo, nullptr, nullptr,
                                                                         j->Riters_out + lo);
        if (st != RCM_OK) return fail(j->table ? "rcm_climate_response" : "rcm_lbl_climate_response", st);
    }
    if (j->species) {
        st = species_rows(sh->s, !j->table, (int)n, j->S_out + lo * 3 * SPJ_NE);
        if (st != RCM_OK) return fail(j->table ? "rcm_species_jacobian" : "rcm_lbl_species_jacobian", st);
    }
    if (j->lbl_nband > 0) {
        st = diagnose_lbl_bands(sh->s, (int)n, j->lbl_nband, j->lbl_bstart, j->forcing_scale, j->B_out + lo * j->lbl_nband * 4);
        if (st != RCM_OK) return fail("rcm_lbl_diagnose_fluxes", st);
    }
}

}  // namespace

int main(int argc, char** argv) {
    std::string atm_path, table_path, lbl_dir, out_path = "output.txt", ckpt_path, resume_path, spectral_path, kernels_path,
        jacobian_path, forcing_path, forcing_scale_arg = "1,2,1,1,1", trop_layers_arg = "4", bands_path, band_size_arg = "100",
        lbl_kernels_path, lbl_jacobian_path, lbl_forcing_path, response_path, lbl_response_path, species_path, lbl_species_path;
    double co2_factor = 1.0;
    int ncol = 1, device = 0, check_every = 250, steps_exact = 0, gpus = 1, fixed_rh = 1;
    long max_steps = 6000;
    unsigned long long seed = 12345;
    double dT = 1e-3;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&]() -> const char* { return (i + 1 < argc) ? argv[++i] : ""; };
        if (a == "--atm") atm_path = val();
        else if (a == "--table") table_path = val();
        else if (a == "--lbl") lbl_dir = val();
        else if (a == "--co2-factor") co2_factor = std::atof(val());
        else if (a == "--ncol") ncol = std::atoi(val());
        else if (a == "--seed") seed = std::strtoull(val(), nullptr, 10);
        else if (a == "--max-steps") max_steps = std::atol(val());
        else if (a == "--check-every") check_every = std::atoi(val());
        else if (a == "--dT") dT = std::atof(val());
        else if (a == "--device") device = std::atoi(val());
        else if (a == "--out") out_path = val();
        else if (a == "--checkpoint") ckpt_path = val();
        else if (a == "--resume") resume_path = val();
        else if (a == "--steps-exact") steps_exact = 1;
        else if (a == "--gpus") gpus = std::atoi(val());
        else if (a == "--spectral-out") spectral_path = val();
        else if (a == "--kernels-out") kernels_path = val();
        else if (a == "--jacobian-out") jacobian_path = val();
        else if (a == "--forcing-out") forcing_path = val();
        else if (a == "--forcing-scale") forcing_scale_arg = val();
        else if (a == "--trop-layers") trop_layers_arg = val();
        else if (a == "--lbl-bands-out") bands_path = val();
        else if (a == "--band-size") band_size_arg = val();
        else if (a == "--lbl-kernels-out") lbl_kernels_path = val();
        else if (a == "--lbl-jacobian-out") lbl_jacobian_path = val();
        else if (a == "--lbl-forcing-out") lbl_forcing_path = val();
        else if (a == "--response-out") response_path = val();
        else if (a == "--lbl-response-out") lbl_response_path = val();
        else if (a == "--fixed-q") fixed_rh = 0;
        else if (a == "--species-jacobian-out") species_path = val();
        else if (a == "--lbl-species-jacobian-out") lbl_species_path = val();
        else {
            std::fprintf(stderr, "rcm_rce: unknown argument %s\n", a.c_str());
            return 1;
        }
    }
    if (atm_path.empty() || (table_path.empty() == lbl_dir.empty()) || ncol < 1 || max_steps < 1 || check_every < 1 || gpus < 1 ||
        gpus > ncol) {
        std::fprintf(stderr, "usage: rcm_rce --atm FILE (--table FILE | --lbl DIR [--co2-factor F]) [--ncol N] [--seed S] [--max-steps M] [--check-every K] "
                             "[--dT K/step] [--device D] [--out FILE] [--checkpoint FILE] [--resume FILE] [--steps-exact] [--gpus N] "
                             "[--spectral-out FILE] [--kernels-out FILE] [--jacobian-out FILE] "
                             "[--forcing-out FILE [--forcing-scale 1,2,1,1,1] [--trop-layers 4]] "
                             "[--lbl-bands-out FILE [--band-size 100] [--forcing-scale 1,2,1,1,1]] [--lbl-kernels-out FILE] "
                             "[--lbl-jacobian-out FILE] [--lbl-forcing-out FILE [--forcing-scale 1,2,1,1,1] [--trop-layers 4]] "
                             "[--response-out FILE [--forcing-scale 1,2,1,1,1] [--trop-layers 4] [--fixed-q]] "
                             "[--lbl-response-out FILE [--forcing-scale 1,2,1,1,1] [--trop-layers 4] [--fixed-q]] "
                             "[--species-jacobian-out FILE] [--lbl-species-jacobian-out FILE]\n");
        return 1;
    }
    if (!lbl_dir.empty() && !spectral_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --spectral-out needs a repwvl table (--table): the line-by-line path has no diagnostic call\n");
        return 1;
    }
    if (!lbl_dir.empty() && !kernels_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --kernels-out needs a repwvl table (--table): with --lbl use --lbl-kernels-out\n");
        return 1;
    }
    if (!lbl_dir.empty() && !jacobian_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --jacobian-out needs a repwvl table (--table): with --lbl use --lbl-jacobian-out\n");
        return 1;
    }
    if (!lbl_dir.empty() && !forcing_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --forcing-out needs a repwvl table (--table): with --lbl use --lbl-forcing-out\n");
        return 1;
    }
    if (lbl_dir.empty() && !lbl_kernels_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --lbl-kernels-out needs line-by-line tables (--lbl)\n");
        return 1;
    }
    if (!lbl_kernels_path.empty()) kernels_path = lbl_kernels_path;  // the same kernels file, from the LBL call
    if (lbl_dir.empty() && !lbl_jacobian_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --lbl-jacobian-out needs line-by-line tables (--lbl)\n");
        return 1;
    }
    if (!lbl_jacobian_path.empty()) jacobian_path = lbl_jacobian_path;  // the same Jacobian file, from the LBL call
    if (lbl_dir.empty() && !lbl_forcing_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --lbl-forcing-out needs line-by-line tables (--lbl)\n");
        return 1;
    }
    if (!lbl_forcing_path.empty()) forcing_path = lbl_forcing_path;  // the same forcing file, from the LBL call
    if (!lbl_dir.empty() && !response_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --response-out needs a repwvl table (--table): with --lbl use --lbl-response-out\n");
        return 1;
    }
    if (lbl_dir.empty() && !lbl_response_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --lbl-response-out needs line-by-line tables (--lbl)\n");
        return 1;
    }
    if (!lbl_response_path.empty()) response_path = lbl_response_path;  // the same response file, from the LBL call
    if (!lbl_dir.empty() && !species_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --species-jacobian-out needs a repwvl table (--table): with --lbl use --lbl-species-jacobian-out\n");
        return 1;
    }
    if (lbl_dir.empty() && !lbl_species_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --lbl-species-jacobian-out needs line-by-line tables (--lbl)\n");
        return 1;
    }
    if (!lbl_species_path.empty()) species_path = lbl_species_path;  // the same species file, from the LBL call
    if (lbl_dir.empty() && !bands_path.empty()) {
        std::fprintf(stderr, "rcm_rce: --lbl-bands-out needs line-by-line tables (--lbl)\n");
        return 1;
    }
    double forcing_scale[5];
    int trop_layers = 0, band_size = 0;
    if (!bands_path.empty()) {  // --forcing-scale: exactly five numbers; --band-size: an integer >= 1
        int k = 0;
        const char* q = forcing_scale_arg.c_str();
        for (char* e = nullptr; k < 5; ++k, q = e + 1) {
            forcing_scale[k] = std::strtod(q, &e);
            if (e == q || (k < 4 && *e != ',') || (k == 4 && *e != '\0')) break;
        }
        char* e = nullptr;
        const long bs = std::strtol(band_size_arg.c_str(), &e, 10);
        if (k < 5 || e == band_size_arg.c_str() || *e != '\0' || bs < 1 || bs > 1000000000L) {
            std::fprintf(stderr, "rcm_rce: --forcing-scale needs five comma-separated factors and --band-size an integer >= 1\n");
            return 1;
        }
        band_size = (int)bs;
    }
    if (!forcing_path.empty() || !response_path.empty()) {  // --forcing-scale: five numbers; --trop-layers: an integer in [0, 19]
        int k = 0;
        const char* q = forcing_scale_arg.c_str();
        for (char* e = nullptr; k < 5; ++k, q = e + 1) {
            forcing_scale[k] = std::strtod(q, &e);
            if (e == q || (k < 4 && *e != ',') || (k == 4 && *e != '\0')) break;
        }
        char* e = nullptr;
        const long tl = std::strtol(trop_layers_arg.c_str(), &e, 10);
        if (k < 5 || e == trop_layers_arg.c_str() || *e != '\0' || tl < 0 || tl > RCM_NLAYER - 1) {
            std::fprintf(stderr, "rcm_rce: --forcing-scale needs five comma-separated factors and --trop-layers an integer in [0, 19]\n");
            return 1;
        }
        trop_layers = (int)tl;
    }

    // ---- the column of the .atm file (main.cpp:396-430) and its ensemble ---------------------------
    constexpr int NLEV = RCM_NLEVEL, NLAY = RCM_NLAYER;
    std::vector<double> cols(9 * NLEV);
    int nrows = 0, nc = 0;
    int st = rcm_read_atm(atm_path.c_str(), NLEV, cols.data(), &nrows, &nc);
    if (st != RCM_OK) return die(atm_path.c_str(), st, nullptr);
    const bool lbl = !lbl_dir.empty();
    if (nrows != NLEV || nc < (lbl ? 6 : 9)) {
        std::fprintf(stderr, "rcm_rce: %s: need 21 levels x %d columns (z p T air H2O O3%s), got %d x %d\n", atm_path.c_str(),
                     lbl ? 6 : 9, lbl ? "" : " CO2 CH4 N2O", nrows, nc);
        return 1;
    }
    if (nc < 9) {  // lbl.arts/README:13-16
        const double well_mixed[3] = {400.0, 1.7, 0.315};
        for (int k = 0; k < 3; ++k)
            for (int i = 0; i < NLEV; ++i) cols[(6 + k) * NLEV + i] = well_mixed[k];
    }
    const double* plevel = &cols[1 * NLEV];
    const double* Tbase = &cols[2 * NLEV];
    const double* vbase = &cols[4 * NLEV];  // H2O, O3, CO2, CH4, N2O: five consecutive columns
    const size_t n = (size_t)ncol;
    std::vector<double> Tlevel(n * NLEV), vlev(n * 5 * NLEV);
    st = rcm_make_ensemble(ncol, seed, plevel, Tbase, vbase, Tlevel.data(), vlev.data());
    if (st != RCM_OK) return die("rcm_make_ensemble", st, nullptr);
    std::vector<double> Tlayer(n * NLAY), vmr9(n * RCM_NSPECIES * NLAY), rel_hum(n * NLAY), player(NLAY), conv(NLAY);
    st = rcm_init_columns(ncol, plevel, Tlevel.data(), vlev.data(), 1.0, Tlayer.data(), vmr9.data(), rel_hum.data(),
                          player.data(), conv.data());  // main.cpp:439-479
    if (st != RCM_OK) return die("rcm_init_columns", st, nullptr);
    std::vector<double> Tsurf(n, 288.2);  // main.cpp:357

    // ---- constants, solar setup (main.cpp:214-264), solver, table ---------------------------------
    rcm_params p;
    rcm_default_params(&p);
    rcm_solar_params sp;
    rcm_default_solar_params(&sp);
    double sol[7];
    rcm_solar_setup(&sp, sol);
    p.solar_irr = sol[6];
    p.dT_converged = dT;
    if (gpus > 1) {
        // ---- one thread and one solver per GPU, NCCL for the block scalars --------------------------------------
        if (rcm_device_count() < gpus) {
            std::fprintf(stderr, "rcm_rce: --gpus %d but %d CUDA device(s) visible\n", gpus, rcm_device_count());
            return 1;
        }
        rcm_table* table = nullptr;
        std::vector<double> wvl, tau5;
        int nwvl = 0;
        if (lbl) {
            const char* names[5] = {"h2o", "co2", "o3", "ch4", "n2o"};
            for (int k = 0; k < 5; ++k) {
                const std::string path = lbl_dir + "/lbl." + names[k] + ".asc";
                int nx = 0, ny = 0;
                double *x = nullptr, *y = nullptr;
                const int rc = rcm_ascii_file2xy2D(path.c_str(), &nx, &ny, &x, &y);
                if (rc != 0 || ny != NLAY || nx < 2 || (k > 0 && (nx != nwvl || std::memcmp(wvl.data(), x, (size_t)nx * sizeof(double)) != 0))) {
                    std::fprintf(stderr, "rcm_rce: %s: reader status %d, %d wavelengths x %d layers\n", path.c_str(), rc, nx, ny);
                    return 1;
                }
                if (k == 0) {
                    nwvl = nx;
                    wvl.assign(x, x + nx);
                    tau5.resize((size_t)5 * nx * NLAY);
                }
                std::memcpy(&tau5[(size_t)k * nx * NLAY], y, (size_t)nx * NLAY * sizeof(double));
                rcm_free(x);
                rcm_free(y);
            }
        } else {
            st = rcm_table_load(table_path.c_str(), &table);
            if (st != RCM_OK) return die(table_path.c_str(), st, nullptr);
        }
        std::vector<double> T(n * NLAY), Ts(n), Eu(n * NLEV);
        std::vector<float> time_h(n);
        int dims[4] = {0, 0, 0, 0};
        std::vector<double> olr, sfc;
        if (!spectral_path.empty()) {
            rcm_table_dims(table, dims);
            olr.resize(n * dims[2]);
            sfc.resize(n * dims[2]);
        }
        std::vector<double> K(kernels_path.empty() ? 0 : n * KERN_NK);
        std::vector<double> H(jacobian_path.empty() ? 0 : n * JAC_NH);
        const bool forcing = !forcing_path.empty();
        std::vector<double> Ff(forcing ? n * 4 : 0), dTf(forcing ? n * NLAY : 0);
        std::vector<int> itf(forcing ? n : 0), ntrop(n, trop_layers);
        const bool response = !response_path.empty();
        std::vector<double> Fr(response ? n * 2 : 0), dTr(response ? n * NLAY : 0), dTsr(response ? n : 0);
        std::vector<int> itr(response ? n : 0);
        std::vector<double> S(species_path.empty() ? 0 : n * 3 * SPJ_NE);
        const std::vector<int> bstart = bands_path.empty() ? std::vector<int>() : lbl_band_starts(nwvl, band_size);
        const int nband = bands_path.empty() ? 0 : (int)bstart.size() - 1;
        std::vector<double> B(n * nband * 4);
        Job job{&p, table, &wvl, &tau5, nwvl, co2_factor, plevel, Tlayer.data(), Tsurf.data(), vmr9.data(), rel_hum.data(), ncol,
                max_steps, check_every, steps_exact, resume_path, ckpt_path, T.data(), Ts.data(), Eu.data(), time_h.data(),
                dims[2], olr.data(), sfc.data(), !kernels_path.empty(), K.data(), !jacobian_path.empty(), H.data(),
                forcing, forcing_scale, ntrop.data(), Ff.data(), dTf.data(), itf.data(), nband, bstart.data(), B.data(),
                response, fixed_rh, Fr.data(), dTr.data(), dTsr.data(), itr.data(), !species_path.empty(), S.data()};
        std::vector<Shard> shards((size_t)gpus);
        std::vector<ncclComm_t> comms((size_t)gpus);
        std::vector<int> devs((size_t)gpus);
        for (int d = 0; d < gpus; ++d) devs[d] = d;
        if (ncclCommInitAll(comms.data(), gpus, devs.data()) != ncclSuccess) {
            std::fprintf(stderr, "rcm_rce: ncclCommInitAll failed for %d GPUs\n", gpus);
            return 1;
        }
        const int base = ncol / gpus, rem = ncol % gpus;  // contiguous blocks, sizes differ by at most one
        for (int d = 0, lo = 0; d < gpus; ++d) {
            shards[d].dev = d;
            shards[d].lo = lo;
            shards[d].hi = lo += base + (d < rem ? 1 : 0);
            shards[d].comm = comms[d];
        }
        std::vector<std::thread> th;
        for (int d = 0; d < gpus; ++d) th.emplace_back(run_shard, &shards[d], &job);
        for (auto& t : th) t.join();
        int bad = 0;
        for (auto& sh : shards)
            if (!sh.err.empty()) {
                std::fprintf(stderr, "rcm_rce: GPU %d: %s\n", sh.dev, sh.err.c_str());
                bad = 1;
            }
        for (auto& sh : shards) {
            if (sh.s) rcm_destroy(sh.s);
            if (sh.comm) ncclCommDestroy(sh.comm);
        }
        if (bad) {
            if (table) rcm_table_free(table);
            return 1;
        }
        if (!spectral_path.empty() &&
            write_spectrum(spectral_path, ncol, dims[2], rcm_table_array(table, 1), rcm_table_array(table, 2), olr.data(), sfc.data())) {
            rcm_table_free(table);
            return 1;
        }
        if (!kernels_path.empty() && write_kernels(kernels_path, ncol, player.data(), plevel[NLAY], K.data())) {
            rcm_table_free(table);
            return 1;
        }
        if (!jacobian_path.empty() && write_jacobian(jacobian_path, ncol, player.data(), H.data())) {
            rcm_table_free(table);
            return 1;
        }
        if (forcing && write_forcing(forcing_path, ncol, player.data(), Ff.data(), dTf.data(), itf.data())) {
            rcm_table_free(table);
            return 1;
        }
        if (response && write_response(response_path, ncol, player.data(), Fr.data(), dTr.data(), dTsr.data(), itr.data())) {
            rcm_table_free(table);
            return 1;
        }
        if (!species_path.empty() && write_species(species_path, ncol, player.data(), S.data())) {
            rcm_table_free(table);
            return 1;
        }
        if (nband > 0 && write_lbl_bands(bands_path, ncol, wvl, bstart, B.data())) return 1;
        if (table) rcm_table_free(table);
        st = rcm_write_profiles(out_path.c_str(), 0, 1, ncol, plevel, T.data(), time_h.data(), ncol > 1);
        if (st != RCM_OK) return die(out_path.c_str(), st, nullptr);
        const rcm_step_scalars& last = shards[0].last;
        double ts_mean = 0.0;
        for (size_t c = 0; c < n; ++c) ts_mean += Ts[c];
        double loop_s = 0.0;
        for (auto& sh : shards) loop_s = sh.loop_s > loop_s ? sh.loop_s : loop_s;
        std::printf("rcm_rce: %d columns on %d GPUs, %ld iterations, %d/%d stationary (< %g K per step), max dT %.3e K, mean TOA net %.4f W/m2, "
                    "mean T_surface %.4f K, member 0: T_surface %.6f K, OLR %.6f W/m2, time %.2f h\n",
                    ncol, gpus, shards[0].done, (int)last.n_converged, ncol, dT, last.max_dT, last.toa_net_sum / ncol, ts_mean / ncol,
                    Ts[0], Eu[0], (double)time_h[0]);
        std::printf("rcm_rce: time loop %.4f s on the slowest GPU = %.4f ms per iteration\n", loop_s, 1e3 * loop_s / (double)shards[0].done);
        return 0;
    }
    std::vector<double> spec_wvl, spec_weight;  // --spectral-out: the table's wavelengths and weights
    std::vector<double> lbl_wvl;                // --lbl-bands-out: the LBL wavelengths
    rcm_solver* s = nullptr;
    st = rcm_create(device, &p, &s);
    if (st != RCM_OK) return die("rcm_create", st, nullptr);
    if (lbl) {
        // the five species tables, README order of the composition: H2O, CO2, O3, CH4, N2O (rcm_set_lbl_tables)
        const char* names[5] = {"h2o", "co2", "o3", "ch4", "n2o"};
        std::vector<double> wvl, tau5;
        int nwvl = 0;
        for (int k = 0; k < 5; ++k) {
            const std::string path = lbl_dir + "/lbl." + names[k] + ".asc";
            int nx = 0, ny = 0;
            double *x = nullptr, *y = nullptr;
            const int rc = rcm_ascii_file2xy2D(path.c_str(), &nx, &ny, &x, &y);  // 0, or the reference's -1 / -2 / -5
            if (rc != 0 || ny != NLAY || nx < 2 || (k > 0 && nx != nwvl)) {
                std::fprintf(stderr, "rcm_rce: %s: reader status %d, %d wavelengths x %d layers (need the same wavelengths in "
                                     "all five files and 20 layers)\n", path.c_str(), rc, nx, ny);
                return 1;
            }
            if (k == 0) {
                nwvl = nx;
                wvl.assign(x, x + nx);
                tau5.resize((size_t)5 * nx * NLAY);
            } else if (std::memcmp(wvl.data(), x, (size_t)nx * sizeof(double)) != 0) {
                std::fprintf(stderr, "rcm_rce: %s: wavelength grid differs from lbl.h2o.asc\n", path.c_str());
                return 1;
            }
            std::memcpy(&tau5[(size_t)k * nx * NLAY], y, (size_t)nx * NLAY * sizeof(double));
            rcm_free(x);
            rcm_free(y);
        }
        // reference profiles of the tables = the .atm file's own column = member 0 (layer VMRs, species 0 and 2 of vmr9)
        st = rcm_set_lbl_tables(s, wvl.data(), tau5.data(), nwvl, &vmr9[0 * NLAY], &vmr9[2 * NLAY], co2_factor);
        if (st != RCM_OK) return die("rcm_set_lbl_tables", st, s);
        lbl_wvl = wvl;
    } else {
        rcm_table* t = nullptr;
        st = rcm_table_load(table_path.c_str(), &t);
        if (st != RCM_OK) return die(table_path.c_str(), st, s);
        st = rcm_set_repwvl_table_from(s, t);
        int dims[4] = {0, 0, 0, 0};
        rcm_table_dims(t, dims);
        spec_wvl.assign(rcm_table_array(t, 1), rcm_table_array(t, 1) + dims[2]);
        spec_weight.assign(rcm_table_array(t, 2), rcm_table_array(t, 2) + dims[2]);
        rcm_table_free(t);
        if (st != RCM_OK) return die("rcm_set_repwvl_table_from", st, s);
    }
    if (!resume_path.empty()) {
        st = rcm_load_checkpoint(s, resume_path.c_str());
        if (st != RCM_OK) return die(resume_path.c_str(), st, s);
        ncol = rcm_column_count(s);
    } else {
        st = rcm_set_columns(s, ncol, plevel, Tlayer.data(), Tsurf.data(), vmr9.data(), rel_hum.data());
        if (st != RCM_OK) return die("rcm_set_columns", st, s);
    }

    // ---- the time loop (main.cpp:531-583), in blocks of check_every fused iterations ---------------
    rcm_step_scalars last{};
    long done = 0;
    rcm_synchronize(s);
    const auto t0 = std::chrono::steady_clock::now();
    if (steps_exact) {
        std::vector<rcm_step_scalars> sc((size_t)check_every);
        while (done < max_steps) {
            const int k = (int)((max_steps - done < check_every) ? (max_steps - done) : check_every);
            st = rcm_advance(s, k, sc.data());
            if (st != RCM_OK) return die("rcm_advance", st, s);
            last = sc[k - 1];
            done += k;
        }
    } else {
        st = rcm_run_to_equilibrium(s, max_steps, check_every, &last, &done);
        if (st != RCM_OK) return die("rcm_run_to_equilibrium", st, s);
    }

    rcm_synchronize(s);
    const double loop_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    // ---- results: the reference's rows for every member, optional checkpoint -----------------------
    const size_t m = (size_t)ncol;
    std::vector<double> T(m * NLAY), Ts(m), Eu(m * NLEV);
    std::vector<float> time_h(m);
    st = rcm_get_state(s, T.data(), Ts.data(), nullptr, time_h.data(), nullptr, Eu.data(), nullptr, nullptr);
    if (st != RCM_OK) return die("rcm_get_state", st, s);
    st = rcm_write_profiles(out_path.c_str(), /*append*/ 0, /*header*/ 1, ncol, plevel, T.data(), time_h.data(),
                            /*column ids*/ ncol > 1);
    if (st != RCM_OK) return die(out_path.c_str(), st, s);
    if (!ckpt_path.empty()) {
        st = rcm_save_checkpoint(s, ckpt_path.c_str());
        if (st != RCM_OK) return die(ckpt_path.c_str(), st, s);
    }
    if (!spectral_path.empty()) {
        const int nw = (int)spec_wvl.size();
        std::vector<double> olr(m * nw), sfc(m * nw);
        st = diagnose_spectrum(s, ncol, nw, olr.data(), sfc.data());
        if (st != RCM_OK) return die("rcm_diagnose_fluxes", st, s);
        if (write_spectrum(spectral_path, ncol, nw, spec_wvl.data(), spec_weight.data(), olr.data(), sfc.data())) return 1;
    }
    if (!kernels_path.empty()) {
        std::vector<double> K(m * KERN_NK);
        st = lbl ? rcm_lbl_radiative_kernels(s, 0, ncol, nullptr, 0, nullptr, nullptr, K.data())
                 : rcm_radiative_kernels(s, 0, ncol, nullptr, nullptr, K.data());
        if (st != RCM_OK) return die(lbl ? "rcm_lbl_radiative_kernels" : "rcm_radiative_kernels", st, s);
        if (write_kernels(kernels_path, ncol, player.data(), plevel[NLAY], K.data())) return 1;
    }
    if (!jacobian_path.empty()) {
        std::vector<double> H(m * JAC_NH);
        st = (lbl ? rcm_lbl_flux_jacobian : rcm_flux_jacobian)(s, 0, ncol, nullptr, nullptr, H.data());
        if (st != RCM_OK) return die(lbl ? "rcm_lbl_flux_jacobian" : "rcm_flux_jacobian", st, s);
        if (write_jacobian(jacobian_path, ncol, player.data(), H.data())) return 1;
    }
    if (!forcing_path.empty()) {
        std::vector<double> Ff(m * 4), dTf(m * NLAY);
        std::vector<int> itf(m), ntrop(m, trop_layers);
        st = (lbl ? rcm_lbl_adjusted_forcing : rcm_adjusted_forcing)(s, 0, ncol, forcing_scale, ntrop.data(), FORCING_TOL,
                                                                    FORCING_MAX_ITER, Ff.data(), dTf.data(), nullptr, nullptr, itf.data());
        if (st != RCM_OK) return die(lbl ? "rcm_lbl_adjusted_forcing" : "rcm_adjusted_forcing", st, s);
        if (write_forcing(forcing_path, ncol, player.data(), Ff.data(), dTf.data(), itf.data())) return 1;
    }
    if (!response_path.empty()) {
        std::vector<double> Fr(m * 2), dTr(m * NLAY), dTsr(m);
        std::vector<int> itr(m), ntrop(m, trop_layers);
        st = (lbl ? rcm_lbl_climate_response : rcm_climate_response)(s, 0, ncol, forcing_scale, ntrop.data(), fixed_rh, FORCING_TOL,
                                                                    FORCING_MAX_ITER, Fr.data(), dTr.data(), dTsr.data(), nullptr,
                                                                    nullptr, itr.data());
        if (st != RCM_OK) return die(lbl ? "rcm_lbl_climate_response" : "rcm_climate_response", st, s);
        if (write_response(response_path, ncol, player.data(), Fr.data(), dTr.data(), dTsr.data(), itr.data())) return 1;
    }
    if (!species_path.empty()) {
        std::vector<double> S(m * 3 * SPJ_NE);
        st = species_rows(s, lbl, ncol, S.data());
        if (st != RCM_OK) return die(lbl ? "rcm_lbl_species_jacobian" : "rcm_species_jacobian", st, s);
        if (write_species(species_path, ncol, player.data(), S.data())) return 1;
    }
    if (!bands_path.empty()) {
        const std::vector<int> bstart = lbl_band_starts((int)lbl_wvl.size(), band_size);
        const int nband = (int)bstart.size() - 1;
        std::vector<double> B(m * nband * 4);
        st = diagnose_lbl_bands(s, ncol, nband, bstart.data(), forcing_scale, B.data());
        if (st != RCM_OK) return die("rcm_lbl_diagnose_fluxes", st, s);
        if (write_lbl_bands(bands_path, ncol, lbl_wvl, bstart, B.data())) return 1;
    }
    double ts_mean = 0.0;
    for (size_t c = 0; c < m; ++c) ts_mean += Ts[c];
    std::printf("rcm_rce: %d columns, %ld iterations, %d/%d stationary (< %g K per step), max dT %.3e K, mean TOA net %.4f W/m2, "
                "mean T_surface %.4f K, member 0: T_surface %.6f K, OLR %.6f W/m2, time %.2f h\n",
                ncol, done, (int)last.n_converged, ncol, dT, last.max_dT, last.toa_net_sum / ncol, ts_mean / ncol, Ts[0], Eu[0],
                (double)time_h[0]);
    std::printf("rcm_rce: time loop %.4f s = %.4f ms per iteration\n", loop_s, 1e3 * loop_s / (double)done);
    rcm_destroy(s);
    return 0;
}
