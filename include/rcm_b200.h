/*
 * rcm_b200.h - C ABI of the B200-native radiative-convective column solver.
 *
 * Drop-in boundary for the thermal hot path of pabloconrat/our_first_climate_model
 * (reference loop body main.cpp:531-583).  The reference has no plugin/FFI layer: its
 * boundary is a handful of C++ free functions.  Every entry point below names the
 * reference interface it replaces.  Plain pointers and sizes only; all host buffers are
 * caller-owned; every function returns an rcm_status (never exits, never throws).
 * One rcm_solver per GPU; calls on one solver are not re-entrant.
 *
 * Array conventions (identical to the reference's): layers/levels are TOP-DOWN (index 0 =
 * top of atmosphere), pressures in hPa, volume mixing ratios as fractions, tau[iwvl][ilyr].
 * The nine species are in read_tau's argument order (repwvl_thermal.h:3-7):
 *   0 H2O, 1 CO2, 2 O3, 3 N2O, 4 CO, 5 CH4, 6 O2, 7 HNO3, 8 N2.
 */
#ifndef RCM_B200_H
#define RCM_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RCM_NLAYER 20 /* Consts::nlayer, main.cpp:78 */
#define RCM_NLEVEL 21 /* Consts::nlevel, main.cpp:79 */
#define RCM_NSPECIES 9

typedef enum {
    RCM_OK = 0,
    RCM_ERR_ARG = 1,      /* bad argument (NULL, size, unsupported dimension) */
    RCM_ERR_STATE = 2,    /* call order (no table / no columns loaded yet) */
    RCM_ERR_CUDA = 3,     /* CUDA runtime error; see rcm_last_error() */
    RCM_ERR_IO = 4,       /* file not found / unreadable */
    RCM_ERR_FORMAT = 5,   /* file is not a supported table / matrix */
    RCM_ERR_NOMEM = 6,
    RCM_ERR_NO_DEVICE = 7 /* no CUDA device: the solver has no CPU fallback */
} rcm_status;

typedef struct rcm_solver rcm_solver; /* opaque, one per GPU */
typedef struct rcm_table rcm_table;   /* opaque host copy of a repwvl lookup table */

/* Model constants; rcm_default_params() fills in the reference's `Consts` (main.cpp:66-92). */
typedef struct {
    int nangle;        /* 30  Consts::nangle (1..64) */
    int cloud_layer;   /* 17  Consts::cloud_layer; < 0 = no grey cloud (cloud_into_tau, main.cpp:266-274) */
    double cloud_tau;  /* 1.0 Consts::tau_s / 2 */
    double dp;         /* 50  hPa, 1000/nlayer (main.cpp:355) */
    double max_dT;     /* 5   K, Consts::max_dT (calculate_timestep, main.cpp:156-162) */
    double dt_cap;     /* 43200 s (main.cpp:158-160) */
    double solar_irr;  /* W/m2, from rcm_solar_setup() (236.882897... for the committed Consts) */
    double dT_converged; /* K, stationarity threshold used for the `converged` count (not in the reference) */
    unsigned species_mask; /* bit s set: species s contributes to tau. Species outside the mask must have
                              VMR == 0 (they then add exactly +0.0 as in repwvl_thermal.cpp:244).
                              Default 0x2F = H2O, CO2, O3, N2O, CH4 - what main.cpp:452-460 feeds. */
} rcm_params;

typedef struct {
    double tau_s, mu_s, g_asym, albedo, daytime, E_0;
    int doublings;
} rcm_solar_params; /* Consts of main.cpp:86-91 */

/* Per-step ensemble diagnostics: the only quantities that ever cross GPUs (one allreduce). */
typedef struct {
    double toa_net_sum; /* sum over columns of solar_irr - E_up[0]  (W/m2) */
    double max_dT;      /* max over columns, layers of |T_sorted(n) - T_sorted(n-1)|  (K) */
    double n_converged; /* number of columns with that change < dT_converged */
    double max_abs_dE;  /* max over columns, layers of |dE| (W/m2) */
} rcm_step_scalars;

/* ---- host-only helpers (no GPU needed) ------------------------------------------------- */
const char* rcm_status_string(int status);
int rcm_default_params(rcm_params* p);
int rcm_default_solar_params(rcm_solar_params* sp);
/* doubling_adding + solar_radiative_transfer_setup (main.cpp:214-264).
 * out7 = r_dir, s_dir, t_dir, r, t, r_total (planetary albedo), solar_irr. */
int rcm_solar_setup(const rcm_solar_params* sp, double* out7);
/* LowerPos (repwvl_thermal.cpp:19-45): index of the table interval used for x. */
long rcm_lowerpos(const double* nodes, int n, double x);

/* Lookup-table loader.  Replaces the NetCDF part of read_tau (repwvl_thermal.cpp:113-176):
 * reads Reduced{10,20,100}Forcing.nc (NetCDF-4/HDF5 subset, SURVEY.md Appendix B) or the flat
 * .rcmtab form of the same data. */
int rcm_table_load(const char* path, rcm_table** out);
void rcm_table_free(rcm_table* t);
/* dims4 = n_tpert (xsec_nbooks), n_species (npages), n_wvl (nrows), n_p (ncols) */
int rcm_table_dims(const rcm_table* t, int* dims4);
/* which: 0 xsec, 1 wvl (ChosenWvls), 2 weight (ChosenWeights), 3 p_grid, 4 t_ref, 5 t_pert, 6 vmrs_ref */
const double* rcm_table_array(const rcm_table* t, int which);

/* 21-level atmosphere file (test.atm / fpda.lbl.atm layout, main.cpp:396-430): skips 4 header
 * lines, reads up to 9 whitespace-separated columns per row.  cols_out [9][max_rows]
 * (column-major per variable: z, p, T, air, H2O, O3, CO2, CH4, N2O); *ncols_out = columns found. */
int rcm_read_atm(const char* path, int max_rows, double* cols_out, int* nrows_out, int* ncols_out);

/* Level -> layer initialisation, the inline part of main() (main.cpp:439-479).
 * Tlevel [ncol][21]; vmr_ppm_level [ncol][5][21] in file order H2O, O3, CO2, CH4, N2O.
 * Outputs: Tlayer [ncol][20], vmr9 [ncol][9][20], rel_hum [ncol][20], player[20], conv[20]. */
int rcm_init_columns(int ncol, const double* plevel_hPa, const double* Tlevel, const double* vmr_ppm_level,
                     double co2_factor, double* Tlayer, double* vmr9, double* rel_hum, double* player,
                     double* conv);

/* Synthetic perturbed-profile ensemble (SURVEY.md section 8(d)); deterministic in `seed`.
 * base_* are one 21-level column; outputs Tlevel [ncol][21], vmr_ppm_level [ncol][5][21]. */
int rcm_make_ensemble(int ncol, unsigned long long seed, const double* plevel_hPa, const double* base_Tlevel,
                      const double* base_vmr_ppm_level, double* Tlevel, double* vmr_ppm_level);

/* Line-by-line table reader: result-identical replacement of ASCII_file2xy2D
 * (lbl.arts/ascii.cpp:1631-1691, ascii.h:63) with flat, caller-freed output.
 * *x [nx], *y [nx*ny] are malloc'ed; free with rcm_free().  Returns 0 or the reference's
 * negative codes: -1 not found, -2 no memory, -5 not rectangular (ascii.h:34-38). */
int rcm_ascii_file2xy2D(const char* filename, int* nx, int* ny, double** x, double** y);
void rcm_free(void* p);
/* Band-integrated Planck radiance (cplkavg.cpp:124-243) on the host; *status as below. */
double rcm_cplkavg_host(double wvllo_nm, double wvlhi_nm, double t, int* status);

/* ---- solver lifecycle ------------------------------------------------------------------ */
int rcm_device_count(void);
int rcm_create(int device, const rcm_params* p, rcm_solver** out);
int rcm_destroy(rcm_solver* s);
const char* rcm_last_error(const rcm_solver* s);
int rcm_set_params(rcm_solver* s, const rcm_params* p);
/* Solver options.  RCM_OPT_ANGLE_CUBES (default 1): visit the quadrature angles in chains
 * mu, mu/3, mu/9 so that two thirds of the transmissions need an exp and the rest are cubes
 * of the previous ones (same mu values, different summation order, ~1e-15 relative). */
#define RCM_OPT_ANGLE_CUBES 0
/* RCM_OPT_ANGLE_PAIRS (default 1, needs the cubes): two chain heads whose node numbers satisfy 3a = 5b, 5a = 7b or
 * 3a = 7b take their transmissions as powers of ONE exp at a virtual node (30 angles: 4 of the 20 exp's per layer
 * and wavelength become 3-4 multiplications; same mu values, ~1e-14 relative). */
#define RCM_OPT_ANGLE_PAIRS 4
/* RCM_OPT_PATH (default 0): 0 = split path ((tile, wavelength-split) units, results independent of shard / GPU count),
 * 1 = the fused tile kernel of round 1 (comparison).  RCM_OPT_MULTI_STEP (default 1, split path): rcm_advance(n >= 2) runs
 * its n steps as ONE persistent launch with per-tile step flags instead of kernel boundaries where a step is only a few
 * rounds of work units per CTA (up to ~34,000 columns per GPU); 0 = always three launches per step, 2 = always one launch.
 * Bit-identical either way. */
#define RCM_OPT_PATH 5
#define RCM_OPT_MULTI_STEP 6
int rcm_set_option(rcm_solver* s, int option, int value);
/* cudaStream_t to launch on (NULL = the solver's own stream). */
int rcm_set_stream(rcm_solver* s, void* cuda_stream);
int rcm_synchronize(rcm_solver* s);

/* Upload a repwvl table (arrays as read by rcm_table_load; xsec in the file's
 * [n_tpert][n_species][n_wvl][n_p] order - the solver re-lays it out for the GPU). */
int rcm_set_repwvl_table(rcm_solver* s, const double* xsec, const double* wvl, const double* weight,
                         const double* p_grid, const double* t_ref, const double* t_pert, int n_tpert,
                         int n_species, int n_wvl, int n_p);
int rcm_set_repwvl_table_from(rcm_solver* s, const rcm_table* t);
/* Wavelengths [nm] and spectral weights alone (what radiative_transfer, main.cpp:320-344, is handed):
 * enough for rcm_radiative_transfer with a caller-supplied tau. */
int rcm_set_spectral_grid(rcm_solver* s, const double* wvl, const double* weight, int n_wvl);

/* Upload line-by-line tables (lbl.arts/README:5-16) and switch the solver to the LBL path:
 * wvl [nwvl] nm ascending, tau5 [5][nwvl][20] in the order H2O, CO2, O3, CH4, N2O (top-down layers, as
 * read by rcm_ascii_file2xy2D), h2o_ref / o3_ref [20] = layer VMRs the H2O / O3 tables were computed for
 * (o3_ref NULL: O3 table used unscaled), co2_factor as `factor` in main.cpp:452-456.
 * tau = tau_H2O*(H2O/h2o_ref) + co2_factor*tau_CO2 + tau_O3*(O3/o3_ref) + tau_CH4 + tau_N2O; the source is
 * cplkavg() over bins bounded by the midpoints between adjacent wavelengths (DESIGN.md section 5). */
int rcm_set_lbl_tables(rcm_solver* s, const double* wvl, const double* tau5, int nwvl, const double* h2o_ref,
                       const double* o3_ref, double co2_factor);
/* Synthetic LBL tables in the reference's format (the real lbl.*.asc are not distributed):
 * wvl [nwvl] log-spaced 4-100 um, tau5 [5][nwvl][20]; deterministic in seed. */
int rcm_make_lbl_tables(int nwvl, unsigned long long seed, const double* plevel_hPa, const double* h2o_vmr_layer,
                        const double* o3_vmr_layer, double* wvl, double* tau5);
/* Write one species table as text: "wavelength[nm] dtau(20 layers, top-down)" per line (lbl.arts/README:5-11). */
int rcm_write_lbl_asc(const char* path, int nwvl, const double* wvl, const double* tau);

/* Column state.  plevel_hPa [21] is shared by the ensemble.  Tlayer [ncol][20], Tsurf [ncol],
 * vmr9 [ncol][9][20], rel_hum [ncol][20].  Resets the step counter to 0 (the first step then
 * uses tau of the initial, unsorted profile exactly as main.cpp:500-504 does). */
int rcm_set_columns(rcm_solver* s, int ncol, const double* plevel_hPa, const double* Tlayer,
                    const double* Tsurf, const double* vmr9, const double* rel_hum);
/* Compact per-step upload for resident ensembles: only T, Tsurf and the H2O..CH4 rows named in
 * species_mask (vmr_active [ncol][n_active][20], ascending species index).  Keeps plevel/rel_hum. */
/* Per-column solar forcing, computed on the device (SURVEY 8(f)3): doubling_adding + solar_radiative_transfer_setup
 * (main.cpp:214-264) with one cloud optical depth / zenith cosine / surface albedo per column.  tau_s, mu_s, albedo:
 * host arrays [ncol] or NULL (then the scalar in *sp).  From the next step on, column c is heated by its own
 * solar_irr[c] instead of rcm_params::solar_irr (main.cpp:341); with cloud_from_tau_s != 0 the thermal grey cloud of
 * column c becomes tau_s[c] / 2 instead of rcm_params::cloud_tau (main.cpp:266-274).  Optional outputs (host, [ncol]):
 * solar_irr_out, r_total_out (planetary albedo).  sp == NULL switches back to the ensemble-wide constants.
 * rcm_set_columns() drops the per-column forcing: call this after it. */
int rcm_set_column_solar(rcm_solver* s, const rcm_solar_params* sp, const double* tau_s, const double* mu_s,
                         const double* albedo, int cloud_from_tau_s, double* solar_irr_out, double* r_total_out);
int rcm_update_columns(rcm_solver* s, const double* Tlayer, const double* Tsurf, const double* vmr_active);
int rcm_set_step_index(rcm_solver* s, long step_index);

/* K1 only: optical depth build = compute part of read_tau (repwvl_thermal.cpp:197-248) +
 * cloud_into_tau (main.cpp:266-274).  tau_out [ncol][nwvl][20] host (NULL = skip the copy);
 * lowpos_p / lowpos_t [ncol][20] in the reference's bottom-up layer order (NULL = skip). */
int rcm_build_tau(rcm_solver* s, double* tau_out, int* lowpos_p, int* lowpos_t);

/* K2-K4 for a GIVEN tau = radiative_transfer (main.cpp:320-344).  tau [ncol][nwvl][20] host,
 * NULL = use the tau of the last rcm_build_tau.  Outputs E_down/E_up [ncol][21], dE [ncol][20]. */
int rcm_radiative_transfer(rcm_solver* s, const double* tau, double* E_down, double* E_up, double* dE);

/* The fused time step (K1-K5), nsteps iterations of main.cpp:531-583 for every column, state
 * resident on the GPU.  scalars_out [nsteps] host (NULL = skip).  Asynchronous pieces are
 * synchronised before return when scalars_out != NULL. */
int rcm_advance(rcm_solver* s, int nsteps, rcm_step_scalars* scalars_out);
/* Same, but leaves the per-step scalars on the device for an allreduce:
 * *d_scalars -> device double[nsteps][4] (layout of rcm_step_scalars), valid until the next call. */
int rcm_advance_async(rcm_solver* s, int nsteps, double** d_scalars);

/* The RCE driver loop: iterate main.cpp:531-583 until the ensemble is stationary.  Advances in blocks of
 * `check_every` fused steps (one launch each) and stops after the first block whose last step moved every
 * column's sorted temperature profile by less than params.dT_converged (n_converged == ncol), or after
 * max_steps.  *last = scalars of the last step done, *steps_done = iterations run by this call (either may be
 * NULL).  One GPU; for N ranks use the same loop with an allreduce of the scalars between the blocks
 * (our_first_climate_model_b200/distributed.py: run_to_equilibrium). */
int rcm_run_to_equilibrium(rcm_solver* s, long max_steps, int check_every, rcm_step_scalars* last, long* steps_done);

/* Download state / last-step fluxes; any pointer may be NULL.  Tlayer [ncol][20], Tsurf [ncol],
 * h2o [ncol][20], time_h [ncol] (float hours, main.cpp:581), E_down/E_up [ncol][21],
 * dE [ncol][20], dt [ncol]. */
int rcm_get_state(rcm_solver* s, double* Tlayer, double* Tsurf, double* h2o, float* time_h, double* E_down,
                  double* E_up, double* dE, double* dt);

/* One call = one reference loop iteration with HOST buffers in and out (what bench.py's e2e
 * leg times): rcm_update_columns + 1 fused step + download of E_down, E_up, dE, Tlayer, Tsurf. */
/* Checkpoint / restart (SURVEY 8(f)4): everything the step reads or carries (T, Tsurf, active VMRs, rel_hum, the
 * previous sorted profile, model time, last dt / fluxes / dE, per-column forcing, step index, pressure grid) in one
 * flat little-endian file.  A solver with the same table and species_mask that loads it continues bit-identically.
 * Tables are not stored.  Errors: RCM_ERR_IO, RCM_ERR_FORMAT (not a checkpoint / truncated), RCM_ERR_STATE (other
 * species_mask or spectral path). */
int rcm_save_checkpoint(rcm_solver* s, const char* path);
int rcm_load_checkpoint(rcm_solver* s, const char* path);
int rcm_column_count(const rcm_solver* s); /* columns currently loaded (rcm_set_columns / rcm_load_checkpoint) */
/* Diagnostic radiation call: the thermal fluxes the NEXT step of the resident ensemble would compute - after its theta-sort
 * and water-vapour feedback, with its grey cloud and solar forcing (main.cpp:536-574) - for the columns [col0, col0 + ncol),
 * per wavelength, optionally with the active species' VMRs scaled.  Changes nothing: state, step counter, scalars and every
 * later step stay bit-identical.  With step_index 0 tau comes from the initial, unsorted profile as in the first step.
 * vmr_scale [nactive] (ascending species index, as vmr_active; NULL = all 1): factor on each active species' layer VMRs as
 * that step would use them (H2O: after the feedback), one rounded multiplication.
 * Outputs (host, any may be NULL): E_down_spec / E_up_spec [ncol][nwvl][21], the contribution of each wavelength (its
 * spectral weight included); E_down / E_up [ncol][21] = those summed over the wavelengths in index order; dE [ncol][20] from
 * them as main.cpp:337-341 (the column's own solar_irr in the lowest layer).  Synchronous.  Works through the range in
 * chunks of at most 8,192 columns with device scratch of its own (about 0.6 GB for 100 wavelengths).
 * Errors: RCM_ERR_ARG for a range outside the loaded columns or a scale that is negative or not finite; RCM_ERR_STATE without
 * table or columns, on the line-by-line path, with another species_mask than the default's five species, or with
 * RCM_OPT_PATH 1. */
int rcm_diagnose_fluxes(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* E_down_spec, double* E_up_spec,
                        double* E_down, double* E_up, double* dE);
/* Radiative kernels (Soden et al. 2008) of the columns [col0, col0 + ncol): analytic derivatives of two fluxes of the NEXT
 * step - output o = 0: E_up[0], the OLR; o = 1: E_down[20], the surface downward flux - at exactly the state
 * rcm_diagnose_fluxes radiates with (after the theta-sort and the water-vapour feedback, with the grey cloud, per-column cloud
 * tau of rcm_set_column_solar included; at step 0 with tau from the initial, unsorted profile), vmr_scale as there.
 * Entries of each output [41]: 0..19 dF/dT_l (W m-2 K-1, layers top-down); 20 dF/dT_surf (exactly 0.0 for o = 1: the surface
 * is black); 21..40 dF/d ln q_l (W m-2 per unit ln q), q_l = H2O VMR of layer l as the step uses it.
 * Definitions: d/dT_l perturbs layer l's temperature in both places it enters - its Planck source and the temperature its tau
 * is interpolated at (the same value except at step 0); d/d ln q_l is taken at fixed T.  Where a clamp is active the derivative
 * is 0: tau at its floor or ceiling, a temperature at or below T_floor in the Planck source.  Exactly on a table temperature
 * node the slope is that of the interval LowerPos picks.
 * Outputs (host, either may be NULL): K_spec [ncol][nwvl][2][41], the contribution of each wavelength (its spectral weight
 * included); K [ncol][2][41] = K_spec summed over the wavelengths in index order.  Synchronous; changes nothing.  Device scratch
 * of its own (about 1.1 GB for 100 wavelengths).  Errors as rcm_diagnose_fluxes; also RCM_ERR_STATE when H2O is not active. */
int rcm_radiative_kernels(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* K_spec, double* K);
/* Flux Jacobians of the columns [col0, col0 + ncol): analytic derivatives of every level's broadband E_down and E_up of the
 * NEXT step (summed over the wavelengths in index order) and of its heating rates, at exactly the state rcm_radiative_kernels
 * differentiates (sort, water-vapour feedback, grey cloud, step-0 rule, vmr_scale), with respect to the same 41 entries
 * x_e and with the same definitions: 0..19 T_l (layers top-down), 20 T_surf, 21..40 ln q_l.
 * Outputs (host, either may be NULL): J [ncol][2][21][41], J[c][0][k][e] = dE_down[k]/dx_e and J[c][1][k][e] = dE_up[k]/dx_e
 * (W m-2 per K resp. per unit ln q); dE_jac [ncol][20][41], d dE_l/dx_e computed from J entry by entry as dE from E
 * (main.cpp:337-341): H[l] = Jd[l] - Jd[l+1] + Ju[l+1] - Ju[l], then H[19] += Jd[20] - Ju[20] (the solar term is constant).
 * Exactly 0.0 by construction: row E_down[0]; dE_down[k]/d(T_l, ln q_l) for l >= k; dE_down[k]/dT_surf; dE_up[k]/d(T_l,
 * ln q_l) for l < k (so row E_up[20] has only its T_surf entry).  Synchronous; changes nothing.  Device scratch of its own
 * (about 0.4 GB, independent of the wavelengths).  Errors as rcm_radiative_kernels. */
int rcm_flux_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac);
/* Stratosphere-adjusted forcing of the columns [col0, col0 + ncol) by fixed dynamical heating (SARF: Manabe & Wetherald;
 * Hansen et al. 1997), next to the instantaneous forcing (IRF).
 * Base state: the state rcm_diagnose_fluxes(..., NULL, ...) radiates (after the theta-sort and the water-vapour feedback,
 * with the grey or per-column cloud and the step-0 rule).  Perturbed state: the same with vmr_scale applied exactly as the
 * other calls apply it (NULL = all 1).
 * Stratosphere: ntrop[c] in [0, 19] (required, never NULL) is the number of stratospheric layers of column c, layers
 * 0 .. ntrop - 1 top-down; the tropopause is level ntrop[c].
 * Adjustment dT: dT_l for l < ntrop is added to layer l's temperature in both places it enters, its Planck source and the
 * temperature its tau is interpolated at (the d/dT_l of rcm_radiative_kernels and rcm_flux_jacobian; at step 0 it moves
 * both the sorted and the unsorted profile).  Troposphere, surface and all VMRs stay fixed; no re-sort, no feedback.
 * Solved for: dE_l(perturbed, T + dT) = dE_l(base, T) for every l < ntrop, by Newton on the ntrop x ntrop block of dE_jac
 * (entries 0 .. ntrop - 1 of rows 0 .. ntrop - 1), re-evaluated at every iterate; FP64 Gaussian elimination with partial
 * pivoting (lowest row on ties).
 * Convergence: a column has converged when max_{l < ntrop} |dE_l - dE_l^base| <= tol (W m-2).  From then on it is frozen:
 * its outputs are those of the evaluation that met the test, and later iterations do not touch it.
 * iters[c]: the number of Newton updates applied; -1 when max_iter updates did not converge, when the linear solve met a
 * zero or non-finite pivot, or when the residual is not finite - the outputs then hold the last evaluated iterate and the
 * call still returns RCM_OK.
 * Outputs (host, any may be NULL), with N_k = E_down[k] - E_up[k] computed as (Ed'[k] - Eu'[k]) - (Ed[k] - Eu[k]):
 * F [ncol][4]: 0 IRF at TOA, 1 IRF at the tropopause level, 2 SARF at TOA, 3 SARF at the tropopause level (W m-2);
 * dT_adj [ncol][20] (K, exactly 0.0 for l >= ntrop); E_down, E_up [ncol][21] broadband fluxes at the adjusted perturbed
 * state; iters [ncol].  Every value is a function of its column alone: ranges, shards and chunks give bit-identical results.
 * Synchronous; changes nothing.  Device scratch of its own: 7,113 doubles and 2 ints per column of a chunk (8,192 at most)
 * plus the tile blocks, twice - 957,219,328 bytes for 8,192 columns and 100 wavelengths (42 x nwvl + 2,913 doubles per
 * column in general).  Errors as rcm_flux_jacobian; also RCM_ERR_ARG when ntrop is NULL or an entry lies outside [0, 19],
 * tol is not finite or not > 0, or max_iter < 1. */
int rcm_adjusted_forcing(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, double tol,
                         int max_iter, double* F, double* dT_adj, double* E_down, double* E_up, int* iters);
/* Diagnostic radiation call of the line-by-line path: the thermal fluxes the NEXT LBL step would compute for the columns
 * [col0, col0 + ncol) - after its theta-sort and water-vapour feedback (none at step 0), with the grey cloud or the per-column
 * cloud tau and solar_irr of rcm_set_column_solar - optionally with scaled species and resolved into bands of wavelengths.
 * Changes nothing: T, Tprev, VMRs, model time, dt, fluxes, step counter, checkpoint bytes and every later step stay as they are.
 * vmr_scale [5] (NULL = all 1): one factor per species in ASCENDING SPECIES INDEX - H2O, CO2, O3, N2O, CH4 (not the table order
 * of rcm_set_lbl_tables).  The perturbed optical depth, defined so that all factors 1 give the step's tau bit for bit:
 *   s_H2O = (f_H2O x h2o) / h2o_ref with h2o the VMR after the feedback, one rounded multiplication before the division;
 *   s_O3  = (f_O3 x o3) / o3_ref, or f_O3 without o3_ref;
 *   column-independent plane = ((f_CO2 x co2_factor) x tau_CO2 + f_CH4 x tau_CH4) + f_N2O x tau_N2O, left to right, each
 *   operation rounded (composed only when one of these three factors is not 1; the tables' own plane otherwise).
 * Broadband outputs (host, any may be NULL): E_down / E_up [ncol][21], dE [ncol][20] (main.cpp:337-341, the column's own
 * solar_irr in dE[19]).  They come from the step's own kernels on copies of the state: unscaled they equal what the next
 * rcm_advance(1) computes, bit for bit.
 * Band outputs (host, either may be NULL): E_down_band / E_up_band [ncol][nband][21]; band b is the sum of each wavelength's own
 * flux over [band_start[b], band_start[b + 1]) in index order, from 0.0 (a band of one wavelength is that wavelength alone).
 * band_start [nband + 1] must satisfy 0 = b_0 < b_1 < ... < b_nband = nwvl; it is read only when a band output is wanted.
 * Every value is a function of its column alone: ranges, chunks and shards give bit-identical rows.  The band pass runs only
 * for band outputs, the broadband pass only for broadband outputs.  Synchronous.
 * Device scratch of its own: two sets for chunks of ch columns (whole tiles of 16, at most 8,192; with band outputs also at most
 * 2e9 / (nwvl x 42 x 8) rounded down to whole tiles, at least 16), each of 8 ch (141 + 42 nchunks_b + 42 nwvl_b + 42 nband_b)
 * + 4 ch + 4 (nband + 1)_b bytes, nchunks = ceil(nwvl / 128), the _b terms only for broadband (nchunks) or band outputs;
 * with CO2, CH4 or N2O scaled also 3 x nwvl x 20 doubles.
 * Errors: RCM_ERR_STATE not on the line-by-line path, without columns, or with another species_mask than the default's five
 * species; RCM_ERR_ARG for a range outside the loaded columns, a factor that is negative or not finite, and with a band output
 * for nband < 1, a NULL band_start or one that does not rise strictly from 0 to nwvl.  Each error leaves the solver usable. */
int rcm_lbl_diagnose_fluxes(rcm_solver* s, int col0, int ncol, const double* vmr_scale, int nband, const int* band_start,
                            double* E_down_band, double* E_up_band, double* E_down, double* E_up, double* dE);
/* Radiative kernels of the line-by-line path: analytic derivatives of the OLR (output 0, E_up[0]) and the surface downward
 * flux (output 1, E_down[20]) of the NEXT LBL step for the columns [col0, col0 + ncol), at exactly the state
 * rcm_lbl_diagnose_fluxes radiates for the same arguments (theta-sorted profile, H2O after the feedback - none at step 0 -,
 * grey or per-column cloud, vmr_scale applied as there).  Entries and outputs as rcm_radiative_kernels, 41 per output:
 * 0..19 dF/dT_l (layers top-down), 20 dF/dT_surf, 21..40 dF/dln q_l (q_l the layer's H2O VMR as the step uses it).
 * LBL tau does not depend on T, so:
 *   d/dT_l moves layer l's Planck source only (fixed q, no re-sort, no feedback); d/dT_surf the surface source (exactly 0.0
 *   for output 1); d/dln q_l = dF/dtau_l x (tau_H2O,l x s_H2O,l) at fixed T, 0 where the tau clamp acts (tau_clamp, on angle
 *   schedules that clamp tau in front of the exp).
 *   dB/dT of the band Planck source, K = sigma/pi x 15/pi^4, f(x) = x^3 / (e^x - 1): on the Simpson branch K T^3 S_n[g],
 *   g(x) = x^4 e^x / (e^x - 1)^2, Simpson's rule on the abscissae, exponentials and order n of B itself (the exact derivative
 *   of the Simpson value); on every other branch 4 B / T - K T^3 (v1 f(v1) - v0 f(v0)) (an overflowing exp: a term of 0);
 *   0 for T < 1e-4.
 * Outputs (host, either may be NULL; both NULL: RCM_OK without work): K [ncol][2][41] the sum over all wavelengths in index
 * order from 0.0; K_band [ncol][nband][2][41], band b the sum over [band_start[b], band_start[b + 1]) in index order from 0.0
 * (K equals K_band of the one band {0, nwvl} bit for bit; a band of one wavelength is that wavelength's contribution).
 * band_start as rcm_lbl_diagnose_fluxes, read only for K_band.  Every value is a function of its column alone: ranges,
 * chunks and shards give bit-identical rows.  Synchronous; changes nothing.
 * Device scratch of its own: two sets for chunks of ch columns (whole tiles of 16, at most 8,192 and at most
 * 2e9 / (nwvl x 82 x 8) rounded down to whole tiles, at least 16), each of 8 ch (182 + 82 nwvl + 82_K + 82 nband_b) + 4 (2 +
 * (nband + 1)_b) bytes rounded up to 256, the _K term only for K, the _b terms only for K_band; with CO2, CH4 or N2O scaled
 * also the 3 x nwvl x 20 doubles of rcm_lbl_diagnose_fluxes.  About 3.8 GB at 20,000 wavelengths.
 * Errors as rcm_lbl_diagnose_fluxes (the band checks for K_band); each leaves the solver usable. */
int rcm_lbl_radiative_kernels(rcm_solver* s, int col0, int ncol, const double* vmr_scale, int nband, const int* band_start,
                              double* K_band, double* K);
/* Flux Jacobians of the line-by-line path: analytic derivatives of every level's broadband E_down and E_up of the NEXT LBL step
 * (summed over the wavelengths in index order) and of its heating rates, for the columns [col0, col0 + ncol), at exactly the
 * state rcm_lbl_radiative_kernels differentiates for the same arguments, with its definitions (d/dT_l through layer l's Planck
 * source alone, d/dln q_l = dF/dtau_l x tau_H2O,l x s_H2O,l, 0 where the tau clamp acts).  Outputs, entries and structural
 * zeros as rcm_flux_jacobian: J [ncol][2][21][41], dE_jac [ncol][20][41] from J as dE from E (main.cpp:337-341).  Rows
 * E_up[0] and E_down[20] of J are rcm_lbl_radiative_kernels' K to rounding (the same terms, summed per level instead of per
 * wavelength).  Both outputs NULL: RCM_OK without work.  Every value is a function of its column alone: ranges, chunks and
 * shards give bit-identical rows.  Synchronous; changes nothing.  Device scratch of its own: two sets for chunks of at most
 * 8,192 columns, each of 2,724 doubles per column (about 0.36 GB, independent of the wavelengths); with CO2, CH4 or N2O
 * scaled also the 3 x nwvl x 20 doubles of rcm_lbl_diagnose_fluxes.  Errors as rcm_lbl_diagnose_fluxes. */
int rcm_lbl_flux_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac);
/* Stratosphere-adjusted forcing of the line-by-line path, as rcm_adjusted_forcing (ntrop, tol, max_iter, convergence, freezing,
 * iters, the outputs F, dT_adj, E_down, E_up and the argument errors) with these substitutions:
 * Base state: what rcm_lbl_diagnose_fluxes(..., NULL, ...) radiates; its E_down, E_up and dE equal the next rcm_advance(1) bit
 * for bit.  Perturbed state: the same with vmr_scale applied exactly as rcm_lbl_diagnose_fluxes applies it, so that the IRF of
 * iterate 0 is rcm_lbl_diagnose_fluxes(vmr_scale) minus the unscaled call, bit for bit.
 * Adjustment: dT_l (l < ntrop) moves layer l's Planck source only (LBL tau does not depend on T; no step-0 rule).
 * Solve: Newton on the ntrop x ntrop block of rcm_lbl_flux_jacobian's dE_jac, re-evaluated at every iterate.
 * Synchronous; changes nothing.  Device scratch of its own: two sets for chunks of at most 8,192 columns, each of
 * 2,956 + 42 ceil(nwvl / 128) doubles and 12 bytes per column (about 1.25 GB at 20,000 wavelengths); with CO2, CH4 or N2O
 * scaled also the 3 x nwvl x 20 doubles of rcm_lbl_diagnose_fluxes.  Errors as rcm_lbl_flux_jacobian, then those of
 * rcm_adjusted_forcing's arguments. */
int rcm_lbl_adjusted_forcing(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, double tol,
                             int max_iter, double* F, double* dT_adj, double* E_down, double* E_up, int* iters);
/* Equilibrium climate response of the columns [col0, col0 + ncol) to a VMR perturbation: the surface warming at fixed lapse
 * rate and, with fixed_rh, fixed relative humidity (Manabe & Wetherald 1967), solved directly by Newton.
 * Base and perturbed states: exactly those of rcm_adjusted_forcing for the same vmr_scale; iterate 0 is rcm_diagnose_fluxes
 * (NULL, resp. vmr_scale) bit for bit.
 * Unknowns: ntrop[c] in [0, 19] (required, never NULL) as there.  Each stratospheric layer l < ntrop has its own dT_l.  The
 * troposphere and the surface share one, dTs, a uniform potential-temperature increment: layer l >= ntrop moves by
 * dT_l = dTs / conv_l, conv_l = (1000 / p_l)^(2/7), and the surface temperature by dTs.  (The model's convective adjustment is
 * the theta-sort and its surface temperature T_19 conv_19: a uniform increment keeps a sorted profile sorted.)
 * Where a temperature change enters: as rcm_adjusted_forcing for the layers (Planck source and the temperature tau is
 * interpolated at; at step 0 both the sorted and the unsorted profile), and the surface's Planck source.
 * Water vapour: with fixed_rh != 0 every layer's H2O is re-evaluated at T + dT by the step's feedback, rel_hum x
 * 6.1094 exp(17.625 Tc / (Tc + 243.04)) / p_l, then multiplied by the H2O factor of vmr_scale as rcm_diagnose_fluxes does
 * (at dT = 0 bit-identical to the step's); fixed_rh needs step_index > 0, since the step applies no feedback at step 0.  With
 * fixed_rh == 0 every VMR stays fixed (fixed absolute humidity), and step 0 is allowed.
 * Solved for, m = ntrop + 1 equations: dE_l(perturbed, x) = dE_l(base) for l < ntrop (fixed dynamical heating), and
 * N_k(perturbed, x) = N_k(base) at the tropopause level k = ntrop, N = E_down - E_up formed as (Ed'[k] - Eu'[k]) -
 * (Ed[k] - Eu[k]); together the TOA net flux is unchanged (with ntrop = 0 this is the TOA balance itself).
 * Newton matrix, re-evaluated at every iterate from rcm_flux_jacobian at that iterate: with D_i the 41 entries of row i of
 * dE_jac (i < ntrop) resp. J_down[ntrop] - J_up[ntrop] (i = ntrop), and gamma_l = 17.625 x 243.04 / (T_l - 273.15 + 243.04)^2
 * at T_l = T_B,l + dT_l (0 with fixed_rh == 0): A[i][j] = D_i[j] + gamma_j D_i[21 + j] for j < ntrop, and A[i][ntrop] =
 * D_i[20] + sum_{l = ntrop}^{19} (D_i[l] + gamma_l D_i[21 + l]) / conv_l in index order.  FP64 Gaussian elimination with
 * partial pivoting (lowest row on ties, NaN refused) as rcm_adjusted_forcing.
 * Convergence and iters as rcm_adjusted_forcing, over all m residuals: max |residual| <= tol (W m-2); -1 for no convergence,
 * a zero or non-finite pivot or a non-finite residual (a column with a runaway greenhouse lands there), RCM_OK all the same.
 * Outputs (host, any may be NULL): F [ncol][2] the IRF at TOA and at the tropopause level (iterate 0; bit for bit
 * rcm_adjusted_forcing's F[c][0..1]); dT [ncol][20] the response profile (K); dTs [ncol] the surface warming (K; for doubled
 * CO2 the model's equilibrium climate sensitivity); E_down, E_up [ncol][21] the fluxes at the solution; iters [ncol].
 * Every value is a function of its column alone: ranges, chunks and shards give bit-identical rows.  Synchronous; changes
 * nothing.  Device scratch of its own: that of rcm_adjusted_forcing, 2,913 + 42 nwvl doubles and 2 ints per column of a chunk
 * (8,192 at most) plus the tile blocks, twice.  Errors as rcm_adjusted_forcing; also RCM_ERR_STATE for fixed_rh at step 0 or
 * without H2O among the active species.  Each error leaves the solver usable. */
int rcm_climate_response(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, int fixed_rh, double tol,
                         int max_iter, double* F, double* dT, double* dTs, double* E_down, double* E_up, int* iters);
/* Equilibrium climate response of the line-by-line path, as rcm_climate_response with rcm_lbl_adjusted_forcing's states: dT and
 * dTs move the Planck sources only (LBL tau does not depend on T; no step-0 rule), with fixed_rh also s_H2O = (f_H2O x h2o) /
 * h2o_ref at T + dT, and the Newton matrix comes from rcm_lbl_flux_jacobian.  Device scratch of its own: that of
 * rcm_lbl_adjusted_forcing, 2,956 + 42 ceil(nwvl / 128) doubles and 12 bytes per column of a chunk, twice.  Errors as
 * rcm_lbl_adjusted_forcing, then those of fixed_rh. */
int rcm_lbl_climate_response(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, int fixed_rh,
                             double tol, int max_iter, double* F, double* dT, double* dTs, double* E_down, double* E_up,
                             int* iters);
/* Species Jacobians of the columns [col0, col0 + ncol): analytic derivatives of every level's broadband E_down and E_up of the
 * NEXT step (summed over the wavelengths in index order) and of its heating rates with respect to the ln VMR of each of the five
 * species in each layer, at exactly the state rcm_flux_jacobian differentiates for the same arguments (sort, water-vapour
 * feedback, grey or per-column cloud, step-0 rule, vmr_scale applied as there).
 * Entries [100]: e = 20 s + l, s in ascending species index as vmr_scale (0 H2O, 1 CO2, 2 O3, 3 N2O, 4 CH4), layers l top-down;
 * entry e is d/d ln x_{s,l}, x_{s,l} the VMR of species s in layer l as the step uses it (W m-2 per unit ln x), at fixed T:
 * no re-sort, no feedback.  dtau_l/dln x_{s,l} is species s's own term of the step's optical depth, numDens_l x (its three-FMA
 * K1 term at layer l) x x_{s,l}; the entry is 0.0 where the tau clamp or floor acts and where x_{s,l} = 0.
 * Outputs (host, either may be NULL; both NULL: RCM_OK without work): J [ncol][2][21][100], J[c][0][k][e] = dE_down[k]/dx_e
 * and J[c][1][k][e] = dE_up[k]/dx_e; dE_jac [ncol][20][100] from J entry by entry as dE from E (main.cpp:337-341).  Structural
 * zeros those of the ln q entries of rcm_flux_jacobian: dE_down[k]/dx_{s,l} for l >= k, dE_up[k]/dx_{s,l} for l < k.  The
 * H2O block (e = 0..19) equals rcm_flux_jacobian's entries 21..40 bit for bit.  Linearised, the change of the fluxes for a
 * profile perturbation of any species is sum_e J[.][e] dln x_e.  Every value is a function of its column alone: ranges, chunks
 * and shards give bit-identical rows.  Synchronous; changes nothing.  Device scratch of its own: two sets for chunks of at
 * most 8,192 columns, each of 6,341 doubles per column plus the tile blocks (about 0.9 GB).  Errors as rcm_flux_jacobian;
 * also RCM_ERR_STATE with any species_mask other than the default 0x2F.  Each leaves the solver usable. */
int rcm_species_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac);
/* Species Jacobians of the line-by-line path: rcm_species_jacobian's entries, outputs, structural zeros and properties at the
 * state rcm_lbl_flux_jacobian differentiates for the same arguments.  dtau_l/dln x_{s,l} is species s's share of tau_l as
 * rcm_lbl_diagnose_fluxes composes it, one rounded product each: tau_H2O,l x s_H2O,l; (f_CO2 x co2_factor) x tau_CO2,l;
 * tau_O3,l x s_O3,l; f_N2O x tau_N2O,l; f_CH4 x tau_CH4,l; 0.0 where the tau clamp acts.  The H2O block equals
 * rcm_lbl_flux_jacobian's entries 21..40 bit for bit.  Device scratch of its own: two sets for chunks of at most 8,192
 * columns, each of 6,382 doubles per column (about 0.84 GB, independent of the wavelengths); with CO2, CH4 or N2O scaled also
 * the 3 x nwvl x 20 doubles of rcm_lbl_diagnose_fluxes.  Errors as rcm_lbl_flux_jacobian; also RCM_ERR_STATE with any
 * species_mask other than the default 0x2F.  Each leaves the solver usable. */
int rcm_lbl_species_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac);
/* Adjoint flux gradients of the columns [col0, col0 + ncol): the derivatives of one weighted sum of each column's broadband
 * fluxes and heating rates of the NEXT step, by one reverse sweep of the radiative transfer instead of full Jacobians.
 * Row r is column c = col0 + r.  Cotangents (host, each may be NULL = zero): w_E_down, w_E_up [ncol][21], w_dE [ncol][20];
 * the objective of column c is
 *   Phi_c = sum_k w_E_down[r][k] E_down[k] + sum_k w_E_up[r][k] E_up[k] + sum_l w_dE[r][l] dE[l],
 * with E and dE the fluxes and heating rates rcm_diagnose_fluxes returns for the same vmr_scale (dE from E as main.cpp:337-341;
 * its solar term is constant).
 * Output (host): grad [ncol][121], grad[r][e] = dPhi_c/dx_e over the entries e = 0..19 T_l (layers top-down), e = 20 T_surf,
 * e = 21 + 20 s + l ln x_{s,l}, s in the order of vmr_scale (0 H2O, 1 CO2, 2 O3, 3 N2O, 4 CH4).  Entries 0..40 are those of
 * rcm_flux_jacobian, entries 21..120 those of rcm_species_jacobian offset by 21, with every definition of those calls: the
 * state they differentiate (sort, water-vapour feedback, grey or per-column cloud, vmr_scale), the step-0 rule for d/dT_l,
 * fixed T for ln x (no re-sort, no feedback), 0 where the tau clamp or floor acts, where T <= T_floor in the Planck source and
 * where a species' VMR is 0.  grad is their contraction with the cotangents, to rounding: sum_k w_E_down[k] J[0][k] +
 * w_E_up[k] J[1][k] + sum_l w_dE[l] dE_jac[l].
 * The cotangents are folded on the host into level cotangents, b_k on E_down[k] and a_k on E_up[k]: b_k = (w_E_down[k] +
 * w_dE[k]) - w_dE[k-1], a_k = (w_E_up[k] - w_dE[k]) + w_dE[k-1], each term where it exists.  The sum over the wavelengths is
 * taken in partials of 5 rounds of 4 wavelengths (wavelengths g, g + 4, ... per group g, the groups in order), then the
 * partials in order: fixed by the table and the angle schedule.  Every value is a function of its column alone: ranges,
 * chunks and shards give bit-identical rows.
 * grad NULL: RCM_OK without work.  All three cotangents NULL: grad filled with 0.0, no launch.  Synchronous; changes nothing.
 * Device scratch of its own: two sets for chunks of at most 8,192 columns, each of 183 + 121 (1 + nsplit) doubles per column,
 * nsplit = ceil(ceil(nwvl / 4) / 5), plus the tile blocks (about 0.15 GB for 100 wavelengths).
 * Errors as rcm_species_jacobian; also RCM_ERR_ARG for a cotangent entry that is not finite (checked on the host before any
 * work).  Each error leaves the solver usable. */
int rcm_flux_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const double* w_E_down, const double* w_E_up,
                      const double* w_dE, double* grad);
/* Adjoint flux gradients of the line-by-line path: rcm_flux_gradient's cotangents, objective, entries, fold and properties at
 * the state rcm_lbl_diagnose_fluxes radiates for the same vmr_scale, with the definitions of rcm_lbl_flux_jacobian (d/dT_l
 * through layer l's Planck source alone, cplkavg_narrow's dB/dT) and rcm_lbl_species_jacobian (each species' share of tau as
 * the rounded product rcm_lbl_diagnose_fluxes composes).  The sum over the wavelengths is taken in partials of 1,024
 * wavelengths (wavelengths g, g + 4, ... of a partial per group g, the groups in order), then the partials in order: fixed by
 * the table.  Device scratch of its own: two sets for chunks of at most 8,192 columns, each of 224 + 121 (1 + ceil(nwvl /
 * 1,024)) doubles per column (about 0.36 GB at 20,000 wavelengths); with CO2, CH4 or N2O scaled also the 3 x nwvl x 20 doubles
 * of rcm_lbl_diagnose_fluxes.  Errors as rcm_lbl_species_jacobian; also RCM_ERR_ARG for a cotangent entry that is not
 * finite.  Each error leaves the solver usable. */
int rcm_lbl_flux_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const double* w_E_down,
                          const double* w_E_up, const double* w_dE, double* grad);
/* Climate-response gradients of the columns [col0, col0 + ncol): the derivatives of the equilibrium surface warming dTs in
 * every species' VMR in every layer of the perturbed state and in an imposed forcing term of every equation, by one adjoint
 * solve of the converged Newton system and one reverse sweep of the radiative transfer.
 * The call runs at exactly the solution rcm_climate_response finds for the same vmr_scale, ntrop, fixed_rh, tol and max_iter
 * (same iterates, same bits).  Write that solution as y = (dT_0 .. dT_{ntrop-1}, dTs), m = ntrop + 1, and the residual as
 * R(y, p) with the equations and order of rcm_climate_response (i < ntrop: the heating rate of layer i; i = ntrop: the net flux
 * at level ntrop).  The derivatives are taken in
 *   p = ln x_{s,l}: a multiplicative perturbation of species s in layer l of the PERTURBED state only (the base state is
 *     fixed); entry e = 20 s + l, s in the order of vmr_scale (0 H2O, 1 CO2, 2 O3, 3 N2O, 4 CH4), layers l top-down; with the
 *     definitions of rcm_species_jacobian at the solution state (the tile block's rows at T_B + dT).  With fixed_rh != 0,
 *     ln x_{H2O,l} is a factor on the feedback's H2O of layer l, i.e. a relative-humidity change;
 *   q_i: an imposed forcing term added to equation i: for i < ntrop an extra heating of stratospheric layer i (W m-2, the
 *     units of dE), for i = ntrop an extra net downward flux at the tropopause level.
 * With A the m x m Newton matrix of rcm_climate_response assembled from the flux Jacobian AT THE SOLUTION (same D_i, gamma_l,
 * conv_l and index order), s = -A^{-T} e_m, solved by the same elimination (partial pivoting, lowest row on ties, NaN refused):
 *   dTs_dF [ncol][21]: dTs/dq_i = s_i for i < ntrop, entry 20 = s_m (K per W m-2: the column's local climate sensitivity
 *     parameter at the tropopause), exactly 0.0 in entries ntrop..19;
 *   dTs_dlnx [ncol][100]: dTs/dp_e = s^T dR/dp_e, the flux gradient (rcm_flux_gradient's entries 21..120 at the solution
 *     state) with the cotangents w_dE[i] = s_i (i < ntrop), w_E_down[ntrop] = s_m, w_E_up[ntrop] = -s_m, every other 0.0,
 *     folded with rcm_flux_gradient's expressions in its order;
 *   dTs [ncol], iters [ncol]: rcm_climate_response's bytes for the same arguments.
 * Any output may be NULL; all NULL: RCM_OK without work.  The rows of dTs_dF and dTs_dlnx are quiet NaN where iters == -1 or
 * where A at the solution has a zero or non-finite pivot (iters keeps the response's value).  Every value is a function of its
 * column alone: ranges, chunks and shards give bit-identical rows.  Synchronous; changes nothing.  Device scratch of its own:
 * that of rcm_climate_response plus 184 + 121 nsplit doubles per column of a chunk (nsplit as rcm_flux_gradient), twice.
 * Errors as rcm_climate_response; also RCM_ERR_STATE with any species_mask other than the default 0x2F.  Each error leaves the
 * solver usable. */
int rcm_climate_response_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, int fixed_rh,
                                  double tol, int max_iter, double* dTs, double* dTs_dF, double* dTs_dlnx, int* iters);
/* Climate-response gradients of the line-by-line path: rcm_climate_response_gradient at the solution of
 * rcm_lbl_climate_response, with A from rcm_lbl_flux_jacobian at the solution and the species entries of
 * rcm_lbl_species_jacobian there (the LBL copies' T_B + dT and s_H2O, each species' rounded share of tau).  Device scratch of its
 * own: that of rcm_lbl_climate_response plus 184 + 121 ceil(nwvl / 1,024) doubles per column of a chunk, twice.  Errors as
 * rcm_lbl_climate_response; also RCM_ERR_STATE with any species_mask other than the default 0x2F. */
int rcm_lbl_climate_response_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop,
                                      int fixed_rh, double tol, int max_iter, double* dTs, double* dTs_dF, double* dTs_dlnx,
                                      int* iters);
/* Batched form of output_conv (main.cpp:102-114): for every column the 20 rows "layer,player,Tlayer,theta,time"
 * ("%d,%f,%f,%f,%f\n", theta = Tlayer * (1000/player)^(2/7) as t_to_theta, main.cpp:123-127; time in hours).
 * column_ids != 0 prefixes every row with the column number ("%d,"); with ncol == 1 and column_ids == 0 the rows are
 * byte-identical to the reference's.  append != 0 appends like the reference's freopen(..., "a"); header != 0 writes
 * the reference's header line (main.cpp:528) first.  Host only. */
int rcm_write_profiles(const char* path, int append, int header, int ncol, const double* plevel_hPa,
                       const double* Tlayer, const float* time_h, int column_ids);
/* One iteration with HOST buffers (what a caller that keeps its state on the host does per step of main.cpp:531-583):
 * uploads Tlayer_in [ncol][20], Tsurf_in [ncol], vmr_active_in [ncol][nactive][20] - each only when not NULL (no VMR upload: the
 * rows of the previous call stay, H2O following the feedback on the device as in the reference loop), runs the step, downloads
 * E_down / E_up [ncol][21], dE / Tlayer_out [ncol][20], Tsurf_out [ncol] (each may be NULL = not wanted); synchronous.
 * On the split path the columns travel in chunks through upload / compute / download streams; with page-locked buffers the
 * pipeline of a steady-state call (second call on, same pointers, no VMR upload) is replayed as one CUDA graph - results are
 * bit-identical to rcm_advance(1) either way.  Environment: RCM_NO_GRAPH=1 keeps the direct calls, RCM_PIPE_CHUNKS=n sets the
 * chunk count.  Errors: RCM_ERR_ARG (no solver), RCM_ERR_STATE without columns / table, RCM_ERR_CUDA. */
int rcm_step_host(rcm_solver* s, const double* Tlayer_in, const double* Tsurf_in, const double* vmr_active_in,
                  double* E_down, double* E_up, double* dE, double* Tlayer_out, double* Tsurf_out);

/* Device-side band Planck (K2 of the LBL path), for parity against cplkavg(): n triples. */
int rcm_cplkavg_device(rcm_solver* s, int n, const double* lo_nm, const double* hi_nm, const double* t,
                       double* out);

/* Introspection for the bench: kernels launched so far, and FP64-pipe microbenchmarks
 * (result in 1e9 thread-instructions/s: which = 0 DFMA, 1 exp(), 2 divide, 3 solver exp). */
long rcm_launch_count(const rcm_solver* s);
/* rcm_step_host in steady state replays its chunk pipeline as one CUDA graph: how often it was captured / replayed. */
int rcm_host_graph_stats(const rcm_solver* s, long* captures, long* replays);
int rcm_fp64_microbench(rcm_solver* s, int which, double* ginstr_per_s);
/* Average device time (ms) of the fused step kernel over the launches since the last reset,
 * measured with CUDA events on the launching stream. */
int rcm_kernel_time_ms(rcm_solver* s, int reset, double* avg_ms, long* n_launches);

#ifdef __cplusplus
}
#endif
#endif /* RCM_B200_H */
