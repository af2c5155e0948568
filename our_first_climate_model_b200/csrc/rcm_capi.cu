// C ABI of the solver (include/rcm_b200.h): handle management, host-side precomputation of
// everything that depends only on the shared pressure grid / wavelength table, uploads,
// launches and downloads.  No CPU fallback: without a CUDA device rcm_create() fails.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <functional>
#include <limits>
#include <string>
#include <vector>

#include "rcm_jac.cuh"
#include "rcm_fdh.cuh"
#include "rcm_ecs.cuh"
#include "rcm_lbl_diag.cuh"
#include "rcm_lbl_jac.cuh"
#include "rcm_lbl_fjac.cuh"
#include "rcm_species.cuh"
#include "rcm_grad.cuh"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

struct rcm_solver {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    rcm_params p{};
    DevConst dc{};
    bool const_dirty = true;
    int opt_angle_cubes = 1;
    int opt_angle_pairs = 1;   // chain heads that share a virtual root take it from one exp (needs opt_angle_cubes)
    int opt_config = 0;        // 0: planned (plan_parts); k > 0: force kShapes[k-1] for the whole ensemble
        // prepare the next wavelength inside the angle loop (0: separate phase)
    int opt_stage_rows = 1;    // K1 reads its table rows from shared memory, staged one wavelength ahead
    int opt_path = 0;          // 0: split path (tile x wavelength-split units) when it applies; 1: fused tile kernel
    int opt_cplk_narrow = 0;   // rcm_cplkavg_device evaluates the LBL kernel's narrow-band variant (tests)
    double tau_clamp = 240.0;  // set by build_angles
    double T_floor = 0.0;      // set by rcm_set_spectral_grid: max over the grid of h*c/(lambda*kB) / 690
    int clampk = 1;
    // table
    bool has_table = false, has_spectral = false;
    std::vector<double> p_grid, t_ref, t_pert, wvl, weight;
    double* d_coef3 = nullptr;  // the split path's rows (rcm_coef3_kernel), rebuilt with d_coef
    double *d_xsec_file = nullptr, *d_coef = nullptr, *d_planck_c = nullptr, *d_planck_k = nullptr, *d_exp_tab = nullptr;
    int* d_species = nullptr;
    bool coef_dirty = true;
    // columns
    int ncol = 0, cap = 0, nactive = 0, h2o_slot = -1;
    int species[RCM_NSPECIES]{};
    bool has_plevel = false;
    double plevel[RCM_NLEVEL]{};
    double *d_T = nullptr, *d_Ts = nullptr, *d_vmr = nullptr, *d_rh = nullptr, *d_Tprev = nullptr;
    float* d_time = nullptr;
    double *d_Ed = nullptr, *d_Eu = nullptr, *d_dE = nullptr, *d_dt = nullptr;
    double *d_diag = nullptr, *d_scalars = nullptr, *d_tau = nullptr, *d_red = nullptr;
    int* d_lowpos = nullptr;
    unsigned* d_ticket = nullptr;  // [diag_steps] ticket counters of rcm_reduce_diag_kernel
    double *d_solar_col = nullptr, *d_cloud_col = nullptr;  // per-column solar forcing / cloud tau (rcm_set_column_solar)
    bool has_col_solar = false, has_col_cloud = false;
    size_t diag_steps = 0, tau_cap = 0;
    long step_index = 0;
    bool tau_valid = false;
    // line-by-line tables
    bool lbl_mode = false;
    int lbl_nwvl = 0;
    double lbl_co2_factor = 1.0;
    bool lbl_has_o3_ref = false;
    double *d_lbl_lo = nullptr, *d_lbl_hi = nullptr, *d_lbl_tau5 = nullptr, *d_lbl_h2o_ref = nullptr,
           *d_lbl_o3_ref = nullptr, *d_sH = nullptr, *d_sO = nullptr, *d_dTstat = nullptr, *d_part = nullptr;
    size_t part_cap = 0;
    // d_lbl_tau5 holds the step's three planes, then the raw CO2, CH4 and N2O planes (rcm_lbl_diagnose_fluxes scales them)
    double* d_lbl_tau3s = nullptr;  // [3][nwvl][20] the step's planes with scaled species (rcm_lbl_diagnose_fluxes)
    size_t tau3s_cap = 0;
    // split path (rcm_split_kernels.cuh)
    unsigned char* d_tile = nullptr;    // [tiles][TILE_BYTES]
    double* d_spart = nullptr;          // [tiles][nsplit][42][16]
    unsigned* d_counter = nullptr;      // [4] work counters: the solver's stream and the three pipeline streams
    unsigned* d_multi = nullptr;        // [2][tile_cap] per-tile counters / step flags of the multi-step unit kernel
    size_t multi_cap = 0;
    int opt_multi = 1;                  // option 6: blocks of steps as ONE launch of the multi-step unit kernel
    size_t tile_cap = 0, spart_cap = 0;
    bool tile_vmr_valid = false;        // the constant species' rows of the tile blocks are current
    std::vector<double> stage;  // host packing buffer
    std::string err;
    long launches = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_free, ev_used;
    cudaStream_t pipe_stream[3] = {nullptr, nullptr, nullptr};  // rcm_step_host's chunk pipeline
    cudaEvent_t pipe_done[3] = {nullptr, nullptr, nullptr}, pipe_start = nullptr;
    // ... of the split path: uploads + K5 prep (high priority), unit kernels alternating on two streams, K5 finish + downloads
    // (high priority); one event per chunk and stage
    // the steady-state call of that pipeline captured as ONE CUDA graph (about 200 runtime calls per step otherwise - with
    // eight ranks on one host the CPU side of the pipeline became its critical path); `sig` + host pointers identify what the
    // graph has baked in, anything else re-captures
    struct HostGraph {
        cudaGraphExec_t exec = nullptr;
        SplitArgs sig{};
        const void* host[7] = {};
        const void* dev[4] = {};
        double dT_converged = 0.0;
        int ncol = 0, nchunk = 0, nkernels = 0;
        long captures = 0, replays = 0;
        bool failed = false;
    } hg;
    cudaStream_t sp_up = nullptr, sp_rt[2] = {nullptr, nullptr}, sp_down = nullptr;
    cudaEvent_t sp_prep[24] = {}, sp_rtdone[24] = {}, sp_end = nullptr;
    double kt_ms = 0.0;
    long kt_n = 0;
    unsigned char* d_diagnose = nullptr;  // rcm_diagnose_fluxes: two sets of (copies of a chunk's state, its tile blocks, fluxes)
    size_t diagnose_bytes = 0;
    cudaStream_t dg_stream[2] = {nullptr, nullptr};  // ... the chunks alternate between two streams and the two sets
    cudaEvent_t dg_fork = nullptr, dg_join[2] = {nullptr, nullptr};
    int* h_fdh_count = nullptr;  // rcm_adjusted_forcing: the active count of each stream's chunk (pinned, read every iteration)
};

namespace {

int fail(rcm_solver* s, int code, const std::string& msg) {
    if (s) s->err = msg;
    return code;
}

int cuda_fail(rcm_solver* s, cudaError_t e, const char* what) {
    return fail(s, RCM_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define CU(call)                                          \
    do {                                                  \
        cudaError_t e__ = (call);                         \
        if (e__ != cudaSuccess) return cuda_fail(s, e__, #call); \
    } while (0)

template <class T>
cudaError_t dalloc(T*& p, size_t n) {
    if (p) cudaFree(p);
    p = nullptr;
    return cudaMalloc((void**)&p, n * sizeof(T));
}

void set_active_species(rcm_solver* s) {
    s->nactive = 0;
    s->h2o_slot = -1;
    for (int k = 0; k < RCM_NSPECIES; ++k)
        if (s->p.species_mask & (1u << k)) {
            if (k == 0) s->h2o_slot = s->nactive;
            s->species[s->nactive++] = k;
        }
}

// Angle schedule.  Quadrature nodes mu_i = dmu/2 + dmu*i (main.cpp:482) = (2i+1)/(2*nangle).  With
// n = 2i+1, 1/mu is proportional to 1/n, hence t(n/3) = t(n)^3: nodes are visited in chains
// n, n/3, n/9, ... so that only the chain heads need an exp.  Summation order over angles
// changes, values of mu do not.  Also fixes tau_clamp / clampk (see exp_scaled in rcm_kernels.cu).
void build_angles(rcm_solver* s) {
    DevConst& d = s->dc;
    const int na = s->p.nangle;
    const double dmu = 1.0 / (double)na;
    d.nangle = na;
    std::vector<std::vector<int>> chains;  // node indices, head first
    struct PairUnit { int type; double inv_mu_root; std::vector<int> a, b; };
    std::vector<PairUnit> pairs;
    if (s->opt_angle_cubes) {
        std::vector<char> used(na, 0);
        for (int i = na - 1; i >= 0; --i) {
            if (used[i]) continue;
            std::vector<int> ch;
            for (int n = 2 * i + 1;; n /= 3) {
                used[(n - 1) / 2] = 1;
                ch.push_back((n - 1) / 2);
                if (n % 3 != 0) break;
            }
            chains.push_back(ch);
        }
        if (s->opt_angle_pairs) {
            // Heads a > b with pa*a == pb*b, (pa,pb) in {(3,5),(5,7),(3,7)}: a maximum matching over these few
            // candidates by exhaustive search (30 angles: 6 candidate edges, 4 disjoint pairs).
            struct Edge { int ca, cb, type, R; };
            std::vector<Edge> edges;
            const int pa_[3] = {3, 5, 3}, pb_[3] = {5, 7, 7};
            for (size_t x = 0; x < chains.size(); ++x)
                for (size_t y = 0; y < chains.size(); ++y) {
                    const int a = 2 * chains[x][0] + 1, b = 2 * chains[y][0] + 1;
                    for (int t = 0; t < 3; ++t)
                        if (a > b && pa_[t] * a == pb_[t] * b) edges.push_back({(int)x, (int)y, t, pa_[t] * a});
                }
            std::vector<int> best, cur;
            std::vector<char> taken(chains.size(), 0);
            std::function<void(size_t)> rec = [&](size_t e) {
                if (cur.size() > best.size()) best = cur;
                if (e >= edges.size() || cur.size() + (edges.size() - e) <= best.size() || edges.size() > 24) return;
                if (!taken[edges[e].ca] && !taken[edges[e].cb]) {
                    taken[edges[e].ca] = taken[edges[e].cb] = 1;
                    cur.push_back((int)e);
                    rec(e + 1);
                    cur.pop_back();
                    taken[edges[e].ca] = taken[edges[e].cb] = 0;
                }
                rec(e + 1);
            };
            rec(0);
            if (best.size() > (size_t)MAX_PAIR) best.resize(MAX_PAIR);
            std::vector<char> gone(chains.size(), 0);
            for (int e : best) {
                const Edge& ed = edges[e];
                pairs.push_back({ed.type, 2.0 * na / (double)ed.R, chains[ed.ca], chains[ed.cb]});
                gone[ed.ca] = gone[ed.cb] = 1;
            }
            std::vector<std::vector<int>> rest;
            for (size_t x = 0; x < chains.size(); ++x)
                if (!gone[x]) rest.push_back(chains[x]);
            chains.swap(rest);
        }
    } else {
        for (int i = 0; i < na; ++i) chains.push_back({i});
    }
    if (chains.size() % 2) chains.push_back({-1});  // padding chain: exp(0) = 1 with zero quadrature weight
    d.nchain = (int)chains.size();
    double sum = 0.0, x_max = 0.0, x_min = 1e300;
    int slot = 0;
    for (int a = 0; a < MAX_ANGLE + 2; ++a) {
        d.chain_len[a] = 1;
        d.neg_inv_mu_l2e[a] = 0.0;
        d.cmu[a] = 0.0;
    }
    auto node_mu = [&](int i) { return dmu / 2.0 + dmu * (double)i; };  // main.cpp:482
    d.npair = (int)pairs.size();
    for (int p = 0; p <= MAX_PAIR; ++p) d.pair_nim[p] = 0.0;
    for (int p = 0; p < d.npair; ++p) {
        d.pair_type[p] = pairs[p].type;
        d.pair_lenA[p] = (int)pairs[p].a.size();
        d.pair_lenB[p] = (int)pairs[p].b.size();
        d.pair_nim[p] = -pairs[p].inv_mu_root * EXP_L2E;
        x_max = std::max(x_max, pairs[p].inv_mu_root);
        for (const std::vector<int>* ch : {&pairs[p].a, &pairs[p].b})
            for (int i : *ch) {
                const double mu = node_mu(i);
                d.cmu[slot] = 2 * M_PI * mu * dmu;
                sum += d.cmu[slot++];
                x_min = std::min(x_min, 1.0 / mu);
            }
    }
    for (int ic = 0; ic < d.nchain; ++ic) {
        d.chain_len[ic] = (int)chains[ic].size();
        for (size_t m = 0; m < chains[ic].size(); ++m, ++slot) {
            if (chains[ic][m] < 0) continue;
            const double mu = node_mu(chains[ic][m]);
            d.cmu[slot] = 2 * M_PI * mu * dmu;
            sum += d.cmu[slot];
            if (m == 0) {
                d.neg_inv_mu_l2e[ic] = (-1.0 / mu) * EXP_L2E;  // times EXP_TAB/ln2, see exp_scaled
                x_max = std::max(x_max, 1.0 / mu);
            }
            x_min = std::min(x_min, 1.0 / mu);
        }
    }
    d.pair_nim[d.npair] = d.neg_inv_mu_l2e[0];  // the last pair unit evaluates the first chain's head
    d.nslot = slot;
    d.csum = sum;
    {
        // h(f) with exp(f c) - 1 = f h(f), c = ln2/EXP_TAB, |f| <= 1/2.
        // 128 entries: Taylor to f^5 with the f^5 term economised (f^5 ~ 0.3125 f^3 - 0.01953125 f on [-1/2, 1/2],
        // Chebyshev), degree 3 in h, max relative error 7.6e-17.
        // 1024 entries: Taylor to f^4 with the f^4 term economised (f^3 ~ 0.1875 f in h), degree 2 in h, 1.4e-16.
        const double ec7[4] = {0x1.62e42fefa3685p-8, 0x1.ebfbdff82c58fp-17, 0x1.c6b09b1799fcbp-26, 0x1.3b2ab6fba4e77p-35};
        const double ec10[4] = {0x1.62e42fefa39efp-11, 0x1.ebfbe033445b4p-23, 0x1.c6b08d704a0c0p-35, 0.0};
        for (int k = 0; k < 4; ++k) d.expc[k] = (EXP_LOG2 == 7) ? ec7[k] : ec10[k];
#ifdef RCM_EXP_DEG_OVERRIDE
        {   // experiment: plain Taylor coefficients of the shorter polynomial
            const double c = 0.6931471805599453 / EXP_TAB;
            const double tay[4] = {c, c * c / 2, c * c * c / 6, c * c * c * c / 24};
            for (int k = 0; k < 4; ++k) d.expc[k] = (k <= EXP_DEG) ? tay[k] : 0.0;
        }
#endif
    }
    // exp_scaled needs |tau/mu|/ln2 <= 1000 for every slot evaluated with exp.  Clamping tau once per layer
    // guarantees that for free - provided the clamped transmission is still zero for every use
    // (exp(-tau_clamp/mu_max) < 1e-40; the fluxes are O(100)).  Otherwise the kernel clamps inside exp.
    s->tau_clamp = 999.0 * 0.6931471805599453 / x_max;
    s->clampk = (s->tau_clamp * x_min > 92.2) ? 0 : 1;
}

// The kernels read the ensemble-wide constants from ONE __constant__ bank per device.  Several solvers
// on one device (tests, the two adapters) therefore take turns: whoever launches next re-uploads its
// constants after the device has drained.  (The intended use is one solver per GPU.)
const rcm_solver* g_const_owner[64] = {nullptr};

int refresh_const(rcm_solver* s) {
    const int dev = s->device & 63;
    if (g_const_owner[dev] != s) {
        CU(cudaDeviceSynchronize());
        s->const_dirty = true;
        g_const_owner[dev] = s;
    }
    if (!s->const_dirty) return RCM_OK;
    CU(cudaStreamSynchronize(s->stream));  // kernels in flight still read the old constants
    DevConst& d = s->dc;
    set_active_species(s);
    d.nactive = s->nactive;
    for (int k = 0; k < RCM_NSPECIES; ++k) d.species[k] = (k < s->nactive) ? s->species[k] : 0;
    d.cloud_layer = s->p.cloud_layer;
    d.cloud_row = s->p.cloud_layer < 0 ? -1 : (s->p.cloud_layer < HALF ? s->p.cloud_layer : 29 - s->p.cloud_layer);
    d.cloud_tau = s->p.cloud_tau;
    for (int r = 0; r < RCM_NLAYER; ++r) d.cloud_w[r] = (r == d.cloud_row) ? 1.0 : 0.0;
    d.dp = s->p.dp;
    d.max_dT = s->p.max_dT;
    d.dt_cap = s->p.dt_cap;
    d.solar_irr = s->p.solar_irr;
    d.dT_converged = s->p.dT_converged;
    build_angles(s);
    if (s->has_table && s->has_plevel) {
        // per-layer quantities of the shared pressure grid, reference expressions
        // (repwvl_thermal.cpp:72, :89, :202, :214, :226, :240), bottom-up index k = 19 - l
        const double avog = 6.02214076e23, molMassAir = 0.0289647, earthAccel = 9.80665;
        double P[RCM_NLEVEL];
        for (int k = 0; k < RCM_NLEVEL; ++k) P[k] = s->plevel[RCM_NLEVEL - 1 - k] * 100.0;
        for (int k = 0; k < RCM_NLAYER; ++k) {
            const int l = RCM_NLAYER - 1 - k;
            const int r = l < HALF ? l : 29 - l;  // pair-order row (see rcm_kernels.cu)
            const double midP = (P[k + 1] + P[k]) / 2;
            const long ip = rcm_lowerpos_impl(s->p_grid.data(), (int)s->p_grid.size(), midP);
            d.ip[l] = (int)ip;
            d.ipcell[r] = r * (d.n_tpert - 1);  // first cell of the layer's block in the per-layer coefficient table
            d.delP[r] = (midP - s->p_grid[ip]) / (s->p_grid[ip + 1] - s->p_grid[ip]);
            d.numDens[r] = (P[k] - P[k + 1]) * avog / molMassAir / earthAccel;
            d.tref_ip[r] = s->t_ref[ip];
        }
    }
    if (s->has_plevel) {
        for (int l = 0; l < RCM_NLAYER; ++l) {
            d.player[l] = (s->plevel[l] + s->plevel[l + 1]) / 2.0;     // main.cpp:472
            d.conv[l] = std::pow(1000.0 / d.player[l], 2.0 / 7.0);     // main.cpp:474
        }
    }
    cudaError_t e = rcm_upload_const(d);
    if (e != cudaSuccess) return cuda_fail(s, e, "upload constants");
    if (s->has_table && s->has_plevel && s->coef_dirty) {
        // bilinear coefficients of the active species per layer: coef[layer row][t interval][wvl][k][4]
        const size_t n = (size_t)RCM_NLAYER * (d.n_tpert - 1) * d.nwvl * s->nactive * 4;
        CU(dalloc(s->d_coef, n));
        CU(dalloc(s->d_species, (size_t)RCM_NSPECIES));
        CU(cudaMemcpyAsync(s->d_species, s->species, sizeof(s->species), cudaMemcpyHostToDevice, s->stream));
        CU(rcm_launch_coef(s->d_xsec_file, s->d_coef, d.n_tpert, d.n_species, d.nwvl, d.n_p, s->nactive, s->d_species,
                           s->stream));
        if (s->nactive == 5) {  // the split path's rows
            const size_t nrows = (size_t)RCM_NLAYER * (d.n_tpert - 1) * d.nwvl;
            CU(dalloc(s->d_coef3, nrows * 16));
            CU(rcm_launch_coef3(s->d_coef, s->d_coef3, nrows, s->stream));
            s->launches += 1;
        }
        CU(cudaStreamSynchronize(s->stream));
        s->launches += 1;
        s->coef_dirty = false;
    }
    s->const_dirty = false;
    return RCM_OK;
}

int ensure_columns(rcm_solver* s, int ncol) {
    if (ncol <= s->cap && s->d_T) return RCM_OK;
    const size_t n = (size_t)ncol;
    CU(dalloc(s->d_T, n * NLAY));
    CU(dalloc(s->d_Ts, n));
    CU(dalloc(s->d_vmr, n * RCM_NSPECIES * NLAY));
    CU(dalloc(s->d_rh, n * NLAY));
    CU(dalloc(s->d_Tprev, n * NLAY));
    CU(dalloc(s->d_time, n));
    CU(dalloc(s->d_Ed, n * NLEV));
    CU(dalloc(s->d_Eu, n * NLEV));
    CU(dalloc(s->d_dE, n * NLAY));
    CU(dalloc(s->d_dt, n));
    CU(dalloc(s->d_lowpos, n * NLAY));
    s->cap = ncol;
    s->diag_steps = 0;
    s->part_cap = 0;
    s->tile_cap = s->spart_cap = 0;
    s->tile_vmr_valid = false;
    if (s->d_dTstat) cudaFree(s->d_dTstat);
    s->d_dTstat = nullptr;
    // the per-column forcing buffers follow the capacity: reallocated by the next rcm_set_column_solar / checkpoint load
    if (s->d_solar_col) cudaFree(s->d_solar_col);
    if (s->d_cloud_col) cudaFree(s->d_cloud_col);
    s->d_solar_col = s->d_cloud_col = nullptr;
    s->has_col_solar = s->has_col_cloud = false;
    return RCM_OK;
}

int ensure_diag(rcm_solver* s, int nsteps) {
    if ((size_t)nsteps <= s->diag_steps && s->d_diag) return RCM_OK;
    CU(dalloc(s->d_diag, (size_t)nsteps * s->cap * 4));
    CU(dalloc(s->d_scalars, (size_t)nsteps * 4));
    CU(dalloc(s->d_red, rcm_reduce_scratch_doubles(nsteps)));
    CU(dalloc(s->d_ticket, (size_t)nsteps));  // one ticket counter per step of the capacity; every reduce launch leaves them at 0
    CU(cudaMemsetAsync(s->d_ticket, 0, (size_t)nsteps * sizeof(unsigned), s->stream));
    s->diag_steps = nsteps;
    return RCM_OK;
}

int ensure_tau(rcm_solver* s) {
    const size_t need = (size_t)s->ncol * s->dc.nwvl * NLAY;
    if (need <= s->tau_cap && s->d_tau) return RCM_OK;
    CU(dalloc(s->d_tau, need));
    s->tau_cap = need;
    return RCM_OK;
}

// CTA shapes: C columns per tile x 128 threads (2 halves x G = 64/C wavelength groups), three CTAs per SM.
// Small CTAs keep the barrier domains small; the time of one tile is proportional to the wavelengths per thread,
// ceil(nwvl / G).  `eff` is the measured relative efficiency of a shape at equal wavelength-rounds.
struct CtaShape { int C, nthreads, per_sm; double eff; };
const CtaShape kShapes[] = {{16, 128, 3, 1.0}, {8, 128, 3, 0.95}, {4, 128, 3, 0.89}, {32, 192, 2, 0.9}, {16, 96, 4, 0.93}};
constexpr int kAutoShapes = 3;  // the first three are the ones the planner picks from

struct Part { int col0, ncols; CtaShape sh; };

double part_cost(const CtaShape& sh, int ncols, int nwvl, int nsm) {
    if (ncols <= 0) return 0.0;
    const long tiles = (ncols + sh.C - 1) / sh.C, slots = (long)nsm * sh.per_sm;
    const long rounds = (tiles + slots - 1) / slots;
    const int G = sh.nthreads / (2 * sh.C);
    return (double)rounds * ((nwvl + G - 1) / G) / sh.eff;
}

// One launch covers the whole ensemble with one tile shape, so that every column sees the same order of
// floating-point additions wherever it sits (replicated columns give bit-identical results).  Tiles are dealt
// to the resident CTAs round-robin; for small ensembles narrower tiles put more SMs to work.
// (Launching a partial last round separately with narrower tiles was measured: no gain - SMs whose CTAs have
// finished leave the FP64 pipe to their neighbours' CTAs - and it breaks the bit-identity above.)
int plan_parts(const rcm_solver* s, int ncol, int nsm, Part* parts) {
    if (s->opt_config > 0 && s->opt_config <= 5) {  // forced shape (benchmarks, tests)
        parts[0] = {0, ncol, kShapes[s->opt_config - 1]};
        return 1;
    }
    const int nwvl = s->dc.nwvl;
    CtaShape best = kShapes[0];
    for (int k = 1; k < kAutoShapes; ++k)
        if (part_cost(kShapes[k], ncol, nwvl, nsm) < part_cost(best, ncol, nwvl, nsm)) best = kShapes[k];
    parts[0] = {0, ncol, best};
    return 1;
}

int nsm_of(const rcm_solver* s) {
    int nsm = 148;
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, s->device);
    return nsm;
}

// One kernel launch for the columns [p.col0, p.col0 + p.ncols) on stream st.
int launch_part(rcm_solver* s, int mode, int nsteps, bool want_diag, const Part& p, int nsm, cudaStream_t st) {
    const size_t o = (size_t)p.col0;
    StepArgs a{};
    a.ncol = p.ncols;
    a.diag_ncol = s->ncol;
    a.C = p.sh.C;
    a.ntiles = (p.ncols + a.C - 1) / a.C;
    a.nthreads = p.sh.nthreads;
    a.clampk = s->clampk;
    a.stage_rows = s->opt_stage_rows;
    a.tau_clamp = s->tau_clamp;
    a.T_floor = s->T_floor;
    a.nsteps = nsteps;
    a.step_index = s->step_index;
    a.coef = s->d_coef;
    a.planck_c = s->d_planck_c;
    a.planck_k = s->d_planck_k;
    a.Tlayer = s->d_T + o * NLAY;
    a.Tsurf = s->d_Ts + o;
    a.vmr = s->d_vmr + o * s->nactive * NLAY;
    a.rel_hum = s->d_rh + o * NLAY;
    a.Tprev = s->d_Tprev + o * NLAY;
    a.time_h = s->d_time + o;
    a.E_down = s->d_Ed + o * NLEV;
    a.E_up = s->d_Eu + o * NLEV;
    a.dE = s->d_dE + o * NLAY;
    a.dt = s->d_dt + o;
    a.diag = want_diag ? s->d_diag + o * 4 : nullptr;
    a.tau_io = s->d_tau ? s->d_tau + o * s->dc.nwvl * NLAY : nullptr;
    a.lowpos_t = s->d_lowpos + o * NLAY;
    a.exp_tab = s->d_exp_tab;
    a.h2o_slot = s->h2o_slot;
    a.solar_col = s->has_col_solar ? s->d_solar_col + o : nullptr;
    a.cloud_col = s->has_col_cloud ? s->d_cloud_col + o : nullptr;
    int per_sm = p.sh.per_sm;
    if (rcm_step_smem_bytes(a.C, s->nactive, a.nthreads) * per_sm > 224 * 1024) per_sm = 1;
    if (const char* e = std::getenv("RCM_CTAS_PER_SM")) {  // occupancy experiments (tools/occupancy_probe.py): fewer resident CTAs
        const int v = std::atoi(e);
        if (v >= 1 && v < per_sm) per_sm = v;
    }
    const int ctas = nsm * per_sm;
    const int grid = a.ntiles < ctas ? a.ntiles : ctas;
    CU(rcm_launch_step(mode, a, s->nactive, grid, st));
    s->launches += 1;
    return RCM_OK;
}


// ---- split path: (tile, wavelength split) units, two kernels per step (rcm_split_kernels.cuh) ----------------------
bool use_split(const rcm_solver* s) {
    return !s->lbl_mode && s->has_table && s->nactive == 5 && s->opt_config == 0 && s->opt_path == 0;
}

struct SplitGeom { int ntiles, nitem, nsplit; };
SplitGeom split_geom(const rcm_solver* s, int ncols) {
    SplitGeom g;
    g.ntiles = (ncols + 15) / 16;
    g.nitem = (s->dc.nwvl + 3) / 4;
    g.nsplit = (g.nitem + rcm_split_ipu() - 1) / rcm_split_ipu();
    return g;
}

int ensure_split(rcm_solver* s) {
    const SplitGeom g = split_geom(s, s->cap);
    const size_t tiles = (size_t)g.ntiles, need_part = tiles * g.nsplit * rcm_split_part_doubles();
    if (tiles > s->tile_cap || !s->d_tile) {
        CU(dalloc(s->d_tile, tiles * rcm_split_tile_bytes()));
        s->tile_cap = tiles;
        s->tile_vmr_valid = false;
    }
    if (need_part > s->spart_cap || !s->d_spart) {
        CU(dalloc(s->d_spart, need_part));
        s->spart_cap = need_part;
    }
    if (tiles > s->multi_cap || !s->d_multi) {
        if (s->d_multi) CU(cudaFree(s->d_multi));
        s->d_multi = nullptr;
        CU(cudaMalloc((void**)&s->d_multi, 2 * tiles * sizeof(unsigned)));
        s->multi_cap = tiles;
    }
    if (!s->d_dTstat) CU(dalloc(s->d_dTstat, (size_t)s->cap));
    if (!s->d_counter) {
        CU(dalloc(s->d_counter, (size_t)4));
        CU(cudaMemsetAsync(s->d_counter, 0, 4 * sizeof(unsigned), s->stream));
    }
    return RCM_OK;
}

// arguments for the columns [col0, col0 + ncols) (col0 a multiple of 16), work counter `which`
SplitArgs split_args(rcm_solver* s, int col0, int ncols, int which) {
    const SplitGeom g = split_geom(s, ncols);
    const size_t o = (size_t)col0, t0 = o / 16;
    SplitArgs a{};
    a.ncol = ncols;
    a.diag_ncol = s->ncol;
    a.ntiles = g.ntiles;
    a.nsplit = g.nsplit;
    a.ipu = rcm_split_ipu();
    a.nitem = g.nitem;
    a.nunits = g.ntiles * g.nsplit;
    a.stage_rows = s->opt_stage_rows;
    a.clampk = s->clampk;
    a.h2o_slot = s->h2o_slot;
    a.tau_clamp = s->tau_clamp;
    a.T_floor = s->T_floor;
    a.coef = s->d_coef3;
    a.planck_c = s->d_planck_c;
    a.planck_k = s->d_planck_k;
    a.exp_tab = s->d_exp_tab;
    a.Tlayer = s->d_T + o * NLAY;
    a.Tsurf = s->d_Ts + o;
    a.vmr = s->d_vmr + o * s->nactive * NLAY;
    a.rel_hum = s->d_rh + o * NLAY;
    a.Tprev = s->d_Tprev + o * NLAY;
    a.time_h = s->d_time + o;
    a.E_down = s->d_Ed + o * NLEV;
    a.E_up = s->d_Eu + o * NLEV;
    a.dE = s->d_dE + o * NLAY;
    a.dt = s->d_dt + o;
    a.diag = s->d_diag + o * 4;
    a.solar_col = s->has_col_solar ? s->d_solar_col + o : nullptr;
    a.cloud_col = s->has_col_cloud ? s->d_cloud_col + o : nullptr;
    a.tile = s->d_tile + t0 * rcm_split_tile_bytes();
    a.part = s->d_spart + t0 * g.nsplit * rcm_split_part_doubles();
    a.dTstat = s->d_dTstat + o;
    a.counter = s->d_counter + which;
    a.quota = 1 << 30;
    return a;
}

int split_grid(const rcm_solver* s, const SplitArgs& a, int nsm) {
    (void)s;
    if (a.quota < a.nunits) return (a.nunits + a.quota - 1) / a.quota;  // CTAs that leave after `quota` units
    int per_sm = 3;
    if (const char* e = std::getenv("RCM_CTAS_PER_SM")) {  // occupancy experiments
        const int v = std::atoi(e);
        if (v >= 1 && v < per_sm) per_sm = v;
    }
    return std::min(a.nunits, nsm * per_sm);
}

// K1-K4 of one step for the columns of `a` on stream st, timed with CUDA events when `timed`
int split_rt(rcm_solver* s, const SplitArgs& a, int nsm, cudaStream_t st, bool timed) {
    std::pair<cudaEvent_t, cudaEvent_t> ev{};
    if (timed) {
        if (!s->ev_free.empty()) {
            ev = s->ev_free.back();
            s->ev_free.pop_back();
        } else {
            CU(cudaEventCreate(&ev.first));
            CU(cudaEventCreate(&ev.second));
        }
        CU(cudaEventRecord(ev.first, st));
    }
    CU(rcm_launch_split_rt(a, split_grid(s, a, nsm), st));
    s->launches += 1;
    if (timed) {
        CU(cudaEventRecord(ev.second, st));
        s->ev_used.push_back(ev);
        if (s->ev_used.size() >= 1024) {
            const int rc = rcm_kernel_time_ms(s, 0, nullptr, nullptr);
            if (rc != RCM_OK) return rc;
        }
    }
    return RCM_OK;
}

// nsteps iterations of main.cpp:531-583: prep, then per step the unit kernel and one K5 kernel that finishes the step
// and prepares the next one.
int split_advance(rcm_solver* s, int nsteps) {
    int st = refresh_const(s);
    if (st != RCM_OK) return st;
    st = ensure_split(s);
    if (st != RCM_OK) return st;
    const int nsm = nsm_of(s);
    const SplitArgs a = split_args(s, 0, s->ncol, 0);
    SplitColFlags f{};
    f.prep = 1;
    f.first = (s->step_index == 0);
    f.write_all_vmr = !s->tile_vmr_valid;
    CU(rcm_launch_split_col(a, f, s->stream));
    s->launches += 1;
    s->tile_vmr_valid = true;
    // ... where a step is only a few rounds of units per CTA (8,192 columns: 5.8; the partial last round and the K5 launches
    // of every step cost 7 % there); with many rounds per step the separate K5 kernel is the cheaper one (65,536 columns:
    // 46 rounds, one launch per block 0.9 % slower than three per step).  opt_multi = 2 forces it (tests).
    static const int multi_rounds = std::getenv("RCM_MULTI_ROUNDS") ? std::atoi(std::getenv("RCM_MULTI_ROUNDS")) : 24;
    const int grid1 = split_grid(s, a, nsm);
    const bool few_rounds = a.nunits < (long long)multi_rounds * grid1;
    // (item numbers are 32-bit: units x steps of one launch, plus the tickets of the CTAs that find the counter exhausted)
    const bool fits = (long long)a.nunits * nsteps + 2LL * grid1 < (1LL << 31);
    if (nsteps >= 2 && fits && (s->opt_multi == 2 || (s->opt_multi == 1 && few_rounds))) {
        // a block of steps as ONE launch: (step, unit) items in step-major order, per-tile step flags instead of kernel
        // boundaries, the K5 body run by the CTA that completes a tile's step (rcm_split_multi_kernel)
        SplitMultiArgs m{};
        m.nsteps = nsteps;
        m.done = s->d_multi;
        m.ready = s->d_multi + a.ntiles;
        CU(cudaMemsetAsync(s->d_multi, 0, 2 * (size_t)a.ntiles * sizeof(unsigned), s->stream));
        SplitArgs am = a;
        am.quota = 1 << 30;
        CU(rcm_launch_split_multi(am, m, split_grid(s, am, nsm), s->stream));
        s->launches += 1;
        return RCM_OK;
    }
    for (int k = 0; k < nsteps; ++k) {
        st = split_rt(s, a, nsm, s->stream, k < 4);  // long blocks: the first steps are timed, the rest run without event records
        if (st != RCM_OK) return st;
        SplitColFlags e{};
        e.finish = 1;
        e.prep = (k + 1 < nsteps);
        e.first = 0;
        e.write_out = (k + 1 == nsteps);
        e.diag_step = k;
        CU(rcm_launch_split_col(a, e, s->stream));
        s->launches += 1;
    }
    return RCM_OK;
}

int launch(rcm_solver* s, int mode, int nsteps, bool want_diag) {
    int st = refresh_const(s);
    if (st != RCM_OK) return st;
    if (mode == MODE_RT ? !s->has_spectral : !s->has_table) return fail(s, RCM_ERR_STATE, "no lookup table loaded");
    if (s->ncol <= 0) return fail(s, RCM_ERR_STATE, "no columns loaded");
    const int nsm = nsm_of(s);
    Part parts[2];
    const int nparts = plan_parts(s, s->ncol, nsm, parts);
    std::pair<cudaEvent_t, cudaEvent_t> ev;
    if (!s->ev_free.empty()) {
        ev = s->ev_free.back();
        s->ev_free.pop_back();
    } else {
        CU(cudaEventCreate(&ev.first));
        CU(cudaEventCreate(&ev.second));
    }
    CU(cudaEventRecord(ev.first, s->stream));
    for (int ip = 0; ip < nparts; ++ip) {
        st = launch_part(s, mode, nsteps, want_diag, parts[ip], nsm, s->stream);
        if (st != RCM_OK) return st;
    }
    CU(cudaEventRecord(ev.second, s->stream));
    if (mode == MODE_STEP) s->ev_used.push_back(ev); else s->ev_free.push_back(ev);
    if (s->ev_used.size() >= 1024) {  // long runs: fold the finished timings so the pool stays small
        st = rcm_kernel_time_ms(s, 0, nullptr, nullptr);
        if (st != RCM_OK) return st;
    }
    return RCM_OK;
}


// rcm_step_host on the split path: the columns travel in chunks of whole tiles through three stages on their own streams,
//   up   (high priority): H2D of the chunk's T / Tsurf / VMRs, K5 prep
//   rt   (two streams, alternating): the unit kernel of the chunk - its CTAs leave after four units, so the slots they
//        hold recycle every ~0.3 ms and the small K5 kernels of the other stages get in without waiting for a whole chunk,
//        and the next chunk's CTAs fill the SMs while this chunk's last units finish (no tail per chunk)
//   down (high priority): K5 finish, D2H of the chunk's results
// Results are bit-identical to rcm_update_columns + rcm_advance + rcm_get_state.
int step_host_split(rcm_solver* s, int nchunk, const double* Tlayer_in, const double* Tsurf_in, const double* vmr_active_in,
                    double* E_down, double* E_up, double* dE, double* Tlayer_out, double* Tsurf_out) {
    int st = ensure_split(s);
    if (st != RCM_OK) return st;
    if (!s->sp_up) {
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // hi = greatest priority (numerically lowest)
        CU(cudaStreamCreateWithPriority(&s->sp_up, cudaStreamNonBlocking, hi));
        CU(cudaStreamCreateWithPriority(&s->sp_down, cudaStreamNonBlocking, hi));
        for (int i = 0; i < 2; ++i) CU(cudaStreamCreateWithPriority(&s->sp_rt[i], cudaStreamNonBlocking, lo));
        for (int i = 0; i < 24; ++i) {
            CU(cudaEventCreateWithFlags(&s->sp_prep[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&s->sp_rtdone[i], cudaEventDisableTiming));
        }
        CU(cudaEventCreateWithFlags(&s->sp_end, cudaEventDisableTiming));
    }
    const int nsm = nsm_of(s);
    const int per = ((s->ncol + nchunk - 1) / nchunk + 15) / 16 * 16;
    // chunk boundaries (whole tiles): the first and the last chunk are quarter-sized, their neighbours three quarters - the
    // upload of the first chunk and the download of the last one are the only copies nothing overlaps
    int bounds[24];
    int nb = 0;
    bounds[nb++] = 0;
    if (nchunk >= 4 && per >= 64) {
        const int q = per / 4 / 16 * 16;
        bounds[nb++] = q;
        for (int c0 = per; c0 < s->ncol - q; c0 += per) bounds[nb++] = c0;
        bounds[nb++] = std::max(bounds[nb - 1], s->ncol - q) / 16 * 16;
    } else {
        for (int c0 = per; c0 < s->ncol; c0 += per) bounds[nb++] = c0;
    }
    bounds[nb] = s->ncol;
    const size_t D = sizeof(double);
    const int na = s->nactive;
    // everything of one call, from the fork off the solver's stream to the scalar reduction after the join
    auto enqueue = [&](bool timed) -> int {
    int nk = 0;
    CU(cudaEventRecord(s->sp_end, s->stream));  // everything queued on the solver's stream so far comes first
    for (cudaStream_t q : {s->sp_up, s->sp_rt[0], s->sp_rt[1], s->sp_down}) CU(cudaStreamWaitEvent(q, s->sp_end, 0));
    for (int k = 0; k < nb; ++k) {
        const int c0 = bounds[k], n = bounds[k + 1] - c0;
        if (n <= 0) continue;
        const size_t o = (size_t)c0;
        cudaStream_t q = s->sp_up;
        if (Tlayer_in) CU(cudaMemcpyAsync(s->d_T + o * NLAY, Tlayer_in + o * NLAY, n * NLAY * D, cudaMemcpyHostToDevice, q));
        if (Tsurf_in) CU(cudaMemcpyAsync(s->d_Ts + o, Tsurf_in + o, n * D, cudaMemcpyHostToDevice, q));
        if (vmr_active_in)
            CU(cudaMemcpyAsync(s->d_vmr + o * na * NLAY, vmr_active_in + o * na * NLAY, (size_t)n * na * NLAY * D,
                               cudaMemcpyHostToDevice, q));
        SplitArgs a = split_args(s, c0, n, 1 + k % 2);
        a.quota = 4;
        SplitArgs ac = a;
        ac.counter = nullptr;  // the K5 kernels run on other streams than the unit kernel: the counter is reset on its own stream
        SplitColFlags f{};
        f.prep = 1;
        f.first = (s->step_index == 0);
        f.write_all_vmr = !s->tile_vmr_valid || vmr_active_in != nullptr;
        CU(rcm_launch_split_col(ac, f, q));
        CU(cudaEventRecord(s->sp_prep[k], q));
        q = s->sp_rt[k % 2];
        CU(cudaStreamWaitEvent(q, s->sp_prep[k], 0));
        CU(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), q));
        st = split_rt(s, a, nsm, q, timed);
        if (st != RCM_OK) return st;
        nk += 3;
        CU(cudaEventRecord(s->sp_rtdone[k], q));
        q = s->sp_down;
        CU(cudaStreamWaitEvent(q, s->sp_rtdone[k], 0));
        SplitColFlags e{};
        e.finish = 1;
        e.write_out = 1;
        CU(rcm_launch_split_col(ac, e, q));
        s->launches += 2;
        if (E_down) CU(cudaMemcpyAsync(E_down + o * NLEV, s->d_Ed + o * NLEV, n * NLEV * D, cudaMemcpyDeviceToHost, q));
        if (E_up) CU(cudaMemcpyAsync(E_up + o * NLEV, s->d_Eu + o * NLEV, n * NLEV * D, cudaMemcpyDeviceToHost, q));
        if (dE) CU(cudaMemcpyAsync(dE + o * NLAY, s->d_dE + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToHost, q));
        if (Tlayer_out) CU(cudaMemcpyAsync(Tlayer_out + o * NLAY, s->d_T + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToHost, q));
        if (Tsurf_out) CU(cudaMemcpyAsync(Tsurf_out + o, s->d_Ts + o, n * D, cudaMemcpyDeviceToHost, q));
    }
    CU(cudaEventRecord(s->sp_end, s->sp_down));  // the last stage of the last chunk: everything before it is done
    CU(cudaStreamWaitEvent(s->stream, s->sp_end, 0));
    CU(rcm_launch_reduce_diag(s->d_diag, 1, s->ncol, s->p.dT_converged, s->d_red, s->d_ticket, s->d_scalars, s->stream));
    s->launches += 1;
    s->hg.nkernels = nk + 1;
    return RCM_OK;
    };  // enqueue

    // Steady state (not the first iteration, VMR rows of the tile blocks current, no VMR upload): the call is the same
    // sequence every time - launch it as one graph.  RCM_NO_GRAPH=1 keeps the direct calls (comparison).
    const bool steady = s->step_index > 0 && s->tile_vmr_valid && !vmr_active_in && !s->hg.failed && !std::getenv("RCM_NO_GRAPH");
    bool launched = false;
    if (steady) {
        rcm_solver::HostGraph& g = s->hg;
        const SplitArgs sig = split_args(s, 0, s->ncol, 1);
        const void* host[7] = {Tlayer_in, Tsurf_in, E_down, E_up, dE, Tlayer_out, Tsurf_out};
        const void* dev[4] = {s->d_diag, s->d_red, s->d_ticket, s->d_scalars};
        const bool same = g.exec && std::memcmp(&g.sig, &sig, sizeof(sig)) == 0 && std::memcmp(g.host, host, sizeof(host)) == 0 &&
                          std::memcmp(g.dev, dev, sizeof(dev)) == 0 && g.dT_converged == s->p.dT_converged && g.ncol == s->ncol &&
                          g.nchunk == nchunk;
        if (!same) {
            if (g.exec) cudaGraphExecDestroy(g.exec);
            g.exec = nullptr;
            cudaGraph_t graph = nullptr;
            const long launches0 = s->launches;
            // asynchronous copies can only be captured from / to page-locked host memory: with pageable buffers stay direct
            bool ok = true;
            for (const void* hp : host) {
                cudaPointerAttributes at{};
                if (hp && (cudaPointerGetAttributes(&at, hp) != cudaSuccess || at.type != cudaMemoryTypeHost)) ok = false;
            }
            cudaGetLastError();
            ok = ok && cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeRelaxed) == cudaSuccess;
            if (ok) {
                ok = enqueue(false) == RCM_OK;
                ok = (cudaStreamEndCapture(s->stream, &graph) == cudaSuccess) && ok && graph;
            }
            s->launches = launches0;  // captured, not launched
            g.captures += 1;
            if (ok) ok = cudaGraphInstantiate(&g.exec, graph, 0) == cudaSuccess;
            if (graph) cudaGraphDestroy(graph);
            if (!ok) {  // direct calls: for this call with pageable buffers, for good when the capture itself failed
                cudaGetLastError();
                g.exec = nullptr;
                bool pinned = true;
                for (const void* hp : host) {
                    cudaPointerAttributes at{};
                    if (hp && (cudaPointerGetAttributes(&at, hp) != cudaSuccess || at.type != cudaMemoryTypeHost)) pinned = false;
                }
                cudaGetLastError();
                if (pinned) g.failed = true;
            } else {
                g.sig = sig;
                std::memcpy(g.host, host, sizeof(host));
                std::memcpy(g.dev, dev, sizeof(dev));
                g.dT_converged = s->p.dT_converged;
                g.ncol = s->ncol;
                g.nchunk = nchunk;
            }
        }
        if (g.exec) {
            CU(cudaGraphLaunch(g.exec, s->stream));
            s->launches += g.nkernels;
            g.replays += 1;
            launched = true;
        }
    }
    if (!launched) {
        st = enqueue(true);
        if (st != RCM_OK) return st;
    }
    s->step_index += 1;
    s->tau_valid = false;
    s->tile_vmr_valid = true;
    CU(cudaStreamSynchronize(s->stream));
    return RCM_OK;
}

}  // namespace

extern "C" {

int rcm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int rcm_create(int device, const rcm_params* p, rcm_solver** out) {
    if (!out) return RCM_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return RCM_ERR_NO_DEVICE;
    if (device < 0 || device >= n) return RCM_ERR_ARG;
    rcm_solver* s = new (std::nothrow) rcm_solver();
    if (!s) return RCM_ERR_NOMEM;
    s->device = device;
    if (p) s->p = *p; else rcm_default_params(&s->p);
    if (s->p.nangle < 1 || s->p.nangle > MAX_ANGLE || s->p.cloud_layer >= RCM_NLAYER) {
        delete s;
        return RCM_ERR_ARG;
    }
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete s;
        return RCM_ERR_CUDA;
    }
    s->stream = s->own_stream;
    // 2^(j/128) with j << 13 pre-subtracted from the high word: exp_scaled adds k << 13 = (m << 20) + (j << 13)
    double tab[EXP_TAB];
    for (int j = 0; j < EXP_TAB; ++j) {
        const double v = std::exp2((double)j / EXP_TAB);
        unsigned long long bits;
        std::memcpy(&bits, &v, 8);
        bits -= (unsigned long long)j << (20 - EXP_LOG2 + 32);
        std::memcpy(&tab[j], &bits, 8);
    }
    if (dalloc(s->d_exp_tab, EXP_TAB) != cudaSuccess ||
        cudaMemcpy(s->d_exp_tab, tab, sizeof(tab), cudaMemcpyHostToDevice) != cudaSuccess) {
        delete s;
        return RCM_ERR_CUDA;
    }
    set_active_species(s);
    *out = s;
    return RCM_OK;
}

int rcm_destroy(rcm_solver* s) {
    if (!s) return RCM_OK;
    cudaSetDevice(s->device);
    cudaStreamSynchronize(s->stream);
    if (g_const_owner[s->device & 63] == s) g_const_owner[s->device & 63] = nullptr;
    void* ptrs[] = {s->d_coef3, s->d_xsec_file, s->d_coef, s->d_species, s->d_planck_c, s->d_planck_k, s->d_exp_tab, s->d_T, s->d_Ts, s->d_vmr, s->d_rh,
                    s->d_Tprev, s->d_time, s->d_lbl_lo, s->d_lbl_hi, s->d_lbl_tau5, s->d_lbl_h2o_ref, s->d_lbl_o3_ref, s->d_lbl_tau3s, s->d_sH, s->d_sO,
                    s->d_dTstat, s->d_part, s->d_Ed, s->d_Eu, s->d_dE, s->d_dt, s->d_diag, s->d_scalars, s->d_red, s->d_tau,
                    s->d_lowpos, s->d_solar_col, s->d_cloud_col, s->d_ticket, s->d_tile, s->d_spart, s->d_counter, s->d_multi, s->d_diagnose};
    for (void* q : ptrs)
        if (q) cudaFree(q);
    for (auto& e : s->ev_free) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    for (auto& e : s->ev_used) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    for (int i = 0; i < 3; ++i) {
        if (s->pipe_stream[i]) cudaStreamDestroy(s->pipe_stream[i]);
        if (s->pipe_done[i]) cudaEventDestroy(s->pipe_done[i]);
    }
    if (s->pipe_start) cudaEventDestroy(s->pipe_start);
    for (cudaStream_t q : {s->sp_up, s->sp_rt[0], s->sp_rt[1], s->sp_down})
        if (q) cudaStreamDestroy(q);
    for (int i = 0; i < 24; ++i) {
        if (s->sp_prep[i]) cudaEventDestroy(s->sp_prep[i]);
        if (s->sp_rtdone[i]) cudaEventDestroy(s->sp_rtdone[i]);
    }
    if (s->sp_end) cudaEventDestroy(s->sp_end);
    for (int i = 0; i < 2; ++i) {
        if (s->dg_stream[i]) cudaStreamDestroy(s->dg_stream[i]);
        if (s->dg_join[i]) cudaEventDestroy(s->dg_join[i]);
    }
    if (s->dg_fork) cudaEventDestroy(s->dg_fork);
    if (s->h_fdh_count) cudaFreeHost(s->h_fdh_count);
    if (s->hg.exec) cudaGraphExecDestroy(s->hg.exec);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    delete s;
    return RCM_OK;
}

const char* rcm_last_error(const rcm_solver* s) { return s ? s->err.c_str() : "null solver"; }

int rcm_set_params(rcm_solver* s, const rcm_params* p) {
    if (!s || !p) return RCM_ERR_ARG;
    if (p->nangle < 1 || p->nangle > MAX_ANGLE || p->cloud_layer >= RCM_NLAYER) return fail(s, RCM_ERR_ARG, "bad params");
    unsigned old = s->p.species_mask;
    s->p = *p;
    if (old != p->species_mask) {
        s->coef_dirty = true;
        s->ncol = 0;  // packed VMR layout changed: columns must be reloaded
    }
    s->const_dirty = true;
    set_active_species(s);
    return RCM_OK;
}

int rcm_set_option(rcm_solver* s, int option, int value) {
    if (!s) return RCM_ERR_ARG;
    if (option == 0) {
        s->opt_angle_cubes = value ? 1 : 0;
        s->const_dirty = true;
        return RCM_OK;
    }
    if (option == 1) {
        s->opt_config = value;
        s->tile_vmr_valid = false;
        return RCM_OK;
    }
    if (option == 2) {
        s->opt_cplk_narrow = value ? 1 : 0;
        return RCM_OK;
    }
    if (option == 3) {
        s->opt_stage_rows = value ? 1 : 0;
        return RCM_OK;
    }
    if (option == 4) {
        s->opt_angle_pairs = value ? 1 : 0;
        s->const_dirty = true;
        return RCM_OK;
    }
    if (option == 5) {
        s->opt_path = value ? 1 : 0;
        s->tile_vmr_valid = false;
        return RCM_OK;
    }
    if (option == 6) {
        s->opt_multi = value < 0 ? 0 : value > 2 ? 2 : value;
        return RCM_OK;
    }
    return fail(s, RCM_ERR_ARG, "unknown option");
}

int rcm_set_stream(rcm_solver* s, void* cuda_stream) {
    if (!s) return RCM_ERR_ARG;
    s->stream = cuda_stream ? (cudaStream_t)cuda_stream : s->own_stream;
    return RCM_OK;
}

int rcm_synchronize(rcm_solver* s) {
    if (!s) return RCM_ERR_ARG;
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->stream));
    return RCM_OK;
}

int rcm_set_repwvl_table(rcm_solver* s, const double* xsec, const double* wvl, const double* weight,
                         const double* p_grid, const double* t_ref, const double* t_pert, int n_tpert, int n_species,
                         int n_wvl, int n_p) {
    if (!s || !xsec || !wvl || !weight || !p_grid || !t_ref || !t_pert) return RCM_ERR_ARG;
    if (n_tpert < 2 || n_tpert > MAX_TPERT || n_species != RCM_NSPECIES || n_wvl < 1 || n_p < 2)
        return fail(s, RCM_ERR_ARG, "unsupported table dimensions");
    CU(cudaSetDevice(s->device));
    const size_t n = (size_t)n_tpert * n_species * n_wvl * n_p;
    CU(dalloc(s->d_xsec_file, n));
    CU(cudaMemcpy(s->d_xsec_file, xsec, n * sizeof(double), cudaMemcpyHostToDevice));
    s->coef_dirty = true;
    {
        int st = rcm_set_spectral_grid(s, wvl, weight, n_wvl);
        if (st != RCM_OK) return st;
    }
    s->p_grid.assign(p_grid, p_grid + n_p);
    s->t_ref.assign(t_ref, t_ref + n_p);
    s->t_pert.assign(t_pert, t_pert + n_tpert);
    s->dc.nwvl = n_wvl;
    s->dc.n_tpert = n_tpert;
    s->dc.n_species = n_species;
    s->dc.n_p = n_p;
    for (int m = 0; m < n_tpert; ++m) s->dc.t_pert[m] = t_pert[m];
    s->has_table = true;
    s->lbl_mode = false;
    s->const_dirty = true;
    s->tau_valid = false;
    s->tau_cap = 0;
    return RCM_OK;
}

int rcm_set_spectral_grid(rcm_solver* s, const double* wvl, const double* weight, int n_wvl) {
    if (!s || !wvl || !weight || n_wvl < 1) return RCM_ERR_ARG;
    CU(cudaSetDevice(s->device));
    // Planck factors that depend on the wavelength alone (main.cpp:188-191):
    //   B = w*2*h*c^2 / (lambda^5 * (exp(h*c/(lambda*kB*T)) - 1)) / 1e9
    const double h = 6.62607e-34, c = 299792458, kB = 1.380649e-23;  // main.cpp:70-72
    std::vector<double> pc(n_wvl), pk(n_wvl);
    double pc_max = 0.0;
    for (int i = 0; i < n_wvl; ++i) {
        const double lam = wvl[i] * 1e-9;
        pc[i] = h * c / (lam * kB);
        pk[i] = weight[i] * 2 * h * std::pow(c, 2) / std::pow(lam, 5) / 1e9;
        if (!(wvl[i] > 0.0) || !std::isfinite(pk[i])) return fail(s, RCM_ERR_ARG, "wavelengths must be positive and finite");
        pc_max = std::max(pc_max, pc[i]);
    }
    // The kernels' exp (exp_scaled) takes exponents up to ~700 and has no overflow path: the Planck exponent
    // h*c/(lambda*kB*T) is kept below 690 by evaluating the source at max(T, T_floor), T_floor = max(h*c/(lambda*kB)) / 690
    // (5.1 K for the repwvl tables; the reference's exp overflows to inf there and its source is 0 - here it is < 1e-299
    // of the Planck factor).  A grid whose floor would reach atmospheric temperatures is refused: this is the thermal path.
    if (pc_max / 690.0 > 20.0)
        return fail(s, RCM_ERR_ARG, "wavelengths below 1043 nm are not supported (thermal solver: the Planck exponent would leave the range of the kernels' exp)");
    s->T_floor = pc_max / 690.0;
    CU(dalloc(s->d_planck_c, (size_t)n_wvl));
    CU(dalloc(s->d_planck_k, (size_t)n_wvl));
    CU(cudaMemcpy(s->d_planck_c, pc.data(), n_wvl * sizeof(double), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(s->d_planck_k, pk.data(), n_wvl * sizeof(double), cudaMemcpyHostToDevice));
    s->wvl.assign(wvl, wvl + n_wvl);
    s->weight.assign(weight, weight + n_wvl);
    if (s->dc.nwvl != n_wvl) {  // a cross-section table of another size can no longer be used
        s->has_table = false;
        s->tau_cap = 0;
    }
    s->dc.nwvl = n_wvl;
    s->has_spectral = true;
    s->lbl_mode = false;
    s->const_dirty = true;
    s->tau_valid = false;
    return RCM_OK;
}

int rcm_set_repwvl_table_from(rcm_solver* s, const rcm_table* t) {
    if (!s || !t) return RCM_ERR_ARG;
    return rcm_set_repwvl_table(s, t->xsec.data(), t->wvl.data(), t->weight.data(), t->p_grid.data(), t->t_ref.data(),
                                t->t_pert.data(), t->n_tpert, t->n_species, t->n_wvl, t->n_p);
}

int rcm_set_lbl_tables(rcm_solver* s, const double* wvl, const double* tau5, int nwvl, const double* h2o_ref,
                       const double* o3_ref, double co2_factor) {
    if (!s || !wvl || !tau5 || nwvl < 2 || !h2o_ref) return RCM_ERR_ARG;
    for (int i = 1; i < nwvl; ++i)
        if (!(wvl[i] > wvl[i - 1])) return fail(s, RCM_ERR_ARG, "LBL wavelengths must be strictly ascending");
    CU(cudaSetDevice(s->device));
    // spectral bins: bounded by the midpoints between adjacent wavelengths, end bins mirrored
    // (builder decision, DESIGN.md section 5; cplkavg() needs hi > lo, cplkavg.cpp:144-146)
    std::vector<double> lo(nwvl), hi(nwvl);
    for (int i = 0; i < nwvl; ++i) {
        const double dl = (i > 0) ? (wvl[i] - wvl[i - 1]) : (wvl[1] - wvl[0]);
        const double dh = (i < nwvl - 1) ? (wvl[i + 1] - wvl[i]) : (wvl[i] - wvl[i - 1]);
        lo[i] = wvl[i] - dl / 2.0;
        hi[i] = wvl[i] + dh / 2.0;
    }
    const size_t n = (size_t)nwvl;
    CU(dalloc(s->d_lbl_lo, 4 * n));  // planes: lo, (hi in d_lbl_hi), whi, wlo, and the narrow-band flags as ints
    CU(dalloc(s->d_lbl_hi, n));
    CU(dalloc(s->d_lbl_tau5, 6 * n * NLAY));
    CU(dalloc(s->d_lbl_h2o_ref, (size_t)NLAY));
    CU(dalloc(s->d_lbl_o3_ref, (size_t)NLAY));
    CU(cudaMemcpy(s->d_lbl_lo, lo.data(), n * sizeof(double), cudaMemcpyHostToDevice));
    {   // per-bin quantities of cplkavg (cplkavg.cpp:141-142, :155), evaluated here once with the reference's expressions
        std::vector<double> wn(2 * n);
        std::vector<int> ok(2 * n, 0);  // (ints in a plane of doubles: 2n ints)
        for (size_t i = 0; i < n; ++i) {
            const double whi = 1.0E7 / lo[i], wlo = 1.0E7 / hi[i];
            wn[i] = whi;
            wn[n + i] = wlo;
            ok[i] = (whi > wlo && wlo >= 0. && (whi - wlo) / whi < 1.e-2) ? 1 : 0;
        }
        CU(cudaMemcpy(s->d_lbl_lo + n, wn.data(), 2 * n * sizeof(double), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(s->d_lbl_lo + 3 * n, ok.data(), n * sizeof(int), cudaMemcpyHostToDevice));
    }
    CU(cudaMemcpy(s->d_lbl_hi, hi.data(), n * sizeof(double), cudaMemcpyHostToDevice));
    {   // device planes: tau_H2O, tau_O3, and the column-independent part f_CO2 * tau_CO2 + tau_CH4 + tau_N2O; behind them the
        // raw CO2, CH4, N2O planes, from which rcm_lbl_diagnose_fluxes composes that part with scaled species
        const size_t plane = n * NLAY;
        std::vector<double> t3(6 * plane);
        std::memcpy(&t3[0], tau5, plane * sizeof(double));
        std::memcpy(&t3[plane], tau5 + 2 * plane, plane * sizeof(double));
        for (size_t i = 0; i < plane; ++i) t3[2 * plane + i] = co2_factor * tau5[plane + i] + tau5[3 * plane + i] + tau5[4 * plane + i];
        std::memcpy(&t3[3 * plane], tau5 + plane, plane * sizeof(double));
        std::memcpy(&t3[4 * plane], tau5 + 3 * plane, 2 * plane * sizeof(double));
        CU(cudaMemcpy(s->d_lbl_tau5, t3.data(), t3.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    CU(cudaMemcpy(s->d_lbl_h2o_ref, h2o_ref, NLAY * sizeof(double), cudaMemcpyHostToDevice));
    s->lbl_has_o3_ref = o3_ref != nullptr;
    if (o3_ref) CU(cudaMemcpy(s->d_lbl_o3_ref, o3_ref, NLAY * sizeof(double), cudaMemcpyHostToDevice));
    s->lbl_nwvl = nwvl;
    s->lbl_co2_factor = co2_factor;
    s->lbl_mode = true;
    // dc.nwvl now counts LBL wavelengths: the repwvl table / spectral grid on the device (d_coef, d_planck_*) are sized
    // for another grid and must not be used with it - they have to be set again to go back to the repwvl path
    if (s->dc.nwvl != nwvl) {
        s->has_table = s->has_spectral = false;
        s->tau_cap = 0;
    }
    s->tau_valid = false;
    s->dc.nwvl = nwvl;
    s->const_dirty = true;
    s->part_cap = 0;
    return RCM_OK;
}

int rcm_set_columns(rcm_solver* s, int ncol, const double* plevel_hPa, const double* Tlayer, const double* Tsurf,
                    const double* vmr9, const double* rel_hum) {
    if (!s || ncol <= 0 || !plevel_hPa || !Tlayer || !Tsurf || !vmr9 || !rel_hum) return RCM_ERR_ARG;
    CU(cudaSetDevice(s->device));
    int st = ensure_columns(s, ncol);
    if (st != RCM_OK) return st;
    s->ncol = ncol;
    if (!s->has_plevel || std::memcmp(s->plevel, plevel_hPa, sizeof(s->plevel)) != 0) s->coef_dirty = true;  // per-layer table
    std::memcpy(s->plevel, plevel_hPa, sizeof(s->plevel));
    s->has_plevel = true;
    s->const_dirty = true;
    set_active_species(s);
    const size_t n = (size_t)ncol;
    // pack the active species rows: [ncol][nactive][20]
    s->stage.resize(n * s->nactive * NLAY);
    for (size_t c = 0; c < n; ++c)
        for (int k = 0; k < s->nactive; ++k)
            std::memcpy(&s->stage[(c * s->nactive + k) * NLAY], vmr9 + (c * RCM_NSPECIES + s->species[k]) * NLAY,
                        NLAY * sizeof(double));
    CU(cudaMemcpyAsync(s->d_vmr, s->stage.data(), s->stage.size() * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(s->d_T, Tlayer, n * NLAY * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(s->d_Tprev, Tlayer, n * NLAY * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(s->d_Ts, Tsurf, n * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(s->d_rh, rel_hum, n * NLAY * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemsetAsync(s->d_time, 0, n * sizeof(float), s->stream));
    CU(cudaStreamSynchronize(s->stream));
    s->step_index = 0;
    s->tau_valid = false;
    s->tile_vmr_valid = false;
    s->has_col_solar = s->has_col_cloud = false;  // per-column forcing belongs to the column set it was given for
    return RCM_OK;
}

int rcm_set_column_solar(rcm_solver* s, const rcm_solar_params* sp, const double* tau_s, const double* mu_s,
                         const double* albedo, int cloud_from_tau_s, double* solar_irr_out, double* r_total_out) {
    if (!s) return RCM_ERR_ARG;
    if (s->ncol <= 0) return fail(s, RCM_ERR_STATE, "rcm_set_columns first");
    CU(cudaSetDevice(s->device));
    if (!sp) {  // back to the ensemble-wide constants of rcm_params
        s->has_col_solar = s->has_col_cloud = false;
        s->tau_valid = false;
        return RCM_OK;
    }
    if (sp->doublings < 0 || sp->doublings > 60) return fail(s, RCM_ERR_ARG, "doublings must be in 0..60");
    if (cloud_from_tau_s && s->p.cloud_layer < 0) return fail(s, RCM_ERR_ARG, "cloud_from_tau_s needs a cloud layer");
    const size_t n = (size_t)s->ncol;
    if (!s->d_solar_col) {
        CU(dalloc(s->d_solar_col, (size_t)s->cap));
        CU(dalloc(s->d_cloud_col, (size_t)s->cap));
    }
    // inputs travel through one scratch allocation [3][n]; r_total comes back through its first row
    double* d_in = nullptr;
    CU(cudaMalloc((void**)&d_in, 3 * n * sizeof(double)));
    const double* src[3] = {tau_s, mu_s, albedo};
    for (int k = 0; k < 3; ++k)
        if (src[k]) {
            cudaError_t e = cudaMemcpyAsync(d_in + k * n, src[k], n * sizeof(double), cudaMemcpyHostToDevice, s->stream);
            if (e != cudaSuccess) { cudaFree(d_in); return cuda_fail(s, e, "upload solar inputs"); }
        }
    double* d_rt = nullptr;
    if (r_total_out) {
        cudaError_t e = cudaMalloc((void**)&d_rt, n * sizeof(double));
        if (e != cudaSuccess) { cudaFree(d_in); return cuda_fail(s, e, "cudaMalloc"); }
    }
    SolarArgs a{};
    a.n = s->ncol;
    a.doublings = sp->doublings;
    a.tau_s = sp->tau_s; a.mu_s = sp->mu_s; a.g_asym = sp->g_asym; a.albedo = sp->albedo; a.daytime = sp->daytime; a.E_0 = sp->E_0;
    a.tau_s_col = tau_s ? d_in : nullptr;
    a.mu_s_col = mu_s ? d_in + n : nullptr;
    a.albedo_col = albedo ? d_in + 2 * n : nullptr;
    a.solar_irr = s->d_solar_col;
    a.r_total = d_rt;
    a.cloud_tau = cloud_from_tau_s ? s->d_cloud_col : nullptr;
    cudaError_t e = rcm_launch_solar(a, s->stream);
    if (e == cudaSuccess && solar_irr_out)
        e = cudaMemcpyAsync(solar_irr_out, s->d_solar_col, n * sizeof(double), cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess && r_total_out)
        e = cudaMemcpyAsync(r_total_out, d_rt, n * sizeof(double), cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    cudaFree(d_in);
    if (d_rt) cudaFree(d_rt);
    if (e != cudaSuccess) return cuda_fail(s, e, "rcm_set_column_solar");
    s->launches += 1;
    s->has_col_solar = true;
    s->has_col_cloud = cloud_from_tau_s != 0;
    s->tau_valid = false;
    return RCM_OK;
}

int rcm_update_columns(rcm_solver* s, const double* Tlayer, const double* Tsurf, const double* vmr_active) {
    if (!s) return RCM_ERR_ARG;
    if (s->ncol <= 0) return fail(s, RCM_ERR_STATE, "rcm_set_columns first");
    CU(cudaSetDevice(s->device));
    const size_t n = (size_t)s->ncol;
    if (Tlayer) CU(cudaMemcpyAsync(s->d_T, Tlayer, n * NLAY * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    if (Tsurf) CU(cudaMemcpyAsync(s->d_Ts, Tsurf, n * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    if (vmr_active)
        CU(cudaMemcpyAsync(s->d_vmr, vmr_active, n * s->nactive * NLAY * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    if (vmr_active) s->tile_vmr_valid = false;
    s->tau_valid = false;
    return RCM_OK;
}

int rcm_set_step_index(rcm_solver* s, long step_index) {
    if (!s || step_index < 0) return RCM_ERR_ARG;
    s->step_index = step_index;
    return RCM_OK;
}

int rcm_build_tau(rcm_solver* s, double* tau_out, int* lowpos_p, int* lowpos_t) {
    if (!s) return RCM_ERR_ARG;
    if (s->lbl_mode) return fail(s, RCM_ERR_STATE, "rcm_build_tau is the repwvl read_tau: set a repwvl table after rcm_set_lbl_tables");
    if (!s->has_table || s->ncol <= 0) return fail(s, RCM_ERR_STATE, "table and columns must be loaded");
    CU(cudaSetDevice(s->device));
    int st = ensure_tau(s);
    if (st != RCM_OK) return st;
    st = launch(s, MODE_TAU, 1, false);
    if (st != RCM_OK) return st;
    const size_t n = (size_t)s->ncol;
    if (tau_out)
        CU(cudaMemcpyAsync(tau_out, s->d_tau, n * s->dc.nwvl * NLAY * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    std::vector<int> lt;
    if (lowpos_t) CU(cudaMemcpyAsync(lowpos_t, s->d_lowpos, n * NLAY * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    if (lowpos_p)
        for (size_t c = 0; c < n; ++c)
            for (int k = 0; k < NLAY; ++k) lowpos_p[c * NLAY + k] = s->dc.ip[NLAY - 1 - k];
    s->tau_valid = true;
    return RCM_OK;
}

int rcm_radiative_transfer(rcm_solver* s, const double* tau, double* E_down, double* E_up, double* dE) {
    if (!s) return RCM_ERR_ARG;
    if (s->lbl_mode) return fail(s, RCM_ERR_STATE, "rcm_radiative_transfer needs a repwvl spectral grid: set one after rcm_set_lbl_tables");
    if (!s->has_spectral || s->ncol <= 0) return fail(s, RCM_ERR_STATE, "spectral grid and columns must be loaded");
    CU(cudaSetDevice(s->device));
    int st = ensure_tau(s);
    if (st != RCM_OK) return st;
    const size_t n = (size_t)s->ncol;
    if (tau) {
        CU(cudaMemcpyAsync(s->d_tau, tau, n * s->dc.nwvl * NLAY * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    } else if (!s->tau_valid) {
        return fail(s, RCM_ERR_STATE, "no tau: pass one or call rcm_build_tau first");
    }
    st = launch(s, MODE_RT, 1, false);
    if (st != RCM_OK) return st;
    if (E_down) CU(cudaMemcpyAsync(E_down, s->d_Ed, n * NLEV * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (E_up) CU(cudaMemcpyAsync(E_up, s->d_Eu, n * NLEV * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (dE) CU(cudaMemcpyAsync(dE, s->d_dE, n * NLAY * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    return RCM_OK;
}

// The LBL kernels' arguments for ncol columns: sizes, species slots and tables; the state pointers are the caller's.
static LblArgs lbl_args(const rcm_solver* s, int ncol) {
    LblArgs a{};
    a.ncol = ncol;
    a.ntiles = (ncol + RCM_LBL_C - 1) / RCM_LBL_C;
    a.nwvl = s->lbl_nwvl;
    // (tile, wavelength chunk) CTAs with a FIXED chunk of 128 wavelengths (32 rounds of the 4 wavelength groups): the
    // order of the spectral sum - registers over a chunk's rounds, groups, chunks - does not depend on how many columns
    // this GPU owns (a shard of an ensemble is bit-identical to the same columns inside the whole), and 4,096 columns x
    // 20,000 wavelengths are 40,192 units for the hardware scheduler to balance instead of 1,792 (4.04 rounds of 444)
    a.chunk_len = 128;
    a.nchunks = (a.nwvl + a.chunk_len - 1) / a.chunk_len;
    a.nact = s->nactive;
    a.h2o_slot = s->h2o_slot;
    a.o3_slot = -1;
    for (int k = 0; k < s->nactive; ++k)
        if (s->species[k] == 2) a.o3_slot = k;
    a.co2_factor = s->lbl_co2_factor;
    a.clampk = s->clampk;
    a.tau_clamp = s->tau_clamp;
    a.wvl_lo = s->d_lbl_lo;
    a.wvl_hi = s->d_lbl_hi;
    a.wn_hi = s->d_lbl_lo + (size_t)s->lbl_nwvl;
    a.wn_lo = s->d_lbl_lo + 2 * (size_t)s->lbl_nwvl;
    a.bin_ok = reinterpret_cast<const int*>(s->d_lbl_lo + 3 * (size_t)s->lbl_nwvl);
    a.tau3 = s->d_lbl_tau5;
    a.h2o_ref = s->d_lbl_h2o_ref;
    a.o3_ref = s->lbl_has_o3_ref ? s->d_lbl_o3_ref : nullptr;
    a.exp_tab = s->d_exp_tab;
    return a;
}

static int lbl_advance(rcm_solver* s, int nsteps) {
    if (s->h2o_slot < 0) return fail(s, RCM_ERR_STATE, "the LBL path needs H2O in species_mask");
    int st = refresh_const(s);
    if (st != RCM_OK) return st;
    const size_t n = (size_t)s->ncol;
    if (!s->d_sH || s->part_cap == 0) {
        CU(dalloc(s->d_sH, (size_t)s->cap * NLAY));
        CU(dalloc(s->d_sO, (size_t)s->cap * NLAY));
        CU(dalloc(s->d_dTstat, (size_t)s->cap));
    }
    LblArgs a = lbl_args(s, s->ncol);
    const size_t need = (size_t)a.nchunks * n * 42;
    if (need > s->part_cap) {
        CU(dalloc(s->d_part, need));
        s->part_cap = need;
    }
    a.Tlayer = s->d_T; a.Tsurf = s->d_Ts; a.vmr = s->d_vmr; a.rel_hum = s->d_rh; a.Tprev = s->d_Tprev;
    a.time_h = s->d_time; a.sH = s->d_sH; a.sO = s->d_sO; a.dTstat = s->d_dTstat; a.part = s->d_part;
    a.E_down = s->d_Ed; a.E_up = s->d_Eu; a.dE = s->d_dE; a.dt = s->d_dt;
    a.solar_col = s->has_col_solar ? s->d_solar_col : nullptr;
    a.cloud_col = s->has_col_cloud ? s->d_cloud_col : nullptr;
    for (int k = 0; k < nsteps; ++k) {
        a.step_index = s->step_index + k;
        a.diag = s->d_diag + (size_t)k * s->ncol * 4;
        std::pair<cudaEvent_t, cudaEvent_t> ev{};
        if (!s->ev_free.empty()) {
            ev = s->ev_free.back();
            s->ev_free.pop_back();
        } else {
            CU(cudaEventCreate(&ev.first));
            CU(cudaEventCreate(&ev.second));
        }
        CU(rcm_launch_lbl_step(a, s->stream, ev.first, ev.second));
        s->ev_used.push_back(ev);
        if (s->ev_used.size() >= 1024) {
            st = rcm_kernel_time_ms(s, 0, nullptr, nullptr);
            if (st != RCM_OK) return st;
        }
        s->launches += 3;
    }
    return RCM_OK;
}

int rcm_advance_async(rcm_solver* s, int nsteps, double** d_scalars) {
    if (!s || nsteps <= 0) return RCM_ERR_ARG;
    if ((!s->has_table && !s->lbl_mode) || s->ncol <= 0) return fail(s, RCM_ERR_STATE, "table and columns must be loaded");
    CU(cudaSetDevice(s->device));
    int st = ensure_diag(s, nsteps);
    if (st != RCM_OK) return st;
    if (s->lbl_mode) {
        st = lbl_advance(s, nsteps);
        if (st != RCM_OK) return st;
        CU(rcm_launch_reduce_diag(s->d_diag, nsteps, s->ncol, s->p.dT_converged, s->d_red, s->d_ticket, s->d_scalars, s->stream));
        s->launches += 1;
        s->step_index += nsteps;
        if (d_scalars) *d_scalars = s->d_scalars;
        return RCM_OK;
    }
    st = use_split(s) ? split_advance(s, nsteps) : launch(s, MODE_STEP, nsteps, true);
    if (st != RCM_OK) return st;
    CU(rcm_launch_reduce_diag(s->d_diag, nsteps, s->ncol, s->p.dT_converged, s->d_red, s->d_ticket, s->d_scalars, s->stream));
    s->launches += 1;
    s->step_index += nsteps;
    s->tau_valid = false;
    if (d_scalars) *d_scalars = s->d_scalars;
    return RCM_OK;
}

int rcm_advance(rcm_solver* s, int nsteps, rcm_step_scalars* scalars_out) {
    int st = rcm_advance_async(s, nsteps, nullptr);
    if (st != RCM_OK) return st;
    if (scalars_out) {
        CU(cudaMemcpyAsync(scalars_out, s->d_scalars, (size_t)nsteps * sizeof(rcm_step_scalars), cudaMemcpyDeviceToHost,
                           s->stream));
        CU(cudaStreamSynchronize(s->stream));
    }
    return RCM_OK;
}

int rcm_run_to_equilibrium(rcm_solver* s, long max_steps, int check_every, rcm_step_scalars* last, long* steps_done) {
    if (!s || max_steps <= 0 || check_every <= 0) return RCM_ERR_ARG;
    if (steps_done) *steps_done = 0;
    std::vector<rcm_step_scalars> sc((size_t)check_every);
    long done = 0;
    while (done < max_steps) {
        const int n = (int)std::min<long>(check_every, max_steps - done);
        const int st = rcm_advance(s, n, sc.data());
        if (st != RCM_OK) return st;
        done += n;
        if (last) *last = sc[n - 1];
        if (steps_done) *steps_done = done;
        if (sc[n - 1].n_converged >= (double)s->ncol) break;
    }
    return RCM_OK;
}

int rcm_get_state(rcm_solver* s, double* Tlayer, double* Tsurf, double* h2o, float* time_h, double* E_down,
                  double* E_up, double* dE, double* dt) {
    if (!s) return RCM_ERR_ARG;
    if (s->ncol <= 0) return fail(s, RCM_ERR_STATE, "no columns loaded");
    CU(cudaSetDevice(s->device));
    const size_t n = (size_t)s->ncol;
    if (Tlayer) CU(cudaMemcpyAsync(Tlayer, s->d_T, n * NLAY * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (Tsurf) CU(cudaMemcpyAsync(Tsurf, s->d_Ts, n * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (time_h) CU(cudaMemcpyAsync(time_h, s->d_time, n * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    if (E_down) CU(cudaMemcpyAsync(E_down, s->d_Ed, n * NLEV * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (E_up) CU(cudaMemcpyAsync(E_up, s->d_Eu, n * NLEV * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (dE) CU(cudaMemcpyAsync(dE, s->d_dE, n * NLAY * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (dt) CU(cudaMemcpyAsync(dt, s->d_dt, n * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (h2o) {
        if (s->h2o_slot < 0) return fail(s, RCM_ERR_STATE, "H2O is not an active species");
        CU(cudaMemcpy2DAsync(h2o, NLAY * sizeof(double), s->d_vmr + (size_t)s->h2o_slot * NLAY,
                             (size_t)s->nactive * NLAY * sizeof(double), NLAY * sizeof(double), n, cudaMemcpyDeviceToHost,
                             s->stream));
    }
    CU(cudaStreamSynchronize(s->stream));
    return RCM_OK;
}

// ------------------------------------------------------------------------------------------
// Diagnostic calls (rcm_diagnose_fluxes, rcm_radiative_kernels, rcm_flux_jacobian, rcm_adjusted_forcing).  The split path's
// prep kernel - the sort, the water-vapour feedback and the table indices of the next step - runs on COPIES of a chunk's T,
// previous profile and VMRs and writes its tile blocks into a scratch buffer; the solver's state, its tile blocks and every
// flag stay as they are.  Chunks of at most 8,192 columns alternate between two streams with a scratch set each (about 0.6 GB
// with 100 wavelengths for the fluxes, 1.1 GB for the radiative kernels, 0.4 GB for the flux Jacobians, whatever the
// wavelengths): the memory-bound sum kernel and the copies of one chunk overlap the radiative transfer of the next, and the
// last round of one chunk's units the first of the next.
// ------------------------------------------------------------------------------------------
extern "C++" {  // (templates)
namespace {

constexpr int kDiagMaxChunk = 8192;

// columns per chunk: whole tiles of 16, at most kDiagMaxChunk
size_t diag_chunk(int ncol) { return (size_t)std::min(kDiagMaxChunk, (ncol + 15) / 16 * 16); }

// the range [col0, col0 + ncol) inside the loaded columns; the factors of vmr_scale (NULL = all 1) into sc
int diag_range(rcm_solver* s, const std::string& fn, int col0, int ncol, const double* vmr_scale, DiagScale& sc) {
    if (col0 < 0 || ncol <= 0 || (long long)col0 + ncol > s->ncol)
        return fail(s, RCM_ERR_ARG, fn + ": columns [" + std::to_string(col0) + ", " + std::to_string((long long)col0 + ncol) +
                                        ") outside the " + std::to_string(s->ncol) + " loaded");
    for (int k = 0; k < 5; ++k) {
        sc.f[k] = vmr_scale ? vmr_scale[k] : 1.0;
        if (!(sc.f[k] >= 0.0) || !std::isfinite(sc.f[k]))
            return fail(s, RCM_ERR_ARG, fn + ": vmr_scale[" + std::to_string(k) + "] must be finite and >= 0");
    }
    return RCM_OK;
}

// the checks every repwvl call makes, then diag_range
int diag_check(rcm_solver* s, const std::string& fn, int col0, int ncol, const double* vmr_scale, DiagScale& sc) {
    if (s->lbl_mode) return fail(s, RCM_ERR_STATE, fn + ": the line-by-line path is not supported");
    if (!s->has_table) return fail(s, RCM_ERR_STATE, fn + ": no lookup table loaded");
    if (s->ncol <= 0) return fail(s, RCM_ERR_STATE, fn + ": no columns loaded");
    if (s->nactive != 5) return fail(s, RCM_ERR_STATE, fn + ": needs the five active species of the default species_mask");
    if (!use_split(s)) return fail(s, RCM_ERR_STATE, fn + ": needs the split path (RCM_OPT_PATH 0, no forced tile shape)");
    return diag_range(s, fn, col0, ncol, vmr_scale, sc);
}

// A chunk's copies of what the prep reads - T, Tprev [ch][20], VMRs [ch][5][20] - its stationarity diagnostic stat [ch]
// (unused), and the tile blocks it writes: the front and the end of every scratch set.
struct DiagState {
    double *T, *Tprev, *vmr, *stat;
    unsigned char* tile;
};

// Hands out a scratch set front to back (doubles first, then ints).  On a null base it only counts.
struct DiagCarve {
    unsigned char* base;
    size_t off = 0;
    template <class T>
    T* take(size_t n) {
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += n * sizeof(T);
        return p;
    }
};

// The device, its constants, two scratch sets for chunks of ch columns and the two streams; work queued on the solver's stream
// comes first.  A set is the state copies, what layout(m, ch, z) takes for the call's own arrays, then the tile blocks at a
// 256-byte boundary (none without tiles: the line-by-line path has none).  The description runs once on a null base for the
// size of a set, then once on each set: the size and the pointers cannot disagree.
template <class Set, class Layout>
int diag_begin(rcm_solver* s, size_t ch, Set (&set)[2], Layout layout, bool tiles = true) {
    CU(cudaSetDevice(s->device));
    const int st = refresh_const(s);
    if (st != RCM_OK) return st;
    auto carve = [&](unsigned char* base, Set& z) {
        DiagCarve m{base};
        z.state.T = m.take<double>(ch * NLAY);
        z.state.Tprev = m.take<double>(ch * NLAY);
        z.state.vmr = m.take<double>(ch * s->nactive * NLAY);
        z.state.stat = m.take<double>(ch);
        layout(m, ch, z);
        m.off = (m.off + 255) / 256 * 256;
        z.state.tile = m.take<unsigned char>(tiles ? ch / 16 * rcm_split_tile_bytes() : 0);
        return (m.off + 255) / 256 * 256;
    };
    Set sized{};
    const size_t set_bytes = carve(nullptr, sized);
    if (2 * set_bytes > s->diagnose_bytes) {
        CU(dalloc(s->d_diagnose, 2 * set_bytes));
        s->diagnose_bytes = 2 * set_bytes;
    }
    for (int k = 0; k < 2; ++k) carve(s->d_diagnose + k * set_bytes, set[k]);
    if (!s->dg_fork) {
        for (int i = 0; i < 2; ++i) {
            CU(cudaStreamCreateWithFlags(&s->dg_stream[i], cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&s->dg_join[i], cudaEventDisableTiming));
        }
        CU(cudaEventCreateWithFlags(&s->dg_fork, cudaEventDisableTiming));
    }
    CU(cudaEventRecord(s->dg_fork, s->stream));
    for (int i = 0; i < 2; ++i) CU(cudaStreamWaitEvent(s->dg_stream[i], s->dg_fork, 0));
    return RCM_OK;
}

// Copies of columns [c0, c0 + n) into d and the prep of the next step on them, tile blocks into d.tile, then the VMR factors
// (sc: NULL = unscaled).  On return d.T holds the sorted profile the step radiates with; a carries the chunk's unit plan.
int diag_prep(rcm_solver* s, cudaStream_t q, int c0, int n, const DiagState& d, const DiagScale* sc, SplitArgs& a) {
    constexpr size_t D = sizeof(double);
    const size_t o = (size_t)c0;
    const int na = s->nactive;
    CU(cudaMemcpyAsync(d.T, s->d_T + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToDevice, q));
    CU(cudaMemcpyAsync(d.Tprev, s->d_Tprev + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToDevice, q));
    CU(cudaMemcpyAsync(d.vmr, s->d_vmr + o * na * NLAY, (size_t)n * na * NLAY * D, cudaMemcpyDeviceToDevice, q));
    a = split_args(s, c0, n, 0);
    a.Tlayer = d.T;
    a.Tprev = d.Tprev;
    a.vmr = d.vmr;
    a.dTstat = d.stat;
    a.tile = d.tile;
    a.counter = nullptr;
    a.part = nullptr;
    a.diag = nullptr;
    a.E_down = a.E_up = a.dE = a.dt = nullptr;
    a.time_h = nullptr;
    SplitColFlags f{};
    f.prep = 1;
    f.first = (s->step_index == 0);
    f.write_all_vmr = 1;
    CU(rcm_launch_split_col(a, f, q));
    if (sc) CU(rcm_launch_diag_scale(d.tile, a.ntiles, *sc, q));
    s->launches += sc ? 2 : 1;
    return RCM_OK;
}

// the solver's stream waits for both streams; then the host waits
int diag_end(rcm_solver* s) {
    for (int i = 0; i < 2; ++i) {
        CU(cudaEventRecord(s->dg_join[i], s->dg_stream[i]));
        CU(cudaStreamWaitEvent(s->stream, s->dg_join[i], 0));
    }
    CU(cudaStreamSynchronize(s->stream));
    return RCM_OK;
}

// what DiagArgs, JacArgs and FjacArgs take from the prep's arguments a: the chunk, the table, the clamp, the tile blocks
template <class A>
A diag_args(const SplitArgs& a) {
    A g{};
    g.ncol = a.ncol;
    g.clampk = a.clampk;
    g.tau_clamp = a.tau_clamp;
    g.coef = a.coef;
    g.planck_c = a.planck_c;
    g.planck_k = a.planck_k;
    g.exp_tab = a.exp_tab;
    g.tile = a.tile;
    return g;
}

// and the (tile, split) units of DiagArgs and JacArgs
template <class A>
A unit_args(const SplitArgs& a) {
    A g = diag_args<A>(a);
    g.ntiles = a.ntiles;
    g.nsplit = a.nsplit;
    g.ipu = a.ipu;
    g.nitem = a.nitem;
    g.nunits = a.nunits;
    return g;
}

// rcm_diag_rt_kernel + rcm_diag_sum_kernel on the tile blocks of the prep a: the spectra dn, up and the broadband Ed, Eu, dE
int diag_fluxes(rcm_solver* s, const SplitArgs& a, cudaStream_t q, double* dn, double* up, double* Ed, double* Eu, double* dE) {
    DiagArgs g = unit_args<DiagArgs>(a);
    g.spec_dn = dn;
    g.spec_up = up;
    g.E_down = Ed;
    g.E_up = Eu;
    g.dE = dE;
    g.solar_col = a.solar_col;
    CU(rcm_launch_diag_rt(g, std::min(g.nunits, 3 * nsm_of(s)), q));
    CU(rcm_launch_diag_sum(g, q));
    s->launches += 2;
    return RCM_OK;
}

// rcm_fjac_kernel on the tile blocks of the prep a, the Planck source at T: J and dE_jac into J, H
int flux_jacobian(rcm_solver* s, const SplitArgs& a, cudaStream_t q, const double* T, double* J, double* H) {
    FjacArgs g = diag_args<FjacArgs>(a);
    g.T_floor = a.T_floor;
    g.wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    g.T = T;
    g.Ts = a.Tsurf;
    g.J = J;
    g.dE_jac = H;
    CU(rcm_launch_fjac(g, q));
    s->launches += 1;
    return RCM_OK;
}

// The chunks of a single-pass call, ch columns each.  Chunk k runs on stream k % 2 with scratch set k % 2 (chunk k + 2 reuses
// the set of chunk k after it on the same stream): prep(z, c0, n, q, a) for its columns [c0, c0 + n), then enqueue(z, a, q).
// Its downloads, download(z, r, n, q) for the output rows [r, r + n), are issued after the kernels of chunk k + 1: into
// pageable memory they block the host.
template <class Set, class Args, class Layout, class Prep, class Enqueue, class Download>
int chunk_loop(rcm_solver* s, int col0, int ncol, size_t ch, bool tiles, Layout layout, Prep prep, Enqueue enqueue,
               Download download) {
    Set set[2];
    int st = diag_begin(s, ch, set, layout, tiles);
    if (st != RCM_OK) return st;
    struct { const Set* z; size_t r; int n; cudaStream_t q; } pend{};
    for (int c0 = col0, k = 0; c0 < col0 + ncol; c0 += (int)ch, ++k) {
        const int n = std::min((int)ch, col0 + ncol - c0);
        const Set& z = set[k % 2];
        cudaStream_t q = s->dg_stream[k % 2];
        Args a;
        if ((st = prep(z, c0, n, q, a)) != RCM_OK) return st;
        if ((st = enqueue(z, a, q)) != RCM_OK) return st;
        if (k > 0 && (st = download(*pend.z, pend.r, pend.n, pend.q)) != RCM_OK) return st;
        pend = {&z, (size_t)(c0 - col0), n, q};
    }
    if ((st = download(*pend.z, pend.r, pend.n, pend.q)) != RCM_OK) return st;
    return diag_end(s);
}

// the repwvl calls: chunks of diag_chunk(ncol) columns, diag_prep (sc: VMR factors or NULL) in front of enqueue
template <class Set, class Layout, class Enqueue, class Download>
int diag_chunks(rcm_solver* s, int col0, int ncol, const DiagScale* sc, Layout layout, Enqueue enqueue, Download download) {
    auto prep = [&](const Set& z, int c0, int n, cudaStream_t q, SplitArgs& a) { return diag_prep(s, q, c0, n, z.state, sc, a); };
    return chunk_loop<Set, SplitArgs>(s, col0, ncol, diag_chunk(ncol), true, layout, prep, enqueue, download);
}

}  // namespace
}  // extern "C++"

int rcm_diagnose_fluxes(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* E_down_spec, double* E_up_spec,
                        double* E_down, double* E_up, double* dE) {
    if (!s) return RCM_ERR_ARG;
    DiagScale sc{};
    const int st = diag_check(s, "rcm_diagnose_fluxes", col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    const int nwvl = s->dc.nwvl;
    constexpr size_t D = sizeof(double);
    struct Set {
        DiagState state;
        double *Ed, *Eu, *dE, *spec_dn, *spec_up;
    };
    return diag_chunks<Set>(
        s, col0, ncol, vmr_scale ? &sc : nullptr,
        [&](DiagCarve& m, size_t ch, Set& z) {  // E_down, E_up [ch][21], dE [ch][20], spectral [2][ch][nwvl][21]
            z.Ed = m.take<double>(ch * NLEV);
            z.Eu = m.take<double>(ch * NLEV);
            z.dE = m.take<double>(ch * NLAY);
            z.spec_dn = m.take<double>(ch * nwvl * NLEV);
            z.spec_up = m.take<double>(ch * nwvl * NLEV);
        },
        [&](const Set& z, const SplitArgs& a, cudaStream_t q) {
            return diag_fluxes(s, a, q, z.spec_dn, z.spec_up, z.Ed, z.Eu, z.dE);
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            const size_t nspec = (size_t)n * nwvl * NLEV;
            if (E_down_spec) CU(cudaMemcpyAsync(E_down_spec + r * nwvl * NLEV, z.spec_dn, nspec * D, cudaMemcpyDeviceToHost, q));
            if (E_up_spec) CU(cudaMemcpyAsync(E_up_spec + r * nwvl * NLEV, z.spec_up, nspec * D, cudaMemcpyDeviceToHost, q));
            if (E_down) CU(cudaMemcpyAsync(E_down + r * NLEV, z.Ed, n * NLEV * D, cudaMemcpyDeviceToHost, q));
            if (E_up) CU(cudaMemcpyAsync(E_up + r * NLEV, z.Eu, n * NLEV * D, cudaMemcpyDeviceToHost, q));
            if (dE) CU(cudaMemcpyAsync(dE + r * NLAY, z.dE, n * NLAY * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// Radiative kernels: rcm_jac_rt_kernel per (column, wavelength), rcm_jac_sum_kernel for the sum over the wavelengths.
int rcm_radiative_kernels(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* K_spec, double* K) {
    if (!s) return RCM_ERR_ARG;
    DiagScale sc{};
    const int st = diag_check(s, "rcm_radiative_kernels", col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->h2o_slot != 0) return fail(s, RCM_ERR_STATE, "rcm_radiative_kernels: needs H2O among the active species");
    const int nwvl = s->dc.nwvl;
    constexpr size_t D = sizeof(double);
    struct Set {
        DiagState state;
        double *K, *K_spec;
    };
    return diag_chunks<Set>(
        s, col0, ncol, vmr_scale ? &sc : nullptr,
        [&](DiagCarve& m, size_t ch, Set& z) {  // K [ch][82], K_spec [ch][nwvl][82]
            z.K = m.take<double>(ch * JAC_NK);
            z.K_spec = m.take<double>(ch * nwvl * JAC_NK);
        },
        [&](const Set& z, const SplitArgs& a, cudaStream_t q) -> int {
            JacArgs g = unit_args<JacArgs>(a);
            g.T_floor = a.T_floor;
            g.wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
            g.T = a.Tlayer;
            g.Ts = a.Tsurf;
            g.K_spec = z.K_spec;
            g.K = z.K;
            CU(rcm_launch_jac_rt(g, std::min(g.nunits, rcm_jac_ctas_per_sm() * nsm_of(s)), q));
            CU(rcm_launch_jac_sum(g, q));
            s->launches += 2;
            return RCM_OK;
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            if (K_spec) CU(cudaMemcpyAsync(K_spec + r * nwvl * JAC_NK, z.K_spec, (size_t)n * nwvl * JAC_NK * D, cudaMemcpyDeviceToHost, q));
            if (K) CU(cudaMemcpyAsync(K + r * JAC_NK, z.K, (size_t)n * JAC_NK * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// Flux Jacobians: rcm_fjac_kernel sums over the wavelengths itself, one warp per column.
int rcm_flux_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac) {
    if (!s) return RCM_ERR_ARG;
    DiagScale sc{};
    const int st = diag_check(s, "rcm_flux_jacobian", col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->h2o_slot != 0) return fail(s, RCM_ERR_STATE, "rcm_flux_jacobian: needs H2O among the active species");
    constexpr size_t D = sizeof(double);
    struct Set {
        DiagState state;
        double *J, *H;
    };
    return diag_chunks<Set>(
        s, col0, ncol, vmr_scale ? &sc : nullptr,
        [&](DiagCarve& m, size_t ch, Set& z) {  // J [ch][2][21][41], dE_jac [ch][20][41]
            z.J = m.take<double>(ch * FJAC_NJ);
            z.H = m.take<double>(ch * FJAC_NH);
        },
        [&](const Set& z, const SplitArgs& a, cudaStream_t q) { return flux_jacobian(s, a, q, a.Tlayer, z.J, z.H); },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            if (J) CU(cudaMemcpyAsync(J + r * FJAC_NJ, z.J, (size_t)n * FJAC_NJ * D, cudaMemcpyDeviceToHost, q));
            if (dE_jac) CU(cudaMemcpyAsync(dE_jac + r * FJAC_NH, z.H, (size_t)n * FJAC_NH * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// the species of the entries of both species-Jacobian calls, in the order of vmr_scale: H2O, CO2, O3, N2O, CH4
constexpr unsigned kSpeciesMask = 0x2F;

// Species Jacobians: the flux Jacobian's chunks, prep and layout, rcm_species_fjac_kernel in place of rcm_fjac_kernel.
int rcm_species_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac) {
    if (!s) return RCM_ERR_ARG;
    DiagScale sc{};
    const int st = diag_check(s, "rcm_species_jacobian", col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->p.species_mask != kSpeciesMask)
        return fail(s, RCM_ERR_STATE, "rcm_species_jacobian: needs the default species_mask (H2O, CO2, O3, N2O, CH4)");
    if (!J && !dE_jac) return RCM_OK;
    constexpr size_t D = sizeof(double);
    struct Set {
        DiagState state;
        double *J, *H;
    };
    return diag_chunks<Set>(
        s, col0, ncol, vmr_scale ? &sc : nullptr,
        [&](DiagCarve& m, size_t ch, Set& z) {  // J [ch][2][21][100], dE_jac [ch][20][100]
            z.J = m.take<double>(ch * SPJ_NJ);
            z.H = m.take<double>(ch * SPJ_NH);
        },
        [&](const Set& z, const SplitArgs& a, cudaStream_t q) -> int {
            SpjacArgs g = diag_args<SpjacArgs>(a);
            g.wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
            g.J = z.J;
            g.dE_jac = z.H;
            CU(rcm_launch_species_fjac(g, q));
            s->launches += 1;
            return RCM_OK;
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            if (J) CU(cudaMemcpyAsync(J + r * SPJ_NJ, z.J, (size_t)n * SPJ_NJ * D, cudaMemcpyDeviceToHost, q));
            if (dE_jac) CU(cudaMemcpyAsync(dE_jac + r * SPJ_NH, z.H, (size_t)n * SPJ_NH * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// ------------------------------------------------------------------------------------------
// Line-by-line calls (rcm_lbl_diagnose_fluxes, rcm_lbl_radiative_kernels): the step's prep kernel on copies of a chunk's T,
// previous profile, VMRs and T_surf, then the species factors; the state stays as it is.
// ------------------------------------------------------------------------------------------
constexpr double kLblStageBytes = 2e9;  // per scratch set: a chunk's per-wavelength staging (band fluxes, kernels)

extern "C++" {
namespace {

// the checks every LBL call makes, then diag_range
int lbl_check(rcm_solver* s, const std::string& fn, int col0, int ncol, const double* vmr_scale, DiagScale& sc) {
    if (!s->lbl_mode) return fail(s, RCM_ERR_STATE, fn + ": needs the line-by-line path (rcm_set_lbl_tables)");
    if (s->ncol <= 0) return fail(s, RCM_ERR_STATE, fn + ": no columns loaded");
    if (s->nactive != 5) return fail(s, RCM_ERR_STATE, fn + ": needs the five active species of the default species_mask");
    return diag_range(s, fn, col0, ncol, vmr_scale, sc);
}

// band_start [nband + 1]: 0 = b_0 < b_1 < ... < b_nband = nwvl
int lbl_band_check(rcm_solver* s, const std::string& fn, int nband, const int* band_start) {
    if (nband < 1 || !band_start) return fail(s, RCM_ERR_ARG, fn + ": band outputs need nband >= 1 and band_start");
    for (int b = 0; b < nband; ++b)
        if (!(band_start[b] < band_start[b + 1]))
            return fail(s, RCM_ERR_ARG, fn + ": band_start must be strictly increasing (entry " + std::to_string(b + 1) + ")");
    if (band_start[0] != 0 || band_start[nband] != s->lbl_nwvl)
        return fail(s, RCM_ERR_ARG, fn + ": band_start must run from 0 to nwvl = " + std::to_string(s->lbl_nwvl));
    return RCM_OK;
}

// The planes the chunks radiate with into tau3: NULL (the tables' own) unless CO2, CH4 or N2O is scaled; then the
// column-independent plane composed anew on the solver's stream, the H2O and O3 planes copied next to it.
int lbl_planes(rcm_solver* s, const DiagScale& sc, const double*& tau3) {
    constexpr size_t D = sizeof(double);
    tau3 = nullptr;
    CU(cudaSetDevice(s->device));
    if (sc.f[1] == 1.0 && sc.f[3] == 1.0 && sc.f[4] == 1.0) return RCM_OK;
    const size_t plane = (size_t)s->lbl_nwvl * NLAY;
    if (s->tau3s_cap < 3 * plane) {
        CU(dalloc(s->d_lbl_tau3s, 3 * plane));
        s->tau3s_cap = 3 * plane;
    }
    CU(cudaMemcpyAsync(s->d_lbl_tau3s, s->d_lbl_tau5, 2 * plane * D, cudaMemcpyDeviceToDevice, s->stream));
    CU(rcm_launch_lbl_plane(s->d_lbl_tau5 + 3 * plane, plane, sc.f[1] * s->lbl_co2_factor, sc.f[4], sc.f[3],
                            s->d_lbl_tau3s + 2 * plane, s->stream));
    s->launches += 1;
    tau3 = s->d_lbl_tau3s;
    return RCM_OK;
}

// What the LBL prep reads and writes besides DiagState: T_surf [ch], sH, sO [ch][20].
struct LblState {
    double *Ts, *sH, *sO;
};

void lbl_take(DiagCarve& m, size_t ch, LblState& l) {
    l.Ts = m.take<double>(ch);
    l.sH = m.take<double>(ch * NLAY);
    l.sO = m.take<double>(ch * NLAY);
}

// Copies of columns [c0, c0 + n) into d and l, the prep of the next step on them, then the H2O and O3 factors (sc: NULL =
// unscaled).  On return l.sH / l.sO and d.T hold what the step radiates with; a carries the chunk's sizes, tables (tau3:
// NULL = the tables' own planes) and the prepared copies.
int lbl_prep(rcm_solver* s, cudaStream_t q, int c0, int n, const DiagState& d, const LblState& l, const double* tau3,
             const DiagScale* sc, LblArgs& a) {
    constexpr size_t D = sizeof(double);
    const size_t o = (size_t)c0;
    CU(cudaMemcpyAsync(d.T, s->d_T + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToDevice, q));
    CU(cudaMemcpyAsync(d.Tprev, s->d_Tprev + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToDevice, q));
    CU(cudaMemcpyAsync(d.vmr, s->d_vmr + o * 5 * NLAY, (size_t)n * 5 * NLAY * D, cudaMemcpyDeviceToDevice, q));
    CU(cudaMemcpyAsync(l.Ts, s->d_Ts + o, n * D, cudaMemcpyDeviceToDevice, q));
    a = lbl_args(s, n);
    a.step_index = s->step_index;
    if (tau3) a.tau3 = tau3;
    a.Tlayer = d.T; a.Tprev = d.Tprev; a.vmr = d.vmr; a.rel_hum = s->d_rh + o * NLAY;
    a.Tsurf = l.Ts; a.sH = l.sH; a.sO = l.sO; a.dTstat = d.stat; a.diag = nullptr;
    a.solar_col = s->has_col_solar ? s->d_solar_col + o : nullptr;
    a.cloud_col = s->has_col_cloud ? s->d_cloud_col + o : nullptr;
    CU(rcm_launch_lbl_prep(a, q));
    if (sc) CU(rcm_launch_lbl_scale(a, sc->f[0], sc->f[2], q));
    s->launches += sc ? 2 : 1;
    return RCM_OK;
}

// columns per chunk of a call that stages row_doubles per (column, wavelength): diag_chunk(ncol), and at most kLblStageBytes of
// staging rounded down to whole tiles, at least one tile
size_t lbl_stage_chunk(const rcm_solver* s, int ncol, size_t row_doubles) {
    const size_t fit = (size_t)(kLblStageBytes / ((double)s->lbl_nwvl * row_doubles * sizeof(double))) / 16 * 16;
    return std::min(diag_chunk(ncol), std::max<size_t>(16, fit));
}

}  // namespace
}  // extern "C++"

// Line-by-line fluxes: the step's three kernels on copies of a chunk (prep, the species factors, rt, finish into scratch), and
// for bands rcm_lbl_band_kernel + rcm_lbl_band_sum_kernel on the same prepared copies, in front of the finish (which moves T).
int rcm_lbl_diagnose_fluxes(rcm_solver* s, int col0, int ncol, const double* vmr_scale, int nband, const int* band_start,
                            double* E_down_band, double* E_up_band, double* E_down, double* E_up, double* dE) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_lbl_diagnose_fluxes";
    DiagScale sc{};
    int st = lbl_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    const int nwvl = s->lbl_nwvl;
    const bool bands = E_down_band || E_up_band, broad = E_down || E_up || dE;
    if (bands && (st = lbl_band_check(s, fn, nband, band_start)) != RCM_OK) return st;
    if (!bands && !broad) return RCM_OK;
    constexpr size_t D = sizeof(double);
    const double* tau3 = nullptr;
    if ((st = lbl_planes(s, sc, tau3)) != RCM_OK) return st;
    const size_t ch = bands ? lbl_stage_chunk(s, ncol, 2 * NLEV) : diag_chunk(ncol);
    const size_t nchunks = (size_t)lbl_args(s, 0).nchunks;
    struct Set {
        DiagState state;
        LblState lbl;
        double *dt, *part, *Ed, *Eu, *dE, *spec_dn, *spec_up, *band_dn, *band_up;
        float* time;
        int* bstart;
    };
    return chunk_loop<Set, LblArgs>(
        s, col0, ncol, ch, false,
        [&](DiagCarve& m, size_t ch, Set& z) {
            lbl_take(m, ch, z.lbl);
            z.dt = m.take<double>(ch);
            z.part = m.take<double>(broad ? nchunks * ch * 2 * NLEV : 0);
            z.Ed = m.take<double>(ch * NLEV);
            z.Eu = m.take<double>(ch * NLEV);
            z.dE = m.take<double>(ch * NLAY);
            z.spec_dn = m.take<double>(bands ? ch * nwvl * NLEV : 0);
            z.spec_up = m.take<double>(bands ? ch * nwvl * NLEV : 0);
            z.band_dn = m.take<double>(bands ? ch * nband * NLEV : 0);
            z.band_up = m.take<double>(bands ? ch * nband * NLEV : 0);
            z.time = m.take<float>(ch);
            z.bstart = m.take<int>(bands ? nband + 1 : 0);
        },
        [&](const Set& z, int c0, int n, cudaStream_t q, LblArgs& a) -> int {
            if (bands) CU(cudaMemcpyAsync(z.bstart, band_start, (nband + 1) * sizeof(int), cudaMemcpyHostToDevice, q));
            const int r = lbl_prep(s, q, c0, n, z.state, z.lbl, tau3, vmr_scale ? &sc : nullptr, a);
            a.time_h = z.time; a.part = z.part; a.E_down = z.Ed; a.E_up = z.Eu; a.dE = z.dE; a.dt = z.dt;
            return r;
        },
        [&](const Set& z, const LblArgs& a, cudaStream_t q) -> int {
            if (bands) {
                CU(rcm_launch_lbl_band(a, z.spec_dn, z.spec_up, q));
                CU(rcm_launch_lbl_band_sum(a.ncol, nwvl, nband, z.bstart, z.spec_dn, z.spec_up, z.band_dn, z.band_up, q));
                s->launches += 2;
            }
            if (broad) {
                CU(rcm_launch_lbl_rt(a, q, nullptr, nullptr));
                CU(rcm_launch_lbl_finish(a, q));
                s->launches += 2;
            }
            return RCM_OK;
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            const size_t nb = (size_t)n * nband * NLEV;
            if (E_down_band) CU(cudaMemcpyAsync(E_down_band + r * nband * NLEV, z.band_dn, nb * D, cudaMemcpyDeviceToHost, q));
            if (E_up_band) CU(cudaMemcpyAsync(E_up_band + r * nband * NLEV, z.band_up, nb * D, cudaMemcpyDeviceToHost, q));
            if (E_down) CU(cudaMemcpyAsync(E_down + r * NLEV, z.Ed, n * NLEV * D, cudaMemcpyDeviceToHost, q));
            if (E_up) CU(cudaMemcpyAsync(E_up + r * NLEV, z.Eu, n * NLEV * D, cudaMemcpyDeviceToHost, q));
            if (dE) CU(cudaMemcpyAsync(dE + r * NLAY, z.dE, n * NLAY * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// Line-by-line radiative kernels: per chunk the prep of the fluxes call, then rcm_lbl_jac_kernel into the staging K_spec and
// rcm_lbl_jac_band_sum_kernel for the bands and for the one band {0, nwvl} of K.  No finish kernel: nothing here moves T.
int rcm_lbl_radiative_kernels(rcm_solver* s, int col0, int ncol, const double* vmr_scale, int nband, const int* band_start,
                              double* K_band, double* K) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_lbl_radiative_kernels";
    DiagScale sc{};
    int st = lbl_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    const int nwvl = s->lbl_nwvl;
    if (K_band && (st = lbl_band_check(s, fn, nband, band_start)) != RCM_OK) return st;
    if (!K_band && !K) return RCM_OK;
    constexpr size_t D = sizeof(double);
    const double* tau3 = nullptr;
    if ((st = lbl_planes(s, sc, tau3)) != RCM_OK) return st;
    const int nb = K_band ? nband : 0;
    const int whole[2] = {0, nwvl};
    const double wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    struct Set {
        DiagState state;
        LblState lbl;
        double *K_spec, *K, *K_band;
        int *whole, *bstart;
    };
    return chunk_loop<Set, LblArgs>(
        s, col0, ncol, lbl_stage_chunk(s, ncol, JAC_NK), false,
        [&](DiagCarve& m, size_t ch, Set& z) {  // K_spec [ch][nwvl][82], K [ch][82], K_band [ch][nband][82]
            lbl_take(m, ch, z.lbl);
            z.K_spec = m.take<double>(ch * nwvl * JAC_NK);
            z.K = m.take<double>(K ? ch * JAC_NK : 0);
            z.K_band = m.take<double>(ch * nb * JAC_NK);
            z.whole = m.take<int>(2);
            z.bstart = m.take<int>(K_band ? nb + 1 : 0);
        },
        [&](const Set& z, int c0, int n, cudaStream_t q, LblArgs& a) -> int {
            if (K) CU(cudaMemcpyAsync(z.whole, whole, sizeof(whole), cudaMemcpyHostToDevice, q));
            if (K_band) CU(cudaMemcpyAsync(z.bstart, band_start, (nb + 1) * sizeof(int), cudaMemcpyHostToDevice, q));
            return lbl_prep(s, q, c0, n, z.state, z.lbl, tau3, vmr_scale ? &sc : nullptr, a);
        },
        [&](const Set& z, const LblArgs& a, cudaStream_t q) -> int {
            CU(rcm_launch_lbl_jac(a, wtau, z.K_spec, q));
            s->launches += 1;
            if (K_band) {
                CU(rcm_launch_lbl_jac_band_sum(a.ncol, nwvl, nb, z.bstart, z.K_spec, z.K_band, q));
                s->launches += 1;
            }
            if (K) {
                CU(rcm_launch_lbl_jac_band_sum(a.ncol, nwvl, 1, z.whole, z.K_spec, z.K, q));
                s->launches += 1;
            }
            return RCM_OK;
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            if (K_band) CU(cudaMemcpyAsync(K_band + r * nb * JAC_NK, z.K_band, (size_t)n * nb * JAC_NK * D, cudaMemcpyDeviceToHost, q));
            if (K) CU(cudaMemcpyAsync(K + r * JAC_NK, z.K, (size_t)n * JAC_NK * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// Line-by-line flux Jacobians: per chunk the prep of the fluxes call, then rcm_lbl_fjac_kernel, which sums over the
// wavelengths itself, one warp per column.  No finish kernel: nothing here moves T.
int rcm_lbl_flux_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_lbl_flux_jacobian";
    DiagScale sc{};
    int st = lbl_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (!J && !dE_jac) return RCM_OK;
    constexpr size_t D = sizeof(double);
    const double* tau3 = nullptr;
    if ((st = lbl_planes(s, sc, tau3)) != RCM_OK) return st;
    const double wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    struct Set {
        DiagState state;
        LblState lbl;
        double *J, *H;
    };
    return chunk_loop<Set, LblArgs>(
        s, col0, ncol, diag_chunk(ncol), false,
        [&](DiagCarve& m, size_t ch, Set& z) {  // J [ch][2][21][41], dE_jac [ch][20][41]
            lbl_take(m, ch, z.lbl);
            z.J = m.take<double>(ch * FJAC_NJ);
            z.H = m.take<double>(ch * FJAC_NH);
        },
        [&](const Set& z, int c0, int n, cudaStream_t q, LblArgs& a) -> int {
            return lbl_prep(s, q, c0, n, z.state, z.lbl, tau3, vmr_scale ? &sc : nullptr, a);
        },
        [&](const Set& z, const LblArgs& a, cudaStream_t q) -> int {
            CU(rcm_launch_lbl_fjac(a, wtau, z.J, z.H, q));
            s->launches += 1;
            return RCM_OK;
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            if (J) CU(cudaMemcpyAsync(J + r * FJAC_NJ, z.J, (size_t)n * FJAC_NJ * D, cudaMemcpyDeviceToHost, q));
            if (dE_jac) CU(cudaMemcpyAsync(dE_jac + r * FJAC_NH, z.H, (size_t)n * FJAC_NH * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// Line-by-line species Jacobians: the LBL flux Jacobian's chunks and prep, rcm_lbl_species_fjac_kernel in place of
// rcm_lbl_fjac_kernel.  The CO2, CH4 and N2O shares come from the tables' raw planes with the factors lbl_planes composes with.
int rcm_lbl_species_jacobian(rcm_solver* s, int col0, int ncol, const double* vmr_scale, double* J, double* dE_jac) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_lbl_species_jacobian";
    DiagScale sc{};
    int st = lbl_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->p.species_mask != kSpeciesMask) return fail(s, RCM_ERR_STATE, fn + ": needs the default species_mask (H2O, CO2, O3, N2O, CH4)");
    if (!J && !dE_jac) return RCM_OK;
    constexpr size_t D = sizeof(double);
    const double* tau3 = nullptr;
    if ((st = lbl_planes(s, sc, tau3)) != RCM_OK) return st;
    const double wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    const double* raw = s->d_lbl_tau5 + 3 * (size_t)s->lbl_nwvl * NLAY;
    struct Set {
        DiagState state;
        LblState lbl;
        double *J, *H;
    };
    return chunk_loop<Set, LblArgs>(
        s, col0, ncol, diag_chunk(ncol), false,
        [&](DiagCarve& m, size_t ch, Set& z) {  // J [ch][2][21][100], dE_jac [ch][20][100]
            lbl_take(m, ch, z.lbl);
            z.J = m.take<double>(ch * SPJ_NJ);
            z.H = m.take<double>(ch * SPJ_NH);
        },
        [&](const Set& z, int c0, int n, cudaStream_t q, LblArgs& a) -> int {
            return lbl_prep(s, q, c0, n, z.state, z.lbl, tau3, vmr_scale ? &sc : nullptr, a);
        },
        [&](const Set& z, const LblArgs& a, cudaStream_t q) -> int {
            CU(rcm_launch_lbl_species_fjac(a, wtau, raw, sc.f[1] * s->lbl_co2_factor, sc.f[4], sc.f[3], z.J, z.H, q));
            s->launches += 1;
            return RCM_OK;
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            if (J) CU(cudaMemcpyAsync(J + r * SPJ_NJ, z.J, (size_t)n * SPJ_NJ * D, cudaMemcpyDeviceToHost, q));
            if (dE_jac) CU(cudaMemcpyAsync(dE_jac + r * SPJ_NH, z.H, (size_t)n * SPJ_NH * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// ------------------------------------------------------------------------------------------
// Flux gradients (rcm_flux_gradient, rcm_lbl_flux_gradient): the species Jacobians' chunks and prep, then one reverse sweep per
// (column, wavelength, angle) with the chunk's level cotangents, partial sums over fixed wavelength ranges, and their sum.
// ------------------------------------------------------------------------------------------
extern "C++" {
namespace {

// The level cotangents of the rows [0, ncol) into co [ncol][42] = {b_0..b_20, a_0..a_20}, w_dE folded in as the adjoint of dE
// from E (main.cpp:337-341: dE_l = Ed_l - Ed_{l+1} + Eu_{l+1} - Eu_l for l < 19, dE_19 = Ed_19 - Eu_19):
//   b_k = (w_Ed[k] + w_dE[k]) - w_dE[k-1],  a_k = (w_Eu[k] - w_dE[k]) + w_dE[k-1],  each term only where it exists.
// RCM_ERR_ARG for a non-finite entry; *any = false when all three are NULL.
int grad_fold(rcm_solver* s, const std::string& fn, int ncol, const double* wEd, const double* wEu, const double* wdE,
              std::vector<double>& co, bool* any) {
    *any = wEd || wEu || wdE;
    if (!*any) return RCM_OK;
    const struct { const double* p; size_t n; const char* name; } in[3] = {
        {wEd, (size_t)ncol * NLEV, "w_E_down"}, {wEu, (size_t)ncol * NLEV, "w_E_up"}, {wdE, (size_t)ncol * NLAY, "w_dE"}};
    for (const auto& v : in)
        if (v.p)
            for (size_t i = 0; i < v.n; ++i)
                if (!std::isfinite(v.p[i]))
                    return fail(s, RCM_ERR_ARG, fn + ": " + v.name + "[" + std::to_string(i / (v.n / ncol)) + "][" +
                                                    std::to_string(i % (v.n / ncol)) + "] is not finite");
    co.assign((size_t)ncol * GRAD_NCO, 0.0);
    for (int r = 0; r < ncol; ++r) {
        double* b = co.data() + (size_t)r * GRAD_NCO;
        double* a = b + NLEV;
        for (int k = 0; k < NLEV; ++k) {
            double bk = wEd ? wEd[(size_t)r * NLEV + k] : 0.0, ak = wEu ? wEu[(size_t)r * NLEV + k] : 0.0;
            if (wdE) {
                const double* w = wdE + (size_t)r * NLAY;
                if (k < NLAY) {
                    bk = bk + w[k];
                    ak = ak - w[k];
                }
                if (k >= 1 && k < NLAY) {
                    bk = bk - w[k - 1];
                    ak = ak + w[k - 1];
                }
            }
            b[k] = bk;
            a[k] = ak;
        }
    }
    return RCM_OK;
}

// rcm_grad_rt_kernel on the tile blocks and units of the prep a, the Planck source at T and Ts, with the level cotangents co:
// partials [ncol][nsplit][121] into part, then rcm_grad_sum_kernel over the splits into grad [ncol][121]
int grad_sweep(rcm_solver* s, const SplitArgs& a, cudaStream_t q, const double* T, const double* Ts, const double* co,
               double* part, double* grad) {
    GradArgs g = unit_args<GradArgs>(a);
    g.T_floor = a.T_floor;
    g.wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    g.T = T;
    g.Ts = Ts;
    g.co = co;
    g.part = part;
    CU(rcm_launch_grad_rt(g, std::min(g.nunits, rcm_grad_ctas_per_sm() * nsm_of(s)), q));
    CU(rcm_launch_grad_sum(g.ncol, g.nsplit, part, grad, q));
    s->launches += 2;
    return RCM_OK;
}

}  // namespace
}  // extern "C++"

// Flux gradients: rcm_grad_rt_kernel per (tile, split) unit into partials [ch][nsplit][121], rcm_grad_sum_kernel over the splits.
int rcm_flux_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const double* w_E_down, const double* w_E_up,
                      const double* w_dE, double* grad) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_flux_gradient";
    DiagScale sc{};
    int st = diag_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->p.species_mask != kSpeciesMask) return fail(s, RCM_ERR_STATE, fn + ": needs the default species_mask (H2O, CO2, O3, N2O, CH4)");
    if (!grad) return RCM_OK;
    std::vector<double> co;
    bool any = false;
    if ((st = grad_fold(s, fn, ncol, w_E_down, w_E_up, w_dE, co, &any)) != RCM_OK) return st;
    if (!any) {
        std::fill(grad, grad + (size_t)ncol * GRAD_NE, 0.0);
        return RCM_OK;
    }
    constexpr size_t D = sizeof(double);
    const int nsplit = split_geom(s, 0).nsplit;
    struct Set {
        DiagState state;
        double *co, *part, *grad;
    };
    return chunk_loop<Set, SplitArgs>(
        s, col0, ncol, diag_chunk(ncol), true,
        [&](DiagCarve& m, size_t ch, Set& z) {  // co [ch][42], part [ch][nsplit][121], grad [ch][121]
            z.co = m.take<double>(ch * GRAD_NCO);
            z.part = m.take<double>(ch * nsplit * GRAD_NE);
            z.grad = m.take<double>(ch * GRAD_NE);
        },
        [&](const Set& z, int c0, int n, cudaStream_t q, SplitArgs& a) -> int {  // diag_chunks' prep, the chunk's cotangents first
            CU(cudaMemcpyAsync(z.co, co.data() + (size_t)(c0 - col0) * GRAD_NCO, (size_t)n * GRAD_NCO * D, cudaMemcpyHostToDevice, q));
            return diag_prep(s, q, c0, n, z.state, vmr_scale ? &sc : nullptr, a);
        },
        [&](const Set& z, const SplitArgs& a, cudaStream_t q) {
            return grad_sweep(s, a, q, a.Tlayer, a.Tsurf, z.co, z.part, z.grad);
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            CU(cudaMemcpyAsync(grad + r * GRAD_NE, z.grad, (size_t)n * GRAD_NE * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

// Line-by-line flux gradients: the LBL species Jacobian's chunks, prep, raw planes and factors, then rcm_lbl_grad_kernel into
// partials [ch][ceil(nwvl / GRAD_LBL_SPAN)][121] and rcm_grad_sum_kernel over the spans.
int rcm_lbl_flux_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const double* w_E_down,
                          const double* w_E_up, const double* w_dE, double* grad) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_lbl_flux_gradient";
    DiagScale sc{};
    int st = lbl_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->p.species_mask != kSpeciesMask) return fail(s, RCM_ERR_STATE, fn + ": needs the default species_mask (H2O, CO2, O3, N2O, CH4)");
    if (!grad) return RCM_OK;
    std::vector<double> co;
    bool any = false;
    if ((st = grad_fold(s, fn, ncol, w_E_down, w_E_up, w_dE, co, &any)) != RCM_OK) return st;
    if (!any) {
        std::fill(grad, grad + (size_t)ncol * GRAD_NE, 0.0);
        return RCM_OK;
    }
    constexpr size_t D = sizeof(double);
    const double* tau3 = nullptr;
    if ((st = lbl_planes(s, sc, tau3)) != RCM_OK) return st;
    const double wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    const double* raw = s->d_lbl_tau5 + 3 * (size_t)s->lbl_nwvl * NLAY;
    const int nspan = (s->lbl_nwvl + GRAD_LBL_SPAN - 1) / GRAD_LBL_SPAN;
    struct Set {
        DiagState state;
        LblState lbl;
        double *co, *part, *grad;
    };
    return chunk_loop<Set, LblArgs>(
        s, col0, ncol, diag_chunk(ncol), false,
        [&](DiagCarve& m, size_t ch, Set& z) {  // co [ch][42], part [ch][nspan][121], grad [ch][121]
            lbl_take(m, ch, z.lbl);
            z.co = m.take<double>(ch * GRAD_NCO);
            z.part = m.take<double>(ch * nspan * GRAD_NE);
            z.grad = m.take<double>(ch * GRAD_NE);
        },
        [&](const Set& z, int c0, int n, cudaStream_t q, LblArgs& a) -> int {
            CU(cudaMemcpyAsync(z.co, co.data() + (size_t)(c0 - col0) * GRAD_NCO, (size_t)n * GRAD_NCO * D, cudaMemcpyHostToDevice, q));
            return lbl_prep(s, q, c0, n, z.state, z.lbl, tau3, vmr_scale ? &sc : nullptr, a);
        },
        [&](const Set& z, const LblArgs& a, cudaStream_t q) -> int {
            CU(rcm_launch_lbl_grad(a, wtau, raw, sc.f[1] * s->lbl_co2_factor, sc.f[4], sc.f[3], z.co, z.part, q));
            CU(rcm_launch_grad_sum(a.ncol, nspan, z.part, z.grad, q));
            s->launches += 2;
            return RCM_OK;
        },
        [&](const Set& z, size_t r, int n, cudaStream_t q) -> int {
            CU(cudaMemcpyAsync(grad + r * GRAD_NE, z.grad, (size_t)n * GRAD_NE * D, cudaMemcpyDeviceToHost, q));
            return RCM_OK;
        });
}

extern "C++" {
namespace {

// the arguments both adjusted-forcing calls check after the solver's state: ntrop [ncol] in [0, 19], tol, max_iter
int fdh_check_args(rcm_solver* s, const std::string& fn, int ncol, const int* ntrop, double tol, int max_iter) {
    if (!ntrop) return fail(s, RCM_ERR_ARG, fn + ": ntrop is NULL");
    for (int c = 0; c < ncol; ++c)
        if (ntrop[c] < 0 || ntrop[c] > FDH_MAXM)
            return fail(s, RCM_ERR_ARG, fn + ": ntrop[" + std::to_string(c) + "] = " + std::to_string(ntrop[c]) + " outside [0, 19]");
    if (!std::isfinite(tol) || !(tol > 0.0)) return fail(s, RCM_ERR_ARG, fn + ": tol must be finite and > 0");
    if (max_iter < 1) return fail(s, RCM_ERR_ARG, fn + ": max_iter must be >= 1");
    return RCM_OK;
}

// The two-slot Newton schedule of the adjusted-forcing calls over the chunks of ch columns from col0.  Slot k runs on its
// stream z.q and carries c0, n, iter and live.  start(z, k, c0) enqueues a chunk up to the check of its iterate 0, whose active
// count lands in h_fdh_count[k]; newton(z) enqueues the Jacobian and the Newton step; check(z, k) the evaluation of iterate
// z.iter and its check; download(z) the chunk's outputs.  The host reads a chunk's active count after every check, and the two
// slots take turns: one chunk's kernels run while the host waits for the other's count.
template <class Slot, class Start, class Check, class Newton, class Download>
int fdh_schedule(rcm_solver* s, Slot (&slot)[2], int col0, int ncol, size_t ch, Start start, Check check, Newton newton,
                 Download download) {
    int st;
    int next = col0;
    for (int k = 0; k < 2 && next < col0 + ncol; ++k, next += (int)ch)
        if ((st = start(slot[k], k, next)) != RCM_OK) return st;
    for (int k = 0; slot[0].live || slot[1].live; k ^= 1) {
        Slot& z = slot[k];
        if (!z.live) continue;
        CU(cudaStreamSynchronize(z.q));
        if (s->h_fdh_count[k] > 0) {  // (none is left after iterate max_iter)
            if ((st = newton(z)) != RCM_OK) return st;
            ++z.iter;
            if ((st = check(z, k)) != RCM_OK) return st;
            continue;
        }
        if ((st = download(z)) != RCM_OK) return st;
        z.live = false;
        if (next < col0 + ncol) {
            if ((st = start(z, k, next)) != RCM_OK) return st;
            next += (int)ch;
        }
    }
    return diag_end(s);
}

}  // namespace
}  // extern "C++"

// Stratosphere-adjusted forcing: the scratch sets, streams, state copies and prep of the calls above.  Per chunk a base
// evaluation (unscaled), the VMR scaling, then Newton iterations: retemper, evaluation (rcm_diag_rt_kernel +
// rcm_diag_sum_kernel), check; while columns are active, the flux Jacobian (rcm_fjac_kernel) and the Newton step.  The host
// reads a chunk's active count after every check.  The chunks of the two streams take turns: one chunk's kernels run while
// the host waits for the other's count.
int rcm_adjusted_forcing(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, double tol, int max_iter,
                         double* F, double* dT_adj, double* E_down, double* E_up, int* iters) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_adjusted_forcing";
    DiagScale sc{};
    int st = diag_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->h2o_slot != 0) return fail(s, RCM_ERR_STATE, fn + ": needs H2O among the active species");
    if ((st = fdh_check_args(s, fn, ncol, ntrop, tol, max_iter)) != RCM_OK) return st;
    const int nwvl = s->dc.nwvl;
    const bool first = (s->step_index == 0);
    const size_t ch = diag_chunk(ncol), D = sizeof(double);
    struct Slot {
        cudaStream_t q;
        int c0 = 0, n = 0, iter = 0;
        bool live = false;
        DiagState state;
        double *Ttau, *Tp, *dT, *Ed0, *Eu0, *dE0, *Ed, *Eu, *dE, *F, *Edo, *Euo, *J, *H, *spec_dn, *spec_up;
        int *ntrop, *iters, *count;
        SplitArgs a;
    } slot[2];
    // T_tau, T + dT, dT [ch][20], E_down, E_up [ch][21] and dE [ch][20] of the base and of the current iterate, F [ch][4], the
    // output E_down, E_up [ch][21], J [ch][2][21][41], dE_jac [ch][20][41], spectral [2][ch][nwvl][21]; ntrop, iters [ch] and
    // the active count
    st = diag_begin(s, ch, slot, [&](DiagCarve& m, size_t, Slot& z) {
        z.Ttau = m.take<double>(ch * NLAY);
        z.Tp = m.take<double>(ch * NLAY);
        z.dT = m.take<double>(ch * NLAY);
        z.Ed0 = m.take<double>(ch * NLEV);
        z.Eu0 = m.take<double>(ch * NLEV);
        z.dE0 = m.take<double>(ch * NLAY);
        z.Ed = m.take<double>(ch * NLEV);
        z.Eu = m.take<double>(ch * NLEV);
        z.dE = m.take<double>(ch * NLAY);
        z.F = m.take<double>(ch * 4);
        z.Edo = m.take<double>(ch * NLEV);
        z.Euo = m.take<double>(ch * NLEV);
        z.J = m.take<double>(ch * FJAC_NJ);
        z.H = m.take<double>(ch * FJAC_NH);
        z.spec_dn = m.take<double>(ch * nwvl * NLEV);
        z.spec_up = m.take<double>(ch * nwvl * NLEV);
        z.ntrop = m.take<int>(ch);
        z.iters = m.take<int>(ch);
        z.count = m.take<int>(1);
    });
    if (st != RCM_OK) return st;
    if (!s->h_fdh_count) CU(cudaMallocHost((void**)&s->h_fdh_count, 2 * sizeof(int)));
    for (int k = 0; k < 2; ++k) slot[k].q = s->dg_stream[k];
    auto fdh_args = [&](const Slot& z) {
        FdhArgs f{};
        f.ncol = z.n;
        f.iter = z.iter;
        f.max_iter = max_iter;
        f.tol = tol;
        f.T_floor = s->T_floor;
        f.tile = z.state.tile;
        f.Tb = z.state.T;
        f.Ttau = first ? z.Ttau : z.state.T;
        f.Tp = z.Tp;
        f.dT = z.dT;
        f.ntrop = z.ntrop;
        f.Ed0 = z.Ed0;
        f.Eu0 = z.Eu0;
        f.dE0 = z.dE0;
        f.Ed = z.Ed;
        f.Eu = z.Eu;
        f.dE = z.dE;
        f.dE_jac = z.H;
        f.iters = z.iters;
        f.F = z.F;
        f.Ed_out = z.Edo;
        f.Eu_out = z.Euo;
        f.nactive = z.count;
        return f;
    };
    // iterate z.iter: the tile blocks at T + dT, their fluxes, the check, the active count into h_fdh_count[k]
    auto check = [&](Slot& z, int k) -> int {
        const FdhArgs f = fdh_args(z);
        CU(rcm_launch_fdh_retemper(f, z.q));
        if ((st = diag_fluxes(s, z.a, z.q, z.spec_dn, z.spec_up, z.Ed, z.Eu, z.dE)) != RCM_OK) return st;
        CU(rcm_launch_fdh_check(f, z.q));
        CU(cudaMemcpyAsync(s->h_fdh_count + k, z.count, sizeof(int), cudaMemcpyDeviceToHost, z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // the flux Jacobian at T + dT and the Newton step
    auto newton = [&](Slot& z) -> int {
        if ((st = flux_jacobian(s, z.a, z.q, z.Tp, z.J, z.H)) != RCM_OK) return st;
        CU(rcm_launch_fdh_newton(fdh_args(z), z.q));
        s->launches += 1;
        return RCM_OK;
    };
    // the chunk [c0, c0 + n): T_tau, prep, base evaluation, scaling, iterate 0
    auto start = [&](Slot& z, int k, int c0) -> int {
        z.c0 = c0;
        z.n = std::min((int)ch, col0 + ncol - c0);
        z.iter = 0;
        z.live = true;
        if (first) CU(cudaMemcpyAsync(z.Ttau, s->d_T + (size_t)c0 * NLAY, z.n * NLAY * D, cudaMemcpyDeviceToDevice, z.q));
        CU(cudaMemcpyAsync(z.ntrop, ntrop + (c0 - col0), z.n * sizeof(int), cudaMemcpyHostToDevice, z.q));
        if ((st = diag_prep(s, z.q, c0, z.n, z.state, nullptr, z.a)) != RCM_OK) return st;
        if ((st = diag_fluxes(s, z.a, z.q, z.spec_dn, z.spec_up, z.Ed0, z.Eu0, z.dE0)) != RCM_OK) return st;
        if (vmr_scale) {
            CU(rcm_launch_diag_scale(z.state.tile, z.a.ntiles, sc, z.q));
            s->launches += 1;
        }
        return check(z, k);
    };
    auto download = [&](const Slot& z) -> int {
        const size_t r = (size_t)(z.c0 - col0);
        if (F) CU(cudaMemcpyAsync(F + r * 4, z.F, z.n * 4 * D, cudaMemcpyDeviceToHost, z.q));
        if (dT_adj) CU(cudaMemcpyAsync(dT_adj + r * NLAY, z.dT, z.n * NLAY * D, cudaMemcpyDeviceToHost, z.q));
        if (E_down) CU(cudaMemcpyAsync(E_down + r * NLEV, z.Edo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (E_up) CU(cudaMemcpyAsync(E_up + r * NLEV, z.Euo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (iters) CU(cudaMemcpyAsync(iters + r, z.iters, z.n * sizeof(int), cudaMemcpyDeviceToHost, z.q));
        return RCM_OK;
    };
    return fdh_schedule(s, slot, col0, ncol, ch, start, check, newton, download);
}

// Line-by-line stratosphere-adjusted forcing: rcm_adjusted_forcing's Newton schedule (fdh_schedule), check and Newton kernels
// on the state rcm_lbl_diagnose_fluxes radiates.  Per chunk: the prep on copies (unscaled, the tables' own planes), the
// prepared T_B and T_surf saved, the base evaluation (the step's rt and finish kernels; the finish moves the copies' T and
// T_surf), the H2O and O3 factors and the composed planes, then per iterate: rcm_lbl_fdh_retemper_kernel (every copy back to
// T_B + dT and the saved T_surf), the evaluation and the check; while columns are active, rcm_lbl_fjac_kernel at T_B + dT and
// the Newton step.  LBL tau does not depend on T: dT moves the Planck source of its layer alone.
int rcm_lbl_adjusted_forcing(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, double tol,
                             int max_iter, double* F, double* dT_adj, double* E_down, double* E_up, int* iters) {
    if (!s) return RCM_ERR_ARG;
    const std::string fn = "rcm_lbl_adjusted_forcing";
    DiagScale sc{};
    int st = lbl_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if ((st = fdh_check_args(s, fn, ncol, ntrop, tol, max_iter)) != RCM_OK) return st;
    const double* tau3 = nullptr;
    if ((st = lbl_planes(s, sc, tau3)) != RCM_OK) return st;
    const size_t ch = diag_chunk(ncol), D = sizeof(double);
    const size_t nchunks = (size_t)lbl_args(s, 0).nchunks;
    const double wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    struct Slot {
        cudaStream_t q;
        int c0 = 0, n = 0, iter = 0;
        bool live = false;
        DiagState state;
        LblState lbl;
        double *Tb, *Ts0, *Tp, *dT, *Ed0, *Eu0, *dE0, *Ed, *Eu, *dE, *F, *Edo, *Euo, *J, *H, *part, *dt;
        float* time;
        int *ntrop, *iters, *count;
        LblArgs a;
    } slot[2];
    // the prep's T_surf, sH, sO; T_B, T_surf as prepared, T_B + dT, dT [ch][20]; E_down, E_up [ch][21] and dE [ch][20] of the
    // base and of the current iterate, F [ch][4], the output E_down, E_up [ch][21], J [ch][2][21][41], dE_jac [ch][20][41],
    // the rt kernel's partials [nchunks][ch][42], the finish's dt and time [ch]; ntrop, iters [ch] and the active count
    st = diag_begin(s, ch, slot, [&](DiagCarve& m, size_t, Slot& z) {
        lbl_take(m, ch, z.lbl);
        z.Tb = m.take<double>(ch * NLAY);
        z.Ts0 = m.take<double>(ch);
        z.Tp = m.take<double>(ch * NLAY);
        z.dT = m.take<double>(ch * NLAY);
        z.Ed0 = m.take<double>(ch * NLEV);
        z.Eu0 = m.take<double>(ch * NLEV);
        z.dE0 = m.take<double>(ch * NLAY);
        z.Ed = m.take<double>(ch * NLEV);
        z.Eu = m.take<double>(ch * NLEV);
        z.dE = m.take<double>(ch * NLAY);
        z.F = m.take<double>(ch * 4);
        z.Edo = m.take<double>(ch * NLEV);
        z.Euo = m.take<double>(ch * NLEV);
        z.J = m.take<double>(ch * FJAC_NJ);
        z.H = m.take<double>(ch * FJAC_NH);
        z.part = m.take<double>(nchunks * ch * 2 * NLEV);
        z.dt = m.take<double>(ch);
        z.time = m.take<float>(ch);
        z.ntrop = m.take<int>(ch);
        z.iters = m.take<int>(ch);
        z.count = m.take<int>(1);
    }, false);
    if (st != RCM_OK) return st;
    if (!s->h_fdh_count) CU(cudaMallocHost((void**)&s->h_fdh_count, 2 * sizeof(int)));
    for (int k = 0; k < 2; ++k) slot[k].q = s->dg_stream[k];
    auto fdh_args = [&](const Slot& z) {
        FdhArgs f{};
        f.ncol = z.n;
        f.iter = z.iter;
        f.max_iter = max_iter;
        f.tol = tol;
        f.T_floor = s->T_floor;
        f.Tb = z.Tb;
        f.Tp = z.Tp;
        f.dT = z.dT;
        f.ntrop = z.ntrop;
        f.Ed0 = z.Ed0;
        f.Eu0 = z.Eu0;
        f.dE0 = z.dE0;
        f.Ed = z.Ed;
        f.Eu = z.Eu;
        f.dE = z.dE;
        f.dE_jac = z.H;
        f.iters = z.iters;
        f.F = z.F;
        f.Ed_out = z.Edo;
        f.Eu_out = z.Euo;
        f.nactive = z.count;
        return f;
    };
    // the step's rt and finish kernels on the chunk's copies: E_down, E_up, dE into Ed, Eu, dE
    auto evaluate = [&](const Slot& z, double* Ed, double* Eu, double* dE) -> int {
        LblArgs a = z.a;
        a.E_down = Ed;
        a.E_up = Eu;
        a.dE = dE;
        CU(rcm_launch_lbl_rt(a, z.q, nullptr, nullptr));
        CU(rcm_launch_lbl_finish(a, z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // iterate z.iter: the copies at T_B + dT, their fluxes, the check, the active count into h_fdh_count[k]
    auto check = [&](Slot& z, int k) -> int {
        const FdhArgs f = fdh_args(z);
        CU(rcm_launch_lbl_fdh_retemper(f, z.a.Tlayer, z.a.Tsurf, z.Ts0, z.q));
        if ((st = evaluate(z, z.Ed, z.Eu, z.dE)) != RCM_OK) return st;
        CU(rcm_launch_fdh_check(f, z.q));
        CU(cudaMemcpyAsync(s->h_fdh_count + k, z.count, sizeof(int), cudaMemcpyDeviceToHost, z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // the flux Jacobian at T_B + dT (Tp, never the copy the finish has moved) and the Newton step
    auto newton = [&](Slot& z) -> int {
        LblArgs a = z.a;
        a.Tlayer = z.Tp;
        a.Tsurf = z.Ts0;
        CU(rcm_launch_lbl_fjac(a, wtau, z.J, z.H, z.q));
        CU(rcm_launch_fdh_newton(fdh_args(z), z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // the chunk [c0, c0 + n): prep, T_B and T_surf saved, base evaluation, scaling, iterate 0
    auto start = [&](Slot& z, int k, int c0) -> int {
        z.c0 = c0;
        z.n = std::min((int)ch, col0 + ncol - c0);
        z.iter = 0;
        z.live = true;
        CU(cudaMemcpyAsync(z.ntrop, ntrop + (c0 - col0), z.n * sizeof(int), cudaMemcpyHostToDevice, z.q));
        if ((st = lbl_prep(s, z.q, c0, z.n, z.state, z.lbl, nullptr, nullptr, z.a)) != RCM_OK) return st;
        z.a.time_h = z.time;
        z.a.part = z.part;
        z.a.dt = z.dt;
        CU(cudaMemcpyAsync(z.Tb, z.a.Tlayer, z.n * NLAY * D, cudaMemcpyDeviceToDevice, z.q));
        CU(cudaMemcpyAsync(z.Ts0, z.a.Tsurf, z.n * D, cudaMemcpyDeviceToDevice, z.q));
        if ((st = evaluate(z, z.Ed0, z.Eu0, z.dE0)) != RCM_OK) return st;
        if (vmr_scale) {
            CU(rcm_launch_lbl_scale(z.a, sc.f[0], sc.f[2], z.q));
            s->launches += 1;
        }
        if (tau3) z.a.tau3 = tau3;
        return check(z, k);
    };
    auto download = [&](const Slot& z) -> int {
        const size_t r = (size_t)(z.c0 - col0);
        if (F) CU(cudaMemcpyAsync(F + r * 4, z.F, z.n * 4 * D, cudaMemcpyDeviceToHost, z.q));
        if (dT_adj) CU(cudaMemcpyAsync(dT_adj + r * NLAY, z.dT, z.n * NLAY * D, cudaMemcpyDeviceToHost, z.q));
        if (E_down) CU(cudaMemcpyAsync(E_down + r * NLEV, z.Edo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (E_up) CU(cudaMemcpyAsync(E_up + r * NLEV, z.Euo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (iters) CU(cudaMemcpyAsync(iters + r, z.iters, z.n * sizeof(int), cudaMemcpyDeviceToHost, z.q));
        return RCM_OK;
    };
    return fdh_schedule(s, slot, col0, ncol, ch, start, check, newton, download);
}

extern "C++" {
namespace {

// the checks both climate-response calls make after fdh_check_args
int ecs_check_args(rcm_solver* s, const std::string& fn, int fixed_rh) {
    if (fixed_rh && s->h2o_slot < 0) return fail(s, RCM_ERR_STATE, fn + ": fixed relative humidity needs H2O among the active species");
    if (fixed_rh && s->step_index == 0)
        return fail(s, RCM_ERR_STATE, fn + ": fixed relative humidity needs a step index > 0 (the step applies no feedback at step 0)");
    return RCM_OK;
}

// The outputs of a climate-response call (NULL: not wanted).
struct EcsOut {
    double *F, *dT, *dTs, *E_down, *E_up;
    int* iters;
};

// The gradient calls' outputs: dTs_dF [ncol][21] and dTs_dlnx [ncol][100] (NULL: not wanted).
struct EcsGrad {
    double *dTs_dF, *dTs_dlnx;
};

// A slot's scratch for the gradient calls' epilogue: co [ch][42], part [ch][npart][121], sum [ch][121], dF [ch][21] (none for
// the response alone, so that its scratch layout stays as it was)
struct EcsGradSet {
    double *co, *part, *sum, *dF;
};

void ecs_grad_take(DiagCarve& m, size_t ch, size_t npart, bool grad, EcsGradSet& g) {
    g.co = m.take<double>(grad ? ch * GRAD_NCO : 0);
    g.part = m.take<double>(grad ? ch * npart * GRAD_NE : 0);
    g.sum = m.take<double>(grad ? ch * GRAD_NE : 0);
    g.dF = m.take<double>(grad ? ch * NLEV : 0);
}

// the epilogue's downloads of the rows [r, r + n): dTs_dF, and entries 21..120 of the sums into dTs_dlnx
int ecs_grad_download(rcm_solver* s, const EcsGrad& o, const EcsGradSet& g, size_t r, int n, cudaStream_t q) {
    constexpr size_t D = sizeof(double);
    if (o.dTs_dF) CU(cudaMemcpyAsync(o.dTs_dF + r * NLEV, g.dF, (size_t)n * NLEV * D, cudaMemcpyDeviceToHost, q));
    if (o.dTs_dlnx)
        CU(cudaMemcpy2DAsync(o.dTs_dlnx + r * SPJ_NE, SPJ_NE * D, g.sum + NLEV, GRAD_NE * D, SPJ_NE * D, n,
                             cudaMemcpyDeviceToHost, q));
    return RCM_OK;
}

// Equilibrium climate response of the repwvl path: rcm_adjusted_forcing's scratch sets, streams, prep, base evaluation, scaling
// and Newton schedule (fdh_schedule) with one more unknown per column, the uniform potential-temperature increment dTs of the
// troposphere and the surface.  Per iterate: rcm_ecs_retemper_kernel (tile blocks at T + dT and Ts + dTs, with fixed RH the
// H2O row), the evaluation and rcm_ecs_check_kernel; while columns are active, the flux Jacobian (rcm_fjac_kernel at T + dT,
// Ts + dTs) and rcm_ecs_newton_kernel.  With grad (the gradient call) the checks add the species mask, and a chunk whose
// active count has reached 0 runs an epilogue before its download: the flux Jacobian at the solution, rcm_ecs_adjoint_kernel
// and the gradient sweep on the retempered tile blocks.
int ecs_response(rcm_solver* s, const std::string& fn, int col0, int ncol, const double* vmr_scale, const int* ntrop,
                 int fixed_rh, double tol, int max_iter, const EcsOut& o, const EcsGrad* grad) {
    DiagScale sc{};
    int st = diag_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if (s->h2o_slot != 0) return fail(s, RCM_ERR_STATE, fn + ": needs H2O among the active species");
    if ((st = fdh_check_args(s, fn, ncol, ntrop, tol, max_iter)) != RCM_OK) return st;
    if ((st = ecs_check_args(s, fn, fixed_rh)) != RCM_OK) return st;
    if (grad && s->p.species_mask != kSpeciesMask)
        return fail(s, RCM_ERR_STATE, fn + ": needs the default species_mask (H2O, CO2, O3, N2O, CH4)");
    if (grad && !o.dTs && !o.iters && !grad->dTs_dF && !grad->dTs_dlnx) return RCM_OK;
    const int nwvl = s->dc.nwvl;
    const bool first = (s->step_index == 0);
    const size_t ch = diag_chunk(ncol), D = sizeof(double);
    const size_t nsplit = split_geom(s, 0).nsplit;
    struct Slot {
        cudaStream_t q;
        int c0 = 0, n = 0, iter = 0;
        bool live = false;
        DiagState state;
        double *Ttau, *Tp, *dT, *Tsp, *dTs, *Ed0, *Eu0, *dE0, *Ed, *Eu, *dE, *F, *Edo, *Euo, *J, *H, *spec_dn, *spec_up;
        EcsGradSet g;
        int *ntrop, *iters, *count;
        SplitArgs a;
    } slot[2];
    // T_tau, T + dT, dT [ch][20], Ts + dTs, dTs [ch], E_down, E_up [ch][21] and dE [ch][20] of the base and of the current
    // iterate, F [ch][2], the output E_down, E_up [ch][21], J [ch][2][21][41], dE_jac [ch][20][41], spectral [2][ch][nwvl][21];
    // the epilogue's scratch; ntrop, iters [ch] and the active count
    st = diag_begin(s, ch, slot, [&](DiagCarve& m, size_t, Slot& z) {
        z.Ttau = m.take<double>(ch * NLAY);
        z.Tp = m.take<double>(ch * NLAY);
        z.dT = m.take<double>(ch * NLAY);
        z.Tsp = m.take<double>(ch);
        z.dTs = m.take<double>(ch);
        z.Ed0 = m.take<double>(ch * NLEV);
        z.Eu0 = m.take<double>(ch * NLEV);
        z.dE0 = m.take<double>(ch * NLAY);
        z.Ed = m.take<double>(ch * NLEV);
        z.Eu = m.take<double>(ch * NLEV);
        z.dE = m.take<double>(ch * NLAY);
        z.F = m.take<double>(ch * 2);
        z.Edo = m.take<double>(ch * NLEV);
        z.Euo = m.take<double>(ch * NLEV);
        z.J = m.take<double>(ch * FJAC_NJ);
        z.H = m.take<double>(ch * FJAC_NH);
        z.spec_dn = m.take<double>(ch * nwvl * NLEV);
        z.spec_up = m.take<double>(ch * nwvl * NLEV);
        ecs_grad_take(m, ch, nsplit, grad, z.g);
        z.ntrop = m.take<int>(ch);
        z.iters = m.take<int>(ch);
        z.count = m.take<int>(1);
    });
    if (st != RCM_OK) return st;
    if (!s->h_fdh_count) CU(cudaMallocHost((void**)&s->h_fdh_count, 2 * sizeof(int)));
    for (int k = 0; k < 2; ++k) slot[k].q = s->dg_stream[k];
    auto ecs_args = [&](const Slot& z) {
        EcsArgs e{};
        e.ncol = z.n;
        e.iter = z.iter;
        e.max_iter = max_iter;
        e.fixed_rh = fixed_rh != 0;
        e.tol = tol;
        e.T_floor = s->T_floor;
        e.f_h2o = sc.f[0];
        e.tile = z.state.tile;
        e.Tb = z.state.T;
        e.Ttau = first ? z.Ttau : z.state.T;
        e.Ts0 = z.a.Tsurf;
        e.rel_hum = z.a.rel_hum;
        e.Tp = z.Tp;
        e.Tsp = z.Tsp;
        e.dT = z.dT;
        e.dTs = z.dTs;
        e.ntrop = z.ntrop;
        e.Ed0 = z.Ed0;
        e.Eu0 = z.Eu0;
        e.dE0 = z.dE0;
        e.Ed = z.Ed;
        e.Eu = z.Eu;
        e.dE = z.dE;
        e.J = z.J;
        e.dE_jac = z.H;
        e.iters = z.iters;
        e.F = z.F;
        e.Ed_out = z.Edo;
        e.Eu_out = z.Euo;
        e.nactive = z.count;
        return e;
    };
    // iterate z.iter: the tile blocks at T + dT, Ts + dTs, their fluxes, the check, the active count into h_fdh_count[k]
    auto check = [&](Slot& z, int k) -> int {
        const EcsArgs e = ecs_args(z);
        CU(rcm_launch_ecs_retemper(e, z.q));
        if ((st = diag_fluxes(s, z.a, z.q, z.spec_dn, z.spec_up, z.Ed, z.Eu, z.dE)) != RCM_OK) return st;
        CU(rcm_launch_ecs_check(e, z.q));
        CU(cudaMemcpyAsync(s->h_fdh_count + k, z.count, sizeof(int), cudaMemcpyDeviceToHost, z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // the flux Jacobian at T + dT, Ts + dTs and the Newton step
    auto newton = [&](Slot& z) -> int {
        SplitArgs a = z.a;
        a.Tsurf = z.Tsp;
        if ((st = flux_jacobian(s, a, z.q, z.Tp, z.J, z.H)) != RCM_OK) return st;
        CU(rcm_launch_ecs_newton(ecs_args(z), z.q));
        s->launches += 1;
        return RCM_OK;
    };
    // the chunk [c0, c0 + n): T_tau, prep, base evaluation, scaling, iterate 0
    auto start = [&](Slot& z, int k, int c0) -> int {
        z.c0 = c0;
        z.n = std::min((int)ch, col0 + ncol - c0);
        z.iter = 0;
        z.live = true;
        if (first) CU(cudaMemcpyAsync(z.Ttau, s->d_T + (size_t)c0 * NLAY, z.n * NLAY * D, cudaMemcpyDeviceToDevice, z.q));
        CU(cudaMemcpyAsync(z.ntrop, ntrop + (c0 - col0), z.n * sizeof(int), cudaMemcpyHostToDevice, z.q));
        if ((st = diag_prep(s, z.q, c0, z.n, z.state, nullptr, z.a)) != RCM_OK) return st;
        if ((st = diag_fluxes(s, z.a, z.q, z.spec_dn, z.spec_up, z.Ed0, z.Eu0, z.dE0)) != RCM_OK) return st;
        if (vmr_scale) {
            CU(rcm_launch_diag_scale(z.state.tile, z.a.ntiles, sc, z.q));
            s->launches += 1;
        }
        return check(z, k);
    };
    // the flux Jacobian at the solution (the tile blocks, Tp and Tsp of the last retemper: a frozen column is not retempered),
    // the adjoint solve and the sweep, then the epilogue's downloads
    auto epilogue = [&](const Slot& z) -> int {
        SplitArgs a = z.a;
        a.Tsurf = z.Tsp;
        if ((st = flux_jacobian(s, a, z.q, z.Tp, z.J, z.H)) != RCM_OK) return st;
        CU(rcm_launch_ecs_adjoint(ecs_args(z), z.g.dF, z.g.co, z.q));
        s->launches += 1;
        if ((st = grad_sweep(s, z.a, z.q, z.Tp, z.Tsp, z.g.co, z.g.part, z.g.sum)) != RCM_OK) return st;
        return ecs_grad_download(s, *grad, z.g, (size_t)(z.c0 - col0), z.n, z.q);
    };
    auto download = [&](const Slot& z) -> int {
        if (grad && (st = epilogue(z)) != RCM_OK) return st;
        const size_t r = (size_t)(z.c0 - col0);
        if (o.F) CU(cudaMemcpyAsync(o.F + r * 2, z.F, z.n * 2 * D, cudaMemcpyDeviceToHost, z.q));
        if (o.dT) CU(cudaMemcpyAsync(o.dT + r * NLAY, z.dT, z.n * NLAY * D, cudaMemcpyDeviceToHost, z.q));
        if (o.dTs) CU(cudaMemcpyAsync(o.dTs + r, z.dTs, z.n * D, cudaMemcpyDeviceToHost, z.q));
        if (o.E_down) CU(cudaMemcpyAsync(o.E_down + r * NLEV, z.Edo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (o.E_up) CU(cudaMemcpyAsync(o.E_up + r * NLEV, z.Euo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (o.iters) CU(cudaMemcpyAsync(o.iters + r, z.iters, z.n * sizeof(int), cudaMemcpyDeviceToHost, z.q));
        return RCM_OK;
    };
    return fdh_schedule(s, slot, col0, ncol, ch, start, check, newton, download);
}

// Line-by-line equilibrium climate response: rcm_lbl_adjusted_forcing's chunks, prep, saved T_B and T_surf, base evaluation,
// scaling and Newton schedule; per iterate rcm_lbl_ecs_retemper_kernel (every copy back to T_B + dT, T_surf + dTs, with fixed
// RH s_H2O at T_B + dT), the evaluation and rcm_ecs_check_kernel; while columns are active, rcm_lbl_fjac_kernel at
// T_B + dT, T_surf + dTs and rcm_ecs_newton_kernel.  grad as in ecs_response; the epilogue is rcm_lbl_fjac_kernel at the
// solution, rcm_ecs_adjoint_kernel, then rcm_lbl_grad_kernel on the copies and planes the last evaluation radiated.
int lbl_ecs_response(rcm_solver* s, const std::string& fn, int col0, int ncol, const double* vmr_scale, const int* ntrop,
                     int fixed_rh, double tol, int max_iter, const EcsOut& o, const EcsGrad* grad) {
    DiagScale sc{};
    int st = lbl_check(s, fn, col0, ncol, vmr_scale, sc);
    if (st != RCM_OK) return st;
    if ((st = fdh_check_args(s, fn, ncol, ntrop, tol, max_iter)) != RCM_OK) return st;
    if ((st = ecs_check_args(s, fn, fixed_rh)) != RCM_OK) return st;
    if (grad && s->p.species_mask != kSpeciesMask)
        return fail(s, RCM_ERR_STATE, fn + ": needs the default species_mask (H2O, CO2, O3, N2O, CH4)");
    if (grad && !o.dTs && !o.iters && !grad->dTs_dF && !grad->dTs_dlnx) return RCM_OK;
    const double* tau3 = nullptr;
    if ((st = lbl_planes(s, sc, tau3)) != RCM_OK) return st;
    const size_t ch = diag_chunk(ncol), D = sizeof(double);
    const size_t nchunks = (size_t)lbl_args(s, 0).nchunks;
    const double wtau = 2 * M_PI * (1.0 / (double)s->p.nangle);
    const double* raw = s->d_lbl_tau5 + 3 * (size_t)s->lbl_nwvl * NLAY;
    const size_t nspan = (s->lbl_nwvl + GRAD_LBL_SPAN - 1) / GRAD_LBL_SPAN;
    struct Slot {
        cudaStream_t q;
        int c0 = 0, n = 0, iter = 0;
        bool live = false;
        DiagState state;
        LblState lbl;
        double *Tb, *Ts0, *Tp, *dT, *Tsp, *dTs, *Ed0, *Eu0, *dE0, *Ed, *Eu, *dE, *F, *Edo, *Euo, *J, *H, *part, *dt;
        EcsGradSet g;
        float* time;
        int *ntrop, *iters, *count;
        LblArgs a;
    } slot[2];
    // the prep's T_surf, sH, sO; T_B, T_surf as prepared, T_B + dT, dT [ch][20], T_surf + dTs, dTs [ch]; E_down, E_up [ch][21]
    // and dE [ch][20] of the base and of the current iterate, F [ch][2], the output E_down, E_up [ch][21], J [ch][2][21][41],
    // dE_jac [ch][20][41], the rt kernel's partials [nchunks][ch][42], the finish's dt, the epilogue's scratch, time [ch];
    // ntrop, iters [ch] and the active count
    st = diag_begin(s, ch, slot, [&](DiagCarve& m, size_t, Slot& z) {
        lbl_take(m, ch, z.lbl);
        z.Tb = m.take<double>(ch * NLAY);
        z.Ts0 = m.take<double>(ch);
        z.Tp = m.take<double>(ch * NLAY);
        z.dT = m.take<double>(ch * NLAY);
        z.Tsp = m.take<double>(ch);
        z.dTs = m.take<double>(ch);
        z.Ed0 = m.take<double>(ch * NLEV);
        z.Eu0 = m.take<double>(ch * NLEV);
        z.dE0 = m.take<double>(ch * NLAY);
        z.Ed = m.take<double>(ch * NLEV);
        z.Eu = m.take<double>(ch * NLEV);
        z.dE = m.take<double>(ch * NLAY);
        z.F = m.take<double>(ch * 2);
        z.Edo = m.take<double>(ch * NLEV);
        z.Euo = m.take<double>(ch * NLEV);
        z.J = m.take<double>(ch * FJAC_NJ);
        z.H = m.take<double>(ch * FJAC_NH);
        z.part = m.take<double>(nchunks * ch * 2 * NLEV);
        z.dt = m.take<double>(ch);
        ecs_grad_take(m, ch, nspan, grad, z.g);
        z.time = m.take<float>(ch);
        z.ntrop = m.take<int>(ch);
        z.iters = m.take<int>(ch);
        z.count = m.take<int>(1);
    }, false);
    if (st != RCM_OK) return st;
    if (!s->h_fdh_count) CU(cudaMallocHost((void**)&s->h_fdh_count, 2 * sizeof(int)));
    for (int k = 0; k < 2; ++k) slot[k].q = s->dg_stream[k];
    auto ecs_args = [&](const Slot& z) {
        EcsArgs e{};
        e.ncol = z.n;
        e.iter = z.iter;
        e.max_iter = max_iter;
        e.fixed_rh = fixed_rh != 0;
        e.tol = tol;
        e.T_floor = s->T_floor;
        e.f_h2o = sc.f[0];
        e.Tb = z.Tb;
        e.Ts0 = z.Ts0;
        e.rel_hum = z.a.rel_hum;
        e.Tp = z.Tp;
        e.Tsp = z.Tsp;
        e.dT = z.dT;
        e.dTs = z.dTs;
        e.T = z.a.Tlayer;
        e.Ts = z.a.Tsurf;
        e.sH = z.a.sH;
        e.h2o_ref = z.a.h2o_ref;
        e.ntrop = z.ntrop;
        e.Ed0 = z.Ed0;
        e.Eu0 = z.Eu0;
        e.dE0 = z.dE0;
        e.Ed = z.Ed;
        e.Eu = z.Eu;
        e.dE = z.dE;
        e.J = z.J;
        e.dE_jac = z.H;
        e.iters = z.iters;
        e.F = z.F;
        e.Ed_out = z.Edo;
        e.Eu_out = z.Euo;
        e.nactive = z.count;
        return e;
    };
    // the step's rt and finish kernels on the chunk's copies: E_down, E_up, dE into Ed, Eu, dE
    auto evaluate = [&](const Slot& z, double* Ed, double* Eu, double* dE) -> int {
        LblArgs a = z.a;
        a.E_down = Ed;
        a.E_up = Eu;
        a.dE = dE;
        CU(rcm_launch_lbl_rt(a, z.q, nullptr, nullptr));
        CU(rcm_launch_lbl_finish(a, z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // iterate z.iter: the copies at T_B + dT, T_surf + dTs, their fluxes, the check, the active count into h_fdh_count[k]
    auto check = [&](Slot& z, int k) -> int {
        const EcsArgs e = ecs_args(z);
        CU(rcm_launch_lbl_ecs_retemper(e, z.q));
        if ((st = evaluate(z, z.Ed, z.Eu, z.dE)) != RCM_OK) return st;
        CU(rcm_launch_ecs_check(e, z.q));
        CU(cudaMemcpyAsync(s->h_fdh_count + k, z.count, sizeof(int), cudaMemcpyDeviceToHost, z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // the flux Jacobian at T_B + dT, T_surf + dTs (Tp, Tsp: never the copies the finish has moved) and the Newton step
    auto newton = [&](Slot& z) -> int {
        LblArgs a = z.a;
        a.Tlayer = z.Tp;
        a.Tsurf = z.Tsp;
        CU(rcm_launch_lbl_fjac(a, wtau, z.J, z.H, z.q));
        CU(rcm_launch_ecs_newton(ecs_args(z), z.q));
        s->launches += 2;
        return RCM_OK;
    };
    // the chunk [c0, c0 + n): prep, T_B and T_surf saved, base evaluation, scaling, iterate 0
    auto start = [&](Slot& z, int k, int c0) -> int {
        z.c0 = c0;
        z.n = std::min((int)ch, col0 + ncol - c0);
        z.iter = 0;
        z.live = true;
        CU(cudaMemcpyAsync(z.ntrop, ntrop + (c0 - col0), z.n * sizeof(int), cudaMemcpyHostToDevice, z.q));
        if ((st = lbl_prep(s, z.q, c0, z.n, z.state, z.lbl, nullptr, nullptr, z.a)) != RCM_OK) return st;
        z.a.time_h = z.time;
        z.a.part = z.part;
        z.a.dt = z.dt;
        CU(cudaMemcpyAsync(z.Tb, z.a.Tlayer, z.n * NLAY * D, cudaMemcpyDeviceToDevice, z.q));
        CU(cudaMemcpyAsync(z.Ts0, z.a.Tsurf, z.n * D, cudaMemcpyDeviceToDevice, z.q));
        if ((st = evaluate(z, z.Ed0, z.Eu0, z.dE0)) != RCM_OK) return st;
        if (vmr_scale) {
            CU(rcm_launch_lbl_scale(z.a, sc.f[0], sc.f[2], z.q));
            s->launches += 1;
        }
        if (tau3) z.a.tau3 = tau3;
        return check(z, k);
    };
    // the flux Jacobian at the solution (Tp, Tsp: never the copies the finish has moved; sH and sO as the last retemper and
    // the scaling left them), the adjoint solve and the sweep with the composed planes, then the epilogue's downloads
    auto epilogue = [&](const Slot& z) -> int {
        LblArgs a = z.a;
        a.Tlayer = z.Tp;
        a.Tsurf = z.Tsp;
        CU(rcm_launch_lbl_fjac(a, wtau, z.J, z.H, z.q));
        CU(rcm_launch_ecs_adjoint(ecs_args(z), z.g.dF, z.g.co, z.q));
        CU(rcm_launch_lbl_grad(a, wtau, raw, sc.f[1] * s->lbl_co2_factor, sc.f[4], sc.f[3], z.g.co, z.g.part, z.q));
        CU(rcm_launch_grad_sum(a.ncol, (int)nspan, z.g.part, z.g.sum, z.q));
        s->launches += 4;
        return ecs_grad_download(s, *grad, z.g, (size_t)(z.c0 - col0), z.n, z.q);
    };
    auto download = [&](const Slot& z) -> int {
        if (grad && (st = epilogue(z)) != RCM_OK) return st;
        const size_t r = (size_t)(z.c0 - col0);
        if (o.F) CU(cudaMemcpyAsync(o.F + r * 2, z.F, z.n * 2 * D, cudaMemcpyDeviceToHost, z.q));
        if (o.dT) CU(cudaMemcpyAsync(o.dT + r * NLAY, z.dT, z.n * NLAY * D, cudaMemcpyDeviceToHost, z.q));
        if (o.dTs) CU(cudaMemcpyAsync(o.dTs + r, z.dTs, z.n * D, cudaMemcpyDeviceToHost, z.q));
        if (o.E_down) CU(cudaMemcpyAsync(o.E_down + r * NLEV, z.Edo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (o.E_up) CU(cudaMemcpyAsync(o.E_up + r * NLEV, z.Euo, z.n * NLEV * D, cudaMemcpyDeviceToHost, z.q));
        if (o.iters) CU(cudaMemcpyAsync(o.iters + r, z.iters, z.n * sizeof(int), cudaMemcpyDeviceToHost, z.q));
        return RCM_OK;
    };
    return fdh_schedule(s, slot, col0, ncol, ch, start, check, newton, download);
}

// The gradient calls around ecs_response / lbl_ecs_response (run): dTs_dF into a buffer of their own when the caller wants
// dTs_dlnx alone, and after the call a row of quiet NaN in dTs_dlnx wherever the adjoint kernel wrote one in dTs_dF (the
// response did not converge, or A at the solution could not be solved).
template <class Run>
int ecs_gradient(int ncol, double* dTs_dF, double* dTs_dlnx, Run run) {
    std::vector<double> own;
    if (!dTs_dF && dTs_dlnx && ncol > 0) {
        own.resize((size_t)ncol * NLEV);
        dTs_dF = own.data();
    }
    const EcsGrad g{dTs_dF, dTs_dlnx};
    const int st = run(g);
    if (st != RCM_OK || !dTs_dlnx) return st;
    for (int c = 0; c < ncol; ++c)
        if (std::isnan(dTs_dF[(size_t)c * NLEV + NLAY]))
            std::fill(dTs_dlnx + (size_t)c * SPJ_NE, dTs_dlnx + (size_t)(c + 1) * SPJ_NE, std::numeric_limits<double>::quiet_NaN());
    return RCM_OK;
}

}  // namespace
}  // extern "C++"

int rcm_climate_response(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, int fixed_rh, double tol,
                         int max_iter, double* F, double* dT, double* dTs, double* E_down, double* E_up, int* iters) {
    if (!s) return RCM_ERR_ARG;
    return ecs_response(s, "rcm_climate_response", col0, ncol, vmr_scale, ntrop, fixed_rh, tol, max_iter,
                        EcsOut{F, dT, dTs, E_down, E_up, iters}, nullptr);
}

int rcm_lbl_climate_response(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, int fixed_rh,
                             double tol, int max_iter, double* F, double* dT, double* dTs, double* E_down, double* E_up,
                             int* iters) {
    if (!s) return RCM_ERR_ARG;
    return lbl_ecs_response(s, "rcm_lbl_climate_response", col0, ncol, vmr_scale, ntrop, fixed_rh, tol, max_iter,
                            EcsOut{F, dT, dTs, E_down, E_up, iters}, nullptr);
}

// Climate-response gradients: the response with its epilogue, of the response's outputs only dTs and iters.
int rcm_climate_response_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop, int fixed_rh,
                                  double tol, int max_iter, double* dTs, double* dTs_dF, double* dTs_dlnx, int* iters) {
    if (!s) return RCM_ERR_ARG;
    return ecs_gradient(ncol, dTs_dF, dTs_dlnx, [&](const EcsGrad& g) {
        return ecs_response(s, "rcm_climate_response_gradient", col0, ncol, vmr_scale, ntrop, fixed_rh, tol, max_iter,
                            EcsOut{nullptr, nullptr, dTs, nullptr, nullptr, iters}, &g);
    });
}

int rcm_lbl_climate_response_gradient(rcm_solver* s, int col0, int ncol, const double* vmr_scale, const int* ntrop,
                                      int fixed_rh, double tol, int max_iter, double* dTs, double* dTs_dF, double* dTs_dlnx,
                                      int* iters) {
    if (!s) return RCM_ERR_ARG;
    return ecs_gradient(ncol, dTs_dF, dTs_dlnx, [&](const EcsGrad& g) {
        return lbl_ecs_response(s, "rcm_lbl_climate_response_gradient", col0, ncol, vmr_scale, ntrop, fixed_rh, tol,
                                max_iter, EcsOut{nullptr, nullptr, dTs, nullptr, nullptr, iters}, &g);
    });
}

// ------------------------------------------------------------------------------------------
// Checkpoint / restart of an ensemble (SURVEY 8(f)4).  One flat little-endian file:
//   "RCMCKPT1", header (int64: ncol, nactive, species_mask, step_index, has_col_solar, has_col_cloud, lbl_mode,
//   nwvl of the table the run used - 0 in files written before it was recorded), plevel[21], then per column arrays in the order of kCkptArrays below.
// Everything the step reads or carries is in it, so a solver that loads the same table and this file continues
// bit-identically (tests/test_gpu_checkpoint.py).  Tables are not stored: they are inputs of the run, not state.
// ------------------------------------------------------------------------------------------
namespace {
struct CkptArray { void* dev; size_t bytes; };

int ckpt_arrays(rcm_solver* s, CkptArray* out, bool col_solar, bool col_cloud) {
    const size_t n = (size_t)s->ncol, D = sizeof(double);
    int k = 0;
    out[k++] = {s->d_T, n * NLAY * D};
    out[k++] = {s->d_Ts, n * D};
    out[k++] = {s->d_vmr, n * s->nactive * NLAY * D};
    out[k++] = {s->d_rh, n * NLAY * D};
    out[k++] = {s->d_Tprev, n * NLAY * D};
    out[k++] = {s->d_time, n * sizeof(float)};
    out[k++] = {s->d_dt, n * D};
    out[k++] = {s->d_Ed, n * NLEV * D};
    out[k++] = {s->d_Eu, n * NLEV * D};
    out[k++] = {s->d_dE, n * NLAY * D};
    if (col_solar) out[k++] = {s->d_solar_col, n * D};
    if (col_cloud) out[k++] = {s->d_cloud_col, n * D};
    return k;
}
}  // namespace

int rcm_column_count(const rcm_solver* s) { return s ? s->ncol : 0; }

int rcm_save_checkpoint(rcm_solver* s, const char* path) {
    if (!s || !path) return RCM_ERR_ARG;
    if (s->ncol <= 0) return fail(s, RCM_ERR_STATE, "no columns loaded");
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->stream));
    FILE* f = std::fopen(path, "wb");
    if (!f) return fail(s, RCM_ERR_IO, std::string("cannot write ") + path);
    const long long hdr[8] = {s->ncol, s->nactive, (long long)s->p.species_mask, s->step_index, s->has_col_solar ? 1 : 0,
                              s->has_col_cloud ? 1 : 0, s->lbl_mode ? 1 : 0, s->dc.nwvl};
    bool ok = std::fwrite("RCMCKPT1", 1, 8, f) == 8 && std::fwrite(hdr, sizeof(hdr), 1, f) == 1 &&
              std::fwrite(s->plevel, sizeof(s->plevel), 1, f) == 1;
    CkptArray arr[12];
    const int na = ckpt_arrays(s, arr, s->has_col_solar, s->has_col_cloud);
    std::vector<char> buf;
    for (int k = 0; k < na && ok; ++k) {
        buf.resize(arr[k].bytes);
        cudaError_t e = cudaMemcpy(buf.data(), arr[k].dev, arr[k].bytes, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            std::fclose(f);
            return cuda_fail(s, e, "checkpoint download");
        }
        ok = std::fwrite(buf.data(), 1, arr[k].bytes, f) == arr[k].bytes;
    }
    ok = (std::fclose(f) == 0) && ok;
    return ok ? RCM_OK : fail(s, RCM_ERR_IO, std::string("short write to ") + path);
}

int rcm_load_checkpoint(rcm_solver* s, const char* path) {
    if (!s || !path) return RCM_ERR_ARG;
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->stream));  // work queued earlier may still read or write the arrays overwritten below
    FILE* f = std::fopen(path, "rb");
    if (!f) return fail(s, RCM_ERR_IO, std::string("cannot read ") + path);
    char magic[8];
    long long hdr[8];
    double plevel[RCM_NLEVEL];
    if (std::fread(magic, 1, 8, f) != 8 || std::memcmp(magic, "RCMCKPT1", 8) != 0 || std::fread(hdr, sizeof(hdr), 1, f) != 1 ||
        std::fread(plevel, sizeof(plevel), 1, f) != 1 || hdr[0] <= 0 || hdr[0] > (1LL << 30)) {
        std::fclose(f);
        return fail(s, RCM_ERR_FORMAT, std::string(path) + " is not a checkpoint of this solver");
    }
    set_active_species(s);
    if ((unsigned)hdr[2] != s->p.species_mask || (int)hdr[1] != s->nactive) {
        std::fclose(f);
        return fail(s, RCM_ERR_STATE, "checkpoint was written with another species_mask");
    }
    if ((hdr[6] != 0) != s->lbl_mode) {
        std::fclose(f);
        return fail(s, RCM_ERR_STATE, "checkpoint belongs to the other spectral path (repwvl / line-by-line)");
    }
    if (hdr[7] != 0 && (s->has_table || s->lbl_mode) && hdr[7] != s->dc.nwvl) {
        std::fclose(f);
        return fail(s, RCM_ERR_STATE, "checkpoint was written with a table of another wavelength count");
    }
    int st = ensure_columns(s, (int)hdr[0]);
    if (st != RCM_OK) {
        std::fclose(f);
        return st;
    }
    s->ncol = (int)hdr[0];
    if ((hdr[4] || hdr[5]) && !s->d_solar_col) {
        cudaError_t e = dalloc(s->d_solar_col, (size_t)s->cap);
        if (e == cudaSuccess) e = dalloc(s->d_cloud_col, (size_t)s->cap);
        if (e != cudaSuccess) {
            std::fclose(f);
            s->ncol = 0;
            return cuda_fail(s, e, "checkpoint: per-column forcing buffers");
        }
    }
    CkptArray arr[12];
    const int na = ckpt_arrays(s, arr, hdr[4] != 0, hdr[5] != 0);
    std::vector<char> buf;
    for (int k = 0; k < na; ++k) {
        buf.resize(arr[k].bytes);
        if (std::fread(buf.data(), 1, arr[k].bytes, f) != arr[k].bytes) {
            std::fclose(f);
            s->ncol = 0;
            return fail(s, RCM_ERR_FORMAT, std::string(path) + " is truncated");
        }
        cudaError_t e = cudaMemcpy(arr[k].dev, buf.data(), arr[k].bytes, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            std::fclose(f);
            s->ncol = 0;
            return cuda_fail(s, e, "checkpoint upload");
        }
    }
    std::fclose(f);
    if (!s->has_plevel || std::memcmp(s->plevel, plevel, sizeof(plevel)) != 0) s->coef_dirty = true;
    std::memcpy(s->plevel, plevel, sizeof(plevel));
    s->has_plevel = true;
    s->const_dirty = true;
    s->step_index = (long)hdr[3];
    s->has_col_solar = hdr[4] != 0;
    s->has_col_cloud = hdr[5] != 0;
    s->tau_valid = false;
    s->tile_vmr_valid = false;
    return RCM_OK;
}

// Host buffers in, one step, host buffers out.  For big repwvl ensembles the columns are cut into chunks that
// travel through three internal streams: while chunk k is stepped, chunk k+1 is on its way up and chunk k-1 on
// its way down (separate copy engines), so the call costs about one step plus one chunk of copies instead of
// step + all copies.  Every chunk is launched with the tile shape of the whole ensemble: results are
// bit-identical to rcm_update_columns + rcm_advance + rcm_get_state.
int rcm_step_host(rcm_solver* s, const double* Tlayer_in, const double* Tsurf_in, const double* vmr_active_in,
                  double* E_down, double* E_up, double* dE, double* Tlayer_out, double* Tsurf_out) {
    if (!s) return RCM_ERR_ARG;
    int max_chunks = 8;
    if (const char* e = std::getenv("RCM_PIPE_CHUNKS")) max_chunks = std::max(1, std::min(16, std::atoi(e)));  // experiments
    const int nchunk = (s && !s->lbl_mode && s->has_table) ? std::min(max_chunks, s->ncol / 4096) : 0;
    if (nchunk < 2) {
        int st = rcm_update_columns(s, Tlayer_in, Tsurf_in, vmr_active_in);
        if (st != RCM_OK) return st;
        st = rcm_advance_async(s, 1, nullptr);
        if (st != RCM_OK) return st;
        return rcm_get_state(s, Tlayer_out, Tsurf_out, nullptr, nullptr, E_down, E_up, dE, nullptr);
    }
    CU(cudaSetDevice(s->device));
    int st = ensure_diag(s, 1);
    if (st != RCM_OK) return st;
    st = refresh_const(s);
    if (st != RCM_OK) return st;
    if (!s->pipe_stream[0]) {
        for (int i = 0; i < 3; ++i) {
            CU(cudaStreamCreateWithFlags(&s->pipe_stream[i], cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&s->pipe_done[i], cudaEventDisableTiming));
        }
        CU(cudaEventCreateWithFlags(&s->pipe_start, cudaEventDisableTiming));
    }
    if (use_split(s))
        return step_host_split(s, nchunk, Tlayer_in, Tsurf_in, vmr_active_in, E_down, E_up, dE, Tlayer_out, Tsurf_out);
    const int nsm = nsm_of(s);
    Part whole[2];
    plan_parts(s, s->ncol, nsm, whole);
    const int C = whole[0].sh.C;
    const int per = ((s->ncol + nchunk - 1) / nchunk + C - 1) / C * C;  // chunk = whole tiles
    CU(cudaEventRecord(s->pipe_start, s->stream));
    for (int i = 0; i < 3; ++i) CU(cudaStreamWaitEvent(s->pipe_stream[i], s->pipe_start, 0));
    const size_t D = sizeof(double);
    const int na = s->nactive;
    for (int k = 0, c0 = 0; c0 < s->ncol; ++k, c0 += per) {
        const int n = std::min(per, s->ncol - c0);
        const size_t o = (size_t)c0;
        cudaStream_t q = s->pipe_stream[k % 3];
        if (Tlayer_in) CU(cudaMemcpyAsync(s->d_T + o * NLAY, Tlayer_in + o * NLAY, n * NLAY * D, cudaMemcpyHostToDevice, q));
        if (Tsurf_in) CU(cudaMemcpyAsync(s->d_Ts + o, Tsurf_in + o, n * D, cudaMemcpyHostToDevice, q));
        if (vmr_active_in)
            CU(cudaMemcpyAsync(s->d_vmr + o * na * NLAY, vmr_active_in + o * na * NLAY, (size_t)n * na * NLAY * D,
                               cudaMemcpyHostToDevice, q));
        const Part p{c0, n, whole[0].sh};
        st = launch_part(s, MODE_STEP, 1, true, p, nsm, q);
        if (st != RCM_OK) return st;
        if (E_down) CU(cudaMemcpyAsync(E_down + o * NLEV, s->d_Ed + o * NLEV, n * NLEV * D, cudaMemcpyDeviceToHost, q));
        if (E_up) CU(cudaMemcpyAsync(E_up + o * NLEV, s->d_Eu + o * NLEV, n * NLEV * D, cudaMemcpyDeviceToHost, q));
        if (dE) CU(cudaMemcpyAsync(dE + o * NLAY, s->d_dE + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToHost, q));
        if (Tlayer_out) CU(cudaMemcpyAsync(Tlayer_out + o * NLAY, s->d_T + o * NLAY, n * NLAY * D, cudaMemcpyDeviceToHost, q));
        if (Tsurf_out) CU(cudaMemcpyAsync(Tsurf_out + o, s->d_Ts + o, n * D, cudaMemcpyDeviceToHost, q));
    }
    for (int i = 0; i < 3; ++i) {
        CU(cudaEventRecord(s->pipe_done[i], s->pipe_stream[i]));
        CU(cudaStreamWaitEvent(s->stream, s->pipe_done[i], 0));
    }
    CU(rcm_launch_reduce_diag(s->d_diag, 1, s->ncol, s->p.dT_converged, s->d_red, s->d_ticket, s->d_scalars, s->stream));
    s->launches += 1;
    s->step_index += 1;
    s->tau_valid = false;
    CU(cudaStreamSynchronize(s->stream));
    return RCM_OK;
}

int rcm_cplkavg_device(rcm_solver* s, int n, const double* lo_nm, const double* hi_nm, const double* t, double* out) {
    if (!s || n <= 0 || !lo_nm || !hi_nm || !t || !out) return RCM_ERR_ARG;
    CU(cudaSetDevice(s->device));
    double* d = nullptr;
    CU(dalloc(d, (size_t)4 * n));
    cudaError_t e = cudaMemcpyAsync(d, lo_nm, n * sizeof(double), cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + n, hi_nm, n * sizeof(double), cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + 2 * (size_t)n, t, n * sizeof(double), cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess) e = rcm_launch_cplkavg(n, d, d + n, d + 2 * (size_t)n, d + 3 * (size_t)n, s->d_exp_tab, s->opt_cplk_narrow, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d + 3 * (size_t)n, n * sizeof(double), cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    cudaFree(d);
    if (e != cudaSuccess) return cuda_fail(s, e, "cplkavg");
    s->launches += 1;
    return RCM_OK;
}

long rcm_launch_count(const rcm_solver* s) { return s ? s->launches : 0; }

int rcm_host_graph_stats(const rcm_solver* s, long* captures, long* replays) {
    if (!s || !captures || !replays) return RCM_ERR_ARG;
    *captures = s->hg.captures;
    *replays = s->hg.replays;
    return RCM_OK;
}

int rcm_fp64_microbench(rcm_solver* s, int which, double* gops) {
    if (!s || !gops || which < 0 || which > 3) return RCM_ERR_ARG;
    CU(cudaSetDevice(s->device));
    int nsm = 148;
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, s->device);
    const int grid = nsm * 8;
    const long iters = (which == 0) ? 40000 : 4000;
    double* d = nullptr;
    CU(dalloc(d, (size_t)grid * 256));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaError_t e = rcm_launch_microbench(which, d, s->d_exp_tab, iters / 10, grid, s->stream);  // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 3 && e == cudaSuccess; ++rep) {
        cudaEventRecord(e0, s->stream);
        e = rcm_launch_microbench(which, d, s->d_exp_tab, iters, grid, s->stream);
        cudaEventRecord(e1, s->stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    if (e != cudaSuccess) return cuda_fail(s, e, "microbench");
    s->launches += 4;
    *gops = (double)grid * 256.0 * 8.0 * (double)iters / (best * 1e-3) / 1e9;
    return RCM_OK;
}

int rcm_kernel_time_ms(rcm_solver* s, int reset, double* avg_ms, long* n_launches) {
    if (!s) return RCM_ERR_ARG;
    CU(cudaSetDevice(s->device));
    CU(cudaStreamSynchronize(s->stream));
    for (auto& ev : s->ev_used) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) {
            s->kt_ms += ms;
            s->kt_n += 1;
        }
        s->ev_free.push_back(ev);
    }
    s->ev_used.clear();
    if (avg_ms) *avg_ms = s->kt_n ? s->kt_ms / s->kt_n : 0.0;
    if (n_launches) *n_launches = s->kt_n;
    if (reset) {
        s->kt_ms = 0.0;
        s->kt_n = 0;
    }
    return RCM_OK;
}

}  // extern "C"
