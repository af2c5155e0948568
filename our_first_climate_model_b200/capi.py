"""ctypes binding of include/rcm_b200.h (one Python method per C entry point)."""
from __future__ import annotations

import ctypes as C
import os
import re
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
NLAY, NLEV, NSPEC = 20, 21, 9
_lib = None


class RcmError(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [("nangle", C.c_int), ("cloud_layer", C.c_int), ("cloud_tau", C.c_double), ("dp", C.c_double),
                ("max_dT", C.c_double), ("dt_cap", C.c_double), ("solar_irr", C.c_double),
                ("dT_converged", C.c_double), ("species_mask", C.c_uint)]


class SolarParams(C.Structure):
    _fields_ = [("tau_s", C.c_double), ("mu_s", C.c_double), ("g_asym", C.c_double), ("albedo", C.c_double),
                ("daytime", C.c_double), ("E_0", C.c_double), ("doublings", C.c_int)]


class StepScalars(C.Structure):
    _fields_ = [("toa_net_sum", C.c_double), ("max_dT", C.c_double), ("n_converged", C.c_double),
                ("max_abs_dE", C.c_double)]


def library_path() -> str:
    # RCM_B200_LIB: another build of the same library (kernel variants under test: tools/build_variants.sh)
    return os.environ.get("RCM_B200_LIB") or os.path.join(_HERE, "lib", "librcm_b200.so")


def header_path() -> str:
    return os.path.join(_ROOT, "include", "rcm_b200.h")


def _declared_symbols():
    try:
        txt = open(header_path()).read()
    except OSError:
        return []
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(rcm_[a-z0-9_A-Z]+)\s*\(", txt)))


DECLARED_SYMBOLS = _declared_symbols()


def build_library(verbose=False):
    """Compile the CUDA extension in-tree for sm_100a (csrc/Makefile)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "-j4"], stdout=out)


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RcmError(f"{path} is missing: build it with our_first_climate_model_b200.build_library() "
                       "(there is no CPU fallback)")
    L = C.CDLL(path)
    L.rcm_status_string.restype = C.c_char_p
    L.rcm_last_error.restype = C.c_char_p
    L.rcm_lowerpos.restype = C.c_long
    L.rcm_table_array.restype = C.POINTER(C.c_double)
    L.rcm_cplkavg_host.restype = C.c_double
    L.rcm_cplkavg_host.argtypes = [C.c_double, C.c_double, C.c_double, C.c_void_p]
    L.rcm_launch_count.restype = C.c_long
    _lib = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _check(st, solver=None):
    if st != 0:
        L = load_library()
        msg = L.rcm_status_string(int(st)).decode()
        if solver is not None:
            extra = L.rcm_last_error(solver).decode()
            if extra:
                msg += ": " + extra
        raise RcmError(f"rcm status {st}: {msg}")


# ---- host-only helpers ------------------------------------------------------------------------
def default_params() -> Params:
    p = Params()
    _check(load_library().rcm_default_params(C.byref(p)))
    return p


def default_solar_params() -> SolarParams:
    sp = SolarParams()
    _check(load_library().rcm_default_solar_params(C.byref(sp)))
    return sp


def solar_setup(sp: SolarParams | None = None) -> dict:
    sp = sp or default_solar_params()
    out = np.zeros(7)
    _check(load_library().rcm_solar_setup(C.byref(sp), _p(out)))
    return dict(zip(["r_dir", "s_dir", "t_dir", "r", "t", "r_total", "solar_irr"], out))


def write_profiles(path: str, plevel, Tlayer, time_h, append=False, header=False, column_ids=False):
    """rcm_write_profiles: the reference's output_conv rows (main.cpp:102-114) for a whole ensemble."""
    T = _f64(Tlayer).reshape(-1, NLAY)
    th = np.ascontiguousarray(np.broadcast_to(time_h, (T.shape[0],)), dtype=np.float32)
    _check(load_library().rcm_write_profiles(path.encode(), C.c_int(int(append)), C.c_int(int(header)),
                                             C.c_int(T.shape[0]), _p(_f64(plevel, (NLEV,))), _p(T), _p(th),
                                             C.c_int(int(column_ids))))


def lowerpos(nodes, x) -> int:
    a = _f64(nodes)
    return int(load_library().rcm_lowerpos(_p(a), C.c_int(a.size), C.c_double(x)))


def device_count() -> int:
    return int(load_library().rcm_device_count())


class Table:
    """Host copy of a repwvl lookup table (rcm_table_load)."""

    def __init__(self, path: str):
        self._h = C.c_void_p()
        _check(load_library().rcm_table_load(path.encode(), C.byref(self._h)))
        d = (C.c_int * 4)()
        _check(_lib.rcm_table_dims(self._h, d))
        self.n_tpert, self.n_species, self.n_wvl, self.n_p = list(d)

    def array(self, which: int, shape):
        ptr = _lib.rcm_table_array(self._h, C.c_int(which))
        if not ptr:
            return None
        n = int(np.prod(shape))
        return np.ctypeslib.as_array(ptr, shape=(n,)).reshape(shape).copy()

    @property
    def xsec(self):
        return self.array(0, (self.n_tpert, self.n_species, self.n_wvl, self.n_p))

    @property
    def wvl(self):
        return self.array(1, (self.n_wvl,))

    @property
    def weight(self):
        return self.array(2, (self.n_wvl,))

    @property
    def p_grid(self):
        return self.array(3, (self.n_p,))

    @property
    def t_ref(self):
        return self.array(4, (self.n_p,))

    @property
    def t_pert(self):
        return self.array(5, (self.n_tpert,))

    @property
    def vmrs_ref(self):
        return self.array(6, (self.n_species, self.n_p))

    def close(self):
        if self._h:
            _lib.rcm_table_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def read_atm(path: str, max_rows: int = 64) -> np.ndarray:
    """-> array [nrows, ncols] (z, p, T, air, H2O, O3, CO2, CH4, N2O)."""
    cols = np.zeros((9, max_rows))
    nr, nc = C.c_int(0), C.c_int(0)
    _check(load_library().rcm_read_atm(path.encode(), C.c_int(max_rows), _p(cols), C.byref(nr), C.byref(nc)))
    return cols[:nc.value, :nr.value].T.copy()


def init_columns(plevel, Tlevel, vmr_ppm_level, co2_factor=1.0) -> dict:
    Tlevel = _f64(Tlevel).reshape(-1, NLEV)
    ncol = Tlevel.shape[0]
    vm = _f64(vmr_ppm_level, (ncol, 5, NLEV))
    pl = _f64(plevel, (NLEV,))
    out = dict(Tlayer=np.zeros((ncol, NLAY)), vmr9=np.zeros((ncol, NSPEC, NLAY)), rel_hum=np.zeros((ncol, NLAY)),
               player=np.zeros(NLAY), conv=np.zeros(NLAY))
    _check(load_library().rcm_init_columns(C.c_int(ncol), _p(pl), _p(Tlevel), _p(vm), C.c_double(co2_factor),
                                           _p(out["Tlayer"]), _p(out["vmr9"]), _p(out["rel_hum"]), _p(out["player"]),
                                           _p(out["conv"])))
    return out


def make_ensemble(ncol, seed, plevel, base_Tlevel, base_vmr_ppm_level):
    pl = _f64(plevel, (NLEV,))
    bT = _f64(base_Tlevel, (NLEV,))
    bv = _f64(base_vmr_ppm_level, (5, NLEV))
    T = np.zeros((ncol, NLEV))
    v = np.zeros((ncol, 5, NLEV))
    _check(load_library().rcm_make_ensemble(C.c_int(ncol), C.c_ulonglong(seed), _p(pl), _p(bT), _p(bv), _p(T), _p(v)))
    return T, v


def make_lbl_tables(nwvl, seed, plevel, h2o_vmr_layer, o3_vmr_layer):
    """Synthetic LBL tables: -> (wvl[nwvl] nm, tau5[5, nwvl, 20]) in the order H2O, CO2, O3, CH4, N2O."""
    wvl = np.zeros(nwvl)
    tau5 = np.zeros((5, nwvl, NLAY))
    _check(load_library().rcm_make_lbl_tables(C.c_int(nwvl), C.c_ulonglong(seed), _p(_f64(plevel, (NLEV,))),
                                              _p(_f64(h2o_vmr_layer, (NLAY,))), _p(_f64(o3_vmr_layer, (NLAY,))),
                                              _p(wvl), _p(tau5)))
    return wvl, tau5


def write_lbl_asc(path, wvl, tau):
    wvl = _f64(wvl)
    _check(load_library().rcm_write_lbl_asc(path.encode(), C.c_int(wvl.size), _p(wvl), _p(_f64(tau, (wvl.size, NLAY)))))


def ascii_file2xy2D(path: str):
    """-> (status, x[nx], y[nx, ny]) with the reference's status codes."""
    L = load_library()
    nx, ny = C.c_int(0), C.c_int(0)
    x, y = C.POINTER(C.c_double)(), C.POINTER(C.c_double)()
    st = L.rcm_ascii_file2xy2D(path.encode(), C.byref(nx), C.byref(ny), C.byref(x), C.byref(y))
    if st != 0:
        return st, None, None
    xa = np.ctypeslib.as_array(x, shape=(nx.value,)).copy() if nx.value else np.zeros(0)
    ya = (np.ctypeslib.as_array(y, shape=(nx.value * max(ny.value, 1),)).copy()[:nx.value * ny.value]
          .reshape(nx.value, ny.value)) if nx.value else np.zeros((0, 0))
    L.rcm_free(x)
    L.rcm_free(y)
    return 0, xa, ya


def cplkavg_host(lo, hi, t):
    st = C.c_int(0)
    v = load_library().rcm_cplkavg_host(float(lo), float(hi), float(t), C.addressof(st))
    return float(v), st.value


# ---- the solver ---------------------------------------------------------------------------------
class Solver:
    """One rcm_solver (one GPU).  Methods map 1:1 to the C entry points."""

    def __init__(self, device: int = 0, params: Params | None = None):
        L = load_library()
        self._h = C.c_void_p()
        self.params = params or default_params()
        st = L.rcm_create(C.c_int(device), C.byref(self.params), C.byref(self._h))
        if st != 0:
            self._h = C.c_void_p()
            _check(st)
        self.ncol = 0
        self.nwvl = 0
        self.stream_ptr = None
        self.nactive = bin(self.params.species_mask).count("1")

    # lifecycle
    def close(self):
        if self._h:
            _lib.rcm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_params(self, params: Params):
        _check(_lib.rcm_set_params(self._h, C.byref(params)), self._h)
        self.params = params
        self.nactive = bin(params.species_mask).count("1")

    def set_option(self, option: int, value: int):
        _check(_lib.rcm_set_option(self._h, C.c_int(option), C.c_int(value)), self._h)

    def set_stream(self, stream_ptr: int | None):
        _check(_lib.rcm_set_stream(self._h, C.c_void_p(stream_ptr or 0)), self._h)
        self.stream_ptr = stream_ptr or None  # None: the solver's own stream (the legacy stream 0 cannot be borrowed)

    def synchronize(self):
        _check(_lib.rcm_synchronize(self._h), self._h)

    # tables
    def set_repwvl_table(self, xsec, wvl, weight, p_grid, t_ref, t_pert):
        xsec = _f64(xsec)
        nt, ns, nw, npp = xsec.shape
        _check(_lib.rcm_set_repwvl_table(self._h, _p(xsec), _p(_f64(wvl)), _p(_f64(weight)), _p(_f64(p_grid)),
                                         _p(_f64(t_ref)), _p(_f64(t_pert)), C.c_int(nt), C.c_int(ns), C.c_int(nw),
                                         C.c_int(npp)), self._h)
        self.nwvl = nw

    def set_spectral_grid(self, wvl, weight):
        """rcm_set_spectral_grid: wavelengths [nm] and spectral weights alone (for rcm_radiative_transfer with a tau
        that was built elsewhere - the `radiative_transfer` signature of main.cpp:320-324)."""
        w = _f64(wvl)
        _check(_lib.rcm_set_spectral_grid(self._h, _p(w), _p(_f64(weight, (w.size,))), C.c_int(w.size)), self._h)
        self.nwvl = w.size

    def set_repwvl_table_from(self, table: Table):
        _check(_lib.rcm_set_repwvl_table_from(self._h, table._h), self._h)
        self.nwvl = table.n_wvl

    def set_lbl_tables(self, wvl, tau5, h2o_ref, o3_ref=None, co2_factor=1.0):
        wvl = _f64(wvl)
        tau5 = _f64(tau5, (5, wvl.size, NLAY))
        o3 = None if o3_ref is None else _f64(o3_ref, (NLAY,))
        _check(_lib.rcm_set_lbl_tables(self._h, _p(wvl), _p(tau5), C.c_int(wvl.size), _p(_f64(h2o_ref, (NLAY,))),
                                       _p(o3), C.c_double(co2_factor)), self._h)
        self.nwvl = wvl.size

    # columns
    def set_columns(self, plevel, Tlayer, Tsurf, vmr9, rel_hum):
        Tl = _f64(Tlayer).reshape(-1, NLAY)
        n = Tl.shape[0]
        Ts = _f64(np.broadcast_to(Tsurf, (n,)))
        _check(_lib.rcm_set_columns(self._h, C.c_int(n), _p(_f64(plevel, (NLEV,))), _p(Tl), _p(Ts),
                                    _p(_f64(vmr9, (n, NSPEC, NLAY))), _p(_f64(rel_hum, (n, NLAY)))), self._h)
        self.ncol = n

    def set_column_solar(self, sp: SolarParams | None = None, tau_s=None, mu_s=None, albedo=None,
                         cloud_from_tau_s: bool = False, clear: bool = False) -> dict | None:
        """rcm_set_column_solar: per-column solar forcing (and optionally the thermal grey cloud) computed on the
        device; returns {'solar_irr', 'r_total'} per column.  clear=True: back to the ensemble-wide constants."""
        if clear:
            _check(_lib.rcm_set_column_solar(self._h, None, None, None, None, C.c_int(0), None, None), self._h)
            return None
        sp = sp or default_solar_params()
        n = self.ncol
        arr = [None if a is None else _f64(np.broadcast_to(a, (n,))) for a in (tau_s, mu_s, albedo)]
        out = dict(solar_irr=np.zeros(n), r_total=np.zeros(n))
        _check(_lib.rcm_set_column_solar(self._h, C.byref(sp), _p(arr[0]), _p(arr[1]), _p(arr[2]),
                                         C.c_int(1 if cloud_from_tau_s else 0), _p(out["solar_irr"]),
                                         _p(out["r_total"])), self._h)
        return out

    def save_checkpoint(self, path: str):
        _check(_lib.rcm_save_checkpoint(self._h, path.encode()), self._h)

    def load_checkpoint(self, path: str):
        _check(_lib.rcm_load_checkpoint(self._h, path.encode()), self._h)
        self.ncol = int(_lib.rcm_column_count(self._h))

    def update_columns(self, Tlayer=None, Tsurf=None, vmr_active=None):
        a = None if Tlayer is None else _f64(Tlayer, (self.ncol, NLAY))
        b = None if Tsurf is None else _f64(Tsurf, (self.ncol,))
        c = None if vmr_active is None else _f64(vmr_active, (self.ncol, self.nactive, NLAY))
        _check(_lib.rcm_update_columns(self._h, _p(a), _p(b), _p(c)), self._h)
        self.synchronize()

    def set_step_index(self, i: int):
        _check(_lib.rcm_set_step_index(self._h, C.c_long(i)), self._h)

    # kernels
    def build_tau(self, want_tau=True, want_lowpos=True):
        tau = np.zeros((self.ncol, self.nwvl, NLAY)) if want_tau else None
        lp = np.zeros((self.ncol, NLAY), dtype=np.int32) if want_lowpos else None
        lt = np.zeros((self.ncol, NLAY), dtype=np.int32) if want_lowpos else None
        _check(_lib.rcm_build_tau(self._h, _p(tau), _p(lp), _p(lt)), self._h)
        return tau, lp, lt

    def radiative_transfer(self, tau=None):
        t = None if tau is None else _f64(tau, (self.ncol, self.nwvl, NLAY))
        Ed = np.zeros((self.ncol, NLEV)); Eu = np.zeros((self.ncol, NLEV)); dE = np.zeros((self.ncol, NLAY))
        _check(_lib.rcm_radiative_transfer(self._h, _p(t), _p(Ed), _p(Eu), _p(dE)), self._h)
        return Ed, Eu, dE

    def _vmr_scale(self, vmr_scale):
        """vmr_scale of the diagnostic calls as contiguous float64 with one factor per active species (None stays None)."""
        if vmr_scale is None:
            return None
        sc = _f64(vmr_scale).ravel()
        if sc.size != self.nactive:
            raise ValueError(f"vmr_scale needs {self.nactive} factors (one per active species), got {sc.size}")
        return sc

    def diagnose_fluxes(self, col0: int = 0, ncol: int | None = None, vmr_scale=None, spectral: bool = True) -> dict:
        """rcm_diagnose_fluxes: the fluxes the next step would compute for columns [col0, col0 + ncol), without changing
        anything.  vmr_scale [nactive]: factors on the active species' VMRs (ascending species index; None = unscaled).
        -> E_down, E_up [ncol, 21], dE [ncol, 20] and, with spectral, E_down_spec / E_up_spec [ncol, nwvl, 21]."""
        n = self.ncol - col0 if ncol is None else int(ncol)
        sc = self._vmr_scale(vmr_scale)
        m = max(n, 0)
        out = dict(E_down=np.zeros((m, NLEV)), E_up=np.zeros((m, NLEV)), dE=np.zeros((m, NLAY)))
        if spectral:
            out["E_down_spec"] = np.zeros((m, self.nwvl, NLEV))
            out["E_up_spec"] = np.zeros((m, self.nwvl, NLEV))
        _check(_lib.rcm_diagnose_fluxes(self._h, C.c_int(col0), C.c_int(n), _p(sc), _p(out.get("E_down_spec")),
                                        _p(out.get("E_up_spec")), _p(out["E_down"]), _p(out["E_up"]), _p(out["dE"])),
               self._h)
        return out

    def lbl_diagnose_fluxes(self, col0: int = 0, ncol: int | None = None, vmr_scale=None, bands=None) -> dict:
        """rcm_lbl_diagnose_fluxes: the fluxes the next line-by-line step would compute for columns [col0, col0 + ncol),
        without changing anything.  vmr_scale [5]: factors on H2O, CO2, O3, N2O, CH4 (ascending species index; None =
        unscaled).  bands: band_start [nband + 1], 0 = b_0 < ... < b_nband = nwvl, or None for no band outputs.
        -> E_down, E_up [ncol, 21], dE [ncol, 20] and, with bands, E_down_band / E_up_band [ncol, nband, 21] (each band the
        sum of its wavelengths' fluxes in index order)."""
        n = self.ncol - col0 if ncol is None else int(ncol)
        sc = self._vmr_scale(vmr_scale)
        m = max(n, 0)
        out = dict(E_down=np.zeros((m, NLEV)), E_up=np.zeros((m, NLEV)), dE=np.zeros((m, NLAY)))
        bs, nband = None, 0
        if bands is not None:
            bs = np.ascontiguousarray(bands, dtype=np.int32).ravel()
            nband = bs.size - 1
            out["E_down_band"] = np.zeros((m, max(nband, 0), NLEV))
            out["E_up_band"] = np.zeros((m, max(nband, 0), NLEV))
        _check(_lib.rcm_lbl_diagnose_fluxes(self._h, C.c_int(col0), C.c_int(n), _p(sc), C.c_int(nband), _p(bs),
                                            _p(out.get("E_down_band")), _p(out.get("E_up_band")), _p(out["E_down"]),
                                            _p(out["E_up"]), _p(out["dE"])), self._h)
        return out

    def lbl_radiative_kernels(self, col0: int = 0, ncol: int | None = None, vmr_scale=None, bands=None) -> dict:
        """rcm_lbl_radiative_kernels: derivatives of the next line-by-line step's OLR (output 0) and surface downward flux
        (output 1) for columns [col0, col0 + ncol), at the state lbl_diagnose_fluxes radiates, without changing anything.
        vmr_scale and bands as in lbl_diagnose_fluxes.
        -> K [ncol, 2, 41] (entries as radiative_kernels; the sum over the wavelengths in index order) with the views
        dOLR_dT, dOLR_dTs, dOLR_dlnq, dSFC_dT, dSFC_dlnq, and with bands K_band [ncol, nband, 2, 41] (each band the sum of
        its wavelengths' contributions in index order)."""
        n = self.ncol - col0 if ncol is None else int(ncol)
        sc = self._vmr_scale(vmr_scale)
        m = max(n, 0)
        K = np.zeros((m, 2, 2 * NLAY + 1))
        bs, nband, Kb = None, 0, None
        if bands is not None:
            bs = np.ascontiguousarray(bands, dtype=np.int32).ravel()
            nband = bs.size - 1
            Kb = np.zeros((m, max(nband, 0), 2, 2 * NLAY + 1))
        _check(_lib.rcm_lbl_radiative_kernels(self._h, C.c_int(col0), C.c_int(n), _p(sc), C.c_int(nband), _p(bs), _p(Kb),
                                              _p(K)), self._h)
        out = dict(K=K, dOLR_dT=K[:, 0, :NLAY], dOLR_dTs=K[:, 0, NLAY], dOLR_dlnq=K[:, 0, NLAY + 1:],
                   dSFC_dT=K[:, 1, :NLAY], dSFC_dlnq=K[:, 1, NLAY + 1:])
        if Kb is not None:
            out["K_band"] = Kb
        return out

    def radiative_kernels(self, col0: int = 0, ncol: int | None = None, vmr_scale=None, spectral: bool = False) -> dict:
        """rcm_radiative_kernels: derivatives of the next step's OLR (output 0) and surface downward flux (output 1) for
        columns [col0, col0 + ncol), without changing anything.  vmr_scale as in diagnose_fluxes.
        -> K [ncol, 2, 41] (entries: dF/dT_l for the 20 layers top-down, dF/dT_surf, dF/dln q_l for the 20 layers) with the
        views dOLR_dT [ncol, 20], dOLR_dTs [ncol], dOLR_dlnq [ncol, 20], dSFC_dT, dSFC_dlnq, and with spectral
        K_spec [ncol, nwvl, 2, 41] (each wavelength's contribution; K is its sum over the wavelengths in index order)."""
        n = self.ncol - col0 if ncol is None else int(ncol)
        sc = self._vmr_scale(vmr_scale)
        m = max(n, 0)
        K = np.zeros((m, 2, 2 * NLAY + 1))
        Ks = np.zeros((m, self.nwvl, 2, 2 * NLAY + 1)) if spectral else None
        _check(_lib.rcm_radiative_kernels(self._h, C.c_int(col0), C.c_int(n), _p(sc), _p(Ks), _p(K)), self._h)
        out = dict(K=K, dOLR_dT=K[:, 0, :NLAY], dOLR_dTs=K[:, 0, NLAY], dOLR_dlnq=K[:, 0, NLAY + 1:],
                   dSFC_dT=K[:, 1, :NLAY], dSFC_dlnq=K[:, 1, NLAY + 1:])
        if spectral:
            out["K_spec"] = Ks
        return out

    def flux_jacobian(self, col0: int = 0, ncol: int | None = None, vmr_scale=None) -> dict:
        """rcm_flux_jacobian: derivatives of the next step's broadband fluxes at every level and of its heating rates for
        columns [col0, col0 + ncol), without changing anything.  vmr_scale as in diagnose_fluxes.  Entries as in
        radiative_kernels (dT_l for the 20 layers top-down, dT_surf, dln q_l for the 20 layers).
        -> J [ncol, 2, 21, 41] (J[:, 0, k] = dE_down[k], J[:, 1, k] = dE_up[k]) and dE_jac [ncol, 20, 41]."""
        n = self.ncol - col0 if ncol is None else int(ncol)
        sc = self._vmr_scale(vmr_scale)
        m = max(n, 0)
        J = np.zeros((m, 2, NLAY + 1, 2 * NLAY + 1))
        H = np.zeros((m, NLAY, 2 * NLAY + 1))
        _check(_lib.rcm_flux_jacobian(self._h, C.c_int(col0), C.c_int(n), _p(sc), _p(J), _p(H)), self._h)
        return dict(J=J, dE_jac=H)

    def adjusted_forcing(self, vmr_scale, ntrop, col0: int = 0, ncol: int | None = None, tol: float = 1e-6,
                         max_iter: int = 20) -> dict:
        """rcm_adjusted_forcing: stratosphere-adjusted forcing by fixed dynamical heating for columns [col0, col0 + ncol),
        without changing anything.  vmr_scale as in diagnose_fluxes (None = unscaled: no forcing); ntrop: the stratospheric
        layers 0 .. ntrop - 1 of every column, an int or an array [ncol] of values in [0, 19]; Newton until
        max_{l < ntrop} |dE_l - dE_l^base| <= tol (W/m2), at most max_iter updates.
        -> F [ncol, 4] with the views IRF_toa, IRF_trop, SARF_toa, SARF_trop (W/m2), dT_adj [ncol, 20] (K), E_down, E_up
        [ncol, 21] at the adjusted perturbed state, iters [ncol] (Newton updates applied, -1: not converged) and
        converged [ncol] (iters >= 0)."""
        n = self.ncol - col0 if ncol is None else int(ncol)
        m = max(n, 0)
        sc = self._vmr_scale(vmr_scale)
        nt = np.asarray(ntrop)
        if nt.ndim == 0:
            nt = np.full(m, int(nt), dtype=np.int32)
        elif nt.shape != (m,):
            raise ValueError(f"ntrop needs one entry per column ({m}), got shape {nt.shape}")
        nt = np.ascontiguousarray(nt, dtype=np.int32)
        F = np.zeros((m, 4))
        dT = np.zeros((m, NLAY))
        Ed, Eu = np.zeros((m, NLEV)), np.zeros((m, NLEV))
        it = np.zeros(m, dtype=np.int32)
        _check(_lib.rcm_adjusted_forcing(self._h, C.c_int(col0), C.c_int(n), _p(sc), _p(nt), C.c_double(tol),
                                         C.c_int(max_iter), _p(F), _p(dT), _p(Ed), _p(Eu), _p(it)), self._h)
        return dict(F=F, IRF_toa=F[:, 0], IRF_trop=F[:, 1], SARF_toa=F[:, 2], SARF_trop=F[:, 3], dT_adj=dT, E_down=Ed,
                    E_up=Eu, iters=it, converged=it >= 0)

    def advance(self, nsteps: int, want_scalars=True):
        sc = (StepScalars * nsteps)() if want_scalars else None
        _check(_lib.rcm_advance(self._h, C.c_int(nsteps), sc), self._h)
        if sc is None:
            return None
        return np.array([[s.toa_net_sum, s.max_dT, s.n_converged, s.max_abs_dE] for s in sc])

    def run_to_equilibrium(self, max_steps: int, check_every: int = 100):
        """rcm_run_to_equilibrium -> (steps done, scalars of the last step [toa_net_sum, max_dT, n_converged, max|dE|])."""
        last, done = StepScalars(), C.c_long(0)
        _check(_lib.rcm_run_to_equilibrium(self._h, C.c_long(max_steps), C.c_int(check_every), C.byref(last),
                                           C.byref(done)), self._h)
        return done.value, np.array([last.toa_net_sum, last.max_dT, last.n_converged, last.max_abs_dE])

    def advance_async(self, nsteps: int) -> int:
        """Launch without waiting; returns the device address of double[nsteps][4] scalars."""
        ptr = C.c_void_p()
        _check(_lib.rcm_advance_async(self._h, C.c_int(nsteps), C.byref(ptr)), self._h)
        return ptr.value

    def get_state(self, want=("Tlayer", "Tsurf", "h2o", "time_h", "E_down", "E_up", "dE", "dt")) -> dict:
        n = self.ncol
        bufs = dict(Tlayer=np.zeros((n, NLAY)), Tsurf=np.zeros(n), h2o=np.zeros((n, NLAY)),
                    time_h=np.zeros(n, dtype=np.float32), E_down=np.zeros((n, NLEV)), E_up=np.zeros((n, NLEV)),
                    dE=np.zeros((n, NLAY)), dt=np.zeros(n))
        args = [_p(bufs[k]) if k in want else None
                for k in ("Tlayer", "Tsurf", "h2o", "time_h", "E_down", "E_up", "dE", "dt")]
        _check(_lib.rcm_get_state(self._h, *args), self._h)
        return {k: v for k, v in bufs.items() if k in want}

    def step_host_ptrs(self, T_in, Ts_in, vmr_in, Ed, Eu, dE, T_out, Ts_out):
        """rcm_step_host on raw host addresses (ints), e.g. pinned torch tensors' data_ptr()."""
        _check(_lib.rcm_step_host(self._h, *[C.c_void_p(x) for x in (T_in, Ts_in, vmr_in, Ed, Eu, dE, T_out, Ts_out)]),
               self._h)

    def step_host(self, Tlayer, Tsurf, vmr_active=None) -> dict:
        """rcm_step_host with numpy arrays: upload T / Tsurf / active VMRs, one step, download the results."""
        n = self.ncol
        T, Ts = _f64(Tlayer), _f64(Tsurf)
        v = None if vmr_active is None else _f64(vmr_active)  # None: the VMRs on the device stay (H2O follows the feedback)
        assert T.shape == (n, NLAY) and Ts.shape == (n,) and (v is None or v.shape == (n, self.nactive, NLAY))
        out = dict(E_down=np.zeros((n, NLEV)), E_up=np.zeros((n, NLEV)), dE=np.zeros((n, NLAY)),
                   Tlayer=np.zeros((n, NLAY)), Tsurf=np.zeros(n))
        _check(_lib.rcm_step_host(self._h, _p(T), _p(Ts), _p(v), _p(out["E_down"]), _p(out["E_up"]), _p(out["dE"]),
                                  _p(out["Tlayer"]), _p(out["Tsurf"])), self._h)
        return out

    def cplkavg_device(self, lo, hi, t):
        lo, hi, t = _f64(lo), _f64(hi), _f64(t)
        out = np.zeros_like(lo)
        _check(_lib.rcm_cplkavg_device(self._h, C.c_int(lo.size), _p(lo), _p(hi), _p(t), _p(out)), self._h)
        return out

    # introspection
    def launch_count(self) -> int:
        return int(_lib.rcm_launch_count(self._h))

    def host_graph_stats(self):
        """(captures, replays) of step_host's steady-state CUDA graph."""
        c, r = C.c_long(0), C.c_long(0)
        _check(_lib.rcm_host_graph_stats(self._h, C.byref(c), C.byref(r)), self._h)
        return c.value, r.value

    def fp64_microbench(self, which: int) -> float:
        v = C.c_double(0)
        _check(_lib.rcm_fp64_microbench(self._h, C.c_int(which), C.byref(v)), self._h)
        return v.value

    def kernel_time_ms(self, reset=False):
        ms, n = C.c_double(0), C.c_long(0)
        _check(_lib.rcm_kernel_time_ms(self._h, C.c_int(int(reset)), C.byref(ms), C.byref(n)), self._h)
        return ms.value, n.value
