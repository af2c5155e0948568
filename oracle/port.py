"""ctypes binding of oracle/liboracle_port.so - the plain-C restatement (rcm_oracle.c).

TEST INFRASTRUCTURE ONLY.  The library is (re)built on demand with gcc.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PATH = os.path.join(_HERE, "liboracle_port.so")
_lib = None
NLAY, NLEV = 20, 21


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Table(C.Structure):
    _fields_ = [("n_tpert", C.c_int), ("n_species", C.c_int), ("n_wvl", C.c_int), ("n_p", C.c_int),
                ("xsec", C.c_void_p), ("wvl", C.c_void_p), ("weight", C.c_void_p), ("p_grid", C.c_void_p),
                ("t_ref", C.c_void_p), ("t_pert", C.c_void_p)]


class SolarParams(C.Structure):
    _fields_ = [("tau_s", C.c_double), ("mu_s", C.c_double), ("g_asym", C.c_double), ("albedo", C.c_double),
                ("daytime", C.c_double), ("E_0", C.c_double), ("doublings", C.c_int)]


class Params(C.Structure):
    _fields_ = [("nlayer", C.c_int), ("nangle", C.c_int), ("cloud_layer", C.c_int), ("cloud_tau", C.c_double),
                ("dp", C.c_double), ("max_dT", C.c_double), ("dt_cap", C.c_double), ("solar_irr", C.c_double)]


def build(force=False):
    src = os.path.join(_HERE, "rcm_oracle.c")
    if force or not os.path.exists(_PATH) or os.path.getmtime(_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "liboracle_port.so"], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_PATH)
        L.rcmo_lowerpos.restype = C.c_long
        L.rcmo_planck.restype = C.c_double
        L.rcmo_planck.argtypes = [C.c_double] * 3
        L.rcmo_magnus.restype = C.c_double
        L.rcmo_magnus.argtypes = [C.c_double]
        L.rcmo_timestep.restype = C.c_double
        L.rcmo_cplkavg.restype = C.c_double
        L.rcmo_cplkavg.argtypes = [C.c_double, C.c_double, C.c_double, C.c_void_p]
        L.rcmo_advance.restype = C.c_int
        L.rcmo_lbl_advance.restype = C.c_int
        _lib = L
    return _lib


def load_rcmtab(path):
    """Read a flat .rcmtab fixture (tools/make_tables.py) -> dict of float64 arrays."""
    with open(path, "rb") as f:
        raw = f.read()
    assert raw[:8] == b"RCMTAB01", "not an .rcmtab file"
    nb, npg, nr, nc = struct.unpack_from("<4Q", raw, 8)
    off = 40
    out = {}
    for name, shape in (("xsec", (nb, npg, nr, nc)), ("wvl", (nr,)), ("weight", (nr,)), ("p_grid", (nc,)),
                        ("t_ref", (nc,)), ("t_pert", (nb,)), ("vmrs_ref", (npg, nc))):
        n = int(np.prod(shape))
        out[name] = np.frombuffer(raw, dtype="<f8", count=n, offset=off).reshape(shape).copy()
        off += 8 * n
    return out


def ctable(tab):
    t = Table(tab["xsec"].shape[0], tab["xsec"].shape[1], tab["xsec"].shape[2], tab["xsec"].shape[3],
              tab["xsec"].ctypes.data, tab["wvl"].ctypes.data, tab["weight"].ctypes.data,
              tab["p_grid"].ctypes.data, tab["t_ref"].ctypes.data, tab["t_pert"].ctypes.data)
    t._keep = tab
    return t


def default_params(solar_irr, cloud_on=True, tau_s=2.0):
    return Params(20, 30, 17 if cloud_on else -1, tau_s / 2.0, 1000.0 / 20, 5.0, 3600.0 * 12, solar_irr)


def solar_setup(tau_s=2.0, mu_s=None, g_asym=0.85, albedo=0.12, daytime=0.5, E_0=1361.0, doublings=20):
    import math
    if mu_s is None:
        mu_s = math.cos(60 * math.pi / 180.0)  # main.cpp:87
    sp = SolarParams(tau_s, mu_s, g_asym, albedo, daytime, E_0, doublings)
    out = np.zeros(7)
    lib().rcmo_solar_setup(C.byref(sp), _p(out))
    return dict(zip(["r_dir", "s_dir", "t_dir", "r", "t", "r_total", "solar_irr"], out))


def lowerpos(a, x):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return int(lib().rcmo_lowerpos(_p(a), C.c_int(len(a)), C.c_double(x)))


def init_columns(plevel, Tlevel, vmr_ppm_level, co2_factor=1.0):
    Tlevel = np.ascontiguousarray(Tlevel, dtype=np.float64).reshape(-1, NLEV)
    ncol = Tlevel.shape[0]
    vm = np.ascontiguousarray(vmr_ppm_level, dtype=np.float64).reshape(ncol, 5, NLEV)
    pl = np.ascontiguousarray(plevel, dtype=np.float64)
    out = dict(Tlayer=np.zeros((ncol, NLAY)), vmr9=np.zeros((ncol, 9, NLAY)), rel_hum=np.zeros((ncol, NLAY)),
               player=np.zeros(NLAY), conv=np.zeros(NLAY))
    lib().rcmo_init_columns(C.c_int(ncol), C.c_int(NLAY), _p(pl), _p(Tlevel), _p(vm), C.c_double(co2_factor),
                            _p(out["Tlayer"]), _p(out["vmr9"]), _p(out["rel_hum"]), _p(out["player"]),
                            _p(out["conv"]))
    return out


def read_tau(tab, plevel, Tlayer, vmr9, cloud_on=True, tau_s=2.0, cloud_layer=17, tau_floor=None):
    """tau [nwvl][20] with the grey cloud in cloud_layer (< 0: none); tau_floor: tau = max(tau, tau_floor) after the cloud,
    the lower clamp the solver's kernels apply where the reference's exp overflows (DESIGN.md section 4)."""
    t = ctable(tab)
    nw = t.n_wvl
    pl = np.ascontiguousarray(plevel, dtype=np.float64)
    T = np.ascontiguousarray(Tlayer, dtype=np.float64)
    v = np.ascontiguousarray(vmr9, dtype=np.float64)
    tau = np.zeros((nw, NLAY)); lp = np.zeros(NLAY, dtype=np.int64); lt = np.zeros(NLAY, dtype=np.int64)
    lib().rcmo_read_tau(C.byref(t), C.c_int(NLEV), _p(pl), _p(T), _p(v), _p(tau), _p(lp), _p(lt))
    if cloud_on:
        lib().rcmo_cloud_into_tau(_p(tau), C.c_int(nw), C.c_int(NLAY), C.c_int(cloud_layer), C.c_double(tau_s / 2.0))
    if tau_floor is not None:
        tau = np.maximum(tau, tau_floor)
    return tau, lp, lt


def radiative_transfer(tau, wvl, weight, Tlayer, T_surface, solar_irr, nangle=30):
    tau = np.ascontiguousarray(tau, dtype=np.float64)
    p = default_params(solar_irr)
    p.nangle = nangle
    Ed = np.zeros(NLEV); Eu = np.zeros(NLEV); dE = np.zeros(NLAY)
    lib().rcmo_radiative_transfer(C.byref(p), C.c_int(tau.shape[0]), _p(tau),
                                  _p(np.ascontiguousarray(wvl, dtype=np.float64)),
                                  _p(np.ascontiguousarray(weight, dtype=np.float64)),
                                  _p(np.ascontiguousarray(Tlayer, dtype=np.float64)), C.c_double(T_surface),
                                  _p(Ed), _p(Eu), _p(dE))
    return Ed, Eu, dE


def advance(tab, plevel, rel_hum, solar_irr, Tlayer, Tsurf, vmr9, nsteps, first_step=0, cloud_on=True,
            time_h=None, want_trace=False, tau_s=2.0, **overrides):
    """overrides: fields of Params (nangle, cloud_layer, max_dT, dt_cap, ...) away from the reference's Consts."""
    t = ctable(tab)
    p = default_params(solar_irr, cloud_on, tau_s)
    for k, v in overrides.items():
        setattr(p, k, v)
    Tl = np.array(Tlayer, dtype=np.float64, order="C").reshape(-1, NLAY)
    ncol = Tl.shape[0]
    Ts = np.array(np.broadcast_to(Tsurf, (ncol,)), dtype=np.float64, order="C")
    v9 = np.array(vmr9, dtype=np.float64, order="C").reshape(ncol, 9, NLAY)
    rh = np.ascontiguousarray(rel_hum, dtype=np.float64).reshape(ncol, NLAY)
    pl = np.ascontiguousarray(plevel, dtype=np.float64)
    th = np.zeros(ncol, dtype=np.float32) if time_h is None else np.array(time_h, dtype=np.float32, order="C")
    Ed = np.zeros((ncol, NLEV)); Eu = np.zeros((ncol, NLEV)); dE = np.zeros((ncol, NLAY)); dt = np.zeros(ncol)
    tr = np.zeros((ncol, nsteps, 24)) if want_trace else None
    nw = lib().rcmo_advance(C.byref(t), C.byref(p), C.c_int(ncol), C.c_int(first_step), C.c_int(nsteps), _p(pl),
                            _p(rh), _p(Tl), _p(Ts), _p(v9), _p(th), _p(Ed), _p(Eu), _p(dE), _p(dt), _p(tr))
    return dict(Tlayer=Tl, Tsurf=Ts, vmr9=v9, time_h=th, E_down=Ed, E_up=Eu, dE=dE, dt=dt, trace=tr, nwvl=nw)


def cplkavg(lo, hi, t):
    st = C.c_int(0)
    v = lib().rcmo_cplkavg(float(lo), float(hi), float(t), C.addressof(st))
    return float(v), st.value


def lbl_bin_edges(wvl):
    wvl = np.ascontiguousarray(wvl, dtype=np.float64)
    lo = np.zeros_like(wvl); hi = np.zeros_like(wvl)
    lib().rcmo_lbl_bin_edges(C.c_int(wvl.size), _p(wvl), _p(lo), _p(hi))
    return lo, hi


def lbl_advance(wvl, tau5, plevel, rel_hum, h2o_ref, o3_scale, co2_factor, solar_irr, Tlayer, Tsurf, h2o, nsteps,
                first_step=0, cloud_on=True, tau_s=2.0):
    p = default_params(solar_irr, cloud_on, tau_s)
    wvl = np.ascontiguousarray(wvl, dtype=np.float64)
    tau5 = np.ascontiguousarray(tau5, dtype=np.float64)
    Tl = np.array(Tlayer, dtype=np.float64, order="C").reshape(-1, NLAY)
    ncol = Tl.shape[0]
    Ts = np.array(np.broadcast_to(Tsurf, (ncol,)), dtype=np.float64, order="C")
    hh = np.array(h2o, dtype=np.float64, order="C").reshape(ncol, NLAY)
    rh = np.ascontiguousarray(rel_hum, dtype=np.float64).reshape(ncol, NLAY)
    o3 = np.ascontiguousarray(o3_scale, dtype=np.float64).reshape(ncol, NLAY)
    href = np.ascontiguousarray(h2o_ref, dtype=np.float64)
    pl = np.ascontiguousarray(plevel, dtype=np.float64)
    Ed = np.zeros((ncol, NLEV)); Eu = np.zeros((ncol, NLEV)); dE = np.zeros((ncol, NLAY)); dt = np.zeros(ncol)
    lib().rcmo_lbl_advance(C.byref(p), C.c_int(wvl.size), _p(wvl), _p(tau5), C.c_int(ncol), C.c_int(first_step),
                           C.c_int(nsteps), _p(pl), _p(rh), _p(href), _p(o3), C.c_double(co2_factor), _p(Tl), _p(Ts),
                           _p(hh), _p(Ed), _p(Eu), _p(dE), _p(dt))
    return dict(Tlayer=Tl, Tsurf=Ts, h2o=hh, E_down=Ed, E_up=Eu, dE=dE, dt=dt)
