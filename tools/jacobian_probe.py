"""GPU probe: cost of the flux-Jacobian call (rcm_flux_jacobian) against a time step and the radiative-kernel call, and the
ensemble-mean radiative relaxation time of every layer.  65,536 columns on Reduced100 after 5 warm-up steps; medians of
synchronous calls (host clock around calls that end in a stream synchronise), (a), (b) and (c) alternated in one loop:
  (a) rcm_advance(1)
  (b) rcm_radiative_kernels, K [ncol][2][41] only
  (c) rcm_flux_jacobian, dE_jac [ncol][20][41] only
Relaxation time of layer l: -(c_p dp 100 / g) / mean_c(d dE_l/dT_l), c_p = 1004 J/kg/K, g = 9.80665 m/s2 (main.cpp:164-176).
python tools/jacobian_probe.py [ncol]"""
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import our_first_climate_model_b200 as rcm  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
NLAY, NE = 20, 41


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def main():
    ncol = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0]
    atm = rcm.read_atm(os.path.join(G, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(ncol, 12345, pl, atm[:, 2].copy(), atm[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev)
    p = rcm.default_params()
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(os.path.join(G, "Reduced100Forcing.rcmtab")))
    s.set_columns(pl, st["Tlayer"], np.full(ncol, 288.2), st["vmr9"], st["rel_hum"])
    s.advance(5)
    nw = s.nwvl
    L = rcm.load_library()
    K = np.zeros((ncol, 2, NE))
    Hj = np.zeros((ncol, NLAY, NE))

    def kern():
        rcm.capi._check(L.rcm_radiative_kernels(s._h, C.c_int(0), C.c_int(ncol), None, None, rcm.capi._p(K)), s._h)

    def fjac():
        rcm.capi._check(L.rcm_flux_jacobian(s._h, C.c_int(0), C.c_int(ncol), None, None, rcm.capi._p(Hj)), s._h)

    for _ in range(3):  # warm-up of every timed call
        s.advance(1)
        kern()
        fjac()
    ta, tb, tc = [], [], []
    for _ in range(10):
        ta.append(timed(lambda: s.advance(1)))
        tb.append(timed(kern))
        tc.append(timed(fjac))
    a, b, c = statistics.median(ta), statistics.median(tb), statistics.median(tc)
    print(f"# tools/jacobian_probe.py on {card} (name, power limit); {ncol} columns, Reduced100 ({nw} wavelengths), "
          f"after 5 + 3 steps")
    print(f"(a) rcm_advance(1)                  median of {len(ta)}: {a:8.3f} ms  (min {min(ta):.3f}, max {max(ta):.3f})")
    print(f"(b) rcm_radiative_kernels, K only   median of {len(tb)}: {b:8.3f} ms  (min {min(tb):.3f}, max {max(tb):.3f})"
          f"  = {b / a:.3f} x (a)")
    print(f"(c) rcm_flux_jacobian, dE_jac only  median of {len(tc)}: {c:8.3f} ms  (min {min(tc):.3f}, max {max(tc):.3f})"
          f"  = {c / a:.3f} x (a), {c / b:.3f} x (b)")
    dEdT = np.diagonal(Hj[:, :, :NLAY], axis1=1, axis2=2).mean(axis=0)
    mass = 1004.0 * p.dp * 100.0 / 9.80665
    print("layer  p_layer/hPa  mean d dE_l/dT_l (W/m2/K)  relaxation time (days)")
    player = (pl[:NLAY] + pl[1:]) / 2.0
    for l in range(NLAY):
        print(f"{l:5d}  {player[l]:11.3f}  {dEdT[l]:25.10f}  {-mass / dEdT[l] / 86400.0:22.4f}")
    s.close()


if __name__ == "__main__":
    main()
