"""GPU probe: cost of the adjusted-forcing call (rcm_adjusted_forcing) against a time step and the flux-Jacobian call, and
the ensemble-mean stratosphere-adjusted forcing of doubled CO2.  65,536 columns on Reduced100 after 5 warm-up steps; medians of
synchronous calls (host clock around calls that end in a stream synchronise), (a), (b) and (c) alternated in one loop:
  (a) rcm_advance(1)
  (b) rcm_flux_jacobian, dE_jac [ncol][20][41] only
  (c) rcm_adjusted_forcing, 2xCO2, ntrop = 4 (layers 0..3, 0-200 hPa), tol 1e-6 W/m2, at most 20 Newton updates; all outputs
The histogram of the Newton updates (iters) and the ensemble means of IRF, SARF and the adjustment of every layer are those of
the first call of (c), at the state after the 5 warm-up steps (the timed loop advances the ensemble further).
python tools/forcing_probe.py [ncol]"""
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
NLAY, NLEV, NE = 20, 21, 41
NTROP = 4
CO2_2X = np.array([1.0, 2.0, 1.0, 1.0, 1.0])


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
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(os.path.join(G, "Reduced100Forcing.rcmtab")))
    s.set_columns(pl, st["Tlayer"], np.full(ncol, 288.2), st["vmr9"], st["rel_hum"])
    s.advance(5)
    nw = s.nwvl
    L = rcm.load_library()
    P = rcm.capi._p
    Hj = np.zeros((ncol, NLAY, NE))
    ntrop = np.full(ncol, NTROP, dtype=np.int32)
    F, dT = np.zeros((ncol, 4)), np.zeros((ncol, NLAY))
    Ed, Eu = np.zeros((ncol, NLEV)), np.zeros((ncol, NLEV))
    iters = np.zeros(ncol, dtype=np.int32)

    def fjac():
        rcm.capi._check(L.rcm_flux_jacobian(s._h, C.c_int(0), C.c_int(ncol), None, None, P(Hj)), s._h)

    def fdh():
        rcm.capi._check(L.rcm_adjusted_forcing(s._h, C.c_int(0), C.c_int(ncol), P(CO2_2X), P(ntrop), C.c_double(1e-6),
                                               C.c_int(20), P(F), P(dT), P(Ed), P(Eu), P(iters)), s._h)

    fdh()  # the state after 5 steps: the physics printed below
    F0, dT0, iters0 = F.copy(), dT.copy(), iters.copy()
    for _ in range(2):  # warm-up of every timed call
        s.advance(1)
        fjac()
        fdh()
    ta, tb, tc = [], [], []
    for _ in range(7):
        ta.append(timed(lambda: s.advance(1)))
        tb.append(timed(fjac))
        tc.append(timed(fdh))
    a, b, c = statistics.median(ta), statistics.median(tb), statistics.median(tc)
    print(f"# tools/forcing_probe.py on {card} (name, power limit); {ncol} columns, Reduced100 ({nw} wavelengths), "
          f"timed from the state after 5 + 2 steps")
    print(f"(a) rcm_advance(1)                       median of {len(ta)}: {a:9.3f} ms  (min {min(ta):.3f}, max {max(ta):.3f})")
    print(f"(b) rcm_flux_jacobian, dE_jac only       median of {len(tb)}: {b:9.3f} ms  (min {min(tb):.3f}, max {max(tb):.3f})"
          f"  = {b / a:.2f} x (a)")
    print(f"(c) rcm_adjusted_forcing, 2xCO2, ntrop 4 median of {len(tc)}: {c:9.3f} ms  (min {min(tc):.3f}, max {max(tc):.3f})"
          f"  = {c / a:.2f} x (a), {c / b:.3f} x (b)")
    print("the first call of (c), at the state after 5 steps:")
    hist = {int(k): int(v) for k, v in zip(*np.unique(iters0, return_counts=True))}
    print(f"Newton updates per column (iters: columns; -1 = not converged): {hist}")
    # a chunk (8,192 columns) iterates until its last column is frozen: its fjac launches are the largest entry
    chunk_max = [int(np.where(iters0[k:k + 8192] < 0, 20, iters0[k:k + 8192]).max()) for k in range(0, ncol, 8192)]
    print(f"Newton updates of each 8,192-column chunk (its slowest column): {chunk_max}")
    mean = F0.mean(axis=0)
    print(f"ensemble means (W/m2): IRF_toa {mean[0]:.6f}  IRF_trop {mean[1]:.6f}  SARF_toa {mean[2]:.6f}  SARF_trop {mean[3]:.6f}")
    player = (pl[:NLAY] + pl[1:]) / 2.0
    print("layer  p_layer/hPa  mean dT_adj (K)")
    for l in range(NLAY):
        print(f"{l:5d}  {player[l]:11.3f}  {dT0[:, l].mean():15.6f}")
    s.close()


if __name__ == "__main__":
    main()
