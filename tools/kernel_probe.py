"""GPU probe: cost of the radiative-kernel call (rcm_radiative_kernels) against a time step and the broadband diagnostic
call, and the ensemble-mean kernels.  65,536 columns on Reduced100 after 5 warm-up steps; medians of synchronous calls (host
clock around calls that end in a stream synchronise), (a), (b) and (c) alternated in one loop:
  (a) rcm_advance(1)
  (b) rcm_diagnose_fluxes, broadband outputs only
  (c) rcm_radiative_kernels, K [ncol][2][41] only
python tools/kernel_probe.py [ncol]"""
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
NLAY = 20


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
    Ed, Eu, dE = np.zeros((ncol, 21)), np.zeros((ncol, 21)), np.zeros((ncol, 20))
    K = np.zeros((ncol, 2, 2 * NLAY + 1))

    def diag():
        rcm.capi._check(L.rcm_diagnose_fluxes(s._h, C.c_int(0), C.c_int(ncol), None, None, None, rcm.capi._p(Ed),
                                              rcm.capi._p(Eu), rcm.capi._p(dE)), s._h)

    def kern():
        rcm.capi._check(L.rcm_radiative_kernels(s._h, C.c_int(0), C.c_int(ncol), None, None, rcm.capi._p(K)), s._h)

    for _ in range(3):  # warm-up of every timed call
        s.advance(1)
        diag()
        kern()
    ta, tb, tc = [], [], []
    for _ in range(20):
        ta.append(timed(lambda: s.advance(1)))
        tb.append(timed(diag))
        tc.append(timed(kern))
    a, b, c = statistics.median(ta), statistics.median(tb), statistics.median(tc)
    d = s.radiative_kernels()
    planck = float(np.mean(d["dOLR_dT"].sum(axis=1) + d["dOLR_dTs"]))
    wv = float(np.mean(d["dOLR_dlnq"].sum(axis=1)))
    print(f"# tools/kernel_probe.py on {card} (name, power limit); {ncol} columns, Reduced100 ({nw} wavelengths), after 5 + 3 steps")
    print(f"(a) rcm_advance(1)                  median of {len(ta)}: {a:8.3f} ms  (min {min(ta):.3f}, max {max(ta):.3f})")
    print(f"(b) rcm_diagnose_fluxes, broadband  median of {len(tb)}: {b:8.3f} ms  (min {min(tb):.3f}, max {max(tb):.3f})"
          f"  = {b / a:.3f} x (a)")
    print(f"(c) rcm_radiative_kernels, K only   median of {len(tc)}: {c:8.3f} ms  (min {min(tc):.3f}, max {max(tc):.3f})"
          f"  = {c / a:.3f} x (a), {c / b:.3f} x (b)")
    print(f"ensemble means: Planck response sum_l dOLR/dT_l + dOLR/dT_s {planck:.10f} W/m2/K, dOLR/dT_s "
          f"{float(np.mean(d['dOLR_dTs'])):.10f} W/m2/K, sum_l dOLR/dln q_l {wv:.10f} W/m2, sum_l dSFC/dT_l "
          f"{float(np.mean(d['dSFC_dT'].sum(axis=1))):.10f} W/m2/K, sum_l dSFC/dln q_l {float(np.mean(d['dSFC_dlnq'].sum(axis=1))):.10f} W/m2")
    s.close()


if __name__ == "__main__":
    main()
