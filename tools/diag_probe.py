"""GPU probe: cost of the diagnostic radiation call (rcm_diagnose_fluxes) against a time step, and the 2xCO2 forcing of the
ensemble.  65,536 columns on Reduced100 after 5 warm-up steps; medians of synchronous calls (host clock around calls that end
in a stream synchronise), (a) and (b) alternated in one loop:
  (a) rcm_advance(1)
  (b) rcm_diagnose_fluxes, broadband outputs only
  (c) the same with both spectral outputs [ncol][nwvl][21] into page-locked host buffers (2.2 GB: bound by the copy)
python tools/diag_probe.py [ncol]"""
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
CO2_2X = [1.0, 2.0, 1.0, 1.0, 1.0]  # active species of the default mask: H2O, CO2, O3, N2O, CH4


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def main():
    import torch  # page-locked host buffers for (c)

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
    spec = [torch.empty(ncol * nw * 21, dtype=torch.float64, pin_memory=True) for _ in range(2)]

    def diag(spectral):
        sp = [C.c_void_p(t.data_ptr()) if spectral else None for t in spec]
        rcm.capi._check(L.rcm_diagnose_fluxes(s._h, C.c_int(0), C.c_int(ncol), None, sp[0], sp[1],
                                              rcm.capi._p(Ed), rcm.capi._p(Eu), rcm.capi._p(dE)), s._h)

    for _ in range(3):  # warm-up of every timed call
        s.advance(1)
        diag(False)
        diag(True)
    ta, tb = [], []
    for _ in range(25):
        ta.append(timed(lambda: s.advance(1)))
        tb.append(timed(lambda: diag(False)))
    tc = [timed(lambda: diag(True)) for _ in range(20)]
    a, b, c = statistics.median(ta), statistics.median(tb), statistics.median(tc)
    one = s.diagnose_fluxes(spectral=False)
    two = s.diagnose_fluxes(vmr_scale=CO2_2X, spectral=False)
    irf_toa = float(np.mean(one["E_up"][:, 0] - two["E_up"][:, 0]))
    irf_sfc = float(np.mean(two["E_down"][:, 20] - one["E_down"][:, 20]))
    print(f"# tools/diag_probe.py on {card} (name, power limit); {ncol} columns, Reduced100 ({nw} wavelengths), after 5 + 3 steps")
    print(f"(a) rcm_advance(1)                       median of {len(ta)}: {a:8.3f} ms  (min {min(ta):.3f}, max {max(ta):.3f})")
    print(f"(b) rcm_diagnose_fluxes, broadband       median of {len(tb)}: {b:8.3f} ms  (min {min(tb):.3f}, max {max(tb):.3f})"
          f"  = {b / a:.3f} x (a)")
    print(f"(c) the same + spectral into pinned host median of {len(tc)}: {c:8.3f} ms  (min {min(tc):.3f}, max {max(tc):.3f})"
          f"  = {c / a:.3f} x (a), {2 * ncol * nw * 21 * 8 / 1e9:.2f} GB copied")
    print(f"ensemble mean OLR {float(np.mean(one['E_up'][:, 0])):.10f} W/m2; 2xCO2 instantaneous forcing: TOA {irf_toa:.10f} W/m2, "
          f"surface E_down {irf_sfc:+.10f} W/m2")
    s.close()


if __name__ == "__main__":
    main()
