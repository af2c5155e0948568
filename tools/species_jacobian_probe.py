"""Cost of the species-Jacobian calls (rcm_species_jacobian, rcm_lbl_species_jacobian) against the flux Jacobian of the same
path, and the linearised 2xCO2 instantaneous forcing they give beside the exact one.
  repwvl: 65,536 columns on Reduced100 after 5 steps; species_jacobian and flux_jacobian alternated.
  LBL:    the bench.py LBL workload, 4,096 columns x 20,000 synthetic wavelengths after 2 steps; the same two calls alternated.
Medians of synchronous calls (host clock around calls that return after a stream synchronise), after one warm-up of each;
then one more call of each under torch.profiler for the device time of the Jacobian kernels alone.
Linearised IRF at level k: ln 2 x sum_l d(E_down[k] - E_up[k])/dln x_{CO2,l}; exact: the difference of two diagnose calls
(CO2 x2 and unscaled).  TOA is level 0, the tropopause level 4.  Prints the card's name and power limit read in the same run.

    python tools/species_jacobian_probe.py [--ncol 65536] [--lbl-ncol 4096] [--lbl-nwvl 20000] [--reps 5] [--out FILE]
"""
import argparse
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))
import our_first_climate_model_b200 as rcm  # noqa: E402
from lbl_diag_probe import lbl_case  # noqa: E402

G = os.path.join(os.path.dirname(ROOT), "tests", "golden")
CO2_2X, NLAY, NTROP = [1.0, 2.0, 1.0, 1.0, 1.0], 20, 4


def alternate(calls, reps):
    for f in calls.values():  # warm-up: modules, scratch allocation
        f()
    times = {k: [] for k in calls}
    for _ in range(reps):
        for k, f in calls.items():
            t0 = time.perf_counter()
            f()
            times[k].append(time.perf_counter() - t0)
    return {k: (1e3 * np.median(v), 1e3 * np.min(v)) for k, v in times.items()}


def kernel_ms(fn, names):
    """device time (ms) of each kernel named in names over one call of fn, summed over its launches (torch.profiler, CUDA)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot = {n: 0.0 for n in names}
    for e in prof.events():
        for n in names:
            if re.search(n + "[<I]", e.name):  # demangled or mangled
                tot[n] += e.device_time / 1e3
    return tot


def irf_lines(J, up2, up1, dn2, dn1):
    """ensemble-mean linearised and exact IRF at TOA and at the tropopause"""
    co2 = J[..., NLAY:2 * NLAY].sum(axis=-1)          # [ncol][2][21]
    lin = np.log(2.0) * (co2[:, 0] - co2[:, 1])       # d(E_down - E_up)
    exact = (dn2 - up2) - (dn1 - up1)
    return [f"2xCO2 IRF at {name} (level {k}): linearised {lin[:, k].mean():.6f} W/m2, exact {exact[:, k].mean():.6f} W/m2"
            for name, k in (("TOA", 0), ("the tropopause", NTROP))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=65536)
    ap.add_argument("--lbl-ncol", type=int, default=4096)
    ap.add_argument("--lbl-nwvl", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the report here")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    lines = [f"card: {card}"]

    # repwvl
    atm = rcm.read_atm(os.path.join(G, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(a.ncol, 12345, pl, atm[:, 2].copy(), atm[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev)
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(os.path.join(G, "Reduced100Forcing.rcmtab")))
    s.set_columns(pl, st["Tlayer"], np.full(a.ncol, 288.2), st["vmr9"], st["rel_hum"])
    s.advance(5)
    t = alternate({"species_jacobian": lambda: s.species_jacobian(), "flux_jacobian": lambda: s.flux_jacobian()}, a.reps)
    lines.append(f"repwvl: {a.ncol} columns x {s.nwvl} wavelengths (Reduced100, after 5 steps), {a.reps} alternated reps")
    for k, (med, mn) in t.items():
        lines.append(f"  {k:17s} median {med:10.2f} ms   min {mn:10.2f} ms   {med / t['flux_jacobian'][0]:6.3f} x flux_jacobian")
    k = {**kernel_ms(lambda: s.species_jacobian(), ["rcm_species_fjac_kernel"]),
         **kernel_ms(lambda: s.flux_jacobian(), ["rcm_fjac_kernel"])}
    lines.append(f"  kernel device time (torch.profiler, one call): rcm_species_fjac_kernel {k['rcm_species_fjac_kernel']:.2f} ms, "
                 f"rcm_fjac_kernel {k['rcm_fjac_kernel']:.2f} ms "
                 f"({k['rcm_species_fjac_kernel'] / k['rcm_fjac_kernel']:.3f} x); the rest of a call is the prep and the "
                 f"downloads of J and dE_jac ({6200 * 8 * a.ncol / 1e9:.2f} GB against {2542 * 8 * a.ncol / 1e9:.2f} GB)")
    J = s.species_jacobian()["J"]
    d2, d1 = s.diagnose_fluxes(vmr_scale=CO2_2X, spectral=False), s.diagnose_fluxes(spectral=False)
    lines += ["  " + x for x in irf_lines(J, d2["E_up"], d1["E_up"], d2["E_down"], d1["E_down"])]
    s.close()
    del J

    # line-by-line
    c = lbl_case(a.lbl_ncol, a.lbl_nwvl, 4242)
    s = rcm.Solver(0)
    s.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
    st = c["st"]
    s.set_columns(c["pl"], st["Tlayer"], c["Tsurf"], st["vmr9"], st["rel_hum"])
    s.advance(2)
    lreps = max(1, min(a.reps, 3))
    t = alternate({"species_jacobian": lambda: s.lbl_species_jacobian(), "flux_jacobian": lambda: s.lbl_flux_jacobian()}, lreps)
    lines.append(f"LBL: {a.lbl_ncol} columns x {a.lbl_nwvl} wavelengths (bench.py LBL case, co2_factor 1, after 2 steps), "
                 f"{lreps} alternated reps")
    for k, (med, mn) in t.items():
        lines.append(f"  {k:17s} median {med:10.2f} ms   min {mn:10.2f} ms   {med / t['flux_jacobian'][0]:6.3f} x flux_jacobian")
    k = {**kernel_ms(lambda: s.lbl_species_jacobian(), ["rcm_lbl_species_fjac_kernel"]),
         **kernel_ms(lambda: s.lbl_flux_jacobian(), ["rcm_lbl_fjac_kernel"])}
    lines.append(f"  kernel device time (torch.profiler, one call): rcm_lbl_species_fjac_kernel "
                 f"{k['rcm_lbl_species_fjac_kernel']:.2f} ms, rcm_lbl_fjac_kernel {k['rcm_lbl_fjac_kernel']:.2f} ms "
                 f"({k['rcm_lbl_species_fjac_kernel'] / k['rcm_lbl_fjac_kernel']:.3f} x)")
    J = s.lbl_species_jacobian()["J"]
    d2, d1 = s.lbl_diagnose_fluxes(vmr_scale=CO2_2X), s.lbl_diagnose_fluxes()
    lines += ["  " + x for x in irf_lines(J, d2["E_up"], d1["E_up"], d2["E_down"], d1["E_down"])]
    s.close()
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
