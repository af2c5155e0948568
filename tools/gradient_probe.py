"""Cost of the adjoint flux-gradient calls (rcm_flux_gradient, rcm_lbl_flux_gradient) beside a step, the radiative kernels and
the two Jacobian calls a gradient otherwise needs (flux_jacobian + species_jacobian, contracted on the host).
  repwvl: 65,536 columns on Reduced100 after 5 steps.
  LBL:    the bench.py LBL workload, 4,096 columns x 20,000 synthetic wavelengths after 2 steps, with the LBL calls.
Medians of synchronous calls (host clock around calls that return after a stream synchronise), the calls alternated, after one
warm-up of each; then one more call of each under torch.profiler (a separate run) for the device time of the calls' main
kernels.  The cotangents are seeded normal numbers on every level's fluxes and heating rates.  Prints the card's name and power
limit read in the same run.

    python tools/gradient_probe.py [--ncol 65536] [--lbl-ncol 4096] [--lbl-nwvl 20000] [--reps 5] [--out FILE]
"""
import argparse
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))
import our_first_climate_model_b200 as rcm  # noqa: E402
from lbl_diag_probe import lbl_case  # noqa: E402
from species_jacobian_probe import alternate  # noqa: E402

G = os.path.join(os.path.dirname(ROOT), "tests", "golden")


def kernel_ms(fn, names):
    """device time (ms) of each kernel named in names over one call of fn, summed over its launches (torch.profiler, CUDA)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot = {n: 0.0 for n in names}
    for e in prof.events():
        for n in names:
            if re.search(n + "[<I(]", e.name):  # demangled (templated or not) or mangled
                tot[n] += e.device_time / 1e3
    return tot


def cotangents(n, seed):
    r = np.random.default_rng(seed)
    return dict(w_E_down=r.normal(size=(n, 21)), w_E_up=r.normal(size=(n, 21)), w_dE=r.normal(size=(n, 20)))


def step(s):
    """one step, synchronised (the steps of the alternation move the state the other calls differentiate: fine for timing)"""
    s.advance(1, want_scalars=False)
    s.synchronize()


def report(lines, t, k, kernels):
    ref = t["flux_jacobian"][0] + t["species_jacobian"][0]
    for name, (med, mn) in t.items():
        lines.append(f"  {name:18s} median {med:10.2f} ms   min {mn:10.2f} ms")
    lines.append(f"  gradient / (flux_jacobian + species_jacobian) = {t['gradient'][0]:.2f} / {ref:.2f} ms = "
                 f"{t['gradient'][0] / ref:.4f}")
    lines.append("  kernel device time (torch.profiler, one call each): " +
                 ", ".join(f"{n} {k[n]:.2f} ms" for n in kernels))


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
    w = cotangents(a.ncol, 1)
    calls = {"gradient": lambda: s.flux_gradient(**w), "radiative_kernels": lambda: s.radiative_kernels(),
             "flux_jacobian": lambda: s.flux_jacobian(), "species_jacobian": lambda: s.species_jacobian(),
             "step": lambda: step(s)}
    t = alternate(calls, a.reps)
    lines.append(f"repwvl: {a.ncol} columns x {s.nwvl} wavelengths (Reduced100, after 5 steps), {a.reps} alternated reps")
    names = ["rcm_grad_rt_kernel", "rcm_grad_sum_kernel", "rcm_jac_rt_kernel", "rcm_fjac_kernel", "rcm_species_fjac_kernel"]
    k = {**kernel_ms(calls["gradient"], names[:2]), **kernel_ms(calls["radiative_kernels"], names[2:3]),
         **kernel_ms(calls["flux_jacobian"], names[3:4]), **kernel_ms(calls["species_jacobian"], names[4:])}
    report(lines, t, k, names)
    s.close()

    # line-by-line
    c = lbl_case(a.lbl_ncol, a.lbl_nwvl, 4242)
    s = rcm.Solver(0)
    s.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
    st = c["st"]
    s.set_columns(c["pl"], st["Tlayer"], c["Tsurf"], st["vmr9"], st["rel_hum"])
    s.advance(2)
    w = cotangents(a.lbl_ncol, 2)
    lreps = max(1, min(a.reps, 3))
    calls = {"gradient": lambda: s.lbl_flux_gradient(**w), "radiative_kernels": lambda: s.lbl_radiative_kernels(),
             "flux_jacobian": lambda: s.lbl_flux_jacobian(), "species_jacobian": lambda: s.lbl_species_jacobian(),
             "step": lambda: step(s)}
    t = alternate(calls, lreps)
    lines.append(f"LBL: {a.lbl_ncol} columns x {a.lbl_nwvl} wavelengths (bench.py LBL case, co2_factor 1, after 2 steps), "
                 f"{lreps} alternated reps")
    names = ["rcm_lbl_grad_kernel", "rcm_grad_sum_kernel", "rcm_lbl_jac_kernel", "rcm_lbl_fjac_kernel",
             "rcm_lbl_species_fjac_kernel"]
    k = {**kernel_ms(calls["gradient"], names[:2]), **kernel_ms(calls["radiative_kernels"], names[2:3]),
         **kernel_ms(calls["flux_jacobian"], names[3:4]), **kernel_ms(calls["species_jacobian"], names[4:])}
    report(lines, t, k, names)
    s.close()
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
