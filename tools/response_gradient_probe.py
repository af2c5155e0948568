"""Cost of the climate-response gradient calls (rcm_climate_response_gradient, rcm_lbl_climate_response_gradient) beside the
climate-response calls at the same arguments, and what they say about the ensemble.
  repwvl: 65,536 columns on Reduced100 after 5 steps, 2xCO2, ntrop 4, fixed RH.
  LBL:    the bench.py LBL workload, 4,096 columns x 20,000 synthetic wavelengths after 2 steps, same arguments.
Medians of synchronous calls (host clock around calls that return after a stream synchronise), the two calls alternated
after one warm-up of each; then one more call of each under torch.profiler (a separate run) for the device time of the
adjoint kernel, the flux-Jacobian kernel (the gradient call's extra Jacobian is the difference to the response call) and the
sweep.  As information only: the ensemble means of lambda_trop and of ln 2 sum_l dTs_dlnx[CO2] at zero forcing (the
linearised 2xCO2 warming), beside the call's own 2xCO2 dTs.  Prints the card's name and power limit read in the same run.

    python tools/response_gradient_probe.py [--ncol 65536] [--lbl-ncol 4096] [--lbl-nwvl 20000] [--reps 5] [--out FILE]
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
CO2_2X = [1.0, 2.0, 1.0, 1.0, 1.0]
NTROP = 4


def kernel_ms(fn, names):
    """{name: (device ms summed over its launches, launches)} over one call of fn (torch.profiler, CUDA)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot = {n: [0.0, 0] for n in names}
    for e in prof.events():
        for n in names:
            if re.search(n + "[<I(]", e.name):  # demangled (templated or not) or mangled
                tot[n][0] += e.device_time / 1e3
                tot[n][1] += 1
    return tot


def measure(lines, s, grad, resp, reps, fjac, sweep):
    calls = {"climate_response": lambda: resp(CO2_2X, NTROP), "gradient": lambda: grad(CO2_2X, NTROP)}
    t = alternate(calls, reps)
    for name, (med, mn) in t.items():
        lines.append(f"  {name:17s} median {med:10.2f} ms   min {mn:10.2f} ms")
    lines.append(f"  gradient / climate_response = {t['gradient'][0]:.2f} / {t['climate_response'][0]:.2f} ms = "
                 f"{t['gradient'][0] / t['climate_response'][0]:.3f}")
    names = ["rcm_ecs_adjoint_kernel", fjac, sweep, "rcm_grad_sum_kernel"]
    kg, kr = kernel_ms(calls["gradient"], names), kernel_ms(calls["climate_response"], names)
    lines.append("  kernel device time (torch.profiler, one gradient call): " +
                 ", ".join(f"{n} {kg[n][0]:.2f} ms ({kg[n][1]} launches)" for n in names))
    lines.append(f"  {fjac} in the response call: {kr[fjac][0]:.2f} ms ({kr[fjac][1]} launches); the gradient's extra "
                 f"Jacobian {kg[fjac][0] - kr[fjac][0]:.2f} ms")
    z = grad(None, NTROP)
    d = grad(CO2_2X, NTROP)
    ok = z["converged"] & d["converged"]
    lin = np.log(2.0) * z["dTs_dlnx"][:, 1].sum(axis=1)
    lines.append(f"  zero forcing (information only): mean lambda_trop {z['lambda_trop'][ok].mean():.6f} K/(W/m2), "
                 f"linearised 2xCO2 warming ln2 sum_l dTs/dln x_CO2 {lin[ok].mean():.6f} K; the call's 2xCO2 dTs "
                 f"{d['dTs'][ok].mean():.6f} K ({int(ok.sum())} columns)")


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
    lines.append(f"repwvl: {a.ncol} columns x {s.nwvl} wavelengths (Reduced100, after 5 steps), 2xCO2, ntrop {NTROP}, "
                 f"fixed RH, tol 1e-6 W/m2; {a.reps} alternated reps")
    measure(lines, s, s.climate_response_gradient, s.climate_response, a.reps, "rcm_fjac_kernel", "rcm_grad_rt_kernel")
    s.close()

    # line-by-line
    c = lbl_case(a.lbl_ncol, a.lbl_nwvl, 4242)
    s = rcm.Solver(0)
    s.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
    st = c["st"]
    s.set_columns(c["pl"], st["Tlayer"], c["Tsurf"], st["vmr9"], st["rel_hum"])
    s.advance(2)
    lreps = max(1, min(a.reps, 2))
    lines.append(f"LBL: {a.lbl_ncol} columns x {a.lbl_nwvl} wavelengths (bench.py LBL case, co2_factor 1, after 2 steps), "
                 f"same arguments; {lreps} alternated reps")
    measure(lines, s, s.lbl_climate_response_gradient, s.lbl_climate_response, lreps, "rcm_lbl_fjac_kernel",
            "rcm_lbl_grad_kernel")
    s.close()
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
