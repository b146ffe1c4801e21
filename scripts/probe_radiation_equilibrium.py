"""Cost of the radiation equilibrium from the tangent map and the envelope (DESIGN.md §4.10): the wall
time and Newton iterations of ``xl.radiation_equilibrium`` on the damping ring of the radiation tests,
``config_petra_like`` and C4 (PETRA IV), and the rate of ``tangent_kernel_radiation`` against
``tangent_kernel`` on C4 (mean-mode radiation on and off).

Wall times are host clocks around the whole call (it ends in a device synchronisation: the orbit is
read back every Newton step); one untimed call first.  Kernel rates from CUDA events around one
``track_tangent`` call each (best of two after a one-turn warm-up).  The card's name, power limit
and SM clocks are read in the same call.

    python scripts/probe_radiation_equilibrium.py [--out profiles/radiation_equilibrium.json]
        [--particles N] [--turns T]
"""
import argparse
import json
import math
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from probe_radiation import gpu_info  # noqa: E402


def _damping_ring():
    import xline_b200 as xl
    from xline_b200 import configs, optics

    theta, els = 0.2, []
    for c in range(8):
        for sgn in (1.0, -1.0):
            els += [xl.Multipole(knl=[0.0, sgn * 0.35], ksl=[0.0, 0.0], length=0.3), xl.DriftExact(length=1.0),
                    xl.Drift(length=0.5), xl.Multipole(knl=[theta, 0.01], ksl=[0.0, 0.0], hxl=theta, length=1.5),
                    xl.DriftExact(length=1.0)]
    u0 = optics.radiation_integrals(xl.Line(els), 6e9, configs.ELECTRON_MASS_EV)["U0"]
    els.append(xl.Cavity(voltage=3 * u0, frequency=5e8, lag=180.0 - math.degrees(math.asin(1 / 3))))
    return xl.Line(els), 6e9, configs.ELECTRON_MASS_EV


def _lpm(cfg):
    line, _, p0c, m0 = cfg
    return line, p0c, m0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--particles", type=int, default=100_000)
    ap.add_argument("--turns", type=int, default=100)
    args = ap.parse_args()

    import numpy as np
    import torch

    import xline_b200 as xl
    from xline_b200 import configs, optics

    if not torch.cuda.is_available():
        raise SystemExit("probe_radiation_equilibrium.py measures on the GPU; no CUDA device found")
    result = {"what": __doc__.split("\n\n")[0], "gpu": gpu_info(), "equilibrium": [], "tangent_rate": {}}
    cases = (("damping_ring", _damping_ring),
             ("petra_like", lambda: _lpm(configs.config_petra_like(n=1))),
             ("C4_petra4", lambda: _lpm(configs.config_petra4(n=1))))
    for name, make in cases:
        line, p0c, m0 = make()
        line.radiation = "mean"
        p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=np.zeros(1))
        xl.radiation_equilibrium(line, p)  # packs and uploads the lattice, loads the kernels
        t0 = time.perf_counter()
        eq = xl.radiation_equilibrium(line, p)
        wall = time.perf_counter() - t0
        r = optics.radiation_integrals(line, p0c, m0)
        row = {"config": name, "elements": len(line.elements), "wall_s": wall, "newton_iterations": eq.iterations,
               "orbit": eq.orbit.tolist(), "damping_times_turns": eq.damping_times.tolist(),
               "integrals_tau": [r["tau_x"], r["tau_y"], r["tau_z"]], "partition": eq.partition.tolist(),
               "partition_sum": float(eq.partition.sum()), "tunes": eq.tunes.tolist(),
               "emittances": eq.emittances.tolist(), "integrals_eps_x": r["eps_x"],
               "sigma_delta": eq.sigma_delta, "integrals_sigma_delta": r["sigma_delta"],
               "sigma_zeta": eq.sigma_zeta, "energy_loss_eV": eq.energy_loss, "integrals_U0_eV": r["U0"]}
        result["equilibrium"].append(row)
        print(json.dumps(row), flush=True)

    line, cols, p0c, m0 = configs.config_petra4(args.particles)
    for rad in (None, "mean"):
        line.radiation = rad
        best = 0.0
        for rep in range(3):
            p = xl.Particles(p0c=p0c, mass0=m0, **cols)
            t = xl.TangentMap(args.particles, device=p.x.device)
            turns = 1 if rep == 0 else args.turns
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            line.track_tangent(p, t, num_turns=turns, radiation=rad is not None)
            b.record()
            torch.cuda.synchronize()
            if rep:
                best = max(best, args.particles * turns / (a.elapsed_time(b) * 1e-3))
        result["tangent_rate"]["radiation_%s" % rad] = {"particle_turns_per_s": best, "alive": int((p.state == 1).sum()),
                                                       "particles": args.particles, "turns": args.turns}
        print(json.dumps({rad or "off": best}), flush=True)
    off, on = (result["tangent_rate"]["radiation_%s" % k]["particle_turns_per_s"] for k in ("None", "mean"))
    result["tangent_rate"]["radiation_over_off"] = on / off
    result["gpu_after"] = gpu_info()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
