"""Cost of tangent-map tracking (Line.track_tangent, csrc/tangent.cu) next to Line.track.

1. Particle-turns per second of track_tangent and of track, measured in the same run, alternating,
   on C2 (LHC with apertures; 1e5 particles x 100 turns) and on C5 (PS Booster with 120
   space-charge kicks; 1e5 particles x 20 turns): one warm-up call each, then `--reps` timed calls
   on fresh copies of the beam (host clock around the call, ending in a synchronise).
2. Registers per thread and the resident warps per SM they allow (ptxas report of the build).
3. An FLI map: 1e5 particles on an (x, y) amplitude grid x 1000 turns of the LHC lattice.

The card's name, power limit and clocks are read in the same run.

    python scripts/probe_tangent.py [--out FILE] [--reps R]
"""
import argparse
import json
import os
import re
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from probe_polygon import gpu_info  # noqa: E402


def _timed(fn):
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def compare(name, line, cols, p0c, m0, turns, reps):
    import numpy as np

    import xline_b200 as xl

    def beam():
        return xl.Particles(p0c=p0c, mass0=m0, device="cuda:0", **{k: np.asarray(v) for k, v in cols.items()})

    n = len(cols["x"])
    out = {"particles": n, "turns": turns, "track_s": [], "track_tangent_s": []}
    for rep in range(reps + 1):
        p, q = beam(), beam()
        t = xl.TangentMap(n, "cuda:0")
        a = _timed(lambda: line.track(p, num_turns=turns))
        b = _timed(lambda: line.track_tangent(q, t, num_turns=turns))
        if rep:  # rep 0 warms up (module load, packing, lattice upload)
            out["track_s"].append(a)
            out["track_tangent_s"].append(b)
        out["survivors_track"], out["survivors_tangent"] = int(p.state.sum()), int(q.state.sum())
    for k in ("track", "track_tangent"):
        best = min(out[k + "_s"])
        out[k + "_particle_turns_per_s"] = n * turns / best
    out["ratio_tangent_over_track_time"] = min(out["track_tangent_s"]) / min(out["track_s"])
    print(name, json.dumps({k: v for k, v in out.items() if not k.endswith("_s")}))
    return out


def registers():
    from xline_b200 import build

    txt = build.ptxas_report().get("tangent", "")
    m = re.search(r"tangent_kernel\S*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                  r"ptxas info\s*: Used (\d+) registers", txt)
    if not m:
        return {"error": "no ptxas report"}
    stack, st, ld, regs = (int(v) for v in m.groups())
    per_thread = (regs + 7) // 8 * 8  # allocation granule of 8 registers per thread (256 per warp)
    warps = min(64, 65536 // (per_thread * 32))
    ctas = warps // 4  # 128-thread CTAs, the default launch
    return {"registers": regs, "stack_bytes": stack, "spill_store_bytes": st, "spill_load_bytes": ld,
            "resident_ctas_per_sm_128_threads": ctas, "resident_warps_per_sm": 4 * ctas,
            "occupancy": 4 * ctas / 64}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch

    import xline_b200 as xl
    from xline_b200 import configs

    res = {"gpu": gpu_info(), "kernel": registers()}
    line, cols, p0c, m0 = configs.config_lhc(100_000)
    res["c2_lhc_apertures"] = compare("C2", line, cols, p0c, m0, 100, args.reps)
    line5, cols5, p0c5, m05 = configs.config_psb(100_000)
    res["c5_psb_spacecharge"] = compare("C5", line5, cols5, p0c5, m05, 20, args.reps)
    # FLI map
    side = 317
    gx, gy = np.meshgrid(np.linspace(1e-5, 1e-3, side), np.linspace(1e-5, 1e-3, side))  # to 10 sigma
    n = 100_000
    z = dict(x=gx.ravel()[:n], y=gy.ravel()[:n])
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda:0", **z)
    t = xl.TangentMap(n, "cuda:0")
    line.track_tangent(xl.Particles(p0c=p0c, mass0=m0, device="cuda:0", x=[1e-4]), xl.TangentMap(1, "cuda:0"))
    dt = _timed(lambda: line.track_tangent(p, t, num_turns=1000))
    fli = t.fli.cpu().numpy()
    alive = p.state.cpu().numpy() == 1
    res["fli_map_lhc"] = {"particles": n, "turns": 1000, "seconds": dt, "particle_turns_per_s": n * 1000 / dt,
                          "survivors": int(alive.sum()),
                          "fli_quantiles_survivors": [float(v) for v in np.quantile(fli[alive], [0.1, 0.5, 0.9])]
                          if alive.any() else None}
    print("FLI map", json.dumps(res["fli_map_lhc"]))
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
