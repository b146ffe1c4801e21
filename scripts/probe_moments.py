"""Cost of beam-moment stores (Line.track(..., moments=BeamMoments(...))) on C2 (LHC, 1 M particles
x 40 turns) and C5 (PS Booster with 120 space-charge kicks, 1 M particles x 400 turns):

    none   -- tracking without stores;
    skip1  -- a store on every turn (launches cut to one turn);
    skip10 -- a store every 10 turns.

Wall time of the call from the host clock around it, ending in a device synchronise; two
alternating repeats after a warm-up.  Reduction-kernel time per store from CUDA events around
200 snapshots of the tracked 1 M-particle beam, and from torch.profiler.  A checksum of the
survivors shows that the stores leave the coordinates as they were.  The card's name, power
limit and SM clocks are read in the same run.

    python scripts/probe_moments.py [--out FILE] [--particles N] [--configs c2,c5]
"""
import argparse
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from probe_polygon import gpu_info  # noqa: E402

TURNS = {"c2": 40, "c5": 400}


def _config(name, n):
    from xline_b200 import configs

    return configs.config_lhc(n) if name == "c2" else configs.config_psb(n)


def _checksum(p):
    ok = p.state == 1
    return repr(float(p.x[ok].sum() + p.py[ok].sum() + p.zeta[ok].sum()))


def _reduction_time(p, reps=200):
    import torch

    import xline_b200 as xl

    for _ in range(10):
        xl.beam_moments(p)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        xl.beam_moments(p)
    e1.record()
    e1.synchronize()
    events_us = e0.elapsed_time(e1) * 1e3 / reps
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(50):
            xl.beam_moments(p)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        if "beam_moments" in ev.key:
            kern[ev.key] = getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 50
    return events_us, kern


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--particles", type=int, default=1_000_000)
    ap.add_argument("--configs", default="c2,c5")
    args = ap.parse_args()

    import torch

    import xline_b200 as xl

    if not torch.cuda.is_available():
        raise SystemExit("probe_moments.py measures on the GPU; no CUDA device found")
    result = {"what": __doc__.split("\n\n")[0], "particles": args.particles, "gpu": gpu_info(), "configs": []}
    for name in args.configs.split(","):
        turns = TURNS[name]
        line, cols, p0c, m0 = _config(name, args.particles)
        cases = {"none": None, "skip1": (turns + 1, 1), "skip10": (turns // 10 + 1, 10)}

        def run(case):
            spec = cases[case]
            m = None if spec is None else xl.BeamMoments(spec[0], skip=spec[1])
            p = xl.Particles(p0c=p0c, mass0=m0, **cols)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            line.track(p, num_turns=turns, moments=m)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            return p, m, dt, line.last_stats["kernel_launches"]

        for case in cases:  # warm-up: module loads, pack caches, launch-length schedule
            p = xl.Particles(p0c=p0c, mass0=m0, **cols)
            line.track(p, num_turns=2, moments=None if cases[case] is None else xl.BeamMoments(3))
        rows = {c: {"case": c, "seconds": [], "particle_turns_per_s": []} for c in cases}
        for rep in range(2):
            for case in (cases if rep == 0 else list(cases)[::-1]):
                p, m, dt, launches = run(case)
                r = rows[case]
                r["seconds"].append(dt)
                r["particle_turns_per_s"].append(int(p.at_turn.sum()) / dt)
                r["launches"] = launches
                r["alive"] = int((p.state == 1).sum())
                r["checksum"] = _checksum(p)
                if m is not None:
                    e = m.emittance()
                    r["stores"] = m.num_stores
                    r["last_store"] = {"turn": int(m.turn[-1]), "count": int(m.count[-1]),
                                       "eps_x": float(e["eps_x"][-1]), "eps_y": float(e["eps_y"][-1]),
                                       "neps_x": float(e["neps_x"][-1])}
        base = min(rows["none"]["seconds"])
        for r in rows.values():
            r["relative_time_to_none"] = min(r["seconds"]) / base
        events_us, kern = _reduction_time(p)
        entry = {"config": name, "turns": turns, "cases": list(rows.values()),
                 "same_checksum": len({r["checksum"] for r in rows.values()}) == 1,
                 "reduction_us_per_store_events": events_us, "reduction_kernel_us_profiler": kern}
        result["configs"].append(entry)
        print(json.dumps(entry), flush=True)
    result["gpu_after"] = gpu_info()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
