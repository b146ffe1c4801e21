"""Cost of synchrotron radiation on the two electron-ring workloads: C4 (PETRA IV, 31 025 thin
elements) and its stand-in ``config_petra_like`` (120 cells), each a dynamic-aperture grid, tracked
with radiation off, in mean mode and in quantum mode (DESIGN.md §4.9).

Particle-turns/s from CUDA events around the tracking kernels (best of two timed runs after a
two-turn warm-up), the slowdown against "off", the radiating records per turn, the card's name,
power limit and SM clocks read in the same call.

    python scripts/probe_radiation.py [--out profiles/radiation.json] [--particles N] [--turns T]
"""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), (v.strip() for v in out.split(","))))
    except (OSError, IndexError, subprocess.SubprocessError) as exc:
        return {"error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--particles", type=int, default=250_000)
    ap.add_argument("--turns", type=int, default=20)
    args = ap.parse_args()

    import torch

    import xline_b200 as xl
    from xline_b200 import configs, lattice

    if not torch.cuda.is_available():
        raise SystemExit("probe_radiation.py measures on the GPU; no CUDA device found")
    result = {"what": __doc__.split("\n\n")[0], "particles": args.particles, "turns": args.turns,
              "gpu": gpu_info(), "cases": []}
    for cfg, fn in (("C4_petra4", configs.config_petra4), ("petra_like", configs.config_petra_like)):
        line, cols, p0c, m0 = fn(args.particles)
        base = None
        for mode in (None, "mean", "quantum"):
            line.radiation = mode
            packed = line.pack()
            best = 0.0
            for rep in range(3):
                p = xl.Particles(p0c=p0c, mass0=m0, **cols)
                line.track(p, num_turns=2 if rep == 0 else args.turns, timed=rep > 0)
                if rep == 0:
                    torch.cuda.synchronize()
                    continue
                st = line.last_stats
                best = max(best, args.particles * args.turns / (st["kernel_ms"] * 1e-3))
            ok = p.state == 1
            row = {"config": cfg, "radiation": mode, "particle_turns_per_s": best, "alive": int(ok.sum()),
                   "records": int(sum(packed.record_counts.values())),
                   "radiating_records": packed.record_counts.get(lattice.T_MULTIPOLE_RAD, 0),
                   "chunks": packed.n_chunks, "regs": st["regs_per_thread"], "kernel_ms": st["kernel_ms"]}
            if base is None:
                base = best
            row["relative_to_off"] = best / base
            result["cases"].append(row)
            print(json.dumps(row), flush=True)
    result["gpu_after"] = gpu_info()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
