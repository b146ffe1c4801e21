"""Cost of polygon apertures on the C2 workload (LHC, 1 M particles x 40 turns, fast kernels):

    (a) C2 as it is (LimitRect after the high-order multipoles, LimitEllipse after the quadrupoles);
    (b) every LimitRect replaced by its 4-vertex LimitPolygon;
    (c) (b) and every LimitEllipse replaced by the 8-vertex octagon inscribed in it;
    (d) C2 plus one 600-vertex polygon (outside the beam): its record makes every chunk of the
        lattice 32 KiB instead of 16 KiB.

Particle-turns/s from CUDA events around the tracking kernels (best of two timed runs after a
two-turn warm-up), a checksum of the survivors, the card's name, power limit and SM clocks.

    python scripts/probe_polygon.py [--out FILE] [--particles N] [--turns T]
"""
import argparse
import json
import math
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


def variants(line):
    import numpy as np

    import xline_b200 as xl

    def rect_poly(e):
        return xl.LimitPolygon(x_vertices=[e.min_x, e.max_x, e.max_x, e.min_x],
                               y_vertices=[e.min_y, e.min_y, e.max_y, e.max_y])

    def octagon(e):
        th = (2 * np.arange(8) + 1) * (math.pi / 8)
        return xl.LimitPolygon(x_vertices=list(e.a * np.cos(th)), y_vertices=list(e.b * np.sin(th)))

    def relined(fn):
        new = xl.Line([fn(e) for e in line.elements], line.element_names)
        new.polygon_apertures = True
        return new

    b = relined(lambda e: rect_poly(e) if type(e).__name__ == "LimitRect" else e)
    kind = {"LimitRect": rect_poly, "LimitEllipse": octagon}
    c = relined(lambda e: kind[type(e).__name__](e) if type(e).__name__ in kind else e)
    th = np.arange(600) * (2 * math.pi / 600)
    r = 0.05 * (1 + 0.05 * np.sin(7 * th))
    d = xl.Line(list(line.elements) + [xl.LimitPolygon(x_vertices=list(r * np.cos(th)),
                                                       y_vertices=list(r * np.sin(th)))],
                list(line.element_names) + ["ngon600"])
    d.polygon_apertures = True
    return [("a_c2", line), ("b_rects_as_polygons", b), ("c_rects_and_ellipses_as_polygons", c),
            ("d_c2_plus_600gon", d)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--particles", type=int, default=1_000_000)
    ap.add_argument("--turns", type=int, default=40)
    args = ap.parse_args()

    import torch

    import xline_b200 as xl
    from xline_b200 import configs, lattice

    if not torch.cuda.is_available():
        raise SystemExit("probe_polygon.py measures on the GPU; no CUDA device found")
    line, cols, p0c, m0 = configs.config_lhc(args.particles)
    result = {"what": __doc__.split("\n\n")[0], "particles": args.particles, "turns": args.turns,
              "gpu": gpu_info(), "cases": []}
    for name, ln in variants(line):
        packed = ln.pack()
        best = 0.0
        for rep in range(2):
            if rep == 0:
                p = xl.Particles(p0c=p0c, mass0=m0, **cols)
                ln.track(p, num_turns=2)
                torch.cuda.synchronize()
            p = xl.Particles(p0c=p0c, mass0=m0, **cols)
            ln.track(p, num_turns=args.turns, timed=True)
            st = ln.last_stats
            best = max(best, int(p.at_turn.sum()) / (st["kernel_ms"] * 1e-3))
        ok = p.state == 1
        chk = float(p.x[ok].double().sum() + p.py[ok].double().sum() + p.zeta[ok].double().sum())
        row = {"case": name, "particle_turns_per_s": best, "alive": int(ok.sum()), "checksum": repr(chk),
               "chunk_words": packed.chunk_words, "polygon_records": packed.record_counts.get(lattice.T_LIMIT_POLYGON, 0),
               "polygon_edges": int(sum(_edges(e) for e in ln.elements)),
               "regs": st["regs_per_thread"], "kernel_ms": st["kernel_ms"]}
        result["cases"].append(row)
        print(json.dumps(row), flush=True)
    base = result["cases"][0]["particle_turns_per_s"]
    for row in result["cases"]:
        row["relative_to_a"] = row["particle_turns_per_s"] / base
    result["gpu_after"] = gpu_info()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


def _edges(e):
    if type(e).__name__ != "LimitPolygon":
        return 0
    y = list(e.y_vertices)
    return sum(1 for k in range(len(y)) if y[k] != y[(k + 1) % len(y)])


if __name__ == "__main__":
    main()
