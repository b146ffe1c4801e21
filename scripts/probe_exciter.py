"""Cost of Exciter records (fast kernels, particle-turns/s from CUDA events around the tracking kernels):

    c2            C2 as it is (LHC with apertures, default kernel);
    c2_ac         C2 + one AC-dipole exciter (order 0) at the start of the line (the polygon twin runs);
    c2_ripple     C2 + one ripple exciter (knl = [0, dk1]) behind every quadrupole;
    c5, c5_ac     C5 (PS Booster with space charge) as it is and with one AC-dipole exciter.

Two repeats, alternating over the cases, each after a two-turn warm-up; the spread of the two is the
noise.  The card's name, power limit and SM clocks are read in the same run, before and after.

    python scripts/probe_exciter.py [--out FILE] [--particles N] [--turns T] [--c5-turns T]
"""
import argparse
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from probe_polygon import gpu_info  # noqa: E402


def cases(particles):
    import math

    import numpy as np
    from scipy.constants import c as clight

    import xline_b200 as xl
    from xline_b200 import configs

    def frev(line, p0c, m0):
        return p0c / math.sqrt(p0c * p0c + m0 * m0) * clight / line.get_length()

    def ac(f, q=0.28):
        return xl.Exciter(knl=[1e-9], samples=np.cos(2 * np.pi * q * np.arange(1000)), sampling_frequency=f, frev=f)

    c2, cols2, p2, m2 = configs.config_lhc(particles)
    f2 = frev(c2, p2, m2)
    c2_ac = xl.Line([ac(f2)] + list(c2.elements), ["ac"] + list(c2.element_names))
    els, names, n_quads = [], [], 0
    ripple = np.sin(2 * np.pi * 0.0371 * np.arange(1000))
    for el, nm in zip(c2.elements, c2.element_names):
        els.append(el)
        names.append(nm)
        if type(el).__name__ == "Multipole" and el.order >= 1 and el.hxl == 0 and float(el.knl[1]) != 0.0:
            els.append(xl.Exciter(knl=[0.0, 1e-6 * float(el.knl[1])], samples=ripple, sampling_frequency=f2, frev=f2))
            names.append(nm + "_ripple")
            n_quads += 1
    c2_ripple = xl.Line(els, names)
    c5, cols5, p5, m5 = configs.config_psb(particles)
    c5_ac = xl.Line([ac(frev(c5, p5, m5))] + list(c5.elements), ["ac"] + list(c5.element_names))
    return n_quads, [("c2", c2, cols2, p2, m2), ("c2_ac", c2_ac, cols2, p2, m2), ("c2_ripple", c2_ripple, cols2, p2, m2),
                     ("c5", c5, cols5, p5, m5), ("c5_ac", c5_ac, cols5, p5, m5)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--particles", type=int, default=1_000_000)
    ap.add_argument("--turns", type=int, default=20)
    ap.add_argument("--c5-turns", type=int, default=20)
    args = ap.parse_args()

    import torch

    import xline_b200 as xl
    from xline_b200 import lattice

    if not torch.cuda.is_available():
        raise SystemExit("probe_exciter.py measures on the GPU; no CUDA device found")
    n_quads, todo = cases(args.particles)
    result = {"what": __doc__.split("\n\n")[0], "particles": args.particles, "turns": args.turns,
              "c5_turns": args.c5_turns, "ripple_exciters": n_quads, "gpu": gpu_info(), "cases": {}}
    for rep in range(2):
        for name, line, cols, p0c, m0 in todo:
            turns = args.c5_turns if name.startswith("c5") else args.turns
            p = xl.Particles(p0c=p0c, mass0=m0, **cols)
            line.track(p, num_turns=2)
            torch.cuda.synchronize()
            p = xl.Particles(p0c=p0c, mass0=m0, **cols)
            line.track(p, num_turns=turns, timed=True)
            st = line.last_stats
            rate = int(p.at_turn.sum()) / (st["kernel_ms"] * 1e-3)
            ok = p.state == 1
            chk = float(p.x[ok].double().sum() + p.py[ok].double().sum() + p.zeta[ok].double().sum())
            packed = line.pack()
            row = result["cases"].setdefault(name, {
                "rates": [], "alive": int(ok.sum()), "checksum": repr(chk), "regs": st["regs_per_thread"],
                "exciter_records": packed.record_counts.get(lattice.T_EXCITER, 0), "chunks": packed.n_chunks,
                "data_words": int(packed.words.size - packed.chunk_words * packed.n_chunks)})
            row["rates"].append(rate)
            print(json.dumps({"case": name, "rep": rep, "particle_turns_per_s": rate}), flush=True)
    for name, row in result["cases"].items():
        r = row["rates"]
        row["particle_turns_per_s"] = max(r)
        row["spread"] = (max(r) - min(r)) / max(r)
        base = result["cases"]["c5" if name.startswith("c5") else "c2"]["particle_turns_per_s"]
        row["relative_to_base"] = row["particle_turns_per_s"] / base
    result["gpu_after"] = gpu_info()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
