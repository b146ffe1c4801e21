"""Measure the beam-field kicks and field Jacobians of every kernel against the 34-digit reference
on the point sets of tests/test_gpu_beamfield_accuracy.py, and write the maxima per configuration
and kernel, next to the float64 oracle's, to profiles/beamfield_accuracy.json (or --out).

    python scripts/probe_beamfield_accuracy.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "beamfield_accuracy.json"))
    args = ap.parse_args()
    import torch

    from tests import test_gpu_beamfield_accuracy as G

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    t0 = time.time()
    kicks, worst = {}, {}
    for cfg in G.CONFIGS:
        res = G.measure(cfg)
        kicks[cfg[0]] = {k: (float("%.3g" % v) if isinstance(v, float) else v) for k, v in res.items()}
        for k, v in res.items():
            if isinstance(v, float):
                worst[k] = max(worst.get(k, 0.0), v)
        print(cfg[0], kicks[cfg[0]], flush=True)
    tangent = {}
    for cfg in G.TAN_CONFIGS:
        rxy, rz = G.measure_tangent(cfg)
        tangent[cfg[0]] = {"xy": float("%.3g" % rxy), "zeta": float("%.3g" % rz)}
        worst["tangent_xy"] = max(worst.get("tangent_xy", 0.0), rxy)
        worst["tangent_zeta"] = max(worst.get("tangent_zeta", 0.0), rz)
        print(cfg[0], tangent[cfg[0]], flush=True)
    out = {
        "what": "max over particles of |kick - kick_ref| / (|fact| (|lambda| T + Lambda |E|)) per configuration "
                "and kernel (tests/test_gpu_beamfield_accuracy.py); 'oracle' is the float64 NumPy/scipy oracle on "
                "the same particles; tangent: the px, py rows of Line.track_tangent against the reference "
                "derivatives over their term scale",
        "gpu": gpu,
        "torch": torch.__version__,
        "seconds": round(time.time() - t0, 1),
        "worst": {k: float("%.3g" % v) for k, v in worst.items()},
        "kick": kicks,
        "tangent": tangent,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out["worst"]))


if __name__ == "__main__":
    main()
