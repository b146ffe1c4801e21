"""Cost of NAFF tunes on the GPU (xl.naff, csrc/naff.cu) and of a footprint job end to end.

1. Kernel time from CUDA events over repeated calls for (n, T) = (1e5, 1024), (1e5, 4096),
   (2e4, 8192), complex signals (a tune, a 10 % harmonic, a 5 % coupling line, noise), generated
   on the device; signals per second; the FP64 operations and bytes per signal the algorithm
   needs (counted below, with the refinement passes per signal taken from the NumPy definition on
   a sample of the same signals) and from them the achieved rate and the share of the bound.
2. A footprint job: C5 (configs.config_psb, 120 space-charge kicks), 1e4 particles x 2048 turns
   with a BeamMonitor at the start of the ring -- tracking time (host clock around the call,
   ending in a synchronise) next to the analysis time (monitor_tunes, both planes).

The card's name, power limit and clocks, and the measured FP64 peak, are read in the same run.

    python scripts/probe_naff.py [--out FILE]
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

CASES = ((100_000, 1024), (100_000, 4096), (20_000, 8192))
HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def flops_per_signal(T, passes):
    """FP64 operations of one complex signal: samples (z, mean, centring, window: ~12 per turn),
    the zero-padded radix-2 FFT (5·M·log2 M), the argmax (3 per bin) and `passes` refinement passes
    of 23 per turn (w·z·e 6, S0 2, S1 4, S2 5, rotation 6).  sincospi calls count as 0."""
    M = 1 << (T - 1).bit_length()
    return 12 * T + 5 * M * (M.bit_length() - 1) + 3 * M + passes * 23 * T


def bytes_per_signal(T):
    """Compulsory DRAM traffic of one complex signal: u and pu read once, tune and amplitude
    written (the kernel reads the samples twice; the second pass is counted apart)."""
    return 16 * T + 16


def _signals(n, T, seed):
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    t = torch.arange(T, dtype=torch.float64, device="cuda")[:, None]
    nu1 = 0.02 + 0.46 * torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    nu2 = 0.02 + 0.46 * torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    u = torch.empty(T, n, dtype=torch.float64, device="cuda")
    pu = torch.empty_like(u)
    for c0 in range(0, n, 8192):  # keep the temporaries small
        c = slice(c0, min(n, c0 + 8192))
        ph1 = 2 * torch.pi * nu1[c] * t
        ph2 = 2 * torch.pi * nu2[c] * t
        u[:, c] = torch.cos(ph1) + 0.1 * torch.cos(2 * ph1) + 0.05 * torch.cos(ph2)
        pu[:, c] = -torch.sin(ph1) - 0.1 * torch.sin(2 * ph1) - 0.05 * torch.sin(ph2)
    u += 1e-6 * torch.randn(T, n, dtype=torch.float64, device="cuda", generator=g)
    return u, pu


def kernel_case(n, T, peak):
    import numpy as np
    import torch

    import xline_b200 as xl
    from tests import naff_oracle as NO

    u, pu = _signals(n, T, seed=n + T)
    for _ in range(2):
        xl.naff(u, pu)
    torch.cuda.synchronize()
    reps, ms = 1, 0.0
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            q, a = xl.naff(u, pu)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        if ms > 500 or reps >= 256:
            break
        reps *= 2
    per_call_s = ms / reps / 1e3
    k = 64
    rq, ra, near, passes = NO.naff(u[:, :k].cpu().numpy(), pu[:, :k].cpu().numpy(), with_passes=True)
    dq = float(np.nanmax(np.abs(q[:k].cpu().numpy() - rq)))
    fl = flops_per_signal(T, float(passes.mean()))
    by = bytes_per_signal(T)
    t_fp64, t_mem = n * fl / peak, n * by / HBM_BYTES_PER_S
    return {"n": n, "T": T, "signal": "complex", "reps": reps, "kernel_ms": per_call_s * 1e3,
            "signals_per_s": n / per_call_s, "refinement_passes_mean": float(passes.mean()),
            "refinement_passes_max": int(passes.max()), "fp64_flops_per_signal": fl,
            "bytes_per_signal": by, "bytes_issued_per_signal": 2 * by - 16,
            "achieved_fp64_flops_per_s": n * fl / per_call_s, "achieved_bytes_per_s": n * by / per_call_s,
            "bound": "fp64" if t_fp64 >= t_mem else "hbm",
            "share_of_bound": max(t_fp64, t_mem) / per_call_s,
            "max_tune_diff_to_numpy_64_signals": dq}


def footprint(n=10_000, turns=2048):
    import numpy as np
    import torch

    import xline_b200 as xl
    from xline_b200 import configs, optics

    line, cols, p0c, m0 = configs.config_psb(n, monitor_stores=turns, monitor_ids=n)
    tw = optics.twiss(line)
    opt = (tw["betx"][0], tw["alfx"][0], tw["bety"][0], tw["alfy"][0])
    p = xl.Particles(p0c=p0c, mass0=m0, **cols)
    line.track(p, num_turns=2)  # warm-up: module loads, pack caches
    line.reset_monitors()
    p = xl.Particles(p0c=p0c, mass0=m0, **cols)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    line.track(p, num_turns=turns)
    torch.cuda.synchronize()
    track_s = time.perf_counter() - t0
    mon = line.elements[0]
    xl.monitor_tunes(mon, optics=opt)
    torch.cuda.synchronize()
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        r = xl.monitor_tunes(mon, optics=opt)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    qx, qy = r["qx"][0].cpu().numpy(), r["qy"][0].cpu().numpy()
    ok = np.isfinite(qx) & np.isfinite(qy)
    return {"config": "c5", "particles": n, "turns": turns, "track_s": track_s,
            "analysis_s": min(times), "analysis_s_all": times, "analysis_over_tracking": min(times) / track_s,
            "alive": int((p.state == 1).sum()), "valid_tunes": int(ok.sum()),
            "qx_range": [float(qx[ok].min()), float(qx[ok].max())], "qy_range": [float(qy[ok].min()), float(qy[ok].max())],
            "twiss_q": [float(tw["qx"] % 1), float(tw["qy"] % 1)]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    args = ap.parse_args()

    import torch

    from xline_b200 import _cabi

    if not torch.cuda.is_available():
        raise SystemExit("probe_naff.py measures on the GPU; no CUDA device found")
    peak, _ = _cabi.measure_fp64_peak()
    result = {"what": __doc__.split("\n\n")[0], "gpu": gpu_info(), "fp64_peak_measured_flops_per_s": peak,
              "hbm_bytes_per_s_datasheet": HBM_BYTES_PER_S, "kernel": []}
    for n, T in CASES:
        row = kernel_case(n, T, peak)
        result["kernel"].append(row)
        print(json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    result["footprint"] = footprint()
    print(json.dumps(result["footprint"]), flush=True)
    result["gpu_after"] = gpu_info()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
