"""Beam moments without a GPU: spec validation, store turns, the layout constants of the C ABI,
the centring / emittance arithmetic on synthetic pairs and the multi-rank fold over gloo, all
against exact rational arithmetic (tests/moments_oracle.py)."""
import ctypes as C
import math
import os
import re
import socket
from fractions import Fraction

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests import moments_oracle as MO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _words(exact):
    """A store holding the exact sums rounded to (hi, lo) pairs."""
    w = [float(exact["n"]), float(exact["n_nonfinite"])]
    for s in exact["sums"]:
        hi = float(s)
        w += [hi, float(s - Fraction(hi))]
    return w


def _beam(n, seed, offset=0.0):
    rng = np.random.default_rng(seed)
    scale = (1e-3, 1e-5, 2e-3, 3e-5, 0.1, 1e-3)
    return {k: offset * s + rng.normal(0, s, n) for k, s in zip(MO.COORDS, scale)}


def test_spec_validation():
    import xline_b200 as xl

    for bad in (dict(num_stores=-1), dict(num_stores=2, start=-1), dict(num_stores=2, skip=0)):
        with pytest.raises(ValueError):
            xl.BeamMoments(device="cpu", **{"num_stores": 1, **bad})
    from xline_b200 import _cabi

    L = _cabi.lib()
    opts = _cabi.TrackOptions()
    for ns, start, skip in ((-1, 0, 1), (1, -1, 1), (1, 0, 0), (1, 0, -3)):
        spec = _cabi.MomentsSpec(ns, start, skip)
        rc = L.xlb_track_device_moments(None, None, C.byref(opts), C.byref(spec), None, None)
        assert rc == -1 and b"spec" in L.xlb_last_error()
    assert L.xlb_track_device_moments(None, None, C.byref(opts), None, None, None) == -1
    spec = _cabi.MomentsSpec(1, 0, 1)
    assert L.xlb_track_device_moments(None, None, C.byref(opts), C.byref(spec), None, None) == -1
    assert b"out is null" in L.xlb_last_error()


def test_store_turns():
    import xline_b200 as xl

    m = xl.BeamMoments(5, start=3, skip=7, device="cpu")
    assert m.turn.tolist() == [3, 10, 17, 24, 31]
    assert xl.BeamMoments(3, device="cpu").turn.tolist() == [0, 1, 2]
    assert xl.BeamMoments(0, device="cpu").data.shape == (0, 56)
    # never written until a call reaches the store's turn
    assert torch.isnan(m.data).all()


def test_layout_constants_match_the_header():
    from xline_b200 import _cabi, moments

    text = open(os.path.join(ROOT, "include", "xline_b200.h")).read()
    defs = dict(re.findall(r"#define (XLB_MOMENT_\w+) (\d+)", text))
    assert int(defs["XLB_MOMENT_WORDS"]) == _cabi.MOMENT_WORDS == MO.WORDS
    assert int(defs["XLB_MOMENT_PAIRS"]) == _cabi.MOMENT_PAIRS == len(moments.PAIRS) == 27
    assert int(defs["XLB_MOMENT_FIRST"]) == _cabi.MOMENT_FIRST
    assert _cabi.MOMENT_FIRST + 2 * _cabi.MOMENT_PAIRS == _cabi.MOMENT_WORDS
    spec = re.search(r"typedef struct xlb_moments_spec \{(.*?)\}", text, re.S).group(1)
    assert re.findall(r"int64_t (\w+);", spec) == [f for f, _ in _cabi.MomentsSpec._fields_]
    assert all(t is C.c_int64 for _, t in _cabi.MomentsSpec._fields_)
    # pair order: the six first moments, then the upper triangle row by row (xx xpx xy ... deltadelta)
    assert moments.PAIRS == MO.PAIRS
    assert moments.pair_index(0) == 0 and moments.pair_index(5) == 5
    assert moments.pair_index(0, 0) == 6 and moments.pair_index(1, 0) == 7 and moments.pair_index(0, 5) == 11
    assert moments.pair_index(1, 1) == 12 and moments.pair_index(5, 5) == 26


@pytest.mark.parametrize("offset", [0.0, 30.0])
def test_centring_and_emittance_against_fractions(offset):
    """mean / cov / emittances from stores of exact sums, against exact rational centring.  The
    offset puts the mean at 30 sigma: Σu·v - Σu·Σv / n then cancels about 10 digits."""
    import xline_b200 as xl

    stores = []
    for seed, n in ((1, 500), (2, 777), (3, 64)):
        cols = _beam(n, seed, offset)
        stores.append(MO.exact_store(cols, np.ones(n, dtype=np.int64)))
    m = xl.BeamMoments(len(stores), device="cpu")
    m.data = torch.tensor([_words(e) for e in stores], dtype=torch.float64)
    m.beta0gamma0 = 7.5
    mean, cov, eps = m.mean.numpy(), m.cov.numpy(), m.emittance()
    assert m.count.tolist() == [500, 777, 64] and m.n_nonfinite.tolist() == [0, 0, 0]
    for s in range(len(stores)):
        emean, ecov = MO.centred(m.data[s].tolist())
        for u in range(6):
            assert MO.ulps(mean[s, u], emean[u]) <= 0.5 + 1e-9, (s, u)
            for v in range(6):
                assert cov[s, u, v] == cov[s, v, u]
                assert MO.ulps(cov[s, u, v], ecov[u][v]) <= 0.5 + 1e-6, (s, u, v)
        for name, k in (("x", 0), ("y", 2), ("zeta", 4)):
            want = MO.emittance_from_cov(cov[s], k)
            assert abs(float(eps["eps_" + name][s]) - want) <= math.ulp(want), (s, name)
        assert float(eps["neps_x"][s]) == float(eps["eps_x"][s]) * 7.5


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _merge_worker(rank, world, port, n_total, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import xline_b200 as xl
        from xline_b200 import sharding

        full = _beam(n_total, 11, offset=2.0)
        state = np.ones(n_total, dtype=np.int64)
        state[::7] = 0
        lo, hi = sharding.shard_bounds(n_total, rank, world)
        mine = MO.exact_store({k: v[lo:hi] for k, v in full.items()}, state[lo:hi])
        m = xl.BeamMoments(2, device="cpu")
        m.data[0] = torch.tensor(_words(mine), dtype=torch.float64)  # store 1 stays unwritten
        merged = sharding.merge_moments(m)
        gathered = [torch.empty_like(merged.data) for _ in range(world)]
        dist.all_gather(gathered, merged.data)
        if rank == 0:
            assert all(torch.equal(g.view(torch.int64), merged.data.view(torch.int64)) for g in gathered)
            exact = MO.exact_store(full, state)
            errs = MO.store_errors(merged.data[0].tolist(), exact)
            # world roundings of the rank sums plus world - 1 additions
            assert max(errs) <= world * MO.DD_ADD_REL, float(max(errs))
            assert torch.isnan(merged.data[1]).all()
            out.put("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(240)
@pytest.mark.parametrize("world", [2, 3])
def test_merge_moments_over_gloo(world):
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_merge_worker, args=(r, world, port, 1001, out)) for r in range(world)]
    for pr in procs:
        pr.start()
    for pr in procs:
        pr.join(200)
    assert all(pr.exitcode == 0 for pr in procs), [pr.exitcode for pr in procs]
    assert not out.empty() and out.get() == "ok"


def test_merge_moments_single_process_is_a_copy():
    import xline_b200 as xl
    from xline_b200 import sharding

    m = xl.BeamMoments(1, device="cpu")
    m.data[0] = torch.arange(56, dtype=torch.float64)
    merged = sharding.merge_moments(m)
    assert merged is not m and torch.equal(merged.data, m.data)
