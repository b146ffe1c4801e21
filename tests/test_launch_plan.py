"""The launch policy of the tracking calls (xline_b200/csrc/launch_plan.h) on the host: the turns a
launch takes, the launch-length ramp, the default kernel shape, the grid of the persistent queue
and the beam-moment store turns.  None of it changes results, only how the work is cut into
launches, so the GPU tests reach it only indirectly; here a small C++ driver around the header
pins each decision."""
import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "xline_b200", "csrc")

DRIVER = r"""
#include <iostream>
#include <string>
#include "launch_plan.h"
using namespace xlb;
int main() {
  std::string f;
  while (std::cin >> f) {
    if (f == "cap") {
      int tpl, turns, chunks;
      std::cin >> tpl >> turns >> chunks;
      std::cout << launch_cap(tpl, turns, chunks) << "\n";
    } else if (f == "rate") {
      double rate;
      int longest;
      std::cin >> rate >> longest;
      std::cout << launch_length_for_rate(rate, longest) << "\n";
    } else if (f == "ramp") {
      double rate;
      int longest, previous;
      std::cin >> rate >> longest >> previous;
      std::cout << ramp_step(rate, longest, previous) << "\n";
    } else if (f == "request") {
      int ppt, threads, strict, beamfields, chi, sms;
      long long n;
      std::cin >> ppt >> threads >> strict >> beamfields >> chi >> n >> sms;
      const LaunchRequest r = launch_request(ppt, threads, strict, beamfields, chi, n, sms);
      std::cout << r.ppt << " " << r.threads << "\n";
    } else if (f == "grid") {
      int blocks, resident, sms;
      std::cin >> blocks >> resident >> sms;
      std::cout << persistent_grid(blocks, resident, sms) << "\n";
    } else if (f == "store") {
      xlb_moments_spec_t spec;
      long long k, turns;
      std::cin >> spec.num_stores >> spec.start >> spec.skip >> k >> turns;
      std::cout << moment_store_turn(spec, k, turns) << "\n";
    } else {
      return 2;
    }
  }
  return 0;
}
"""


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    d = tmp_path_factory.mktemp("launch_plan")
    src, exe = str(d / "driver.cpp"), str(d / "driver")
    with open(src, "w") as fh:
        fh.write(DRIVER)
    subprocess.run([cxx, "-std=c++17", "-O2", "-I", CSRC, "-o", exe, src], check=True)

    def run(*queries):
        text = "".join(" ".join(str(v) for v in q) + "\n" for q in queries)
        res = subprocess.run([exe], input=text, capture_output=True, text=True, check=True)
        return [tuple(int(v) for v in line.split()) if " " in line else int(line)
                for line in res.stdout.splitlines()]

    return run


def test_launch_cap(plan):
    assert plan(
        ("cap", 0, 150, 1), ("cap", 0, 151, 1),       # automatic: one launch up to 150 turns, else 100
        ("cap", -1, 1000, 1), ("cap", -7, 123, 1),    # negative: every turn in one launch
        ("cap", 7, 1000, 1), ("cap", 7, 3, 1),        # positive: itself
    ) == [150, 100, 1000, 123, 7, 7]
    # a launch streams at most 2^31 chunks
    cap = 0x7FFFFFFF // 1000
    assert plan(("cap", -1, 0x7FFFFFFF, 1000), ("cap", 5_000_000, 10_000_000, 1000),
                ("cap", 0, 10**9, 1000), ("cap", -1, 10, 0x7FFFFFFF)) == [cap, cap, 100, 1]


def test_launch_length_from_loss_rate(plan):
    assert plan(("rate", 0, 100), ("rate", -0.0, 100), ("rate", -1, 100)) == [100, 100, 100]
    rates = [1.0, 0.5, 0.06, 0.01, 0.003, 1e-3, 6e-4, 1e-6]
    want = []
    for r in rates:
        length = 0.06 / r
        want.append(100 if length >= 100 else (1 if length < 1.0 else int(length)))
    assert plan(*[("rate", repr(r), 100) for r in rates]) == want
    assert want[:4] == [1, 1, 1, 6] and want[-1] == 100


def test_ramp_never_more_than_doubles(plan):
    lengths = [1]
    for _ in range(8):
        lengths.append(plan(("ramp", 0, 100, lengths[-1]))[0])
    assert lengths == [1, 2, 4, 8, 16, 32, 64, 100, 100]
    # a higher loss rate shortens the next launch at once
    assert plan(("ramp", 0.01, 100, 64), ("ramp", 1e-6, 100, 3), ("ramp", 0, 0x7FFFFFFF, 0x7FFFFFF0)) == \
        [6, 6, 0x7FFFFFFF]


def test_default_particles_per_thread(plan):
    sms = 148
    thin = [("request", 0, 0, 0, 0, 0, n, sms) for n in (10**6, 227_328, 227_327, 18_944, 18_943, 1)]
    assert plan(*thin) == [(4, 128), (4, 128), (2, 128), (2, 128), (1, 128), (1, 128)]
    assert plan(
        ("request", 0, 0, 0, 0, 1, 10**6, sms),        # chi column: three
        ("request", 0, 0, 0, 0, 1, 170_495, sms),      # ... two below 3 x 128 x 3 per SM
        ("request", 0, 0, 1, 0, 0, 10**6, sms),        # strict: three
        ("request", 0, 0, 0, 1, 0, 10**6, sms),        # beam fields: two in 256-thread CTAs
        ("request", 0, 0, 0, 1, 0, 100, sms),          # ... whatever the beam
        ("request", 0, 256, 0, 0, 0, 100, sms),        # the caller's CTA size keeps four
        ("request", 3, 0, 0, 0, 0, 100, sms),          # the caller's particles per thread
        ("request", 1, 0, 0, 1, 0, 10**6, sms),
    ) == [(3, 128), (2, 128), (3, 128), (2, 256), (2, 256), (4, 256), (3, 128), (1, 256)]


def test_persistent_grid(plan):
    assert plan(("grid", 2000, 444, 148), ("grid", 2000, 454, 148), ("grid", 160, 444, 148),
                ("grid", 250, 444, 148)) == [444, 444, 148, 235]


def test_moment_store_turns(plan):
    # (num_stores, start, skip, k, num_turns)
    assert plan(("store", 3, 0, 5, 0, 10), ("store", 3, 0, 5, 1, 10), ("store", 3, 0, 5, 2, 10),
                ("store", 3, 0, 5, 3, 10)) == [0, 5, 10, 11]
    assert plan(("store", 3, 11, 1, 0, 10), ("store", 5, 0, 4, 3, 10)) == [11, 11]
    # start + k * skip would overflow: no store left
    big = 2**62
    assert plan(("store", 10, 1, big, 2, 10), ("store", 10, 3, 2**63 - 1, 0, 10),
                ("store", 10, 0, 2**63 - 1, 1, big)) == [11, 3, big + 1]
