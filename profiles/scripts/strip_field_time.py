"""Device time of sweeps of the single large lattice in a uniform longitudinal field: SingleLattice2D(65536)
(config 5's lattice, one strip, exchange_every = 8) at beta = 0.44 and h in {0, 0.1, 1.0}; h = 0 runs the
zero-field kernel (k_strip_phase), h != 0 the field kernel (k_strip_phase_field).  Time = the library's CUDA
events around ising_strip_sweeps (Strip.stats()["device_ms"]), after a warm-up, over windows of at least 1 s;
the three fields are measured in turn, `--rounds` times.  The card's name, power limit and SM clock are read
in the same run and written next to the numbers.  Sweeps only: no observables inside the windows.

    python profiles/scripts/strip_field_time.py [--out profiles/r04_strip_field_time.log] [--rounds 3]"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.getcwd())
import numpy as np

import pyisingmontecarlo_b200 as pkg

FIELDS = (0.0, 0.1, 1.0)


def window(lat, beta, h, min_ms=1000.0):
    """(device ms, sweeps) of one window of >= min_ms in the field h"""
    n = 64
    while True:
        lat.strip.stats(reset=True)
        lat.sweeps(np.full(n, beta), h)
        ms = lat.strip.stats()["device_ms"]
        if ms >= min_ms:
            return ms, n
        n = int(n * 1.2 * min_ms / max(ms, 1e-3)) + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r04_strip_field_time.log"))
    ap.add_argument("--L", type=int, default=65536)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    L, beta = args.L, 0.44
    lat = pkg.SingleLattice2D(L, seed=1)
    for h in FIELDS:                                               # warm-up: modules, every kernel, the clocks
        lat.sweeps(np.full(32, beta), h)
    rates = {h: [] for h in FIELDS}
    lines = []
    for r in range(args.rounds):
        for h in FIELDS if r % 2 == 0 else FIELDS[::-1]:
            ms, n = window(lat, beta, h)
            rate = float(L) * L * n / (ms * 1e-3)
            rates[h].append(rate)
            lines.append(f"  round {r}  h = {h:<4}  {n:5d} sweeps in {ms:8.1f} ms  {1e3 * ms / n:8.1f} us/sweep  "
                         f"{rate / 1e12:6.3f} x 10^12 flips/s")
    card_after = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader"],
                                capture_output=True, text=True).stdout.strip().splitlines()[0]
    out = [f"strip_field_time.py: SingleLattice2D({L}) (one strip, exchange_every = 8), beta = {beta}, windows >= 1 s",
           f"card (name, power limit, SM clock, max SM clock): {card}",
           f"after the runs (SM clock, power draw): {card_after}",
           "device time = the library's CUDA events around ising_strip_sweeps; flips/s = L^2 * sweeps / time", ""]
    out += lines + ["", "median over the rounds:"]
    base = float(np.median(rates[0.0]))
    for h in FIELDS:
        med = float(np.median(rates[h]))
        kern = "k_strip_phase" if h == 0.0 else "k_strip_phase_field"
        out.append(f"  h = {h:<4} {kern:20s} {med / 1e12:6.3f} x 10^12 flips/s   {med / base:5.2f}x of h = 0  "
                   f"(spread {min(rates[h]) / 1e12:.3f} .. {max(rates[h]) / 1e12:.3f})")
    text = "\n".join(out) + "\n"
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
