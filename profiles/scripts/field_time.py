"""Device time per sweep of a torus in a uniform longitudinal field: config 3's lattice (64^3 +-J x
1024 replicas) at beta = 0.5 and h in {0.1, 1.0} on three paths,
  (a) field     Graph.torus(..., field=h): the bit-sliced field kernel (k_sweep_field)
  (b) float     the same torus as an edge list with biases h: the float-field kernel (k_sweep_real)
  (c) no field  Graph.torus(...): today's zero-field path (row walk)
with and without per-sweep energies.  Time = the library's CUDA events (SimStats.sweep_device_ms).
The card's name, power limit and SM clock are read in the same run and written next to the numbers.

    python profiles/scripts/field_time.py [--out profiles/r03_field_time.log] [--sweeps 40]"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.getcwd())
import numpy as np

from pyisingmontecarlo_b200 import _native as nat


def per_sweep_ms(sim, nsweeps, energies):
    betas = np.full(nsweeps, 0.5)
    sim.sweeps(betas[:3], per_sweep_energies=energies)             # warm-up: modules, scratch buffers
    sim.reset_stats()
    sim.sweeps(betas, per_sweep_energies=energies)
    return sim.stats()["sweep_device_ms"] / nsweeps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r03_field_time.log"))
    ap.add_argument("--sweeps", type=int, default=40)
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    ctx = nat.Context.get(0)
    dims, E = (64, 64, 64), 1024
    plain = nat.Graph.torus(ctx, dims, j0=1.0, pmj=True, j_seed=2024)
    a, b, j = plain.edges()
    N = plain.nvars
    lines = [f"field_time.py: {dims[0]}^3 +-J x {E} replicas, beta 0.5, {args.sweeps} sweeps per measurement",
             f"card (name, power limit, SM clock, max SM clock): {card}",
             "device time per sweep (library CUDA events, SimStats.sweep_device_ms); flips/s = E * N / time", ""]
    for h in (0.1, 1.0):
        graphs = {"(a) field": nat.Graph.torus(ctx, dims, j0=1.0, pmj=True, j_seed=2024, field=h),
                  "(b) float": nat.Graph.from_edges(ctx, N, a, b, j, np.full(N, h)),
                  "(c) no field": plain}
        for energies in (False, True):
            ms = {}
            for name, g in graphs.items():
                sim = nat.Sim(g, E, 5)
                ms[name] = per_sweep_ms(sim, args.sweeps, energies)
                sim.close()
            mode = "with per-sweep energies" if energies else "sweeps only"
            lines.append(f"h = {h}, {mode}:")
            for name, t in ms.items():
                lines.append(f"  {name:13s} {1e3 * t:9.1f} us/sweep  {E * N / (t * 1e-3) / 1e9:8.2f} Gflips/s")
            lines.append(f"  field / float flips/s = {ms['(b) float'] / ms['(a) field']:.2f}x, "
                         f"field / no-field flips/s = {ms['(c) no field'] / ms['(a) field']:.2f}x")
    text = "\n".join(lines) + "\n"
    print(text, end="")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
