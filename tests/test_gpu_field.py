"""Tori in a uniform longitudinal field on the device (k_sweep_field, csrc/sweep_field.cu; run with
-m gpu on a B200): bit for bit against the field mirror (tests/field_mirror.c: msc_mirror_run_field)
at every instantiation the launcher picks, at config 3's size and as a shard; the h = 0 field graph
against the plain torus; per-sweep energies against numpy; the Lattice face through every driver,
in law against the float-field path; and every refusal."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from field_check import energies_from_states, mirror_field
from mirror_check import assert_same, families, instances, launched

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def field_instance(dims, E, planes, rounds, pmj):
    """k_sweep_field<DIM, PMJ, K, ROUNDS, V> as launch_sweep_field picks it (V from the word count)"""
    W = -(-E // 32)
    V = 4 if W % 4 == 0 else (2 if W % 2 == 0 else 1)
    return (3 if len(dims) == 3 and dims[2] > 1 else 2, pmj, planes, rounds, V)


# dims, E, pmj, j0, h, betas, planes, rounds, offset
CASES = {
    "c3_shape_pmj": ((8, 6, 4), 128, True, -1.0, 0.3, [0.2, 0.9, 0.9], 6, 7, 96),
    "dE0_classes_v1": ((4, 4, 6), 96, True, -1.0, 2.0, [0.5, 3.0], 5, 10, 0),
    "antiferro_v2": ((6, 4, 4), 64, False, 1.0, -0.1, [0.25, 0.6], 7, 7, 32),
    "2d_all_up_uphill": ((16, 8), 128, False, -1.0, 7.0, [0.3, 0.44], 6, 10, 0),
    "2d_pmj_ragged": ((12, 6), 40, True, -1.5, 0.15, [0.4, 2.5], 7, 10, 160),
    "2d_dE0_high_beta": ((10, 10), 70, False, -0.5, 1.0, [1.0, 4.0], 5, 7, 64),
    "3d_ferro_v4": ((16, 16, 16), 256, False, -0.7, 1.4, [0.6, 2.0], 6, 7, 0),
    "grid_wrap": ((4, 80, 64), 32, True, -1.0, -7.0, [0.3, 1.5], 6, 7, 224),   # 5120 rows > 32 blocks per SM
}
C3_BETAS = [0.2, 0.5, 0.8, 1.1]


def _case(native, oracle, name):
    dims, E, pmj, j0, h, betas, planes, rounds, off = CASES[name]
    ctx = native.Context.get(0)
    g = native.Graph.torus(ctx, dims, j0=j0, pmj=pmj, j_seed=3, field=h)
    a, b, j = g.edges()
    en_ref, st_ref = mirror_field(a, b, j, g.nvars, g.colors(), E, 17, betas, h, replica_offset=off, planes=planes,
                                  rounds=rounds, per_sweep=True)
    sim = native.Sim(g, E, 17, replica_offset=off, planes=planes, rounds=rounds)
    en, names = launched(lambda: sim.sweeps(betas, per_sweep_energies=True))
    assert_same(sim.states(), st_ref, en, en_ref, name, off)
    assert (sim.energies() == en_ref[:, -1]).all(), name
    sim.close()
    return names


def _config3(native, oracle):
    """64^3 +-J x 1024 in h = 0.3: words 0 and 31 against the mirror; the 96-replica shard at offset
    128 equals words 4 .. 6 of the unsharded run"""
    ctx = native.Context.get(0)
    g = native.Graph.torus(ctx, (64, 64, 64), j0=1.0, pmj=True, j_seed=2024, field=0.3)
    a, b, j = g.edges()
    colors = g.colors()
    sim = native.Sim(g, 1024, 31337)
    en, names = launched(lambda: sim.sweeps(C3_BETAS, per_sweep_energies=True))
    st = sim.states()
    sim.close()
    for w in (0, 31):
        en_ref, st_ref = mirror_field(a, b, j, g.nvars, colors, 32, 31337, C3_BETAS, 0.3, replica_offset=32 * w,
                                      per_sweep=True)
        assert_same(st[32 * w:32 * w + 32], st_ref, en[32 * w:32 * w + 32], en_ref, f"config 3 word {w}", 32 * w)
    shard = native.Sim(g, 96, 31337, replica_offset=128)
    en_s, names_s = launched(lambda: shard.sweeps(C3_BETAS, per_sweep_energies=True))
    assert_same(shard.states(), st[128:224], en_s, en[128:224], "config 3 shard", 128)
    shard.close()
    return names, names_s


ZERO_FIELD = {"zero_field_2d": ((64, 64), False, -1.0, 64), "zero_field_3d_pmj": ((16, 16, 16), True, 1.0, 128)}


def _zero_field(native, name):
    """h = 0 through ising_graph_torus_field equals ising_graph_torus bit for bit, states and energies"""
    dims, pmj, j0, E = ZERO_FIELD[name]
    ctx = native.Context.get(0)
    betas = [0.3, 0.44, 1.0, 2.0]
    out, names = [], None
    for field in (None, 0.0):
        g = native.Graph.torus(ctx, dims, j0=j0, pmj=pmj, j_seed=9, field=field)
        sim = native.Sim(g, E, 123)
        if field is None:
            en = sim.sweeps(betas, per_sweep_energies=True)
        else:
            en, names = launched(lambda: sim.sweeps(betas, per_sweep_energies=True))
        out.append((sim.states(), en, sim.energies()))
        sim.close()
    assert_same(out[1][0], out[0][0], out[1][1], out[0][1], name)
    assert (out[0][2] == out[1][2]).all(), name
    return names


def _lattice(native):
    """the Lattice face: a global bias on a torus runs the field kernel"""
    import pyisingmontecarlo_b200 as pkg

    lat = pkg.Lattice.torus((16, 16), j=-1.0, seed_gen=11)
    lat.set_global_bias(0.2)
    _, names = launched(lambda: lat.run_monte_carlo(0.35, 20, 64, only_basic_moves=True))
    return names


# The profiler attaches CUPTI to its process; in a pytest process that also ran it, later profiled
# tests of other files missed kernels (DESIGN section 2, item 7): every profiled run happens here.
_CHILD = (
    "import json, sys\n"
    "sys.path[:0] = [%r, %r]\n"
    "import oracle_lib, test_gpu_field as T\n"
    "from pyisingmontecarlo_b200 import _native as nat\n"
    "res = {n: T._case(nat, oracle_lib, n) for n in T.CASES}\n"
    "res['config3'], res['config3_shard'] = T._config3(nat, oracle_lib)\n"
    "res.update({n: T._zero_field(nat, n) for n in T.ZERO_FIELD})\n"
    "res['lattice'] = T._lattice(nat)\n"
    "json.dump(res, open(sys.argv[1], 'w'))\n") % (ROOT, os.path.join(ROOT, "tests"))


def test_field_kernels_match_mirror(native):
    """Every case equals the mirror bit for bit, and the h = 0 field graph the plain torus (asserted
    in one child process, which records the kernels it launched); each ran the k_sweep_field
    instantiation the launcher's rule gives and no float-field kernel."""
    e = {k: v for k, v in os.environ.items() if not k.startswith("ISING_")}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "kernels.json")
        res = subprocess.run([sys.executable, "-c", _CHILD, path], env=e, timeout=900, capture_output=True, text=True)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
        got = json.load(open(path))
    want = {n: field_instance(c[0], c[1], c[6], c[7], c[2]) for n, c in CASES.items()}
    want["config3"] = (3, True, 6, 7, 4)            # W = 32 -> V = 4
    want["config3_shard"] = (3, True, 6, 7, 1)      # W = 3 -> V = 1
    want["zero_field_2d"] = (2, False, 6, 7, 2)      # W = 2
    want["zero_field_3d_pmj"] = (3, True, 6, 7, 4)   # W = 4
    want["lattice"] = (2, False, 6, 7, 2)
    assert set(got) == set(want)
    for name, names in got.items():
        assert instances(names, "k_sweep_field") == {want[name]}, (name, names)
        assert "k_sweep_real" not in " ".join(names), (name, names)
        assert families(names) == {"k_sweep_field", "k_nsat_stencil"}, (name, names)


def test_energies_every_replica_every_sweep(native):
    ctx = native.Context.get(0)
    h = 0.37
    g = native.Graph.torus(ctx, (32, 32, 16), j0=1.0, pmj=True, j_seed=5, field=h)
    a, b, j = g.edges()
    sim = native.Sim(g, 1000, 41)
    for t, beta in enumerate((0.45, 1.2, 1.2)):
        en = sim.sweeps([beta], per_sweep_energies=True)
        ref = energies_from_states(sim.states(), a, b, j, h)
        assert (en[:, 0] == ref).all(), f"sweep {t}: {(en[:, 0] != ref).sum()} energies differ"
        assert (sim.energies() == ref).all()
        m = sim.magnetization()
        assert (m == (2.0 * sim.states().sum(axis=1) - g.nvars)).all()
    sim.close()


def _moments(x):
    per_rep = x.mean(axis=1)
    return per_rep.mean(), per_rep.std(ddof=1) / np.sqrt(len(per_rep))


def test_lattice_drivers_in_a_field(native):
    """Lattice.torus(...).set_global_bias(h): all four drivers and the observables loop give energies
    that match their states and sample the law of the float-field path (the same torus as an edge
    list with set_global_bias) within 4 sigma"""
    import pyisingmontecarlo_b200 as pkg

    dims, beta, h, E = (16, 16), 0.35, 0.2, 512
    lat = pkg.Lattice.torus(dims, j=-1.0, seed_gen=11)
    lat.set_global_bias(h)
    a, b, j = lat.graph().edges()
    assert lat.graph().field == h
    en, st = lat.run_monte_carlo(beta, 20, 64, only_basic_moves=True)
    assert (en == energies_from_states(st, a, b, j, h)).all()
    en, st = lat.run_monte_carlo_annealing([(0, 0.1), (20, beta)], 20, 64, only_basic_moves=True)
    assert (en == energies_from_states(st, a, b, j, h)).all()
    en, st = lat.run_monte_carlo_annealing_and_get_energies([(0, 0.1), (20, beta)], 20, 64, only_basic_moves=True)
    assert en.shape == (64, 20) and (en[:, -1] == energies_from_states(st, a, b, j, h)).all()
    en, st = lat.run_monte_carlo_sampling(beta, 6, 64, only_basic_moves=True, thermalization_time=5, sampling_freq=2)
    assert en.shape == (64, 3) and all((en[:, k] == energies_from_states(st[:, k], a, b, j, h)).all() for k in range(3))
    e_f, m_f, _ = lat.run_monte_carlo_observables(beta, 400, E, thermalization_time=300, sampling_freq=2)
    edges = [((int(x), int(y)), float(w)) for x, y, w in zip(a, b, j)]
    ref = pkg.Lattice(edges, seed_gen=12)
    ref.set_global_bias(h)
    e_r, m_r, _ = ref.run_monte_carlo_observables(beta, 400, E, thermalization_time=300, sampling_freq=2)
    for x, y, what in ((e_f, e_r, "E"), (m_f, m_r, "M")):
        (mx, sx), (my, sy) = _moments(x), _moments(y)
        assert abs(mx - my) < 4 * np.hypot(sx, sy), (what, mx, sx, my, sy)
    assert _moments(m_f)[0] > 0                                       # h > 0 favours up spins


def test_refusals(native):
    import pyisingmontecarlo_b200 as pkg

    ctx = native.Context.get(0)
    with pytest.raises(ValueError, match="finite"):
        native.Graph.torus(ctx, (8, 8), field=float("nan"))
    with pytest.raises(ValueError, match="finite"):
        native.Graph.torus(ctx, (8, 8), field=float("inf"))
    g = native.Graph.torus(ctx, (8, 8, 8), j0=-1.0, field=0.5)
    with pytest.raises(NotImplementedError, match="GENERAL_LAYOUT"):
        native.Sim(g, 64, 1, general_layout=True)
    sim = native.Sim(g, 64, 1)
    with pytest.raises(NotImplementedError, match="per-experiment betas"):
        sim.set_betas(np.full(64, 0.5))
    with pytest.raises(NotImplementedError, match="edge and worm moves"):
        sim.set_moves(edge_passes=1)
    with pytest.raises(NotImplementedError, match="edge and worm moves"):
        sim.set_moves(edge_passes=0, worms=1)
    sim.sweeps([0.5])                                                 # still usable after the refusals
    sim.close()
    with pytest.raises(NotImplementedError, match="tempering"):
        native.Tempering(g, [0.3, 0.5], 1)
    lat = pkg.Lattice.torus((8, 8), j=-1.0, seed_gen=1)
    lat.set_global_bias(0.4)
    with pytest.raises(NotImplementedError, match="replay"):
        lat.replay(0.5, np.zeros((1, 4), dtype=np.uint32), np.full((1, 4), 0.5), np.zeros((1, 64), dtype=bool))
    lat.non_basic_moves = True
    with pytest.raises(NotImplementedError, match="edge and worm moves"):
        lat.run_monte_carlo(0.5, 2, 32, only_basic_moves=False)
    lat2 = pkg.Lattice.torus((8, 8), j=-1.0, seed_gen=1)
    lat2.set_individual_bias(3, 0.5)
    with pytest.raises(NotImplementedError, match="individual"):
        lat2.run_monte_carlo(0.5, 2, 32, only_basic_moves=True)
