"""The row-walk sweep (k_sweep_rows, csrc/sweep_rows.cuh) and the other per-phase sweep kernels of
lattices above the thread-block-cluster limit, compared bit for bit with the scalar mirror
(oracle/msc_mirror.c) on the device, at every launch shape the library picks (run with -m gpu on
a B200).

A decision depends only on (seed, site, global replica word, sweep), so msc_mirror(E = 32 k,
replica_offset = 32 w) reproduces words w .. w + k - 1 of a larger run: full-size runs are checked
word by word.  Every case records the sweep kernels it launched (torch.profiler, CUDA activity)
and asserts the instantiation that the launcher's shape rules, restated below with the device's
SM count, say it must take; a case that loses its path fails under its own name.
"""
import json
import os
import subprocess
import sys
import tempfile
from dataclasses import dataclass, field

import numpy as np
import pytest

from mirror_check import (assert_same, check_words, device_sms, families, instances, launched,
                          pow2_ceil)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------
# the launcher's dispatch restated (api_sim.cu: sim_sweeps_coop, sweep_cluster.cu,
# sweep_rows_launch.cuh: rows_phase / rows_shape / launch_sweep_rows_dim)
# ---------------------------------------------------------------------------------------------
def _layout(dims, E):
    Lx, Ly, Lz = (list(dims) + [1, 1])[:3]
    W = -(-E // 32)
    return dict(Lxh=Lx // 2, Ly=Ly, Lz=Lz, halfN=Lx * Ly * Lz // 2, W=W,
                V=4 if W % 4 == 0 else (2 if W % 2 == 0 else 1))


def _rows_shape(lay, threads):
    groups = lay["W"] // lay["V"]
    wx = 32 if groups >= 32 else pow2_ceil(groups)
    by = threads // wx
    bxh = min(pow2_ceil(lay["Lxh"]), by)
    nrs = by // bxh
    while nrs > 1 and lay["Ly"] % nrs:
        nrs //= 2
    if nrs > 64:                                            # ROWS_DESC_CHUNK
        return None
    return dict(threads=threads, wx=wx, bxh=bxh, nrs=nrs, xtiles=-(-lay["Lxh"] // bxh),
                wtiles=-(-groups // wx))


def rows_phase(dims, E, acc, sms):
    """Shape of one colour phase of k_sweep_rows (acc: the accumulating phase), None when the row
    walk does not take it."""
    lay = _layout(dims, E)
    V = lay["V"]
    small = V == 4 and lay["halfN"] * (lay["W"] // V) * 2 < sms * 768 * (5 if acc else 3)
    sh = _rows_shape(lay, 128) if small else None
    if small and (sh is None or sh["bxh"] * sh["nrs"] < V):
        small = False
    if not small:
        sh = _rows_shape(lay, 256)
    if sh is None or (acc and sh["bxh"] * sh["nrs"] < V):
        return None
    return dict(sh, V=V, small=small, multirow=sh["nrs"] > 1)


def counter_copies(E):
    """copies of a sweep's satisfied-bond counters with per-sweep energies (ising_sim_sweeps)"""
    cw = -(-E // 32) * 32
    return max(1, min(16, 4096 // cw))


def sweep_path(dims, E, acc, sms):
    """'cluster', or the set of k_sweep_rows template argument tails (V, ACC, MULTIROW, SMALL) one
    sweep launches, with the shapes of its two colour phases."""
    lay = _layout(dims, E)
    words = lay["halfN"] * lay["W"]
    if words <= (8192 if acc else 16384):
        return "cluster", None
    phases = [rows_phase(dims, E, False, sms), rows_phase(dims, E, acc, sms)]
    assert all(phases), (dims, E, acc)
    kerns = {(p["V"], a, p["multirow"], p["small"]) for p, a in zip(phases, (False, acc))}
    return kerns, phases


# ---------------------------------------------------------------------------------------------
# kernel names from the profiler
# ---------------------------------------------------------------------------------------------
def rows_instances(names):
    """template arguments (DIM, PMJ, K, ROUNDS, V, ACC, MULTIROW, SMALL) of every k_sweep_rows"""
    return instances(names, "k_sweep_rows")


def _dim(dims):
    return 2 if len(dims) == 2 else 3


def assert_path(names, dims, E, acc, pmj, sms, label):
    """the sweep kernels of one run are the ones the restated dispatch names"""
    want, _ = sweep_path(dims, E, acc, sms)
    fam = families(names)
    print(f"{label}: {sorted(fam)} {sorted(rows_instances(names))}")
    if want == "cluster":
        assert "k_sweep_stencil_cluster" in fam and "k_sweep_rows" not in fam, (label, names)
        return
    got = rows_instances(names)
    want = {(_dim(dims), pmj, 6, 7) + t for t in want}
    assert got == want, (label, "k_sweep_rows instances", sorted(got), "expected", sorted(want))
    assert fam <= {"k_sweep_rows"}, (label, names)


# ---------------------------------------------------------------------------------------------
# 1. shape matrix: every branch of the launcher, full-replica mirror
# ---------------------------------------------------------------------------------------------
BETAS = np.array([0.35, 0.8, 1.2, 1.2])   # most decisions at 1.2 go through ties


@dataclass
class Case:
    name: str
    dims: tuple
    E: int
    j0: float
    pmj: bool
    seed: int
    offset: int = 0
    reach: dict = field(default_factory=dict)   # mode -> "cluster" or properties of its phase

    @property
    def what(self):
        if self.pmj:
            return f"+-{abs(self.j0):g}J"
        return ("ferro" if self.j0 < 0 else "antiferro") + ("" if abs(self.j0) == 1 else f" |J|={abs(self.j0):g}")


CASES = [
    Case("small_multirow_3d", (64, 64, 64), 128, 1.0, True, 11,
         reach=dict(plain=dict(small=True, multirow=True, nrs=4, V=4),
                    acc=dict(small=True, multirow=True, nrs=4, V=4))),
    Case("mixed_shapes_in_one_sweep", (64, 64, 64), 256, -1.0, False, 12,
         reach=dict(plain=dict(small=False, threads=256, V=4), acc=dict(small=True, threads=128, V=4))),
    Case("w4_256_wx1", (96, 96, 64), 128, 1.0, False, 13,
         reach=dict(plain=dict(small=False, wx=1, multirow=True, V=4),
                    acc=dict(small=False, wx=1, multirow=True, V=4))),
    Case("v1_ragged_tiles", (64, 48), 2080, -0.37, False, 14,
         reach=dict(plain=dict(V=1, xtiles=4, wtiles=3), acc=dict(V=1, xtiles=4, wtiles=3))),
    Case("acc_above_8192_words", (128, 128), 40, 2.0, True, 15,
         reach=dict(plain="cluster", acc=dict(V=2, multirow=True))),
    Case("plain_above_16384_words", (128, 132), 40, -1.0, False, 16,
         reach=dict(plain=dict(V=2), acc=dict(V=2))),
    Case("acc_at_8192_words", (128, 64), 40, 1.0, False, 17, reach=dict(plain="cluster", acc="cluster")),
    Case("noncube_ragged", (8, 24, 12), 1000, 1.0, True, 18,
         reach=dict(plain=dict(V=4, multirow=True), acc=dict(V=4, multirow=True))),
    Case("nrs_halved_by_ly", (8, 6, 24), 1000, -1.0, False, 19,
         reach=dict(plain=dict(small=True, nrs=2), acc=dict(small=True, nrs=2))),
    Case("wtiles9_v1", (8, 8, 8), 8200, 1.0, True, 20,
         reach=dict(plain=dict(V=1, wtiles=9), acc=dict(V=1, wtiles=9))),
    Case("xtiles8_wtiles2", (64, 64), 8192, 1.0, False, 21,
         reach=dict(plain=dict(V=4, xtiles=8, wtiles=2), acc=dict(V=4, xtiles=8, wtiles=2))),
    Case("v1_offset_gw0", (32, 32, 16), 96, 0.5, True, 22, offset=64,
         reach=dict(plain=dict(V=1), acc=dict(V=1))),
    Case("cluster_3d_8192_words", (16, 16, 8), 256, 1.0, True, 23, reach=dict(plain="cluster", acc="cluster")),
]
CASE = {c.name: c for c in CASES}


def check_reach(case, sms):
    """the case still reaches the branch it is meant for"""
    for mode, want in case.reach.items():
        acc = mode == "acc"
        path, _ = sweep_path(case.dims, case.E, acc, sms)
        if want == "cluster":
            assert path == "cluster", f"{case.name} ({mode}) no longer runs in the cluster kernel"
            continue
        assert path != "cluster", f"{case.name} ({mode}) now runs in the cluster kernel"
        ph = rows_phase(case.dims, case.E, acc, sms)
        got = {k: ph[k] for k in want}
        assert got == want, f"{case.name} ({mode}) reaches {got}, meant for {want}"


def run_case(native, oracle, case, check_kernels=True, sms=None):
    """Both runs of a case (plain sweeps; per-sweep energies) against the mirror, bit for bit.
    Returns {mode: kernel names}."""
    ctx = native.Context.get(0)
    g = native.Graph.torus(ctx, case.dims, j0=case.j0, pmj=case.pmj, j_seed=case.seed)
    a, b, j = g.edges()
    en_ref, st_ref = oracle.msc_mirror(a, b, j, g.nvars, g.colors(), case.E, case.seed, BETAS,
                                       replica_offset=case.offset, per_sweep=True)
    out = {}
    for acc in (False, True):
        mode = "acc" if acc else "plain"
        label = f"{case.name} [{case.dims} x {case.E}, {case.what}, {mode}]"
        sim = native.Sim(g, case.E, case.seed, replica_offset=case.offset)
        en, names = launched(lambda: sim.sweeps(BETAS, per_sweep_energies=acc))
        assert_same(sim.states(), st_ref, en, en_ref if acc else None, label, case.offset)
        assert (sim.energies() == en_ref[:, -1]).all(), label
        sim.close()
        if check_kernels:
            assert_path(names, case.dims, case.E, acc, case.pmj, sms, label)
        out[mode] = names
    return out


@pytest.fixture(scope="module")
def sms(native):
    native.Context.get(0)
    return device_sms()


def test_profile_records_library_kernels(native, sms):
    """CUPTI records the kernels of libising_b200 (its own stream and runtime) with their template
    arguments: every path assertion of this file rests on it"""
    ctx = native.Context.get(0)
    g = native.Graph.torus(ctx, (64, 64, 64), j0=1.0, pmj=True, j_seed=1)
    sim = native.Sim(g, 128, 1)
    _, names = launched(lambda: sim.sweeps([0.5]))
    assert rows_instances(names), names
    assert_path(names, (64, 64, 64), 128, False, True, sms, "probe")


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_shape_matrix_matches_mirror(native, oracle, sms, case):
    check_reach(case, sms)
    run_case(native, oracle, case, sms=sms)


# ---------------------------------------------------------------------------------------------
# 2. full BASELINE sizes, word by word
# ---------------------------------------------------------------------------------------------
C3_BETAS = np.linspace(0.1, 1.2, 1000, endpoint=False)[::90]   # 12 sweeps across bench.py's c3 ramp


def test_config3_words_match_mirror(native, oracle, sms):
    """BASELINE config 3 (64^3 +-J x 1024, 256-thread shape): words 0, 15 and 31"""
    ctx = native.Context.get(0)
    dims = (64, 64, 64)
    g = native.Graph.torus(ctx, dims, j0=1.0, pmj=True, j_seed=2024)
    sim = native.Sim(g, 1024, 31337)
    en, names = launched(lambda: sim.sweeps(C3_BETAS, per_sweep_energies=True))
    assert_path(names, dims, 1024, True, True, sms, "config 3")
    st = sim.states()
    sim.close()
    check_words(oracle, g, 1024, 31337, C3_BETAS, (0, 15, 31), en, lambda w: st[32 * w:32 * w + 32], "config 3")


def test_config3_shard_words_match_mirror(native, oracle, sms):
    """the 128-replica shard at offset 896 (8-GPU split: 128-thread shape, gw0 = 28): all words"""
    ctx = native.Context.get(0)
    dims = (64, 64, 64)
    g = native.Graph.torus(ctx, dims, j0=1.0, pmj=True, j_seed=2024)
    sim = native.Sim(g, 128, 31337, replica_offset=896)
    en, names = launched(lambda: sim.sweeps(C3_BETAS, per_sweep_energies=True))
    assert_path(names, dims, 128, True, True, sms, "config 3 shard")
    assert rows_phase(dims, 128, True, sms)["small"]
    st = sim.states()
    sim.close()
    check_words(oracle, g, 128, 31337, C3_BETAS, range(4), en, lambda w: st[32 * w:32 * w + 32],
                "config 3 shard", offset=896)


def test_config2_last_word_matches_mirror(native, oracle, sms):
    """BASELINE config 2 (4096^2 ferromagnet x 1024, beta 0.43): word 31 over 2 sweeps.  The mirror
    holds the 33.5 M-edge list, its adjacency and 32 states (about 2 GB of host memory)."""
    ctx = native.Context.get(0)
    dims = (4096, 4096)
    g = native.Graph.torus(ctx, dims, j0=-1.0)
    betas = [0.43, 0.43]
    sim = native.Sim(g, 1024, 31337)
    en, names = launched(lambda: sim.sweeps(betas, per_sweep_energies=True))
    assert_path(names, dims, 1024, True, False, sms, "config 2")
    col = sim.packed()[:, 31].copy()      # bit b of word 31 = replica 992 + b
    sim.close()
    bits = ((col[None, :] >> np.arange(32, dtype=np.uint32)[:, None]) & 1).astype(bool)
    del col
    check_words(oracle, g, 1024, 31337, betas, (31,), en, lambda w: bits, "config 2")
    del bits


# ---------------------------------------------------------------------------------------------
# 3. every replica, every sweep: per-sweep energies against numpy at every counter-copy count
# ---------------------------------------------------------------------------------------------
COPY_E = [128, 1024, 2048, 4096, 1000]


@pytest.mark.parametrize("E", COPY_E, ids=[f"E{E}_copies{counter_copies(E)}" for E in COPY_E])
def test_every_replica_every_sweep(native, sms, E):
    """Single-sweep calls with per-sweep energies on a lattice above the cluster limit (32 x 32 x 16
    +-J): the accumulating phase spreads its atomics over 16 / 4 / 2 / 1 copies of the counters;
    every replica's energy equals an int64 recomputation from the returned states, and so does
    energies()."""
    ctx = native.Context.get(0)
    dims = (32, 32, 16)
    g = native.Graph.torus(ctx, dims, j0=1.0, pmj=True, j_seed=5)
    a, b, j = g.edges()
    ai, bi, jj = a.astype(np.intp), b.astype(np.intp), j.astype(np.int64)
    assert (jj == j).all()
    sim = native.Sim(g, E, 40 + E)
    for t, beta in enumerate((0.45, 1.2, 1.2)):
        en, names = launched(lambda: sim.sweeps([beta], per_sweep_energies=True))
        assert_path(names, dims, E, True, True, sms, f"E={E} sweep {t}")
        s = sim.states().view(np.int8)
        e_np = np.empty(E, dtype=np.int64)
        for r in range(0, E, 256):
            x = s[r:r + 256] * np.int8(2) - np.int8(1)
            e_np[r:r + 256] = ((x[:, ai] * x[:, bi]).astype(np.int64) * jj).sum(1)
        bad = np.flatnonzero(en[:, 0] != e_np)
        assert len(bad) == 0, (f"E={E} sweep {t}: {len(bad)} per-sweep energies differ, first replica "
                               f"{bad[:1]}: {en[bad[:1], 0]} vs {e_np[bad[:1]]}")
        assert (sim.energies() == e_np).all(), f"E={E} sweep {t}: energies()"
    sim.close()


# ---------------------------------------------------------------------------------------------
# 4. the other per-phase kernels above the cluster limit
# ---------------------------------------------------------------------------------------------
def test_per_replica_beta_above_cluster_limit(native, oracle):
    """set_betas on a lattice above the cluster limit runs k_sweep_stencil_perbeta (the row walk
    has no per-replica tables), with and without per-sweep energies"""
    ctx = native.Context.get(0)
    dims, E, seed = (32, 32, 16), 96, 77
    g = native.Graph.torus(ctx, dims, j0=1.0, pmj=True, j_seed=6)
    betas_e = np.linspace(0.3, 1.3, E)
    a, b, j = g.edges()
    en_ref, st_ref = oracle.msc_mirror(a, b, j, g.nvars, g.colors(), E, seed, None, per_replica_beta=betas_e,
                                       nsweeps=4, per_sweep=True)
    for acc in (False, True):
        sim = native.Sim(g, E, seed)
        sim.set_betas(betas_e)
        en, names = launched(lambda: sim.sweeps(4, per_sweep_energies=acc))
        assert families(names) == {"k_sweep_stencil_perbeta"}, names
        assert_same(sim.states(), st_ref, en, en_ref if acc else None, f"per-replica beta acc={acc}")
        assert (sim.energies() == en_ref[:, -1]).all()
        sim.close()


@pytest.mark.parametrize("planes,rounds", [(5, 7), (7, 7), (6, 10), (5, 10)])
def test_per_row_fallback_above_cluster_limit(native, oracle, planes, rounds):
    """planes 5 / 7 or Philox-10 above the cluster limit: the one-row-per-block k_sweep_stencil
    (the row walk covers 6 planes and 7 rounds only)"""
    ctx = native.Context.get(0)
    dims, E, seed = (32, 32, 16), 128, 78
    g = native.Graph.torus(ctx, dims, j0=1.0, pmj=True, j_seed=7)
    a, b, j = g.edges()
    en_ref, st_ref = oracle.msc_mirror(a, b, j, g.nvars, g.colors(), E, seed, BETAS, planes=planes,
                                       rounds=rounds, per_sweep=True)
    for acc in (False, True):
        sim = native.Sim(g, E, seed, planes=planes, rounds=rounds)
        en, names = launched(lambda: sim.sweeps(BETAS, per_sweep_energies=acc))
        assert families(names) == {"k_sweep_stencil"}, names
        # k_sweep_stencil<DIM, PMJ, K, ROUNDS, V, ACC>: both phases plain, or plain + accumulating
        want = {(3, True, planes, rounds, 4, a) for a in {False, acc}}
        assert instances(names, "k_sweep_stencil") == want, names
        assert_same(sim.states(), st_ref, en, en_ref if acc else None, f"planes {planes} rounds {rounds} acc={acc}")
        sim.close()


# ---------------------------------------------------------------------------------------------
# 5. knobs that change no result (read once per process: one child per knob)
# ---------------------------------------------------------------------------------------------
def _no_small(case, mode, names):
    inst = rows_instances(names)
    assert inst and not any(t[7] for t in inst), names


def _v1(case, mode, names):
    fam = families(names)
    assert "k_sweep_stencil" in fam and "k_sweep_rows" not in fam, names


def _split_acc(case, mode, names):
    inst = rows_instances(names)
    assert inst and not any(t[5] for t in inst), names
    assert ("k_nsat_rows" in families(names)) == (mode == "acc"), names


def _no_cluster(case, mode, names):
    fam = families(names)
    assert "k_sweep_rows" in fam and "k_sweep_stencil_cluster" not in fam, names


def _coop(case, mode, names):
    assert families(names) == {"k_sweep_stencil_coop"}, names


KNOBS = [
    ({"ISING_NO_PDL": "1"}, ["small_multirow_3d", "v1_ragged_tiles", "acc_above_8192_words"], None),
    ({"ISING_ROWS_NO_SMALL": "1"}, ["small_multirow_3d", "xtiles8_wtiles2"], _no_small),
    ({"ISING_SWEEP_V1": "1"}, ["small_multirow_3d", "v1_ragged_tiles", "plain_above_16384_words"], _v1),
    ({"ISING_ROWS_SPLIT_ACC": "1"}, ["small_multirow_3d", "v1_offset_gw0"], _split_acc),
    ({"ISING_ROWS_GRID_PCT": "40"}, ["small_multirow_3d", "noncube_ragged", "wtiles9_v1"], None),
    ({"ISING_NO_CLUSTER": "1"}, ["acc_at_8192_words", "cluster_3d_8192_words"], _no_cluster),
    ({"ISING_NO_CLUSTER": "1", "ISING_COOP": "1"}, ["acc_at_8192_words", "cluster_3d_8192_words"], _coop),
    ({"ISING_COOP": "1"}, ["small_multirow_3d"], _coop),   # 2^19 site-words: the cooperative limit
]

_CHILD = (
    "import json, sys\n"
    "sys.path[:0] = [%r, %r]\n"
    "import oracle_lib, test_gpu_row_walk as T\n"
    "from pyisingmontecarlo_b200 import _native as nat\n"
    "res = {n: T.run_case(nat, oracle_lib, T.CASE[n], check_kernels=False) for n in sys.argv[2:]}\n"
    "json.dump(res, open(sys.argv[1], 'w'))\n") % (ROOT, os.path.join(ROOT, "tests"))


@pytest.mark.parametrize("env,cases,check", KNOBS, ids=["+".join(f"{k}={v}" for k, v in e.items()) for e, _, _ in KNOBS])
def test_knob_changes_no_result(native, sms, env, cases, check):
    """Every case equals the mirror with the knob set (asserted in the child); the kernels show the
    knob took effect.  Knobs that only change launch attributes or grid sizes keep the default
    instantiations."""
    e = {k: v for k, v in os.environ.items() if not k.startswith("ISING_")}
    e.update(env)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "kernels.json")
        res = subprocess.run([sys.executable, "-c", _CHILD, path] + cases, env=e, timeout=900,
                             capture_output=True, text=True)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
        with open(path) as f:
            got = json.load(f)
    for name in cases:
        case = CASE[name]
        for mode, names in got[name].items():
            if check is None:
                assert_path(names, case.dims, case.E, mode == "acc", case.pmj, sms, f"{name} ({mode})")
            else:
                check(case, mode, names)
