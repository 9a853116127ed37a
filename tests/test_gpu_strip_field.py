"""One large 2D lattice in a uniform longitudinal field on the device (k_strip_phase_field, csrc/strip_field.cu;
run with -m gpu on a B200): every instantiation bit for bit against the field strip mirror
(tests/strip_field_mirror.c) through ising_strip_set_field + phases and through ising_strip_sweeps_field at
every exchange depth, with the kernel chosen per sweep by h != 0; strips exchanging by hand; the opt-in fused
pass; SingleLattice2D's energy and magnetization; the law against Lattice.torus(...).set_global_bias; every
refusal; and NCCL strips on several GPUs."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from mirror_check import instances, launched
from strip_field_check import mirror_single_field, strip_energy

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INSTANCES = [(K, R, Lx) for K in (5, 6, 7) for R in (7, 10) for Lx in (64, 128, 256)]   # Wr = 1 / 2 / 4 -> V
PHASE_BETAS = [0.3, 0.44, 2.0, 0.44]
SCHED_BETAS = [0.3, 0.44, 1.5, 0.44, 0.7, 0.2, 0.6]


def _case(K, R, Lx):
    """coupling, constant field and field schedule of one instantiation (|J| and h vary over the cases)"""
    i = INSTANCES.index((K, R, Lx))
    jabs = (0.5, 1.0, 1.5)[i % 3]
    j = jabs if i % 4 == 1 else -jabs
    h = (0.1, -0.1, 2.0, 4.0, 7.0, -7.0)[i % 6] * jabs
    fields = [h, -h, 0.0, 2.0 * jabs, -0.0, h, -2.0 * jabs]
    return j, h, fields


def _instance(nat, K, R, Lx):
    """set_field + phases, then sweeps_field at exchange_every 0 / 1 / 3 / 8: the mirror's bits; -> kernel names
    of the phase run"""
    ctx = nat.Context.get(0)
    Ly = 16
    j, h, fields = _case(K, R, Lx)
    seed = 1000 + 7 * Lx + K
    strip = nat.Strip(ctx, Lx, Ly, 0, Ly, j, seed, K, R)
    strip.set_field(h)

    def phases():
        for beta in PHASE_BETAS:
            for colour in (0, 1):
                strip.wrap_local(1 - colour)
                strip.phase(colour, beta)

    _, names = launched(phases)
    ref, _, _ = mirror_single_field(Lx, Ly, j, seed, PHASE_BETAS, h, K, R)
    got = strip.rows()
    assert (got == ref).all(), (K, R, Lx, "phases", int((got != ref).sum()))
    strip.close()
    ref, _, _ = mirror_single_field(Lx, Ly, j, seed, SCHED_BETAS, fields, K, R)
    for k in (0, 1, 3, 8):
        s = nat.Strip(ctx, Lx, Ly, 0, Ly, j, seed, K, R, ghost=16)
        s.sweeps(SCHED_BETAS, None, k, fields=fields)
        got = s.rows()
        assert (got == ref).all(), (K, R, Lx, "exchange_every", k, int((got != ref).sum()))
        s.close()
    return names


SCHEDULE = [0.5, 0.0, -0.5, -0.0, 2.0, 0.0, -7.0]


def _per_sweep(nat, k):
    """sweeps_field one sweep at a time: kernel names of each sweep; the whole schedule equals the mirror"""
    ctx = nat.Context.get(0)
    Lx, Ly = 256, 16
    s = nat.Strip(ctx, Lx, Ly, 0, Ly, -1.0, 31, ghost=16)
    names = []
    for beta, h in zip(SCHED_BETAS, SCHEDULE):
        _, n = launched(lambda: s.sweeps([beta], None, k, fields=[h]))
        names.append(n)
    ref, _, _ = mirror_single_field(Lx, Ly, -1.0, 31, SCHED_BETAS, SCHEDULE)
    assert (s.rows() == ref).all(), k
    s.close()
    return names


# The profiler attaches CUPTI to its process (DESIGN section 2, item 7): every profiled run happens here.
_CHILD = (
    "import json, sys\n"
    "sys.path[:0] = [%r, %r]\n"
    "import test_gpu_strip_field as T\n"
    "from pyisingmontecarlo_b200 import _native as nat\n"
    "res = {'%%d,%%d,%%d' %% c: T._instance(nat, *c) for c in T.INSTANCES}\n"
    "res.update({'sweeps_k%%d' %% k: T._per_sweep(nat, k) for k in (1, 3)})\n"
    "json.dump(res, open(sys.argv[1], 'w'))\n") % (ROOT, os.path.join(ROOT, "tests"))


def test_every_instantiation_matches_mirror(native):
    """K 5/6/7 x rounds 7/10 x V 1/2/4 against the mirror, as phases and as library loops at every exchange
    depth (asserted in one child process, which records the kernels); each phase run launched only the
    instantiation launch_strip_phase_field picks, and sweeps_field ran k_strip_phase_field exactly for the
    sweeps with h != 0 and k_strip_phase for the others"""
    e = {k: v for k, v in os.environ.items() if not k.startswith("ISING_")}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "kernels.json")
        res = subprocess.run([sys.executable, "-c", _CHILD, path], env=e, timeout=900, capture_output=True, text=True)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
        got = json.load(open(path))
    for K, R, Lx in INSTANCES:
        names = got["%d,%d,%d" % (K, R, Lx)]
        Wr = Lx // 64
        V = 4 if Wr % 4 == 0 else (2 if Wr % 2 == 0 else 1)
        assert instances(names, "k_strip_phase_field") == {(K, R, V)}, (K, R, Lx, names)
        assert not instances(names, "k_strip_phase"), names
    for k in (1, 3):
        per = got["sweeps_k%d" % k]
        assert len(per) == len(SCHEDULE)
        for h, names in zip(SCHEDULE, per):
            field, plain = instances(names, "k_strip_phase_field"), instances(names, "k_strip_phase")
            if h != 0.0:
                assert field == {(6, 7, 4)} and not plain, (k, h, names)
            else:
                assert plain == {(6, 7, 4)} and not field, (k, h, names)


def test_strips_in_a_field_reproduce_single_strip(native):
    """Three strips exchanging by hand - one row per phase, and 4 rows of both colours per 2 sweeps with
    phase_ext - equal one strip in a field schedule that changes sign and passes through 0"""
    ctx = native.Context.get(0)
    Lx, Ly, G = 128, 24, 4
    bounds = ((0, 6), (6, 16), (16, 24))
    betas = (0.4, 0.5, 0.3, 0.6)
    fields = (0.3, 0.0, -0.3, -2.0)
    whole = native.Strip(ctx, Lx, Ly, 0, Ly, -1.0, 5)
    for beta, h in zip(betas, fields):
        whole.set_field(h)
        for colour in (0, 1):
            whole.wrap_local(1 - colour)
            whole.phase(colour, beta)
    ref, _, _ = mirror_single_field(Lx, Ly, -1.0, 5, betas, fields)
    assert (whole.rows() == ref).all()
    parts = [native.Strip(ctx, Lx, Ly, lo, hi, -1.0, 5) for lo, hi in bounds]
    for beta, h in zip(betas, fields):
        for p in parts:
            p.set_field(h)
        for colour in (0, 1):
            for k, p in enumerate(parts):
                up, down = parts[(k - 1) % 3], parts[(k + 1) % 3]
                p.set_ghost(1 - colour, 0, up.get_boundary(1 - colour, 1))
                p.set_ghost(1 - colour, 1, down.get_boundary(1 - colour, 0))
            for p in parts:
                p.phase(colour, beta)
    assert (np.concatenate([p.rows() for p in parts]) == ref).all()
    deep = [native.Strip(ctx, Lx, Ly, lo, hi, -1.0, 5, ghost=G) for lo, hi in bounds]
    for i in range(0, len(betas), 2):
        bufs = []
        for p in deep:
            b = np.empty((2, 2, G, p.words), dtype=np.uint32)
            p.halo_deep(0, G, b)
            bufs.append(b)
        for k, p in enumerate(deep):
            r = np.empty((2, 2, G, p.words), dtype=np.uint32)
            r[0] = bufs[(k - 1) % 3][1]
            r[1] = bufs[(k + 1) % 3][0]
            p.halo_deep(1, G, r)
        for q in range(4):
            for p in deep:
                p.set_field(fields[i + q // 2])
                p.phase_ext(q & 1, betas[i + q // 2], 3 - q, advance=bool(q & 1), sync=True)
    assert (np.concatenate([p.rows() for p in deep]) == ref).all()


_FUSED = (
    "import os, sys\n"
    "sys.path[:0] = [%r, %r]\n"
    "from pyisingmontecarlo_b200 import _native as nat\n"
    "from strip_field_check import mirror_single_field\n"
    "assert os.environ.get('ISING_STRIP_FUSE') == '1'\n"
    "ctx = nat.Context.get(0)\n"
    "betas, fields = [0.3, 0.44, 0.8, 0.44, 0.5, 0.2], [0.2, 0.0, -0.4, 0.0, 3.0, 0.0]\n"
    "for Lx, Ly, k in ((256, 32, 2), (1024, 48, 3)):\n"
    "    ref, _, _ = mirror_single_field(Lx, Ly, -1.0, 21, betas, fields)\n"
    "    s = nat.Strip(ctx, Lx, Ly, 0, Ly, -1.0, 21, ghost=2 * k)\n"
    "    s.sweeps(betas, None, k, fields=fields)\n"
    "    assert (s.rows() == ref).all(), (Lx, Ly, k)\n"
    "    # one sweep per call: launches of each sweep (fused pass 1, phases 2)\n"
    "    t, per = nat.Strip(ctx, Lx, Ly, 0, Ly, -1.0, 21, ghost=2 * k), []\n"
    "    for b, h in zip(betas, fields):\n"
    "        t.stats(reset=True)\n"
    "        t.sweeps([b], None, k, fields=[h])\n"
    "        per.append(t.stats()['launches'])\n"
    "    assert (t.rows() == ref).all(), (Lx, Ly, k)\n"
    "    assert all(n == 2 for n, h in zip(per, fields) if h != 0.0), per\n"
    "    assert any(n == 1 for n, h in zip(per, fields) if h == 0.0), per\n"
    "    print(Lx, Ly, k, 'launches per sweep', per)\n"
    "print('STRIP_FIELD_FUSED_OK')\n") % (ROOT, os.path.join(ROOT, "tests"))


def test_fused_knob_changes_no_bit_in_a_field(native):
    """ISING_STRIP_FUSE=1 (in a process of its own): a field schedule keeps the mirror's bits; sweeps with
    h != 0 run the two phase launches, and h = 0 sweeps do take the fused pass"""
    env = dict(os.environ, ISING_STRIP_FUSE="1", ISING_STRIP_FUSE_MIN_ROWS="1")
    res = subprocess.run([sys.executable, "-c", _FUSED], capture_output=True, text=True, timeout=600, env=env)
    assert "STRIP_FIELD_FUSED_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]


@pytest.mark.parametrize("k", [0, 2])
def test_single_lattice_energy_and_magnetization(native, k):
    """SingleLattice2D in a schedule: after every sweep energy() = |J|(2N - 2 n_sat) - h M and magnetization()
    = 2 up - N with the mirror's counts; the field property follows the schedule"""
    import pyisingmontecarlo_b200 as pkg

    Lx, Ly, j = 128, 16, -1.5
    betas = [0.3, 0.44, 0.8, 0.44, 0.6]
    fields = [0.45, 0.0, -0.45, -3.0, 0.15]
    lat = pkg.SingleLattice2D(Lx, Ly, j=j, seed=77, exchange_every=k, field=0.45)
    assert lat.field == 0.45
    ref, nsat, up = mirror_single_field(Lx, Ly, j, 77, betas, fields)
    lat.sweeps(betas[:1])                                            # in the field given at construction
    for t in range(1, len(betas)):
        assert lat.energy() == strip_energy(j, fields[t - 1], Lx * Ly, int(nsat[t - 1]), int(up[t - 1]))
        assert lat.magnetization() == 2 * int(up[t - 1]) - Lx * Ly
        lat.sweeps(betas[t:t + 1], fields[t:t + 1])
        assert lat.field == fields[t]
    assert (lat.local_rows() == ref).all()
    assert lat.energy() == strip_energy(j, fields[-1], Lx * Ly, int(nsat[-1]), int(up[-1]))
    lat2 = pkg.SingleLattice2D(Lx, Ly, j=j, seed=77, exchange_every=k)
    lat2.sweeps(betas, fields)                                      # the whole schedule in one call
    assert (lat2.local_rows() == ref).all() and lat2.field == fields[-1]
    lat3 = pkg.SingleLattice2D(Lx, Ly, j=j, seed=77, exchange_every=k)
    lat3.set_field(0.45)
    lat3.sweeps(betas[:1])
    lat3.sweeps(betas[1:], 0.0)                                      # a scalar: one field for every sweep
    ref0, _, _ = mirror_single_field(Lx, Ly, j, 77, betas, [0.45] + [0.0] * (len(betas) - 1))
    assert (lat3.local_rows() == ref0).all() and lat3.field == 0.0


def test_statistics_against_the_torus_field_path(native):
    """1024^2 ferromagnet at beta = 0.5, h = 0.05 from the all-up state: <E>/N and <m> of the single lattice
    (batch means over sweeps) within 4 sigma of Lattice.torus((1024, 1024)).set_global_bias(0.05) (32 replicas)"""
    import pyisingmontecarlo_b200 as pkg

    L, beta, h, therm, nsamp = 1024, 0.5, 0.05, 200, 400
    N = L * L
    lat = pkg.SingleLattice2D(L, seed=13, field=h)
    lat.set_all(True)
    lat.sweeps([beta] * therm)
    es, ms = [], []
    for _ in range(nsamp // 8):
        lat.sweeps([beta] * 8)
        es.append(lat.energy() / N)
        ms.append(lat.magnetization() / N)
    es, ms = np.array(es), np.array(ms)
    tor = pkg.Lattice.torus((L, L), j=-1.0, seed_gen=14)
    tor.set_global_bias(h)
    tor.set_initial_state(np.ones(N, dtype=bool))
    e_t, m_t, _ = tor.run_monte_carlo_observables(beta, nsamp, 32, thermalization_time=therm, sampling_freq=8,
                                                  overlaps=False)

    def batch(x, nb=10):
        b = x[: len(x) // nb * nb].reshape(nb, -1).mean(axis=1)
        return b.mean(), b.std(ddof=1) / np.sqrt(nb)

    def reps(x):
        per = x.mean(axis=1) / N
        return per.mean(), per.std(ddof=1) / np.sqrt(len(per))

    for (ms_, ss), (mt, st), what in ((batch(es), reps(e_t), "E"), (batch(ms), reps(m_t), "m")):
        assert abs(ms_ - mt) < 4 * np.hypot(ss, st), (what, ms_, ss, mt, st)
    assert ms.mean() > 0.9


def test_refusals(native):
    import pyisingmontecarlo_b200 as pkg

    with pytest.raises(ValueError, match="finite"):
        pkg.SingleLattice2D(64, 4, field=float("nan"))
    lat = pkg.SingleLattice2D(64, 4)
    for bad in (float("nan"), float("inf"), -float("inf")):
        with pytest.raises(ValueError, match="finite"):
            lat.set_field(bad)
        with pytest.raises(ValueError, match="finite"):
            lat.sweeps([0.4, 0.4], [0.1, bad])
        with pytest.raises(ValueError, match="finite"):
            lat.strip.set_field(bad)
        with pytest.raises(ValueError, match="finite"):
            lat.strip.sweeps([0.4], fields=[bad])
    with pytest.raises(ValueError, match="one value per beta"):
        lat.sweeps([0.4, 0.4, 0.4], [0.1, 0.2])
    with pytest.raises(ValueError, match="one value per beta"):
        lat.strip.sweeps([0.4, 0.4], fields=[0.1])
    assert lat.field == 0.0
    lat.sweeps([0.4], [0.2])                                         # still usable after the refusals
    assert lat.field == 0.2


def test_multi_gpu_field_strips_under_torchrun(native):
    """Runs tests/multi_gpu_strip_field_check.py on every visible GPU (skipped on a 1-GPU box)."""
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = min(n, 4)
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                          "--master-addr", "127.0.0.1", "--master-port", "29537",
                          os.path.join(ROOT, "tests", "multi_gpu_strip_field_check.py")],
                         capture_output=True, text=True, timeout=240)
    assert "MULTI_GPU_STRIP_FIELD_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
