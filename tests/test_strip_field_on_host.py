"""The field strip kernel's own source (csrc/strip_field.cu), run on the host, against the field strip
mirror (CPU suite).

One large 2D lattice bit-packed along x in a uniform longitudinal field h keeps integer energy classes:
the class of a site is (spin, satisfied bonds), dE = 2|J|(2 n_sat - 4) + 2 h sigma, and k_strip_phase_field
compares the Philox planes with exact host thresholds per class.  tests/host_emulation/emu_strip_field.cpp
runs it one OS thread per CUDA thread, as one strip and as three strips exchanging ghost rows (one row per
phase, or 2k rows of both colours per k sweeps with the redundant ghost-row updates of phase_ext), on whole
and partial row ranges, and the bits must equal tests/strip_field_mirror.c: msc_mirror_single_field.  The
mirror itself is pinned twice without a device: at h = 0 the kernel equals msc_mirror_single, and on a
64 x 4 lattice the mirror samples the law of the torus field mirror (msc_mirror_run_field), which also fixes
the sign of h."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from field_check import mirror_field
from strip_field_check import mirror_single_field, schedule, strip_energy
from test_device_source_on_host import CSRC, EMU, layout_index, prepare_sources, strip_pack, strip_unpack, torus


def prepare_strip_field_sources(dst):
    """prepared/ of prepare_sources plus strip_field.cu without its launchers and its dependent-launch
    control (exact, asserted cuts)"""
    prepare_sources(dst)
    src = open(os.path.join(CSRC, "strip_field.cu")).read()
    marker = "template <int V>\nstatic int strip_field_dispatch("
    assert src.count(marker) == 1, "launchers of strip_field.cu"
    src = src[:src.find(marker)] + "\n}  // namespace ising\n"
    for ptx in ('    asm volatile("griddepcontrol.launch_dependents;");\n',
                '    asm volatile("griddepcontrol.wait;" ::: "memory");\n'):
        assert src.count(ptx) == 1, ptx
        src = src.replace(ptx, "")
    code = re.sub(r"//.*", "", src)
    assert "<<<" not in src and "asm" not in code and "__shared__" not in code and code.count("__global__") == 1
    open(os.path.join(dst, "strip_field_kernel.cuh"), "w").write(src)


@pytest.fixture(scope="module")
def emu_sf(tmp_path_factory):
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if shutil.which("g++") is None or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA toolkit headers (vector types) to build the host emulation")
    build = str(tmp_path_factory.mktemp("strip_field_emulation"))
    prepare_strip_field_sources(os.path.join(build, "prepared"))
    so = os.path.join(build, "libemu_strip_field.so")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-w",
                          "-I", EMU, "-I", build, "-I", cuda_inc, os.path.join(EMU, "emu_strip_field.cpp"), "-o", so],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    lib = C.CDLL(so)
    lib.emu_strip_phase_field.restype = C.c_int
    lib.emu_strip_phase_field.argtypes = [C.c_void_p] + [C.c_uint32] * 7 + [C.c_uint64, C.c_uint32, C.c_double, C.c_double,
                                                                           C.c_double, C.c_int, C.c_int, C.c_uint32,
                                                                           C.c_uint32, C.c_uint32]
    return lib


def run_strips(emu, init, j, seed, betas, fields, K, rounds, nstrips=1, mode="phase", k=1, sms=2):
    """The kernel on `nstrips` equal strips of the lattice `init` (bool[Ly, Lx]), exchanging ghost rows by hand:
    mode "phase"  one row of the colour about to be read per phase, the local rows in one launch;
    mode "pieces" the same with the local rows in three launches (first row, interior, last row), as the
                  overlapped exchange of SingleLattice2D issues them;
    mode "deep"   2 nb rows of both colours per batch of nb <= k sweeps, phase q of the batch on the local
                  rows plus 2 nb - 1 - q ghost rows on each side (ising_strip_phase_ext)."""
    Ly, Lx = init.shape
    Wr, rows = Lx // 64, Ly // nstrips
    G = 2 * k if mode == "deep" else 1
    assert rows * nstrips == Ly and rows % 2 == 0 and G <= rows
    full = strip_pack(init, Wr)
    strips = []
    for s in range(nstrips):
        buf = np.zeros((2, rows + 2 * G, Wr), dtype=np.uint32)
        buf[:, G:G + rows] = full[:, s * rows:(s + 1) * rows]
        strips.append(buf)

    def exchange(colours, d):
        for s, buf in enumerate(strips):
            for c in colours:
                buf[c, G - d:G] = strips[(s - 1) % nstrips][c, G + rows - d:G + rows]
                buf[c, G + rows:G + rows + d] = strips[(s + 1) % nstrips][c, G:G + d]

    def phase(c, t, r0, r1):
        for s, buf in enumerate(strips):
            rc = emu.emu_strip_phase_field(buf.ctypes.data, Wr, rows, s * rows, Ly, G, c, t, seed,
                                           0xFFFFFFFF if j > 0 else 0, float(betas[t]), abs(j), float(fields[t]), K,
                                           rounds, r0, r1 - r0, sms)
            assert rc == 0, rc

    betas, fields = schedule(betas, fields)
    if mode == "deep":
        i = 0
        while i < len(betas):
            nb = min(k, len(betas) - i)
            exchange((0, 1), 2 * nb)
            for q in range(2 * nb):
                ext = 2 * nb - 1 - q
                phase(q & 1, i + q // 2, G - ext, G + rows + ext)
            i += nb
    else:
        for t in range(len(betas)):
            for c in (0, 1):
                exchange((1 - c,), 1)
                if mode == "pieces":
                    for r0, r1 in ((G + 1, G + rows - 1), (G, G + 1), (G + rows - 1, G + rows)):
                        phase(c, t, r0, r1)
                else:
                    phase(c, t, G, G + rows)
    return strip_unpack(np.concatenate([b[:, G:G + rows] for b in strips], axis=1), Lx)


# Lx, Ly, j, h / |J|, betas, planes, rounds, strips, mode, k
CASES = [
    (64, 8, -1.0, 0.1, [0.3, 0.44, 2.0], 6, 7, 1, "phase", 1),          # Wr = 1 (V = 1)
    (128, 12, 1.0, -0.1, [0.25, 0.6, 3.0], 5, 10, 3, "phase", 1),       # antiferromagnet, V = 2, three strips
    (192, 8, -0.5, 2.0, [0.5, 3.0, 4.0], 7, 7, 2, "pieces", 1),         # Wr = 3; h = 2|J|: classes with dE = 0
    (256, 8, -1.5, 4.0, [0.3, 1.0], 6, 10, 1, "pieces", 1),             # V = 4, |J| = 1.5, h = 4|J|
    (256, 12, 0.5, 7.0, [0.2, 0.44, 1.5], 7, 10, 3, "deep", 2),         # h = 7|J|: every up class uphill
    (128, 16, -1.0, -7.0, [0.3, 0.8, 0.44], 5, 7, 1, "deep", 1),        # h = -7|J|, one strip wrapping deep
    (64, 8, 1.5, 2.0, [0.4, 5.0, 5.0], 6, 7, 2, "deep", 2),             # antiferromagnet |J| = 1.5, high beta: ties
]


@pytest.mark.parametrize("Lx,Ly,j,hj,betas,K,rounds,nstrips,mode,k", CASES)
def test_field_strip_source_equals_the_mirror(emu_sf, Lx, Ly, j, hj, betas, K, rounds, nstrips, mode, k):
    rng = np.random.default_rng(Lx * 7 + Ly + K)
    init = rng.integers(0, 2, size=(Ly, Lx)).astype(bool)
    seed, h = 0x0123456789ABCDEF + Lx, hj * abs(j)
    got = run_strips(emu_sf, init, j, seed, betas, h, K, rounds, nstrips, mode, k)
    ref, nsat, up = mirror_single_field(Lx, Ly, j, seed, betas, h, K, rounds, state=init)
    assert (got == ref).all(), f"kernel source on the host differs from the mirror: {(got != ref).sum()} spins"
    assert (got != init).mean() > 0.02                                   # (the sweeps did move the spins)
    assert up[-1] == ref.sum()


# a field reversal through zero, changing inside the batches of the deep exchange
SCHEDULE_BETAS = [0.44, 0.44, 0.6, 0.6, 0.44, 1.0, 0.44]
SCHEDULE_FIELDS = [0.5, -0.5, 0.0, -0.0, 2.0, -2.0, 0.1]


@pytest.mark.parametrize("nstrips,mode,k", [(1, "phase", 1), (3, "pieces", 1), (3, "deep", 3), (1, "deep", 4)])
def test_field_schedule_equals_the_mirror(emu_sf, nstrips, mode, k):
    Lx, Ly = 128, 24
    rng = np.random.default_rng(5)
    init = rng.integers(0, 2, size=(Ly, Lx)).astype(bool)
    got = run_strips(emu_sf, init, -1.0, 77, SCHEDULE_BETAS, SCHEDULE_FIELDS, 6, 7, nstrips, mode, k)
    ref, _, _ = mirror_single_field(Lx, Ly, -1.0, 77, SCHEDULE_BETAS, SCHEDULE_FIELDS, state=init)
    assert (got == ref).all(), f"{(got != ref).sum()} spins differ"


@pytest.mark.parametrize("Lx,Ly,j,K,rounds,nstrips", [(128, 8, -1.0, 6, 7, 1), (256, 12, 0.5, 7, 10, 3)])
def test_field_kernel_at_zero_field_is_the_plain_mirror(emu_sf, oracle, Lx, Ly, j, K, rounds, nstrips):
    """k_strip_phase_field forced to h = +-0 (the library runs k_strip_phase there) gives msc_mirror_single's
    bits: the thresholds of the classes at h = 0 are the plain strip's, the dE <= 0 classes flip as there"""
    rng = np.random.default_rng(Lx)
    init = rng.integers(0, 2, size=(Ly, Lx)).astype(bool)
    betas = [0.3, 0.44, 0.7]
    _, ref = oracle.msc_mirror_single(Lx, Ly, j, 99, betas, planes=K, rounds=rounds, state=init)
    for h in (0.0, -0.0):
        got = run_strips(emu_sf, init, j, 99, betas, h, K, rounds, nstrips)
        assert (got == ref).all(), (h, (got != ref).sum())
    ref_f, _, _ = mirror_single_field(Lx, Ly, j, 99, betas, [0.0, -0.0, 0.0], K, rounds, state=init)
    assert (ref_f == ref).all()


@pytest.mark.parametrize("beta,h", [(0.4, 0.3), (0.3, -0.8)])
def test_strip_field_mirror_samples_the_torus_field_law(beta, h):
    """64 x 4 ferromagnet: <E>/N and <m> of the strip mirror (independent chains, one per seed) within 4 sigma
    of the torus field mirror's (replicas of the same lattice as an edge list); the sign of m follows h"""
    Lx, Ly, N = 64, 4, 256
    burn, nsamp, chains = 60, 120, 96
    rng = np.random.default_rng(0)
    a, b, jj = torus((Lx, Ly, 1), rng, False, -1.0)
    _, colors = layout_index((Lx, Ly, 1))
    # torus mirror: replicas, E and m after every sweep of the sampling window
    _, st = mirror_field(a, b, jj, N, colors, chains, 3, [beta] * burn, h)
    e_t, m_t = [], []
    for t in range(nsamp):
        en, st = mirror_field(a, b, jj, N, colors, chains, 3, [beta], h, states=st, sweep0=burn + t)
        e_t.append(en / N)
        m_t.append(st.mean(axis=1) * 2 - 1)
    e_t, m_t = np.array(e_t).T, np.array(m_t).T                            # [chain, sample]
    # strip mirror: one chain per seed
    e_s, m_s = [], []
    for seed in range(chains):
        _, nsat, up = mirror_single_field(Lx, Ly, -1.0, 1000 + seed, [beta] * (burn + nsamp), h)
        e_s.append(strip_energy(-1.0, h, N, nsat[burn:], up[burn:]) / N)
        m_s.append((2 * up[burn:] - N) / N)
    e_s, m_s = np.array(e_s), np.array(m_s)

    def moments(x):
        per_chain = x.mean(axis=1)
        return per_chain.mean(), per_chain.std(ddof=1) / np.sqrt(len(per_chain))

    for x, y, what in ((e_s, e_t, "E"), (m_s, m_t, "m")):
        (mx, sx), (my, sy) = moments(x), moments(y)
        assert abs(mx - my) < 4 * np.hypot(sx, sy), (what, mx, sx, my, sy)
    assert np.sign(m_s.mean()) == np.sign(h)
