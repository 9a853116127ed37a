"""The field kernels' own source (csrc/sweep_field.cu), run on the host, against the field mirror (CPU suite).

A torus in a uniform longitudinal field h keeps integer energy classes: the class of a site is
(spin, satisfied bonds), dE = 2|J|(2 n_sat - 2 DIM) + 2 h sigma, and the bit-sliced kernel compares the
Philox planes with exact host thresholds per class.  tests/host_emulation/ runs k_sweep_field and
k_energy_field one OS thread per CUDA thread (as test_device_source_on_host.py does for the other
kernels) and the bits and per-sweep energies must equal tests/field_mirror.c: msc_mirror_run_field.
The mirror itself is pinned twice without a device: at h = 0 it is msc_mirror_run, and on a 4 x 4
torus in a field it samples the exact Boltzmann law (which also fixes the sign of h)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from field_check import energies_from_states, exact_moments, mirror_field
from test_device_source_on_host import CSRC, EMU, ROOT, bond_masks, layout_index, pack, prepare_sources, torus, unpack


def prepare_field_sources(dst):
    """prepared/ of prepare_sources plus sweep_field.cu without its launchers (exact, asserted cut)"""
    prepare_sources(dst)
    src = open(os.path.join(CSRC, "sweep_field.cu")).read()
    marker = "template <int DIM, bool PMJ, int K, int ROUNDS, int V>\nstatic int field_launch("
    assert src.count(marker) == 1, "launchers of sweep_field.cu"
    src = src[:src.find(marker)] + "\n}  // namespace ising\n"
    code = re.sub(r"//.*", "", src)
    assert "<<<" not in src and "asm" not in code and "__shared__" not in code and code.count("__global__") == 2
    assert "static void field_launch_shape(" in src
    open(os.path.join(dst, "field_kernels.cuh"), "w").write(src)


@pytest.fixture(scope="module")
def emu_field(tmp_path_factory):
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if shutil.which("g++") is None or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA toolkit headers (vector types) to build the host emulation")
    build = str(tmp_path_factory.mktemp("field_emulation"))
    prepare_field_sources(os.path.join(build, "prepared"))
    so = os.path.join(build, "libemu_field.so")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-w",
                          "-I", EMU, "-I", build, "-I", cuda_inc, os.path.join(EMU, "emu_field.cpp"), "-o", so],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    lib = C.CDLL(so)
    lib.emu_sweep_field.restype = C.c_int
    lib.emu_sweep_field.argtypes = [C.c_int] + [C.c_uint32] * 4 + [C.c_int, C.c_void_p, C.c_uint32, C.c_void_p,
                                   C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_double, C.c_double,
                                   C.c_double, C.c_uint32]
    lib.emu_energy_field.restype = None
    lib.emu_energy_field.argtypes = [C.c_void_p, C.c_void_p] + [C.c_uint64] * 3 + [C.c_double, C.c_uint64, C.c_double,
                                                                                  C.c_uint64, C.c_void_p, C.c_uint64,
                                                                                  C.c_uint64]
    return lib


CASES = [
    # dims, E, V, pmj, j0, h, betas, planes, rounds, gw0, sms
    ((8, 6, 4), 128, 4, True, -1.0, 0.3, [0.2, 0.9], 6, 7, 3, 2),           # config 3's shape, +-J in a field
    ((4, 4, 6), 96, 1, True, -1.0, 2.0, [0.5, 3.0], 5, 10, 0, 1),           # h = 2|J|: classes with dE = 0; ties
    ((6, 4, 2), 64, 2, False, 1.0, -0.1, [0.25, 0.6], 7, 7, 1, 2),          # antiferromagnet, h = -0.1|J|, Lz = 2
    ((16, 8, 1), 128, 4, False, -1.0, 7.0, [0.3, 0.44], 6, 10, 0, 2),       # 2D, h = 7|J|: every up class uphill
    ((12, 6, 1), 40, 2, True, -1.5, 0.15, [0.4, 2.5], 7, 10, 5, 1),         # |J| = 1.5, h = 0.1|J|, ragged E
    ((10, 10, 1), 70, 1, False, -0.5, 1.0, [1.0, 4.0], 5, 7, 2, 1),         # h = 2|J| at |J| = 0.5, high beta
    ((6, 6, 6), 64, 2, False, -0.7, 1.4, [0.6, 2.0], 6, 7, 0, 1),           # 3D h = 2|J|; 36 rows > 32 blocks: grid wrap
    ((4, 8, 8), 32, 1, True, -1.0, -7.0, [0.3, 1.5], 6, 7, 7, 1),           # h = -7|J|; 64 rows over 32 blocks
]


@pytest.mark.parametrize("dims,E,V,pmj,j0,h,betas,planes,rounds,gw0,sms", CASES)
def test_field_source_equals_the_mirror(emu_field, dims, E, V, pmj, j0, h, betas, planes, rounds, gw0, sms):
    rng = np.random.default_rng(abs(hash((dims, E, V, pmj, h))) & 0xFFFF)
    dim = 3 if dims[2] > 1 else 2
    a, b, j = torus(dims, rng, pmj, j0)
    N = dims[0] * dims[1] * dims[2]
    _, colors = layout_index(dims)
    W = (E + 31) // 32
    if W % V:
        W += V - W % V                                                    # pad words are idle replicas
    init = rng.integers(0, 2, size=(E, N)).astype(bool)
    seed, sweep0 = 0x0123456789ABCDEF, 11
    words = pack(init, dims, W)
    jm = None
    if pmj:                                                               # [2][2 dim][halfN] as upload_stencil_masks
        m8 = bond_masks(dims, a, b, j)
        jm = np.ascontiguousarray(m8.reshape(2, N // 2, 8)[:, :, :2 * dim].transpose(0, 2, 1))
    antiferro = 0xFFFFFFFF if (not pmj and j0 > 0) else 0
    cw = 32 * W
    nsat_hist = np.zeros((len(betas), cw), dtype=np.uint64)
    up_hist = np.zeros((len(betas), cw), dtype=np.uint64)
    for t, beta in enumerate(betas):
        rc = emu_field.emu_sweep_field(dim, dims[0], dims[1], dims[2], W, V, None if jm is None else jm.ctypes.data,
                                       antiferro, words.ctypes.data, seed, sweep0 + t, gw0, planes, rounds, float(beta),
                                       abs(j0), float(h), sms)
        assert rc == 0, rc
        st = unpack(words, dims, E)
        s = st.astype(np.int64) * 2 - 1
        nsat_hist[t, :E] = ((s[:, a.astype(np.int64)] * s[:, b.astype(np.int64)] * np.sign(j)[None, :]) < 0).sum(axis=1)
        up_hist[t, :E] = st.sum(axis=1)
    en = np.zeros((E, len(betas)))
    emu_field.emu_energy_field(nsat_hist.ctypes.data, up_hist.ctypes.data, E, cw, len(betas), abs(j0), len(a), float(h),
                               N, en.ctypes.data, len(betas), 0)
    got = unpack(words, dims, E)
    en_ref, st_ref = mirror_field(a, b, j, N, colors, E, seed, betas, h, replica_offset=32 * gw0, planes=planes,
                                  rounds=rounds, states=init, sweep0=sweep0, per_sweep=True)
    assert (got == st_ref).all(), f"kernel source on the host differs from the mirror: {(got != st_ref).sum()} spins"
    assert (en == en_ref).all()
    assert (en[:, -1] == energies_from_states(got, a, b, j, h)).all()
    assert (got != init).mean() > 0.02                                    # (the sweeps did move the spins)


@pytest.mark.parametrize("dims,pmj,j0", [((8, 6, 4), True, -1.0), ((10, 6, 1), False, 1.0), ((6, 6, 6), False, -0.5)])
def test_field_mirror_at_zero_field_is_the_plain_mirror(oracle, dims, pmj, j0):
    rng = np.random.default_rng(7)
    a, b, j = torus(dims, rng, pmj, j0)
    N = dims[0] * dims[1] * dims[2]
    _, colors = layout_index(dims)
    betas = [0.1, 0.44, 1.0, 3.0]
    for E, offset in ((64, 0), (45, 96)):
        en0, st0 = oracle.msc_mirror(a, b, j, N, colors, E, 99, betas, replica_offset=offset, per_sweep=True)
        en1, st1 = mirror_field(a, b, j, N, colors, E, 99, betas, 0.0, replica_offset=offset, per_sweep=True)
        assert (st0 == st1).all() and (en0 == en1).all()
        en_neg, st_neg = mirror_field(a, b, j, N, colors, E, 99, betas, -0.0, replica_offset=offset, per_sweep=True)
        assert (st0 == st_neg).all() and (en0 == en_neg).all()


@pytest.mark.parametrize("beta,h", [(0.4, 0.3), (0.3, -0.8)])
def test_field_mirror_samples_the_exact_law(oracle, beta, h):
    """4 x 4 ferromagnetic torus: <E> and <m> of the mirror within 4 sigma of exact enumeration; with
    h > 0 the up spins (set bits) are favoured, E = sum J s s' - h sum s."""
    dims = (4, 4, 1)
    rng = np.random.default_rng(0)
    a, b, j = torus(dims, rng, False, -1.0)
    N = 16
    _, colors = layout_index(dims)
    e_ex, m_ex = exact_moments(a, b, j, N, beta, h)
    R, chunk, nchunk = 256, 4, 150
    _, st = mirror_field(a, b, j, N, colors, R, 5, [beta] * 50, h)     # thermalise
    es, ms = [], []
    for k in range(nchunk):
        en, st = mirror_field(a, b, j, N, colors, R, 5, [beta] * chunk, h, states=st, sweep0=50 + chunk * k)
        es.append(en)
        ms.append(st.mean(axis=1) * 2 - 1)
    es, ms = np.array(es), np.array(ms)                                   # [chunk, replica]
    for x, ref in ((es, e_ex), (ms, m_ex)):
        per_rep = x.mean(axis=0)
        mean, err = per_rep.mean(), per_rep.std(ddof=1) / np.sqrt(R)
        assert abs(mean - ref) < 4 * err + 1e-12, (mean, ref, err)
    assert np.sign(ms.mean()) == np.sign(h)
