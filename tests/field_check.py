"""Helpers of the field tests (test_field_on_host.py, test_gpu_field.py): the field mirror
(tests/field_mirror.c: msc_mirror_run_field on top of the unchanged oracle/msc_mirror.c, built here
with the oracle's flags),
and the exact law of a small torus in a field."""
import ctypes as C
import itertools
import os
import shutil
import subprocess
import tempfile

import numpy as np

_P = C.c_void_p
_U64 = C.c_uint64
HERE = os.path.dirname(os.path.abspath(__file__))
_handle = None


def _lib():
    """tests/field_mirror.c compiled once per process into a temporary directory (the tree may be read-only)"""
    global _handle
    if _handle is not None:
        return _handle
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    tmp = tempfile.mkdtemp(prefix="field_mirror_")
    out = os.path.join(tmp, "libfield_mirror.so")
    res = subprocess.run([cc, "-O2", "-fPIC", "-fopenmp", "-fvisibility=hidden", "-ffp-contract=off", "-shared", "-o", out,
                          os.path.join(HERE, "field_mirror.c"), "-lm"], capture_output=True, text=True)
    assert res.returncode == 0, "field mirror build failed:\n" + res.stdout + res.stderr
    h = C.CDLL(out)
    shutil.rmtree(tmp, ignore_errors=True)            # the loaded mapping stays valid
    f = h.msc_mirror_run_field
    f.restype = C.c_int
    f.argtypes = [_U64, _U64, _P, _P, _P, _P, C.c_uint32, _U64, _U64, _U64, C.c_int, C.c_int, C.c_int, _P, _P,
                  _U64, _U64, _P, _P, _P, C.c_int, C.c_double]
    _handle = h
    return h


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def mirror_field(a, b, j, nvars, colors, E, seed, betas, h, *, replica_offset=0, planes=6, rounds=7,
                 init_state=None, states=None, sweep0=0, per_sweep=False):
    """msc_mirror_run_field: the production sweep in the uniform field h (one beta per sweep).
    -> (energies [E, nsweeps] when per_sweep else [E], states bool[E, nvars])"""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    j = np.ascontiguousarray(j, dtype=np.float64)
    colors = np.ascontiguousarray(colors, dtype=np.uint32)
    betas = np.ascontiguousarray(betas, dtype=np.float64)
    randomize = int(states is None and init_state is None)
    st = np.zeros((E, nvars), dtype=np.uint8) if states is None else np.ascontiguousarray(states, dtype=np.uint8).copy()
    init = None if init_state is None else np.ascontiguousarray(init_state, dtype=np.uint8)
    eps = np.zeros((E, len(betas))) if per_sweep else None
    fin = np.zeros(E)
    rc = _lib().msc_mirror_run_field(nvars, len(a), _p(a), _p(b), _p(j), _p(colors), int(colors.max()) + 1, E,
                                     int(seed), replica_offset, planes, rounds, randomize, _p(init), _p(betas),
                                     len(betas), sweep0, _p(st), _p(eps), _p(fin), 0, float(h))
    assert rc == 0, rc
    return (eps if per_sweep else fin), st.astype(bool)


def energies_from_states(states, a, b, j, h):
    """E = sum J s s' - h sum s (s = +1 for True), as the library forms it: |J| (nbonds - 2 nsat) + h (N - 2 up)"""
    s = states.astype(np.int64) * 2 - 1
    nsat = ((s[:, a.astype(np.int64)] * s[:, b.astype(np.int64)] * np.sign(j)[None, :]) < 0).sum(axis=1)
    up = states.sum(axis=1).astype(np.int64)
    jabs = abs(float(j[0]))
    return jabs * (len(a) - 2 * nsat).astype(np.float64) + h * (states.shape[1] - 2 * up).astype(np.float64)


def exact_moments(a, b, j, nvars, beta, h):
    """<E>, <m> (m = sum s / N) of the Boltzmann law by enumeration of all 2^nvars states"""
    s = np.array(list(itertools.product([-1, 1], repeat=nvars)), dtype=np.float64)
    en = (s[:, a.astype(np.int64)] * s[:, b.astype(np.int64)] * j[None, :]).sum(axis=1) - h * s.sum(axis=1)
    w = np.exp(-beta * (en - en.min()))
    w /= w.sum()
    return float((w * en).sum()), float((w * s.mean(axis=1)).sum())
