"""Helpers of the field strip tests (test_strip_field_on_host.py, test_gpu_strip_field.py): the field strip
mirror (tests/strip_field_mirror.c: msc_mirror_single_field and its band variant on top of the unchanged
oracle/msc_mirror.c, built here with the oracle's flags) and the energy the library forms from its counts."""
import ctypes as C
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
    """tests/strip_field_mirror.c compiled once per process into a temporary directory (the tree may be read-only)"""
    global _handle
    if _handle is not None:
        return _handle
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    tmp = tempfile.mkdtemp(prefix="strip_field_mirror_")
    out = os.path.join(tmp, "libstrip_field_mirror.so")
    res = subprocess.run([cc, "-O2", "-fPIC", "-fopenmp", "-fvisibility=hidden", "-ffp-contract=off", "-shared", "-o", out,
                          os.path.join(HERE, "strip_field_mirror.c"), "-lm"], capture_output=True, text=True)
    assert res.returncode == 0, "strip field mirror build failed:\n" + res.stdout + res.stderr
    h = C.CDLL(out)
    shutil.rmtree(tmp, ignore_errors=True)            # the loaded mapping stays valid
    h.msc_mirror_single_field.restype = C.c_int
    h.msc_mirror_single_field.argtypes = [_U64, _U64, C.c_double, _U64, C.c_int, C.c_int, C.c_int, _P, _P, _U64, _P,
                                          _P, _P]
    h.msc_mirror_single_band_field.restype = C.c_int
    h.msc_mirror_single_band_field.argtypes = [_U64, _U64, _U64, C.c_double, _U64, C.c_int, C.c_int, C.c_int, _P, _P,
                                               _U64, _P]
    _handle = h
    return h


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def schedule(betas, fields):
    """(betas, fields) as f64 arrays of one length; a scalar field applies to every sweep"""
    betas = np.ascontiguousarray(np.atleast_1d(betas), dtype=np.float64)
    fields = np.ascontiguousarray(np.broadcast_to(np.asarray(fields, dtype=np.float64), betas.shape))
    return betas, fields


def mirror_single_field(Lx, Ly, j, seed, betas, fields, planes=6, rounds=7, state=None):
    """The field strip as the device runs it, one (beta, h) per sweep, from the Philox initial state or
    from `state`.  -> (state bool[Ly, Lx], satisfied bonds int64[nsweeps], up spins int64[nsweeps])"""
    betas, fields = schedule(betas, fields)
    st = np.zeros((Ly, Lx), dtype=np.uint8) if state is None else np.ascontiguousarray(state, dtype=np.uint8).copy()
    nsat = np.zeros(len(betas), dtype=np.int64)
    up = np.zeros(len(betas), dtype=np.int64)
    rc = _lib().msc_mirror_single_field(Lx, Ly, float(j), int(seed), planes, rounds, int(state is None), _p(betas),
                                        _p(fields), len(betas), _p(st), _p(nsat), _p(up))
    assert rc == 0, rc
    return st.astype(bool), nsat, up


def mirror_band_field(Lx, y0, nrows, j, seed, betas, fields, planes=6, rounds=7):
    """Rows y0 .. y0 + nrows - 1 of a large lattice in the field schedule; after n sweeps the rows
    [2 n, nrows - 2 n) equal the full lattice's."""
    betas, fields = schedule(betas, fields)
    st = np.zeros((nrows, Lx), dtype=np.uint8)
    rc = _lib().msc_mirror_single_band_field(Lx, y0, nrows, float(j), int(seed), planes, rounds, 1, _p(betas),
                                             _p(fields), len(betas), _p(st))
    assert rc == 0, rc
    return st.astype(bool)


def strip_energy(j, h, nsites, nsat, up):
    """E = |J| (2 N - 2 n_sat) - h M, M = 2 up - N: SingleLattice2D.energy() from the counts"""
    if h == 0.0:
        return abs(j) * (2 * nsites - 2 * nsat)
    return abs(j) * (2 * nsites - 2 * nsat) - h * (2 * up - nsites)
