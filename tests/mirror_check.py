"""Helpers of the device-against-mirror tests (test_gpu_row_walk.py, test_gpu_general_graph.py): the
kernels a call launched, as torch.profiler records them, and where a device run first left the
scalar mirror (oracle/msc_mirror.c)."""
import re

import numpy as np


def pow2_ceil(v):
    r = 1
    while r < v:
        r *= 2
    return r


def random_regular(n, d, rng):
    """random d-regular graph (pairing model, self loops and multi-edges rejected) -> (a, b)"""
    while True:
        stubs = np.repeat(np.arange(n, dtype=np.int64), d)
        rng.shuffle(stubs)
        a, b = stubs[0::2], stubs[1::2]
        if (a == b).any():
            continue
        key = np.minimum(a, b) * n + np.maximum(a, b)
        if len(np.unique(key)) != len(key):
            continue
        return a, b


# ---------------------------------------------------------------------------------------------
# kernel names from the profiler
# ---------------------------------------------------------------------------------------------
def _targs(text):
    out = []
    for t in text.split(","):
        t = re.sub(r"^\(\w+\)", "", t.strip())
        out.append(t == "true" if t in ("true", "false") else int(t.rstrip("uU")))
    return tuple(out)


def launched(fn):
    """(fn(), names of the CUDA kernels the process launched meanwhile)"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, sorted({e.name for e in prof.events()})


def instances(names, kernel):
    """template arguments of every instantiation of `kernel` among the names"""
    pat = re.compile(r"\b" + kernel + r"<([^<>]*)>")
    return {_targs(m.group(1)) for n in names for m in [pat.search(n)] if m}


def families(names):
    fam = set()
    for n in names:
        m = re.search(r"(k_sweep_\w+|k_nsat_\w+)", n)
        if m:
            fam.add(m.group(1))
    return fam


def device_sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------
# comparison with the mirror
# ---------------------------------------------------------------------------------------------
def first_diff(st_gpu, st_ref, en_gpu, en_ref, offset=0):
    """where the device left the mirror first: replica word, replica, sweep / site"""
    msg = []
    if en_gpu is not None:
        bad = np.argwhere(en_gpu != en_ref)
        if len(bad):
            e, t = bad[np.lexsort((bad[:, 0], bad[:, 1]))[0]]
            msg.append(f"{len(bad)} energies differ; first at sweep {t}, replica {offset + e} "
                       f"(global word {(offset + e) // 32}): {en_gpu[e, t]} vs {en_ref[e, t]}")
    bad = np.argwhere(st_gpu != st_ref)
    if len(bad):
        e, n = bad[0]
        msg.append(f"{len(bad)} spins differ; first at replica {offset + e} (global word "
                   f"{(offset + e) // 32}), site {n}")
    return "; ".join(msg)


def assert_same(st_gpu, st_ref, en_gpu, en_ref, label, offset=0):
    ok = (st_gpu == st_ref).all() and (en_gpu is None or (en_gpu == en_ref).all())
    assert ok, f"{label}: {first_diff(st_gpu, st_ref, en_gpu, en_ref, offset)}"


def check_words(oracle, graph, E, seed, betas, words, en_gpu, word_states, label, offset=0, edges=None,
                per_replica_beta=None, **mirror_kw):
    """Replica words `words` of a run of E experiments at replica_offset `offset`: states and
    per-sweep energies equal msc_mirror run on those words alone (the ragged last word with its
    true tail, since the mirror ranks ties over real replicas only).  word_states(w) ->
    bool[32 or tail, nvars].  per_replica_beta: the run's E betas (betas is then the sweep count)."""
    a, b, j = graph.edges() if edges is None else edges
    colors = graph.colors()
    for w in words:
        k = min(32, E - 32 * w)
        if per_replica_beta is not None:
            mirror_kw.update(per_replica_beta=per_replica_beta[32 * w:32 * w + k], nsweeps=betas)
        en_ref, st_ref = oracle.msc_mirror(a, b, j, graph.nvars, colors, k, seed,
                                           None if per_replica_beta is not None else betas,
                                           replica_offset=offset + 32 * w, per_sweep=True, **mirror_kw)
        assert_same(word_states(w), st_ref, en_gpu[32 * w:32 * w + k], en_ref,
                    f"{label} word {w}", offset + 32 * w)


def word_bits(packed, w, k=32):
    """bool[k, nvars]: replicas 32 w .. 32 w + k - 1 of a packed state uint32[nvars, W]"""
    col = packed[:, w]
    return ((col[None, :] >> np.arange(k, dtype=np.uint32)[:, None]) & 1).astype(bool)
