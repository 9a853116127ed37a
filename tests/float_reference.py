"""TEST INFRASTRUCTURE: an f64 restatement of the float-field path, decision by decision.

Graphs outside the integer classes (real couplings, a bias, degree > 15; DESIGN.md D4) run on
k_sweep_real, k_edge_moves and k_worm_moves: an f32 local field per replica bit, the fast
exponential, and one 32-bit Philox word u per decision, accepted iff u < p 2^32.  They cannot
be bit-exact against f64, but u is exact, so f64 knows every decision except those where u
falls in a narrow band around p 2^32.  This module draws the same words (csrc/philox.h) and
takes the same decisions in f64; `decide` bounds what the kernel's f32 arithmetic can make of
p, and a decision whose u lies inside those bounds is "in band".  Replicas are independent (own
field, own uniform, own beta), so a replica that meets an in-band decision is dropped from the
comparison from then on (`Chain.determined`) and every other replica must equal the kernel bit
for bit.

What the kernels compute (csrc/sweep_general.cu, csrc/moves.cu):
  sweep      per colour class (ascending): dE = 2 s_i (b_i - sum_k J_ik s_k), accept iff
             dE <= 0 or u < exp(-beta dE) 2^32; Philox counter (site, replica word, t, call),
             call = (replica bit) / 4, u = word (replica bit) % 4.
  edge move  per pass, per class of the strong edge colouring (ascending): both spins of bond
             (a, b) flip, dE over the bonds that join a or b to the rest of the graph plus both
             bias terms; p = wrel min(1, exp(-beta dE)), wrel = |J| / max |J| with importance
             sampling, else 1; counter (edge id, replica word, t, call | pass << 8 | TAG_EDGE << 24).
  worm       per worm k: counter (replica, k, t, call | TAG_WORM << 24), word m = component m % 4
             of call m / 4; start = umul64hi(w0 << 32 | w1, nvars), u = w2, step t goes to
             nbr[row[head] + umulhi(w(2 + t), deg(head))]; a chain that bites itself (or meets a
             site without bonds) is abandoned; p = min(1, deg(first) / deg(last) exp(-beta dE)).

The error bounds of `decide`: the f32 field sums `terms` products of f32 couplings (exact: the
couplings are f32, the spins +-1) and the bias.  For the moves |dE_f32 - dE| <= 2 (terms + 2)
2^-23 (sum|J| + |b|) (recursive summation, one more rounding for b - h, generous by 2x); the sweep
takes the tighter 2^-24 per addition times the running sum it forms (`sweep_delta`), which keeps
dense graphs (SK, degree 255) determined at beta = 1e6; where every coupling and bias is a multiple
of a power of two q and every sum stays below 2^24 q (+-J, integer fields) the f32 sums are exact
and the bound is 0.  __expf(x) has at most
2 + floor(1.173 |x|) ulp of error (CUDA C++ Programming Guide, intrinsic functions); the f32
rounding of beta, of -beta dE and of the products with wrel or the degree ratio add at most
|x| + 2 ulp more, so the kernel's p is within (4 + 2|x|) 2^-23 of exp(-beta dE_f32) in relative
terms.  On the host the emulation takes glibc's expf (< 1 ulp), which the same bound covers.
Plain numpy and scipy; nothing here imports the library.
"""
import math

import numpy as np
import scipy.sparse as sp

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
TAG_ACCEPT, TAG_EDGE, TAG_WORM = 0, 4, 5
U32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def philox(c0, c1, c2, c3, k0, k1, rounds):
    """Philox4x32-R of csrc/philox.h, vectorised over broadcast counters -> 4 uint64 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & U32 for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    for _ in range(rounds):
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        c = [(p1 >> _S32) ^ c[1] ^ k0, p1 & U32, (p0 >> _S32) ^ c[3] ^ k1, p0 & U32]
        k0 = (k0 + np.uint64(W0)) & U32
        k1 = (k1 + np.uint64(W1)) & U32
    return c


def keys(seed):
    seed = int(seed) & (2**64 - 1)
    return seed & 0xFFFFFFFF, seed >> 32


def _word(r, j):
    """component j (array, 0..3) of Philox outputs r"""
    return np.choose(np.asarray(j, dtype=np.int64), r)


def _f32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def decide(u, de, delta, beta, factor=1.0, kind="sweep"):
    """(accept, in_band) of decisions with Philox words u (uint64), f64 energy changes de, bounds
    delta on the kernel's f32 error of de, inverse temperatures beta and proposal factors (wrel,
    degree ratio).  accept is the exact rule u < p 2^32, p = min(1, factor g(de)) with
    g = exp(-beta max(dE, 0)) for kind "sweep" and "edge", exp(-beta dE) for "worm".  in_band: the
    kernel's f32 dE and __expf could decide either way.  The kernels' own rules:
      sweep  dE <= 0 accepts, else u < trunc(exp 2^32) saturated at 2^32 - 1 (u = 2^32 - 1 rejects)
      edge   p = (dE > 0 ? exp : 1) wrel; p >= 1 accepts, else u < trunc(p 2^32)
      worm   p = ratio exp; p >= 1 accepts, else u < trunc(p 2^32)"""
    de, delta = np.asarray(de, dtype=np.float64), np.asarray(delta, dtype=np.float64)
    beta = np.asarray(beta, dtype=np.float64)
    factor = np.asarray(factor, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64)                         # exact: u < 2^32
    arg = (lambda x: x) if kind == "worm" else (lambda x: np.maximum(x, 0.0))
    with np.errstate(over="ignore", invalid="ignore"):
        p = np.minimum(1.0, factor * np.exp(-beta * arg(de)))
        # the kernel's dE lies in [de - delta, de + delta], its p within a relative eps of factor g
        x = beta * (np.abs(de) + delta) if kind == "worm" else beta * np.maximum(de + delta, 0.0)
        eps = np.minimum((4.0 + 2.0 * x) * 2.0**-23, 0.5)          # x: the largest argument of __expf
        p_hi = np.minimum(1.0, factor * np.exp(-beta * arg(de - delta)) * (1 + eps))
        p_lo = np.minimum(1.0, factor * np.exp(-beta * arg(de + delta)) * (1 - eps))
    accept = u < p * 2.0**32
    downhill = de + delta <= 0                                  # the kernel's dE <= 0 as well
    if kind == "sweep":
        sure_accept = downhill | (u + 1.0 <= np.minimum(p_lo * 2.0**32, 2.0**32 - 1))
    else:
        sure_accept = (p_lo >= 1.0) | (u + 1.0 <= p_lo * 2.0**32)
        if kind == "edge":
            sure_accept |= downhill & (factor == 1.0)           # p = 1 exactly, no exponential
    sure_reject = (p_hi < 1.0) & (u >= p_hi * 2.0**32)          # u >= p_hi 2^32 >= trunc(p_k 2^32)
    return accept, ~(sure_accept | sure_reject)


def field_delta(terms, abs_sum, exact=False):
    """bound on the f32 error of a dE summed from `terms` couplings over a magnitude abs_sum"""
    d = 2.0 * (np.asarray(terms, dtype=np.float64) + 2.0) * 2.0**-23 * np.asarray(abs_sum, dtype=np.float64)
    return d * 0.0 if exact else d


def sweep_delta(g, s, sites, h):
    """[E, |C|] bound on |dE_f32 - dE| of the sweep from the partial sums the kernel forms: adding
    term k in f32 errs by at most 2^-24 |partial sum k|, b - h by 2^-24 |b - h|, dE = 2 s (b - h)
    doubles it; the second-order terms are bounded by n^2 2^-48 sum|J| (a 1 % margin on top)"""
    u = 2.0**-24
    lo, hi = g.row[sites], g.row[sites + 1]
    n = hi - lo
    idx = np.concatenate([np.arange(l, h_) for l, h_ in zip(lo, hi)]) if n.sum() else np.zeros(0, np.int64)
    if len(idx) == 0:
        return np.zeros((s.shape[0], len(sites)))
    c = s[:, g.nbr[idx]] * g.jcsr[idx]
    cs = np.cumsum(c, axis=1)
    starts = np.concatenate([[0], np.cumsum(n)[:-1]])
    base = np.where(starts > 0, cs[:, np.maximum(starts - 1, 0)], 0.0)
    seg = np.repeat(np.arange(len(sites)), n)
    partial = np.abs(cs - base[:, seg])
    tot = np.zeros((s.shape[0], len(sites)))
    nz = n > 0
    tot[:, nz] = np.add.reduceat(partial, starts[nz], axis=1)
    e_h = u * tot + (n ** 2) * u * u * 4 * g.abs_j[sites]
    e = e_h + u * (np.abs(g.bq[sites] - h) + e_h)
    return 2.0 * 1.01 * e


class Graph:
    """The graph as the float kernels see it: couplings and biases rounded to f32 (jf / biasf),
    CSR with neighbours ascending and ties in edge-list order (csrc/graph.cpp: build_csr), the
    colour classes of the sweeps and the classes of the strong edge colouring (edge id = index in
    the edge list)."""

    def __init__(self, nvars, a, b, j, bias=None, colors=None, edge_classes=None):
        self.n = int(nvars)
        self.a = np.asarray(a, dtype=np.int64)
        self.b = np.asarray(b, dtype=np.int64)
        self.j = np.asarray(j, dtype=np.float64)                # f64: what the energies use
        self.bias = np.zeros(self.n) if bias is None else np.asarray(bias, dtype=np.float64)
        self.jq, self.bq = _f32(self.j), _f32(self.bias)        # f32-rounded: what the sweeps use
        n, m = self.n, len(self.a)
        src = np.concatenate([self.a, self.b])
        dst = np.concatenate([self.b, self.a])
        order = np.lexsort((np.concatenate([np.arange(m)] * 2), dst, src))
        self.row = np.zeros(n + 1, dtype=np.int64)
        np.add.at(self.row, src + 1, 1)
        self.row = np.cumsum(self.row)
        self.nbr = dst[order]
        self.jcsr = np.concatenate([self.jq, self.jq])[order]
        self.deg = np.diff(self.row)
        self.abs_j = np.zeros(n)
        np.add.at(self.abs_j, src, np.abs(np.concatenate([self.jq, self.jq])))
        # J[i, k] = sum of the f32 couplings of the bonds between i and k (multi-edges add up)
        self.J = sp.csr_matrix((np.concatenate([self.jq, self.jq]), (src, dst)), shape=(n, n))
        self.J.sum_duplicates()
        self.Jabs = sp.csr_matrix((np.abs(np.concatenate([self.jq, self.jq])), (src, dst)), shape=(n, n))
        self.Jabs.sum_duplicates()
        self.mult = sp.csr_matrix((np.ones(2 * m), (src, dst)), shape=(n, n))
        self.mult.sum_duplicates()
        # every coupling and bias a multiple of q = 2^e and every sum a move forms below 2^24 q (e.g.
        # +-J): the f32 fields are exact and the bounds on their error vanish
        vals = np.concatenate([self.jq, self.bq])
        vals = vals[vals != 0]
        mant, ex = np.frexp(vals)
        m24 = np.abs(mant * 2.0**24).astype(np.int64)
        low = (m24 & -m24).astype(np.float64)                        # lowest set bit of the 24-bit mantissa
        q = float((low * np.ldexp(1.0, ex - 24)).min()) if len(vals) else 1.0
        self.exact = bool(16 * (self.abs_j + np.abs(self.bq)).max() <= 2.0**24 * q)
        self.colors = None if colors is None else np.asarray(colors, dtype=np.int64)
        self.classes = None
        if colors is not None:
            self.classes = [np.nonzero(self.colors == c)[0] for c in range(int(self.colors.max()) + 1)]
        self.edge_cls = None
        if edge_classes is not None:
            ec = np.asarray(edge_classes, dtype=np.int64)
            self.edge_cls = [np.nonzero(ec == c)[0] for c in range(int(ec.max()) + 1)]
            wj = np.abs(self.j).astype(np.float32).astype(np.float64)
            jmax = np.abs(self.j).max()
            self.wrel = (wj / jmax).astype(np.float32).astype(np.float64) if jmax > 0 else np.ones(m)

    @classmethod
    def from_native(cls, g, bias=None):
        """through the library's Graph.edges(), colors(), edge_classes() (a ctypes object)"""
        a, b, j = g.edges()
        return cls(g.nvars, a, b, j, bias, g.colors(), g.edge_classes())

    def pair(self, x, y, M):
        return np.asarray(M[x, y]).ravel()

    def energies(self, states):
        """exact f64 energies sum_edges J s_a s_b - sum_i b_i s_i (math.fsum) of bool[E, n]"""
        s = np.asarray(states, dtype=np.float64) * 2 - 1
        terms = np.concatenate([s[:, self.a] * s[:, self.b] * self.j, -s * self.bias], axis=1)
        return np.array([math.fsum(r) for r in terms])

    def energy_bound(self):
        """bound on |k_energy_real - exact|: 2 nedges + nvars f64 additions over sum|J| + sum|b|"""
        return (2 * len(self.a) + self.n) * 2.0**-52 * (np.abs(self.j).sum() + np.abs(self.bias).sum())


class Chain:
    """E replicas of the float path: states bool[E, n], global replica index rep[e] (Philox replica
    word rep // 32, bit rep % 32; the worms' experiment index), a `determined` mask and counts."""

    def __init__(self, graph, states, seed, rep0=0, rounds=7, rep=None):
        self.g = graph
        self.s = np.array(states, dtype=bool)
        self.E = self.s.shape[0]
        self.rep = (rep0 + np.arange(self.E)).astype(np.uint64) if rep is None else np.asarray(rep, dtype=np.uint64)
        self.k0, self.k1 = keys(seed)
        self.rounds = rounds
        self.determined = np.ones(self.E, dtype=bool)
        self.in_band = 0
        self.decisions = 0

    def _take(self, accept, band, live=None):
        """accept / band [E, k]: count, drop replicas with an in-band decision"""
        if live is None:
            live = np.ones(accept.shape, dtype=bool)
        band = band & live
        self.in_band += int(band.sum())
        self.decisions += int(live.sum())
        self.determined &= ~band.any(axis=1)
        return accept & live

    def _beta(self, beta):
        return np.broadcast_to(np.asarray(beta, dtype=np.float64), (self.E,))[:, None]

    def sweep(self, t, beta):
        """one colour-class sweep at timestep t; beta scalar or per replica [E]"""
        g, beta = self.g, self._beta(beta)
        word, bit = self.rep >> np.uint64(5), self.rep & np.uint64(31)
        for sites in g.classes:
            s = self.s.astype(np.float64) * 2 - 1
            h = np.asarray((g.J[:, sites].T @ s.T).T)            # [E, |C|]
            si = s[:, sites]
            de = 2 * si * (g.bq[sites] - h)
            r = philox(sites[None, :], word[:, None], t, (bit >> np.uint64(2))[:, None] | (TAG_ACCEPT << 24),
                       self.k0, self.k1, self.rounds)
            u = _word(r, (bit & np.uint64(3))[:, None].astype(np.int64))
            delta = np.zeros(de.shape) if g.exact else sweep_delta(g, s, sites, h)
            acc, band = decide(u, de, delta, beta)
            acc = self._take(acc, band)
            self.s[:, sites] ^= acc

    def edge_pass(self, t, beta, p, importance=False):
        g, beta = self.g, self._beta(beta)
        word, bit = self.rep >> np.uint64(5), self.rep & np.uint64(31)
        for ids in g.edge_cls:
            s = self.s.astype(np.float64) * 2 - 1
            ea, eb = g.a[ids], g.b[ids]
            jab, mab = g.pair(ea, eb, g.J), g.pair(ea, eb, g.mult)
            F = np.asarray((g.J[:, np.concatenate([ea, eb])].T @ s.T).T)
            ha = F[:, :len(ids)] - s[:, eb] * jab                # bonds between a and b keep their energy
            hb = F[:, len(ids):] - s[:, ea] * jab
            de = 2 * s[:, ea] * (g.bq[ea] - ha) + 2 * s[:, eb] * (g.bq[eb] - hb)
            r = philox(ids[None, :], word[:, None], t,
                       (bit >> np.uint64(2))[:, None] | np.uint64(p << 8) | np.uint64(TAG_EDGE << 24),
                       self.k0, self.k1, self.rounds)
            u = _word(r, (bit & np.uint64(3))[:, None].astype(np.int64))
            jab_abs = g.pair(ea, eb, g.Jabs)
            terms = g.deg[ea] + g.deg[eb] - 2 * mab
            mag = g.abs_j[ea] + g.abs_j[eb] - 2 * jab_abs + np.abs(g.bq[ea]) + np.abs(g.bq[eb])
            acc, band = decide(u, de, field_delta(terms, mag, g.exact)[None, :], beta,
                               g.wrel[ids][None, :] if importance else 1.0, kind="edge")
            acc = self._take(acc, band)
            self.s[:, ea] ^= acc
            self.s[:, eb] ^= acc

    def worms(self, t, beta, nworms, length):
        g, beta = self.g, self._beta(beta)[:, 0]
        E, n = self.E, g.n
        idx = np.arange(E)
        for k in range(nworms):
            calls = {}

            def w(m):
                c = m >> 2
                if c not in calls:
                    calls[c] = philox(self.rep, k, t, c | (TAG_WORM << 24), self.k0, self.k1, self.rounds)
                return calls[c][m & 3]

            hi, lo = w(0), w(1)
            path = np.zeros((E, length), dtype=np.int64)
            path[:, 0] = ((hi * np.uint64(n) + ((lo * np.uint64(n)) >> _S32)) >> _S32).astype(np.int64)
            u = w(2)
            ok = np.ones(E, dtype=bool)
            for st in range(1, length):
                head = path[:, st - 1]
                d = g.deg[head]
                ok &= d > 0
                pick = ((w(2 + st) * d.astype(np.uint64)) >> _S32).astype(np.int64)
                nxt = g.nbr[np.minimum(g.row[head] + pick, len(g.nbr) - 1)]
                ok &= ~(path[:, :st] == nxt[:, None]).any(axis=1)
                path[:, st] = nxt
            s = self.s.astype(np.float64) * 2 - 1
            F = np.asarray(g.J.T @ s.T).T                            # fields [E, n] (J symmetric)
            sp_ = s[idx[:, None], path]                              # [E, L]
            de = np.zeros(E)
            for a_ in range(length):
                h = F[idx, path[:, a_]]
                for b_ in range(length):
                    if b_ != a_:
                        h = h - g.pair(path[:, a_], path[:, b_], g.J) * sp_[:, b_]
                de += 2 * sp_[:, a_] * (g.bq[path[:, a_]] - h)
            terms = g.deg[path].sum(axis=1) + length
            mag = (g.abs_j[path] + np.abs(g.bq[path])).sum(axis=1)
            dl = g.deg[path[:, -1]]
            ratio = g.deg[path[:, 0]] / np.maximum(dl, 1) if length > 1 else np.ones(E)
            acc, band = decide(u, de, field_delta(terms, mag, g.exact), beta, ratio, kind="worm")
            acc = self._take(acc[:, None], band[:, None], ok[:, None])[:, 0]
            rows = np.nonzero(acc)[0]
            for a_ in range(length):
                self.s[rows, path[rows, a_]] ^= True

    def timestep(self, t, beta, spin_sweeps=1, edge_passes=0, worms=0, worm_len=4, importance=False):
        """one timestep as csrc/api_sim.cu enqueues it (sim_one_sweep / sim_non_basic_moves)"""
        if spin_sweeps:
            self.sweep(t, beta)
        for p in range(edge_passes):
            self.edge_pass(t, beta, p, importance)
        if worms:
            self.worms(t, beta, worms, worm_len)
