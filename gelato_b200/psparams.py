"""Flipped Legendre-Gauss-Radau mesh parameters (host side, computed once).

Mirror of the reference's transcription helper
(/root/reference/lib/SectionParameters.py:30-103 `PSparams`,
/root/reference/lib/PSfunctions.py:149-208 `nodes_LGR` /
`differentiation_matrix_LGR`): same public methods and the same values, bit for
bit -- the differentiation matrix is evaluated with the reference's Lagrange
product/sum operation order (PSfunctions.py:64-88) but vectorised over all
(row, column) entries, so an n = 50 section costs milliseconds instead of the
reference's O(n^4) Python loops.
"""
import numpy as np
from scipy import special


def lgr_nodes(n):
    """n flipped LGR collocation points in (-1, 1], last one = +1."""
    roots, _ = special.j_roots(n - 1, 0, 1)
    return np.sort(-np.hstack((-1.0, roots)))


def lgr_diff_matrix(n, tau=None):
    """D[n, n+1]: derivative at the n LGR points of the Lagrange basis over
    the n+1 support points {-1} U tau.  Same operation order as the reference's
    nested loops, hence identical bits."""
    if tau is None:
        tau = lgr_nodes(n)
    tn = np.hstack((-1.0, tau))  # support points
    npts = n + 1
    t_eval = tn[1:]  # rows
    # den[i] = prod_{m != i} (tn[i] - tn[m]), sequential in m
    den = np.ones(npts)
    for m in range(npts):
        upd = den * (tn - tn[m])
        den = np.where(np.arange(npts) != m, upd, den)
    # num[k, i] = sum_{j != i} prod_{m != i, m != j} (t_k - tn[m])
    T = t_eval[:, None] * np.ones((1, npts))  # t per row, broadcast over columns i
    col = np.arange(npts)[None, :]
    num = np.zeros((n, npts))
    for j in range(npts):
        num_j = np.ones((n, npts))
        for m in range(npts):
            if m == j:
                continue
            upd = num_j * (T - tn[m])
            num_j = np.where(col != m, upd, num_j)
        num = np.where(col != j, num + num_j, num)
    return num / den[None, :]


_MESH = {}  # n -> (tau, D), read-only: a study of many scenarios builds the same meshes again and again


def mesh_tables(n):
    """(tau[n], D[n, n+1]) of an n-node section, computed once per process (read-only arrays)."""
    if n not in _MESH:
        tau = lgr_nodes(n)
        D = lgr_diff_matrix(n, tau)
        tau.setflags(write=False)
        D.setflags(write=False)
        _MESH[n] = (tau, D)
    return _MESH[n]


def lgr_points(n):
    """lgr_nodes(n), with n = 1 allowed: the one flipped LGR point is +1."""
    return lgr_nodes(n) if n > 1 else np.ones(1)


def interval_points(pts, a, b):
    """Points in [-1, 1] (the last one +1) mapped affinely onto [a, b], the last one exactly b."""
    out = a + (np.asarray(pts, dtype=np.float64) + 1.0) * ((b - a) / 2.0)
    out[-1] = b
    return out


def check_intervals(n, counts, breaks=None):
    """(counts, breaks) of a section of n nodes made of K = len(counts) LGR intervals, validated: every count >= 1 and
    their sum n, breaks the K - 1 interior breakpoints, strictly increasing inside (-1, 1) (None: equal widths).
    ValueError otherwise."""
    counts = [int(c) for c in counts]
    K = len(counts)
    if K < 1 or min(counts) < 1 or sum(counts) != n:
        raise ValueError("interval node counts must be >= 1 and add up to the section's %d nodes, got %r" % (n, counts))
    if breaks is None:
        breaks = [-1.0 + 2.0 * k / K for k in range(1, K)]
    breaks = np.array(breaks, dtype=np.float64).reshape(-1)
    b = np.hstack((-1.0, breaks, 1.0))
    if breaks.size != K - 1 or not np.all(np.isfinite(breaks)) or not np.all(b[1:] > b[:-1]):
        raise ValueError("%d intervals need %d interior breakpoints, strictly increasing inside (-1, 1), got %r"
                         % (K, K - 1, breaks.tolist()))
    return counts, breaks


def composite_tables(counts, breaks):
    """(tau[n], D[n, n+1]) of a section made of LGR intervals (check_intervals): interval k over [b_k, b_k+1] has its
    n_k flipped LGR points mapped into it (its last one exactly b_k+1), and its rows of D are lgr_diff_matrix(n_k) * 2 /
    w_k in its support columns c_k .. c_k + n_k (c_k = n_0 + .. + n_k-1), every other entry exactly 0."""
    n = sum(counts)
    b = np.hstack((-1.0, breaks, 1.0))
    tau, D = np.empty(n), np.zeros((n, n + 1))
    c = 0
    for k, nk in enumerate(counts):
        pts = lgr_points(nk)
        tau[c:c + nk] = interval_points(pts, b[k], b[k + 1])
        D[c:c + nk, c:c + nk + 1] = lgr_diff_matrix(nk, pts) * (2.0 / (b[k + 1] - b[k]))
        c += nk
    return tau, D


class PSparams:
    """Per-section node counts, LGR points, differentiation matrices and the
    index arithmetic of the decision vector (reference: SectionParameters.py).

    intervals[i] (optional): None, one LGR interval as the reference has it, or (counts, breaks) of a composite section
    of several LGR intervals (check_intervals, composite_tables; DESIGN.md section 11).  Every user of tau and D reads a
    composite section as it reads any other: only values change, never the layout."""

    def __init__(self, num_nodes, intervals=None):
        self._num_nodes = [int(n) for n in num_nodes]
        self._num_sections = len(self._num_nodes)
        if intervals is None:
            intervals = [None] * self._num_sections
        if len(intervals) != self._num_sections:
            raise ValueError("one interval entry per section is needed")
        self._tau, self._D, self._int = [], [], []
        for n, iv in zip(self._num_nodes, intervals):
            if iv is not None:
                counts, breaks = check_intervals(n, *iv)
                iv = None if len(counts) == 1 else (counts, breaks)
            if iv is None:
                tau, D = mesh_tables(n)
                self._int.append(([n], np.empty(0), [0]))
            else:
                tau, D = composite_tables(*iv)
                tau.setflags(write=False)
                D.setflags(write=False)
                self._int.append((iv[0], iv[1], [int(v) for v in np.concatenate(([0], np.cumsum(iv[0])[:-1]))]))
            self._tau.append(tau)
            self._D.append(D)
        self._index_start_u = [int(v) for v in np.concatenate(([0], np.cumsum(self._num_nodes)[:-1]))]
        self._N = int(sum(self._num_nodes))

    def _check(self, i):
        if i < 0 or i >= self._num_sections:
            raise ValueError("Index out of range")

    def tau(self, i):
        self._check(i)
        return self._tau[i]

    def D(self, i):
        self._check(i)
        return self._D[i]

    def nodes(self, i):
        self._check(i)
        return self._num_nodes[i]

    def intervals(self, i):
        """(counts, breaks, support columns) of section i: the node count of each LGR interval, the interior
        breakpoints in section tau and the first support column c_k of each; ([n], [], [0]) for one interval."""
        self._check(i)
        return self._int[i]

    def index_start_u(self, i):
        return self._index_start_u[i]

    def index_end_u(self, i):
        return self._index_start_u[i] + self._num_nodes[i]

    def index_start_x(self, i):
        return self._index_start_u[i] + i

    def index_end_x(self, i):
        return self.index_start_x(i) + self._num_nodes[i] + 1

    def num_u(self):
        return self._N

    def num_x(self):
        return self._N + self._num_sections

    def num_sections(self):
        return self._num_sections

    def time_nodes(self, i, to, tf):
        t = np.zeros(self._num_nodes[i] + 1)
        t[0] = to
        t[1:] = self.tau(i) * (tf - to) / 2 + (tf + to) / 2
        return t

    def get_index(self, section):
        """(ua, ub, xa, xb, n) of a section: control rows ua..ub-1, state rows xa..xb-1."""
        ua = self._index_start_u[section]
        n = self._num_nodes[section]
        return ua, ua + n, ua + section, ua + section + n + 1, n

    def __getitem__(self, i):
        self._check(i)
        return {"index_start": self._index_start_u[i], "nodes": self._num_nodes[i], "D": self._D[i], "tau": self._tau[i]}
