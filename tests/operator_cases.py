"""Seeded synthetic operators for the sparse and mesh-layer kernels, and a float64 reference of what those kernels compute.

The template mesh's operators (tests/golden/operators_template5k.npz) have properties the kernels could silently depend
on: a symmetric L_hat (so CSR(L) and CSR(L^T) are the same arrays), degrees <= ~9, five fixed vertex counts, empty rows
only as a suffix, no duplicates / self loops / hubs, D matrices that select distinct vertices and U matrices with 3
entries per row.  The families below break each of these.

An operator case is an `Op`: the (edge_index, norm) pair that ChebConv_batch.norm hands to the layers
(out[t] += norm[e] * x[edge_index[0][e]] for edge_index[1][e] == t) or a torch sparse COO matrix for pooling, plus the
same matrix as a float64 scipy CSR built from the fp32 values the device receives.  No product imports: the tests pass
these through the real operators.from_edges / from_sparse.

The reference (cheb_ref_fwd / cheb_ref_bwd / pool_ref) works on vertex-major float64 arrays [N, B, F]; its backward is
the adjoint form (S_k = T_k(L^T) G), so it never materialises per-edge gathers."""
from dataclasses import dataclass
from typing import Optional

import numpy as np
import scipy.sparse as sp
import torch

from tests.helpers import OPERATORS_NPZ


@dataclass
class Op:
    name: str
    n_rows: int
    n_cols: int
    rows: np.ndarray            # int64, COO order as handed to the product (duplicates kept)
    cols: np.ndarray
    vals: np.ndarray            # float32

    @property
    def csr(self) -> sp.csr_matrix:
        """float64 CSR of the fp32 operator (duplicates summed in float64)"""
        return sp.csr_matrix((self.vals.astype(np.float64), (self.rows, self.cols)), shape=(self.n_rows, self.n_cols))

    @property
    def nnz(self) -> int:
        return int(self.rows.shape[0])

    def edges(self):
        """(edge_index [2, E] int64, norm [E] fp32) of L_hat: source = column, target = row"""
        ei = torch.from_numpy(np.vstack((self.cols, self.rows)).astype(np.int64))
        return ei, torch.from_numpy(self.vals.astype(np.float32))

    def sparse(self) -> torch.Tensor:
        """uncoalesced torch sparse COO [n_rows, n_cols], as the reference's model.py hands its D / U matrices over"""
        idx = torch.from_numpy(np.vstack((self.rows, self.cols)).astype(np.int64))
        return torch.sparse_coo_tensor(idx, torch.from_numpy(self.vals.astype(np.float32)), (self.n_rows, self.n_cols),
                                       check_invariants=False)


def _op(name, n_rows, n_cols, rows, cols, vals) -> Op:
    return Op(name, int(n_rows), int(n_cols), np.asarray(rows, np.int64), np.asarray(cols, np.int64),
              np.asarray(vals, np.float32))


def _cheb_norm_np(src, dst, n, w=None):
    """oracle.cheb_norm restated on numpy: self loops dropped, norm_e = -deg^-1/2[src] * w_e * deg^-1/2[dst] with the
    degree summed over the source index (nn/conv.py:541-555); inf -> 0"""
    keep = src != dst
    src, dst = src[keep], dst[keep]
    w = np.ones(src.shape[0], np.float32) if w is None else np.asarray(w, np.float32)[keep]
    deg = np.zeros(n, np.float32)
    np.add.at(deg, src, w)
    with np.errstate(divide="ignore"):
        dis = np.where(deg > 0, deg.astype(np.float32) ** np.float32(-0.5), np.float32(0))
    return src, dst, (-dis[src] * w * dis[dst]).astype(np.float32)


# ---------------------------------------------------------------------------------------------
# families
# ---------------------------------------------------------------------------------------------
def template_adjacency(lvl: int):
    """(src, dst, N) of the template's adjacency at a level (both directions of every edge)"""
    d = np.load(OPERATORS_NPZ)
    return d[f"A{lvl}_row"].astype(np.int64), d[f"A{lvl}_col"].astype(np.int64), int(d["num_nodes"][lvl])


def template_L(lvl: int) -> Op:
    src, dst, n = template_adjacency(lvl)
    s, t, v = _cheb_norm_np(src, dst, n)
    return _op(f"template{lvl}", n, n, t, s, v)


def relabelled(lvl: int, seed: int) -> Op:
    """the template's L_hat under a random vertex permutation: still symmetric, but every row's columns span the mesh"""
    src, dst, n = template_adjacency(lvl)
    p = np.random.default_rng(seed).permutation(n)
    s, t, v = _cheb_norm_np(p[src], p[dst], n)
    return _op(f"relabelled{lvl}", n, n, t, s, v)


def directed(lvl: int, seed: int, both: bool) -> Op:
    """template edges kept in one random direction each (both=False), or in both directions with independent weights
    (both=True), normalised as ChebConv_batch.norm does: L_hat is not symmetric"""
    src, dst, n = template_adjacency(lvl)
    rng = np.random.default_rng(seed)
    und = src < dst
    a, b = src[und], dst[und]
    if both:
        s, t = np.concatenate((a, b)), np.concatenate((b, a))
        w = rng.uniform(0.2, 2.0, s.shape[0]).astype(np.float32)
    else:
        flip = rng.random(a.shape[0]) < 0.5
        s, t = np.where(flip, b, a), np.where(flip, a, b)
        w = None
    s, t, v = _cheb_norm_np(s, t, n, w)
    return _op(f"directed{lvl}{'w' if both else '1'}", n, n, t, s, v)


def _scale_rows(rows, vals, n, rng, lo=0.5, hi=0.95):
    """each non-empty row scaled to an absolute row sum in [lo, hi]: ||L||_inf <= 0.95 keeps T_k bounded"""
    s = np.zeros(n)
    np.add.at(s, rows, np.abs(vals))
    target = rng.uniform(lo, hi, n)
    f = np.where(s > 0, target / np.where(s > 0, s, 1.0), 0.0)
    return (vals * f[rows]).astype(np.float32)


def irregular(n: int, seed: int, deg=(4, 8), hubs=0, hub_deg=(200, 1000), isolated=0, dups=0, loops=0,
              n_active: Optional[int] = None, hub_rows=None) -> Op:
    """a random square operator on n vertices: base degree in [deg[0], deg[1]] (columns without repetition),
    `hubs` rows of degree in hub_deg (at `hub_rows` if given), `isolated` vertices scattered through the middle with
    no entry in their row or column (empty rows that are not a suffix), `dups` duplicated (row, col) entries and `loops`
    self-loop entries; values of both signs, rows scaled to an absolute sum <= 0.95.  With n_active < n the graph lives
    on the first n_active vertices and the rest have no edges (the closed-form rows of mvb_cheb_*)."""
    rng = np.random.default_rng(seed)
    na = n if n_active is None else n_active
    iso = np.zeros(n, bool)
    iso[na:] = True
    if isolated:
        mid = np.arange(min(1, na - 1), max(na - 1, 1))
        iso[rng.choice(mid, size=min(isolated, mid.shape[0]), replace=False)] = True
    live = np.flatnonzero(~iso)
    rows, cols = [], []
    if hub_rows is None:
        hub_rows = rng.choice(live, size=min(hubs, live.shape[0]), replace=False) if hubs else np.zeros(0, np.int64)
    hub_set = set(int(h) for h in hub_rows)
    for r in live:
        if r in hub_set:
            d = int(rng.integers(hub_deg[0], hub_deg[1] + 1))
        else:
            d = int(rng.integers(deg[0], deg[1] + 1))
        d = min(d, live.shape[0])
        c = rng.choice(live, size=d, replace=False)
        rows.append(np.full(d, r))
        cols.append(c)
    rows = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    cols = np.concatenate(cols) if cols else np.zeros(0, np.int64)
    if dups and rows.shape[0]:
        j = rng.choice(rows.shape[0], size=dups)
        rows, cols = np.concatenate((rows, rows[j])), np.concatenate((cols, cols[j]))
    if loops and live.shape[0]:
        r = rng.choice(live, size=min(loops, live.shape[0]), replace=False)
        rows, cols = np.concatenate((rows, r)), np.concatenate((cols, r))
    perm = rng.permutation(rows.shape[0])                       # COO order as given: not sorted by row
    rows, cols = rows[perm], cols[perm]
    vals = rng.uniform(0.2, 1.0, rows.shape[0]) * rng.choice([-1.0, 1.0], rows.shape[0])
    vals = _scale_rows(rows, vals, n, rng)
    return _op(f"irregular{n}", n, n, rows, cols, vals)


def selection(n_in: int, n_out: int, seed: int, repeat: int = 0) -> Op:
    """D [n_out, n_in]: one 1.0 per row at distinct vertices in random (unsorted) order; `repeat` > 0 makes that many
    rows select a vertex another row already selects"""
    rng = np.random.default_rng(seed)
    cols = rng.choice(n_in, size=n_out, replace=False)
    if repeat:
        r = rng.choice(np.arange(1, n_out), size=repeat, replace=False)
        cols[r] = cols[rng.integers(0, r.min(), size=repeat)]
    rows = np.arange(n_out)
    perm = rng.permutation(n_out)
    return _op(f"sel{n_out}x{n_in}{'rep' if repeat else ''}", n_out, n_in, rows[perm], cols[perm], np.ones(n_out))


def weighted_down(n_in: int, n_out: int, seed: int) -> Op:
    """D [n_out, n_in] with 2 weighted entries per row (not a selection)"""
    rng = np.random.default_rng(seed)
    rows = np.repeat(np.arange(n_out), 2)
    cols = np.concatenate([rng.choice(n_in, size=2, replace=False) for _ in range(n_out)])
    vals = rng.uniform(0.1, 0.9, 2 * n_out)
    return _op(f"wdown{n_out}x{n_in}", n_out, n_in, rows, cols, vals)


def upsample(n_out: int, n_in: int, seed: int, max_per_row: int = 4) -> Op:
    """U [n_out, n_in] with 0..max_per_row entries per row (barycentric-like positive weights, some rows empty)"""
    rng = np.random.default_rng(seed)
    cnt = rng.integers(0, max_per_row + 1, n_out)
    rows = np.repeat(np.arange(n_out), cnt)
    cols = np.concatenate([rng.choice(n_in, size=c, replace=c > n_in) for c in cnt]) if cnt.sum() else np.zeros(0, np.int64)
    vals = rng.uniform(0.05, 1.0, rows.shape[0])
    perm = rng.permutation(rows.shape[0])
    return _op(f"up{n_out}x{n_in}", n_out, n_in, rows[perm], cols[perm], vals[perm])


def asymmetry(op: Op) -> float:
    """||L - L^T||_F / ||L||_F"""
    m = op.csr
    return float(sp.linalg.norm(m - m.T) / sp.linalg.norm(m))


# ---------------------------------------------------------------------------------------------
# shared-memory and plan arithmetic of the kernels, restated to place cases on either side of a boundary
# ---------------------------------------------------------------------------------------------
SMEM_CAP = 227 * 1024
ST_ECAP, ST_RCAP = 4096, 592


def _al(v, a):
    return (v + a - 1) // a * a


def mesh_tc_smem(n, n_in, nnz, k, width_in, width_acc, c):
    """(fits, has_second_lo_plane) of the tensor-core mesh kernels' shared-memory layout (csrc/mvb_mesh_tc.cu
    mesh_tc_layout) for a cluster of c CTAs per mesh"""
    wl = width_in // c
    tiles = (n + 127) // 128
    if width_in % c or wl not in (8, 16, 32) or width_acc not in (16, 32) or tiles * width_acc > 512:
        return False, False
    rb = wl * 4
    plane = _al(max(n_in, tiles * 128) * rb, 1024)
    if c == 2:
        plane = max(plane, _al(n * (width_acc // 2) * 4, 1024))
    o = 3 * plane + 2 * _al(k * width_acc * rb, 1024) + _al(n * 8, 16) + _al(nnz * 8, 16) + _al(n * 4, 16) + 32
    lo2 = o + plane + 4096 + 1024 <= SMEM_CAP
    if lo2:
        o = _al(o, 1024) + plane
    return o + 1024 <= SMEM_CAP, lo2


def stream_bands(op: Op, b: int, sw: int, sms: int):
    """entries of every CTA's row band of the streaming layer (csrc/mvb_stream_tc.cu stream_plan_sw), or None when the
    plan does not cover (N, B, sw)"""
    n = op.n_rows
    if b % sw:
        return None
    nslabs, rpt = b // sw, 128 // sw
    nrb_max = sms // nslabs
    if nrb_max < 1:
        return None
    rp = _al((n + nrb_max - 1) // nrb_max, rpt)
    if rp > ST_RCAP or (rp // rpt) * 16 > 512:
        return None
    rowptr = np.concatenate(([0], np.cumsum(np.bincount(op.rows, minlength=n))))
    return np.array([rowptr[min(r + rp, n)] - rowptr[r] for r in range(0, n, rp)])


# ---------------------------------------------------------------------------------------------
# float64 reference (vertex-major arrays [N, B, F])
# ---------------------------------------------------------------------------------------------
def _mm(m: sp.csr_matrix, x: np.ndarray) -> np.ndarray:
    return np.asarray(m @ x.reshape(x.shape[0], -1)).reshape((m.shape[0],) + x.shape[1:])


def cheb_ref_fwd(x, L: sp.csr_matrix, w, bias=None, U: Optional[sp.csr_matrix] = None):
    """-> (pre-activation [N,B,Fout], T_0): T_0 = x or U x, T_1 = L T_0, T_k = 2 L T_{k-1} - T_{k-2}, sum_k T_k W_k + b"""
    t0 = _mm(U, x) if U is not None else x
    pre = np.einsum("nbi,io->nbo", t0, w[0])
    tp, t = None, t0
    for k in range(1, w.shape[0]):
        tp, t = t, (_mm(L, t) if k == 1 else 2.0 * _mm(L, t) - tp)
        pre += np.einsum("nbi,io->nbo", t, w[k])
    if bias is not None:
        pre = pre + bias
    return pre, t0


def cheb_ref_bwd(g, t0, L: sp.csr_matrix, w, U: Optional[sp.csr_matrix] = None):
    """adjoint form for G = dY * [y > 0] [N,B,Fout]: S_k = T_k(L^T) G, dW_k = T_0^T S_k, db = sum G,
    dX = U^T sum_k S_k W_k^T  -> (dx, dw, db)"""
    lt = L.T.tocsr()
    dw = np.empty(w.shape)
    dt0 = np.zeros(t0.shape)
    sp_, s = None, g
    for k in range(w.shape[0]):
        if k:
            sp_, s = s, (_mm(lt, s) if k == 1 else 2.0 * _mm(lt, s) - sp_)
        dw[k] = np.einsum("nbi,nbo->io", t0, s)
        dt0 += np.einsum("nbo,io->nbi", s, w[k])
    dx = _mm(U.T.tocsr(), dt0) if U is not None else dt0
    return dx, dw, g.sum(axis=(0, 1))


def pool_ref(x, P: sp.csr_matrix):
    return _mm(P, x)


def pool_ref_bwd(dy, P: sp.csr_matrix):
    return _mm(P.T.tocsr(), dy)


def irregular_nnz(n: int, nnz: int, seed: int) -> Op:
    """a random square operator with exactly nnz entries at uniformly random (row, col) (duplicates and self loops
    included), vertex n - 1 used so that n_active == n; rows scaled as in `irregular`"""
    rng = np.random.default_rng(seed)
    rows, cols = rng.integers(0, n, nnz), rng.integers(0, n, nnz)
    rows[0] = n - 1
    vals = rng.uniform(0.2, 1.0, nnz) * rng.choice([-1.0, 1.0], nnz)
    return _op(f"random{n}x{nnz}", n, n, rows, cols, _scale_rows(rows, vals, n, rng))
