"""Operator hand-off: the reference's uncoalesced COO operators (model.py:24-32) and the
(edge_index, norm) pairs of ChebConv_batch.norm (nn/conv.py:541-555) -> immutable CSR +
transpose-CSR on the device, built once per operator and cached.

The build is the host routine `mvb_csr_from_coo_host` (stable counting sort: entries of a row stay
in COO order, duplicates kept), so it can be tested without a GPU; the arrays are then uploaded.

Values that need a gradient (a `norm` computed from learned edge weights) change every step: they take the
value-free EdgePattern, cached by the index tensor alone, and are bound to it on the device per call."""
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib


def csr_from_coo_host(rows: np.ndarray, cols: np.ndarray, vals: np.ndarray, n_rows: int, n_cols: int,
                      transpose: bool = False) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """numpy in / numpy out wrapper of the C ABI host routine (CSR of P, or of P^T)."""
    rows = np.ascontiguousarray(rows, dtype=np.int64)
    cols = np.ascontiguousarray(cols, dtype=np.int64)
    vals = np.ascontiguousarray(vals, dtype=np.float32)
    nnz = int(rows.shape[0])
    n_out_rows, n_out_cols = (n_cols, n_rows) if transpose else (n_rows, n_cols)
    rowptr = np.zeros(n_out_rows + 1, dtype=np.int32)
    colidx = np.zeros(max(nnz, 1), dtype=np.int32)
    v = np.zeros(max(nnz, 1), dtype=np.float32)
    rc = _lib.lib.mvb_csr_from_coo_host(n_out_rows, n_out_cols, nnz, rows.ctypes.data, cols.ctypes.data,
                                        vals.ctypes.data, 1 if transpose else 0, rowptr.ctypes.data,
                                        colidx.ctypes.data, v.ctypes.data)
    _lib.check(rc, "mvb_csr_from_coo_host")
    return rowptr, colidx[:nnz], v[:nnz]


class MeshOperator:
    """A fixed sparse operator P [n_rows, n_cols] resident on one device as CSR(P) and CSR(P^T)."""

    def __init__(self, rows, cols, vals, n_rows: int, n_cols: int, device):
        rows = np.asarray(rows)
        cols = np.asarray(cols)
        vals = np.asarray(vals)
        self.n_rows, self.n_cols, self.nnz = int(n_rows), int(n_cols), int(rows.shape[0])
        self.device = torch.device(device)
        rp, ci, v = csr_from_coo_host(rows, cols, vals, n_rows, n_cols, transpose=False)
        rpt, cit, vt = csr_from_coo_host(rows, cols, vals, n_rows, n_cols, transpose=True)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.device)  # noqa: E731
        self.rowptr, self.colidx, self.vals = up(rp), up(ci), up(v)
        self.rowptr_t, self.colidx_t, self.vals_t = up(rpt), up(cit), up(vt)
        # one nonzero per row with value 1 at distinct columns (the D matrices, mesh_operations.py:72-85): pure row
        # selection.  The fused kernels invert it (inv[sel[r]] = r), so a column selected twice must take the SpMM path
        self.is_selection = bool(self.nnz == n_rows and np.all(np.diff(rp) == 1) and np.all(v == 1.0)
                                 and np.unique(ci).shape[0] == self.nnz)
        # square operators: rows >= n_active are empty and no entry references a column >= n_active
        # (the coarse operator applied to a finer tensor, models/cheb_VAE.py:288) -> closed-form rows
        self.n_active = self.n_rows
        if n_rows == n_cols:
            self.n_active = int(max(rows.max(), cols.max())) + 1 if self.nnz else 0

    def csr_bytes(self) -> int:
        return (self.n_rows + 1) * 4 + self.nnz * 8


_CACHE: Dict[tuple, Tuple[MeshOperator, tuple]] = {}


def _key(idx: torch.Tensor, val: Optional[torch.Tensor], n_rows: int, n_cols: int, kind: str, device):
    return (kind, idx.data_ptr(), idx._version, None if val is None else (val.data_ptr(), val._version),
            int(idx.shape[-1]), n_rows, n_cols, str(idx.device), str(device))


def from_edges(edge_index: torch.Tensor, norm: torch.Tensor, n: int, device=None) -> MeshOperator:
    """L_hat as used by propagate with flow='source_to_target' (nn/conv.py:172): out[t] sums
    norm[e] * x[edge_index[0][e]] over edges with edge_index[1][e] == t; N comes from x (size=None,
    nn/conv.py:160-169), so a coarse operator on a finer tensor simply has empty rows."""
    device = norm.device if device is None else torch.device(device)
    key = _key(edge_index, norm, n, n, "edges", device)
    hit = _CACHE.get(key)
    if hit is None:
        ei = edge_index.detach().cpu().numpy()
        op = MeshOperator(ei[1], ei[0], norm.detach().float().cpu().numpy(), n, n, device)
        _CACHE[key] = hit = (op, (edge_index, norm))      # keep the keyed storages alive
    return hit[0]


def from_sparse(mat: torch.Tensor, device=None) -> MeshOperator:
    """A torch sparse COO matrix used through _indices()/_values() exactly as given (nn/pool.py:19)."""
    idx, val = mat._indices(), mat._values()
    device = val.device if device is None else torch.device(device)
    key = _key(idx, val, int(mat.shape[0]), int(mat.shape[1]), "coo", device)
    hit = _CACHE.get(key)
    if hit is None:
        i = idx.detach().cpu().numpy()
        op = MeshOperator(i[0], i[1], val.detach().float().cpu().numpy(), int(mat.shape[0]), int(mat.shape[1]),
                          device)
        _CACHE[key] = hit = (op, (idx, val, mat))
    return hit[0]


class EdgePattern:
    """The pattern of an L_hat whose values change from call to call (computed from learned edge weights): CSR(L) and
    CSR(L^T) without values, with perm / perm_t mapping each CSR slot to its COO entry.  `bind(norm)` fills the values
    of both orientations on the device (mvb_csr_values): no host round trip, nothing cached per call."""

    def __init__(self, edge_index: torch.Tensor, n: int, device):
        ei = edge_index.detach().cpu().numpy()
        rows, cols = ei[1], ei[0]
        self.n_rows = self.n_cols = int(n)
        self.nnz = int(rows.shape[0])
        self.device = torch.device(device)
        ones = np.ones(self.nnz, np.float32)
        rp, ci, _ = csr_from_coo_host(rows, cols, ones, n, n, transpose=False)
        rpt, cit, _ = csr_from_coo_host(rows, cols, ones, n, n, transpose=True)
        perm, perm_t = coo_permutations(rows, cols)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(self.device)  # noqa: E731
        self.rowptr, self.colidx, self.perm = up(rp), up(ci), up(perm)
        self.rowptr_t, self.colidx_t, self.perm_t = up(rpt), up(cit), up(perm_t)
        self.device = self.rowptr.device            # with its index: compared with the values' device in bind()
        self.is_selection = False
        self.n_active = int(max(rows.max(), cols.max())) + 1 if self.nnz else 0

    def bind(self, norm: torch.Tensor) -> "BoundOperator":
        """the operator with values `norm` [nnz] (fp32, on this pattern's device, COO order of edge_index)"""
        if norm.dtype != torch.float32 or norm.device != self.device or tuple(norm.shape) != (self.nnz,):
            raise _lib.MvbError(f"operator values: expected float32 [{self.nnz}] on {self.device}, got {norm.dtype} "
                                f"{tuple(norm.shape)} on {norm.device}")
        norm = norm.detach().contiguous()
        vals = torch.empty(max(self.nnz, 1), device=self.device, dtype=torch.float32)
        vals_t = torch.empty_like(vals)
        _lib.check(_lib.lib.mvb_csr_values(self.nnz, self.perm.data_ptr(), self.perm_t.data_ptr(), norm.data_ptr(),
                                           vals.data_ptr(), vals_t.data_ptr(), _lib.stream_ptr()), "mvb_csr_values")
        return BoundOperator(self, vals, vals_t)


class BoundOperator:
    """An EdgePattern with the values of one call: what MeshOperator offers, plus `pattern` (for perm)"""

    def __init__(self, pattern: EdgePattern, vals: torch.Tensor, vals_t: torch.Tensor):
        self.pattern, self.vals, self.vals_t = pattern, vals, vals_t

    def __getattr__(self, name):
        return getattr(self.pattern, name)


def coo_permutations(rows: np.ndarray, cols: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """(perm, perm_t): the COO entry behind each slot of CSR(P) and of CSR(P^T) as csr_from_coo_host orders them (its
    stable counting sort keeps the COO order within a row, i.e. a stable argsort of the rows, resp. columns)"""
    return (np.argsort(np.asarray(rows), kind="stable").astype(np.int32),
            np.argsort(np.asarray(cols), kind="stable").astype(np.int32))


_PATTERNS: Dict[tuple, Tuple[EdgePattern, torch.Tensor]] = {}


def pattern_from_edges(edge_index: torch.Tensor, n: int, device=None) -> EdgePattern:
    """the cached pattern of the L_hat with entries (edge_index[1][e], edge_index[0][e]) on n vertices, keyed by the
    index tensor (identity and version), n and the device - not by any values"""
    device = edge_index.device if device is None else torch.device(device)
    key = _key(edge_index, None, n, n, "pattern", device)
    hit = _PATTERNS.get(key)
    if hit is None:
        _PATTERNS[key] = hit = (EdgePattern(edge_index, n, device), edge_index)
    return hit[0]


def edge_operator(edge_index: torch.Tensor, norm: torch.Tensor, n: int, device):
    """(operator, values) for functional.cheb_conv: the cached pattern and norm as fp32 values when norm needs a
    gradient, else the value-keyed cached operator and None"""
    if norm.requires_grad and torch.is_grad_enabled():
        return pattern_from_edges(edge_index, n, device), norm.to(device=device, dtype=torch.float32)
    return from_edges(edge_index, norm, n, device), None


def clear_cache():
    _CACHE.clear()
    _PATTERNS.clear()
