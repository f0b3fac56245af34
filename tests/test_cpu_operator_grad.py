"""CPU checks of the value-free operator pattern behind the gradient with respect to the operator values: the COO
permutations perm / perm_t reproduce the CSR values of the host COO->CSR routine exactly (both orientations), and
ChebConv_batch.norm with edge weights is PyG's 'sym' normalisation (the oracle shim) without its cancelling diagonal."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import mesh_vae_oracle as O
from tests import operator_cases as C
from tests.helpers import OPERATORS_NPZ, ROOT


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    return meshvae_b200


def _template_coo():
    """(name, rows, cols, vals, n_rows, n_cols): the template's L_hat at levels 0-4 (rows = targets, as from_edges
    hands them over), its D1 and its U0"""
    d = np.load(OPERATORS_NPZ)
    out = []
    for lvl in range(5):
        op = C.template_L(lvl)
        out.append((f"A{lvl}", op.rows, op.cols, op.vals, op.n_rows, op.n_cols))
    for name in ("D1", "U0"):
        shape = d[f"{name}_shape"]
        out.append((name, d[f"{name}_row"].astype(np.int64), d[f"{name}_col"].astype(np.int64),
                    d[f"{name}_val"].astype(np.float32), int(shape[0]), int(shape[1])))
    return out


def _edge_cases():
    """duplicates (also of whole rows), explicit zeros, empty rows inside and at the end, unsorted COO order"""
    rng = np.random.default_rng(3)
    rows = np.array([5, 0, 2, 2, 0, 5, 2, 3, 3, 0, 2, 5], np.int64)
    cols = np.array([1, 4, 2, 2, 4, 0, 6, 3, 3, 1, 2, 1], np.int64)
    vals = rng.uniform(-1, 1, rows.shape[0]).astype(np.float32)
    vals[[3, 7]] = 0.0
    return [("dups_zeros_tail", rows, cols, vals, 9, 9),            # rows 1, 4, 6-8 empty; columns 5, 7, 8 empty
            ("irregular", *(lambda o: (o.rows, o.cols, o.vals, o.n_rows, o.n_cols))(
                C.irregular(200, seed=4, hubs=2, hub_deg=(40, 80), isolated=5, dups=15, loops=6, n_active=180)))]


@pytest.mark.parametrize("case", _template_coo() + _edge_cases(), ids=lambda c: c[0])
def test_coo_permutations_reproduce_csr_values(mvb, case):
    _, rows, cols, vals, n_rows, n_cols = case
    perm, perm_t = mvb.operators.coo_permutations(rows, cols)
    for transpose, p in ((False, perm), (True, perm_t)):
        rp, ci, v = mvb.operators.csr_from_coo_host(rows, cols, vals, n_rows, n_cols, transpose=transpose)
        assert p.dtype == np.int32 and np.array_equal(np.sort(p), np.arange(rows.shape[0]))
        assert np.array_equal(vals[p].view(np.int32), v.view(np.int32))          # bit for bit, zeros and signs too
        assert np.array_equal((cols if not transpose else rows)[p], ci)


@pytest.mark.parametrize("case", _edge_cases(), ids=lambda c: c[0])
def test_edge_pattern_matches_mesh_operator(mvb, case):
    """the pattern's CSR arrays and n_active are MeshOperator's; its perm / perm_t pick MeshOperator's values"""
    _, rows, cols, vals, n, _ = case
    ei = torch.from_numpy(np.vstack((cols, rows)))
    pat = mvb.operators.EdgePattern(ei, n, "cpu")
    ref = mvb.operators.MeshOperator(rows, cols, vals, n, n, "cpu")
    for a in ("rowptr", "colidx", "rowptr_t", "colidx_t"):
        assert torch.equal(getattr(pat, a), getattr(ref, a)), a
    assert pat.n_active == ref.n_active and pat.nnz == ref.nnz
    assert torch.equal(torch.from_numpy(vals)[pat.perm.long()], ref.vals)
    assert torch.equal(torch.from_numpy(vals)[pat.perm_t.long()], ref.vals_t)


def _pyg_shim_chebconv():
    """the oracle's PyG 2.0.4 ChebConv restatement, imported without leaving its shim packages in sys.modules"""
    before = set(sys.modules)
    sys.path.insert(0, os.path.join(ROOT, "oracle", "shims"))
    try:
        from torch_geometric.nn.conv.cheb_conv import ChebConv
    finally:
        sys.path.pop(0)
        for name in set(sys.modules) - before:
            if name.split(".")[0] in ("torch_geometric", "torch_scatter"):
                del sys.modules[name]
    return ChebConv


@pytest.mark.parametrize("lvl", [0, 2, 4])
def test_cheb_norm_with_edge_weights_matches_pyg(mvb, lvl):
    A, _, _, nn_ = O.load_operators(OPERATORS_NPZ)
    idx, n = A[lvl]._indices(), nn_[lvl]
    g = torch.Generator().manual_seed(lvl)
    w = torch.rand(idx.shape[1], generator=g, dtype=torch.float64) * 1.8 + 0.2
    loops = torch.arange(3)                          # a few self loops: both drop them (and their weights)
    idx = torch.cat((idx, torch.stack((loops, loops))), 1)
    w = torch.cat((w, torch.full((3,), 5.0, dtype=torch.float64)))
    ei, norm = mvb.ChebConv_batch.norm(idx, n, w, torch.float64)
    shim = _pyg_shim_chebconv()(1, 1, 2)
    ei_p, norm_p = shim.__norm__(idx, n, w, "sym", torch.tensor(2.0, dtype=torch.float64), dtype=torch.float64)
    e = ei.shape[1]
    # PyG appends n loops of +1 (get_laplacian) and n of -1 (lambda_max = 2): they cancel
    assert ei_p.shape[1] == e + 2 * n
    assert torch.equal(norm_p[e:e + n], torch.ones(n, dtype=torch.float64))
    assert torch.equal(norm_p[e + n:], -torch.ones(n, dtype=torch.float64))
    assert torch.equal(ei, ei_p[:, :e])
    torch.testing.assert_close(norm, norm_p[:e], rtol=1e-15, atol=0)
    # the same values, differentiably, as the oracle's ChebConv_batch.norm
    wr = w.clone().requires_grad_(True)
    _, nr = O.cheb_norm(idx, n, wr)
    torch.testing.assert_close(mvb.ChebConv_batch.norm(idx, n, wr)[1], nr, rtol=0, atol=0)
