"""CPU checks of tests/operator_cases.py: the synthetic operator families have the properties they are meant to have,
the float64 reference agrees with the oracle's ChebConv_batch / SurfacePool run in float64 under autograd, and
MeshOperator classifies the pooling matrices (a D that selects one vertex twice is not a selection)."""
import numpy as np
import pytest
import torch

from tests import operator_cases as C
from oracle import mesh_vae_oracle as O


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    return meshvae_b200


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / np.abs(b).max())


# ---------------------------------------------------------------------------------------------
# generator properties
# ---------------------------------------------------------------------------------------------
def test_template_family_matches_oracle_cheb_norm():
    A, _, _, nn_ = O.load_operators(C.OPERATORS_NPZ)
    for lvl in range(5):
        op = C.template_L(lvl)
        ei, norm = O.cheb_norm(A[lvl]._indices(), nn_[lvl])
        ref = torch.sparse_coo_tensor(torch.stack((ei[1], ei[0])), norm.double(), (nn_[lvl],) * 2).to_dense().numpy()
        assert np.array_equal(op.csr.toarray(), ref)
        assert C.asymmetry(op) == 0.0


@pytest.mark.parametrize("lvl", [0, 2, 3])
def test_relabelled_is_a_permuted_template(lvl):
    t, r = C.template_L(lvl), C.relabelled(lvl, seed=lvl)
    assert C.asymmetry(r) == 0.0
    assert r.nnz == t.nnz and np.allclose(np.sort(r.vals), np.sort(t.vals))
    # the column band of a row is as wide as the mesh
    m = r.csr
    spans = [np.ptp(m.indices[m.indptr[i]:m.indptr[i + 1]]) for i in range(m.shape[0]) if m.indptr[i + 1] > m.indptr[i]]
    assert np.median(spans) > r.n_rows / 4


@pytest.mark.parametrize("lvl,both", [(0, False), (1, True), (2, False), (3, True), (4, False)])
def test_directed_family_is_asymmetric(lvl, both):
    op = C.directed(lvl, seed=lvl, both=both)
    assert C.asymmetry(op) > 0.1
    # one-way edges: the oracle's ChebConv_batch.norm of the same edge list gives the same values
    if not both:
        ei, norm = op.edges()
        e2, n2 = O.cheb_norm(ei, op.n_rows)
        assert torch.equal(e2, ei) and torch.allclose(n2, norm, rtol=1e-6, atol=0)


def test_irregular_family_structure():
    op = C.irregular(600, seed=1, hubs=3, isolated=7, dups=20, loops=9)
    m = op.csr
    deg = np.diff(np.concatenate(([0], np.cumsum(np.bincount(op.rows, minlength=op.n_rows)))))
    assert deg.max() >= 200                                                  # hubs
    empty = np.flatnonzero(deg == 0)
    assert empty.shape[0] >= 7 and empty.max() < op.n_rows - 1               # empty rows in the middle, not a suffix
    pairs = op.rows * op.n_cols + op.cols
    assert np.unique(pairs).shape[0] < pairs.shape[0]                        # duplicate entries
    assert np.any(op.rows == op.cols)                                        # self loops
    assert not np.all(np.diff(op.rows) >= 0)                                 # COO not sorted by row
    assert np.abs(m).sum(axis=1).max() <= 0.95 + 1e-6
    assert C.asymmetry(op) > 0.1
    tail = C.irregular(300, seed=2, n_active=260)
    assert max(tail.rows.max(), tail.cols.max()) < 260


def test_pooling_families():
    d = C.selection(500, 125, seed=3)
    assert np.unique(d.cols).shape[0] == 125 and not np.all(np.diff(d.cols) > 0)
    r = C.selection(500, 125, seed=3, repeat=3)
    assert np.unique(r.cols).shape[0] == 122
    w = C.weighted_down(500, 125, seed=4)
    assert np.all(np.bincount(w.rows) == 2)
    for m, n in ((500, 125), (100, 400)):
        u = C.upsample(m, n, seed=5)
        cnt = np.bincount(u.rows, minlength=m)
        assert cnt.min() == 0 and cnt.max() == 4


def test_stream_band_arithmetic():
    """dense-band operators overflow every CTA's staging area, hub-band operators only some of them"""
    dense = C.irregular(4998, seed=6, deg=(40, 48))
    hub = C.irregular(4998, seed=7, deg=(4, 8), hub_rows=np.arange(5, 1600, 400), hub_deg=(4200, 4400))
    for sw in (8, 16):
        assert C.stream_bands(dense, 64, sw, 148).min() > C.ST_ECAP
        bands = C.stream_bands(hub, 64, sw, 148)
        assert bands.max() > C.ST_ECAP and bands.min() <= C.ST_ECAP


# ---------------------------------------------------------------------------------------------
# the float64 reference pinned to the oracle (float64 under torch autograd)
# ---------------------------------------------------------------------------------------------
def _oracle_layer(x, op, w, b, relu, u=None, d=None, gy_seed=11):
    """oracle composition [SurfacePool(U)] -> ChebConv_batch -> [ReLU] -> [SurfacePool(D)] in float64; logical
    [B, N, F] tensors -> (y, dx, dw, db, gy, mask) with the incoming gradient gy"""
    xo = torch.from_numpy(x).permute(1, 0, 2).clone().requires_grad_()
    wo = torch.from_numpy(w).clone().requires_grad_()
    bo = torch.from_numpy(b).clone().requires_grad_()
    h = xo
    if u is not None:
        ut = u.sparse()
        h = O.surface_pool(h, ut._indices(), ut._values().double(), ut.shape)
    ei, norm = op.edges()
    pre = O.cheb_conv_batch(h, ei, norm.double(), wo, bo)
    y = torch.relu(pre) if relu else pre
    if d is not None:
        dt = d.sparse()
        y = O.surface_pool(y, dt._indices(), dt._values().double(), dt.shape)
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(gy_seed), dtype=torch.float64)
    y.backward(gy)
    vm = lambda t: t.detach().permute(1, 0, 2).numpy()                      # noqa: E731
    return vm(y), vm(xo.grad), wo.grad.numpy(), bo.grad.numpy(), vm(gy), vm((pre > 0).double())


def _reference_layer(x, op, w, b, relu, u=None, d=None, gy=None):
    U = u.csr if u is not None else None
    pre, t0 = C.cheb_ref_fwd(x, op.csr, w, b, U)
    mask = (pre > 0).astype(np.float64) if relu else np.ones_like(pre)
    y = pre * mask
    if d is not None:
        y = C.pool_ref(y, d.csr)
        gconv = C.pool_ref_bwd(gy, d.csr)
    else:
        gconv = gy
    dx, dw, db = C.cheb_ref_bwd(gconv * mask, t0, op.csr, w, U)
    return y, dx, dw, db


SMALL = {
    "template2": lambda: C.template_L(2), "template3": lambda: C.template_L(3), "template4": lambda: C.template_L(4),
    "relabelled3": lambda: C.relabelled(3, 1), "directed3": lambda: C.directed(3, 2, False),
    "directed4w": lambda: C.directed(4, 3, True),
    "irregular": lambda: C.irregular(90, seed=4, hubs=2, hub_deg=(40, 60), isolated=5, dups=12, loops=6),
    "tail": lambda: C.irregular(70, seed=5, n_active=50, dups=3, loops=2),
}


# polygon_order 6 (the default config) on every case, and the other orders a config may ask for: K = 1 (T_0 alone) and
# K = 2 (T_1 without a 2 L T - T step) are where a restated recurrence most easily goes wrong
REF_ORDERS = [(c, 6) for c in SMALL] + [(c, k) for c in SMALL for k in (1, 2, 3, 8)]


@pytest.mark.parametrize("case,K", REF_ORDERS, ids=[c if k == 6 else f"{c}-K{k}" for c, k in REF_ORDERS])
@pytest.mark.parametrize("kind", ["plain", "enc", "dec", "wdec"])
def test_reference_matches_oracle_float64(case, kind, K):
    op = SMALL[case]()
    n = op.n_rows
    rng = np.random.default_rng(len(case) * 7 + len(kind) + (0 if K == 6 else 100 * K))
    fin, fout, b = 5, 7, 3
    u = d = None
    n_in = n
    if kind == "enc":
        d = C.selection(n, max(n // 4, 1), seed=1)
    elif kind == "dec":
        n_in = max(n // 3, 2)
        u = C.upsample(n, n_in, seed=2)
    elif kind == "wdec":
        d = C.weighted_down(n, max(n // 3, 1), seed=3)
    x = rng.standard_normal((n_in, b, fin))
    w = rng.standard_normal((K, fin, fout)) * 0.3
    bias = rng.standard_normal(fout) * 0.1
    for relu in (False, True):
        yo, dxo, dwo, dbo, gy, _ = _oracle_layer(x, op, w, bias, relu, u, d)
        y, dx, dw, db = _reference_layer(x, op, w, bias, relu, u, d, gy)
        for a, ref in ((y, yo), (dx, dxo), (dw, dwo), (db, dbo)):
            assert _rel(a, ref) <= 1e-12


@pytest.mark.parametrize("m,n,kind", [(125, 500, "sel"), (125, 500, "rep"), (125, 500, "wdown"), (400, 100, "up"),
                                      (60, 200, "up")])
def test_pool_reference_matches_oracle_float64(m, n, kind):
    op = {"sel": lambda: C.selection(n, m, 1), "rep": lambda: C.selection(n, m, 1, repeat=4),
          "wdown": lambda: C.weighted_down(n, m, 2), "up": lambda: C.upsample(m, n, 3)}[kind]()
    rng = np.random.default_rng(m + n)
    x = rng.standard_normal((n, 4, 6))
    gy = rng.standard_normal((m, 4, 6))
    xo = torch.from_numpy(x).permute(1, 0, 2).clone().requires_grad_()
    t = op.sparse()
    yo = O.surface_pool(xo, t._indices(), t._values().double(), t.shape)
    yo.backward(torch.from_numpy(gy).permute(1, 0, 2))
    assert _rel(C.pool_ref(x, op.csr), yo.detach().permute(1, 0, 2).numpy()) <= 1e-12
    assert _rel(C.pool_ref_bwd(gy, op.csr), xo.grad.permute(1, 0, 2).numpy()) <= 1e-12


# ---------------------------------------------------------------------------------------------
# MeshOperator on the host: selection and n_active
# ---------------------------------------------------------------------------------------------
def test_is_selection_requires_distinct_columns(mvb):
    M = mvb.operators.MeshOperator
    assert M([0, 1, 2], [5, 9, 7], [1.0, 1.0, 1.0], 3, 10, "cpu").is_selection
    assert not M([0, 1, 2], [5, 5, 7], [1.0, 1.0, 1.0], 3, 10, "cpu").is_selection
    assert not M([0, 1, 2], [5, 6, 7], [1.0, 0.5, 1.0], 3, 10, "cpu").is_selection
    for op, sel in ((C.selection(500, 125, 1), True), (C.selection(500, 125, 1, repeat=1), False),
                    (C.weighted_down(500, 125, 2), False)):
        assert mvb.operators.from_sparse(op.sparse(), "cpu").is_selection == sel


def test_mesh_operator_n_active_on_cpu(mvb):
    op = C.irregular(300, seed=2, n_active=260)
    ei, norm = op.edges()
    m = mvb.operators.from_edges(ei, norm, 300, "cpu")
    assert m.n_active == 260 and m.nnz == op.nnz
    assert np.array_equal(m.rowptr.numpy(), np.concatenate(([0], np.cumsum(np.bincount(op.rows, minlength=300)))))
