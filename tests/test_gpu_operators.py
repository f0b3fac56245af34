"""The sparse and mesh-layer kernels on operators other than the template's (tests/operator_cases.py), against a float64
reference of the same operation: non-symmetric L_hat (a kernel that used L where L^T is meant passes on the template),
irregular degree / hubs / duplicates / self loops / empty rows in the middle, an isolated tail (n_active < N), unsorted
and repeated row selections, weighted down-sampling, up-sampling with 0-4 entries per row, vertex counts at the tile
edges, operators on either side of the kernels' shared-memory boundaries, and row bands of the streaming layer that
overflow its staging area.

Gates: rel_err < 1e-4 and elem_err <= 1 (tests/helpers.py) for y, dx, dW and db; the ReLU mask is the device's, and a
decision may differ from the reference only where the reference pre-activation is within 1e-5 max|y| of zero.  Exact
invariants: bit-identical results run to run, and fused_recurrence=1 bit-identical to the step-by-step recurrence."""
import numpy as np
import pytest
import torch

from tests import operator_cases as C
from tests.helpers import rel_err, elem_err

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-4
MAX_ERR = {}          # entry point -> largest rel_err seen (printed at the end of the module with pytest -s)


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    yield meshvae_b200
    print("\nlargest rel_err per entry point: " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(MAX_ERR.items())))


def _reset(mvb):
    mvb._lib.tune("mesh_tc=1,0;stream_tc=0,16;fused_recurrence=1")
    mvb._lib.lib.mvb_set_tensor_cores(1)


def _dev(a, grad=False):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(DEV).requires_grad_(grad)


def _gate(entry, what, dev, ref):
    d, r = dev.detach().double().cpu(), torch.from_numpy(np.asarray(ref, np.float64))
    e = rel_err(d, r)
    MAX_ERR[entry] = max(MAX_ERR.get(entry, 0.0), e)
    assert e < TOL, f"{entry} {what}: rel_err {e:.3e}"
    ee = elem_err(d, r)
    assert ee <= 1.0, f"{entry} {what}: elem_err {ee:.3f}"


def _l_op(mvb, op: C.Op):
    ei, norm = op.edges()
    return mvb.operators.from_edges(ei.to(DEV), norm.to(DEV), op.n_rows, DEV)


def _p_op(mvb, op: C.Op):
    return mvb.operators.from_sparse(op.sparse().to(DEV), DEV)


def _inputs(seed, n_in, b, fin, fout, k, bias=True):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n_in, b, fin)), rng.standard_normal((k, fin, fout)) * 0.1,
            rng.standard_normal(fout) * 0.1 if bias else None, rng)


def _check_layer(entry, fn, op, x, w, bias, relu, u=None, d=None, need_dx=True, rng=None):
    """run fn(x, w, b) -> y (vertex-major, autograd) on the device, backward with a random dY, and gate y / dx / dW / db
    against the float64 reference of [U] -> ChebConv -> [ReLU] -> [D] (the ReLU mask taken from the device output)"""
    xg, wg = _dev(x, need_dx), _dev(w, True)
    bg = _dev(bias, True) if bias is not None else None
    yg = fn(xg, wg, bg)
    pre, t0 = C.cheb_ref_fwd(x, op.csr, w, bias, u.csr if u is not None else None)
    pre_out = C.pool_ref(pre, d.csr) if d is not None else pre
    assert tuple(yg.shape) == pre_out.shape
    if relu:
        assert d is None or d.csr.max() == 1.0 and np.all(np.diff(d.csr.indptr) == 1), "ReLU before a weighted D"
        mask = (yg.detach().cpu().numpy() > 0).astype(np.float64)
        flips = mask != (pre_out > 0)
        assert np.all(np.abs(pre_out[flips]) <= 1e-5 * np.abs(pre_out).max()), "a ReLU decision differs from the reference"
    else:
        mask = np.ones_like(pre_out)
    gy = rng.standard_normal(pre_out.shape)
    yg.backward(_dev(gy))
    g = gy * mask
    g_conv = C.pool_ref_bwd(g, d.csr) if d is not None else g
    dx, dw, db = C.cheb_ref_bwd(g_conv, t0, op.csr, w, u.csr if u is not None else None)
    _gate(entry, "y", yg, pre_out * mask)
    if need_dx:
        _gate(entry, "dx", xg.grad, dx)
    _gate(entry, "dW", wg.grad, dw)
    if bias is not None:
        _gate(entry, "db", bg.grad, db)
    return yg


# ---------------------------------------------------------------------------------------------
# operator cases
# ---------------------------------------------------------------------------------------------
SQUARE = {
    "irregular300": lambda: C.irregular(300, seed=1, hubs=3, hub_deg=(200, 290), isolated=9, dups=30, loops=12),
    "directed1w": lambda: C.directed(1, seed=2, both=True),
    "directed2": lambda: C.directed(2, seed=3, both=False),
    "relabelled2": lambda: C.relabelled(2, seed=4),
    "tail300": lambda: C.irregular(300, seed=5, n_active=241, dups=10, loops=5, isolated=4),
}
EDGE_N = [1, 2, 127, 128, 129, 255, 256, 257]


def _edge_op(n):
    return C.irregular(n, seed=n, dups=min(n, 5), loops=min(n, 3), isolated=2 if n > 8 else 0)


# ---------------------------------------------------------------------------------------------
# mvb_spmm
# ---------------------------------------------------------------------------------------------
SPMM_OPS = {**{k: SQUARE[k] for k in ("irregular300", "directed2", "tail300")},
            "up400x100": lambda: C.upsample(400, 100, seed=6), "wdown80x300": lambda: C.weighted_down(300, 80, seed=7)}


@pytest.mark.parametrize("case", list(SPMM_OPS))
@pytest.mark.parametrize("b,f", [(4, 16), (3, 5)])
def test_spmm(mvb, case, b, f):
    op = SPMM_OPS[case]()
    L = mvb._lib
    m = _p_op(mvb, op) if op.n_rows != op.n_cols else _l_op(mvb, op)
    rng = np.random.default_rng(b * 100 + f)
    x = rng.standard_normal((op.n_cols, b, f))
    z, w = rng.standard_normal((2, op.n_rows, b, f))
    lx = C.pool_ref(x, op.csr)
    xg, zg, wg = _dev(x), _dev(z), _dev(w)
    for alpha, beta, use_z, use_w in ((2.0, -1.0, True, True), (0.5, 0.0, False, False), (1.0, 0.25, True, False),
                                      (-1.0, 0.0, False, True)):
        y = torch.full((op.n_rows, b, f), float("nan"), device=DEV)
        L.check(L.lib.mvb_spmm(op.n_rows, op.n_cols, L.ptr(m.rowptr), L.ptr(m.colidx), L.ptr(m.vals), L.ptr(xg), L.ptr(y),
                               L.ptr(zg) if use_z else None, L.ptr(wg) if use_w else None, alpha, beta, b * f,
                               L.stream_ptr()), "mvb_spmm")
        ref = alpha * lx + (beta * z if use_z else 0.0) + (w if use_w else 0.0)
        _gate("mvb_spmm", f"a={alpha} b={beta}", y, ref)
        if use_w:                       # y aliasing w (the reverse recurrence's in-place update): the same bits
            wa = wg.clone()
            L.check(L.lib.mvb_spmm(op.n_rows, op.n_cols, L.ptr(m.rowptr), L.ptr(m.colidx), L.ptr(m.vals), L.ptr(xg),
                                   L.ptr(wa), L.ptr(zg) if use_z else None, L.ptr(wa), alpha, beta, b * f, L.stream_ptr()),
                    "mvb_spmm")
            assert torch.equal(wa, y)


# ---------------------------------------------------------------------------------------------
# mvb_pool_fwd / _bwd, Pool
# ---------------------------------------------------------------------------------------------
POOL_OPS = {"sel": (lambda: C.selection(1250, 313, 1), True), "sel_rep": (lambda: C.selection(1250, 313, 2, repeat=9), False),
            "wdown": (lambda: C.weighted_down(900, 300, 3), False), "up_more": (lambda: C.upsample(1250, 313, 4), False),
            "up_fewer": (lambda: C.upsample(200, 700, 5), False)}


@pytest.mark.parametrize("case", list(POOL_OPS))
@pytest.mark.parametrize("b,f", [(3, 16), (2, 3)])
def test_pool(mvb, case, b, f):
    mk, is_sel = POOL_OPS[case]
    op = mk()
    p = _p_op(mvb, op)
    assert p.is_selection == is_sel
    rng = np.random.default_rng(len(case) + f)
    x, dy = rng.standard_normal((op.n_cols, b, f)), rng.standard_normal((op.n_rows, b, f))
    xg = _dev(x, True)
    y = mvb.functional.pool(xg, p)
    y.backward(_dev(dy))
    _gate("mvb_pool", "y", y, C.pool_ref(x, op.csr))
    _gate("mvb_pool", "dx", xg.grad, C.pool_ref_bwd(dy, op.csr))
    y1 = mvb.Pool(_dev(x).permute(1, 0, 2), op.sparse().to(DEV))
    _gate("Pool", "y", y1.permute(1, 0, 2), C.pool_ref(x, op.csr))


# ---------------------------------------------------------------------------------------------
# mvb_cheb_fwd / _bwd through cheb_conv
# ---------------------------------------------------------------------------------------------
# (Fin, Fout): 16 -> 16 takes the adjoint-form backward (Fout <= 1.2 Fin), 16 -> 32 the basis form, 3 -> 16 the padded
# 3-channel input
CONV_CASES = [(c, tc, fin, fout, k, relu) for c in SQUARE for (tc, fin, fout, k, relu) in
              [(1, 16, 16, 6, True), (0, 16, 16, 6, True), (1, 16, 32, 3, True), (0, 16, 32, 2, False), (1, 3, 16, 1, False),
               (1, 32, 16, 6, False)]]


@pytest.mark.parametrize("case,tc,fin,fout,k,relu", CONV_CASES)
def test_cheb_conv(mvb, case, tc, fin, fout, k, relu):
    op = SQUARE[case]()
    lo = _l_op(mvb, op)
    assert (lo.n_active < op.n_rows) == (case == "tail300")
    x, w, bias, rng = _inputs(hash((case, fin, fout, k)) % 1000, op.n_rows, 3, fin, fout, k)
    mvb._lib.lib.mvb_set_tensor_cores(tc)
    try:
        _check_layer("mvb_cheb", lambda a, b_, c: mvb.functional.cheb_conv(a, b_, c, lo, relu), op, x, w, bias, relu, rng=rng)
    finally:
        _reset(mvb)


@pytest.mark.parametrize("n", EDGE_N)
def test_cheb_conv_vertex_counts(mvb, n):
    op = _edge_op(n)
    lo = _l_op(mvb, op)
    x, w, bias, rng = _inputs(n, n, 5, 16, 16, 6)
    _check_layer("mvb_cheb", lambda a, b_, c: mvb.functional.cheb_conv(a, b_, c, lo, True), op, x, w, bias, True, rng=rng)


def _k_ids(cases, k_col=-1):
    """pytest ids of a case table with a polygon-order column: the K = 6 rows keep the ids they had before the column
    existed, the other orders get a -K<k> suffix"""
    return ["-".join(str(v) for i, v in enumerate(c) if i != k_col % len(c)) + ("" if c[k_col] == 6 else f"-K{c[k_col]}")
            for c in cases]


# (Fin, Fout, K): the default order, and K = 2 / 3 / 8 (no 2 L T - T step, one, and more steps than the default)
RECUR_CASES = [(16, 16, 6), (16, 32, 6), (16, 16, 2), (16, 32, 3), (16, 16, 8), (16, 32, 8)]


@pytest.mark.parametrize("case", ["irregular300", "directed1w", "tail300"])
@pytest.mark.parametrize("fin,fout,k", RECUR_CASES, ids=_k_ids(RECUR_CASES))
def test_fused_recurrence_is_bit_identical_on_other_operators(mvb, case, fin, fout, k):
    """the one-kernel recurrence of small levels sums in the order of the step-by-step SpMM launches"""
    op = SQUARE[case]()
    lo = _l_op(mvb, op)
    x, w, bias, rng = _inputs(7, op.n_rows, 6, fin, fout, k)
    dy = _dev(rng.standard_normal((op.n_rows, 6, fout)))
    res = []
    try:
        for fused in (1, 0):
            mvb._lib.tune(f"fused_recurrence={fused}")
            xg, wg, bg = _dev(x, True), _dev(w, True), _dev(bias, True)
            y = mvb.functional.cheb_conv(xg, wg, bg, lo, True)
            y.backward(dy)
            res.append((y.detach(), xg.grad, wg.grad, bg.grad))
    finally:
        _reset(mvb)
    for a, b_ in zip(*res):
        assert torch.equal(a, b_)


# ---------------------------------------------------------------------------------------------
# mvb_cheb_sel_fwd / _bwd through cheb_conv_sel
# ---------------------------------------------------------------------------------------------
SEL_CASES = [("irregular300", 0, 4), ("irregular300", 0, 16), ("directed1w", 0, 32), ("relabelled2", 0, 16),
             ("irregular300", 5, 16), ("directed2", 3, 4)]


@pytest.mark.parametrize("case,repeat,fin", SEL_CASES)
def test_cheb_conv_sel(mvb, case, repeat, fin):
    op = SQUARE[case]()
    d = C.selection(op.n_rows, (op.n_rows + 3) // 4, seed=fin + repeat, repeat=repeat)
    lo, do = _l_op(mvb, op), _p_op(mvb, d)
    fout, k = 16, (3 if fin == 32 else 6)
    x, w, bias, rng = _inputs(fin * 3 + repeat, op.n_rows, 5, fin, fout, k)
    Fn = mvb.functional
    xv = _dev(x)
    fused = Fn.cheb_conv_sel_supported(xv, _dev(w), lo, do)
    assert fused == (repeat == 0), "a repeated selection must take the composition path"

    def run(a, b_, c):
        if fused:
            return Fn.cheb_conv_sel(a, b_, c, lo, do, relu=True)
        return Fn.pool(Fn.cheb_conv(a, b_, c, lo, True), do)
    _check_layer("mvb_cheb_sel", run, op, x, w, bias, True, d=d, need_dx=False, rng=rng)


# ---------------------------------------------------------------------------------------------
# mvb_cheb_layer_fwd / _bwd through cheb_layer
# ---------------------------------------------------------------------------------------------
MODES = ["mesh_tc=1,0", "mesh_tc=1,1", "mesh_tc=1,2", "mesh_tc=0,0"]
LAYER_OPS = {**SQUARE, "relabelled3": lambda: C.relabelled(3, seed=14)}
# (operator, kind, B, Fin, Fout, relu, K)
LAYER_CASES = [("directed2", "enc", 8, 16, 16, True, 6), ("directed2", "dec", 8, 16, 32, True, 6),
               ("relabelled2", "enc", 16, 32, 32, True, 6), ("irregular300", "plain", 4, 16, 16, True, 6),
               ("irregular300", "dec", 6, 32, 16, True, 6), ("directed1w", "plain", 8, 16, 16, True, 6),
               ("irregular300", "wenc", 4, 16, 16, False, 6), ("directed2", "enc_rep", 4, 16, 16, True, 6),
               ("tail300", "plain", 4, 16, 16, True, 6)]
# the orders a config may ask for (the tensor-core mesh kernels take K <= 16).  The backward reduces dW in plane groups of
# at most 128 / Fout planes (csrc/mvb_mesh_tc.cu wgrad_group): one group on the tensor cores (Fout 16: K <= 6; Fout 32:
# K <= 3), one group too wide for them that falls to the FFMA reduction (Fout 16: K 7-8; Fout 32: K 4), several groups
# each finalized into its own slice of dW (Fout 16: K 9, 16; Fout 32: K 5-16).  Operators whose T_k stay bounded at
# K = 16: row sums <= 0.95, or a symmetric normalised L_hat
LAYER_CASES += [("irregular300", ("enc", "dec", "plain")[i % 3], 8, 16, 16, True, k) for i, k in enumerate((1, 2, 3, 4, 5, 7, 8, 9, 16))]
LAYER_CASES += [("relabelled2", ("dec", "plain", "enc")[i % 3], 8, 32 if k % 2 else 16, 32, True, k)
                for i, k in enumerate((1, 2, 3, 4, 5, 7, 8, 9, 16))]
# widths only the FFMA mesh kernels take
LAYER_CASES += [("directed2", "enc", 4, 8, 8, True, 2), ("irregular300", "dec", 4, 8, 8, False, 7),
                ("relabelled3", "plain", 4, 64, 64, True, 3), ("relabelled3", "enc", 8, 64, 64, True, 9)]


def _layer_ops(op, kind, seed):
    n = op.n_rows
    u = d = None
    if kind == "enc":
        d = C.selection(n, (n + 3) // 4, seed)
    elif kind == "enc_rep":
        d = C.selection(n, (n + 3) // 4, seed, repeat=4)
    elif kind == "wenc":
        d = C.weighted_down(n, (n + 3) // 4, seed)
    elif kind == "dec":
        u = C.upsample(n, (n + 3) // 4, seed)
    return u, d


def _run_layer_case(mvb, op, kind, b, fin, fout, relu, mode, k=6, expect_fused=None):
    u, d = _layer_ops(op, kind, b + fin)
    lo = _l_op(mvb, op)
    uo = _p_op(mvb, u) if u is not None else None
    do = _p_op(mvb, d) if d is not None else None
    n_in = u.n_cols if u is not None else op.n_rows
    x, w, bias, rng = _inputs(b * 7 + fin, n_in, b, fin, fout, k)
    Fn = mvb.functional
    sup = Fn.cheb_layer_supported(op.n_rows, b, fin, fout, k, lo, uo, do)
    if expect_fused is not None:
        assert sup == expect_fused, f"cheb_layer_supported = {sup} under {mode}"
    c0 = mvb._lib.lib.mvb_launch_count()
    counted = {}

    def run(a, b_, c):
        y = Fn.cheb_layer(a, b_, c, lo, uo, do, relu=relu)
        counted["fwd"] = mvb._lib.lib.mvb_launch_count() - c0
        return y
    _check_layer("mvb_cheb_layer" if sup else "composition", run, op, x, w, bias, relu, u=u, d=d, rng=rng)
    if sup:
        assert counted["fwd"] == 1, "the fused layer is one launch"
    return sup


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case,kind,b,fin,fout,relu,k", LAYER_CASES, ids=_k_ids(LAYER_CASES))
def test_cheb_layer(mvb, case, kind, b, fin, fout, relu, k, mode):
    op = LAYER_OPS[case]()
    mvb._lib.tune(mode)
    try:
        # a selection with a repeated vertex, a weighted D and an isolated tail are not the fused kernels' layers
        fits = kind not in ("wenc", "enc_rep") and case != "tail300"
        _run_layer_case(mvb, op, kind, b, fin, fout, relu, mode, k=k,
                        expect_fused=(False if not fits else (True if mode == "mesh_tc=1,0" else None)))
    finally:
        _reset(mvb)


@pytest.mark.parametrize("n", EDGE_N)
def test_cheb_layer_vertex_counts(mvb, n):
    op = _edge_op(n)
    _run_layer_case(mvb, op, "plain", 4, 16, 16, True, "auto")


def _bisect_capacity(mvb, fin, fout, b, k, deg):
    sup = lambda n: bool(mvb._lib.lib.mvb_cheb_layer_supported(n, b, fin, fout, k, deg * n, n, 0, n))    # noqa: E731
    lo, hi = 1, 4096
    assert sup(lo) and not sup(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if sup(mid) else (lo, mid)
    return lo


@pytest.mark.parametrize("fin,fout", [(16, 16), (16, 32), (32, 32), (32, 16)])
def test_cheb_layer_capacity_edge(mvb, fin, fout):
    """the largest plain layer mvb_cheb_layer_supported accepts (7 entries per row, 8 meshes) runs fused; one vertex
    more falls back to the composition and is still right"""
    b, k, deg = 8, 6, 7
    n_max = _bisect_capacity(mvb, fin, fout, b, k, deg)
    for n, fused in ((n_max, True), (n_max + 1, False)):
        op = C.irregular_nnz(n, deg * n, seed=n)
        _run_layer_case(mvb, op, "plain", b, fin, fout, True, "auto", expect_fused=fused)


def _tc_boundary_cases():
    """N = 768 (6 tiles of 128) with 16-wide planes: the nnz at which one CTA stops holding the mesh and at which the
    second lo plane stops fitting (csrc/mvb_mesh_tc.cu mesh_tc_layout), and one entry past each"""
    n, k = 768, 6
    out = []
    for which in (0, 1):                    # 0: one CTA fits, 1: the second lo plane fits
        nnz = 0
        while C.mesh_tc_smem(n, n, nnz + 2, k, 16, 16, 1)[which]:
            nnz += 2
        assert nnz > n // 2
        out += [(n, nnz), (n, nnz + 2)]
    return out


@pytest.mark.parametrize("n,nnz", _tc_boundary_cases())
@pytest.mark.parametrize("mode,b", [("mesh_tc=1,1", 8), ("mesh_tc=1,2", 8), ("mesh_tc=1,0", 120)])
def test_cheb_layer_shared_memory_boundaries(mvb, n, nnz, mode, b):
    op = C.irregular_nnz(n, nnz, seed=nnz)
    mvb._lib.tune(mode)
    try:
        _run_layer_case(mvb, op, "plain", b, 16, 16, True, mode)
    finally:
        _reset(mvb)


# ---------------------------------------------------------------------------------------------
# mvb_cheb_stream_fwd / _bwd (the row-streaming layer of level 0)
# ---------------------------------------------------------------------------------------------
STREAM_OPS = {
    "directed0": (lambda: C.directed(0, seed=8, both=False), "none"),
    "directed0w": (lambda: C.directed(0, seed=9, both=True), "none"),
    "relabelled0": (lambda: C.relabelled(0, seed=10), "none"),
    "dense": (lambda: C.irregular(4998, seed=11, deg=(40, 48)), "all"),
    "hubband": (lambda: C.irregular(4998, seed=12, deg=(4, 8), hub_rows=np.arange(5, 1600, 400), hub_deg=(4200, 4400)),
                "some"),
}
# (operator, kind, B, meshes per slab, K): the streaming kernel takes K <= 8
STREAM_CASES = [("directed0", "dec", 64, 16, 6), ("directed0w", "plain", 64, 8, 6), ("relabelled0", "dec", 64, 8, 6),
                ("dense", "plain", 64, 8, 6), ("dense", "dec", 64, 16, 6), ("hubband", "plain", 64, 8, 6),
                ("hubband", "dec", 64, 16, 6),
                ("directed0", "dec", 64, 16, 1), ("relabelled0", "plain", 64, 8, 2), ("hubband", "dec", 64, 16, 3),
                ("dense", "plain", 64, 8, 8), ("relabelled0", "dec", 64, 16, 8)]


def _run_stream_case(mvb, op, kind, b, sw, overflow=None, k=6):
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    if overflow is not None:
        bands = C.stream_bands(op, b, sw, sms)
        assert bands is not None
        over = bands > C.ST_ECAP
        assert {"none": not over.any(), "all": over.all(), "some": over.any() and not over.all()}[overflow], bands
    u = C.upsample(op.n_rows, 1250, seed=b + sw, max_per_row=3) if kind == "dec" else None
    lo = _l_op(mvb, op)
    uo = _p_op(mvb, u) if u is not None else None
    n_in = u.n_cols if u is not None else op.n_rows
    x, w, bias, rng = _inputs(sw + b + (0 if k == 6 else 100 * k), n_in, b, 16, 16, k)
    Fn = mvb.functional
    mvb._lib.tune(f"stream_tc=1,{sw}")
    try:
        assert Fn.cheb_stream_supported(op.n_rows, b, 16, 16, k, lo, uo, None)
        c0 = mvb._lib.lib.mvb_launch_count()
        _check_layer("mvb_cheb_stream", lambda a, b_, c: Fn.cheb_layer(a, b_, c, lo, uo, None, relu=True), op, x, w, bias,
                     True, u=u, rng=rng)
        assert mvb._lib.lib.mvb_launch_count() - c0 >= 2
    finally:
        _reset(mvb)


@pytest.mark.parametrize("case,kind,b,sw,k", STREAM_CASES, ids=_k_ids(STREAM_CASES))
def test_cheb_stream(mvb, case, kind, b, sw, k):
    mk, overflow = STREAM_OPS[case]
    _run_stream_case(mvb, mk(), kind, b, sw, overflow, k=k)


def test_cheb_stream_smallest_and_ragged(mvb):
    """the smallest N at 16 meshes that mvb_cheb_stream_supported accepts, and N + 1 (a ragged last row block)"""
    b = 16
    mvb._lib.tune("stream_tc=1,8")
    try:
        sup = lambda n: bool(mvb._lib.lib.mvb_cheb_stream_supported(n, b, 16, 16, 6, n, 0, n))      # noqa: E731
        lo, hi = 1, 4998
        assert sup(hi) and not sup(lo)
        while hi - lo > 1:
            mid = (lo + hi) // 2
            lo, hi = (lo, mid) if sup(mid) else (mid, hi)
    finally:
        _reset(mvb)
    for n in (hi, hi + 1):
        _run_stream_case(mvb, C.irregular(n, seed=n, hubs=2, hub_deg=(300, 600), isolated=5, dups=20, loops=5), "plain", b, 8)


# ---------------------------------------------------------------------------------------------
# run-to-run determinism on irregular operators
# ---------------------------------------------------------------------------------------------
# one other order per path: K = 9 and 16 reduce dW of the mesh kernels in several plane groups
DET_CASES = [("conv_adjoint", 6), ("conv_basis", 6), ("layer", 6), ("layer_ffma", 6), ("stream", 6),
             ("conv_adjoint", 2), ("conv_basis", 8), ("layer", 9), ("layer_ffma", 3), ("stream", 8), ("layer", 16)]


@pytest.mark.parametrize("path,k", DET_CASES, ids=_k_ids(DET_CASES))
def test_bit_identical_run_to_run(mvb, path, k):
    op = C.irregular(4998, seed=13, hubs=4, hub_deg=(900, 1000), isolated=20, dups=50, loops=20) if path == "stream" \
        else SQUARE["irregular300"]()
    lo = _l_op(mvb, op)
    fout = 32 if path == "conv_basis" else 16
    b = 64 if path == "stream" else 8
    x, w, bias, rng = _inputs(17, op.n_rows, b, 16, fout, k)
    dy = _dev(rng.standard_normal((op.n_rows, b, fout)))
    Fn = mvb.functional
    if path == "stream":
        mvb._lib.tune("stream_tc=1,16")
    elif path == "layer_ffma":
        mvb._lib.tune("mesh_tc=0,0")
    try:
        outs = []
        for _ in range(3):
            xg, wg, bg = _dev(x, True), _dev(w, True), _dev(bias, True)
            if path.startswith("conv"):
                y = Fn.cheb_conv(xg, wg, bg, lo, True)
            else:
                assert Fn.cheb_layer_supported(op.n_rows, b, 16, fout, k, lo, None, None)
                y = Fn.cheb_layer(xg, wg, bg, lo, None, None, relu=True)
            y.backward(dy)
            outs.append((y.detach(), xg.grad, wg.grad, bg.grad))
    finally:
        _reset(mvb)
    for o in outs[1:]:
        assert all(torch.equal(a, b_) for a, b_ in zip(outs[0], o))
