"""The Chebyshev convolution at the polygon orders and filter widths a config can ask for, against float64 references.

The reference reads `polygon_order` and `num_conv_filters` from the user's config, one entry per level, and cheb_VAE /
cheb_GCN hand them straight to the kernels, which pick their implementation by K and by plane width:

  * step path (mvb_cheb_fwd / _bwd): the tcgen05 row GEMM tc_rowgemm_kernel<W, K> (4-wide planes: K <= 8, packed into one
    16- or 32-column tile; 16-wide: K <= 6; 32-wide: K <= 3; any output width up to 256, padded to 16), the weight-gradient
    reduction tc_wgrad_kernel<K, W/4> (K*W + 1 <= 128 feature rows, output width <= 32), the FFMA kernels beyond those,
    and the closed-form rows of an operator with an isolated tail (weights folded as W0 - W2 + W4 - ...), in the adjoint
    form of the backward (dx wanted, Fout <= 1.2 Fin) and the basis form (Fout > 1.2 Fin, or no dx);
  * row selection (mvb_cheb_sel_*): the planar layouts only, else the model composes conv + pool;
  * whole models against the oracle run in float64.

The mesh-resident layers, the streaming layer and the determinism checks take K as one more column of their case tables
in tests/test_gpu_operators.py.  Gates as there: rel_err < 1e-4 and elem_err <= 1 against tests/operator_cases.py's
float64 reference, the ReLU mask taken from the device."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import mesh_vae_oracle as O
from tests import operator_cases as C
from tests.helpers import OPERATORS_NPZ, rel_err, seeded_state_dict
from tests.test_gpu_operators import MAX_ERR, _check_layer, _dev, _inputs, _l_op, _p_op, _reset

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-4
GTOL = 1e-3       # whole-model gradients: see test_cheb_vae_matches_oracle_at_other_shapes (test_gpu_heads_shapes.py)


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    yield meshvae_b200
    print("\nlargest rel_err per entry point: " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(MAX_ERR.items())))


def _rows_op(n_active):
    """an operator whose active prefix is n_active rows (B = 1: the tensor-core thresholds are on rows = n_active * B),
    followed by 9 closed-form rows"""
    return C.irregular(n_active + 9, seed=n_active, n_active=n_active, isolated=3, dups=4, loops=2)


STEP_OPS = {"tail300": lambda: C.irregular(300, seed=5, n_active=241, dups=10, loops=5, isolated=4),
            **{f"rows{n}": (lambda n=n: _rows_op(n)) for n in (127, 129, 255, 257)}}

# (operator, tensor cores, Fin, Fout, K, B, dx wanted).  241 active rows x B = 2: 482 rows, over both tensor-core
# thresholds (row GEMM: 128 rows, weight gradient: 256 rows), + 59 x 2 closed-form rows
STEP_CASES = []
for _k in range(1, 9):
    # 4-wide planes (the padded 3-channel input, and 4 -> 4): tc_rowgemm<4, K>, tc_wgrad<K, 1> in both forms,
    # the adjoint-form dx contraction tc_rowgemm<4, K>, fold_rows_* for the closed-form rows
    STEP_CASES += [("tail300", 1, 4, 4, _k, 2, True), ("tail300", 1, 3, 16, _k, 2, False)]
for _k in range(1, 7):
    # 16-wide planes: tc_rowgemm<16, K>, tc_wgrad<K, 4> (adjoint: K*16 rows of S; basis: K*16 + 1 with the bias row)
    STEP_CASES += [("tail300", 1, 16, 16, _k, 2, True), ("tail300", 1, 16, 32, _k, 2, True)]
for _k in range(1, 4):
    # 32-wide planes: tc_rowgemm<32, K>, tc_wgrad<K, 8>
    STEP_CASES += [("tail300", 1, 32, 32, _k, 2, True), ("tail300", 1, 32, 16, _k, 2, False)]
# beyond the planar layouts: FFMA contraction and reduction (32 -> 32 at K = 8: the register tiles' limit, 512)
STEP_CASES += [("tail300", 1, 16, 16, 7, 2, True), ("tail300", 1, 16, 16, 8, 2, True), ("tail300", 1, 16, 32, 8, 2, False),
               ("tail300", 1, 32, 32, 4, 2, True), ("tail300", 1, 32, 32, 8, 2, True)]
# output widths other than 16 / 32: padded tensor-core output tiles (4, 8, 12: adjoint form; 20, 24, 28: basis form)
for _fo, _k in ((4, 3), (8, 5), (12, 6), (20, 2), (24, 4), (28, 6)):
    STEP_CASES += [("tail300", 1, 16, _fo, _k, 2, True)]
STEP_CASES += [("tail300", 1, 16, 12, 4, 2, False), ("tail300", 1, 32, 4, 2, 2, False)]
# the FFMA kernels alone (mvb_set_tensor_cores(0))
STEP_CASES += [("tail300", 0, 4, 4, 2, 2, True), ("tail300", 0, 4, 4, 8, 2, True), ("tail300", 0, 3, 16, 5, 2, False),
               ("tail300", 0, 16, 16, 1, 2, True), ("tail300", 0, 16, 16, 8, 2, True), ("tail300", 0, 16, 28, 5, 2, True),
               ("tail300", 0, 32, 32, 2, 2, True), ("tail300", 0, 16, 12, 6, 2, True)]
# row counts on either side of the tensor-core thresholds, and 13 full 128-row tiles + a ragged one (241 x 7 = 1687)
for _n in (127, 129, 255, 257):
    STEP_CASES += [(f"rows{_n}", 1, 16, 16, 3, 1, True), (f"rows{_n}", 1, 4, 16, 8, 1, False)]
STEP_CASES += [("tail300", 1, 16, 16, 4, 7, True), ("tail300", 1, 3, 16, 7, 7, False), ("tail300", 1, 4, 32, 2, 7, True)]


def _step_id(c):
    op, tc, fin, fout, k, b, dx = c
    return f"{op}-tc{tc}-{fin}to{fout}-K{k}-B{b}-{'dx' if dx else 'nodx'}"


@pytest.mark.parametrize("case,tc,fin,fout,k,b,need_dx", STEP_CASES, ids=[_step_id(c) for c in STEP_CASES])
def test_cheb_conv_orders_and_widths(mvb, case, tc, fin, fout, k, b, need_dx):
    op = STEP_OPS[case]()
    lo = _l_op(mvb, op)
    assert lo.n_active < op.n_rows
    relu = (fin + fout + k) % 2 == 0
    x, w, bias, rng = _inputs(fin * 1000 + fout * 10 + k, op.n_rows, b, fin, fout, k)
    mvb._lib.lib.mvb_set_tensor_cores(tc)
    try:
        _check_layer("mvb_cheb", lambda a, b_, c: mvb.functional.cheb_conv(a, b_, c, lo, relu), op, x, w, bias, relu,
                     need_dx=need_dx, rng=rng)
    finally:
        _reset(mvb)


def test_step_cases_take_both_backward_forms(mvb):
    """the grid above runs each K of the planar layouts in the adjoint and in the basis form of the backward"""
    uses_basis = mvb._lib.lib.mvb_cheb_bwd_uses_basis
    forms = {}
    for _, tc, fin, fout, k, _, dx in STEP_CASES:
        if tc:
            forms.setdefault(((fin + 3) // 4 * 4, k), set()).add(uses_basis((fin + 3) // 4 * 4, (fout + 3) // 4 * 4, int(dx)))
    for fin, kmax in ((4, 8), (16, 6), (32, 3)):
        for k in range(1, kmax + 1):
            assert forms[(fin, k)] == {0, 1}, (fin, k)


# ---------------------------------------------------------------------------------------------
# row selection (mvb_cheb_sel_*): the planar layouts of tc_rowgemm / tc_wgrad, and one step past each limit
# ---------------------------------------------------------------------------------------------
SEL_FOUT = (4, 8, 20, 32)
SEL_CASES = ([(3 if k % 3 == 0 else 4, SEL_FOUT[k % 4], k) for k in range(1, 9)] +
             [(16, SEL_FOUT[k % 4], k) for k in range(1, 7)] + [(32, SEL_FOUT[k % 4], k) for k in range(1, 4)])
SEL_PAST = [(4, 16, 9), (16, 16, 7), (32, 16, 4)]


@pytest.mark.parametrize("fin,fout,k", SEL_CASES + SEL_PAST,
                         ids=[f"{fi}to{fo}-K{k}" for fi, fo, k in SEL_CASES + SEL_PAST])
def test_cheb_conv_sel_orders(mvb, fin, fout, k):
    op = C.irregular(300, seed=21, hubs=2, hub_deg=(100, 200), isolated=5, dups=10, loops=4)
    d = C.selection(op.n_rows, 75, seed=k)
    lo, do = _l_op(mvb, op), _p_op(mvb, d)
    b = 4                                                   # 75 kept rows x 4 meshes = 300 rows >= 256
    x, w, bias, rng = _inputs(fin * 100 + k, op.n_rows, b, fin, fout, k)
    Fn = mvb.functional
    fused = Fn.cheb_conv_sel_supported(_dev(x), _dev(w), lo, do)
    assert fused == ((fin, fout, k) not in SEL_PAST)
    finp = (fin + 3) // 4 * 4
    assert bool(mvb._lib.lib.mvb_cheb_sel_supported(op.n_rows, b, finp, fout, k, d.n_rows)) == fused

    def run(a, b_, c):
        if fused:
            return Fn.cheb_conv_sel(a, b_, c, lo, do, relu=True)
        return Fn.pool(Fn.cheb_conv(a, b_, c, lo, True), do)         # what cheb_VAE._layer composes then
    _check_layer("mvb_cheb_sel" if fused else "composition", run, op, x, w, bias, True, d=d, need_dx=False, rng=rng)


# ---------------------------------------------------------------------------------------------
# whole models against the oracle in float64, on the same seeded weights
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ops():
    return O.load_operators(OPERATORS_NPZ)


def _config(**kw):
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    cfg["dropout"] = 0.0
    cfg.update(kw)
    return cfg


def _vae_batch(b, n, classes, z, seed):
    """x [B,N,3], labels over `classes` (every class present), reparameterisation noise [B,z]"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, n, 3, generator=g)
    y = torch.arange(b)[torch.randperm(b, generator=g)] % classes
    return x, y, torch.randn(b, z, generator=g)


def _vae_pair(mvb, ops, cfg, seed=7):
    A, D, U, nn_ = ops
    ref = O.OracleChebVAE(3, cfg, D, U, A, nn_)
    ref.load_state_dict(seeded_state_dict(ref, seed))
    ref.double()
    net = mvb.cheb_VAE(3, copy.deepcopy(cfg), [d.to(DEV) for d in D], [u.to(DEV) for u in U], [a.to(DEV) for a in A], nn_,
                       model=cfg["model"])
    net.load_state_dict(seeded_state_dict(net, seed))
    return ref, net.to(DEV)


def _vae_forward(ref, net, cfg, nn0, batch, seed):
    x, y, eps = _vae_batch(batch, nn0, cfg["num_classes"], cfg["num_style"], seed)
    y_hot = F.one_hot(y, cfg["num_classes"])
    ref.train(); net.train()
    outs_ref = ref(x.double(), x.double(), y_hot.double(), m_type="train", eps=eps.double())
    outs_net = net(x.cuda(), x.double().cuda(), y_hot.cuda(), m_type="train", eps=eps.cuda())
    return outs_ref, outs_net


def _check_outputs(outs_ref, outs_net):
    lo, co, ro, (ko, reco, zo), yho = outs_ref
    lg, cg, rg, (kg, recg, zg), yhg = outs_net
    assert torch.isfinite(lg).all() and torch.isfinite(rg).all()
    assert int(cg) == int(co)
    for what, a, r in (("loss", lg, lo), ("recon", rg, ro), ("kld", kg, ko), ("rec", recg, reco), ("z", zg, zo),
                       ("y_hat", yhg, yho)):
        e = rel_err(a, r)
        MAX_ERR["cheb_VAE"] = max(MAX_ERR.get("cheb_VAE", 0.0), e)
        assert e < TOL, f"{what}: rel_err {e:.3e}"


def _check_grads(ref, net, entry):
    po = dict(ref.named_parameters())
    for name, p in net.named_parameters():
        if po[name].grad is None:
            assert p.grad is None, name
            continue
        e = rel_err(p.grad, po[name].grad)
        MAX_ERR[entry + " grad"] = max(MAX_ERR.get(entry + " grad", 0.0), e)
        assert e < GTOL, f"{name}: rel_err {e:.3e}"


VAE_CONFIGS = {
    # every layer at another K; the output layer (closed-form rows on the finest mesh) folds at K = 8
    "orders23458": dict(polygon_order=[2, 3, 4, 5, 8]),
    # a K = 1 level (encoder level 2 / decoder level 1) and K = 7 on the level-1 mesh kernel
    "orders87163": dict(polygon_order=[8, 7, 1, 6, 3]),
    # widths only the FFMA step path takes (24: not a power-of-two number of quads), 8-wide levels, three classes
    "widths8_24": dict(num_conv_filters=[8, 8, 24, 24, 24], num_classes=3, num_style=8),
}


@pytest.mark.parametrize("name", list(VAE_CONFIGS))
def test_cheb_vae_matches_oracle_at_other_orders_and_widths(mvb, ops, name):
    cfg = _config(**VAE_CONFIGS[name])
    ref, net = _vae_pair(mvb, ops, cfg)
    outs_ref, outs_net = _vae_forward(ref, net, cfg, ops[3][0], 16, 21)
    outs_ref[0].backward()
    outs_net[0].backward()
    _check_outputs(outs_ref, outs_net)
    _check_grads(ref, net, "cheb_VAE")


def test_cheb_vae_48_wide_layers_raise_in_backward(mvb, ops):
    """16, 32, 48, 48, 48: the 48-wide levels take the step path (no mesh kernel takes 12 quads), whose FFMA
    weight-gradient reduction holds at most 512 register tiles of 4 x 4 (include/mvb.h, mvb_cheb_bwd) - at K = 6 the
    decoder's 48 -> 32 layer needs 48 x 12 = 576 of them, its 48 -> 48 layers 72 x 12.  The forward pass is right; the
    backward pass raises MvbError before the reduction runs, never a wrong gradient."""
    cfg = _config(num_conv_filters=[16, 32, 48, 48, 48])
    ref, net = _vae_pair(mvb, ops, cfg)
    outs_ref, outs_net = _vae_forward(ref, net, cfg, ops[3][0], 16, 23)
    _check_outputs(outs_ref, outs_net)
    with pytest.raises(mvb._lib.MvbError, match="wgrad: K\\*Fin x Fout"):
        outs_net[0].backward()
    torch.cuda.synchronize()


@pytest.mark.parametrize("k", [3, 8])
def test_cheb_gcn_matches_oracle_at_other_orders(mvb, ops, k):
    A, D, U, nn_ = ops
    cfg = _config(polygon_order=[k] * 5)
    ref = O.OracleChebGCN(6, copy.deepcopy(cfg), D, U, A, nn_)
    ref.load_state_dict(seeded_state_dict(ref, 9))
    ref.double()
    net = mvb.cheb_GCN(6, copy.deepcopy(cfg), [d.to(DEV) for d in D], [u.to(DEV) for u in U], [a.to(DEV) for a in A], nn_)
    net.load_state_dict(seeded_state_dict(net, 9))
    net = net.to(DEV)
    g = torch.Generator().manual_seed(13 + k)
    x = torch.randn(4, nn_[0], 6, generator=g)
    y = torch.tensor([0, 1, 1, 0])
    lo = ref(x.double())
    F.cross_entropy(lo, y).backward()
    lg = net(x.cuda())
    F.cross_entropy(lg, y.cuda()).backward()
    e = rel_err(lg, lo)
    MAX_ERR["cheb_GCN"] = max(MAX_ERR.get("cheb_GCN", 0.0), e)
    assert e < TOL, f"logits: rel_err {e:.3e}"
    _check_grads(ref, net, "cheb_GCN")


def test_train_engine_captured_step_at_other_orders(mvb, ops):
    """the captured training step at polygon_order 2, 3, 4, 5, 8 is the same bits as the eager step: the workspaces
    that depend on K are sized right under capture"""
    from meshvae_b200.engine import TrainEngine
    A, D, U, nn_ = ops
    cfg = _config(polygon_order=[2, 3, 4, 5, 8], dropout=0.2)
    B = 16
    batches = [_vae_batch(B, nn_[0], 2, 16, 700 + s) for s in range(2)]
    finals, losses = [], []
    for use_graph in (True, False):
        net = mvb.cheb_VAE(3, copy.deepcopy(cfg), [d.to(DEV) for d in D], [u.to(DEV) for u in U], [a.to(DEV) for a in A], nn_)
        net.load_state_dict(seeded_state_dict(net, 11))
        net = net.to(DEV)
        eng = TrainEngine(net, B, lr=1e-3, weight_decay=5e-4, use_graph=use_graph)
        eng.capture(warmup=1)
        ls = [eng.step(x, x.double(), y, eps_host=eps) for x, y, eps in batches]
        assert all(np.isfinite(v) for v in ls), ls
        losses.append(ls)
        finals.append([p.detach().clone() for p in net.parameters()])
        del eng, net
    assert losses[0] == losses[1]
    for a, r in zip(*finals):
        assert torch.equal(a, r)
