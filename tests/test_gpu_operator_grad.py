"""The Chebyshev convolution differentiated with respect to its operator values (a `norm` that requires grad, e.g.
computed from learned edge weights), against the oracle's ChebConv_batch / cheb_norm and the PyG restatement run in
float64 autograd on the CPU.  Gates as in test_gpu_conv_orders.py: rel_err < 1e-4 and elem_err <= 1 per tensor,
whole-model gradients rel_err < 1e-3."""
import copy
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import mesh_vae_oracle as O
from tests import operator_cases as C
from tests.helpers import OPERATORS_NPZ, ROOT, elem_err, rel_err, seeded_state_dict

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-4
GTOL = 1e-3


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    return meshvae_b200


def _gate(what, dev, ref, tol=TOL):
    d, r = dev.detach().double().cpu(), ref.detach().double().cpu()
    assert tuple(d.shape) == tuple(r.shape), what
    e = rel_err(d, r)
    assert e < tol, f"{what}: rel_err {e:.3e}"
    ee = elem_err(d, r)
    assert ee <= 1.0, f"{what}: elem_err {ee:.3f}"


def _gate_grad(what, dev, ref):
    """a gradient; where the reference's graph never uses the tensor (K = 1) its gradient is None and ours all zero"""
    if ref is None:
        assert torch.count_nonzero(dev) == 0, what
    else:
        _gate(what, dev, ref)


def _coarse_on_fine():
    """the coarsest template operator on a 313-vertex tensor: n_active = 20 < N (models/cheb_VAE.py:288)"""
    op = C.template_L(4)
    return C.Op("coarse", 313, 313, op.rows, op.cols, op.vals)


OPS = {**{f"t{l}": (lambda l=l: C.template_L(l)) for l in range(5)},
       "relab1": lambda: C.relabelled(1, seed=3),
       "irr": lambda: C.irregular(300, seed=8, hubs=2, hub_deg=(60, 120), dups=12, loops=3, isolated=4),
       "dir2": lambda: C.directed(2, seed=2, both=True),
       "coarse": _coarse_on_fine}

# (operator, tensor cores, Fin, Fout, K, B, ReLU, bias, dx wanted)
CASES = [
    # the template's levels at the widths of the model's layers
    ("t0", 1, 16, 16, 6, 2, True, True, True), ("t0", 1, 3, 16, 6, 2, True, True, False),
    ("t1", 1, 16, 32, 6, 4, True, True, True), ("t2", 1, 32, 32, 3, 64, True, True, True),
    ("t3", 1, 16, 16, 6, 64, True, True, True), ("t4", 1, 16, 3, 6, 64, False, False, True),
    # K = 1 (d_norm all zero), 2, 3, 8
    ("t2", 1, 16, 16, 1, 2, True, True, True), ("t2", 1, 16, 16, 2, 2, False, True, True),
    ("t2", 1, 4, 4, 3, 64, True, False, True), ("t2", 1, 16, 16, 8, 1, True, True, False),
    ("t3", 1, 4, 4, 8, 2, False, True, True),
    # operators other than the template's: relabelled, hubs + duplicates + self loops, not symmetric, n_active < N
    ("relab1", 1, 16, 16, 6, 2, True, True, True), ("irr", 1, 16, 32, 6, 2, True, True, True),
    ("irr", 1, 16, 16, 8, 1, False, True, False), ("dir2", 1, 16, 16, 6, 2, True, True, True),
    ("dir2", 1, 32, 32, 2, 2, False, False, True), ("coarse", 1, 16, 3, 6, 2, False, False, True),
    ("coarse", 1, 16, 16, 3, 2, True, True, True),
    # the FFMA kernels alone
    ("t2", 0, 16, 16, 6, 2, True, True, True), ("irr", 0, 3, 16, 3, 2, True, True, False),
    ("dir2", 0, 16, 3, 8, 1, False, False, True),
]


def _id(c):
    op, tc, fin, fout, k, b, relu, bias, dx = c
    return f"{op}-tc{tc}-{fin}to{fout}-K{k}-B{b}{'-relu' if relu else ''}{'-bias' if bias else ''}{'-dx' if dx else ''}"


def _inputs(seed, n, b, fin, fout, k, bias):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, b, fin, generator=g, dtype=torch.float64)
    w = torch.randn(k, fin, fout, generator=g, dtype=torch.float64) * 0.1
    bb = torch.randn(fout, generator=g, dtype=torch.float64) * 0.1 if bias else None
    return x, w, bb, g


def _device_layer(mvb, ei, norm, x, w, bb, relu, need_dx, n):
    """the layer through functional.cheb_conv on the cached pattern, norm a leaf that requires grad"""
    leaves = [x.float().to(DEV).requires_grad_(need_dx), w.float().to(DEV).requires_grad_(True),
              None if bb is None else bb.float().to(DEV).requires_grad_(True), norm.float().to(DEV).requires_grad_(True)]
    pat = mvb.operators.pattern_from_edges(ei.to(DEV), n, DEV)
    y = mvb.functional.cheb_conv(leaves[0], leaves[1], leaves[2], pat, relu, norm=leaves[3])
    return y, leaves


@pytest.mark.parametrize("case,tc,fin,fout,k,b,relu,bias,need_dx", CASES, ids=[_id(c) for c in CASES])
def test_operator_gradient(mvb, case, tc, fin, fout, k, b, relu, bias, need_dx):
    op = OPS[case]()
    ei, norm = op.edges()
    x, w, bb, g = _inputs(fin * 1000 + fout * 10 + k, op.n_rows, b, fin, fout, k, bias)
    mvb._lib.lib.mvb_set_tensor_cores(tc)
    try:
        y, (xg, wg, bg, ng) = _device_layer(mvb, ei, norm, x, w, bb, relu, need_dx, op.n_rows)
        gy = torch.randn(y.shape, generator=g, dtype=torch.float64)
        y.backward(gy.float().to(DEV))
        torch.cuda.synchronize()
    finally:
        mvb._lib.lib.mvb_set_tensor_cores(1)
    # float64 reference: the oracle's ChebConv_batch on [B, N, F], the ReLU mask taken from the device output
    xr, wr, nr = x.clone().requires_grad_(True), w.clone().requires_grad_(True), norm.double().requires_grad_(True)
    br = None if bb is None else bb.clone().requires_grad_(True)
    pre = O.cheb_conv_batch(xr.transpose(0, 1), ei, nr, wr, br).transpose(0, 1)
    mask = (y.detach().cpu() > 0).double() if relu else torch.ones_like(pre)
    if relu:
        flips = mask != (pre.detach() > 0).double()
        assert bool((pre.detach()[flips.bool()].abs() <= 1e-5 * pre.detach().abs().max()).all())
    (pre * mask * gy).sum().backward()
    _gate("y", y, pre * mask)
    _gate_grad("d_norm", ng.grad, nr.grad)
    _gate("dW", wg.grad, wr.grad)
    if need_dx:
        _gate("dx", xg.grad, xr.grad)
    else:
        assert xg.grad is None
    if bias:
        _gate("db", bg.grad, br.grad)
    if k == 1:
        assert nr.grad is None and torch.count_nonzero(ng.grad) == 0


@pytest.mark.parametrize("case,fin,fout,need_dx", [("t1", 16, 32, True), ("irr", 3, 16, False), ("t3", 16, 32, True),
                                                   ("coarse", 16, 32, False)])
def test_frozen_norm_gives_the_same_bits(mvb, case, fin, fout, need_dx):
    """where mvb_cheb_bwd takes the basis form, dx / dW / db of mvb_cheb_bwd_op are its bits"""
    finp = fin + (-fin) % 4
    assert mvb._lib.lib.mvb_cheb_bwd_uses_basis(finp, fout, int(need_dx)) == 1
    op = OPS[case]()
    ei, norm = op.edges()
    x, w, bb, g = _inputs(5, op.n_rows, 8, fin, fout, 6, True)
    gy = torch.randn(op.n_rows, 8, fout, generator=g).to(DEV)
    outs = []
    for learned in (False, True):
        xg = x.float().to(DEV).requires_grad_(need_dx)
        wg, bg = w.float().to(DEV).requires_grad_(True), bb.float().to(DEV).requires_grad_(True)
        if learned:
            ng = norm.to(DEV).requires_grad_(True)
            y = mvb.functional.cheb_conv(xg, wg, bg, mvb.operators.pattern_from_edges(ei.to(DEV), op.n_rows, DEV), True, norm=ng)
        else:
            y = mvb.functional.cheb_conv(xg, wg, bg, mvb.operators.from_edges(ei.to(DEV), norm.to(DEV), op.n_rows, DEV), True)
        y.backward(gy)
        outs.append((y.detach(), xg.grad, wg.grad, bg.grad))
    for a, r in zip(*outs):
        assert (a is None and r is None) or torch.equal(a, r)


def test_operator_gradient_is_deterministic(mvb):
    op = OPS["irr"]()
    ei, norm = op.edges()
    x, w, bb, g = _inputs(9, op.n_rows, 4, 16, 16, 6, True)
    grads = []
    for _ in range(2):
        y, (xg, wg, bg, ng) = _device_layer(mvb, ei, norm, x, w, bb, True, True, op.n_rows)
        y.backward(torch.ones_like(y))
        grads.append(ng.grad)
    assert torch.equal(grads[0], grads[1])


def _edge_weights(idx, seed, dtype=torch.float32, device=DEV):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(idx.shape[1], generator=g, dtype=torch.float64) * 1.5 + 0.25).to(device=device, dtype=dtype)


def test_learned_edge_weights_through_cheb_conv_batch(mvb):
    A, _, _, nn_ = O.load_operators(OPERATORS_NPZ)
    idx, n = A[2]._indices(), nn_[2]
    w0 = _edge_weights(idx, 1)
    conv = mvb.ChebConv_batch(16, 16, 6).to(DEV)
    ref = O.OracleChebVAE._Conv(16, 16, 6).double()
    with torch.no_grad():
        ref.weight.copy_(conv.weight.double().cpu())
        ref.bias.copy_(conv.bias.double().cpu())
    x = torch.randn(3, n, 16, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    wd = w0.clone().requires_grad_(True)
    ei_d = mvb.ChebConv_batch.norm(idx.to(DEV), n)[0]
    norm_d = mvb.ChebConv_batch.norm(idx.to(DEV), n, wd)[1]
    y = conv(x.float().to(DEV), ei_d, norm_d)
    (y.double().cpu() ** 2).sum().backward()
    wr = w0.double().cpu().requires_grad_(True)
    ei_r, norm_r = O.cheb_norm(idx, n, wr)
    yr = ref(x, ei_r, norm_r)
    (yr ** 2).sum().backward()
    _gate("y", y, yr)
    _gate("w.grad", wd.grad, wr.grad)
    _gate("dW", conv.weight.grad, ref.weight.grad)


def _pyg_shim_chebconv():
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


@pytest.mark.parametrize("k", [1, 3, 6])
def test_learned_edge_weights_through_pyg_chebconv(mvb, k):
    A, _, _, nn_ = O.load_operators(OPERATORS_NPZ)
    idx, n = A[1]._indices(), nn_[1]
    loops = torch.arange(0, n, 97)                       # self loops with their own weights: dropped by both
    idx = torch.cat((idx, torch.stack((loops, loops))), 1)
    w0 = _edge_weights(idx, 3)
    conv = mvb.ChebConv(16, 32, k).to(DEV)
    ref = _pyg_shim_chebconv()(16, 32, k).double()
    ref.load_state_dict({kk: v.double().cpu() for kk, v in conv.state_dict().items()})
    x = torch.randn(2, n, 16, generator=torch.Generator().manual_seed(k), dtype=torch.float64)
    wd = w0.clone().requires_grad_(True)
    y = conv(x.float().to(DEV), idx.to(DEV), edge_weight=wd)
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(7), dtype=torch.float64)
    (y.double().cpu() * gy).sum().backward()
    wr = w0.double().cpu().requires_grad_(True)
    yr = ref(x, idx, edge_weight=wr)
    (yr * gy).sum().backward()
    _gate("y", y, yr)
    _gate_grad("w.grad", wd.grad, wr.grad)
    # a frozen weight tensor takes the same path without a gradient (the degree sums are CUDA scatter-adds, whose
    # order is not fixed: the same values to rounding, not the same bits)
    with torch.no_grad():
        y2 = conv(x.float().to(DEV), idx.to(DEV), edge_weight=w0)
    assert not y2.requires_grad
    _gate("y, frozen weights", y2, yr)


def test_fresh_and_updated_norms_neither_sync_nor_grow_the_caches(mvb):
    A, _, _, nn_ = O.load_operators(OPERATORS_NPZ)
    idx, n = A[2]._indices().to(DEV), nn_[2]
    ei, base = mvb.ChebConv_batch.norm(idx, n)
    conv = mvb.ChebConv_batch(16, 16, 6).to(DEV)
    x = torch.randn(4, n, 16, device=DEV)
    leaf = base.clone().requires_grad_(True)
    conv(x, ei, leaf).sum().backward()                   # builds the pattern once
    sizes = (len(mvb.operators._CACHE), len(mvb.operators._PATTERNS))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")               # a host synchronisation in the loop raises
    try:
        _fresh_and_updated(conv, x, ei, base, leaf)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert (len(mvb.operators._CACHE), len(mvb.operators._PATTERNS)) == sizes


def _fresh_and_updated(conv, x, ei, base, leaf):
    for i in range(50):
        if i % 2:
            with torch.no_grad():
                leaf.mul_(1.001)                          # in place: a new _version of the same storage
            conv(x, ei, leaf).sum().backward()
        else:
            fresh = (base * (1.0 + 0.01 * i)).requires_grad_(True)     # a new tensor every call
            conv(x, ei, fresh).sum().backward()
            assert fresh.grad is not None


def test_learned_norm_layer_in_a_cuda_graph(mvb):
    op = C.template_L(2)
    ei, norm0 = op.edges()
    ei = ei.to(DEV)
    conv = mvb.ChebConv_batch(16, 16, 6).to(DEV)
    conv.fuse_relu = True
    x = torch.randn(2, op.n_rows, 16, device=DEV)
    gy = torch.randn(2, op.n_rows, 16, device=DEV)
    leaf = norm0.to(DEV).requires_grad_(True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):                                # warm-up: pattern, side stream, allocator
            conv(x, ei, leaf).mul(gy).sum().backward()
    torch.cuda.current_stream().wait_stream(s)
    leaf.grad = None
    conv.weight.grad = conv.bias.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y = conv(x, ei, leaf)
        y.mul(gy).sum().backward()
    ref = O.OracleChebVAE._Conv(16, 16, 6).double()
    with torch.no_grad():
        ref.weight.copy_(conv.weight.double().cpu())
        ref.bias.copy_(conv.bias.double().cpu())
    g = torch.Generator().manual_seed(4)
    for step in range(3):
        new = norm0 * (1.0 + 0.2 * torch.rand(norm0.shape, generator=g))
        with torch.no_grad():
            leaf.copy_(new.to(DEV))
        graph.replay()
        torch.cuda.synchronize()
        nr = new.double().requires_grad_(True)
        yr = F.relu(ref(x.double().cpu(), ei.cpu(), nr))
        (yr * gy.double().cpu()).sum().backward()
        _gate(f"y replay {step}", y, yr)
        _gate(f"d_norm replay {step}", leaf.grad, nr.grad)


def test_cheb_vae_learned_edge_weights_match_oracle(mvb):
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    cfg["dropout"] = 0.0
    ref = O.OracleChebVAE(3, cfg, D, U, A, nn_)
    ref.load_state_dict(seeded_state_dict(ref, 7))
    ref.double()
    net = mvb.cheb_VAE(3, copy.deepcopy(cfg), [d.to(DEV) for d in D], [u.to(DEV) for u in U], [a.to(DEV) for a in A], nn_,
                       model=cfg["model"])
    net.load_state_dict(seeded_state_dict(net, 7))
    net = net.to(DEV)
    w_net = [_edge_weights(A[i]._indices(), 10 + i).requires_grad_(True) for i in range(len(nn_))]
    w_ref = [w.detach().double().cpu().requires_grad_(True) for w in w_net]
    net.A_norm = tuple(mvb.ChebConv_batch.norm(A[i]._indices().to(DEV), nn_[i], w_net[i])[1] for i in range(len(nn_)))
    ref.A_norm = tuple(O.cheb_norm(A[i]._indices(), nn_[i], w_ref[i])[1] for i in range(len(nn_)))
    b = 2
    g = torch.Generator().manual_seed(31)
    x = torch.randn(b, nn_[0], 3, generator=g)
    y_hot = F.one_hot(torch.tensor([0, 1]), cfg["num_classes"])
    eps = torch.randn(b, cfg["num_style"], generator=g)
    ref.train(); net.train()
    lr = ref(x.double(), x.double(), y_hot.double(), m_type="train", eps=eps.double())[0]
    ln = net(x.cuda(), x.double().cuda(), y_hot.cuda(), m_type="train", eps=eps.cuda())[0]
    lr.backward()
    ln.backward()
    assert rel_err(ln, lr) < TOL
    for i in range(len(nn_)):
        e = rel_err(w_net[i].grad, w_ref[i].grad)
        assert e < GTOL, f"edge weights of level {i}: rel_err {e:.3e}"
    po = dict(ref.named_parameters())
    for name, p in net.named_parameters():
        if po[name].grad is not None:
            e = rel_err(p.grad, po[name].grad)
            assert e < GTOL, f"{name}: rel_err {e:.3e}"
