"""GPU parity of the mesh-resident fused coarse-level layers (mvb_cheb_layer_fwd/bwd through the C
ABI; models/cheb_VAE.py:264-265, 284-285) against (1) the CPU oracle's SurfacePool / ChebConv_batch
composition on the same seeded inputs and (2) the step-by-step CUDA path (pool + cheb_conv + pool).
fp32 tolerance 1e-4 relative (max|a-b| / max|b| per tensor); measured <= 3e-6."""
import pytest
import torch

from tests.helpers import OPERATORS_NPZ, rel_err, elem_err
from oracle import mesh_vae_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    return meshvae_b200


@pytest.fixture(scope="module")
def ops():
    return O.load_operators(OPERATORS_NPZ)


def _rand(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


# (kind, level of the conv, batch, Fin, Fout, relu, bias)
CASES = [("enc", 2, 64, 16, 16, True, True), ("enc", 3, 64, 16, 32, True, True), ("dec", 3, 64, 32, 32, True, True),
         ("dec", 2, 64, 32, 16, True, True), ("plain", 2, 5, 16, 16, False, True), ("plain", 3, 1, 32, 8, True, False),
         ("enc", 2, 3, 8, 16, True, True), ("dec", 2, 100, 16, 32, False, True), ("plain", 4, 7, 32, 32, True, True),
         # level 1 (1250 vertices): only the tensor-core mesh kernels (a 2-CTA cluster per mesh) hold it
         ("enc", 1, 64, 16, 16, True, True), ("dec", 1, 64, 16, 16, True, True), ("plain", 1, 3, 16, 16, False, False),
         ("dec", 1, 9, 16, 32, True, True), ("enc", 1, 160, 32, 16, True, True)]
# implementation behind mvb_cheb_layer_*: tensor-core mesh kernels with the automatic cluster size, forced to one /
# two CTAs per mesh, and the FFMA mesh kernels (mvb_tune "mesh_tc=enable,ctas")
MODES = ["mesh_tc=1,0", "mesh_tc=1,1", "mesh_tc=1,2", "mesh_tc=0,0"]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("kind,lvl,b,fin,fout,relu,bias", CASES)
def test_fused_layer_matches_oracle_and_stepwise(mvb, ops, kind, lvl, b, fin, fout, relu, bias, mode):
    mvb._lib.tune(mode)
    try:
        _fused_layer_case(mvb, ops, kind, lvl, b, fin, fout, relu, bias, mode)
    finally:
        mvb._lib.tune("mesh_tc=1,0")


def _fused_layer_case(mvb, ops, kind, lvl, b, fin, fout, relu, bias, mode):
    A, D, U, nn_ = ops
    Fn = mvb.functional
    n = nn_[lvl]
    K = 6
    ei, norm = O.cheb_norm(A[lvl]._indices(), n)
    up = U[lvl] if kind == "dec" else None            # U[lvl]: level lvl+1 -> lvl
    down = D[lvl] if kind == "enc" else None          # D[lvl]: level lvl -> lvl+1
    n_in = up.shape[1] if up is not None else n
    x = _rand(b, n_in, fin, seed=1)
    w = _rand(K, fin, fout, seed=2, scale=0.1)
    bs = _rand(fout, seed=3, scale=0.1) if bias else None
    # ---- fused kernel ----
    dev = torch.device("cuda:0")
    l_op = mvb.operators.from_edges(ei.to(dev), norm.to(dev), n, dev)
    u_op = None if up is None else mvb.operators.from_sparse(up.to(dev), dev)
    d_op = None if down is None else mvb.operators.from_sparse(down.to(dev), dev)
    if not Fn.cheb_layer_supported(n, b, fin, fout, K, l_op, u_op, d_op):
        # (level 1 fits shared memory only with 16-wide planes in both directions - the shapes the models have there)
        assert mode != "mesh_tc=1,0" or (lvl == 1 and (fin, fout) != (16, 16)), "the automatic mode must cover this case"
        pytest.skip(f"{mode} does not cover this shape")
    xg = Fn.to_vertex_major(x.to(dev)).clone().requires_grad_()
    wg = w.to(dev).requires_grad_()
    bg = bs.to(dev).requires_grad_() if bias else None
    c0 = mvb._lib.lib.mvb_launch_count()
    yg = Fn.cheb_layer(xg, wg, bg, l_op, u_op, d_op, relu=relu)
    assert mvb._lib.lib.mvb_launch_count() - c0 == 1, "the fused layer must be ONE launch"
    # ---- oracle (CPU): the reference's module composition, with the ReLU mask the device produced (a pre-activation
    # within rounding error of 0 may land on either side; such a flip moves dW by a whole row's contribution) ----
    xr, wr = x.clone().requires_grad_(), w.clone().requires_grad_()
    br = bs.clone().requires_grad_() if bias else None
    h = O.surface_pool(xr, up._indices(), up._values(), up.shape) if up is not None else xr
    h = O.cheb_conv_batch(h, ei, norm, wr, br)
    if relu:
        mask = torch.ones_like(h)
        ydev = Fn.from_vertex_major(yg).detach().cpu()
        if down is not None:
            di = down._indices()
            rows = torch.empty(down.shape[0], dtype=torch.long)
            rows[di[0]] = di[1]                      # output row r of the pooled tensor is conv row rows[r]
        else:
            rows = torch.arange(n)
        mask[:, rows] = (ydev > 0).float()
        flips = int(((h.detach()[:, rows] > 0).float() != mask[:, rows]).sum())
        assert flips <= 4, f"{flips} ReLU decisions differ from the oracle"
        h = h * mask
    yr = O.surface_pool(h, down._indices(), down._values(), down.shape) if down is not None else h
    gy = _rand(*yr.shape, seed=4)
    yr.backward(gy)
    yg.backward(Fn.to_vertex_major(gy.to(dev)).contiguous())
    assert rel_err(Fn.from_vertex_major(yg), yr) < TOL
    assert rel_err(Fn.from_vertex_major(xg.grad), xr.grad) < TOL
    assert rel_err(wg.grad, wr.grad) < TOL
    if bias:
        assert rel_err(bg.grad, br.grad) < TOL
    # per-element gate: rtol 1e-4 with an absolute floor of 1e-4 of the tensor's RMS
    assert elem_err(Fn.from_vertex_major(yg), yr) <= 1.0
    assert elem_err(Fn.from_vertex_major(xg.grad), xr.grad) <= 1.0
    assert elem_err(wg.grad, wr.grad) <= 1.0
    if bias:
        assert elem_err(bg.grad, br.grad) <= 1.0
    # ---- step-by-step CUDA path on the same inputs ----
    xs = xg.detach().clone().requires_grad_()
    ws = wg.detach().clone().requires_grad_()
    bsg = bg.detach().clone().requires_grad_() if bias else None
    h = Fn.pool(xs, u_op) if u_op is not None else xs
    h = Fn.cheb_conv(h, ws, bsg, l_op, relu)
    ys = Fn.pool(h, d_op) if d_op is not None else h
    ys.backward(Fn.to_vertex_major(gy.to(dev)).contiguous())
    assert rel_err(yg, ys) < TOL and rel_err(xg.grad, xs.grad) < TOL and rel_err(wg.grad, ws.grad) < TOL


# level 0 (4998 vertices): the row-streaming fused layer (mvb_cheb_stream_*, csrc/mvb_stream_tc.cu) - one persistent launch
# per direction behind the same cheb_layer call.  64 meshes = the benchmark shape; 24 / 20 meshes: fewer slabs, a ragged last
# row block; plain = no up-sampling prologue.  sw = meshes per slab (8 / 16; mvb_tune
# stream_tc=1,sw; 0 = automatic)
STREAM_CASES = [("dec", 0, 64, 16, 16, True, True, 8), ("dec", 0, 64, 16, 16, True, True, 16), ("dec", 0, 24, 16, 16, True, False, 8),
                ("plain", 0, 40, 16, 16, False, True, 0), ("plain", 0, 64, 16, 16, True, True, 0)]


@pytest.mark.parametrize("kind,lvl,b,fin,fout,relu,bias,sw", STREAM_CASES)
def test_stream_layer_matches_oracle_and_stepwise(mvb, ops, kind, lvl, b, fin, fout, relu, bias, sw):
    A, D, U, nn_ = ops
    dev = torch.device("cuda:0")
    ei, norm = O.cheb_norm(A[lvl]._indices(), nn_[lvl])
    l_op = mvb.operators.from_edges(ei.to(dev), norm.to(dev), nn_[lvl], dev)
    u_op = mvb.operators.from_sparse(U[lvl].to(dev), dev) if kind == "dec" else None
    mvb._lib.tune(f"stream_tc=1,{sw}")
    try:
        assert mvb.functional.cheb_stream_supported(nn_[lvl], b, fin, fout, 6, l_op, u_op, None)
        _fused_layer_case(mvb, ops, kind, lvl, b, fin, fout, relu, bias, "mesh_tc=1,0")
    finally:
        mvb._lib.tune("stream_tc=0,16")


def test_stream_layer_is_deterministic_and_can_be_switched_off(mvb, ops):
    A, D, U, nn_ = ops
    Fn = mvb.functional
    dev = torch.device("cuda:0")
    n = nn_[0]
    ei, norm = O.cheb_norm(A[0]._indices(), n)
    l_op = mvb.operators.from_edges(ei.to(dev), norm.to(dev), n, dev)
    u_op = mvb.operators.from_sparse(U[0].to(dev), dev)
    x = _rand(u_op.n_cols, 64, 16, seed=5).to(dev).requires_grad_()
    w = _rand(6, 16, 16, seed=6, scale=0.1).to(dev).requires_grad_()
    bias = _rand(16, seed=7, scale=0.1).to(dev).requires_grad_()
    outs = []
    mvb._lib.tune("stream_tc=1")           # opt-in (the default training step keeps the step-by-step kernels at this level)
    try:
        assert Fn.cheb_stream_supported(n, 64, 16, 16, 6, l_op, u_op, None)
        for _ in range(3):
            x.grad = w.grad = bias.grad = None
            y = Fn.cheb_layer(x, w, bias, l_op, u_op, None, relu=True)
            y.square().sum().backward()
            outs.append((y.detach().clone(), x.grad.clone(), w.grad.clone(), bias.grad.clone()))
    finally:
        mvb._lib.tune("stream_tc=0")
    for o in outs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(outs[0], o))
    # the recurrence is the step kernels' arithmetic: switched off, the composition path gives the same basis, and the
    # outputs agree to the 3xTF32 rounding of the two contraction orders
    assert not Fn.cheb_stream_supported(n, 64, 16, 16, 6, l_op, u_op, None)
    y2 = Fn.cheb_layer(x.detach(), w.detach(), bias.detach(), l_op, u_op, None, relu=True)
    assert rel_err(outs[0][0], y2) < 1e-5


def test_fused_layer_is_deterministic_and_needs_no_input_grad(mvb, ops):
    A, D, U, nn_ = ops
    Fn = mvb.functional
    dev = torch.device("cuda:0")
    n = nn_[2]
    ei, norm = O.cheb_norm(A[2]._indices(), n)
    l_op = mvb.operators.from_edges(ei.to(dev), norm.to(dev), n, dev)
    d_op = mvb.operators.from_sparse(D[2].to(dev), dev)
    x = _rand(n, 64, 16, seed=5).to(dev)                     # no grad: dx is skipped
    w = _rand(6, 16, 16, seed=6, scale=0.1).to(dev).requires_grad_()
    outs = []
    for _ in range(2):
        w.grad = None
        y = Fn.cheb_layer(x, w, None, l_op, None, d_op, relu=True)
        y.square().sum().backward()
        outs.append((y.detach().clone(), w.grad.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_unsupported_levels_fall_back(mvb, ops):
    A, D, U, nn_ = ops
    Fn = mvb.functional
    dev = torch.device("cuda:0")
    ei, norm = O.cheb_norm(A[0]._indices(), nn_[0])
    l_op = mvb.operators.from_edges(ei.to(dev), norm.to(dev), nn_[0], dev)
    assert not Fn.cheb_layer_supported(nn_[0], 4, 16, 16, 6, l_op, None, None)      # level 0 does not fit shared memory
    x = _rand(nn_[0], 2, 16, seed=7).to(dev)
    w = _rand(6, 16, 16, seed=8, scale=0.1).to(dev)
    y = Fn.cheb_layer(x, w, None, l_op, None, None, relu=True)                       # composition path
    assert torch.equal(y, Fn.cheb_conv(x, w, None, l_op, True))

