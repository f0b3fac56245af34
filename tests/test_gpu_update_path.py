"""The rest of the training step against float64 (tests/update_reference.py) at every shape a config or a batch can give
it: the loss epilogue (mvb_vae_loss_fwd/bwd), the latent element-wise kernels, the dense layers (mvb_linear_fwd/bwd), the
fused Adam updates (mvb_adam_step, mvb_adam_step_hp, engine.FlatAdam) and the fused data-parallel reduce + Adam
(mvb_dp_reduce_adam) at every world size the kernel takes.

Tolerances are derived, not tuned.  U = 2^-24 is the unit roundoff of fp32: one rounded fp32 operation is off by at most
U relative.  The derivation of each bound is next to it.  Run with -s to see every measured error next to its bound."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import update_reference as R
from tests.helpers import elem_err, rel_err
from tests.test_gpu_heads_shapes import keep_mask

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
LOG_SIGMA = 1.0009117126464844          # softclip(1, -6) in fp32, the model's log sigma


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    return meshvae_b200


def _report(name, value, bound=1.0):
    print(f"ERR {name}: {value:.3g} (bound {bound:.3g})")
    assert value <= bound, (name, value, bound)


def bound_err(a, ref, bound):
    """max over the elements of |a - ref| / bound (passes when <= 1); bound is a per-element error bound"""
    a, ref = a.detach().double().cpu(), ref.detach().double().cpu()
    assert a.shape == ref.shape, (tuple(a.shape), tuple(ref.shape))
    d = (a - ref).abs()
    bound = torch.as_tensor(bound, dtype=torch.float64).expand_as(d)
    if bool(((d > 0) & (bound <= 0)).any()):
        return math.inf
    return float((d / bound.clamp_min(1e-300)).max()) if d.numel() else 0.0


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# σ = expf(log σ) is fp32 on the device and in the reference model (log_sigma.exp() of an fp32 tensor); the device expf
# is within 2 ulps of the correctly rounded value and the CPU's within 0.5, so the two σ differ by up to 2.5 ulps = 5U
# relative, and (x - recon)^2 / σ^2 by up to 10U.  log σ = 0 makes σ = 1 exactly on both sides.
def _sig(log_sigma):
    return 0.0 if log_sigma == 0.0 else 10 * U


# ================================================ the loss epilogue ================================================
def _loss_inputs(b, n, z, ncls, c, ld, dt, seed):
    g = _gen(seed)
    recon_vm = torch.randn(n, b, ld, generator=g)              # the padding floats are random: they must be ignored
    x = (recon_vm[..., :c].permute(1, 0, 2) + 0.5 * torch.randn(b, n, c, generator=g)).to(dt).contiguous()
    mu, lv = torch.randn(b, z, generator=g), 0.5 * torch.randn(b, z, generator=g)
    y_hat = torch.softmax(2 * torch.randn(b, ncls, generator=g), 1)
    lab = torch.randint(0, ncls, (b,), generator=g)
    lab[-1] = ncls - 1                                         # a label in the last class
    y = F.one_hot(lab, ncls)
    return recon_vm, x, mu, lv, y_hat, y


def _loss_bounds(recon_vm, x, mu, lv, y_hat, y, c, log_sigma, gloss):
    """reference values and per-element error bounds of every output of mvb_vae_loss_fwd / _bwd"""
    f32 = x.dtype == torch.float32
    recon = recon_vm[..., :c].permute(1, 0, 2)
    ref = R.vae_loss(recon, x, mu, lv, y_hat, y, log_sigma)
    grads = R.vae_loss_grads(recon, x, mu, lv, y_hat, y, log_sigma, gloss)
    grads["dnll"] = R.vae_loss_grads(recon, x, mu, lv, y_hat, y, log_sigma, recon.shape[0])["d_recon"]   # (recon - x) / σ^2
    sig = _sig(log_sigma)
    m, l = mu.double(), lv.double()
    bnd = {}
    # kld[b] = -0.5 sum_j (1 + lv - mu^2 - exp(lv)) in fp32, j ascending (16 lanes + a shuffle tree): each term's four
    # roundings and expf's 2 ulps are <= 6U of the terms' magnitudes, and the Z-term sum adds <= Z U of them
    mag = 0.5 * (1 + l.abs() + m * m + l.exp()).sum(-1)
    bnd["kld"] = (mu.shape[1] + 6) * U * mag
    # rec[b]: every term 0.5 ((x - recon) / σ)^2 + log σ + log(2π)/2 is positive.  fp32 x: a difference, a product by
    # 1/σ, a square, a scale and an add: <= 8U per term (10U with margin), fp64 accumulation.  fp64 x: fp64 throughout.
    r_rec = (10 * U if f32 else 1e-12) + sig
    bnd["rec"] = r_rec * ref["rec"]
    # loss = mean_b(kld + rec - 2 log q), every term >= 0: the three bounds add up; log q: logf's ulp on |log q| plus
    # U absolute (q = y_hat[label] exactly: y is one-hot)
    logq = (y_hat.double() * y.double()).sum(-1).log()
    bnd["loss"] = (bnd["kld"] + bnd["rec"] + 2 * (2 * U * logq.abs() + U)).mean() + 1e-12 * float(ref["loss"])
    # dnll = (recon - x) / σ^2: fp32 x: a difference, 1/(σ σ) (two roundings), a product: 4U; fp64 x: one cast, U
    r_dnll = (4 * U if f32 else U) + sig
    # d_recon = (float)(gloss / B) * dnll: two more roundings
    bnd["d_recon"] = (r_dnll + 2 * U) * grads["d_recon"].abs()
    bnd["d_mu"] = 2 * U * grads["d_mu"].abs()
    s = abs(gloss) / mu.shape[0]
    # d_logvar = s 0.5 (expf(lv) - 1): expf's 2 ulps are absolute in the difference (6U e^lv with the other roundings)
    bnd["d_logvar"] = 3 * U * grads["d_logvar"].abs() + s * 0.5 * 6 * U * l.exp()
    bnd["d_yhat"] = 3 * U * grads["d_yhat"].abs()
    return ref, grads, bnd, r_dnll


def _check_loss(tag, got, ref, grads, bnd, r_dnll, c, ld, check_grads=True):
    loss, kld, rec, correct, dnll = got[:5]
    _report(f"{tag} loss", bound_err(loss.reshape(1), ref["loss"].reshape(1), bnd["loss"]))
    _report(f"{tag} kld", bound_err(kld, ref["kld"], bnd["kld"]))
    _report(f"{tag} rec", bound_err(rec, ref["rec"], bnd["rec"]))
    assert int(correct) == ref["correct"], tag
    d_ref = grads["dnll"]
    _report(f"{tag} dnll", bound_err(dnll[..., :c].permute(1, 0, 2), d_ref, r_dnll * d_ref.abs()))
    if ld > c:
        assert torch.equal(dnll[..., c:], torch.zeros_like(dnll[..., c:])), "padding of dnll must be zero"
    if check_grads:
        d_recon, d_mu, d_lv, d_yh = got[5:]
        if ld > c:
            assert torch.equal(d_recon[..., c:], torch.zeros_like(d_recon[..., c:]))
        _report(f"{tag} d_recon", bound_err(d_recon[..., :c].permute(1, 0, 2), grads["d_recon"], bnd["d_recon"]))
        _report(f"{tag} d_mu", bound_err(d_mu, grads["d_mu"], bnd["d_mu"]))
        _report(f"{tag} d_logvar", bound_err(d_lv, grads["d_logvar"], bnd["d_logvar"]))
        _report(f"{tag} d_yhat", bound_err(d_yh, grads["d_yhat"], bnd["d_yhat"]))


def _loss_abi(mvb, recon_vm, x, mu, lv, y_hat, y, c, log_sigma, gloss, outs=(True, True, True, True), dnll_out=None):
    """mvb_vae_loss_fwd then mvb_vae_loss_bwd through the C ABI; recon_vm / x may be (offset) views.  Returns
    (loss, kld, rec, correct, dnll, d_recon, d_mu, d_logvar, d_yhat), None for an output not asked for."""
    L = mvb._lib
    n, b, ld = recon_vm.shape
    z, ncls = mu.shape[1], y_hat.shape[1]
    dev = recon_vm.device
    loss = torch.empty((), device=dev, dtype=torch.float64)
    kld = torch.empty(b, device=dev)
    rec = torch.empty(b, device=dev, dtype=torch.float64)
    correct = torch.empty((), device=dev, dtype=torch.int64)
    dnll = torch.empty(n, b, ld, device=dev) if dnll_out is None else dnll_out
    ws_bytes = L.lib.mvb_vae_loss_workspace_bytes(b, n)
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    L.check(L.lib.mvb_vae_loss_fwd(b, n, c, z, ncls, L.ptr(recon_vm), ld, L.ptr(x), int(x.dtype == torch.float64), L.ptr(mu),
                                   L.ptr(lv), L.ptr(y_hat), L.ptr(y), log_sigma, L.ptr(loss), L.ptr(kld), L.ptr(rec),
                                   L.ptr(correct), L.ptr(dnll), L.ptr(ws), ws_bytes, L.stream_ptr()), "mvb_vae_loss_fwd")
    g = torch.tensor(gloss, device=dev, dtype=torch.float64)
    d = [torch.full(t.shape, float("nan"), device=dev) if want else None
         for want, t in zip(outs, (dnll, mu, lv, y_hat))]
    L.check(L.lib.mvb_vae_loss_bwd(b, n, ld, z, ncls, L.ptr(dnll), L.ptr(mu), L.ptr(lv), L.ptr(y_hat), L.ptr(y), L.ptr(g),
                                   *[L.ptr(t) for t in d], L.stream_ptr()), "mvb_vae_loss_bwd")
    torch.cuda.synchronize()
    return [loss, kld, rec, correct, dnll] + d


# (B, N, Z, ncls, (C, ld)): every B, N, Z, ncls and (C, ld) of the sweep at least once; B > 64 runs the finalize kernel's
# later passes (64 meshes each), B > 32 the second batch tile of the partial kernel, N = 4998 more than 128 vertex chunks.
# The shared-memory tile is 32 vertices unless C * sizeof(x) + 4 ld exceeds 48: (6, 8) and (12, 12) take 16 (fp32, and
# (6, 8) in fp64), (12, 12) in fp64 takes 8.
LOSS_CASES = [(1, 1, 1, 1, (1, 1)), (31, 7, 5, 2, (3, 3)), (32, 33, 16, 3, (3, 4)), (33, 313, 17, 10, (6, 8)),
              (64, 4998, 64, 2, (3, 4)), (65, 313, 256, 32, (12, 12)), (1023, 33, 17, 3, (12, 12)),
              (1025, 4998, 16, 2, (3, 4)), (1025, 7, 256, 32, (6, 8)), (65, 4998, 5, 10, (1, 1)), (1023, 313, 64, 1, (3, 3))]


@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
@pytest.mark.parametrize("b,n,z,ncls,cl", LOSS_CASES)
def test_loss_epilogue_matches_float64(mvb, b, n, z, ncls, cl, dt):
    """functional.vae_loss (forward and autograd backward with the upstream gradient 0.375) at the case's shape"""
    c, ld = cl
    log_sigma = LOG_SIGMA if LOSS_CASES.index((b, n, z, ncls, cl)) % 2 else 0.0
    recon_vm, x, mu, lv, y_hat, y = _loss_inputs(b, n, z, ncls, c, ld, dt, seed=b * 7 + n + z)
    gloss = 0.375                    # exact in fp32: the fp32 loss's upstream gradient is the same number
    ref, grads, bnd, r_dnll = _loss_bounds(recon_vm, x, mu, lv, y_hat, y, c, log_sigma, gloss)
    leaves = [t.cuda().requires_grad_() for t in (recon_vm, mu, lv, y_hat)]
    loss, kld, rec, correct = mvb.functional.vae_loss(leaves[0], x.cuda(), leaves[1], leaves[2], leaves[3], y.cuda(),
                                                      log_sigma=log_sigma, channels=c)
    assert loss.dtype == dt and rec.dtype == dt
    torch.autograd.backward(loss, torch.tensor(gloss, device="cuda", dtype=dt))
    torch.cuda.synchronize()
    # the dnll plane itself comes from the C ABI call (autograd keeps it internal); bit-identical forward outputs
    got = _loss_abi(mvb, recon_vm.cuda(), x.cuda(), mu.cuda(), lv.cuda(), y_hat.cuda(), y.cuda(), c, log_sigma, gloss)
    assert torch.equal(kld, got[1]) and int(correct) == int(got[3])
    if dt == torch.float64:
        assert torch.equal(loss, got[0]) and torch.equal(rec, got[2])
    tag = f"loss B{b} N{n} Z{z} cls{ncls} C{c}/{ld} {'f64' if dt == torch.float64 else 'f32'}"
    _check_loss(tag, got, ref, grads, bnd, r_dnll, c, ld)
    for a, b_ in zip([t.grad for t in leaves], got[5:]):
        assert torch.equal(a, b_), "autograd and the C ABI backward differ"


@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
def test_loss_offset_views_and_null_outputs(mvb, dt):
    """x_gt and recon offset by one element (the scalar cp.async staging), dnll offset by one float (the scalar store of
    the padded-entry path): the same bits as the aligned call.  NULL outputs in the backward call."""
    b, n, z, ncls, c, ld = 65, 313, 16, 2, 3, 4
    recon_vm, x, mu, lv, y_hat, y = (t.cuda() for t in _loss_inputs(b, n, z, ncls, c, ld, dt, seed=3))
    base = _loss_abi(mvb, recon_vm, x, mu, lv, y_hat, y, c, LOG_SIGMA, 1.5)
    rbuf = torch.empty(recon_vm.numel() + 1, device="cuda")
    rbuf[1:].copy_(recon_vm.reshape(-1))
    xbuf = torch.empty(x.numel() + 1, device="cuda", dtype=dt)
    xbuf[1:].copy_(x.reshape(-1))
    dbuf = torch.empty(recon_vm.numel() + 1, device="cuda")
    off = _loss_abi(mvb, rbuf[1:].view(n, b, ld), xbuf[1:].view(b, n, c), mu, lv, y_hat, y, c, LOG_SIGMA, 1.5,
                    dnll_out=dbuf[1:].view(n, b, ld))
    for i, (a, r) in enumerate(zip(off, base)):
        assert torch.equal(a, r), i
    # any subset of the backward outputs: the others are not written, the requested ones are the same bits
    for outs in [(False, True, False, False), (True, False, False, True), (False, False, True, False)]:
        part = _loss_abi(mvb, recon_vm, x, mu, lv, y_hat, y, c, LOG_SIGMA, 1.5, outs=outs)
        for want, a, r in zip(outs, part[5:], base[5:]):
            assert (a is None) if not want else torch.equal(a, r)


def test_loss_first_maximum_wins_and_run_to_run(mvb):
    """ties in y_hat: the first maximal class is the prediction, as torch.argmax; labels in the last class"""
    b, n, z, ncls = 96, 33, 16, 4
    recon_vm, x, mu, lv, _, _ = _loss_inputs(b, n, z, ncls, 3, 4, torch.float64, seed=8)
    rows = torch.tensor([[0.25, 0.25, 0.25, 0.25], [0.1, 0.4, 0.4, 0.1], [0.4, 0.1, 0.1, 0.4], [0.0, 0.0, 0.5, 0.5]])
    y_hat = rows.repeat(b // 4, 1)
    lab = torch.arange(b) % ncls
    lab[3::4] = 3                   # [.., 0.5, 0.5] with label 3: the tie goes to class 2, so this one is wrong
    y = F.one_hot(lab, ncls)
    ref = R.vae_loss(recon_vm[..., :3].permute(1, 0, 2), x, mu, lv, y_hat, y, LOG_SIGMA)
    args = [t.cuda() for t in (recon_vm, x, mu, lv, y_hat, y)]
    got1 = _loss_abi(mvb, *args, 3, LOG_SIGMA, 1.0)
    got2 = _loss_abi(mvb, *args, 3, LOG_SIGMA, 1.0)
    assert int(got1[3]) == ref["correct"]
    for a, r in zip(got1, got2):
        assert torch.equal(a, r)


@pytest.mark.parametrize("dt,c_ok", [(torch.float64, 16), (torch.float32, 24)], ids=["x64", "x32"])
def test_loss_widest_entry_and_the_refusal_past_it(mvb, dt, c_ok):
    """the staging tile needs at least 8 vertices of (C ground-truth values + ld reconstruction floats) x 32 meshes in
    48 KB: C = ld = 16 with fp64 x_gt, 24 with fp32.  One more channel is refused with MvbError, not launched."""
    b, n, z, ncls = 40, 45, 16, 2
    recon_vm, x, mu, lv, y_hat, y = _loss_inputs(b, n, z, ncls, c_ok, c_ok, dt, seed=4)
    ref, grads, bnd, r_dnll = _loss_bounds(recon_vm, x, mu, lv, y_hat, y, c_ok, LOG_SIGMA, 1.0)
    got = _loss_abi(mvb, *[t.cuda() for t in (recon_vm, x, mu, lv, y_hat, y)], c_ok, LOG_SIGMA, 1.0)
    _check_loss(f"loss widest C{c_ok}", got, ref, grads, bnd, r_dnll, c_ok, c_ok)
    recon_vm, x, mu, lv, y_hat, y = _loss_inputs(b, n, z, ncls, c_ok + 1, c_ok + 1, dt, seed=4)
    with pytest.raises(mvb._lib.MvbError, match="too large"):
        _loss_abi(mvb, *[t.cuda() for t in (recon_vm, x, mu, lv, y_hat, y)], c_ok + 1, LOG_SIGMA, 1.0)


def test_pack_vertex_major_offset_output(mvb):
    """the C == 3, Cp == 4 path writes 16-byte entries: an output view offset by one float takes the scalar stores"""
    L = mvb._lib
    b, n = 16, 96
    x = torch.randn(b, n, 3, generator=_gen(5)).cuda()
    outs = []
    for shift in (0, 1):
        buf = torch.full((n * b * 4 + 1,), float("nan"), device="cuda")
        o = buf[shift:shift + n * b * 4].view(n, b, 4)
        L.check(L.lib.mvb_pack_vertex_major(b, n, 3, 4, L.ptr(x), L.ptr(o), L.stream_ptr()), "mvb_pack_vertex_major")
        outs.append(o)
    torch.cuda.synchronize()
    ref = torch.cat([x.permute(1, 0, 2), torch.zeros(n, b, 1, device="cuda")], 2)
    assert torch.equal(outs[0], ref) and torch.equal(outs[1], ref)


# ========================================== the latent element-wise kernels ==========================================
def _past_grid_cap():
    """elements beyond what one pass of the capped grid covers (ew_grid: 16 blocks of 256 threads per SM)"""
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 16 * 256 + 37


def test_reparam_past_the_grid_cap(mvb):
    n = _past_grid_cap()
    g = _gen(6)
    mu, lv, eps, dz = torch.randn(n, generator=g), 0.5 * torch.randn(n, generator=g), torch.randn(n, generator=g), torch.randn(n, generator=g)
    cu = [t.cuda() for t in (mu, lv, eps, dz)]
    z = mvb.functional.reparameterize(cu[0].requires_grad_(), cu[1].requires_grad_(), cu[2])
    z.backward(cu[3])
    std = (0.5 * lv.double()).exp()
    zr = eps.double() * std + mu.double()
    # z = fmaf(eps, expf(0.5 lv), mu): expf's 2 ulps + the product's rounding are relative to |eps std| (the sum can
    # cancel), one more U relative to |z|
    _report("reparam z", bound_err(z, zr, 5 * U * (eps.double() * std).abs() + U * zr.abs()))
    assert torch.equal(cu[0].grad, cu[3])
    d = dz.double() * eps.double() * 0.5 * std
    _report("reparam dlogvar", bound_err(cu[1].grad, d, 7 * U * d.abs()))       # expf 2 ulps + 3 products


@pytest.mark.parametrize("b,z", [(1, 1), (1025, 17), (300, 256)])
def test_kld_kernels(mvb, b, z):
    g = _gen(b + z)
    mu, lv, gout = torch.randn(b, z, generator=g), 0.5 * torch.randn(b, z, generator=g), torch.randn(b, generator=g)
    cm, cl = mu.cuda().requires_grad_(), lv.cuda().requires_grad_()
    k = mvb.functional.kld(cm, cl)
    k.backward(gout.cuda())
    m, l = mu.double(), lv.double()
    kr = -0.5 * (1 + l - m * m - l.exp()).sum(-1)
    # the sequential fp32 sum of Z terms: as the loss's kld bound
    _report(f"kld B{b} Z{z}", bound_err(k, kr, (z + 6) * U * 0.5 * (1 + l.abs() + m * m + l.exp()).sum(-1)))
    gd = gout.double()[:, None]
    _report(f"kld d_mu B{b} Z{z}", bound_err(cm.grad, gd * m, U * (gd * m).abs()))
    dl = gd * 0.5 * (l.exp() - 1)
    _report(f"kld d_logvar B{b} Z{z}", bound_err(cl.grad, dl, 3 * U * dl.abs() + gd.abs() * 0.5 * 6 * U * l.exp()))


@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
def test_gaussian_nll_past_the_grid_cap(mvb, dt):
    n = _past_grid_cap()
    g = _gen(7)
    mu, x, gout = torch.randn(n, generator=g), torch.randn(n, generator=g).to(dt), torch.randn(n, generator=g).to(dt)
    cm = mu.cuda().requires_grad_()
    out = mvb.functional.gaussian_nll(cm, x.cuda(), LOG_SIGMA)
    out.backward(gout.cuda())
    sigma = R.loss_sigma(LOG_SIGMA)
    t = (x.double() - mu.double()) / sigma
    ref = 0.5 * t * t + float(torch.tensor(LOG_SIGMA, dtype=torch.float32)) + R.LOG_2PI_HALF
    f32 = dt == torch.float32
    # positive terms: fp32 <= 8U per value (as the loss's rec), fp64 exact but for σ
    _report(f"nll {dt}", bound_err(out, ref, ((10 * U if f32 else 1e-12) + _sig(LOG_SIGMA)) * ref.abs()))
    d = gout.double() * (mu.double() - x.double()) / (sigma * sigma)
    _report(f"nll d_mu {dt}", bound_err(cm.grad, d, ((5 * U if f32 else U) + _sig(LOG_SIGMA)) * d.abs()))


# ================================================ the dense layers ================================================
def _lin_tol(length):
    """rtol = RMS floor of an fp32 dot product of `length` terms summed in sequence: each partial sum is rounded once,
    so the error is a random walk of `length` roundings of partial sums that grow like sqrt(k); its standard deviation
    is about U sqrt(length) / 2.45 of the RMS of the result.  8 U sqrt(length) is 4.5 standard deviations with a margin
    of four; 4U more for the bias, the ReLU and the dropout scale."""
    return 8 * U * math.sqrt(length) + 4 * U


def _linear_abi(mvb, x, x_vm_f, w, b, relu, p, seed, offset, y_vm_f, gy, want_dx=True):
    """mvb_linear_fwd then mvb_linear_bwd through the C ABI.  x is [M,K] (x_vm_f 0) or [K/F,M,F]; y / gy likewise."""
    L = mvb._lib
    n, k = w.shape
    m = x.shape[1] if x_vm_f else x.shape[0]
    y = torch.full(((n // y_vm_f, m, y_vm_f) if y_vm_f else (m, n)), float("nan"), device="cuda")
    L.check(L.lib.mvb_linear_fwd(m, k, n, L.ptr(x), x_vm_f, L.ptr(w), L.ptr(b), int(relu), p, seed, None, offset, L.ptr(y),
                                 y_vm_f, L.stream_ptr()), "mvb_linear_fwd")
    dx = torch.full_like(x, float("nan")) if want_dx else None
    dw = torch.full_like(w, float("nan"))
    db = torch.full((n,), float("nan"), device="cuda") if b is not None else None
    L.check(L.lib.mvb_linear_bwd(m, k, n, L.ptr(x), x_vm_f, L.ptr(w), L.ptr(y), L.ptr(gy), y_vm_f, int(relu), p, L.ptr(dx),
                                 L.ptr(dw), L.ptr(db), L.stream_ptr()), "mvb_linear_bwd")
    torch.cuda.synchronize()
    return y, dx, dw, db


def _vm_to_rows(t, f):
    """[V,M,F] vertex-major -> the logical [M, V*F]"""
    return t.permute(1, 0, 2).reshape(t.shape[1], -1) if f else t


def _run_linear(mvb, tag, m, k, n, x_vm_f=0, y_vm_f=0, relu=True, bias=True, p=0.0, want_dx=True, seed=0):
    g = _gen(seed + m + k + n)
    xl = torch.randn(m, k, generator=g)
    w = torch.randn(n, k, generator=g) / math.sqrt(k)
    b = 0.1 * torch.randn(n, generator=g) if bias else None
    gyl = torch.randn(m, n, generator=g)
    x = xl.reshape(m, k // x_vm_f, x_vm_f).permute(1, 0, 2).contiguous() if x_vm_f else xl
    gy = gyl.reshape(m, n // y_vm_f, y_vm_f).permute(1, 0, 2).contiguous() if y_vm_f else gyl
    dseed, doff = 0x5EED0000 + seed, 11
    y, dx, dw, db = _linear_abi(mvb, x.cuda(), x_vm_f, w.cuda(), None if b is None else b.cuda(), relu, p, dseed, doff,
                                y_vm_f, gy.cuda(), want_dx)
    yl = _vm_to_rows(y, y_vm_f)
    keep = keep_mask(dseed, doff, m, n, p) if p > 0 else None
    yr = R.linear_fwd(xl, w, b, relu=relu, keep=keep, p=p)
    tk = _lin_tol(k)
    _report(f"{tag} y", elem_err(yl, yr, tk, tk))
    if keep is not None:
        assert bool((yl.cpu()[torch.from_numpy(~keep)] == 0).all()), "a dropped unit is not zero"
    dxr, dwr, dbr = R.linear_bwd(xl, w, yl, gyl, relu=relu, p=p)      # the mask of the backward pass is y > 0
    tm, tn = _lin_tol(m), _lin_tol(n)
    _report(f"{tag} dW", elem_err(dw, dwr, tm, tm))
    if bias:
        _report(f"{tag} db", elem_err(db, dbr, tm, tm))
    if want_dx:
        _report(f"{tag} dx", elem_err(_vm_to_rows(dx, x_vm_f), dxr, tn, tn))


MS = [1, 31, 32, 33, 64, 65, 300, 512]
ENC = [(f, v) for f in (4, 8, 16, 24, 32, 48, 64) for v in (1, 20, 79, 313)]


@pytest.mark.parametrize("f,v", ENC)
def test_enc_lin_vertex_major_input(mvb, f, v):
    """x.reshape(B, V*F) of the coarsest level's [V, B, F] buffer: K = V*F from 4 to 20032; K > 640 takes further K
    chunks in the forward kernel (K = 1280: exactly two)"""
    i = ENC.index((f, v))
    m = MS[i % len(MS)]
    _run_linear(mvb, f"enc_lin F{f} V{v} M{m}", m, v * f, 72, x_vm_f=f, relu=True, bias=i % 3 != 0, p=0.2 if i % 2 else 0.0,
                want_dx=i % 4 != 1, seed=i)


@pytest.mark.parametrize("k,m", [(3, 1), (18, 33), (66, 65), (258, 512)])
def test_dec_lin(mvb, k, m):
    """dec_lin: K = C + Z (e.g. 2 + 16, 2 + 64, 2 + 256), hidden width 512; K = 3 and 18 and 66 are not multiples of 4"""
    _run_linear(mvb, f"dec_lin K{k} M{m}", m, k, 512, relu=True, bias=True, p=0.2, seed=k)


@pytest.mark.parametrize("f,v,m", [(32, 20, 64), (32, 79, 31), (16, 79, 300), (48, 20, 65), (8, 313, 33), (64, 20, 1),
                                   (4, 313, 512), (24, 79, 32)])
def test_dec_lin_2_vertex_major_output(mvb, f, v, m):
    """x.reshape(B, V, F) written as [V, B, F]: N = V*F up to 2528 > 640 takes further N chunks in the dx tiles"""
    _run_linear(mvb, f"dec_lin_2 F{f} V{v} M{m}", m, 96, v * f, y_vm_f=f, relu=True, bias=True, p=0.2 if m % 2 else 0.0,
                seed=f + v)


@pytest.mark.parametrize("m,k,n,relu,bias", [(33, 641, 37, True, True), (65, 1283, 641, False, False), (1, 7, 5, False, True),
                                             (300, 1280, 1281, True, False)])
def test_linear_scalar_staging(mvb, m, k, n, relu, bias):
    """K or N not a multiple of 4: the scalar cp.async staging, in the K and N chunks past 640 too"""
    _run_linear(mvb, f"linear M{m} K{k} N{n}", m, k, n, relu=relu, bias=bias, seed=1)


def test_linear_vertex_major_width_6(mvb):
    """a vertex-major width that is not a multiple of 4 (scalar staging of the vertex-major views) on both sides"""
    _run_linear(mvb, "linear vm6 in", 65, 6 * 107, 96, x_vm_f=6, relu=True, bias=True, p=0.2, seed=2)
    _run_linear(mvb, "linear vm6 out", 33, 96, 6 * 107, y_vm_f=6, relu=True, bias=True, seed=3)


@pytest.mark.parametrize("m,k,n,x_vm_f,y_vm_f", [(64, 640, 512, 32, 0), (65, 96, 2528, 0, 32), (33, 641, 37, 0, 0)])
def test_linear_deferred_weight_gradient_is_bit_identical(mvb, m, k, n, x_vm_f, y_vm_f):
    """mvb_tune("defer_wgrad=1"): the dx tiles alone on the stream, dW / db on side lane 1, joined with
    mvb_side_join_lane(stream, 1) - the same bits as the one-launch form"""
    L = mvb._lib
    g = _gen(m + k + n)
    xl, w, b, gyl = torch.randn(m, k, generator=g), torch.randn(n, k, generator=g) / math.sqrt(k), torch.randn(n, generator=g), torch.randn(m, n, generator=g)
    x = (xl.reshape(m, k // x_vm_f, x_vm_f).permute(1, 0, 2).contiguous() if x_vm_f else xl).cuda()
    gy = (gyl.reshape(m, n // y_vm_f, y_vm_f).permute(1, 0, 2).contiguous() if y_vm_f else gyl).cuda()
    w, b = w.cuda(), b.cuda()
    one = _linear_abi(mvb, x, x_vm_f, w, b, True, 0.2, 5, 0, y_vm_f, gy)
    try:
        L.tune("defer_wgrad=1")
        dx, dw, db = torch.empty_like(x), torch.full_like(w, float("nan")), torch.full_like(b, float("nan"))
        L.check(L.lib.mvb_linear_bwd(m, k, n, L.ptr(x), x_vm_f, L.ptr(w), L.ptr(one[0]), L.ptr(gy), y_vm_f, 1, 0.2, L.ptr(dx),
                                     L.ptr(dw), L.ptr(db), L.stream_ptr()), "mvb_linear_bwd")
        L.check(L.lib.mvb_side_join_lane(L.stream_ptr(), 1), "mvb_side_join_lane")
    finally:
        L.tune("defer_wgrad=0")
    torch.cuda.synchronize()
    assert torch.equal(dx, one[1]) and torch.equal(dw, one[2]) and torch.equal(db, one[3])


# ==================================================== Adam ====================================================
def _f32(v):
    return float(np.float32(v))


def adam_p_rtol(beta1, beta2, t, fresh):
    """relative bound on the kernel's parameter increment lr/bc1 * m / (sqrt(v/bc2) + eps) against the float64 step.
    - 12U: the roundings of the ten or so fp32 operations on the increment (sqrtf, rsqrtf's 2 ulps, the divisions);
    - powf is within 2 ulps of beta^t, and 1 - beta^t cancels: 4U beta^t / (1 - beta^t) on bc1, half that on bc2
      (it sits under the square root).
    - The kernel computes 1 - beta and beta^t from the fp32 beta; torch uses the double.  At beta2 = 0.999 the fp32
      1 - beta2 is 1.29e-5 smaller (relatively), at beta1 = 0.9 2.4e-7.  From the zero state at t = 1 this cancels
      exactly: v / (1 - beta2) = g^2 on both sides (`fresh`).  From any other state it does not: the new v differs
      by up to that 1.29e-5 and 1 - beta2^t by |beta2^t - fp32 beta2^t| / (1 - beta2^t), both halved by the root."""
    b1f, b2f = _f32(beta1), _f32(beta2)
    r = 12 * U + 4 * U * b1f ** t / (1 - b1f ** t) + 2 * U * b2f ** t / (1 - b2f ** t)
    if not fresh:
        d1 = abs((1 - b1f) - (1 - beta1)) / (1 - beta1) + abs(b1f ** t - beta1 ** t) / (1 - beta1 ** t)
        d2 = abs((1 - b2f) - (1 - beta2)) / (1 - beta2) + abs(b2f ** t - beta2 ** t) / (1 - beta2 ** t)
        r += d1 + 0.5 * d2
    return r


def _adam_bounds(p0, g, m0, v0, t, lr, betas, eps, wd, gs, fresh=False):
    """the float64 step from the fp32 state (p0, m0, v0) at counter t, and per-element bounds of the kernel's error"""
    pr, mr, vr = R.adam_step(p0, g, m0, v0, t, lr, betas, eps, wd, gs)
    b1, b2 = betas
    geff = (g.double() * gs).abs() + wd * p0.double().abs()         # the terms of g * grad_scale + wd * p
    # m = fmaf(b1, m, (1 - b1) g): the fp32 1 - b1 (see adam_p_rtol) on the new term, and 4U of both terms' magnitudes
    d1 = abs((1 - _f32(b1)) - (1 - b1)) / (1 - b1)
    m_b = (d1 + 4 * U) * (b1 * m0.double().abs() + (1 - b1) * geff) + 1e-300
    # v = fmaf(b2, v, (1 - b2) g g): the same with the fp32 1 - b2 - the 1.29e-5 at b2 = 0.999 - on the g^2 term
    d2 = abs((1 - _f32(b2)) - (1 - b2)) / (1 - b2)
    v_b = (d2 + 6 * U) * (b2 * v0.double() + (1 - b2) * geff * geff) + 1e-300
    # p: half an ulp of the new value for the final subtraction, the increment's relative bound, and m's absolute bound
    # carried through lr / bc1 / denom (m may be the small difference of its two terms; the increment is then small too)
    denom = vr.sqrt() / math.sqrt(1 - b2 ** t) + eps
    p_b = U * pr.abs() + adam_p_rtol(b1, b2, t, fresh) * (pr - p0.double()).abs() + lr / (1 - b1 ** t) * m_b / denom + 1e-300
    return (pr, mr, vr), (p_b, m_b, v_b)


def _adam_check(tag, got, p0, g, m0, v0, t, lr, betas, eps, wd, gs, fresh=False):
    """the kernel's (p, m, v) after one step from the fp32 state (p0, m0, v0) at counter t, against the float64 step"""
    ref, bnd = _adam_bounds(p0, g, m0, v0, t, lr, betas, eps, wd, gs, fresh)
    e = {k_: bound_err(a, r, b) for k_, a, r, b in zip("pmv", got, ref, bnd)}
    for k_, v_ in e.items():
        _report(f"{tag} {k_}", v_)
    return e


def _adam_abi(mvb, which, p, g, m, v, step, hp):
    """one mvb_adam_step (which == 0) or mvb_adam_step_hp (1) on copies; -> (p, m, v, step)"""
    L = mvb._lib
    p, m, v = p.clone(), m.clone(), v.clone()
    st = torch.tensor(step, device="cuda", dtype=torch.int64)
    if which == 0:
        L.check(L.lib.mvb_adam_step(p.numel(), L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), L.ptr(st), *hp, L.stream_ptr()),
                "mvb_adam_step")
    else:
        h = torch.tensor(hp, device="cuda", dtype=torch.float32)
        L.check(L.lib.mvb_adam_step_hp(p.numel(), L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), L.ptr(st), L.ptr(h), L.stream_ptr()),
                "mvb_adam_step_hp")
    torch.cuda.synchronize()
    return p, m, v, int(st)


def _cheb_vae_flat_size():
    from oracle import mesh_vae_oracle as O
    from tests.helpers import OPERATORS_NPZ
    from meshvae_b200 import dp
    A, D, U_, nn_ = O.load_operators(OPERATORS_NPZ)
    net = O.OracleChebVAE(3, O.DEFAULT_CONFIG, D, U_, A, nn_)
    return dp.flat_layout([p for name, p in net.named_parameters() if not name.startswith("dec_lin_1")], 32)[1]


def _adam_state(n, seed, zero=False):
    g = _gen(seed)
    p, gr = torch.randn(n, generator=g), torch.randn(n, generator=g)
    if zero:
        return p, gr, torch.zeros(n), torch.zeros(n)
    return p, gr, 0.01 * torch.randn(n, generator=g), 1e-4 * torch.rand(n, generator=g)


@pytest.mark.parametrize("n", [1, 3, 255, 256, 257, 303105, "cheb_VAE"])
def test_adam_entry_points_match_float64(mvb, n):
    """mvb_adam_step and mvb_adam_step_hp, bit-identical to each other, against the float64 step; 303105 elements are
    one past what the capped grid (8 blocks of 256 per SM) covers in one pass"""
    n = _cheb_vae_flat_size() if n == "cheb_VAE" else n
    hpv = (1e-3, 0.9, 0.999, 1e-8, 5e-4, 1.0)
    for t0, zero in [(0, True), (9, False)]:
        p, gr, m, v = _adam_state(n, seed=n + t0, zero=zero)
        cu = [a.cuda() for a in (p, gr, m, v)]
        got0 = _adam_abi(mvb, 0, *cu, t0, hpv)
        got1 = _adam_abi(mvb, 1, *cu, t0, hpv)
        for a, b in zip(got0[:3], got1[:3]):
            assert torch.equal(a, b)
        assert got0[3] == got1[3] == t0 + 1
        _adam_check(f"adam n{n} t{t0 + 1}", got0[:3], p, gr, m, v, t0 + 1, hpv[0], hpv[1:3], hpv[3], hpv[4], hpv[5],
                    fresh=zero and t0 == 0)


def test_adam_trajectory_one_step_at_a_time(mvb):
    """300 steps of mvb_adam_step_hp, each compared with the float64 step taken from the kernel's own fp32 state (so
    differences do not compound); the learning rate changes at step 150"""
    n = 4115
    g = _gen(12)
    p = torch.randn(n, generator=g).cuda()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    step = torch.zeros((), device="cuda", dtype=torch.int64)
    hp = [1e-3, 0.9, 0.999, 1e-8, 5e-4, 1.0]
    hyper = torch.tensor(hp, device="cuda")
    L = mvb._lib
    worst = {"p": 0.0, "m": 0.0, "v": 0.0}
    for t in range(1, 301):
        if t == 150:
            hp[0] = 3e-4
            hyper[0] = hp[0]
        gr = (torch.randn(n, generator=g) * (1 + 0.01 * t)).cuda()
        p0, m0, v0 = p.cpu(), m.cpu(), v.cpu()
        L.check(L.lib.mvb_adam_step_hp(n, L.ptr(p), L.ptr(gr), L.ptr(m), L.ptr(v), L.ptr(step), L.ptr(hyper), L.stream_ptr()))
        torch.cuda.synchronize()
        assert int(step) == t
        ref, bnd = _adam_bounds(p0, gr.cpu(), m0, v0, t, hp[0], (0.9, 0.999), 1e-8, 5e-4, 1.0, fresh=t == 1)
        e = {k_: bound_err(a, r, b) for k_, a, r, b in zip("pmv", (p, m, v), ref, bnd)}
        for k_ in worst:
            assert e[k_] <= 1.0, (t, k_, e[k_])
            worst[k_] = max(worst[k_], e[k_])
    for k_, v_ in worst.items():
        _report(f"adam trajectory {k_}", v_)


@pytest.mark.parametrize("t0", [1, 10, 1000, 1000000])
def test_adam_step_counter_preset(mvb, t0):
    """the counter preset (a restored optimizer) reaches the bias corrections: t0 + 1 in the step"""
    hpv = (1e-3, 0.9, 0.999, 1e-8, 5e-4, 1.0)
    p, gr, m, v = _adam_state(1031, seed=t0)
    got = _adam_abi(mvb, 1, *[a.cuda() for a in (p, gr, m, v)], t0, hpv)
    assert got[3] == t0 + 1
    _adam_check(f"adam t{t0 + 1}", got[:3], p, gr, m, v, t0 + 1, *hpv[:1], hpv[1:3], *hpv[3:])


@pytest.mark.parametrize("lr,betas,eps,wd,gs", [(1e-3, (0.9, 0.999), 1e-8, 0.0, 1.0), (1e-3, (0.9, 0.999), 1e-8, 0.1, 1.0),
                                                (1e-2, (0.5, 0.9), 1e-3, 5e-4, 1.0 / 3.0), (3e-4, (0.5, 0.9), 1e-8, 0.1, 1.0 / 3.0)])
def test_adam_hyper_parameters(mvb, lr, betas, eps, wd, gs):
    hpv = (lr, *betas, eps, wd, gs)
    p, gr, m, v = _adam_state(777, seed=int(wd * 1000) + int(eps * 1e4))
    for which in (0, 1):
        got = _adam_abi(mvb, which, *[a.cuda() for a in (p, gr, m, v)], 4, hpv)
        _adam_check(f"adam lr{lr} b{betas} eps{eps} wd{wd} gs{gs:.3f} [{which}]", got[:3], p, gr, m, v, 5, lr, betas, eps, wd, gs)


def test_adam_zero_learning_rate_and_zero_gradients(mvb):
    p, gr, m, v = _adam_state(1000, seed=3)
    cu = [a.cuda() for a in (p, gr, m, v)]
    hpv = (0.0, 0.9, 0.999, 1e-8, 5e-4, 1.0)
    got = _adam_abi(mvb, 1, *cu, 6, hpv)
    assert torch.equal(got[0], cu[0]), "lr = 0 must leave p unchanged"
    _adam_check("adam lr0", got[:3], p, gr, m, v, 7, *hpv[:1], hpv[1:3], *hpv[3:])
    assert not torch.equal(got[1], cu[2]) and not torch.equal(got[2], cu[3])
    # zero gradients without weight decay: from the zero state nothing moves, from another state the moments decay
    z = torch.zeros_like(cu[1])
    hpv = (1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0)
    got = _adam_abi(mvb, 1, cu[0], z, torch.zeros_like(z), torch.zeros_like(z), 0, hpv)
    assert torch.equal(got[0], cu[0]) and not got[1].any() and not got[2].any()
    got = _adam_abi(mvb, 0, cu[0], z, cu[2], cu[3], 2, hpv)
    _adam_check("adam zero grad", got[:3], p, torch.zeros_like(gr), m, v, 3, *hpv[:1], hpv[1:3], *hpv[3:])


def test_flat_adam_matches_torch_adam_after_restore_at_step_37(mvb):
    """torch.optim.Adam (fp32, CUDA) runs 37 steps; its state dict goes into a FlatAdam through
    formats.load_adam_state_dict; both then take 5 more steps on the same gradients.  A step count that did not reach
    the bias correction (t = 1 instead of 38) would move p by about 6 times the right increment."""
    from meshvae_b200 import formats
    from meshvae_b200.engine import FlatAdam
    g = _gen(37)
    net = torch.nn.Sequential(torch.nn.Linear(13, 7), torch.nn.Linear(7, 3)).cuda()
    net2 = torch.nn.Sequential(torch.nn.Linear(13, 7), torch.nn.Linear(7, 3)).cuda()
    opt = torch.optim.Adam(net.parameters(), lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-4, foreach=False)
    grads = [[torch.randn(p.shape, generator=g).cuda() for p in net.parameters()] for _ in range(42)]
    for s in range(37):
        for p, gr in zip(net.parameters(), grads[s]):
            p.grad = gr
        opt.step()
    net2.load_state_dict(net.state_dict())
    flat = FlatAdam(list(net2.parameters()), lr=1.0)
    formats.load_adam_state_dict(flat, net2, opt.state_dict())
    assert int(flat.step_count) == 37
    for s in range(37, 42):
        p0 = flat.flat_p.clone()
        m0, v0 = flat.m.clone(), flat.v.clone()
        for view, gr in zip(flat.grad_views, grads[s]):
            view.copy_(gr)
        flat.step()
        for p, gr in zip(net.parameters(), grads[s]):
            p.grad = gr
        opt.step()
        torch.cuda.synchronize()
        _adam_check(f"FlatAdam step {s + 1}", (flat.flat_p, flat.m, flat.v), p0.cpu(), flat.flat_g.cpu(), m0.cpu(), v0.cpu(),
                    s + 1, 2e-3, (0.9, 0.999), 1e-8, 5e-4, 1.0)
        for p, q in zip(net.parameters(), net2.parameters()):
            st = opt.state[p]
            assert int(float(st["step"])) == int(flat.step_count) == s + 1
            # torch's fp32 Adam and the kernel differ by about 1e-5 of an increment of ~2e-3 (the kernel's fp32
            # 1 - beta2, see adam_p_rtol) and a few ulps: far below 1e-6 of the parameters' scale
            assert rel_err(q, p) < 1e-6


# ========================================= data-parallel reduce + Adam =========================================
def _dp_run(mvb, world, steps=2):
    """`world` ranks on one device and one stream, one after another: before each rank's launch every pad word is
    2^30, so each wait for a peer's signal passes at once (signals are epoch numbers, here 1 and 2) and no kernel waits
    for another.  Buckets: [0, 4) channel 0, [4, 1024) channel 1, [1024, 2228) channel 0, an empty one at 2228 on
    channel 1; the first bucket of a step ticks the counter; max_ctas 0, 1, 3."""
    L, lib = mvb._lib, mvb._lib.lib
    n = 2228
    buckets = [(0, 4, 0, 1, 0), (4, 1020, 1, 0, 1), (1024, n - 1024, 0, 0, 3), (n, 0, 1, 0, 0)]
    dev = torch.device("cuda")
    g = _gen(world)
    pad_words = int(lib.mvb_dp_pad_bytes()) // 4
    pads = torch.zeros(world, pad_words, device=dev, dtype=torch.int32)
    arr = ctypes.c_void_p * world
    pad_ptrs = arr(*[pads[r].data_ptr() for r in range(world)])
    grads = [torch.empty(n, device=dev) for _ in range(world)]
    grad_ptrs = arr(*[t.data_ptr() for t in grads])
    p_init = torch.randn(n, generator=g).to(dev)
    reps = [dict(p=p_init.clone(), m=torch.zeros(n, device=dev), v=torch.zeros(n, device=dev), gsum=torch.empty(n, device=dev),
                 step=torch.zeros((), device=dev, dtype=torch.int64),
                 state=torch.zeros(int(lib.mvb_dp_state_bytes()) // 4, device=dev, dtype=torch.int32)) for _ in range(world)]
    hpv = (1e-3, 0.9, 0.999, 1e-8, 5e-4, 1.0 / world)
    hyper = torch.tensor(hpv, device=dev)
    st = L.stream_ptr()
    for s in range(1, steps + 1):
        for gr in grads:
            gr.copy_(torch.randn(n, generator=g) * (1 + s))
        p0, m0, v0 = reps[0]["p"].cpu(), reps[0]["m"].cpu(), reps[0]["v"].cpu()
        for r, rp in enumerate(reps):
            pads.fill_(1 << 30)
            L.check(lib.mvb_dp_begin(world, r, 2, pad_ptrs, L.ptr(rp["state"]), st), "mvb_dp_begin")
            for off, cnt, ch, tick, max_ctas in buckets:
                pads.fill_(1 << 30)
                L.check(lib.mvb_dp_reduce_adam(world, r, ch, off, cnt, L.ptr(rp["p"]), grad_ptrs, L.ptr(rp["m"]), L.ptr(rp["v"]),
                                               L.ptr(rp["gsum"]), L.ptr(rp["step"]), tick, L.ptr(hyper), pad_ptrs,
                                               L.ptr(rp["state"]), max_ctas, st), "mvb_dp_reduce_adam")
        torch.cuda.synchronize()
        gs_ref = R.rank_order_sum(grads)
        for r, rp in enumerate(reps):
            assert int(rp["state"][1]) == 0, f"rank {r}: a wait for a peer's signal timed out"
            assert int(rp["state"][0]) == s and int(rp["step"]) == s
            assert torch.equal(rp["gsum"], gs_ref), f"rank {r}: the gradient sum is not the fp32 rank-order sum"
            for k_ in ("p", "m", "v"):
                assert torch.equal(rp[k_], reps[0][k_]), f"rank {r}: {k_} differs from rank 0"
        _adam_check(f"dp world {world} step {s}", (reps[0]["p"], reps[0]["m"], reps[0]["v"]), p0, gs_ref.cpu(), m0, v0, s,
                    hpv[0], hpv[1:3], hpv[3], hpv[4], hpv[5], fresh=s == 1)


@pytest.mark.parametrize("world", list(range(1, 17)))
def test_dp_reduce_adam_every_world_size(mvb, world):
    """world 1-16 (mvb_dp_max_world): the kernel reads peers eight at a time, so world 9-16 runs a second group"""
    assert mvb._lib.lib.mvb_dp_max_world() == 16
    _dp_run(mvb, world)
