"""The sigma-VAE decoder variances (optimal and learned log sigma, include/mvb.h mvb_vae_loss_sigma_fwd/_bwd and
mvb_gaussian_nll_sigma_fwd/_bwd) against float64 autograd, at their edges, under CUDA-graph capture, and through the
training engine.

sc(t) = -6 + softplus(t + 6), n = N*C; optimal: log sigma = sc(0.5 log(SSE / (B n))), learned: log sigma = sc(s);
rec_b = 0.5 SSE_b / sigma^2 + n (log sigma + 0.5 log 2 pi); the rest of the loss is models/cheb_VAE.py:321-346."""
import copy
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import update_reference as R
from tests.helpers import elem_err, rel_err
from tests.test_gpu_step_modes import _batch, _config, _net, _restore

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-4
GLOSS = 0.375


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    return meshvae_b200


@pytest.fixture(scope="module")
def ops():
    from oracle import mesh_vae_oracle as O
    from tests.helpers import OPERATORS_NPZ
    return O.load_operators(OPERATORS_NPZ)


def _gate(what, dev, ref):
    d, r = dev.detach().double().cpu(), ref.detach().double().cpu()
    assert torch.isfinite(d).all(), f"{what}: not finite"
    e = rel_err(d, r)
    assert e < TOL, f"{what}: rel_err {e:.3e}"
    ee = elem_err(d.reshape(-1), r.reshape(-1))
    assert ee <= 1.0, f"{what}: elem_err {ee:.3f}"


# ---------------------------------------------------------------------------------------------------------------------
# float64 restatement
# ---------------------------------------------------------------------------------------------------------------------
def sc(t):
    return -6.0 + torch.logaddexp(t + 6.0, torch.zeros_like(t))


def ref_sigma_loss(recon, x, mu, lv, y_hat, y, mode, s=None, gloss=GLOSS):
    """recon / x [B,N,C] mesh-major; float64 autograd of gloss * loss -> dict of values and gradients"""
    r, m, l, yh = (t.detach().to("cpu", torch.float64).requires_grad_() for t in (recon, mu, lv, y_hat))
    xx, yy = x.detach().to("cpu", torch.float64), y.detach().to("cpu", torch.float64)
    b, n = r.shape[0], r.shape[1] * r.shape[2]
    sse_b = ((r - xx) ** 2).sum((1, 2))
    sp = None
    if mode == "optimal":
        t = 0.5 * torch.log(sse_b.sum() / (b * n))
    else:
        sp = torch.tensor(float(np.float32(s)), dtype=torch.float64, requires_grad=True)       # s is an fp32 parameter
        t = sp
    ls = sc(t)
    rec = 0.5 * sse_b * torch.exp(-2.0 * ls) + n * (ls + R.LOG_2PI_HALF)
    kld = -0.5 * (1.0 + l - m * m - l.exp()).sum(-1)
    logq = (yh * yy).sum(-1).log()
    loss = (kld + rec - 2.0 * logq).mean()
    (gloss * loss).backward()
    out = {"loss": loss.detach(), "kld": kld.detach(), "rec": rec.detach(), "log_sigma": ls.detach(), "d_recon": r.grad,
           "d_mu": m.grad, "d_logvar": l.grad, "d_yhat": yh.grad, "sse": sse_b.sum().detach()}
    if sp is not None:
        out["d_s"] = sp.grad
    return out


def _inputs(b, n, c, ld, dt, seed, scale=0.5):
    """recon_vm [N,B,ld] (junk in the padding), x [B,N,C] of dtype dt; y_hat has the label's entry exactly 1 (so that
    log q = 0 on both sides and the fp64 loss can be held to 1e-12)"""
    g = torch.Generator().manual_seed(seed)
    recon_vm = torch.randn(n, b, ld, generator=g)
    x = (recon_vm[..., :c].permute(1, 0, 2).double() + scale * torch.randn(b, n, c, generator=g, dtype=torch.float64)).to(dt)
    mu, lv = torch.randn(b, 16, generator=g), 0.5 * torch.randn(b, 16, generator=g)
    lab = torch.randint(0, 2, (b,), generator=g)
    y = F.one_hot(lab, 2)
    y_hat = y.float()
    return recon_vm, x.contiguous(), mu, lv, y_hat, y


def _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, mode, s=0.0, gloss=GLOSS):
    """functional.vae_loss forward and autograd backward on the device -> dict"""
    leaves = [t.to(DEV).requires_grad_() for t in (recon_vm, mu, lv, y_hat)]
    sp = torch.nn.Parameter(torch.full((), float(s), device=DEV)) if mode == "learned" else None
    loss, kld, rec, correct, ls = mvb.functional.vae_loss(leaves[0], x.to(DEV), leaves[1], leaves[2], leaves[3], y.to(DEV),
                                                          log_sigma=sp if mode == "learned" else "optimal", channels=c,
                                                          return_log_sigma=True)
    torch.autograd.backward(loss, torch.tensor(gloss, device=DEV, dtype=loss.dtype))
    torch.cuda.synchronize()
    out = {"loss": loss, "kld": kld, "rec": rec, "correct": correct, "log_sigma": ls, "d_recon_vm": leaves[0].grad,
           "d_recon": leaves[0].grad[..., :c].permute(1, 0, 2), "d_mu": leaves[1].grad, "d_logvar": leaves[2].grad,
           "d_yhat": leaves[3].grad}
    if sp is not None:
        out["d_s"] = sp.grad
    return out


CASES = [(b, n, ld) for b in (1, 3, 64, 300) for n in (1, 20, 4998) for ld in (3, 4)]


@pytest.mark.parametrize("mode", ["optimal", "learned"])
@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
@pytest.mark.parametrize("b,n,ld", CASES, ids=[f"B{b}-N{n}-ld{ld}" for b, n, ld in CASES])
def test_sigma_loss_matches_float64(mvb, b, n, ld, dt, mode):
    c = 3
    recon_vm, x, mu, lv, y_hat, y = _inputs(b, n, c, ld, dt, seed=b * 31 + n + ld)
    s = 0.3
    got = _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, mode, s)
    ref = ref_sigma_loss(recon_vm[..., :c].permute(1, 0, 2), x, mu, lv, y_hat, y, mode, s)
    assert got["loss"].dtype == dt and got["rec"].dtype == dt
    for k in ("loss", "kld", "rec", "log_sigma", "d_recon", "d_mu", "d_logvar", "d_yhat") + (("d_s",) if mode == "learned" else ()):
        _gate(f"{mode} B{b} N{n} ld{ld} {dt} {k}", got[k], ref[k])
    if ld > c:
        assert torch.count_nonzero(got["d_recon_vm"][..., c:]) == 0, "the padding lane carries no gradient"
    if dt == torch.float64:
        # the loss in fp64 throughout, with the kld terms the device adds (fp32 as in the reference model, gated above)
        exact = float((got["kld"].double().cpu() + ref["rec"]).mean())
        loss = float(got["loss"].detach())
        assert abs(loss - exact) <= 1e-12 * abs(exact), (loss, exact)


# ---------------------------------------------------------------------------------------------------------------------
# edge cases
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
def test_perfect_reconstruction_is_finite(mvb, dt):
    """SSE = 0: optimal log sigma = sc(-inf) = -6, rec = n (-6 + log(2 pi)/2), d_recon = 0; learned: finite, d_s = gloss n sc'"""
    b, n, c = 64, 4998, 3
    recon_vm, _, mu, lv, y_hat, y = _inputs(b, n, c, 4, dt, seed=5)
    x = recon_vm[..., :c].permute(1, 0, 2).to(dt).contiguous()
    for mode in ("optimal", "learned"):
        got = _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, mode, s=0.0)
        for k, v in got.items():
            assert torch.isfinite(v.double()).all(), (mode, k)
        assert torch.count_nonzero(got["d_recon_vm"]) == 0
        if mode == "optimal":
            assert float(got["log_sigma"]) == -6.0
            ref_rec = torch.full((b,), n * c * (-6.0 + R.LOG_2PI_HALF), dtype=torch.float64)
        else:
            ref = ref_sigma_loss(recon_vm[..., :c].permute(1, 0, 2), x, mu, lv, y_hat, y, mode, 0.0)
            ref_rec = ref["rec"]
            _gate("learned SSE=0 d_s", got["d_s"], ref["d_s"])
            _gate("learned SSE=0 log_sigma", got["log_sigma"], ref["log_sigma"])
        _gate(f"{mode} SSE=0 rec", got["rec"], ref_rec)


@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
def test_clipped_optimal_sigma_matches_float64(mvb, dt):
    """an error of 1e-6: 0.5 log(SSE / (B n)) ~ -13.8, where the soft clip holds log sigma near -6"""
    b, n, c = 64, 4998, 3
    recon_vm, x, mu, lv, y_hat, y = _inputs(b, n, c, 4, dt, seed=6, scale=1e-6)
    got = _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, "optimal")
    ref = ref_sigma_loss(recon_vm[..., :c].permute(1, 0, 2), x, mu, lv, y_hat, y, "optimal")
    assert -6.0 < float(ref["log_sigma"]) < -5.99
    for k in ("loss", "rec", "log_sigma", "d_recon"):
        _gate(f"clipped {dt} {k}", got[k], ref[k])


def test_optimal_sigma_is_stationary(mvb):
    """with the clip inactive (log sigma ~ 10, where sc(t) = t to 1e-7) the gradient through sigma vanishes: d_recon is
    that of the constant-sigma epilogue run at the same sigma, to the rounding of that sigma to fp32"""
    b, n, c = 64, 4998, 3
    recon_vm, x, mu, lv, y_hat, y = _inputs(b, n, c, 4, torch.float64, seed=7, scale=math.exp(10.0))
    got = _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, "optimal")
    ls = float(got["log_sigma"])
    assert 9.9 < ls < 10.1
    r = recon_vm.to(DEV).requires_grad_()
    loss, *_ = mvb.functional.vae_loss(r, x.to(DEV), mu.to(DEV), lv.to(DEV), y_hat.to(DEV), y.to(DEV), log_sigma=ls, channels=c)
    torch.autograd.backward(loss, torch.tensor(GLOSS, device=DEV, dtype=torch.float64))
    fixed = r.grad[..., :c].permute(1, 0, 2)
    # log sigma as an fp32 argument is off by up to half an ulp of 10 (4.8e-7), sigma^-2 by twice that relative; the
    # gradient through the optimal sigma is ~2 exp(-16) = 2.3e-7 of the direct term
    d = (got["d_recon"] - fixed).abs()
    assert bool((d <= 4e-6 * fixed.abs() + 1e-30).all()), float((d / fixed.abs().clamp_min(1e-30)).max())


def test_learned_sigma_at_the_optimum_has_no_gradient(mvb):
    """sigma^2 = SSE / (B n) is where d rec / d s vanishes"""
    b, n, c = 64, 4998, 3
    recon_vm, x, mu, lv, y_hat, y = _inputs(b, n, c, 4, torch.float64, seed=8)
    sse = float(((recon_vm[..., :c].permute(1, 0, 2).double() - x) ** 2).sum())
    target = 0.5 * math.log(sse / (b * n * c))
    s = math.log(math.expm1(target + 6.0)) - 6.0           # sc(s) = target
    got = _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, "learned", s=s)
    # s is an fp32 parameter: rounding it (3e-8 relative) moves 1 - SSE sigma^-2 by ~2 sc'(s)^2 |s| 6e-8
    assert abs(float(got["d_s"])) <= 1e-6 * GLOSS * n * c, float(got["d_s"])
    assert abs(float(got["log_sigma"]) - target) < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# determinism, capture, no host synchronisation
# ---------------------------------------------------------------------------------------------------------------------
def test_same_bits_every_run(mvb):
    b, n, c = 300, 4998, 3
    recon_vm, x, mu, lv, y_hat, y = _inputs(b, n, c, 4, torch.float64, seed=9)
    for mode in ("optimal", "learned"):
        a = _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, mode, s=0.2)
        for _ in range(2):
            bb = _run(mvb, recon_vm, x, mu, lv, y_hat, y, c, mode, s=0.2)
            for k in a:
                assert torch.equal(a[k], bb[k]), (mode, k)


def test_captured_optimal_sigma_follows_new_inputs(mvb):
    Fn = mvb.functional
    b, n, c = 64, 4998, 3
    st = [t.to(DEV) for t in _inputs(b, n, c, 4, torch.float64, seed=10)]
    recon = st[0].clone().requires_grad_()

    def step():
        recon.grad = None
        out = Fn.vae_loss(recon, st[1], st[2], st[3], st[4], st[5], log_sigma="optimal", channels=c, return_log_sigma=True)
        out[0].backward()
        return out

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    recon.grad = torch.zeros_like(recon)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        recon.grad = None
        out = Fn.vae_loss(recon, st[1], st[2], st[3], st[4], st[5], log_sigma="optimal", channels=c, return_log_sigma=True)
        out[0].backward()
    grad = recon.grad
    out = [t.detach() for t in out]          # the static outputs; the captured autograd graph is not kept alive
    seen = set()
    for k in range(3):
        new = _inputs(b, n, c, 4, torch.float64, seed=100 + k, scale=0.25 * (k + 1))
        with torch.no_grad():
            recon.copy_(new[0].to(DEV))
        st[1].copy_(new[1].to(DEV))
        g.replay()
        torch.cuda.synchronize()
        eager = step()
        torch.cuda.synchronize()
        assert torch.equal(out[0], eager[0]) and torch.equal(out[4], eager[4]) and torch.equal(out[2], eager[2])
        assert torch.equal(grad, recon.grad)
        seen.add(float(out[4]))
    assert len(seen) == 3, "log sigma did not follow the inputs"


def test_captured_learned_sigma_follows_adam(mvb):
    """loss, backward into the flat gradient buffer and Adam, captured once: each replay reads the s that the previous
    replay's Adam wrote; an eager run of the same sequence gives the same bits"""
    from meshvae_b200.engine import FlatAdam
    Fn = mvb.functional
    b, n, c = 64, 4998, 3
    ins = [t.to(DEV) for t in _inputs(b, n, c, 4, torch.float64, seed=11)]

    def make():
        sp = torch.nn.Parameter(torch.zeros((), device=DEV))
        opt = FlatAdam([sp], lr=0.05, weight_decay=5e-4)
        sp._mvb_grad_sink = opt.grad_views[0]
        return sp, opt

    def step(sp, opt):
        out = Fn.vae_loss(ins[0], ins[1], ins[2], ins[3], ins[4], ins[5], log_sigma=sp, channels=c, return_log_sigma=True)
        out[0].backward()
        opt.step()
        return out

    sp_e, opt_e = make()
    eager = []
    for _ in range(4):
        out = step(sp_e, opt_e)
        eager.append((out[0].clone(), out[4].clone(), sp_e.detach().clone()))
    sp, opt = make()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):           # warm-up, then the optimizer state is reset
        step(sp, opt)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    opt.flat_p.zero_(); opt.m.zero_(); opt.v.zero_(); opt.step_count.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step(sp, opt)
    prev = None
    for loss_e, ls_e, s_e in eager:
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out[0], loss_e) and torch.equal(out[4], ls_e) and torch.equal(sp.detach(), s_e)
        if prev is not None:
            assert float(out[4]) != prev
        prev = float(out[4])
    assert float(sp) != 0.0


@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
@pytest.mark.parametrize("kind", ["optimal", "learned"])
def test_logpdf_gaussian_nll_with_device_log_sigma(mvb, dt, kind):
    """logpdf.gaussian_nll with the sigma-VAE's own log sigma, a CUDA tensor with gradient: no host synchronisation, and
    autograd through both arguments matches float64"""
    g = torch.Generator().manual_seed(12)
    mu0 = torch.randn(8, 313, 3, generator=g)
    x0 = (mu0.double() + 0.3 * torch.randn(8, 313, 3, generator=g, dtype=torch.float64)).to(dt)
    gout = torch.randn(8, 313, 3, generator=g, dtype=torch.float64)

    def expr(mu, x, s, lp):
        ls = lp.softclip(((x - mu) ** 2).mean().sqrt().log(), -6) if kind == "optimal" else lp.softclip(s, -6)
        return lp.gaussian_nll(mu, ls, x)

    class _RefLp:             # the reference's logpdf.py:22-28 in torch
        softclip = staticmethod(lambda t, m: m + F.softplus(t - m))
        gaussian_nll = staticmethod(lambda mu, ls, x: 0.5 * torch.pow((x - mu) / ls.exp(), 2) + ls + R.LOG_2PI_HALF)

    mo = mu0.double().requires_grad_()
    so = torch.tensor([0.4], dtype=torch.float64, requires_grad=True)
    ref = expr(mo, x0.double(), so, _RefLp)
    ref.backward(gout)
    mg = mu0.to(DEV).requires_grad_()
    sg = torch.tensor([0.4], device=DEV, requires_grad=True)
    xg, gg = x0.to(DEV), gout.to(DEV, dt)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = expr(mg, xg, sg, mvb.logpdf)
        out.backward(gg)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert out.dtype == dt
    _gate(f"nll {kind} {dt} out", out, ref)
    _gate(f"nll {kind} {dt} d_mu", mg.grad, mo.grad)
    if kind == "learned":
        _gate(f"nll {kind} {dt} d_s", sg.grad, so.grad)


def test_gaussian_nll_d_log_sigma_is_deterministic(mvb):
    g = torch.Generator().manual_seed(13)
    mu = torch.randn(3_000_000, generator=g).to(DEV)
    x = torch.randn(3_000_000, generator=g).to(DEV)
    grads = []
    for _ in range(3):
        ls = torch.tensor(0.1, device=DEV, requires_grad=True)
        mvb.functional.gaussian_nll(mu, x, ls).sum().backward()
        grads.append(ls.grad.clone())
    assert all(torch.equal(grads[0], t) for t in grads[1:])


# ---------------------------------------------------------------------------------------------------------------------
# the training engine
# ---------------------------------------------------------------------------------------------------------------------
def _sigma_net(mvb, ops, cfg, mode):
    net = _net(mvb, ops, cfg)
    net.set_decoder_sigma(mode)
    return net


def _engine_run(mvb, ops, cfg, mode, b, steps, serial, monkeypatch):
    """-> (losses, log sigmas, flat_g after step 0, flat_p after the steps and a ragged step)"""
    from meshvae_b200.engine import TrainEngine
    L = mvb._lib
    real = L.defer_side_chains
    try:
        if serial:
            L.tune("pdl=0")
            monkeypatch.setattr(L, "defer_side_chains", lambda on: real(False))
        net = _sigma_net(mvb, ops, cfg, mode)
        eng = TrainEngine(net, b, lr=1e-3, weight_decay=5e-4, use_graph=not serial)
        eng.capture(warmup=1)
        losses, sigmas, g0 = [], [], None
        for s in range(steps):
            x, y, eps = _batch(b, ops[3][0], cfg["num_classes"], cfg["num_style"], 900 + s)
            losses.append(eng.step(x.pin_memory(), x.double().pin_memory(), y.pin_memory(), eps_host=eps.pin_memory()))
            sigmas.append(float(eng.log_sigma))
            if s == 0:
                g0 = eng.opt.flat_g.clone()
        rb = b // 2 + 1
        x, y, eps = _batch(rb, ops[3][0], cfg["num_classes"], cfg["num_style"], 77)
        out = eng.ragged_step(x.to(DEV), x.double().to(DEV), F.one_hot(y, cfg["num_classes"]).to(DEV), eps.to(DEV))
        losses.append(float(out[0]))
        torch.cuda.synchronize()
        return losses, sigmas, g0, eng.opt.flat_p.clone()
    finally:
        monkeypatch.setattr(L, "defer_side_chains", real)
        _restore(mvb)


ENGINE = [(m, b, p) for m in ("optimal", "learned") for b in (64, 300) for p in (0.0, 0.2)]


@pytest.mark.parametrize("mode,b,p", ENGINE, ids=[f"{m}-B{b}-p{p}" for m, b, p in ENGINE])
def test_engine_sigma_step_is_bit_identical_to_serial(mvb, ops, monkeypatch, mode, b, p):
    cfg = _config("default", p)
    la, sa, ga, pa = _engine_run(mvb, ops, cfg, mode, b, 3, False, monkeypatch)
    lb, sb, gb, pb = _engine_run(mvb, ops, cfg, mode, b, 3, True, monkeypatch)
    assert all(np.isfinite(v) for v in la), la
    assert la == lb, (la, lb)
    assert sa == sb, (sa, sb)
    assert len(set(sa)) == len(sa), f"log sigma did not change from step to step: {sa}"
    assert torch.equal(ga, gb), "step-0 gradients differ"
    assert torch.equal(pa, pb), "parameters differ after three steps and a ragged step"


def test_engine_learned_sigma_step0_matches_float64(mvb, ops, monkeypatch):
    """the serial engine's first step in the learned mode: the loss terms, log sigma, d_s (in the flat gradient buffer) and
    Adam's update of s against float64, from the step's own reconstruction and latent outputs"""
    from meshvae_b200.engine import TrainEngine
    Fn, L = mvb.functional, mvb._lib
    cfg = _config("default", 0.0)
    b = 64
    x, y, eps = _batch(b, ops[3][0], cfg["num_classes"], cfg["num_style"], 4242)
    seen = {}
    real_loss = Fn.vae_loss

    def spy(recon_vm, x_gt, mu, logvar, y_hat, yy, *a, **kw):
        seen["args"] = [t.detach().clone() for t in (recon_vm, x_gt, mu, logvar, y_hat, yy)]
        seen["channels"] = kw.get("channels")
        return real_loss(recon_vm, x_gt, mu, logvar, y_hat, yy, *a, **kw)

    real = L.defer_side_chains
    try:
        L.tune("pdl=0")
        monkeypatch.setattr(L, "defer_side_chains", lambda on: real(False))
        net = _sigma_net(mvb, ops, cfg, "learned")
        with torch.no_grad():
            net.log_sigma.fill_(0.25)
        eng = TrainEngine(net, b, lr=1e-3, weight_decay=5e-4, use_graph=False)
        eng.capture(warmup=1)
        i = [k for k, p in enumerate(eng.opt.params) if p is net.log_sigma]
        assert len(i) == 1
        # bucket 1 of the flat buffer: behind every convolution weight (bucket 2, the front)
        assert all(o < eng.opt.offsets[i[0]] for p, o in zip(eng.opt.params, eng.opt.offsets) if p.dim() == 3)
        monkeypatch.setattr(Fn, "vae_loss", spy)
        loss = eng.step(x.pin_memory(), x.double().pin_memory(), y.pin_memory(), eps_host=eps.pin_memory())
        monkeypatch.setattr(Fn, "vae_loss", real_loss)
        torch.cuda.synchronize()
        d_s = eng.opt.grad_views[i[0]].clone()
        s1 = float(net.log_sigma)
        ls, rec, kld = eng.log_sigma.clone(), eng.rec.clone(), eng.kld.clone()
    finally:
        monkeypatch.setattr(L, "defer_side_chains", real)
        _restore(mvb)
    recon_vm, x_gt, mu, logvar, y_hat, yy = seen["args"]
    c = seen["channels"] or recon_vm.shape[2]
    ref = ref_sigma_loss(recon_vm[..., :c].permute(1, 0, 2), x_gt, mu, logvar, y_hat, yy, "learned", 0.25, gloss=1.0)
    _gate("engine loss", torch.tensor(loss), ref["loss"])
    _gate("engine rec", rec, ref["rec"])
    _gate("engine kld", kld, ref["kld"])
    _gate("engine log_sigma", ls, ref["log_sigma"])
    _gate("engine d_s", d_s, ref["d_s"])
    p1, _, _ = R.adam_step(torch.tensor(0.25), ref["d_s"], torch.tensor(0.0), torch.tensor(0.0), 1, 1e-3, weight_decay=5e-4)
    assert abs(s1 - float(p1)) <= 1e-6 * abs(float(p1)), (s1, float(p1))


def test_checkpoint_round_trips_learned_sigma(mvb, ops, tmp_path):
    from meshvae_b200 import formats
    from meshvae_b200.engine import TrainEngine
    cfg = _config("default", 0.0)
    b = 16

    def batch(seed):
        x, y, eps = _batch(b, ops[3][0], cfg["num_classes"], cfg["num_style"], seed)
        return x.pin_memory(), x.double().pin_memory(), y.pin_memory(), eps.pin_memory()

    net = _sigma_net(mvb, ops, cfg, "learned")
    eng = TrainEngine(net, b, use_graph=False)
    eng.capture(warmup=1)
    for s in range(2):
        x, xg, y, eps = batch(50 + s)
        eng.step(x, xg, y, eps_host=eps)
    path = formats.save_model(net, eng.opt, 2, 0.0, 0.0, str(tmp_path))
    ck = torch.load(path, weights_only=False)
    assert "log_sigma" in ck["state_dict"] and float(ck["state_dict"]["log_sigma"]) != 0.0
    idx = [k for k, p in enumerate(net.parameters()) if p is net.log_sigma][0]
    assert idx in ck["optimizer"]["state"]

    net2 = _net(mvb, ops, cfg, seed=99)
    net2.set_decoder_sigma("learned", init=-1.0)
    eng2 = TrainEngine(net2, b, use_graph=False)
    eng2.capture(warmup=1)
    formats.load_model(net2, path, eng2.opt)
    for k, v in net.state_dict().items():
        assert torch.equal(v, net2.state_dict()[k]), k
    assert torch.equal(eng.opt.m, eng2.opt.m) and torch.equal(eng.opt.v, eng2.opt.v)
    x, xg, y, eps = batch(60)
    l1 = eng.step(x, xg, y, eps_host=eps)
    l2 = eng2.step(x, xg, y, eps_host=eps)
    assert l1 == l2 and torch.equal(eng.opt.flat_p, eng2.opt.flat_p)
