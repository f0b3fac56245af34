"""The importance-weighted estimate of the held-out log-likelihood (include/mvb.h mvb_iw_sample, mvb_iw_log_weights,
mvb_iw_reduce; cheb_VAE.log_likelihood; loop.log_likelihood): each stage against float64 on the device's own inputs, the
whole estimate against the float64 oracle with the same weights and samples, its identities, the statistics of the
sampler, and its launch behaviour (determinism, CUDA-graph capture, no host synchronisation).

With S samples z_s ~ q(z | x, y) = N(mu, exp(logvar)) per mesh, n = N*C and the decoder's log sigma:
  log w_s = log p(x | z_s, y) - log r_s,  log p(x | z) = -SSE / (2 sigma^2) - n (log sigma + 0.5 log 2 pi),
  log r_s = log q(z_s | x, y) - log p(z_s) = sum_j (-eps_j^2/2 - logvar_j/2 + z_j^2/2);
  log_px = log mean_s exp(log w_s), elbo = mean_s log w_s, ess = (sum_s w_s)^2 / sum_s w_s^2."""
import copy
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import mesh_vae_oracle as O
from tests import update_reference as R
from tests.helpers import rel_err, seeded_state_dict
from tests.test_gpu_step_modes import _config, _net

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-4            # end to end: the fp32 device model against the fp64 oracle
EXACT = 1e-12         # a stage against float64 on the device's own inputs


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    return meshvae_b200


@pytest.fixture(scope="module")
def ops():
    from tests.helpers import OPERATORS_NPZ
    return O.load_operators(OPERATORS_NPZ)


# ---------------------------------------------------------------------------------------------------------------------
# float64 restatement (tests/test_cpu_loglik.py holds it to torch.distributions and torch.logsumexp)
# ---------------------------------------------------------------------------------------------------------------------
def sc(t):
    return -6.0 + torch.logaddexp(t + 6.0, torch.zeros_like(t))


def ref_log_r(eps, logvar, z):
    """log q(z | x, y) - log p(z) summed over the last (latent) dimension"""
    return (-0.5 * eps ** 2 - 0.5 * logvar + 0.5 * z ** 2).sum(-1)


def ref_log_pxz(recon, x, log_sigma: float):
    """log N(x; recon, sigma^2 I) summed over the last two (vertex, coordinate) dimensions"""
    n = recon.shape[-1] * recon.shape[-2]
    sse = ((recon - x) ** 2).sum((-1, -2))
    return -0.5 * sse * math.exp(-2.0 * log_sigma) - n * (log_sigma + R.LOG_2PI_HALF)


def ref_reduce(log_w):
    """log_w [B,S] -> (log_px, elbo, ess) [B]"""
    s = log_w.shape[1]
    m = log_w.max(1, keepdim=True).values
    e = torch.exp(log_w - m)
    return m[:, 0] + torch.log(e.sum(1)) - math.log(s), log_w.mean(1), e.sum(1) ** 2 / (e ** 2).sum(1)


def ref_log_w(ref, x, x_gt, y_hot, eps, log_sigma: float, chunk=256):
    """the float64 oracle (eval) on the device's samples: log_w [B,S]"""
    with torch.no_grad():
        y64 = y_hot.double().cpu()
        h = ref.encoder(x.double().cpu())
        hh = torch.cat([y64, h], -1)
        mu, lv = ref.z_mean(hh), ref.z_log_var(hh)
        e = eps.double().cpu()
        b, s, _ = e.shape
        z = mu[:, None] + torch.exp(0.5 * lv)[:, None] * e
        zin = torch.cat([y64[:, None].expand(b, s, -1), z], -1).reshape(b * s, -1)
        recon = torch.cat([ref.decoder(zin[i:i + chunk]) for i in range(0, b * s, chunk)]).reshape(b, s, x.shape[1], -1)
        return ref_log_pxz(recon, x_gt.double().cpu()[:, None], log_sigma) - ref_log_r(e, lv[:, None], z)


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _inputs(b, n, classes, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, n, 3, generator=g)
    y = torch.arange(b)[torch.randperm(b, generator=g)] % classes
    return x.to(DEV), F.one_hot(y, classes).to(DEV)


def _model(mvb, ops, cfg_name, mode, seed=7, x=None, y_hot=None):
    """the device model in a decoder sigma mode: learned s = 0.3; optimal: the sigma of one training forward"""
    net = _net(mvb, ops, _config(cfg_name, 0.0), seed)
    if mode != "fixed":
        net.set_decoder_sigma(mode, init=0.3)
    if mode == "optimal":
        net.train()
        with torch.no_grad():
            net(x, x.double(), y_hot, m_type="train", eps=torch.zeros(x.shape[0], net.z, device=DEV))
        assert net.train_log_sigma is not None
    return net


def _oracle(ops, cfg_name, seed=7):
    A, D, U, nn_ = ops
    cfg = _config(cfg_name, 0.0)
    ref = O.OracleChebVAE(3, copy.deepcopy(cfg), D, U, A, nn_)
    ref.load_state_dict(seeded_state_dict(ref, seed))
    return ref.double().eval()


def _log_sigma(net):
    return float(net._likelihood_log_sigma(None, DEV))


def _eps(b, s, z, seed):
    """the samples log_likelihood draws with generator=torch.Generator(device).manual_seed(seed)"""
    return torch.randn((b, s, z), generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV)


def _ll(net, x, x_gt, y_hot, s, chunk, seed, **kw):
    return net.log_likelihood(x, x_gt, y_hot, s, chunk, torch.Generator(device=DEV).manual_seed(seed), **kw)


def _decode(net, zcat):
    """the decoder as log_likelihood runs it -> (recon_vm, channels)"""
    recon = net.decoder(zcat)
    padded, net._recon_padded = net._recon_padded, None
    if padded is not None and recon.data_ptr() == padded.data_ptr():
        return padded, recon.shape[2]
    return recon.permute(1, 0, 2).contiguous(), None


# ---------------------------------------------------------------------------------------------------------------------
# each stage against float64 on the device's own inputs
# ---------------------------------------------------------------------------------------------------------------------
STAGES = [(b, s) for b in (1, 3, 64) for s in (1, 2, 17, 128)]


@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
@pytest.mark.parametrize("b,s", STAGES, ids=[f"B{b}-S{s}" for b, s in STAGES])
def test_stages_match_float64(mvb, ops, b, s, dt):
    Fn = mvb.functional
    net = _model(mvb, ops, "default", "fixed")
    net.eval()
    x, y_hot = _inputs(b, ops[3][0], 2, seed=b * 7 + s)
    x_gt = x.to(dt)
    with torch.no_grad():
        h = net.encoder(x)
        _, mu, lv, _, _ = Fn.vae_heads(h, y_hot, None, net.classifier_layer, net.z_mean, net.z_log_var)
        eps = _eps(b, s, net.z, seed=s)
        zcat, log_r = Fn.iw_sample(mu, lv, eps, y_hot)
        # the sampler's z is the reparameterisation kernel's, bit for bit, and its one-hot part is y
        z_rep = Fn.reparameterize(mu.repeat_interleave(s, 0), lv.repeat_interleave(s, 0), eps.reshape(b * s, -1))
        assert torch.equal(zcat[:, 2:], z_rep)
        assert torch.equal(zcat[:, :2], y_hot.float().repeat_interleave(s, 0))
        ref_r = ref_log_r(eps.double().reshape(b * s, -1), lv.double().repeat_interleave(s, 0), zcat[:, 2:].double())
        assert log_r.dtype == torch.float64 and rel_err(log_r, ref_r) <= EXACT
        # log w from the device's reconstructions, written into columns [s0, s0 + s) of a wider buffer
        recon_vm, c = _decode(net, zcat)
        ls = torch.tensor(0.37, device=DEV, dtype=torch.float64)
        s0 = 3
        log_w = torch.full((b, s + 5), 7.0, device=DEV, dtype=torch.float64)
        Fn.iw_log_weights(recon_vm, x_gt, ls, log_r, log_w, s0, c)
        recon = recon_vm[..., :3].permute(1, 0, 2).reshape(b, s, -1, 3)
        # the kernel's squared errors: differences in x_gt's precision, squares and sums in fp64
        d = (recon.to(dt) - x_gt[:, None]).double()
        sse = (d ** 2).sum((-1, -2))
        ref_w = -0.5 * sse * math.exp(-0.74) - 3 * x.shape[1] * (0.37 + R.LOG_2PI_HALF) - ref_r.reshape(b, s)
        assert rel_err(log_w[:, s0:s0 + s], ref_w) <= EXACT
        assert bool((log_w[:, :s0] == 7.0).all()) and bool((log_w[:, s0 + s:] == 7.0).all()), "columns outside the chunk"
        # the reduction, and its copy of the weights
        lw = log_w[:, s0:s0 + s].contiguous()
        log_px, elbo, ess, lw_copy = Fn.iw_reduce(lw, return_log_w=True)
        assert torch.equal(lw_copy, lw)
        for what, got, want in zip(("log_px", "elbo", "ess"), (log_px, elbo, ess), ref_reduce(lw.cpu())):
            assert got.dtype == torch.float64 and rel_err(got, want) <= EXACT, what


def test_reduce_matches_float64_on_spread_weights(mvb):
    """weights over a range of a few hundred nats (ess far below S) and S beyond a warp's lanes"""
    g = torch.Generator().manual_seed(3)
    for b, s in ((1, 1), (5, 33), (64, 128), (3, 4096)):
        lw = (-2.0e4 + 60.0 * torch.randn(b, s, generator=g, dtype=torch.float64)).to(DEV)
        got = mvb.functional.iw_reduce(lw)
        want = ref_reduce(lw.cpu())
        for what, a, r in zip(("log_px", "elbo", "ess"), got, want):
            assert rel_err(a, r) <= EXACT, (b, s, what)


# ---------------------------------------------------------------------------------------------------------------------
# end to end against the float64 oracle: same weights, same samples
# ---------------------------------------------------------------------------------------------------------------------
# (B, S, sample_chunk, x_gt dtype, sigma mode, config): every B, S, chunk, dtype and mode of the plan, both latent sizes
# (16 in the default config, 8 in the other), kept to about 2000 oracle decodes
E2E = [(1, 128, 5, torch.float64, "fixed", "default"),
       (3, 17, 5, torch.float32, "learned", "default"),
       (64, 2, 1, torch.float64, "optimal", "default"),
       (3, 1, 1, torch.float32, "fixed", "default"),
       (64, 17, 17, torch.float64, "fixed", "default"),
       (64, 1, 1, torch.float32, "learned", "orders87163_widths8_24"),
       (3, 17, 17, torch.float64, "optimal", "orders87163_widths8_24"),
       (1, 2, 2, torch.float32, "fixed", "orders87163_widths8_24"),
       (3, 128, 128, torch.float32, "learned", "orders87163_widths8_24")]


@pytest.mark.parametrize("b,s,chunk,dt,mode,cfg", E2E,
                         ids=[f"B{b}-S{s}-chunk{c}-{'x64' if d == torch.float64 else 'x32'}-{m}-{g}" for b, s, c, d, m, g in E2E])
def test_log_likelihood_matches_oracle(mvb, ops, b, s, chunk, dt, mode, cfg):
    classes = _config(cfg, 0.0)["num_classes"]
    x, y_hot = _inputs(b, ops[3][0], classes, seed=100 + b + s)
    net = _model(mvb, ops, cfg, mode, x=x, y_hot=y_hot)
    net.train()
    log_px, elbo, ess, log_w = _ll(net, x, x.to(dt), y_hot, s, chunk, seed=s, return_log_w=True)
    assert net.training, "the model's mode is restored"
    for t in (log_px, elbo, ess, log_w):
        assert t.dtype == torch.float64 and t.device == DEV
    assert tuple(log_w.shape) == (b, s) and tuple(log_px.shape) == (b,)
    ref = _oracle(ops, cfg)
    ls = _log_sigma(net)
    if mode == "fixed":
        assert ls == mvb.functional.LOG_SIGMA_DEFAULT
    elif mode == "learned":
        assert abs(ls - float(sc(torch.tensor(float(np.float32(0.3)), dtype=torch.float64)))) <= 1e-15
    else:
        assert ls == float(net.train_log_sigma)
    want_w = ref_log_w(ref, x, x.to(dt), y_hot, _eps(b, s, net.z, seed=s), ls)
    want = ref_reduce(want_w)
    for what, got, r in (("log_w", log_w, want_w), ("log_px", log_px, want[0]), ("elbo", elbo, want[1])):
        assert torch.isfinite(got).all(), what
        e = rel_err(got, r)
        assert e < TOL, f"{what}: rel_err {e:.3e}"
    assert bool((ess >= 1.0 - 1e-12).all()) and bool((ess <= s * (1.0 + 1e-12)).all())


# ---------------------------------------------------------------------------------------------------------------------
# identities
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [torch.float32, torch.float64], ids=["x32", "x64"])
@pytest.mark.parametrize("mode", ["learned", "fixed"])
def test_zero_noise_single_sample_is_the_loss_epilogue(mvb, ops, mode, dt):
    """eps = 0, S = 1: log w_b = -rec_b - sum_j (-logvar_j/2 + mu_j^2/2) with rec_b from the loss epilogue at z = mu, on
    the same decoder bits.  Bounds: 1e-12 relative where the epilogue's rec is fp64 arithmetic on the same squared
    errors (the sigma-VAE epilogue, learned sigma, fp64 x_gt).  The constant-sigma epilogue uses sigma = expf(log sigma)
    rounded to fp32 (sigma^-2 off by up to 2.4e-7 relative) and, with fp32 x_gt, fp32 NLL terms; with fp32 x_gt rec is
    returned in fp32 (6e-8 relative): there the bound is 1e-6 of |rec|."""
    Fn = mvb.functional
    b = 64
    x, y_hot = _inputs(b, ops[3][0], 2, seed=21)
    x_gt = x.to(dt)
    net = _model(mvb, ops, "default", mode)
    net.eval()
    with torch.no_grad():
        _, _, _, (kld, rec, z_), _ = net(x, x_gt, y_hot, m_type="test")
        h = net.encoder(x)
        _, mu, lv, _, _ = Fn.vae_heads(h, y_hot, None, net.classifier_layer, net.z_mean, net.z_log_var)
        zcat, log_r = Fn.iw_sample(mu, lv, torch.zeros(b, 1, net.z, device=DEV), y_hot)
        assert torch.equal(zcat[:, 2:], z_), "z = mu at eps = 0"
        recon_vm, c = _decode(net, zcat)
        log_w = torch.empty(b, 1, device=DEV, dtype=torch.float64)
        Fn.iw_log_weights(recon_vm, x_gt, net._likelihood_log_sigma(None, DEV), log_r, log_w, 0, c)
    want = -rec.double().cpu() - (-0.5 * lv.double() + 0.5 * mu.double() ** 2).sum(-1).cpu()
    got = log_w[:, 0].cpu()
    exact = mode == "learned" and dt == torch.float64
    bound = (EXACT * want.abs()) if exact else (1e-6 * rec.double().abs().cpu())
    assert bool(((got - want).abs() <= bound).all()), float(((got - want).abs() / want.abs()).max())


def test_single_sample_and_jensen(mvb, ops):
    b = 64
    x, y_hot = _inputs(b, ops[3][0], 2, seed=22)
    net = _model(mvb, ops, "default", "fixed")
    log_px, elbo, ess, log_w = _ll(net, x, x.double(), y_hot, 1, None, seed=1, return_log_w=True)
    assert torch.equal(log_px, log_w[:, 0]) and torch.equal(elbo, log_w[:, 0])
    assert torch.equal(ess, torch.ones_like(ess))
    for s in (2, 17, 128):
        log_px, elbo, ess = _ll(net, x, x.double(), y_hot, s, 32, seed=s)
        assert bool((log_px >= elbo).all()), s
        assert bool((ess >= 1.0 - 1e-12).all()) and bool((ess <= s * (1.0 + 1e-12)).all())


def test_explicit_log_sigma_reproduces_the_modes(mvb, ops):
    b, s = 3, 17
    x, y_hot = _inputs(b, ops[3][0], 2, seed=23)
    net = _model(mvb, ops, "default", "fixed")
    fixed = _ll(net, x, x.double(), y_hot, s, 5, seed=9)
    for explicit in (mvb.functional.LOG_SIGMA_DEFAULT,
                     torch.tensor([mvb.functional.LOG_SIGMA_DEFAULT], device=DEV, dtype=torch.float32)):
        got = _ll(net, x, x.double(), y_hot, s, 5, seed=9, log_sigma=explicit)
        assert all(torch.equal(a, c) for a, c in zip(fixed, got))
    # an explicit value overrides a mode; "learned" agrees with its own sc(s) passed explicitly
    net.set_decoder_sigma("learned", init=0.3)
    learned = _ll(net, x, x.double(), y_hot, s, 5, seed=9)
    got = _ll(net, x, x.double(), y_hot, s, 5, seed=9, log_sigma=net._likelihood_log_sigma(None, DEV))
    assert all(torch.equal(a, c) for a, c in zip(learned, got))
    other = _ll(net, x, x.double(), y_hot, s, 5, seed=9, log_sigma=mvb.functional.LOG_SIGMA_DEFAULT)
    assert all(torch.equal(a, c) for a, c in zip(fixed, other))


def test_optimal_sigma_is_that_of_the_training_step(mvb, ops):
    """an evaluation forward (what loop.evaluate runs on every test batch) fits the optimal sigma to its own batch and
    leaves it in last_log_sigma; log_likelihood keeps scoring with the sigma of the last training step, on the evaluated
    meshes too"""
    b, s, n = 3, 17, ops[3][0]
    x, y_hot = _inputs(b, n, 2, seed=30)
    net = _model(mvb, ops, "default", "optimal", x=x, y_hot=y_hot)
    trained = float(net.train_log_sigma)
    assert float(net._likelihood_log_sigma(None, DEV)) == trained
    x2, y2 = _inputs(b, n, 2, seed=31)
    x2 = 3.0 * x2
    before = [_ll(net, xx, xx.double(), yy, s, 5, seed=3) for xx, yy in ((x, y_hot), (x2, y2))]
    net.eval()
    with torch.no_grad():
        net(x2, x2.double(), y2, m_type="test")
    assert float(net.last_log_sigma) != trained, "the evaluation forward fitted a sigma of its own"
    assert float(net.train_log_sigma) == trained and float(net._likelihood_log_sigma(None, DEV)) == trained
    after = [_ll(net, xx, xx.double(), yy, s, 5, seed=3) for xx, yy in ((x, y_hot), (x2, y2))]
    for u, v in zip(before, after):
        assert all(torch.equal(p, q) for p, q in zip(u, v))


def test_engine_step_sets_the_optimal_sigma(mvb, ops):
    """the captured training step's optimal sigma is the one log_likelihood reads, after an evaluation forward too"""
    from meshvae_b200.engine import TrainEngine
    from tests.test_gpu_step_modes import _batch
    cfg = _config("default", 0.0)
    b, n = 16, ops[3][0]
    net = _net(mvb, ops, cfg)
    net.set_decoder_sigma("optimal")
    eng = TrainEngine(net, b)
    eng.capture(warmup=1)
    seen = set()
    for step in range(2):
        x, y, eps = _batch(b, n, cfg["num_classes"], cfg["num_style"], 300 + step)
        eng.step(x.pin_memory(), x.double().pin_memory(), y.pin_memory(), eps_host=eps.pin_memory())
        torch.cuda.synchronize()
        assert float(net._likelihood_log_sigma(None, DEV)) == float(eng.log_sigma)
        seen.add(float(eng.log_sigma))
    assert len(seen) == 2, "the sigma follows the training steps"
    x2, y2 = _inputs(b, n, 2, seed=32)
    net.eval()
    with torch.no_grad():
        net(3.0 * x2, 3.0 * x2.double(), y2, m_type="test")
    assert float(net._likelihood_log_sigma(None, DEV)) == float(eng.log_sigma)


# ---------------------------------------------------------------------------------------------------------------------
# statistics of the sampler
# ---------------------------------------------------------------------------------------------------------------------
def test_mean_log_r_is_the_analytic_kld(mvb, ops):
    """E_q[log q(z) - log p(z)] = KL(q || p): the sample mean of log r over S = 4096 draws lies within 5 standard errors of
    the kld of the loss epilogue"""
    Fn = mvb.functional
    b, s = 3, 4096
    x, y_hot = _inputs(b, ops[3][0], 2, seed=24)
    net = _model(mvb, ops, "default", "fixed")
    net.eval()
    with torch.no_grad():
        _, _, _, (kld, _, _), _ = net(x, x.double(), y_hot, m_type="test")
        h = net.encoder(x)
        _, mu, lv, _, _ = Fn.vae_heads(h, y_hot, None, net.classifier_layer, net.z_mean, net.z_log_var)
        _, log_r = Fn.iw_sample(mu, lv, _eps(b, s, net.z, seed=2024), y_hot)
    lr = log_r.reshape(b, s).cpu()
    mean, se = lr.mean(1), lr.std(1) / math.sqrt(s)
    k = kld.double().cpu()
    assert bool(((mean - k).abs() <= 5.0 * se).all()), (mean, k, se)


# ---------------------------------------------------------------------------------------------------------------------
# launch behaviour
# ---------------------------------------------------------------------------------------------------------------------
def test_same_bits_every_run_and_chunks_agree(mvb, ops):
    b, s = 64, 128
    x, y_hot = _inputs(b, ops[3][0], 2, seed=25)
    net = _model(mvb, ops, "default", "fixed")
    a = _ll(net, x, x.double(), y_hot, s, 32, seed=4, return_log_w=True)
    again = _ll(net, x, x.double(), y_hot, s, 32, seed=4, return_log_w=True)
    assert all(torch.equal(u, v) for u, v in zip(a, again))
    for chunk in (1, 5, None):
        other = _ll(net, x, x.double(), y_hot, s, chunk, seed=4, return_log_w=True)
        for what, u, v in zip(("log_px", "elbo", "ess", "log_w"), a, other):
            if what != "ess":
                assert rel_err(v, u) < TOL, (chunk, what)


def test_captured_call_replays_the_eager_bits(mvb, ops):
    b, s, chunk = 3, 17, 5
    x, y_hot = _inputs(b, ops[3][0], 2, seed=26)
    x_gt = x.double()
    net = _model(mvb, ops, "default", "learned")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        net.log_likelihood(x, x_gt, y_hot, s, chunk)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = net.log_likelihood(x, x_gt, y_hot, s, chunk, return_log_w=True)
    seen = set()
    for seed in (5, 6):
        torch.cuda.manual_seed(seed)
        g.replay()
        torch.cuda.synchronize()
        torch.cuda.manual_seed(seed)
        eager = net.log_likelihood(x, x_gt, y_hot, s, chunk, return_log_w=True)
        torch.cuda.synchronize()
        assert all(torch.equal(u, v) for u, v in zip(out, eager)), seed
        seen.add(float(out[0][0]))
    assert len(seen) == 2, "the replays drew the same samples"
    # the learned sigma is read on the device at every replay
    with torch.no_grad():
        net.log_sigma.fill_(-0.4)
    torch.cuda.manual_seed(5)
    g.replay()
    torch.cuda.manual_seed(5)
    eager = net.log_likelihood(x, x_gt, y_hot, s, chunk, return_log_w=True)
    torch.cuda.synchronize()
    assert all(torch.equal(u, v) for u, v in zip(out, eager))


def test_eager_call_never_synchronises(mvb, ops):
    b, s = 3, 17
    x, y_hot = _inputs(b, ops[3][0], 2, seed=27)
    net = _model(mvb, ops, "default", "learned")
    gen = torch.Generator(device=DEV).manual_seed(1)
    net.log_likelihood(x, x.double(), y_hot, s, 5, gen)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = net.log_likelihood(x, x.double(), y_hot, s, 5, gen)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(t).all()) for t in out)


def test_loop_log_likelihood(mvb, ops):
    """loop.log_likelihood over a loader of the evaluate kind: the per-mesh values of the model call on each batch (one
    generator across the batches), their means and the names in loader order"""
    n = ops[3][0]
    g = torch.Generator().manual_seed(28)
    batches = []
    for i, b in enumerate((4, 3)):
        x = torch.randn(b, n, 3, generator=g)
        y = torch.arange(b) % 2
        batches.append((x, x.double(), y, [f"m{i}_{k}.obj" for k in range(b)], None, None, None, None))
    net = _model(mvb, ops, "default", "fixed")
    res = mvb.loop.log_likelihood(net, batches, DEV, 9, sample_chunk=4, seed=3)
    gen = torch.Generator(device=DEV).manual_seed(3)
    want = [net.log_likelihood(bt[0].to(DEV), bt[1].to(DEV), F.one_hot(bt[2], 2).to(DEV), 9, 4, gen) for bt in batches]
    for i, k in enumerate(("log_px", "elbo", "ess")):
        w = torch.cat([t[i] for t in want]).cpu().numpy()
        assert res[k].dtype == np.float64 and np.array_equal(res[k], w), k
        assert res[k + "_mean"] == float(w.mean())
    assert res["names"] == [f"m{i}_{k}.obj" for i, b in enumerate((4, 3)) for k in range(b)]


# ---------------------------------------------------------------------------------------------------------------------
# errors
# ---------------------------------------------------------------------------------------------------------------------
def test_errors(mvb, ops):
    Err = mvb.MvbError
    b = 3
    x, y_hot = _inputs(b, ops[3][0], 2, seed=29)
    net = _model(mvb, ops, "default", "fixed")
    for s, chunk in ((0, None), (-1, None), (4, 0)):
        with pytest.raises(Err):
            net.log_likelihood(x, x.double(), y_hot, s, chunk)
    with pytest.raises(Err):
        net.log_likelihood(x, x.double()[:, :-1], y_hot, 4)            # ground truth of another mesh size
    with pytest.raises(Err):
        net.log_likelihood(x, x.double()[:2], y_hot, 4)                # another batch
    with pytest.raises(Err):
        net.log_likelihood(x, x.double(), F.one_hot(torch.arange(b) % 3, 3).to(DEV), 4)     # another number of classes
    with pytest.raises(Err):
        net.log_likelihood(x, x.double(), y_hot, 4, log_sigma=torch.zeros(2, device=DEV))
    with pytest.raises(Err):
        net.log_likelihood(x.cpu(), x.double(), y_hot, 4)
    with pytest.raises(Err):
        net.log_likelihood(x, x.double().cpu(), y_hot, 4)
    with pytest.raises(Err):
        net.log_likelihood(x, x.double(), y_hot, 4, log_sigma=torch.tensor(0.5))
    net.set_decoder_sigma("optimal")
    with pytest.raises(Err, match="optimal"):
        net.log_likelihood(x, x.double(), y_hot, 4)
    net.log_likelihood(x, x.double(), y_hot, 4, log_sigma=0.5)          # an explicit sigma is enough
    Fn = mvb.functional
    mu, lv = torch.zeros(b, 16, device=DEV), torch.zeros(b, 16, device=DEV)
    with pytest.raises(Err):
        Fn.iw_sample(mu, lv, torch.zeros(b, 2, 8, device=DEV), y_hot)
    with pytest.raises(Err):
        Fn.iw_sample(mu, lv, torch.zeros(b, 0, 16, device=DEV), y_hot)
    with pytest.raises(Err):
        Fn.iw_sample(mu.cpu(), lv.cpu(), torch.zeros(b, 2, 16), y_hot.cpu())
    log_r = torch.zeros(b * 2, device=DEV, dtype=torch.float64)
    recon = torch.zeros(20, b * 2, 3, device=DEV)
    ls = torch.zeros((), device=DEV, dtype=torch.float64)
    with pytest.raises(Err):
        Fn.iw_log_weights(recon, torch.zeros(b, 20, 3, device=DEV), ls, log_r, torch.zeros(b, 3, device=DEV, dtype=torch.float64), 2)
    with pytest.raises(Err):
        Fn.iw_log_weights(recon, torch.zeros(b, 21, 3, device=DEV), ls, log_r, torch.zeros(b, 2, device=DEV, dtype=torch.float64))
    with pytest.raises(Err):
        Fn.iw_reduce(torch.zeros(b, 2, device=DEV))
