"""CPU checks of the importance-weighted log-likelihood estimate (tests/test_gpu_loglik.py holds the kernels to these): the
float64 restatement of log r, log p(x | z) and the reduction against torch.distributions.Normal.log_prob sums and
torch.logsumexp, and the refusals that need no GPU."""
import copy
import math

import pytest
import torch
from torch.distributions import Normal

import meshvae_b200 as mvb
from meshvae_b200 import _lib
from oracle import mesh_vae_oracle as O
from tests.helpers import OPERATORS_NPZ
from tests.test_gpu_loglik import ref_log_pxz, ref_log_r, ref_reduce, sc


def test_log_r_is_log_q_minus_log_p():
    """sum_j (-eps^2/2 - logvar/2 + z^2/2) = log N(z; mu, exp(logvar)) - log N(z; 0, 1), z = mu + exp(logvar/2) eps"""
    g = torch.Generator().manual_seed(1)
    b, s, zd = 4, 9, 16
    mu = torch.randn(b, 1, zd, generator=g, dtype=torch.float64)
    lv = 0.7 * torch.randn(b, 1, zd, generator=g, dtype=torch.float64)
    eps = torch.randn(b, s, zd, generator=g, dtype=torch.float64)
    z = mu + torch.exp(0.5 * lv) * eps
    want = Normal(mu, torch.exp(0.5 * lv)).log_prob(z).sum(-1) - Normal(0.0, 1.0).log_prob(z).sum(-1)
    got = ref_log_r(eps, lv, z)
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)


def test_log_pxz_is_the_gaussian_decoder_density():
    g = torch.Generator().manual_seed(2)
    b, s, n = 3, 5, 79
    recon = torch.randn(b, s, n, 3, generator=g, dtype=torch.float64)
    x = torch.randn(b, 1, n, 3, generator=g, dtype=torch.float64)
    for ls in (-1.3, 0.0, mvb.functional.LOG_SIGMA_DEFAULT):
        want = Normal(recon, math.exp(ls)).log_prob(x.expand_as(recon)).sum((-1, -2))
        assert torch.allclose(ref_log_pxz(recon, x, ls), want, rtol=1e-12, atol=0)


def test_reduction_is_logsumexp():
    g = torch.Generator().manual_seed(3)
    for b, s in ((1, 1), (3, 2), (5, 17), (2, 4096)):
        lw = -3.0e4 + 40.0 * torch.randn(b, s, generator=g, dtype=torch.float64)
        log_px, elbo, ess = ref_reduce(lw)
        assert torch.allclose(log_px, torch.logsumexp(lw, 1) - math.log(s), rtol=1e-14, atol=0)
        assert torch.allclose(elbo, lw.mean(1), rtol=1e-14, atol=0)
        w = torch.exp(lw - lw.max(1, keepdim=True).values)
        assert torch.allclose(ess, torch.exp(2 * torch.logsumexp(lw, 1) - torch.logsumexp(2 * lw, 1)), rtol=1e-10, atol=0)
        assert torch.allclose(ess, w.sum(1) ** 2 / (w ** 2).sum(1), rtol=1e-14, atol=0)
        assert bool((log_px >= elbo - 1e-9).all())
        if s == 1:
            assert torch.equal(log_px, lw[:, 0]) and torch.equal(ess, torch.ones(b, dtype=torch.float64))


def test_learned_log_sigma_restatement_is_the_softclip():
    t = torch.tensor([-40.0, -6.0, 0.3, 25.0], dtype=torch.float64)
    assert torch.allclose(sc(t), O.softclip(t, -6), rtol=1e-14, atol=0)


def test_log_likelihood_has_no_cpu_path():
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    net = mvb.cheb_VAE(3, cfg, D, U, A, nn_, model=cfg["model"])
    x = torch.randn(2, nn_[0], 3)
    y = torch.eye(2, dtype=torch.int64)
    with pytest.raises(mvb.MvbError):
        net.log_likelihood(x, x.double(), y, 4)
    Fn = mvb.functional
    with pytest.raises(mvb.MvbError):
        Fn.iw_sample(torch.zeros(2, 16), torch.zeros(2, 16), torch.zeros(2, 3, 16), y)
    with pytest.raises(mvb.MvbError):
        Fn.iw_log_weights(torch.zeros(20, 6, 3), torch.zeros(2, 20, 3), torch.zeros((), dtype=torch.float64),
                          torch.zeros(6, dtype=torch.float64), torch.zeros(2, 3, dtype=torch.float64))
    with pytest.raises(mvb.MvbError):
        Fn.iw_reduce(torch.zeros(2, 3, dtype=torch.float64))


def test_log_weights_refuse_more_reconstructions_than_one_launch_covers():
    """the SSE partial kernel tiles the B*S reconstructions 32 at a time over grid.y (at most 65535 tiles): beyond
    2097120 per call the entry point says so (MVB_EINVAL) before any launch; at the limit it goes on to the workspace
    check (MVB_EWORKSPACE with an empty one) - dummy pointers, nothing is launched either way"""
    p = 256
    rc = _lib.lib.mvb_iw_log_weights(64, 32769, 4998, 3, p, 4, p, 1, p, p, 32769, 0, p, p, 0, None)
    assert rc == -1 and "at most 2097120" in _lib.last_error(), _lib.last_error()
    rc = _lib.lib.mvb_iw_log_weights(32, 65535, 4998, 3, p, 4, p, 1, p, p, 65535, 0, p, p, 0, None)
    assert rc == -4, _lib.last_error()
