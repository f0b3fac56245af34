"""CPU checks of the sigma-VAE decoder variances (tests/test_gpu_loss_sigma.py holds the kernels to these): the float64
restatement of the loss against the sigma-VAE's own torch expressions, the model's sigma modes and state-dict contract,
and the training engine's refusal of the optimal sigma under data parallelism."""
import copy
import math

import pytest
import torch
import torch.nn.functional as F

import meshvae_b200 as mvb
from oracle import mesh_vae_oracle as O
from tests.helpers import OPERATORS_NPZ
from tests.test_gpu_loss_sigma import ref_sigma_loss, sc


def _net():
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    return mvb.cheb_VAE(3, cfg, D, U, A, nn_, model=cfg["model"])


@pytest.mark.parametrize("mode", ["optimal", "learned"])
def test_float64_restatement_is_the_sigma_vae_loss(mode):
    """ref_sigma_loss against the sigma-VAE code's form: softclip(log_sigma, -6), gaussian_nll(...).sum(-1).sum(-1) and
    (optimal) log_sigma = ((x - mu)**2).mean().sqrt().log() - values and gradients"""
    g = torch.Generator().manual_seed(1)
    b, n, c = 5, 79, 3
    recon = torch.randn(b, n, c, generator=g)
    x = recon.double() + 0.4 * torch.randn(b, n, c, generator=g, dtype=torch.float64)
    mu, lv = torch.randn(b, 16, generator=g), 0.5 * torch.randn(b, 16, generator=g)
    y = F.one_hot(torch.randint(0, 2, (b,), generator=g), 2)
    y_hat = torch.softmax(torch.randn(b, 2, generator=g), 1)
    ref = ref_sigma_loss(recon, x, mu, lv, y_hat, y, mode, s=0.3)
    r, m, l, yh = (t.double().requires_grad_() for t in (recon, mu, lv, y_hat))
    s = torch.tensor([0.3], dtype=torch.float32).double().requires_grad_()
    raw = ((x - r) ** 2).mean().sqrt().log() if mode == "optimal" else s
    ls = O.softclip(raw, -6)
    rec = O.gaussian_nll(r, ls, x).sum(-1).sum(-1)
    loss = (O.kld(m, l) + rec - 2 * (yh * y).sum(-1).log()).mean()
    (0.375 * loss).backward()
    assert torch.allclose(ref["loss"], loss.detach(), rtol=1e-13, atol=0)
    assert torch.allclose(ref["rec"], rec.detach(), rtol=1e-13, atol=0)
    assert torch.allclose(ref["log_sigma"], ls.detach().reshape(()), rtol=1e-13, atol=0)
    for k, t in (("d_recon", r), ("d_mu", m), ("d_logvar", l), ("d_yhat", yh)):
        assert torch.allclose(ref[k], t.grad, rtol=1e-10, atol=1e-13), k
    if mode == "learned":
        assert torch.allclose(ref["d_s"], s.grad.reshape(()), rtol=1e-10, atol=0)
    assert float(sc(torch.tensor(-math.inf, dtype=torch.float64))) == -6.0


def test_decoder_sigma_modes_and_state_dict():
    net = _net()
    keys = set(net.state_dict())
    assert net.sigma_mode == "fixed" and net.log_sigma == mvb.functional.LOG_SIGMA_DEFAULT
    net.set_decoder_sigma("optimal")
    assert net.log_sigma == "optimal" and set(net.state_dict()) == keys
    net.set_decoder_sigma("learned", init=0.5)
    assert set(net.state_dict()) == keys | {"log_sigma"}
    assert isinstance(net.log_sigma, torch.nn.Parameter) and net.log_sigma.shape == () and float(net.log_sigma.detach()) == 0.5
    assert any(p is net.log_sigma for p in net.parameters())
    net.set_decoder_sigma("fixed")
    assert set(net.state_dict()) == keys and net.log_sigma == mvb.functional.LOG_SIGMA_DEFAULT
    with pytest.raises(ValueError):
        net.set_decoder_sigma("optimal_sigma_VAE")


def test_engine_rejects_optimal_sigma_with_data_parallelism(monkeypatch):
    from meshvae_b200 import engine
    net = _net()
    net.set_decoder_sigma("optimal")
    monkeypatch.setattr(engine.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(engine.dist, "get_world_size", lambda: 2)
    with pytest.raises(mvb.MvbError, match="optimal decoder sigma"):
        engine.TrainEngine(net, 4)


def test_sigma_paths_have_no_cpu_fallback():
    r, x = torch.randn(20, 2, 3), torch.randn(2, 20, 3)
    mu, lv, yh, y = torch.randn(2, 16), torch.randn(2, 16), torch.full((2, 2), 0.5), torch.eye(2, dtype=torch.int64)
    with pytest.raises(mvb.MvbError):
        mvb.functional.vae_loss(r, x, mu, lv, yh, y, log_sigma="optimal")
    with pytest.raises(mvb.MvbError):
        mvb.functional.vae_loss(r, x, mu, lv, yh, y, log_sigma="learned")
    with pytest.raises(mvb.MvbError):
        mvb.logpdf.gaussian_nll(torch.randn(4), torch.zeros(1, requires_grad=True), torch.randn(4))
