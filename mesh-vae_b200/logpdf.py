"""Drop-in for the three logpdf.py functions on the hot path (logpdf.py:7-8 KLD, :22-23
gaussian_nll, :24-28 softclip), backed by CUDA kernels.  The fused loss epilogue used by the model
mirror is `functional.vae_loss`; these exist so the reference's own `loss_function`
(models/cheb_VAE.py:321-346) runs unchanged."""
import torch
import torch.nn.functional as F

from . import functional as Fn


def KLD(mu, logvar):
    return Fn.kld(mu, logvar)


def softclip(tensor, min):  # noqa: A002  (reference signature)
    """min + softplus(tensor - min) on a 1-element tensor: init-grade arithmetic, left to torch."""
    return min + F.softplus(tensor - min)


def gaussian_nll(mu, log_sigma, x):
    """0.5 ((x - mu)/exp(log_sigma))^2 + log_sigma + 0.5 log(2 pi); log_sigma is a 1-element tensor: the constant of
    models/cheb_VAE.py:328-329, or a sigma-VAE log sigma (a parameter, or the optimal
    softclip(((x - mu)**2).mean().sqrt().log(), -6)) through which the gradient flows.  A CUDA log_sigma is read on the
    device (no host synchronisation); a constant host one is passed by value as before."""
    if isinstance(log_sigma, torch.Tensor):
        if log_sigma.numel() != 1:
            raise ValueError(f"gaussian_nll: log_sigma must have one element, got {tuple(log_sigma.shape)}")
        if log_sigma.is_cuda or log_sigma.requires_grad:
            log_sigma = log_sigma.to(mu.device)
        else:
            log_sigma = float(log_sigma)
    mu_b, x_b = torch.broadcast_tensors(mu, x)
    return Fn.gaussian_nll(mu_b, x_b, log_sigma)
