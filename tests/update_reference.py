"""Plain float64 restatements of the rest of the training step, for the kernel tests of tests/test_gpu_update_path.py:

- the loss of models/cheb_VAE.py:321-346 (KLD, Gaussian NLL with softclip(1, -6), the log sum(y_hat * y) term, `correct`
  with torch's first-index argmax) and its gradients;
- Linear + ReLU + inverted dropout (forward, and dW / db / dx from the forward output, as mvb_linear_bwd defines them);
- one Adam step exactly as torch.optim.Adam (single-tensor, L2-style weight decay) writes it, hyper-parameters as Python
  doubles;
- the rank-order gradient sum of the fused data-parallel update, followed by that Adam step.

Everything runs on the CPU in float64 (the gradient sum excepted: it is the fp32 rank-order sum the kernel must reproduce
bit for bit).  tests/test_cpu_update_reference.py pins these restatements to the oracle and to torch."""
import math

import torch

LOG_2PI_HALF = 0.5 * math.log(2.0 * math.pi)


def _d(t):
    return t.detach().to("cpu", torch.float64)


def loss_sigma(log_sigma: float) -> float:
    """sigma as the reference model computes it: log_sigma.exp() on an fp32 tensor (models/cheb_VAE.py:328-329), then
    promoted to float64 by the fp64 ground truth"""
    return float(torch.tensor(log_sigma, dtype=torch.float32).exp())


def vae_loss(recon, x, mu, logvar, y_hat, y, log_sigma: float):
    """recon, x [B,N,C] (recon mesh-major here); mu / logvar [B,Z]; y_hat [B,ncls]; y [B,ncls] one-hot.
    -> dict(loss, kld[B], rec[B], correct) in float64 (correct an int)"""
    r, xx, m, lv, yh, yy = _d(recon), _d(x), _d(mu), _d(logvar), _d(y_hat), _d(y)
    ls = float(torch.tensor(log_sigma, dtype=torch.float32))
    sigma = loss_sigma(log_sigma)
    kld = -0.5 * (1.0 + lv - m * m - lv.exp()).sum(-1)
    rec = (0.5 * ((xx - r) / sigma) ** 2 + ls + LOG_2PI_HALF).sum(-1).sum(-1)
    logqy = (yh * yy).sum(-1).log()
    loss = (kld + rec - 2.0 * logqy).mean()
    correct = int((torch.argmax(_d(y_hat), 1) == torch.argmax(_d(y), 1)).sum())
    return {"loss": loss, "kld": kld, "rec": rec, "correct": correct}


def vae_loss_grads(recon, x, mu, logvar, y_hat, y, log_sigma: float, gloss: float = 1.0):
    """gradients of gloss * loss: d_recon [B,N,C], d_mu, d_logvar [B,Z], d_yhat [B,ncls] (float64)"""
    r, xx, m, lv, yh, yy = _d(recon), _d(x), _d(mu), _d(logvar), _d(y_hat), _d(y)
    sigma = loss_sigma(log_sigma)
    s = gloss / r.shape[0]
    q = (yh * yy).sum(-1, keepdim=True)
    return {"d_recon": s * (r - xx) / (sigma * sigma), "d_mu": s * m, "d_logvar": s * 0.5 * (lv.exp() - 1.0),
            "d_yhat": s * (-2.0) * yy / q}


def linear_fwd(x, w, b=None, relu: bool = False, keep=None, p: float = 0.0):
    """y = dropout_p(relu?(x W^T + b)); x [M,K], w [N,K], keep [M,N] bool (None: no dropout)"""
    y = _d(x) @ _d(w).t()
    if b is not None:
        y = y + _d(b)
    if relu:
        y = y.clamp_min(0.0)
    if keep is not None:
        y = y * torch.as_tensor(keep, dtype=torch.float64) / (1.0 - p)
    return y


def linear_bwd(x, w, y, gy, relu: bool = False, p: float = 0.0):
    """-> (dx, dW, db) for gp = gy * [y > 0] / (1 - p) (relu; y the forward OUTPUT, whose zeros are the clamped and the
    dropped units) or gp = gy"""
    g = _d(gy)
    if relu:
        g = g * (_d(y) > 0).to(torch.float64) / (1.0 - p)
    return g @ _d(w), g.t() @ _d(x), g.sum(0)


def adam_step(p, g, m, v, step: int, lr: float, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
              grad_scale: float = 1.0):
    """one step of torch.optim.Adam (_single_tensor_adam, amsgrad off) on the gradient grad_scale * g; `step` is the
    counter AFTER its increment (1 on the first step).  -> (p, m, v) float64"""
    p, g, m, v = _d(p), _d(g) * grad_scale, _d(m), _d(v)
    b1, b2 = float(betas[0]), float(betas[1])
    if weight_decay != 0:
        g = g + weight_decay * p
    m = m + (1.0 - b1) * (g - m)                       # exp_avg.lerp_(grad, 1 - beta1)
    v = v * b2 + (1.0 - b2) * (g * g)                  # exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    denom = v.sqrt() / math.sqrt(bc2) + eps
    return p - (lr / bc1) * (m / denom), m, v


def rank_order_sum(grads):
    """the fp32 sum g0 + g1 + ... in rank order, as every rank of the fused data-parallel update forms it"""
    s = grads[0].clone()
    for g in grads[1:]:
        s += g
    return s


def dp_reduce_adam(p, grads, m, v, step: int, lr: float, betas, eps: float, weight_decay: float, grad_scale: float):
    """the rank-order sum of the ranks' gradients followed by one Adam step -> (p, m, v, grad_sum)"""
    gs = rank_order_sum([g.detach().cpu() for g in grads])
    return (*adam_step(p, gs, m, v, step, lr, betas, eps, weight_decay, grad_scale), gs)
