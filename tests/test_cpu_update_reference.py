"""The float64 restatements of tests/update_reference.py pinned on the CPU: the loss against the oracle's loss function
(models/cheb_VAE.py:321-346) and its autograd, the Adam step against torch.optim.Adam, the dense layer against
F.linear.  All in float64, so every bound here is 1e-12."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import mesh_vae_oracle as O
from tests import update_reference as R
from tests.helpers import rel_err

LOG_SIGMA = float(O.softclip(torch.Tensor([1]), -6))


def _loss_inputs(b, n, c, z, ncls, seed):
    g = torch.Generator().manual_seed(seed)
    recon = torch.randn(b, n, c, generator=g, dtype=torch.float64)
    x = torch.randn(b, n, c, generator=g, dtype=torch.float64)
    mu, lv = torch.randn(b, z, generator=g, dtype=torch.float64), 0.3 * torch.randn(b, z, generator=g, dtype=torch.float64)
    y_hat = torch.softmax(torch.randn(b, ncls, generator=g, dtype=torch.float64), 1)
    y = F.one_hot(torch.randint(0, ncls, (b,), generator=g), ncls)
    return recon, x, mu, lv, y_hat, y


def test_loss_matches_oracle_loss_function():
    for b, n, c, z, ncls in [(5, 33, 3, 16, 2), (9, 7, 6, 17, 10), (1, 1, 1, 1, 1)]:
        recon, x, mu, lv, y_hat, y = _loss_inputs(b, n, c, z, ncls, seed=b + n)
        # the oracle's loss_function (only `self` is unused in it)
        leaves = [t.clone().requires_grad_() for t in (recon, mu, lv, y_hat)]
        lo, co, ko, ro = O.OracleChebVAE.loss_function(None, x, leaves[0], leaves[1], leaves[2], y, leaves[3])
        (0.37 * lo).backward()
        got = R.vae_loss(recon, x, mu, lv, y_hat, y, LOG_SIGMA)
        assert rel_err(got["loss"], lo) < 1e-12 and rel_err(got["kld"], ko) < 1e-12 and rel_err(got["rec"], ro) < 1e-12
        assert got["correct"] == int(co)
        gr = R.vae_loss_grads(recon, x, mu, lv, y_hat, y, LOG_SIGMA, gloss=0.37)
        for name, leaf in zip(("d_recon", "d_mu", "d_logvar", "d_yhat"), leaves):
            assert rel_err(gr[name], leaf.grad) < 1e-12, name


def test_loss_correct_takes_the_first_maximum():
    """ties in y_hat: torch.argmax returns the first maximal index, and so must the restatement"""
    y_hat = torch.tensor([[0.25, 0.25, 0.5, 0.5], [0.5, 0.5, 0.0, 0.0], [0.25, 0.25, 0.25, 0.25]], dtype=torch.float64)
    y = F.one_hot(torch.tensor([3, 0, 3]), 4)
    got = R.vae_loss(torch.zeros(3, 1, 1), torch.zeros(3, 1, 1), torch.zeros(3, 2), torch.zeros(3, 2), y_hat, y, LOG_SIGMA)
    assert got["correct"] == 1          # row 0 predicts class 2 (first of the tie), row 1 class 0, row 2 class 0


def test_adam_step_matches_torch_adam_over_50_steps():
    """torch.optim.Adam on float64 parameters with weight decay, betas (0.5, 0.9), a gradient scale folded in, and the
    learning rate changed mid-run"""
    g = torch.Generator().manual_seed(0)
    shapes = [(7, 5), (3,), (1,)]
    params = [torch.randn(*s, generator=g, dtype=torch.float64).requires_grad_() for s in shapes]
    opt = torch.optim.Adam(params, lr=3e-3, betas=(0.5, 0.9), eps=1e-6, weight_decay=0.1, foreach=False)
    state = [(p.detach().clone(), torch.zeros_like(p), torch.zeros_like(p)) for p in params]
    scale = 1.0 / 3.0
    for step in range(1, 51):
        if step == 20:
            opt.param_groups[0]["lr"] = 1e-2
        lr = opt.param_groups[0]["lr"]
        grads = [torch.randn(*s, generator=g, dtype=torch.float64) for s in shapes]
        for p, gr in zip(params, grads):
            p.grad = gr * scale
        opt.step()
        state = [R.adam_step(p, gr, m, v, step, lr, (0.5, 0.9), 1e-6, 0.1, scale) for (p, m, v), gr in zip(state, grads)]
        for p, (pr, mr, vr) in zip(params, state):
            st = opt.state[p]
            assert rel_err(pr, p) < 1e-12 and rel_err(mr, st["exp_avg"]) < 1e-12 and rel_err(vr, st["exp_avg_sq"]) < 1e-12


def test_linear_matches_f_linear():
    g = torch.Generator().manual_seed(1)
    m, k, n, p = 37, 29, 11, 0.2
    x, w, b = (torch.randn(*s, generator=g, dtype=torch.float64) for s in ((m, k), (n, k), (n,)))
    gy = torch.randn(m, n, generator=g, dtype=torch.float64)
    keep = np.random.default_rng(2).random((m, n)) >= p
    for relu, drop, bias in [(False, False, False), (True, False, True), (True, True, True)]:
        xr, wr = x.clone().requires_grad_(), w.clone().requires_grad_()
        br = b.clone().requires_grad_() if bias else None
        y = F.linear(xr, wr, br)
        if relu:
            y = F.relu(y)
        if drop:
            y = y * torch.from_numpy(keep).double() / (1 - p)
        y.backward(gy)
        got = R.linear_fwd(x, w, b if bias else None, relu=relu, keep=keep if drop else None, p=p if drop else 0.0)
        assert rel_err(got, y) < 1e-12
        dx, dw, db = R.linear_bwd(x, w, got, gy, relu=relu, p=p if drop else 0.0)
        assert rel_err(dx, xr.grad) < 1e-12 and rel_err(dw, wr.grad) < 1e-12
        if bias:
            assert rel_err(db, br.grad) < 1e-12


def test_rank_order_sum_is_left_to_right_fp32():
    a = torch.tensor([1.0, 2.0 ** 24], dtype=torch.float32)
    b = torch.tensor([2.0 ** -24, 1.0], dtype=torch.float32)
    c = torch.tensor([-1.0, -(2.0 ** 24)], dtype=torch.float32)
    # (a + b) + c: the small terms are rounded away first; another order would keep them
    assert torch.equal(R.rank_order_sum([a, b, c]), (a + b) + c)
    assert not torch.equal(R.rank_order_sum([a, c, b]), (a + b) + c)
