"""The fused VAE heads (mvb_vae_heads_fwd/bwd: classifier + softmax, z_mean, z_log_var on cat(y, h), the
reparameterisation and cat(y, z); models/cheb_VAE.py:206-223, 253-258, 309-319) at the shapes a user's config can
ask for - any batch, hidden width and latent size, up to 32 classes, with dropout - against the same heads written
with torch on the CPU in fp64.  The classifier's dropout mask is checked against an independent numpy restatement of
the library's Philox4x32-10 key (seed, offset, b*H + j)."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import OPERATORS_NPZ, seeded_state_dict, seeded_batch, rel_err, elem_err
from oracle import mesh_vae_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    return meshvae_b200


# ---- Philox4x32-10 and the keep decision of csrc/mvb_dense.cu (philox4x32_10, drop_keep), restated in numpy ----
def _philox4x32_10(c, k):
    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    mask = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, dtype=np.uint64) & mask for x in c]
    k0, k1 = np.uint64(k[0]), np.uint64(k[1])
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]                    # exact: both factors < 2^32
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0, k1 = (k0 + W0) & mask, (k1 + W1) & mask
    return c


def keep_mask(seed: int, offset: int, b: int, hdim: int, p: float) -> np.ndarray:
    """[b, hdim] bool: element (i, j) is kept; counter (idx / 4, 0, offset lo, offset hi), key (seed lo, seed hi), word
    idx % 4 of the output, idx = i*hdim + j; kept when (word >> 8) * 2^-24 >= p in fp32"""
    idx = np.arange(b * hdim, dtype=np.uint64)
    n = np.zeros_like(idx)
    r = _philox4x32_10([idx >> np.uint64(2), n, n + np.uint64(offset & 0xFFFFFFFF), n + np.uint64((offset >> 32) & 0xFFFFFFFF)],
                       (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    lane = (idx & np.uint64(3)).astype(np.int64)
    word = np.choose(lane, r)
    u = (word >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return (u >= np.float32(p)).reshape(b, hdim)


# ---- inputs and the fp64 CPU reference ----
def _inputs(b, hdim, z, c, seed):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(b, hdim, generator=g)
    y = F.one_hot(torch.randint(0, c, (b,), generator=g), c)
    eps = torch.randn(b, z, generator=g)
    ws = [torch.randn(c, hdim, generator=g) / hdim ** 0.5, torch.randn(c, generator=g) * 0.1,
          torch.randn(z, c + hdim, generator=g) / (c + hdim) ** 0.5, torch.randn(z, generator=g) * 0.1,
          torch.randn(z, c + hdim, generator=g) / (c + hdim) ** 0.5, torch.randn(z, generator=g) * 0.1]
    ups = [torch.randn(b, c, generator=g), torch.randn(b, z, generator=g), torch.randn(b, z, generator=g),
           torch.randn(b, z, generator=g), torch.randn(b, c + z, generator=g)]
    return h, y, eps, ws, ups


def _reference(h, y, eps, ws, ups, keep=None, p=0.0):
    """fp64 outputs (y_hat, mu, logvar, z, zcat) and gradients (g_h, dWc, dbc, dWm, dbm, dWv, dbv); ups entries may be
    None (no gradient from that output)"""
    hr = h.double().requires_grad_()
    wr = [w.double().requires_grad_() for w in ws]
    hd = hr if keep is None else hr * torch.from_numpy(keep).double() / (1.0 - p)
    y_hat = torch.softmax(F.linear(hd, wr[0], wr[1]), 1)
    hc = torch.cat([y.double(), hr], 1)
    mu, lv = F.linear(hc, wr[2], wr[3]), F.linear(hc, wr[4], wr[5])
    zz = mu + eps.double() * torch.exp(0.5 * lv) if eps is not None else mu
    zcat = torch.cat([y.double(), zz], 1)
    outs = (y_hat, mu, lv, zz, zcat)
    used = [(o, u.double()) for o, u in zip(outs, ups) if u is not None]
    grads = torch.autograd.grad([o for o, _ in used], [hr] + wr, [u for _, u in used], allow_unused=True)
    grads = [torch.zeros_like(t) if gr is None else gr for gr, t in zip(grads, [hr] + wr)]
    return [o.detach() for o in outs], grads


def _heads_abi(mvb, h, y, eps, ws, ups, p=0.0, seed=0, offset=0):
    """mvb_vae_heads_fwd then mvb_vae_heads_bwd through the C ABI (NULL for the upstream gradients that are None)"""
    L = mvb._lib
    b, hdim = h.shape
    c, z = ws[0].shape[0], ws[2].shape[0]
    dev = torch.device("cuda")
    hg, yg = h.to(dev), y.to(dev, torch.int64).contiguous()
    eg = None if eps is None else eps.to(dev)
    wg = [w.to(dev).contiguous() for w in ws]
    y_hat, mu, lv, zz = (torch.empty(b, n, device=dev) for n in (c, z, z, z))
    zcat = torch.empty(b, c + z, device=dev)
    L.check(L.lib.mvb_vae_heads_fwd(b, hdim, z, c, L.ptr(hg), L.ptr(yg), L.ptr(eg), *[L.ptr(w) for w in wg], float(p), seed,
                                    None, offset, L.ptr(y_hat), L.ptr(mu), L.ptr(lv), L.ptr(zz), L.ptr(zcat), L.stream_ptr()),
            "mvb_vae_heads_fwd")
    ug = [None if u is None else u.to(dev).contiguous() for u in ups]
    g_h = torch.full_like(hg, float("nan"))
    dws = [torch.full_like(w, float("nan")) for w in wg]           # every element must be overwritten
    L.check(L.lib.mvb_vae_heads_bwd(b, hdim, z, c, L.ptr(hg), L.ptr(yg), L.ptr(eg), L.ptr(wg[0]), L.ptr(wg[2]), L.ptr(wg[4]),
                                    L.ptr(y_hat), L.ptr(lv), float(p), seed, None, offset, *[L.ptr(u) for u in ug],
                                    L.ptr(g_h), *[L.ptr(d) for d in dws], L.stream_ptr()), "mvb_vae_heads_bwd")
    torch.cuda.synchronize()
    return [y_hat, mu, lv, zz, zcat], [g_h] + dws


def _assert_close(got, ref, names):
    for a, r, name in zip(got, ref, names):
        assert torch.isfinite(a).all(), name
        assert rel_err(a, r) < TOL, (name, rel_err(a, r))
        assert elem_err(a, r) <= 1.0, (name, elem_err(a, r))


OUT_NAMES = ("y_hat", "mu", "logvar", "z", "zcat")
GRAD_NAMES = ("g_h", "dWc", "dbc", "dWm", "dbm", "dWv", "dbv")
SHAPES = [(1, 512, 16, 2), (257, 512, 16, 2), (512, 512, 16, 2), (1000, 512, 16, 2),
          (64, 512, 48, 2), (64, 512, 64, 2), (300, 1024, 128, 2),
          (64, 1562, 16, 2), (64, 4096, 256, 3), (7, 100, 5, 10)]


@pytest.mark.parametrize("b,hdim,z,c", SHAPES)
@pytest.mark.parametrize("which", ["all", "some", "test_mode"])
def test_heads_match_torch(mvb, b, hdim, z, c, which):
    """all five outputs and all eight gradients; "some": only y_hat and z receive a gradient (the other three
    upstream gradients are NULL); "test_mode": eps = NULL (z = mu), no gradient from y_hat / logvar"""
    h, y, eps, ws, ups = _inputs(b, hdim, z, c, seed=b + hdim + z + c)
    if which == "some":
        ups = [ups[0], None, None, ups[3], None]
    elif which == "test_mode":
        eps = None
        ups = [None, ups[1], None, ups[3], ups[4]]
    ref_o, ref_g = _reference(h, y, eps, ws, ups)
    got_o, got_g = _heads_abi(mvb, h, y, eps, ws, ups)
    _assert_close(got_o, ref_o, OUT_NAMES)
    _assert_close(got_g, ref_g, GRAD_NAMES)


@pytest.mark.parametrize("b,z", [(64, 16), (512, 16), (512, 64)])
def test_classifier_dropout_matches_independent_mask(mvb, b, z):
    """p = 0.2: the classifier reads h * mask / (1 - p) with the mask of the numpy restatement, the z heads read h
    (quirk 8); forward and backward against torch.  At 64 meshes the one-launch kernels run, at 512 the tiled backward,
    at 512 x 64 latents the tiled forward and backward."""
    hdim, c, p = 512, 2, 0.2
    seed, offset = 0x1234_5678_9ABC_DEF0, (7 << 32) + 3
    h, y, eps, ws, ups = _inputs(b, hdim, z, c, seed=11)
    keep = keep_mask(seed, offset, b, hdim, p)
    assert abs(keep.mean() - (1 - p)) < 0.01
    ref_o, ref_g = _reference(h, y, eps, ws, ups, keep=keep, p=p)
    got_o, got_g = _heads_abi(mvb, h, y, eps, ws, ups, p=p, seed=seed, offset=offset)
    _assert_close(got_o, ref_o, OUT_NAMES)
    _assert_close(got_g, ref_g, GRAD_NAMES)
    # the mask matters: without it the classifier's output is far from what the kernel computed
    no_mask, _ = _reference(h, y, eps, ws, ups)
    assert rel_err(got_o[0], no_mask[0]) > 100 * TOL


def _heads_autograd(mvb, h, y, eps, ws, ups, p, rng):
    mods = [torch.nn.Linear(ws[0].shape[1], ws[0].shape[0]), torch.nn.Linear(ws[2].shape[1], ws[2].shape[0]),
            torch.nn.Linear(ws[4].shape[1], ws[4].shape[0])]
    for m, (w, bias) in zip(mods, [(ws[0], ws[1]), (ws[2], ws[3]), (ws[4], ws[5])]):
        m.weight.data.copy_(w)
        m.bias.data.copy_(bias)
        m.cuda()
    hg = h.cuda().requires_grad_()
    outs = mvb.functional.vae_heads(hg, y.cuda(), eps.cuda(), *mods, p=p, rng=rng)
    torch.autograd.backward(list(outs), [u.cuda() for u in ups])
    torch.cuda.synchronize()
    return [o.detach() for o in outs], [hg.grad] + [t.grad for m in mods for t in (m.weight, m.bias)]


def test_first_rows_of_a_large_call_equal_a_smaller_call(mvb):
    """the mask is keyed by the row within the call: rows [0, 256) of a 512-mesh call with dropout are the same bits as
    a 256-mesh call with the same (seed, offset) - outputs and the input gradient"""
    hdim, z, c, p = 512, 16, 2, 0.2
    h, y, eps, ws, ups = _inputs(512, hdim, z, c, seed=5)
    rng = (0xC0FFEE, None, 41)
    o_big, g_big = _heads_autograd(mvb, h, y, eps, ws, ups, p, rng)
    o_small, g_small = _heads_autograd(mvb, h[:256], y[:256], eps[:256], ws, [u[:256] for u in ups], p, rng)
    for a, s, name in zip(o_big, o_small, OUT_NAMES):
        assert torch.equal(a[:256], s), name
    assert torch.equal(g_big[0][:256], g_small[0])


def test_bit_identical_run_to_run(mvb):
    b, hdim, z, c, p = 512, 512, 64, 2, 0.2
    h, y, eps, ws, ups = _inputs(b, hdim, z, c, seed=9)
    rng = (77, None, 5)
    o1, g1 = _heads_autograd(mvb, h, y, eps, ws, ups, p, rng)
    o2, g2 = _heads_autograd(mvb, h, y, eps, ws, ups, p, rng)
    for a, r in zip(o1 + g1, o2 + g2):
        assert torch.equal(a, r)


# ---- the whole model at latent sizes, hidden widths and batches the one-launch heads kernels do not hold ----
@pytest.mark.parametrize("batch,num_style,num_hidden", [(16, 64, 1024), (300, 16, 512)])
def test_cheb_vae_matches_oracle_at_other_shapes(mvb, batch, num_style, num_hidden):
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    cfg["dropout"] = 0.0
    cfg["num_style"], cfg["num_hidden"] = num_style, num_hidden
    ref = O.OracleChebVAE(3, cfg, D, U, A, nn_)
    ref.load_state_dict(seeded_state_dict(ref, 7))
    dev = torch.device("cuda:0")
    net = mvb.cheb_VAE(3, copy.deepcopy(cfg), [d.to(dev) for d in D], [u.to(dev) for u in U], [a.to(dev) for a in A], nn_,
                       model=cfg["model"])
    net.load_state_dict(seeded_state_dict(net, 7))
    net = net.to(dev)
    x, y, _ = seeded_batch(batch, nn_[0], 21)
    eps = torch.randn(batch, num_style, generator=torch.Generator().manual_seed(22))
    y_hot = F.one_hot(y, 2)
    ref.train(); net.train()
    lo, co, ro, (ko, reco, zo), yho = ref(x, x.double(), y_hot, m_type="train", eps=eps)
    lo.backward()
    lg, cg, rg, (kg, recg, zg), yhg = net(x.cuda(), x.double().cuda(), y_hot.cuda(), m_type="train", eps=eps.cuda())
    lg.backward()
    assert rel_err(lg, lo) < TOL and int(cg) == int(co) and rel_err(rg, ro) < TOL
    assert rel_err(kg, ko) < TOL and rel_err(recg, reco) < TOL and rel_err(yhg, yho) < TOL and rel_err(zg, zo) < TOL
    # gradients: 1e-3, the bound of test_gpu_parity.py's whole-model test at 64 meshes and for the same reason - ReLU
    # decisions within fp32 rounding of zero land on the other side than in the oracle's summation order, and one flip
    # moves a weight gradient by a whole row's contribution.  With this test's eps such flips occur at 16 meshes too:
    # measured on a B200, 2.3e-4 on dec_lin.weight at (num_style 64, num_hidden 1024), and the same 2.3e-4 with the
    # model's dense layers run by torch on the GPU instead of the fused kernels (6.2e-4 for both at the default config
    # with this eps) - the gap is the flips, not the heads.  Outputs stay at 1e-4.
    gtol = 1e-3
    po = dict(ref.named_parameters())
    for name, p in net.named_parameters():
        if po[name].grad is None:
            assert p.grad is None
        else:
            assert rel_err(p.grad, po[name].grad) < gtol, name


# ---- the captured training step at 512 meshes per GPU with dropout 0.2 (strong scaling, global batch 512) ----
def test_train_engine_512_meshes_with_dropout(mvb):
    from meshvae_b200.engine import TrainEngine
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    cfg["dropout"] = 0.2
    dev = torch.device("cuda:0")
    B = 512
    batches = [seeded_batch(B, nn_[0], 600 + s) for s in range(3)]
    finals, losses = [], []
    for use_graph in (True, False):
        net = mvb.cheb_VAE(3, copy.deepcopy(cfg), [d.to(dev) for d in D], [u.to(dev) for u in U], [a.to(dev) for a in A], nn_)
        net.load_state_dict(seeded_state_dict(net, 11))
        net = net.to(dev)
        eng = TrainEngine(net, B, lr=1e-3, weight_decay=5e-4, use_graph=use_graph)
        eng.capture(warmup=1)
        ls = [eng.step(x, x.double(), y, eps_host=eps) for x, y, eps in batches]
        assert all(np.isfinite(l) for l in ls), ls
        losses.append(ls)
        finals.append([p.detach().clone() for p in net.parameters()])
        del eng, net
    # same kernels, same masks (keyed by the device step counter), same order: the same bits
    assert losses[0] == losses[1]
    for a, r in zip(*finals):
        assert torch.equal(a, r)
