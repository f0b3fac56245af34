"""Host-side mirror of the reference model `cheb_VAE` (models/cheb_VAE.py:104-351) composed from the
native modules: same constructor signature, method names, return tuple and state-dict keys
(`cheb.{i}.weight/.bias`, `cheb_dec.{i}.weight/.bias` with `cheb_dec.4.bias` absent, `enc_lin`,
`dec_lin`, `dec_lin_1` (dead, quirk 7), `dec_lin_2`, `z_mean`, `z_log_var`, `classifier_layer`),
so checkpoints written by main.py:32-39 load unchanged.  The reference file itself also runs
unchanged on top of the `compat/` import shims; this mirror exists because the reference tree is
not present on the GPU box and because it can use the fused entry points:

  * ReLU fused into the contraction epilogue of every conv that the reference follows with
    F.relu (models/cheb_VAE.py:264,285);
  * the loss epilogue (models/cheb_VAE.py:321-346) as one fused kernel pair on the vertex-major
    reconstruction;
  * reparameterisation noise either from the CPU generator as the reference draws it
    (models/cheb_VAE.py:316, `noise="cpu"`) or from the device generator (`noise="device"`,
    CUDA-graph capturable).
"""
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as Fn
from . import operators
from ._lib import MvbError
from .conv import ChebConv_batch
from .pool import SurfacePool


class cheb_VAE(nn.Module):
    def __init__(self, num_features, config, downsample_matrices, upsample_matrices, adjacency_matrices, num_nodes,
                 model="MSE_VAE"):
        super().__init__()
        self.n_layers = config["n_layers"]
        self.filters = [num_features] + list(config["num_conv_filters"])
        self.K = config["polygon_order"]
        self.downsample_matrices = downsample_matrices
        self.upsample_matrices = upsample_matrices
        self.adjacency_matrices = adjacency_matrices
        pairs = [ChebConv_batch.norm(adjacency_matrices[i]._indices(), num_nodes[i]) for i in range(len(num_nodes))]
        self.A_edge_index = tuple(p[0] for p in pairs)
        self.A_norm = tuple(p[1] for p in pairs)

        f = self.filters
        self.cheb = nn.ModuleList([ChebConv_batch(f[i], f[i + 1], self.K[i]) for i in range(len(f) - 2)])
        self.cheb_dec = nn.ModuleList([ChebConv_batch(f[-i - 1], f[-i - 2], self.K[i]) for i in range(len(f) - 1)])
        self.cheb_dec[-1].bias = None          # no bias on the output conv (models/cheb_VAE.py:135)
        for conv in list(self.cheb) + list(self.cheb_dec)[:-1]:
            conv.fuse_relu = True              # every one of these is followed by F.relu in the reference
        self.pool = SurfacePool()

        self.num_class = config["num_classes"]
        self.z = config["num_style"]
        self.num_hidden = config["num_hidden"]
        flat = downsample_matrices[-1].shape[0] * f[-1]
        self.classifier_layer = nn.Linear(self.num_hidden, self.num_class)
        self.z_mean = nn.Linear(self.num_hidden + self.num_class, self.z)
        self.z_log_var = nn.Linear(self.num_hidden + self.num_class, self.z)
        self.enc_lin = nn.Linear(flat, self.num_hidden)
        self.dec_lin = nn.Linear(self.z + self.num_class, self.num_hidden)
        self.dec_lin_1 = nn.Linear(self.z + self.num_class, self.num_hidden)
        self.dec_lin_2 = nn.Linear(self.num_hidden, flat)
        self.dropout = nn.Dropout(p=config["dropout"])
        self.reset_parameters()
        self.type = model
        self.noise = "cpu"
        # decoder Gaussian log sigma: the reference's constant (quirk 6; `model` above does not change it, as in the
        # reference), or a sigma-VAE variant chosen with set_decoder_sigma
        self.sigma_mode = "fixed"
        self.log_sigma = Fn.LOG_SIGMA_DEFAULT
        self.last_log_sigma = None
        self.train_log_sigma = None
        # fused dense bottleneck (row f2): one launch per Linear(+ReLU+dropout), one for the three heads
        self.fused_dense = True
        # coarse levels: pool + conv + ReLU (+ pool) as one mesh-resident kernel (Fn.cheb_layer)
        self.fused_layers = True
        self.keep_encoder_conv_out = False
        self._recon_padded = None
        self.encoder_conv_out = None
        self.A_num_nodes = tuple(int(n) for n in num_nodes)
        self.dropout_stream = Fn.DropoutStream()

    def set_decoder_sigma(self, mode: str, init: float = 0.0):
        """The decoder likelihood's log sigma (Rybkin et al., "Simple and Effective VAE Training with Calibrated Decoders"):
          "fixed"   - the reference's constant softclip(1, -6) (models/cheb_VAE.py:328-329), the default;
          "optimal" - the batch's optimal sigma, sc(0.5 log(SSE / (B N C))), sc(t) = -6 + softplus(t + 6), computed on
                      the device in the loss epilogue, with its gradient;
          "learned" - sc(s) with s a scalar Parameter `log_sigma` initialised to `init`, trained with the others.
        Only "learned" adds a state-dict key (`log_sigma`).  Choose the mode before an engine.TrainEngine is built on the
        model: the engine lays out its flat parameter buffer from the parameters it finds then."""
        if mode not in ("fixed", "optimal", "learned"):
            raise ValueError(f"set_decoder_sigma: mode is 'fixed', 'optimal' or 'learned', got {mode!r}")
        if "log_sigma" in self._parameters:
            del self._parameters["log_sigma"]
        if mode == "learned":
            dev = next(self.parameters()).device
            self.log_sigma = nn.Parameter(torch.full((), float(init), device=dev, dtype=torch.float32))
        else:
            self.log_sigma = Fn.LOG_SIGMA_DEFAULT if mode == "fixed" else "optimal"
        self.sigma_mode = mode
        self.last_log_sigma = None
        self.train_log_sigma = None

    def reset_parameters(self):
        nn.init.normal_(self.enc_lin.weight, 0, 0.1)
        nn.init.normal_(self.dec_lin.weight, 0, 0.1)

    def set_param(self, alpha, beta):
        self.alpha, self.beta = alpha, beta

    @staticmethod
    def _act(conv, y):
        """F.relu of models/cheb_VAE.py:264,285 - already applied inside the conv epilogue when fused"""
        return y if conv.fuse_relu else F.relu(y)

    def _layer(self, x, conv, lvl, up=None, down=None):
        """one step of the encoder loop (conv, relu, pool(D): models/cheb_VAE.py:264-265) or of the decoder
        loop (pool(U), conv, relu: :284-285); coarse levels run as ONE mesh-resident kernel per direction.  An operator
        computed from learned edge weights (A_norm[lvl] requires grad) takes the composition: only ChebConv_batch
        differentiates its values"""
        learned = self.A_norm[lvl].requires_grad and torch.is_grad_enabled()
        if self.fused_layers and x.is_cuda and conv.fuse_relu and not learned:
            l_op = operators.from_edges(self.A_edge_index[lvl], self.A_norm[lvl], self.A_num_nodes[lvl], x.device)
            u_op = None if up is None else operators.from_sparse(up, x.device)
            d_op = None if down is None else operators.from_sparse(down, x.device)
            fin, fout = conv.weight.shape[1], conv.weight.shape[2]
            if fin % 4 == 0 and fout % 4 == 0:
                y = Fn.cheb_layer_fused(Fn.to_vertex_major(x), conv.weight, conv.bias, l_op, u_op, d_op, relu=True)
                if y is not None:
                    return Fn.from_vertex_major(y)
            if u_op is None and fout % 4 == 0:
                # level 0 (too large for a mesh-resident kernel): conv + ReLU + row selection, only the rows D keeps are
                # contracted / reduced over (first encoder layer: its input needs no gradient)
                xv = Fn.to_vertex_major(x)
                if Fn.cheb_conv_sel_supported(xv, conv.weight, l_op, d_op):
                    return Fn.from_vertex_major(Fn.cheb_conv_sel(xv, conv.weight, conv.bias, l_op, d_op, relu=True))
        if up is not None:
            x = self.pool(x, up)
        x = self._act(conv, conv(x, self.A_edge_index[lvl], self.A_norm[lvl]))
        if down is not None:
            x = self.pool(x, down)
        return x

    # ---- sub-networks (logical [B, N, F] tensors; physically vertex-major views) -----------------
    def encoder(self, x):
        if x.is_cuda and not x.requires_grad and x.shape[2] % 4:
            # 3-channel input: one kernel to the zero-padded vertex-major layout (the first conv pads its weight to match)
            x = Fn.from_vertex_major(Fn.pack_input(x))
        for i in range(self.n_layers):
            x = self._layer(x, self.cheb[i], i, down=self.downsample_matrices[i])
        if self.keep_encoder_conv_out:
            # one-shot hand-over to the step engine, which splits the backward pass (gradient buckets) at this
            # tensor and clears the attribute at once - a lasting reference would keep the step's autograd graph alive
            self.encoder_conv_out = x
        if self.fused_dense and x.is_cuda:
            # x.reshape(B, 640) of models/cheb_VAE.py:270 is read straight from the vertex-major buffer
            return Fn.linear(Fn.to_vertex_major(x), self.enc_lin.weight, self.enc_lin.bias, relu=True, p=self._p(),
                             rng=self.dropout_stream.site(0), x_vm=True)
        x = x.reshape(x.shape[0], self.enc_lin.in_features)
        return self.dropout(F.relu(self.enc_lin(x)))

    def _p(self) -> float:
        return float(self.dropout.p) if self.training else 0.0

    def classifier(self, x):
        if self.fused_dense and x.is_cuda and not x.requires_grad and not (self.training and self.dropout.p > 0):
            # inference.py:88 / main.py:42-49 (classifier_): softmax(classifier_layer(x)) from the heads kernel
            # (its other outputs are discarded); no cuBLAS / ATen launch on the forward-only path
            y0 = torch.zeros((x.shape[0], self.num_class), device=x.device, dtype=torch.int64)
            return Fn.vae_heads(x, y0, None, self.classifier_layer, self.z_mean, self.z_log_var)[0]
        return F.softmax(self.classifier_layer(self.dropout(x)), dim=1)

    def decoder(self, z):
        if self.fused_dense and z.is_cuda:
            x = Fn.linear(z, self.dec_lin.weight, self.dec_lin.bias, relu=True, p=self._p(), rng=self.dropout_stream.site(2))
            # x.reshape(B, -1, 32) of models/cheb_VAE.py:281 is written straight in the vertex-major layout
            x = Fn.linear(x, self.dec_lin_2.weight, self.dec_lin_2.bias, relu=True, p=self._p(),
                          rng=self.dropout_stream.site(3), y_vm_f=self.filters[-1])
            x = Fn.from_vertex_major(x)
        else:
            x = self.dropout(F.relu(self.dec_lin(z)))
            x = self.dropout(F.relu(self.dec_lin_2(x)))
            x = x.reshape(x.shape[0], -1, self.filters[-1])
        for i in range(self.n_layers):
            lvl = self.n_layers - i - 1
            x = self._layer(x, self.cheb_dec[i], lvl, up=self.upsample_matrices[lvl])
        # quirk 1: the output conv runs the COARSEST operator on the finest mesh (models/cheb_VAE.py:288)
        conv = self.cheb_dec[-1]
        if x.is_cuda and not conv.fuse_relu:
            # the 3-channel output stays in its 4-float entries: the returned [B,N,3] tensor is a view, and
            # loss_function reads the padded buffer in place (handed over once through _recon_padded)
            op, vals = operators.edge_operator(self.A_edge_index[-1], self.A_norm[-1], x.size(1), x.device)
            y = Fn.cheb_conv(Fn.to_vertex_major(x), conv.weight, conv.bias, op, False, keep_padding=True, norm=vals)
            fout = conv.weight.shape[2]
            if y.shape[2] != fout:
                self._recon_padded = y
            return Fn.from_vertex_major(y)[..., :fout]
        return conv(x, self.A_edge_index[-1], self.A_norm[-1])

    def sample(self, y, z):
        x = self.decoder(torch.cat([y, z], -1))
        self._recon_padded = None       # no loss follows a sampled decode: drop the hand-over reference at once
        return x.reshape(z.shape[0], -1, self.filters[0])

    def _draw_eps(self, shape, like):
        if self.noise == "device":
            return torch.randn(shape, device=like.device, dtype=like.dtype)
        return torch.normal(mean=0, std=1, size=tuple(shape)).to(like.device)      # CPU generator, models/cheb_VAE.py:316

    def reparameterize(self, mu, logvar, eps: Optional[torch.Tensor] = None):
        if eps is None:
            eps = self._draw_eps(mu.shape, mu)
        return Fn.reparameterize(mu, logvar, eps)

    def loss_function(self, x, recon_x, z, mu_z, logvar_z, y, y_hat):
        """as the reference's; with a sigma-VAE decoder sigma the log sigma used is left in `last_log_sigma` (fp64 0-dim
        device tensor), and in training mode also in `train_log_sigma`: the sigma of the last training step, which an
        evaluation forward does not replace (log_likelihood's optimal sigma)"""
        padded, self._recon_padded = self._recon_padded, None           # one-shot hand-over from decoder()
        if padded is not None and recon_x.data_ptr() == padded.data_ptr() and recon_x.shape[1] == padded.shape[0]:
            recon_vm, channels = padded, recon_x.shape[2]
        else:
            recon_vm, channels = Fn.to_vertex_major(recon_x), None
        out = Fn.vae_loss(recon_vm, x, mu_z, logvar_z, y_hat, y, self.log_sigma, channels=channels,
                          return_log_sigma=self.sigma_mode != "fixed")
        loss, kld, rec, correct = out[:4]
        if self.sigma_mode != "fixed":
            self.last_log_sigma = out[4]
            if self.training:
                self.train_log_sigma = out[4]
        return loss, correct, kld, rec

    def forward_recon(self, data, y, m_type="test", eps: Optional[torch.Tensor] = None):
        """everything of forward() that does not need the ground truth: encoder, heads, decoder
        (models/cheb_VAE.py:195-243).  -> (recon, z, x_mean, x_var, z_, y_hat).  The step engine runs this
        part while the ground-truth batch is still on its way to the device."""
        if isinstance(data, torch.Tensor):
            x, batch_size = data, data.shape[0]
        else:
            x, batch_size = data.x, data.num_graphs
        x = x.reshape(batch_size, -1, self.filters[0])
        self.dropout_stream.advance()
        h = self.encoder(x)
        if self.fused_dense and h.is_cuda:
            if m_type == "train" and eps is None:
                eps = self._draw_eps((batch_size, self.z), h)
            y_hat, x_mean, x_var, z_, z = Fn.vae_heads(h, y, eps if m_type == "train" else None, self.classifier_layer,
                                                       self.z_mean, self.z_log_var, p=self._p(),
                                                       rng=self.dropout_stream.site(1))
        else:
            y_hat = self.classifier(h)
            h = torch.cat([y, h], -1)
            x_mean, x_var = self.z_mean(h), self.z_log_var(h)
            z_ = self.reparameterize(x_mean, x_var, eps) if m_type == "train" else x_mean
            z = torch.cat([y, z_], -1)
        recon = self.decoder(z).reshape(batch_size, -1, self.filters[0])
        return recon, z, x_mean, x_var, z_, y_hat

    def _likelihood_log_sigma(self, log_sigma, dev) -> torch.Tensor:
        """the decoder log sigma of log_likelihood as a 0-dim fp64 device tensor (never read back to the host)"""
        if isinstance(log_sigma, torch.Tensor):
            Fn._req_cuda(log_sigma, "log_likelihood log_sigma", None)
            if log_sigma.numel() != 1:
                raise MvbError(f"log_likelihood: log_sigma has {log_sigma.numel()} elements, expected 1")
            return log_sigma.detach().reshape(()).to(torch.float64)
        if log_sigma is not None:
            if isinstance(log_sigma, str):
                raise MvbError(f"log_likelihood: log_sigma is a float or a 1-element CUDA tensor, got {log_sigma!r}")
            return torch.full((), float(log_sigma), device=dev, dtype=torch.float64)
        if self.sigma_mode == "learned":
            t = self.log_sigma.detach().double() + 6.0
            return -6.0 + torch.logaddexp(t, torch.zeros_like(t))
        if self.sigma_mode == "optimal":
            if self.train_log_sigma is None:
                raise MvbError("log_likelihood: the optimal decoder sigma is taken from the last training step, and the model "
                               "has not trained in this mode; pass log_sigma=")
            return self.train_log_sigma.detach().reshape(()).to(dev, torch.float64)
        return torch.full((), float(self.log_sigma), device=dev, dtype=torch.float64)

    def log_likelihood(self, x, x_gt, y_onehot, samples: int, sample_chunk: Optional[int] = None,
                       generator: Optional[torch.Generator] = None, log_sigma=None, return_log_w: bool = False):
        """Importance-weighted estimate of log p(x | y) per mesh with `samples` (S) draws from q(z | x, y):
        log w_s = log p(x | z_s, y) + log p(z_s) - log q(z_s | x, y), and
          log_px = log (1/S) sum_s w_s   (a lower bound of log p(x | y) in expectation, tight as S grows),
          elbo   = (1/S) sum_s log w_s   (the Monte-Carlo ELBO),
          ess    = (sum_s w_s)^2 / sum_s w_s^2   (the effective sample size of the weights, between 1 and S),
        each an fp64 [B] device tensor; return_log_w=True appends log w [B, S].  x [B,N,F] the (z-scored) input, x_gt
        [B,N,F] fp32 / fp64 its ground truth, y_onehot [B, num_classes]; densities are those of these coordinates.

        The model runs in eval mode (no dropout) under no_grad, and its mode is restored afterwards.  The encoder and heads
        run once; eps = torch.randn((B, S, num_style), generator=generator, device=x.device) is drawn once, so the result
        does not depend on `sample_chunk`; the decoder runs on sample_chunk * B meshes at a time (default: all S).  No host
        synchronisation: the call can be captured in a CUDA graph (with the default generator, or one registered with it).

        The decoder's log sigma: `log_sigma` (a float or a 1-element CUDA tensor) when given, else that of the model's
        decoder sigma mode - the constant (fixed), sc(s) of the parameter (learned), or `train_log_sigma`, the sigma of the
        last training step (optimal: MvbError when there is none; the sigma is never derived from the data scored)."""
        if isinstance(x, torch.Tensor):
            b = x.shape[0]
        else:
            x, b = x.x, x.num_graphs
        Fn._req_cuda(x, "log_likelihood x")
        Fn._req_cuda(x_gt, "log_likelihood x_gt", None)
        Fn._req_cuda(y_onehot, "log_likelihood y", None)
        s_total = int(samples)
        chunk = s_total if sample_chunk is None else int(sample_chunk)
        if s_total < 1 or chunk < 1:
            raise MvbError(f"log_likelihood: samples={samples} and sample_chunk={sample_chunk} must be >= 1")
        chunk = min(chunk, s_total)
        x = x.reshape(b, -1, self.filters[0])
        if x.shape[1] != self.A_num_nodes[0] or x_gt.dim() != 3 or tuple(x_gt.shape) != tuple(x.shape):
            raise MvbError(f"log_likelihood: x {tuple(x.shape)} and x_gt {tuple(x_gt.shape)} must both be "
                           f"({b}, {self.A_num_nodes[0]}, {self.filters[0]})")
        dev = x.device
        ls = self._likelihood_log_sigma(log_sigma, dev)
        was_training = self.training
        self.eval()
        try:
            with torch.no_grad():
                h = self.encoder(x)
                _, mu, logvar, _, _ = Fn.vae_heads(h, y_onehot, None, self.classifier_layer, self.z_mean, self.z_log_var)
                eps = torch.randn((b, s_total, self.z), generator=generator, device=dev, dtype=torch.float32)
                log_w = torch.empty((b, s_total), device=dev, dtype=torch.float64)
                for s0 in range(0, s_total, chunk):
                    zcat, log_r = Fn.iw_sample(mu, logvar, eps[:, s0:s0 + chunk], y_onehot)
                    recon = self.decoder(zcat)
                    padded, self._recon_padded = self._recon_padded, None
                    if padded is not None and recon.data_ptr() == padded.data_ptr():
                        recon_vm, channels = padded, recon.shape[2]
                    else:
                        recon_vm, channels = Fn.to_vertex_major(recon), None
                    Fn.iw_log_weights(recon_vm, x_gt, ls, log_r, log_w, s0, channels)
                return Fn.iw_reduce(log_w, return_log_w)
        finally:
            self.train(was_training)

    def forward(self, data, x_gt, y, supervise=True, m_type="test", eps: Optional[torch.Tensor] = None):
        self.supervise = supervise
        recon, z, x_mean, x_var, z_, y_hat = self.forward_recon(data, y, m_type, eps)
        loss, correct, kld, rec_loss = self.loss_function(x_gt, recon, z, x_mean, x_var, y, y_hat)
        return loss, correct, recon, [kld, rec_loss, z_], y_hat
