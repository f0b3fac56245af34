"""Training-step engine for `cheb_VAE`: the per-batch body of main.py:67-85 (H2D of the batch,
forward, backward, optimizer step, loss read-back) with every device operation captured once in
CUDA graphs and replayed, one process per GPU.

Data parallel (new - the reference is single device, main.py:194-195): each rank owns a
contiguous slice of the global batch; the gradient of the global-batch mean loss is the average
of the per-rank gradients, exchanged as ONE flat fp32 buffer with one NCCL all-reduce over
NVLink / NVSwitch between the backward graph and the optimizer graph; the 1/world_size scaling is
folded into the fused Adam kernel (`mvb_adam_step`).  `dec_lin_1` never receives a gradient
(quirk 7) and is excluded from the flat buffers, exactly as torch's Adam skips it.
"""
import os
from typing import Optional

import torch
import torch.distributed as dist

from . import _lib, dp
from ._lib import lib, check, ptr, stream_ptr


class _HyperGroup(dict):
    """optimizer.param_groups[0] of torch.optim.Adam: item assignment reaches the device-resident hyper-parameters"""

    def __init__(self, opt):
        super().__init__(lr=opt.lr, betas=opt.betas, eps=opt.eps, weight_decay=opt.weight_decay, amsgrad=False)
        self._opt = opt

    def __setitem__(self, key, value):
        super().__setitem__(key, value)
        if key in ("lr", "betas", "eps", "weight_decay"):
            setattr(self._opt, key, value)


class FlatAdam:
    """Adam(lr, betas, eps, weight_decay) with torch.optim.Adam's arithmetic (main.py:251) as one
    fused kernel over a flat parameter buffer; parameters are re-pointed to views of that buffer."""

    ALIGN = 32          # elements: every parameter starts on a 128-byte boundary of the flat buffers, so that
                        # the kernels' 16-byte vector / cp.async paths apply to parameter and gradient views

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, grad_buffer_factory=None):
        self.params = [p for p in params]
        dev = self.params[0].device
        self.offsets, self.n = dp.flat_layout(self.params, self.ALIGN)
        # padding elements stay exactly zero: p = g = 0 => m = v = 0 and the update is 0
        self.flat_p = torch.zeros(self.n, device=dev, dtype=torch.float32)
        for p, o in zip(self.params, self.offsets):
            k = p.numel()
            self.flat_p[o:o + k].copy_(p.detach().reshape(-1))
            p.data = self.flat_p[o:o + k].view_as(p)
        # (data parallel: the gradient buffer may live in peer-mapped memory - dp.PeerBuffers - for the fused exchange)
        self.flat_g = grad_buffer_factory(self.n) if grad_buffer_factory is not None else torch.zeros(self.n, device=dev, dtype=torch.float32)
        self.grad_views = dp.flat_views(self.flat_g, self.params, self.offsets)
        self.m = torch.zeros_like(self.flat_p)
        self.v = torch.zeros_like(self.flat_p)
        self.step_count = torch.zeros((), device=dev, dtype=torch.int64)
        # hyper-parameters live in DEVICE memory (lr, beta1, beta2, eps, weight_decay, grad_scale): the kernel reads them
        # at run time, so a captured step graph follows `opt.lr = ...` / `set_lr()` (the per-epoch schedule of
        # main.py:266-269) and formats.load_adam_state_dict without re-capture
        self._hp_host = [float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), 1.0]
        self.hyper = torch.tensor(self._hp_host, device=dev, dtype=torch.float32)
        # the view torch.optim.Adam offers to main.py:266-269 (`for p in optimizer.param_groups: p['lr'] = ...`)
        self.param_groups = [_HyperGroup(self)]

    def _set_hp(self, i: int, v: float):
        v = float(v)
        if self._hp_host[i] != v:
            self._hp_host[i] = v
            self.hyper[i:i + 1].copy_(torch.tensor([v], dtype=torch.float32), non_blocking=False)

    lr = property(lambda self: self._hp_host[0], lambda self, v: self._set_hp(0, v))
    eps = property(lambda self: self._hp_host[3], lambda self, v: self._set_hp(3, v))
    weight_decay = property(lambda self: self._hp_host[4], lambda self, v: self._set_hp(4, v))
    grad_scale = property(lambda self: self._hp_host[5], lambda self, v: self._set_hp(5, v))

    @property
    def betas(self):
        return (self._hp_host[1], self._hp_host[2])

    @betas.setter
    def betas(self, b):
        self._set_hp(1, b[0])
        self._set_hp(2, b[1])

    def set_lr(self, lr: float):
        """learning rate of the NEXT step, captured graphs included"""
        self.lr = lr

    def pack_grads(self):
        """one multi-tensor copy of the per-parameter gradients into the flat exchange buffer"""
        dp.pack_grads(self.params, self.grad_views)

    def step_peers(self, peer, grad_scale: float = 1.0, lo: int = 0, hi: Optional[int] = None, channel: int = 0, tick: bool = True,
                   max_ctas: int = 0):
        """all-reduce over the peers' gradient buffers + Adam in ONE launch (mvb_dp_reduce_adam) for the elements [lo, hi)
        of the flat buffers (a gradient bucket)"""
        self.grad_scale = grad_scale
        hi = self.n if hi is None else hi
        check(lib.mvb_dp_reduce_adam(peer.world, peer.rank, channel, lo, hi - lo, ptr(self.flat_p), peer.grad_ptrs, ptr(self.m),
                                     ptr(self.v), None, ptr(self.step_count), 1 if tick else 0, ptr(self.hyper), peer.pad_ptrs,
                                     ptr(peer.state), max_ctas, stream_ptr()), "mvb_dp_reduce_adam")

    def step(self, grad_scale: float = 1.0):
        self.grad_scale = grad_scale
        check(lib.mvb_adam_step_hp(self.n, ptr(self.flat_p), ptr(self.flat_g), ptr(self.m), ptr(self.v),
                                   ptr(self.step_count), ptr(self.hyper), stream_ptr()), "mvb_adam_step_hp")


class TrainEngine:
    def __init__(self, net, batch: int, lr=1e-3, weight_decay=5e-4, x_gt_dtype=torch.float64, use_graph=True,
                 distributed: Optional[bool] = None, graph_comm: bool = True, fused_dp: Optional[bool] = None):
        self.net = net
        self.dev = next(net.parameters()).device
        self.batch = batch
        self.world = dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1
        self.sigma_mode = getattr(net, "sigma_mode", "fixed")
        if self.sigma_mode == "optimal" and self.world > 1:
            # each rank would derive sigma from its own shard's error, not from the global batch's
            raise _lib.MvbError("TrainEngine: the optimal decoder sigma needs the whole batch's error; it is not supported "
                                f"with {self.world} data-parallel ranks (use 'fixed' or 'learned')")
        self.distributed = (self.world > 1) if distributed is None else distributed
        self.graph_comm = graph_comm            # data parallel: capture the all-reduces inside the step graph
        self.one_graph = False
        self._capturing_one_graph = False
        self.n_vert = net.adjacency_matrices[0].shape[0]
        self.feat = net.filters[0]
        # which parameters receive gradients is a property of the graph (dec_lin_1 is dead): probe once
        # the step's four input tensors are views of ONE flat device buffer (256-byte aligned pieces), so that the
        # double-buffered path moves a staged batch into place with a single device-to-device copy
        self._in_spec = [((batch, self.n_vert, self.feat), torch.float32), ((batch, self.n_vert, self.feat), x_gt_dtype),
                         ((batch, net.z), torch.float32), ((batch, net.num_class), torch.int64)]
        self._in_flat, (self.x, self.x_gt, self.eps, self.y_hot) = self._alloc_inputs()
        self.y_hot[:, 0] = 1
        net.train()
        net.zero_grad(set_to_none=True)
        loss, *_ = net(self.x, self.x_gt, self.y_hot, m_type="train", eps=self.eps)
        loss.backward()
        live = dp.live_parameters(list(net.parameters()))
        net.zero_grad(set_to_none=True)
        # Flat-buffer order = gradient buckets for data parallelism.  Bucket 2 (front of the buffer, ~30 KB): the
        # encoder convolutions, whose gradients are the last ones of the backward pass, and the 3-channel
        # convolutions, whose gradients arrive through autograd.  Bucket 1: everything else (99 % of the bytes),
        # final once the backward pass reaches the encoder's last pooled output - its all-reduce runs on NCCL's
        # stream while the encoder backward (a second graph) computes.
        self._enc_ids = {id(p) for p in getattr(net, "cheb", torch.nn.ModuleList()).parameters()}
        # (round 2) every convolution's weights go to the late bucket: their gradients come from the deferred
        # weight-gradient side chains (joined once, at the end of the backward pass), and together they are ~100 KB -
        # the early bucket then holds exactly the dense layers (99 % of the bytes), all produced on the main stream
        # before the cut, and its all-reduce overlaps the whole encoder backward without an early join
        conv_ids = self._enc_ids | {id(p) for p in getattr(net, "cheb_dec", torch.nn.ModuleList()).parameters()}
        late = [p for p in live if id(p) in conv_ids or (p.dim() == 3 and (p.shape[1] % 4 or p.shape[2] % 4))]
        late_ids = {id(p) for p in late}
        live = late + [p for p in live if id(p) not in late_ids]
        # Data parallel on one node: the gradient exchange and Adam are ONE launch that reads the peers' flat gradient
        # buffers over NVLink (csrc/mvb_dp.cu) - no NCCL call in the step, no bucket split.  fused_dp=None: used when the
        # process group is NCCL and the peer mapping succeeds on every rank, else the bucketed NCCL all-reduces below.
        self.peer = None
        want = fused_dp if fused_dp is not None else os.environ.get("MVB_FUSED_DP", "1") != "0"
        if self.distributed and self.world > 1 and want and self.dev.type == "cuda" and dist.get_backend() == "nccl":
            n_flat = dp.flat_layout(live, FlatAdam.ALIGN)[1]
            try:
                self.peer = dp.PeerBuffers(n_flat, self.dev)
            except Exception as e:  # noqa: BLE001
                if fused_dp:
                    raise
                import warnings
                warnings.warn(f"TrainEngine: peer-memory gradient exchange unavailable ({e}); using NCCL all-reduces")
        if self.distributed and self.world > 1 and (self.peer is None or os.environ.get("MVB_DP_PDL", "1") == "0"):
            # Programmatic dependent launch and the data-parallel graph (2 GPUs, same box, ms per step): with the exchange
            # branch on an ordinary-priority stream 0.9913 with PDL / 0.9627 without (the CTAs parked in griddepcontrol.wait take
            # the block slots the exchange kernel needs); with the branch on a HIGHEST-priority stream 0.9424 with PDL (the mesh
            # kernels' CTAs are already resident when the exchange launches, and its few CTAs win the slots that free up) but
            # 1.07-1.54 without (the exchange CTAs are placed first, one per SM, and every mesh kernel - one CTA per WHOLE SM -
            # waits for them).  So: PDL stays on with the peer-memory exchange (MVB_DP_PDL=0 switches it off) and goes off
            # for the NCCL fallback, whose kernels run on NCCL's own ordinary-priority stream.
            _lib.tune("pdl=0")
        self.opt = FlatAdam(live, lr=lr, weight_decay=weight_decay,
                            grad_buffer_factory=(lambda n: self.peer.flat_g) if self.peer is not None else None)
        self.split = self.opt.offsets[len(late)] if (self.distributed and use_graph and hasattr(net, "keep_encoder_conv_out")
                                                     and 0 < len(late) < len(live)) else 0
        if os.environ.get("MVB_DP_SPLIT") == "0":          # A/B: one all-reduce of the whole buffer at the end of the backward pass
            self.split = 0
        if hasattr(net, "dropout_stream"):
            # fresh dropout masks on every graph replay: the fused dense kernels add Adam's device step
            # counter to their Philox offset; per-rank streams (SURVEY.md 8(e))
            rank = dist.get_rank() if self.world > 1 else 0
            net.dropout_stream.offset_dev = self.opt.step_count
            net.dropout_stream.seed = (net.dropout_stream.seed + 7919 * rank) & 0xFFFFFFFFFFFFFFFF
        # Gradient sinks: the backward kernels write dW / db straight into the parameter's view of the flat
        # exchange buffer (no per-parameter allocation, no pack copy).  A second probe step finds the few
        # parameters whose gradient still arrives through torch autograd (the 3-channel convolutions, whose
        # weights pass through the differentiable zero-padding of functional.cheb_conv): those are copied.
        for p, v in zip(self.opt.params, self.opt.grad_views):
            p._mvb_grad_sink = v
        net.zero_grad(set_to_none=True)
        loss, *_ = net(self.x, self.x_gt, self.y_hot, m_type="train", eps=self.eps)
        loss.backward()
        self.loose = [(p, v) for p, v in zip(self.opt.params, self.opt.grad_views) if p.grad is not None]
        for p, v in zip(self.opt.params, self.opt.grad_views):
            if p.grad is None:
                p.grad = v                      # the sink IS the gradient
        self.loss = torch.zeros((), device=self.dev, dtype=torch.float64)
        self.kld = self.rec = self.correct = self.recon = None
        # the decoder log sigma of the last step (fp64 0-dim device tensor): the constant, or the sigma-VAE one the loss
        # epilogue derived (a tensor of the step graph, updated by every replay like kld / rec / correct)
        self.log_sigma = None if self.sigma_mode != "fixed" else \
            torch.full((), float(torch.tensor(net.log_sigma, dtype=torch.float32)), device=self.dev, dtype=torch.float64)
        self.use_graph = use_graph
        self.g_fb = self.g_opt = self.g_enc = None
        self._cut = self._cut_grad = None
        self.launches_per_step = None
        self._copy_stream = self._gt_ready = None
        self._stage = self._stage_flat = self._ev_staged = self._ev_consumed = self._h_small = None
        self._staged = False
        self._fwd_out = None
        self._bg_ctas = 0

    def release(self):
        """Detach the engine from the model: remove the gradient sinks (while they are installed the backward kernels
        OVERWRITE the flat gradient buffer and hand `None` to autograd - a torch optimizer driving the same net afterwards
        would skip those parameters, and gradient accumulation would not accumulate) and give the dropout streams back
        their host counter.  Parameters stay views of the flat parameter buffer (values preserved)."""
        for p in self.opt.params:
            if hasattr(p, "_mvb_grad_sink"):
                del p._mvb_grad_sink
            p.grad = None
        if hasattr(self.net, "dropout_stream"):
            self.net.dropout_stream.offset_dev = None
        self.g_fb = self.g_opt = self.g_enc = None

    def _alloc_inputs(self):
        offs, n = [], 0
        for shape, dt in self._in_spec:
            offs.append(n)
            nbytes = torch.empty((), dtype=dt).element_size()
            for d in shape:
                nbytes *= d
            n += (nbytes + 255) // 256 * 256
        flat = torch.zeros(n, device=self.dev, dtype=torch.uint8)
        views = []
        for (shape, dt), o in zip(self._in_spec, offs):
            k = torch.empty((), dtype=dt).element_size()
            for d in shape:
                k *= d
            views.append(flat[o:o + k].view(dt).view(shape))
        return flat, views

    # ---- device work of one step -------------------------------------------------------------
    def _fwd(self):
        """part A of the step: everything that does not need the ground-truth batch"""
        if self.peer is not None:      # new epoch: the peers have finished reading this rank's gradient buffer
            self._dp_begin()
        for p, _ in self.loose:
            p.grad = None
        self.net.keep_encoder_conv_out = bool(self.split)
        self._fwd_out = self.net.forward_recon(self.x, self.y_hot, m_type="train", eps=self.eps)
        if self.split:
            self._cut, self.net.encoder_conv_out = self.net.encoder_conv_out, None

    def _loss_bwd(self, part: int = 0):
        """part B: loss (needs x_gt), backward, gradients of the few autograd-routed parameters.
        part 0 = all of it; part 1 = down to the encoder's last pooled output (every gradient of bucket 1 is then
        final); part 2 = the encoder convolutions."""
        if part in (0, 1):
            recon, z, mu, logvar, z_, y_hat = self._fwd_out
            loss, correct, kld, rec = self.net.loss_function(self.x_gt, recon, z, mu, logvar, self.y_hot, y_hat)
            self.loss.copy_(loss.detach())
            # per-batch statistics of main.py:83-85: the tensors stay device-resident (static addresses under
            # graph replay); stats() reduces them on demand instead of inside every step
            self.kld, self.rec, self.correct = kld, rec, correct
            if self.sigma_mode != "fixed":
                self.log_sigma = self.net.last_log_sigma
            self.recon = recon.detach()         # [B,N,3] view of the decoder buffer (no autograd graph attached)
            self._fwd_out = None
        _lib.defer_side_chains(True)          # weight-gradient chains of the conv layers run beside the following layers
        try:
            sel = self._backward_part(part, loss if part in (0, 1) else None)
        finally:
            # joined at the end of the backward pass; after part 1 only when a stream capture ends there (the
            # three-graph scheme) - in the one-graph step the chains of the decoder keep running under the encoder backward
            if part != 1 or not self._capturing_one_graph:
                _lib.side_join()
            else:
                _lib.side_join(lane=1)          # the dense layers' dW / db (bucket 1) must be final before its all-reduce
            _lib.defer_side_chains(False)
        if sel:       # autograd-routed gradients into their views (all of them live in bucket 2)
            torch._foreach_copy_([v for _, v in sel], [p.grad for p, _ in sel])

    def _backward_part(self, part: int, loss):
        if part == 0:
            loss.backward()
            self._cut = None
            sel = self.loose
        elif part == 1:
            sel = [(p, v) for p, v in self.loose if id(p) not in self._enc_ids]
            grads = torch.autograd.grad(loss, [self._cut] + [p for p, _ in sel])
            self._cut_grad = grads[0]
            for (p, _), g in zip(sel, grads[1:]):
                p.grad = g
        else:
            sel = [(p, v) for p, v in self.loose if id(p) in self._enc_ids]
            torch.autograd.backward([self._cut], [self._cut_grad])
            self._cut = self._cut_grad = None
        return sel

    def _fwd_bwd(self):
        self._fwd()
        self._loss_bwd()

    def stats(self):
        """(mean kld, mean rec_loss, correct) of the last step - main.py:83-85 reads these per batch (the decoder log sigma
        of the step is `log_sigma`)"""
        return float(self.kld.mean()), float(self.rec.mean()), int(self.correct)

    def _dp_begin(self):
        check(lib.mvb_dp_begin(self.peer.world, self.peer.rank, 2 if self.split else 1, self.peer.pad_ptrs, ptr(self.peer.state),
                               stream_ptr()), "mvb_dp_begin")

    def _optim(self):
        if self.peer is None:
            self.opt.step(1.0 / self.world)
        elif self.split:        # the two gradient buckets, one after the other (warm-up and ragged steps; the captured step overlaps them)
            self._optim_bucket(1)
            self._optim_bucket(2)
        else:
            self.opt.step_peers(self.peer, 1.0 / self.world)

    def _optim_bucket(self, which: int, background: bool = False):
        """fused exchange + Adam of one gradient bucket: 1 = everything behind `split` (the dense layers - final once the
        backward pass has reached the encoder), 2 = the convolutions in front of it"""
        if which == 1:
            self.opt.step_peers(self.peer, 1.0 / self.world, lo=self.split, hi=self.opt.n, channel=0, tick=True,
                                max_ctas=self._bg_ctas if background else 0)
        else:
            self.opt.step_peers(self.peer, 1.0 / self.world, lo=0, hi=self.split, channel=1, tick=False)

    def capture(self, warmup: int = 3):
        """warm up on a side stream (lazy init, cuBLAS workspaces), then capture the graphs"""
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        state = (self.opt.flat_p.clone(), self.opt.m.clone(), self.opt.v.clone(), self.opt.step_count.clone())
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self._fwd_bwd()
                self._optim()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        # warm-up must not train: restore parameters and optimizer state
        self.opt.flat_p.copy_(state[0]); self.opt.m.copy_(state[1]); self.opt.v.copy_(state[2])
        self.opt.step_count.copy_(state[3])
        if not self.use_graph:
            c0 = lib.mvb_launch_count()
            self._fwd_bwd(); self._optim()
            self.launches_per_step = lib.mvb_launch_count() - c0
            self.opt.flat_p.copy_(state[0]); self.opt.m.copy_(state[1]); self.opt.v.copy_(state[2])
            self.opt.step_count.copy_(state[3])
            return
        c0 = lib.mvb_launch_count()
        # ONE graph on a single GPU: forward, an EXTERNAL event-wait node (the ground-truth H2D copy that
        # step() issues on the copy stream - the fp64 ground truth is 2/3 of the H2D bytes and is only needed by
        # the loss), loss + backward, Adam.  Data parallel: the optimizer is a second graph so that the NCCL
        # all-reduce of the flat gradient buffer runs between the two.
        self._copy_stream = torch.cuda.Stream()
        self._gt_ready = torch.cuda.Event()
        self._gt_ready.record(self._copy_stream)
        torch.cuda.synchronize()
        # all captures on ONE stream: autograd replays a node's backward on the stream of its forward, so the
        # encoder backward (its own graph when the gradient buckets are split) must be captured on that stream
        cap = torch.cuda.Stream()
        self.one_graph = not self.distributed or self.peer is not None
        if self.peer is not None:
            # data parallel through peer memory: the whole step - exchange included - is kernels of this library
            dist.barrier()
            g = torch.cuda.CUDAGraph()
            # (highest priority with PDL on - see __init__; ordinary priority when PDL is off)
            side = torch.cuda.Stream(priority=-1) if os.environ.get("MVB_DP_PDL", "1") != "0" else torch.cuda.Stream()
            self._bg_ctas = int(os.environ.get("MVB_DP_BG_CTAS", "40"))          # 8 GPUs: 16 -> 0.984 ms, 40 -> 0.965, 74 -> 0.974, 148 -> 0.973
            with torch.cuda.graph(g, stream=cap):
                self._fwd()
                check(lib.mvb_stream_wait_external_event(stream_ptr(), self._gt_ready.cuda_event), "mvb_stream_wait_external_event")
                if self.split:
                    # bucket 1 (the dense layers, 99 % of the bytes) is exchanged and stepped on a side branch of the graph
                    # while the encoder backward computes; the small bucket of the convolutions follows at the end
                    self._capturing_one_graph = True
                    try:
                        self._loss_bwd(1)
                        side.wait_stream(cap)
                        with torch.cuda.stream(side):
                            self._optim_bucket(1, background=True)
                        self._loss_bwd(2)
                    finally:
                        self._capturing_one_graph = False
                    cap.wait_stream(side)
                    self._optim_bucket(2)
                else:
                    self._loss_bwd(0)
                    self._optim()
            self.g_fb = g
            self.launches_per_step = lib.mvb_launch_count() - c0
            torch.cuda.synchronize()
            return
        if self.distributed and self.graph_comm:
            # Data parallel, ONE graph: the bucketed NCCL all-reduces are captured with the step (NCCL enqueues on its own
            # stream; fork / join become graph edges), so a step is a single replay - no host launch between backward,
            # exchange and optimizer, and the big bucket still overlaps the encoder backward.
            try:
                warm = torch.zeros(8, device=self.dev)
                dist.all_reduce(warm)                       # communicator set-up outside the capture
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                self._capturing_one_graph = True
                with torch.cuda.graph(g, stream=cap):
                    self._fwd()
                    check(lib.mvb_stream_wait_external_event(stream_ptr(), self._gt_ready.cuda_event), "mvb_stream_wait_external_event")
                    if self.split:
                        self._loss_bwd(1)
                        w1 = dist.all_reduce(self.opt.flat_g[self.split:], op=dist.ReduceOp.SUM, async_op=True)
                        self._loss_bwd(2)
                        w2 = dist.all_reduce(self.opt.flat_g[:self.split], op=dist.ReduceOp.SUM, async_op=True)
                        w1.wait()
                        w2.wait()
                    else:
                        self._loss_bwd(0)
                        dist.all_reduce(self.opt.flat_g, op=dist.ReduceOp.SUM)
                    self._optim()
                self._capturing_one_graph = False
                self.g_fb, self.one_graph = g, True
                self.launches_per_step = lib.mvb_launch_count() - c0
                torch.cuda.synchronize()
                return
            except Exception as e:  # noqa: BLE001  (a build of torch / NCCL that cannot capture collectives): three graphs below
                self._capturing_one_graph = False
                import warnings
                warnings.warn(f"TrainEngine: the data-parallel step could not be captured as one graph ({e}); "
                              "falling back to three graphs with host-launched all-reduces")
                torch.cuda.synchronize()
                self.opt.flat_p.copy_(state[0]); self.opt.m.copy_(state[1]); self.opt.v.copy_(state[2])
                self.opt.step_count.copy_(state[3])
                c0 = lib.mvb_launch_count()
        self.g_fb = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_fb, stream=cap):
            self._fwd()
            check(lib.mvb_stream_wait_external_event(stream_ptr(), self._gt_ready.cuda_event), "mvb_stream_wait_external_event")
            self._loss_bwd(1 if self.split else 0)
            if not self.distributed:
                self._optim()
        if self.distributed:
            if self.split:
                self.g_enc = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.g_enc, pool=self.g_fb.pool(), stream=cap):
                    self._loss_bwd(2)
            self.g_opt = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g_opt, pool=self.g_fb.pool(), stream=cap):
                self._optim()
        self.launches_per_step = lib.mvb_launch_count() - c0
        torch.cuda.synchronize()

    def device_step(self):
        """one training step on inputs already resident in the static device buffers"""
        if self.use_graph and self.one_graph:
            self.g_fb.replay()               # the whole step, collectives included
            return
        if self.use_graph:
            self.g_fb.replay()
        else:
            self._fwd()
            if self._gt_ready is not None:
                torch.cuda.current_stream().wait_event(self._gt_ready)
            self._loss_bwd()
        if self.distributed and self.peer is None:
            if self.use_graph and self.split:
                # bucket 1 is reduced on NCCL's stream while graph g_enc computes the encoder backward
                w1 = dist.all_reduce(self.opt.flat_g[self.split:], op=dist.ReduceOp.SUM, async_op=True)
                self.g_enc.replay()
                w2 = dist.all_reduce(self.opt.flat_g[:self.split], op=dist.ReduceOp.SUM, async_op=True)
                w1.wait()
                w2.wait()
            else:
                dp.allreduce_sum_(self.opt.flat_g)
        if self.use_graph:
            if self.distributed and self.peer is None:
                self.g_opt.replay()
        else:
            self._optim()

    # ---- the public per-batch call (host buffers in, loss out) ---------------------------------
    def step(self, x_host: torch.Tensor, x_gt_host: torch.Tensor, y_host: torch.Tensor,
             eps_host: Optional[torch.Tensor] = None, sync: bool = True) -> Optional[float]:
        """x_host [B,N,3] f32, x_gt_host [B,N,3] f64/f32, y_host [B] int64 labels (pinned host memory for
        asynchronous copies).  Mirrors main.py:69-85: H2D, one-hot, step, loss read-back.  The ground truth
        travels on a second stream while the forward pass runs."""
        main = torch.cuda.current_stream()
        self.x.copy_(x_host, non_blocking=True)
        if eps_host is None:   # the reference draws the noise on the CPU generator (cheb_VAE.py:316)
            eps_host = torch.normal(mean=0, std=1, size=(self.batch, self.net.z))
        self.eps.copy_(eps_host, non_blocking=True)
        # one-hot on the host, then H2D, as main.py:71 does
        self.y_hot.copy_(torch.nn.functional.one_hot(y_host, self.net.num_class), non_blocking=True)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
            self._gt_ready = torch.cuda.Event()
        self._copy_stream.wait_stream(main)          # the previous step's loss kernel has read x_gt
        with torch.cuda.stream(self._copy_stream):
            self.x_gt.copy_(x_gt_host, non_blocking=True)
            self._gt_ready.record(self._copy_stream)
        self.device_step()
        if not sync:                     # the epoch loop (loop.train_epoch) accumulates on the device instead
            return None
        return float(self.loss)          # D2H read of the step's loss (synchronises)

    # ---- input double-buffering: batch i+1 travels to the device while step i computes ------------------------
    def stage(self, x_host: torch.Tensor, x_gt_host: torch.Tensor, y_host: torch.Tensor,
              eps_host: Optional[torch.Tensor] = None) -> None:
        """Enqueue the host->device copies of the NEXT batch on the copy stream and return at once (pinned host
        tensors).  The copies land in staging buffers; `step_prefetched` moves them into the step's static buffers
        (device-to-device, a few microseconds) when the previous step no longer reads those."""
        if self._stage is None:
            self._stage_flat, self._stage = self._alloc_inputs()
            self._ev_staged, self._ev_consumed = torch.cuda.Event(), torch.cuda.Event()
            self._ev_consumed.record(torch.cuda.current_stream())
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
            self._gt_ready = torch.cuda.Event()
        if self._h_small is None:
            # pinned homes for the two small host-made operands: a copy from pageable memory would synchronise the
            # copy stream on the host - behind the 11 MB of mesh data - before anything else could be launched
            self._h_small = (torch.empty(self.eps.shape, dtype=self.eps.dtype).pin_memory(),
                             torch.empty(self.y_hot.shape, dtype=self.y_hot.dtype).pin_memory())
        else:
            self._ev_staged.synchronize()           # the previous copies out of the pinned homes have been made
        if eps_host is None:
            eps_host = torch.normal(mean=0, std=1, size=(self.batch, self.net.z))
        self._h_small[0].copy_(eps_host)
        self._h_small[1].copy_(torch.nn.functional.one_hot(y_host, self.net.num_class))
        cs = self._copy_stream
        cs.wait_event(self._ev_consumed)            # the staging buffers have been emptied
        with torch.cuda.stream(cs):
            for dst, src in zip(self._stage, (x_host, x_gt_host, self._h_small[0], self._h_small[1])):
                dst.copy_(src, non_blocking=True)
            self._ev_staged.record(cs)
        self._staged = True

    def step_prefetched(self, next_batch=None, sync: bool = True) -> Optional[float]:
        """One step on the batch handed to `stage()` earlier; `next_batch` = (x_host, x_gt_host, y_host[, eps_host]) is
        staged while this step computes.  Same work per step as `step()` - every batch is copied from the host once
        and the loss is read back - with the copy of batch i+1 overlapping the kernels of step i."""
        if not self._staged:
            raise RuntimeError("step_prefetched: no staged batch (call stage() first)")
        main = torch.cuda.current_stream()
        main.wait_event(self._ev_staged)
        self._in_flat.copy_(self._stage_flat)         # one device-to-device copy for all four inputs
        self._ev_consumed.record(main)
        self._gt_ready.record(main)                  # the step graph's external wait node: the ground truth is in place
        self._staged = False
        self.device_step()                           # launched first: the copies below then overlap its kernels
        if next_batch is not None:
            self.stage(*next_batch)
        if not sync:
            return None
        return float(self.loss)

    def wait_staged(self) -> None:
        """make the current stream wait for the staged copies (for timing: the interval then covers the H2D)"""
        if self._staged:
            torch.cuda.current_stream().wait_event(self._ev_staged)

    def ragged_step(self, x: torch.Tensor, x_gt: torch.Tensor, y_hot: torch.Tensor, eps: Optional[torch.Tensor] = None,
                    grad_weight: float = 1.0):
        """the last, smaller batch of an epoch (DataLoader without drop_last, main.py:256): same kernels, same flat
        optimizer, not graph-replayed (the graphs are captured for `batch` meshes).  Device tensors in.
        Data parallel: EVERY rank must take this path for the same step (one all-reduce of the whole flat buffer, where
        the graph path issues two bucketed ones - loop.train_epoch decides from the global batch size); `grad_weight`
        = dp.ragged_weight(...) makes the average over ranks the gradient of the global-batch mean when the slices
        are unequal (0 for a rank that only holds a stand-in item)."""
        if self.peer is not None:
            self._dp_begin()
        for p, _ in self.loose:
            p.grad = None
        self.net.keep_encoder_conv_out = False
        if eps is None:
            eps = torch.normal(mean=0, std=1, size=(x.shape[0], self.net.z)).to(self.dev)
        loss, correct, recon, (kld, rec, _), _ = self.net(x, x_gt, y_hot, m_type="train", eps=eps)
        loss.backward()
        if self.loose:
            torch._foreach_copy_([v for _, v in self.loose], [p.grad for p, _ in self.loose])
        if self.distributed:
            if grad_weight != 1.0:
                self.opt.flat_g.mul_(float(grad_weight))
            if self.peer is None:
                dp.allreduce_sum_(self.opt.flat_g)
        self._optim()
        return loss.detach(), kld, rec, correct, recon.detach()

    def h2d_bytes(self) -> int:
        return (self.x.numel() * self.x.element_size() + self.x_gt.numel() * self.x_gt.element_size()
                + self.eps.numel() * 4 + self.y_hot.numel() * 8)

    def d2h_bytes(self) -> int:
        return 8
