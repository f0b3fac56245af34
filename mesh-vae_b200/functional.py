"""torch.autograd glue over the C ABI.  PyTorch supplies device memory, streams and the autograd
tape; all arithmetic of the hot path happens in libmvb_sm100a.so.  Tensors that cross into the
library are fp32 CUDA tensors in the VERTEX-MAJOR layout [N, B, F] (see include/mvb.h).

No CPU fallback: a non-CUDA tensor raises."""
from typing import Optional

import torch

from . import _lib
from ._lib import lib, check, ptr, stream_ptr
from .operators import MeshOperator

LOG_SIGMA_DEFAULT = 1.0009117126464844      # softclip(1, -6) in fp32 (models/cheb_VAE.py:328-329)


def _req_cuda(t: torch.Tensor, name: str, dtype=torch.float32):
    if not t.is_cuda:
        raise _lib.MvbError(f"{name}: expected a CUDA tensor - this package has no CPU path")
    if dtype is not None and t.dtype != dtype:
        raise _lib.MvbError(f"{name}: expected {dtype}, got {t.dtype}")


def _sink(t):
    """Gradient sink of a Parameter: a contiguous view (of the engine's flat gradient buffer) that the
    backward kernels write straight into; the Function then returns None for that input, so autograd
    neither allocates nor copies (engine.TrainEngine installs the sinks; absent = ordinary autograd)."""
    return None if t is None else getattr(t, "_mvb_grad_sink", None)


def _grad_outs(sinks, w, n_bias):
    """(dw, db) for a backward kernel to write: the Parameters' gradient sinks where installed, else new tensors;
    db is None when n_bias is None (no bias)"""
    sw, sb = sinks
    dw = sw if sw is not None else torch.empty_like(w)
    if n_bias is None:
        return dw, None
    return dw, (sb if sb is not None else torch.empty(n_bias, device=w.device, dtype=torch.float32))


def _park_or_join(ctx, tensors):
    """deferred mode: park the tensors a backward call's pending side chain still reads or writes until side_join, or
    join now when a gradient goes back to autograd (it must be complete on this stream) instead of into a sink"""
    if not _lib._deferred["on"]:
        return
    sw, sb = ctx.sinks
    if sw is not None and (sb is not None or not ctx.has_bias):
        _lib._deferred["keep"].append(tensors)
    else:
        _lib.side_join()


def _ret(sinks, dw, db):
    """backward's return values for (weight, bias): None for a gradient that went into its sink"""
    sw, sb = sinks
    return (None if sw is not None else dw), (None if sb is not None else db)


def to_vertex_major(x: torch.Tensor) -> torch.Tensor:
    """logical [B, N, F] (any strides) -> physical [N, B, F] contiguous; free when x is already a
    permuted view of a vertex-major buffer (which is what every module of this package returns)."""
    xt = x.permute(1, 0, 2)
    return xt if xt.is_contiguous() else xt.contiguous()


def from_vertex_major(x_vm: torch.Tensor) -> torch.Tensor:
    """physical [N, B, F] -> logical [B, N, F] strided view (no copy)."""
    return x_vm.permute(1, 0, 2)


class _ChebConvFn(torch.autograd.Function):
    """mvb_cheb_fwd / mvb_cheb_bwd  (nn/conv.py:557-577 and its autograd).  With `norm` (the COO values of an
    operators.EdgePattern) the operator is bound to those values here, and when `norm` needs a gradient the backward
    pass is mvb_cheb_bwd_op, which also returns d_norm."""

    @staticmethod
    def forward(ctx, x_vm, weight, bias, op, relu: bool, norm=None):
        _req_cuda(x_vm, "cheb_conv x")
        _req_cuda(weight, "cheb_conv weight")
        n, b, fin = x_vm.shape
        k, fin_w, fout = weight.shape
        if fin_w != fin:
            raise _lib.MvbError(f"cheb_conv: x has {fin} features, weight expects {fin_w}")
        if op.n_rows != n or op.n_cols != n:
            raise _lib.MvbError(f"cheb_conv: operator is {op.n_rows}x{op.n_cols}, tensor has {n} vertices")
        if norm is not None:
            op = op.bind(norm)
        x_vm = x_vm.contiguous()
        w = weight.contiguous()
        bb = None if bias is None else bias.contiguous()
        na = op.n_active
        basis = torch.empty((max(k - 1, 0), na, b, fin), device=x_vm.device, dtype=torch.float32)
        y = torch.empty((n, b, fout), device=x_vm.device, dtype=torch.float32)
        check(lib.mvb_cheb_fwd(n, b, fin, fout, k, na, op.nnz, ptr(op.rowptr), ptr(op.colidx), ptr(op.vals), ptr(x_vm), ptr(w),
                               ptr(bb), 1 if relu else 0, ptr(basis) if basis.numel() else None, ptr(y), stream_ptr()),
              "mvb_cheb_fwd")
        ctx.op, ctx.relu, ctx.has_bias = op, relu, bias is not None
        ctx.sinks = (_sink(weight), _sink(bias))
        ctx.op_grad = norm is not None and ctx.needs_input_grad[5]
        # the adjoint-form backward recomputes its planes from dY: the forward basis is then a temporary (the operator
        # gradient reads it: always the basis form)
        keep = ctx.op_grad or bool(lib.mvb_cheb_bwd_uses_basis(fin, fout, 1 if ctx.needs_input_grad[0] else 0))
        ctx.save_for_backward(x_vm, basis if keep else None, w, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_vm, basis, w, y = ctx.saved_tensors
        op = ctx.op
        n, b, fin = x_vm.shape
        k, _, fout = w.shape
        dy = dy.contiguous()
        need_dx = ctx.needs_input_grad[0]
        dx = torch.empty_like(x_vm) if need_dx else None
        dw, db = _grad_outs(ctx.sinks, w, fout if ctx.has_bias else None)
        na = op.n_active
        basis_p = ptr(basis) if (basis is not None and basis.numel()) else None
        if ctx.op_grad:
            d_norm = torch.empty(op.nnz, device=w.device, dtype=torch.float32)
            ws_bytes = lib.mvb_cheb_bwd_op_workspace_bytes(n, b, fin, fout, k, na)
            ws = torch.empty(ws_bytes, device=w.device, dtype=torch.uint8)
            check(lib.mvb_cheb_bwd_op(n, b, fin, fout, k, na, op.nnz, ptr(op.rowptr), ptr(op.colidx), ptr(op.perm),
                                      ptr(op.rowptr_t), ptr(op.colidx_t), ptr(op.vals_t), ptr(x_vm), basis_p, ptr(w),
                                      ptr(y) if ctx.relu else None, ptr(dy), ptr(dx), ptr(dw), ptr(db), ptr(d_norm), ptr(ws),
                                      ws_bytes, stream_ptr()), "mvb_cheb_bwd_op")
            return dx, *_ret(ctx.sinks, dw, db), None, None, d_norm
        ws_bytes = lib.mvb_cheb_bwd_workspace_bytes(n, b, fin, fout, k, na, 1 if need_dx else 0)
        ws = torch.empty(ws_bytes, device=w.device, dtype=torch.uint8)
        check(lib.mvb_cheb_bwd(n, b, fin, fout, k, na, op.nnz, ptr(op.rowptr_t), ptr(op.colidx_t), ptr(op.vals_t), ptr(x_vm),
                               basis_p, ptr(w), ptr(y) if ctx.relu else None,
                               ptr(dy), ptr(dx),
                               ptr(dw), ptr(db), ptr(ws), ws_bytes, stream_ptr()), "mvb_cheb_bwd")
        _park_or_join(ctx, (ws, x_vm, basis, w, y, dy, dw, db))
        return dx, *_ret(ctx.sinks, dw, db), None, None, None


def cheb_conv(x_vm: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], op: MeshOperator,
              relu: bool = False, pad_to_quads: bool = True, keep_padding: bool = False,
              norm: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x_vm [N,B,Fin] -> [N,B,Fout] (vertex-major in, vertex-major out).

    With `norm` (fp32 [nnz], COO order), `op` is an operators.EdgePattern and norm its values: the result is
    differentiable with respect to norm.

    Feature widths that are not a multiple of 4 (the 3-channel mesh coordinates at the encoder
    input and the decoder output) are zero-padded to the next multiple of 4 around the kernel call,
    so that every plane is made of whole 16-byte quads: the SpMM takes its vector path and the
    contractions run on the tcgen05 kernels instead of the scalar FFMA fallback.  Zero features /
    zero weight columns do not change any result; the padding ops are differentiable torch glue
    (autograd slices the padded weight gradient back)."""
    fin_x, fin, fout = x_vm.shape[2], weight.shape[1], weight.shape[2]
    if fin_x != fin and not (fin_x > fin and fin_x == fin + (-fin) % 4):
        raise _lib.MvbError(f"cheb_conv: x has {fin_x} features, weight expects {fin}")
    pin, pout = (-fin) % 4, (-fout) % 4
    if not pad_to_quads or (pin == 0 and pout == 0):
        return _ChebConvFn.apply(x_vm, weight, bias, op, relu, norm)
    if pin and fin_x == fin:             # (an input packed by pack_input already carries the zero column)
        x_vm = torch.nn.functional.pad(x_vm, (0, pin))
    w = torch.nn.functional.pad(weight, (0, pout, 0, pin))
    b = bias if (bias is None or pout == 0) else torch.nn.functional.pad(bias, (0, pout))
    y = _ChebConvFn.apply(x_vm, w, b, op, relu, norm)
    if pout and keep_padding:
        return y                         # [N,B,fout+pout]: the caller slices a view and hands the padded buffer to the loss
    return y[..., :fout] if pout else y


class _ChebConvSelFn(torch.autograd.Function):
    """mvb_cheb_sel_fwd / mvb_cheb_sel_bwd: ChebConv (+bias, ReLU) followed by the row selection of a down-sampling
    operator (models/cheb_VAE.py:264-265) for a layer whose input needs no gradient (the first encoder layer)."""

    @staticmethod
    def forward(ctx, x_vm, weight, bias, op: MeshOperator, d_op: MeshOperator, relu: bool):
        _req_cuda(x_vm, "cheb_conv_sel x")
        n, b, fin = x_vm.shape
        k, _, fout = weight.shape
        x_vm, w = x_vm.contiguous(), weight.contiguous()
        bb = None if bias is None else bias.contiguous()
        n_sel = d_op.n_rows
        basis = torch.empty((max(k - 1, 0), n, b, fin), device=x_vm.device, dtype=torch.float32)
        y = torch.empty((n_sel, b, fout), device=x_vm.device, dtype=torch.float32)
        check(lib.mvb_cheb_sel_fwd(n, b, fin, fout, k, op.nnz, ptr(op.rowptr), ptr(op.colidx), ptr(op.vals), ptr(x_vm), ptr(w),
                                   ptr(bb), 1 if relu else 0, n_sel, ptr(d_op.colidx), ptr(basis) if basis.numel() else None,
                                   ptr(y), stream_ptr()), "mvb_cheb_sel_fwd")
        ctx.d_op, ctx.relu, ctx.has_bias = d_op, relu, bias is not None
        ctx.sinks = (_sink(weight), _sink(bias))
        ctx.save_for_backward(x_vm, basis, w, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_vm, basis, w, y = ctx.saved_tensors
        n, b, fin = x_vm.shape
        k, _, fout = w.shape
        dy = dy.contiguous()
        dw, db = _grad_outs(ctx.sinks, w, fout if ctx.has_bias else None)
        ws_bytes = lib.mvb_cheb_sel_bwd_workspace_bytes(fin, fout, k)
        ws = torch.empty(ws_bytes, device=w.device, dtype=torch.uint8)
        check(lib.mvb_cheb_sel_bwd(n, b, fin, fout, k, ptr(x_vm), ptr(basis) if basis.numel() else None, ptr(y) if ctx.relu else None,
                                   ptr(dy), ctx.d_op.n_rows, ptr(ctx.d_op.colidx), ptr(dw), ptr(db), ptr(ws), ws_bytes, stream_ptr()),
              "mvb_cheb_sel_bwd")
        return None, *_ret(ctx.sinks, dw, db), None, None, None


def cheb_conv_sel_supported(x_vm: torch.Tensor, weight: torch.Tensor, op: MeshOperator, d_op: Optional[MeshOperator]) -> bool:
    """the conv + row-selection kernels cover this layer: a selection D, an input without gradient, plane widths of
    the tensor-core kernels (3 input channels count as 4: zero padded)"""
    if d_op is None or not d_op.is_selection or x_vm.requires_grad or not x_vm.is_cuda:
        return False
    if op.n_active != op.n_rows or op.n_rows != x_vm.shape[0]:
        return False
    k, fin, fout = weight.shape
    finp = fin + (-fin) % 4
    return bool(lib.mvb_cheb_sel_supported(op.n_rows, x_vm.shape[1], finp, fout, k, d_op.n_rows))


def cheb_conv_sel(x_vm: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], op: MeshOperator, d_op: MeshOperator,
                  relu: bool = True) -> torch.Tensor:
    """x_vm [N,B,Fin] (no gradient) -> [n_sel,B,Fout] = act(conv(x))[rows D keeps]; see cheb_conv for the zero padding of
    3-channel inputs (the padded weight's gradient is sliced back by autograd)."""
    fin_x, fin = x_vm.shape[2], weight.shape[1]
    pin = (-fin) % 4
    if pin and fin_x == fin:
        x_vm = torch.nn.functional.pad(x_vm, (0, pin))
    w = torch.nn.functional.pad(weight, (0, 0, 0, pin)) if pin else weight
    return _ChebConvSelFn.apply(x_vm, w, bias, op, d_op, relu)


def pack_input(x: torch.Tensor) -> torch.Tensor:
    """[B,N,C] mesh-major input (no gradient) -> vertex-major [N,B,Cp] with Cp = C rounded up to 4, zero padded:
    one kernel instead of the transpose copy + fill + padded copy."""
    _req_cuda(x, "pack_input x")
    b, n, c = x.shape
    cp = c + (-c) % 4
    x = x.contiguous()
    out = torch.empty((n, b, cp), device=x.device, dtype=torch.float32)
    check(lib.mvb_pack_vertex_major(b, n, c, cp, ptr(x), ptr(out), stream_ptr()), "mvb_pack_vertex_major")
    return out


class _PoolFn(torch.autograd.Function):
    """mvb_pool_fwd / mvb_pool_bwd  (nn/pool.py:13-23; models/cheb_cls.py:22-27)."""

    @staticmethod
    def forward(ctx, x_vm, op: MeshOperator):
        _req_cuda(x_vm, "pool x")
        n, b, f = x_vm.shape
        if n != op.n_cols:
            raise _lib.MvbError(f"pool: operator has {op.n_cols} columns, tensor has {n} vertices")
        x_vm = x_vm.contiguous()
        y = torch.empty((op.n_rows, b, f), device=x_vm.device, dtype=torch.float32)
        check(lib.mvb_pool_fwd(op.n_rows, op.n_cols, ptr(op.rowptr), ptr(op.colidx), ptr(op.vals), ptr(x_vm), ptr(y), b * f,
                               stream_ptr()), "mvb_pool_fwd")
        ctx.op = op
        return y

    @staticmethod
    def backward(ctx, dy):
        op = ctx.op
        dy = dy.contiguous()
        _, b, f = dy.shape
        dx = torch.empty((op.n_cols, b, f), device=dy.device, dtype=torch.float32)
        check(lib.mvb_pool_bwd(op.n_cols, op.n_rows, ptr(op.rowptr_t), ptr(op.colidx_t), ptr(op.vals_t), ptr(dy), ptr(dx), b * f,
                               stream_ptr()), "mvb_pool_bwd")
        return dx, None


def pool(x_vm: torch.Tensor, op: MeshOperator) -> torch.Tensor:
    """x_vm [N,B,F] -> [M,B,F] = P x (vertex-major)."""
    return _PoolFn.apply(x_vm, op)


class _ReparamFn(torch.autograd.Function):
    """mvb_vae_reparam_fwd / _bwd  (models/cheb_VAE.py:309-319)."""

    @staticmethod
    def forward(ctx, mu, logvar, eps):
        _req_cuda(mu, "reparam mu")
        mu, logvar, eps = mu.contiguous(), logvar.contiguous(), eps.contiguous()
        _req_cuda(eps, "reparam eps")
        z = torch.empty_like(mu)
        check(lib.mvb_vae_reparam_fwd(mu.numel(), ptr(mu), ptr(logvar), ptr(eps), ptr(z), stream_ptr()),
              "mvb_vae_reparam_fwd")
        ctx.save_for_backward(logvar, eps)
        return z

    @staticmethod
    def backward(ctx, dz):
        logvar, eps = ctx.saved_tensors
        dz = dz.contiguous()
        dmu, dlv = torch.empty_like(dz), torch.empty_like(dz)
        check(lib.mvb_vae_reparam_bwd(dz.numel(), ptr(logvar), ptr(eps), ptr(dz), ptr(dmu), ptr(dlv), stream_ptr()),
              "mvb_vae_reparam_bwd")
        return dmu, dlv, None


def reparameterize(mu, logvar, eps):
    return _ReparamFn.apply(mu, logvar, eps)


def _loss_operands(recon_vm, x_gt, mu, logvar, y_hat, y, channels: int):
    """checked, contiguous operands of the loss epilogue, its sizes (n, b, c, z, ncls, ld, x_gt is fp64) and its
    outputs (loss, kld, rec, correct, dnll, workspace, workspace bytes)"""
    _req_cuda(recon_vm, "vae_loss recon")
    _req_cuda(x_gt, "vae_loss x_gt", None)
    if x_gt.dtype not in (torch.float32, torch.float64):
        raise _lib.MvbError(f"vae_loss: x_gt must be fp32 or fp64, got {x_gt.dtype}")
    n, b, ld = recon_vm.shape                    # entries of ld floats, the first `channels` are the reconstruction
    c = channels
    if tuple(x_gt.shape) != (b, n, c) or c > ld:
        raise _lib.MvbError(f"vae_loss: x_gt is {tuple(x_gt.shape)}, expected {(b, n, c)}")
    z = mu.shape[1]
    ncls = y_hat.shape[1]
    recon_vm, x_gt = recon_vm.contiguous(), x_gt.contiguous()
    mu, logvar, y_hat = mu.contiguous(), logvar.contiguous(), y_hat.contiguous()
    y = y.to(torch.int64).contiguous()
    dev = recon_vm.device
    f64 = x_gt.dtype == torch.float64
    loss = torch.empty((), device=dev, dtype=torch.float64)
    kld = torch.empty(b, device=dev, dtype=torch.float32)
    rec = torch.empty(b, device=dev, dtype=torch.float64)
    correct = torch.empty((), device=dev, dtype=torch.int64)
    dnll = torch.empty_like(recon_vm)
    ws_bytes = lib.mvb_vae_loss_workspace_bytes(b, n)
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    return (recon_vm, x_gt, mu, logvar, y_hat, y), (n, b, c, z, ncls, ld, f64), (loss, kld, rec, correct, dnll, ws, ws_bytes)


class _VaeLossFn(torch.autograd.Function):
    """mvb_vae_loss_fwd / _bwd  (models/cheb_VAE.py:321-346)."""

    @staticmethod
    def forward(ctx, recon_vm, x_gt, mu, logvar, y_hat, y, log_sigma: float, channels: int):
        (recon_vm, x_gt, mu, logvar, y_hat, y), (n, b, c, z, ncls, ld, f64), (loss, kld, rec, correct, dnll, ws, ws_bytes) = \
            _loss_operands(recon_vm, x_gt, mu, logvar, y_hat, y, channels)
        check(lib.mvb_vae_loss_fwd(b, n, c, z, ncls, ptr(recon_vm), ld, ptr(x_gt), 1 if f64 else 0, ptr(mu), ptr(logvar),
                                   ptr(y_hat), ptr(y), float(log_sigma), ptr(loss), ptr(kld), ptr(rec), ptr(correct),
                                   ptr(dnll), ptr(ws), ws_bytes, stream_ptr()), "mvb_vae_loss_fwd")
        ctx.save_for_backward(dnll, mu, logvar, y_hat, y)
        ctx.dims = (b, n, ld, z, ncls)
        ctx.set_materialize_grads(False)          # no zero tensors for the undefined grads of kld / rec / correct
        if not f64:                     # all-fp32 call (inference.py:87): the reference returns fp32
            loss, rec = loss.float(), rec.float()
        ctx.mark_non_differentiable(kld, rec, correct)
        return loss, kld, rec, correct

    @staticmethod
    def backward(ctx, gloss, _gk, _gr, _gc):
        dnll, mu, logvar, y_hat, y = ctx.saved_tensors
        b, n, c, z, ncls = ctx.dims
        g = gloss.to(torch.float64).contiguous()
        need = ctx.needs_input_grad
        d_recon = torch.empty_like(dnll) if need[0] else None
        d_mu = torch.empty_like(mu) if need[2] else None
        d_lv = torch.empty_like(logvar) if need[3] else None
        d_yh = torch.empty_like(y_hat) if need[4] else None
        check(lib.mvb_vae_loss_bwd(b, n, c, z, ncls, ptr(dnll), ptr(mu), ptr(logvar), ptr(y_hat), ptr(y), ptr(g),
                                   ptr(d_recon), ptr(d_mu), ptr(d_lv), ptr(d_yh), stream_ptr()), "mvb_vae_loss_bwd")
        return d_recon, None, d_mu, d_lv, d_yh, None, None, None


SIGMA_STATE_DOUBLES = 8          # include/mvb.h: mvb_vae_loss_sigma_fwd's sigma_state


class _VaeLossSigmaFn(torch.autograd.Function):
    """mvb_vae_loss_sigma_fwd / _bwd: the loss with the sigma-VAE decoder log sigma, optimal (s_param None) or learned
    (sc(s_param), s_param a 1-element fp32 CUDA tensor whose gradient the backward kernel writes)."""

    @staticmethod
    def forward(ctx, recon_vm, x_gt, mu, logvar, y_hat, y, s_param, channels: int):
        (recon_vm, x_gt, mu, logvar, y_hat, y), (n, b, c, z, ncls, ld, f64), (loss, kld, rec, correct, dnll, ws, ws_bytes) = \
            _loss_operands(recon_vm, x_gt, mu, logvar, y_hat, y, channels)
        if s_param is not None:
            _req_cuda(s_param, "vae_loss log_sigma parameter")
            if s_param.numel() != 1:
                raise _lib.MvbError(f"vae_loss: a learned log_sigma has one element, got {tuple(s_param.shape)}")
        state = torch.empty(SIGMA_STATE_DOUBLES, device=recon_vm.device, dtype=torch.float64)
        s = None if s_param is None else s_param.detach().contiguous()
        check(lib.mvb_vae_loss_sigma_fwd(b, n, c, z, ncls, ptr(recon_vm), ld, ptr(x_gt), 1 if f64 else 0, ptr(mu), ptr(logvar),
                                         ptr(y_hat), ptr(y), 1 if s is None else 2, ptr(s), ptr(state), ptr(loss), ptr(kld),
                                         ptr(rec), ptr(correct), ptr(dnll), ptr(ws), ws_bytes, stream_ptr()),
              "mvb_vae_loss_sigma_fwd")
        ctx.save_for_backward(dnll, state, mu, logvar, y_hat, y)
        ctx.dims = (b, n, ld, z, ncls)
        ctx.s_sink = _sink(s_param)
        ctx.s_like = s_param
        ctx.set_materialize_grads(False)
        if not f64:
            loss, rec = loss.float(), rec.float()
        ctx.mark_non_differentiable(kld, rec, correct, state)
        return loss, kld, rec, correct, state

    @staticmethod
    def backward(ctx, gloss, _gk, _gr, _gc, _gs):
        dnll, state, mu, logvar, y_hat, y = ctx.saved_tensors
        b, n, c, z, ncls = ctx.dims
        g = gloss.to(torch.float64).contiguous()
        need = ctx.needs_input_grad
        d_recon = torch.empty_like(dnll) if need[0] else None
        d_mu = torch.empty_like(mu) if need[2] else None
        d_lv = torch.empty_like(logvar) if need[3] else None
        d_yh = torch.empty_like(y_hat) if need[4] else None
        d_s = None
        if need[6]:
            d_s = ctx.s_sink if ctx.s_sink is not None else torch.empty_like(ctx.s_like, memory_format=torch.contiguous_format)
        check(lib.mvb_vae_loss_sigma_bwd(b, n, c, z, ncls, ptr(dnll), ptr(state), ptr(mu), ptr(logvar), ptr(y_hat), ptr(y),
                                         ptr(g), ptr(d_recon), ptr(d_mu), ptr(d_lv), ptr(d_yh), ptr(d_s), stream_ptr()),
              "mvb_vae_loss_sigma_bwd")
        return d_recon, None, d_mu, d_lv, d_yh, None, (None if ctx.s_sink is not None else d_s), None


def vae_loss(recon_vm, x_gt, mu, logvar, y_hat, y, log_sigma=LOG_SIGMA_DEFAULT, channels: Optional[int] = None,
             return_log_sigma: bool = False):
    """-> (loss, kld[B], rec_loss[B], correct); only `loss` carries gradient (as main.py:80 uses it).
    recon_vm [N,B,ld]; `channels` (default ld) < ld: the decoder's padded output buffer is read in place.

    log_sigma, the decoder's Gaussian log sigma:
      * a float: that constant (the reference's softclip(1, -6) by default);
      * "optimal": the sigma-VAE optimal sigma, sc(0.5 log(SSE / (B N C))) with sc(t) = -6 + softplus(t + 6) and SSE the
        batch's squared error, computed on the device; the gradient flows through it;
      * a 1-element fp32 CUDA tensor s (a parameter): the learned sigma-VAE sigma sc(s); s receives its gradient.
    return_log_sigma=True appends the log sigma used, an fp64 0-dim device tensor."""
    c = int(recon_vm.shape[2] if channels is None else channels)
    if isinstance(log_sigma, str) and log_sigma != "optimal":
        raise _lib.MvbError(f"vae_loss: log_sigma is a float, 'optimal' or a parameter tensor, got {log_sigma!r}")
    if isinstance(log_sigma, (str, torch.Tensor)):
        out = _VaeLossSigmaFn.apply(recon_vm, x_gt, mu, logvar, y_hat, y, None if isinstance(log_sigma, str) else log_sigma, c)
        return (*out[:4], out[4][0]) if return_log_sigma else out[:4]
    out = _VaeLossFn.apply(recon_vm, x_gt, mu, logvar, y_hat, y, log_sigma, c)
    if not return_log_sigma:
        return out
    ls = float(torch.tensor(float(log_sigma), dtype=torch.float32))        # the kernel's log sigma is an fp32 argument
    return (*out, torch.full((), ls, device=recon_vm.device, dtype=torch.float64))


# ---------------------------------------------------------------------------------------------
# importance-weighted log-likelihood estimate (include/mvb.h: mvb_iw_*); forward only, no autograd
# ---------------------------------------------------------------------------------------------
def iw_sample(mu, logvar, eps, y_onehot):
    """mu, logvar [B,Z] fp32, eps [B,S,Z] fp32, y_onehot [B,C] -> (zcat [B*S, C+Z] fp32, row b*S + s = cat(y_b, z) with
    z = eps * exp(logvar/2) + mu; log_r [B*S] fp64 = log q(z | x, y) - log p(z))"""
    for t, name in ((mu, "mu"), (logvar, "logvar"), (eps, "eps")):
        _req_cuda(t, f"iw_sample {name}")
    _req_cuda(y_onehot, "iw_sample y", None)
    if mu.dim() != 2 or tuple(logvar.shape) != tuple(mu.shape):
        raise _lib.MvbError(f"iw_sample: mu {tuple(mu.shape)} and logvar {tuple(logvar.shape)} must be the same [B, Z]")
    b, z = mu.shape
    if eps.dim() != 3 or eps.shape[0] != b or eps.shape[2] != z or eps.shape[1] < 1:
        raise _lib.MvbError(f"iw_sample: eps is {tuple(eps.shape)}, expected ({b}, S, {z})")
    if y_onehot.dim() != 2 or y_onehot.shape[0] != b:
        raise _lib.MvbError(f"iw_sample: y is {tuple(y_onehot.shape)}, expected ({b}, C)")
    s, c = eps.shape[1], y_onehot.shape[1]
    mu, logvar, eps = mu.contiguous(), logvar.contiguous(), eps.contiguous()
    y = y_onehot.to(torch.int64).contiguous()
    zcat = torch.empty((b * s, c + z), device=mu.device, dtype=torch.float32)
    log_r = torch.empty(b * s, device=mu.device, dtype=torch.float64)
    check(lib.mvb_iw_sample(b, s, z, c, ptr(mu), ptr(logvar), ptr(eps), ptr(y), ptr(zcat), ptr(log_r), stream_ptr()),
          "mvb_iw_sample")
    return zcat, log_r


def iw_log_weights(recon_vm, x_gt, log_sigma, log_r, log_w, s0: int = 0, channels: Optional[int] = None):
    """Writes columns [s0, s0 + S) of log_w [B, S_total] (fp64, in place): log w = log p(x_b | z) - log_r with
    log p(x | z) = -SSE / (2 sigma^2) - N C (log sigma + log(2 pi)/2).  recon_vm [N, B*S, ld] vertex-major (column b*S + s;
    the first `channels` (default ld) floats of an entry are the reconstruction), x_gt [B,N,C] fp32 / fp64, log_sigma a
    0-dim (or 1-element) fp64 CUDA tensor, log_r [B*S] fp64 from iw_sample.  -> log_w"""
    _req_cuda(recon_vm, "iw_log_weights recon")
    _req_cuda(x_gt, "iw_log_weights x_gt", None)
    _req_cuda(log_sigma, "iw_log_weights log_sigma", torch.float64)
    _req_cuda(log_r, "iw_log_weights log_r", torch.float64)
    _req_cuda(log_w, "iw_log_weights log_w", torch.float64)
    if x_gt.dtype not in (torch.float32, torch.float64):
        raise _lib.MvbError(f"iw_log_weights: x_gt must be fp32 or fp64, got {x_gt.dtype}")
    if log_sigma.numel() != 1:
        raise _lib.MvbError(f"iw_log_weights: log_sigma has {log_sigma.numel()} elements, expected 1")
    n, bs, ld = recon_vm.shape
    c = int(ld if channels is None else channels)
    b = x_gt.shape[0]
    if x_gt.dim() != 3 or tuple(x_gt.shape[1:]) != (n, c) or c > ld or b < 1 or bs % b:
        raise _lib.MvbError(f"iw_log_weights: x_gt is {tuple(x_gt.shape)}, recon {tuple(recon_vm.shape)}: expected x_gt (B, {n}, {c}) "
                            f"with B dividing {bs}")
    s = bs // b
    if log_w.dim() != 2 or log_w.shape[0] != b or not log_w.is_contiguous() or s0 < 0 or s0 + s > log_w.shape[1]:
        raise _lib.MvbError(f"iw_log_weights: log_w {tuple(log_w.shape)} has no contiguous columns [{s0}, {s0 + s}) for {b} meshes")
    if tuple(log_r.shape) != (bs,):
        raise _lib.MvbError(f"iw_log_weights: log_r is {tuple(log_r.shape)}, expected ({bs},)")
    recon_vm, x_gt, log_r, ls = recon_vm.contiguous(), x_gt.contiguous(), log_r.contiguous(), log_sigma.contiguous()
    ws_bytes = lib.mvb_iw_log_weights_workspace_bytes(b, s, n)
    ws = torch.empty(ws_bytes, device=recon_vm.device, dtype=torch.uint8)
    check(lib.mvb_iw_log_weights(b, s, n, c, ptr(recon_vm), ld, ptr(x_gt), int(x_gt.dtype == torch.float64), ptr(ls), ptr(log_r),
                                 log_w.shape[1], int(s0), ptr(log_w), ptr(ws), ws_bytes, stream_ptr()), "mvb_iw_log_weights")
    return log_w


def iw_reduce(log_w, return_log_w: bool = False):
    """log_w [B,S] fp64 -> (log_px, elbo, ess), fp64 [B]: log mean_s exp(log w), mean_s log w and the effective sample size
    (sum_s w)^2 / sum_s w^2; return_log_w=True appends a copy of log_w"""
    _req_cuda(log_w, "iw_reduce log_w", torch.float64)
    if log_w.dim() != 2 or log_w.shape[0] < 1 or log_w.shape[1] < 1:
        raise _lib.MvbError(f"iw_reduce: log_w is {tuple(log_w.shape)}, expected (B, S)")
    b, s = log_w.shape
    log_w = log_w.contiguous()
    out = [torch.empty(b, device=log_w.device, dtype=torch.float64) for _ in range(3)]
    copy = torch.empty_like(log_w) if return_log_w else None
    check(lib.mvb_iw_reduce(b, s, ptr(log_w), ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(copy), stream_ptr()), "mvb_iw_reduce")
    return (*out, copy) if return_log_w else tuple(out)


class _KldFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu, logvar):
        _req_cuda(mu, "KLD mu")
        mu, logvar = mu.contiguous(), logvar.contiguous()
        b, z = mu.shape
        out = torch.empty(b, device=mu.device, dtype=torch.float32)
        check(lib.mvb_kld_fwd(b, z, ptr(mu), ptr(logvar), ptr(out), stream_ptr()), "mvb_kld_fwd")
        ctx.save_for_backward(mu, logvar)
        return out

    @staticmethod
    def backward(ctx, g):
        mu, logvar = ctx.saved_tensors
        b, z = mu.shape
        g = g.to(torch.float32).contiguous()
        dmu, dlv = torch.empty_like(mu), torch.empty_like(logvar)
        check(lib.mvb_kld_bwd(b, z, ptr(mu), ptr(logvar), ptr(g), ptr(dmu), ptr(dlv), stream_ptr()), "mvb_kld_bwd")
        return dmu, dlv


def kld(mu, logvar):
    return _KldFn.apply(mu, logvar)


class _GaussianNllFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu, x, log_sigma: float):
        _req_cuda(mu, "gaussian_nll mu")
        _req_cuda(x, "gaussian_nll x", None)
        if x.dtype not in (torch.float32, torch.float64) or x.shape != mu.shape:
            raise _lib.MvbError("gaussian_nll: x must be fp32/fp64 with the shape of mu")
        mu_c, x_c = mu.contiguous(), x.contiguous()
        out = torch.empty_like(x_c)
        f64 = x.dtype == torch.float64
        check(lib.mvb_gaussian_nll_fwd(mu_c.numel(), ptr(mu_c), ptr(x_c), 1 if f64 else 0, float(log_sigma), ptr(out),
                                       stream_ptr()), "mvb_gaussian_nll_fwd")
        ctx.save_for_backward(mu_c, x_c)
        ctx.log_sigma, ctx.f64 = float(log_sigma), f64
        return out

    @staticmethod
    def backward(ctx, g):
        mu_c, x_c = ctx.saved_tensors
        g = g.to(x_c.dtype).contiguous()
        d_mu = torch.empty_like(mu_c)
        check(lib.mvb_gaussian_nll_bwd(mu_c.numel(), ptr(mu_c), ptr(x_c), 1 if ctx.f64 else 0, ctx.log_sigma, ptr(g),
                                       ptr(d_mu), stream_ptr()), "mvb_gaussian_nll_bwd")
        return d_mu, None, None


class _GaussianNllSigmaFn(torch.autograd.Function):
    """mvb_gaussian_nll_sigma_fwd / _bwd: log_sigma a 0-dim fp32 / fp64 CUDA tensor, differentiable"""

    @staticmethod
    def forward(ctx, mu, x, log_sigma):
        _req_cuda(mu, "gaussian_nll mu")
        _req_cuda(x, "gaussian_nll x", None)
        _req_cuda(log_sigma, "gaussian_nll log_sigma", None)
        if x.dtype not in (torch.float32, torch.float64) or x.shape != mu.shape:
            raise _lib.MvbError("gaussian_nll: x must be fp32/fp64 with the shape of mu")
        if log_sigma.dtype not in (torch.float32, torch.float64):
            raise _lib.MvbError(f"gaussian_nll: log_sigma must be fp32 or fp64, got {log_sigma.dtype}")
        mu_c, x_c, ls = mu.contiguous(), x.contiguous(), log_sigma.contiguous()
        out = torch.empty_like(x_c)
        f64, ls64 = x.dtype == torch.float64, ls.dtype == torch.float64
        check(lib.mvb_gaussian_nll_sigma_fwd(mu_c.numel(), ptr(mu_c), ptr(x_c), int(f64), ptr(ls), int(ls64), ptr(out),
                                             stream_ptr()), "mvb_gaussian_nll_sigma_fwd")
        ctx.save_for_backward(mu_c, x_c, ls)
        return out

    @staticmethod
    def backward(ctx, g):
        mu_c, x_c, ls = ctx.saved_tensors
        n = mu_c.numel()
        g = g.to(x_c.dtype).contiguous()
        d_mu = torch.empty_like(mu_c)
        d_ls = torch.empty((), device=mu_c.device, dtype=torch.float64)
        ws_bytes = lib.mvb_gaussian_nll_sigma_workspace_bytes(n)
        ws = torch.empty(max(ws_bytes, 8), device=mu_c.device, dtype=torch.uint8)
        if n == 0:
            d_ls.zero_()
        else:
            check(lib.mvb_gaussian_nll_sigma_bwd(n, ptr(mu_c), ptr(x_c), int(x_c.dtype == torch.float64), ptr(ls),
                                                 int(ls.dtype == torch.float64), ptr(g), ptr(d_mu), ptr(d_ls), ptr(ws), ws_bytes,
                                                 stream_ptr()), "mvb_gaussian_nll_sigma_bwd")
        return d_mu, None, d_ls.to(ls.dtype)


def gaussian_nll(mu, x, log_sigma):
    """log_sigma a float (a host constant) or a 1-element CUDA tensor (read on the device, differentiable)"""
    if isinstance(log_sigma, torch.Tensor):
        if log_sigma.numel() != 1:
            raise _lib.MvbError(f"gaussian_nll: log_sigma has {log_sigma.numel()} elements, expected 1")
        return _GaussianNllSigmaFn.apply(mu, x, log_sigma.reshape(()))
    return _GaussianNllFn.apply(mu, x, log_sigma)


# ---------------------------------------------------------------------------------------------
# dense bottleneck (SURVEY.md 8(f) row f2): fused Linear(+ReLU+dropout) and the three VAE heads
# ---------------------------------------------------------------------------------------------
class DropoutStream:
    """Counter-based dropout stream shared by the fused dense kernels: a mask is a pure function of
    (seed + site, offset, element), offset = host counter + *device counter.  The backward pass
    regenerates the mask from the same triple; a captured CUDA graph gets fresh masks on every replay
    through the device counter (the engine points it at Adam's device step counter)."""

    def __init__(self, seed: int = 0x5EED):
        self.seed = int(seed)
        self.offset_host = 0
        self.offset_dev: Optional[torch.Tensor] = None     # int64 scalar on the device, or None

    def advance(self):
        # with a device counter attached (the engine points it at Adam's step counter, which every step - replayed or
        # eager - increments) the host offset must stay frozen: advancing both would hand two different steps the same
        # sum, i.e. the same masks at every site
        if self.offset_dev is None:
            self.offset_host += 1

    def site(self, site_id: int):
        return ((self.seed + 0x9E3779B97F4A7C15 * (site_id + 1)) & 0xFFFFFFFFFFFFFFFF, self.offset_dev, self.offset_host)


_NO_RNG = (0, None, 0)
VAE_HEADS_MAX_BATCH = 256      # the largest batch of the one-launch heads kernels at the default shapes (larger: tiled kernels)


class _LinearFn(torch.autograd.Function):
    """mvb_linear_fwd / mvb_linear_bwd: y = dropout(relu(x W^T + b)) (torch.nn.Linear + F.relu +
    nn.Dropout, models/cheb_VAE.py:270-272, 276-281).  x is [M,K] row-major, or - x_vm - a
    vertex-major activation [V,M,F] standing for x.reshape(M, V*F); likewise the output."""

    @staticmethod
    def forward(ctx, x, weight, bias, relu: bool, p: float, rng, x_vm: bool, y_vm_f: int):
        _req_cuda(x, "linear x")
        _req_cuda(weight, "linear weight")
        x = x.contiguous()
        w = weight.contiguous()
        n, k = w.shape
        if x_vm:
            v, m, f = x.shape
            if v * f != k:
                raise _lib.MvbError(f"linear: vertex-major input {tuple(x.shape)} does not flatten to {k} features")
            x_vm_f = f
        else:
            m = x.shape[0]
            if x.dim() != 2 or x.shape[1] != k:
                raise _lib.MvbError(f"linear: input {tuple(x.shape)} does not match weight {tuple(w.shape)}")
            x_vm_f = 0
        if y_vm_f:
            if n % y_vm_f:
                raise _lib.MvbError(f"linear: {n} outputs do not split into vertices of {y_vm_f} features")
            y = torch.empty((n // y_vm_f, m, y_vm_f), device=x.device, dtype=torch.float32)
        else:
            y = torch.empty((m, n), device=x.device, dtype=torch.float32)
        bb = None if bias is None else bias.contiguous()
        seed, off_dev, off_host = rng if p > 0 else _NO_RNG
        check(lib.mvb_linear_fwd(m, k, n, ptr(x), x_vm_f, ptr(w), ptr(bb), 1 if relu else 0, float(p), seed, ptr(off_dev),
                                 off_host, ptr(y), y_vm_f, stream_ptr()), "mvb_linear_fwd")
        ctx.dims = (m, k, n, x_vm_f, y_vm_f, relu, float(p))
        ctx.has_bias = bias is not None
        ctx.sinks = (_sink(weight), _sink(bias))
        ctx.save_for_backward(x, w, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w, y = ctx.saved_tensors
        m, k, n, x_vm_f, y_vm_f, relu, p = ctx.dims
        gy = gy.contiguous()
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dw, db = _grad_outs(ctx.sinks, w, n if ctx.has_bias else None)
        check(lib.mvb_linear_bwd(m, k, n, ptr(x), x_vm_f, ptr(w), ptr(y), ptr(gy), y_vm_f, 1 if relu else 0, p, ptr(dx), ptr(dw),
                                 ptr(db), stream_ptr()), "mvb_linear_bwd")
        if dx is not None:          # without dx there is no split launch and nothing on the side chain
            _park_or_join(ctx, (x, w, y, gy, dw, db))
        return dx, *_ret(ctx.sinks, dw, db), None, None, None, None, None


def linear(x, weight, bias=None, relu: bool = False, p: float = 0.0, rng=_NO_RNG, x_vm: bool = False, y_vm_f: int = 0):
    """Fused dense layer.  `p > 0` needs `relu=True` (the backward recovers the dropout mask from y == 0)."""
    if p > 0 and not relu:
        raise _lib.MvbError("linear: dropout without ReLU is not supported by the fused kernel")
    return _LinearFn.apply(x, weight, bias, relu, float(p), rng, x_vm, int(y_vm_f))


class _VaeHeadsFn(torch.autograd.Function):
    """mvb_vae_heads_fwd / _bwd: classifier + softmax, z_mean, z_log_var on cat(y, h), the
    reparameterisation and cat(y, z) (models/cheb_VAE.py:206-223, 253-258, 309-319)."""

    @staticmethod
    def forward(ctx, h, y_onehot, eps, wc, bc, wm, bm, wv, bv, p: float, rng):
        _req_cuda(h, "vae_heads h")
        h = h.contiguous()
        b, hd = h.shape
        c, z = wc.shape[0], wm.shape[0]
        if wc.shape[1] != hd or wm.shape[1] != c + hd or tuple(wv.shape) != tuple(wm.shape):
            raise _lib.MvbError("vae_heads: weight shapes do not match h / the one-hot width")
        y_onehot = y_onehot.to(torch.int64).contiguous()
        if tuple(y_onehot.shape) != (b, c):
            raise _lib.MvbError(f"vae_heads: y is {tuple(y_onehot.shape)}, expected {(b, c)}")
        eps_c = None if eps is None else eps.contiguous()
        ctx_params = (wc, bc, wm, bm, wv, bv)
        wc, bc, wm, bm, wv, bv = (t.contiguous() for t in (wc, bc, wm, bm, wv, bv))
        dev = h.device
        y_hat = torch.empty((b, c), device=dev, dtype=torch.float32)
        mu = torch.empty((b, z), device=dev, dtype=torch.float32)
        logvar = torch.empty_like(mu)
        zz = torch.empty_like(mu)
        zcat = torch.empty((b, c + z), device=dev, dtype=torch.float32)
        seed, off_dev, off_host = rng if p > 0 else _NO_RNG
        check(lib.mvb_vae_heads_fwd(b, hd, z, c, ptr(h), ptr(y_onehot), ptr(eps_c), ptr(wc), ptr(bc), ptr(wm), ptr(bm), ptr(wv),
                                    ptr(bv), float(p), seed, ptr(off_dev), off_host, ptr(y_hat), ptr(mu), ptr(logvar), ptr(zz),
                                    ptr(zcat), stream_ptr()), "mvb_vae_heads_fwd")
        ctx.save_for_backward(h, y_onehot, eps_c, wc, wm, wv, y_hat, logvar)
        ctx.cfg = (b, hd, z, c, float(p), seed, off_dev, off_host)
        ctx.sinks = tuple(_sink(t) for t in (ctx_params[0], ctx_params[1], ctx_params[2], ctx_params[3], ctx_params[4], ctx_params[5]))
        return y_hat, mu, logvar, zz, zcat

    @staticmethod
    def backward(ctx, g_yhat, g_mu, g_logvar, g_z, g_zcat):
        h, y_onehot, eps, wc, wm, wv, y_hat, logvar = ctx.saved_tensors
        b, hd, z, c, p, seed, off_dev, off_host = ctx.cfg
        gs = [None if g is None else g.contiguous() for g in (g_yhat, g_mu, g_logvar, g_z, g_zcat)]
        g_h = torch.empty_like(h)
        sk = ctx.sinks
        dwc, dbc = _grad_outs(sk[0:2], wc, c)
        dwm, dbm = _grad_outs(sk[2:4], wm, z)
        dwv, dbv = _grad_outs(sk[4:6], wv, z)
        check(lib.mvb_vae_heads_bwd(b, hd, z, c, ptr(h), ptr(y_onehot), ptr(eps), ptr(wc), ptr(wm), ptr(wv), ptr(y_hat),
                                    ptr(logvar), p, seed, ptr(off_dev), off_host, ptr(gs[0]), ptr(gs[1]), ptr(gs[2]), ptr(gs[3]),
                                    ptr(gs[4]), ptr(g_h), ptr(dwc), ptr(dbc), ptr(dwm), ptr(dbm), ptr(dwv), ptr(dbv),
                                    stream_ptr()), "mvb_vae_heads_bwd")
        return (g_h, None, None, *_ret(sk[0:2], dwc, dbc), *_ret(sk[2:4], dwm, dbm), *_ret(sk[4:6], dwv, dbv), None, None)


def vae_heads(h, y_onehot, eps, classifier, z_mean, z_log_var, p: float = 0.0, rng=_NO_RNG):
    """-> (y_hat, mu, logvar, z, cat(y, z)); `classifier`, `z_mean`, `z_log_var` are the model's
    nn.Linear modules (their Parameters receive the gradients); eps=None means z = mu (test mode).
    One call covers any batch, hidden width and latent size (at most 32 classes): the library picks the one-launch
    kernels where they fit and the tiled ones elsewhere, with the same results and the same dropout mask."""
    args = (classifier.weight, classifier.bias, z_mean.weight, z_mean.bias, z_log_var.weight, z_log_var.bias)
    return _VaeHeadsFn.apply(h, y_onehot, eps, *args, float(p), rng)


# ---------------------------------------------------------------------------------------------
# mesh-resident fused layers for the coarse levels (models/cheb_VAE.py:264-265, 284-285)
# ---------------------------------------------------------------------------------------------
def _fused_layer_kind(n: int, b: int, fin: int, fout: int, k: int, l_op: MeshOperator, u_op: Optional[MeshOperator],
                      d_op: Optional[MeshOperator]) -> Optional[str]:
    """"mesh" (the mesh-resident kernels), "stream" (the row-streaming kernels) or None (neither covers the layer)"""
    if l_op.n_active != n or l_op.n_rows != n:
        return None
    if d_op is not None and not d_op.is_selection:
        return None
    n_in = u_op.n_cols if u_op is not None else n
    n_out = d_op.n_rows if d_op is not None else n
    if lib.mvb_cheb_layer_supported(n, b, fin, fout, k, l_op.nnz, n_in, u_op.nnz if u_op is not None else 0, n_out):
        return "mesh"
    return "stream" if cheb_stream_supported(n, b, fin, fout, k, l_op, u_op, d_op) else None


def cheb_layer_supported(n: int, b: int, fin: int, fout: int, k: int, l_op: MeshOperator, u_op: Optional[MeshOperator],
                         d_op: Optional[MeshOperator]) -> bool:
    return _fused_layer_kind(n, b, fin, fout, k, l_op, u_op, d_op) is not None


def cheb_stream_supported(n: int, b: int, fin: int, fout: int, k: int, l_op: MeshOperator, u_op: Optional[MeshOperator],
                          d_op: Optional[MeshOperator]) -> bool:
    """the row-streaming fused layer (mvb_cheb_stream_*): levels too large for shared memory, no row selection"""
    if d_op is not None or l_op.n_active != n or l_op.n_rows != n:
        return False
    n_in = u_op.n_cols if u_op is not None else n
    return bool(lib.mvb_cheb_stream_supported(n, b, fin, fout, k, n_in, 1 if u_op is not None else 0, n))


class _ChebLayerFn(torch.autograd.Function):
    """mvb_cheb_layer_fwd / _bwd: [pool(U)] -> ChebConv -> ReLU -> [pool(D)] for one coarse level, one
    launch per direction.  Saves only its input and output (the basis is recomputed in shared memory)."""

    @staticmethod
    def forward(ctx, x_vm, weight, bias, l_op: MeshOperator, u_op, d_op, relu: bool):
        _req_cuda(x_vm, "cheb_layer x")
        _req_cuda(weight, "cheb_layer weight")
        x_vm = x_vm.contiguous()
        w = weight.contiguous()
        n_in, b, fin = x_vm.shape
        k, fin_w, fout = w.shape
        n = l_op.n_rows
        if fin_w != fin:
            raise _lib.MvbError(f"cheb_layer: x has {fin} features, weight expects {fin_w}")
        if (u_op.n_cols if u_op is not None else n) != n_in:
            raise _lib.MvbError(f"cheb_layer: x has {n_in} vertices, the layer expects {u_op.n_cols if u_op is not None else n}")
        n_out = d_op.n_rows if d_op is not None else n
        bb = None if bias is None else bias.contiguous()
        y = torch.empty((n_out, b, fout), device=x_vm.device, dtype=torch.float32)
        u = u_op
        check(lib.mvb_cheb_layer_fwd(n, b, fin, fout, k, ptr(l_op.rowptr), ptr(l_op.colidx), ptr(l_op.vals), l_op.nnz, n_in,
                                     ptr(u.rowptr) if u else None, ptr(u.colidx) if u else None, ptr(u.vals) if u else None,
                                     u.nnz if u else 0, n_out, ptr(d_op.colidx) if d_op is not None else None, ptr(x_vm), ptr(w),
                                     ptr(bb), 1 if relu else 0, ptr(y), stream_ptr()), "mvb_cheb_layer_fwd")
        ctx.ops = (l_op, u_op, d_op)
        ctx.relu, ctx.has_bias = relu, bias is not None
        ctx.sinks = (_sink(weight), _sink(bias))
        ctx.save_for_backward(x_vm, w, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_vm, w, y = ctx.saved_tensors
        l_op, u, d_op = ctx.ops
        n_in, b, fin = x_vm.shape
        k, _, fout = w.shape
        n = l_op.n_rows
        n_out = d_op.n_rows if d_op is not None else n
        dy = dy.contiguous()
        dx = torch.empty_like(x_vm) if ctx.needs_input_grad[0] else None
        dw, db = _grad_outs(ctx.sinks, w, fout if ctx.has_bias else None)
        ws_bytes = lib.mvb_cheb_layer_bwd_workspace_bytes(n, b, fin, fout, k, 1 if u is not None else 0)
        ws = torch.empty(ws_bytes, device=w.device, dtype=torch.uint8)
        check(lib.mvb_cheb_layer_bwd(n, b, fin, fout, k, ptr(l_op.rowptr), ptr(l_op.colidx), ptr(l_op.vals), ptr(l_op.rowptr_t),
                                     ptr(l_op.colidx_t), ptr(l_op.vals_t), l_op.nnz, n_in,
                                     ptr(u.rowptr) if u else None, ptr(u.colidx) if u else None, ptr(u.vals) if u else None,
                                     ptr(u.rowptr_t) if u else None, ptr(u.colidx_t) if u else None, ptr(u.vals_t) if u else None,
                                     u.nnz if u else 0, n_out, ptr(d_op.colidx) if d_op is not None else None, ptr(x_vm), ptr(w),
                                     ptr(y) if ctx.relu else None, ptr(dy), ptr(dx), ptr(dw), ptr(db), ptr(ws), ws_bytes,
                                     stream_ptr()), "mvb_cheb_layer_bwd")
        _park_or_join(ctx, (ws, x_vm, w, dy, dw, db))
        return dx, *_ret(ctx.sinks, dw, db), None, None, None, None


class _ChebStreamFn(torch.autograd.Function):
    """mvb_cheb_stream_fwd / _bwd: [pool(U)] -> ChebConv -> ReLU at a level too large for shared memory (level 0), one
    persistent launch per direction; saves only its input and output."""

    @staticmethod
    def forward(ctx, x_vm, weight, bias, l_op: MeshOperator, u_op, relu: bool):
        _req_cuda(x_vm, "cheb_layer x")
        _req_cuda(weight, "cheb_layer weight")
        x_vm = x_vm.contiguous()
        w = weight.contiguous()
        n_in, b, fin = x_vm.shape
        k, fin_w, fout = w.shape
        n = l_op.n_rows
        if fin_w != fin:
            raise _lib.MvbError(f"cheb_layer: x has {fin} features, weight expects {fin_w}")
        if (u_op.n_cols if u_op is not None else n) != n_in:
            raise _lib.MvbError(f"cheb_layer: x has {n_in} vertices, the layer expects {u_op.n_cols if u_op is not None else n}")
        bb = None if bias is None else bias.contiguous()
        y = torch.empty((n, b, fout), device=x_vm.device, dtype=torch.float32)
        u = u_op
        ws_bytes = lib.mvb_cheb_stream_fwd_workspace_bytes(n, b, fin, fout, k, 1 if u is not None else 0)
        ws = torch.empty(ws_bytes, device=w.device, dtype=torch.uint8)
        check(lib.mvb_cheb_stream_fwd(n, b, fin, fout, k, ptr(l_op.rowptr), ptr(l_op.colidx), ptr(l_op.vals), l_op.nnz, n_in,
                                      ptr(u.rowptr) if u else None, ptr(u.colidx) if u else None, ptr(u.vals) if u else None,
                                      u.nnz if u else 0, ptr(x_vm), ptr(w), ptr(bb), 1 if relu else 0, ptr(y), ptr(ws), ws_bytes,
                                      stream_ptr()), "mvb_cheb_stream_fwd")
        ctx.ops = (l_op, u_op)
        ctx.relu, ctx.has_bias = relu, bias is not None
        ctx.sinks = (_sink(weight), _sink(bias))
        ctx.save_for_backward(x_vm, w, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_vm, w, y = ctx.saved_tensors
        l_op, u = ctx.ops
        n_in, b, fin = x_vm.shape
        k, _, fout = w.shape
        n = l_op.n_rows
        dy = dy.contiguous()
        dx = torch.empty_like(x_vm) if ctx.needs_input_grad[0] else None
        dw, db = _grad_outs(ctx.sinks, w, fout if ctx.has_bias else None)
        ws_bytes = lib.mvb_cheb_stream_bwd_workspace_bytes(n, b, fin, fout, k, 1 if u is not None else 0)
        ws = torch.empty(ws_bytes, device=w.device, dtype=torch.uint8)
        check(lib.mvb_cheb_stream_bwd(n, b, fin, fout, k, ptr(l_op.rowptr_t), ptr(l_op.colidx_t), ptr(l_op.vals_t), l_op.nnz, n_in,
                                      ptr(u.rowptr) if u else None, ptr(u.colidx) if u else None, ptr(u.vals) if u else None,
                                      ptr(u.rowptr_t) if u else None, ptr(u.colidx_t) if u else None, ptr(u.vals_t) if u else None,
                                      u.nnz if u else 0, ptr(x_vm), ptr(w), ptr(y) if ctx.relu else None, ptr(dy), ptr(dx), ptr(dw),
                                      ptr(db), ptr(ws), ws_bytes, stream_ptr()), "mvb_cheb_stream_bwd")
        _park_or_join(ctx, (ws, x_vm, w, dy, dw, db))
        return dx, *_ret(ctx.sinks, dw, db), None, None, None


def cheb_layer_fused(x_vm, weight, bias, l_op: MeshOperator, u_op: Optional[MeshOperator] = None,
                     d_op: Optional[MeshOperator] = None, relu: bool = True) -> Optional[torch.Tensor]:
    """cheb_layer as one fused kernel per direction - the mesh-resident kernels when the level fits shared memory, else
    the row-streaming kernels - or None when neither covers the layer"""
    if not x_vm.is_cuda:
        return None
    kind = _fused_layer_kind(l_op.n_rows, x_vm.shape[1], x_vm.shape[2], weight.shape[2], weight.shape[0], l_op, u_op, d_op)
    if kind == "mesh":
        return _ChebLayerFn.apply(x_vm, weight, bias, l_op, u_op, d_op, relu)
    if kind == "stream":
        return _ChebStreamFn.apply(x_vm, weight, bias, l_op, u_op, relu)
    return None


def cheb_layer(x_vm, weight, bias, l_op: MeshOperator, u_op: Optional[MeshOperator] = None,
               d_op: Optional[MeshOperator] = None, relu: bool = True):
    """[U prologue] -> Chebyshev conv (+bias, ReLU) -> [D row selection] on vertex-major tensors: the fused
    kernels when they cover the level (cheb_layer_fused), else the composition of pool / cheb_conv / pool."""
    y = cheb_layer_fused(x_vm, weight, bias, l_op, u_op, d_op, relu)
    if y is not None:
        return y
    if u_op is not None:
        x_vm = pool(x_vm, u_op)
    y = cheb_conv(x_vm, weight, bias, l_op, relu)
    if d_op is not None:
        y = pool(y, d_op)
    return y


def recon_error(recon, mean, std, s, R, m, gt_mesh, per_vertex: bool = False, mesh: bool = False):
    """Per-mesh reconstruction error of the train / evaluate / inference loops (main.py:88-93, :139-146;
    inference.py:100-127) on the device: recon [B,N,3] (any strides - the model's output is a view of the
    vertex-major decoder buffer and is read in place), mean/std [N,3] (norm.npz), s [B] / R [B,3,3] /
    m [B,1,3] or [B,3] (Procrustes), gt_mesh [B,N,3] (None with mesh=True: only the back-transform).
    -> (mean_err [B], max_err [B]) fp64 device tensors; `mean_err.mean()` is main.py:93's `diff`.
    per_vertex=True appends diff [B,N] fp32 (main.py:146), mesh=True the back-transformed mesh [B,N,3] fp32."""
    _req_cuda(recon, "recon_error recon")
    b, n, c = recon.shape
    if c != 3:
        raise _lib.MvbError("recon_error: meshes have 3 coordinates")
    if gt_mesh is None and not mesh:
        raise _lib.MvbError("recon_error: no ground truth and no mesh output requested")
    rv = recon.permute(1, 0, 2)                      # [N,B,3] view
    if rv.stride(2) == 1 and rv.stride(0) == b * rv.stride(1) and rv.stride(1) >= 3:
        ld = rv.stride(1)                            # in place: entries of ld floats (3, or 4 for the padded decoder output)
    else:
        rv, ld = rv.contiguous(), 3
    dev = recon.device
    # small operands: one asynchronous copy each (pinned host tensors make them truly asynchronous); the ground-truth
    # meshes are read in the precision they arrive in (fp32 from the loader, data.py:133) - no conversion pass
    f32 = lambda t: torch.as_tensor(t).to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()      # noqa: E731
    f64 = lambda t: torch.as_tensor(t).to(device=dev, non_blocking=True).to(torch.float64).contiguous()        # noqa: E731
    mean, std = f32(mean).reshape(n, 3), f32(std).reshape(n, 3)
    s, R, m = f64(s).reshape(b), f64(R).reshape(b, 3, 3), f64(m).reshape(b, 3)
    gt = None
    if gt_mesh is not None:
        gt = torch.as_tensor(gt_mesh)
        if gt.dtype not in (torch.float32, torch.float64):
            gt = gt.to(torch.float32)
        gt = gt.to(dev, non_blocking=True).reshape(b, n, 3).contiguous()
    mean_err = torch.empty(b, device=dev, dtype=torch.float64)
    max_err = torch.empty(b, device=dev, dtype=torch.float64)
    verr = torch.empty((b, n), device=dev, dtype=torch.float32) if (per_vertex and gt is not None) else None
    mesh_out = torch.empty((b, n, 3), device=dev, dtype=torch.float32) if mesh else None
    ws_bytes = lib.mvb_recon_error_workspace_bytes(b, n)
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    check(lib.mvb_recon_error(b, n, ld, ptr(rv), ptr(mean), ptr(std), ptr(s), ptr(R), ptr(m), ptr(gt),
                              int(gt is not None and gt.dtype == torch.float64), ptr(mean_err), ptr(max_err), ptr(verr), ptr(mesh_out), ptr(ws), ws_bytes, stream_ptr()), "mvb_recon_error")
    out = (mean_err, max_err)
    if per_vertex:
        out += (verr,)
    if mesh:
        out += (mesh_out,)
    return out


class EpochMeter:
    """Running totals of one epoch of main.py's train() / evaluate() (main.py:60-65, 83-86, 93, 96) on the device:
    `add` is one launch and no synchronisation; `read` is the single device->host transfer of the epoch."""

    def __init__(self, device):
        self.acc = torch.zeros(8, device=device, dtype=torch.float64)

    def reset(self):
        self.acc.zero_()

    def add(self, loss, kld, rec, correct=None, mean_err=None):
        b = kld.shape[0]
        if loss.dtype not in (torch.float32, torch.float64) or rec.dtype not in (torch.float32, torch.float64):
            raise _lib.MvbError("EpochMeter.add: loss / rec must be fp32 or fp64")
        kld = kld.detach().float().contiguous()
        rec, loss = rec.detach().contiguous(), loss.detach().contiguous()
        if correct is not None:
            correct = correct.detach().to(torch.int64).contiguous()
        if mean_err is not None:
            mean_err = mean_err.detach().to(torch.float64).contiguous()
        check(lib.mvb_epoch_meter_add(b, ptr(loss), int(loss.dtype == torch.float64), ptr(kld), ptr(rec),
                                      int(rec.dtype == torch.float64), ptr(correct), ptr(mean_err), ptr(self.acc),
                                      stream_ptr()), "mvb_epoch_meter_add")

    def read(self):
        """-> dict(loss, kld, rec_loss, error, accuracy, count): the per-sample means main.py returns"""
        a = self.acc.cpu().numpy()
        n = max(a[5], 1.0)
        return {"loss": a[0] / n, "kld": a[1] / n, "rec_loss": a[2] / n, "error": a[3] / n, "accuracy": a[4] / n,
                "count": int(a[5])}
