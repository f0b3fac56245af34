/*
 * mvb.h  --  C ABI of libmvb_sm100a.so, the B200-native (sm_100a) kernels for the Mesh-VAE hot path.
 *
 * The reference (ZOUKaifeng/Mesh-VAE) is pure Python and has NO FFI layer: its boundary for this
 * path is the Python module namespace (SURVEY.md 8(b)).  Every entry point below therefore names
 * the reference Python symbol (file:line under the reference tree) whose arithmetic it replaces;
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every `float*` / `int*` / `double*` / `void*` data pointer is a DEVICE pointer owned by the
 *     caller (mvb_csr_from_coo_host is the one exception: HOST pointers, runs on the CPU);
 *   - kernels are enqueue-only on `stream` (a cudaStream_t passed as void*): no allocation, no
 *     synchronisation, CUDA-graph capturable; scratch memory is an explicit `workspace` whose
 *     size the matching *_workspace_bytes() query returns;
 *   - activations are VERTEX-MAJOR: a logical [B, N, F] reference tensor is stored as
 *     [N, B, F] contiguous (row = (vertex, mesh), B*F contiguous floats per vertex);
 *   - sparse operators are CSR with int32 indices and fp32 values, entries of a row kept in the
 *     COO order the reference hands over (deterministic summation order);
 *   - return value: MVB_OK (0) or a negative MVB_E* code; mvb_last_error() gives the text
 *     (thread-local).  There is no CPU fallback: without a CUDA device every compute entry
 *     point fails with MVB_ECUDA.
 */
#ifndef MVB_H_
#define MVB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVB_OK 0
#define MVB_EINVAL (-1) /* bad size / null pointer / unsupported combination */
#define MVB_ECUDA (-2)  /* CUDA runtime error (launch failure, no device)   */
#define MVB_EALIGN (-3) /* pointer not aligned as documented                */
#define MVB_EWORKSPACE (-4) /* workspace too small                          */

#define MVB_VERSION 100

/* ---- library info ------------------------------------------------------------------------ */
int mvb_version(void);             /* MVB_VERSION */
int mvb_sm_arch(void);             /* 100: the only architecture compiled in (sm_100a) */
const char *mvb_last_error(void);  /* text of the last error on this thread ("" if none) */
/* compute capability (major*10+minor) of the current device, or MVB_ECUDA when there is none */
int mvb_device_cc(void);
/* number of CUDA kernels this library has launched (or captured) in this process so far; bench.py
 * reports the per-step delta as "gpu_launches" */
int64_t mvb_launch_count(void);
/* enable (default) / disable the tcgen05 3xTF32 tensor-core kernels for the dense contractions;
 * disabled, the strict-fp32 FFMA kernels run everywhere.  Returns the previous setting. */
int mvb_set_tensor_cores(int enable);
/* Run-time switches for tests and the step engine - not part of the operator API.  spec is a list
 * "key=a[,b];key=..." (keys: mesh_tc, fused_recurrence, stream_tc, pdl, defer_wgrad; documented next to mvb_tune in
 * csrc/mvb_api.cu); any other key is rejected with MVB_EINVAL.  mesh_tc / fused_recurrence / stream_tc select between
 * implementations tested against each other; pdl and defer_wgrad change only how kernels are launched and joined.  The
 * mvb Python package applies the environment variable MVB_TUNE through this call when it is imported. */
int mvb_tune(const char *spec);
/* Deferred side chains: with mvb_tune("defer_wgrad=1") the weight-gradient work of these calls runs on an internal
 * per-device side stream and is NOT joined into the caller's stream before the call returns - it then overlaps the
 * following layers' backward kernels:
 *   lane 0: mvb_cheb_bwd in the adjoint form (mvb_cheb_bwd_uses_basis == 0), mvb_cheb_layer_bwd when its tensor-core
 *           kernel runs, mvb_cheb_stream_bwd;
 *   lane 1: mvb_linear_bwd with dx (its dW / db tiles run as a launch of their own).
 * No other call defers.  The pending chain of each call reads or writes:
 *   mvb_cheb_bwd (adjoint form): workspace, x, dweight, and dy when y_for_relu is NULL (without ReLU the chain reduces
 *           dy itself; with it, the masked copy in the workspace) - dbias is reduced on `stream` before the call returns;
 *   mvb_cheb_layer_bwd, mvb_cheb_stream_bwd: workspace, dweight, dbias, and x when there is no U prologue (with one,
 *           the up-sampled T_0 in the workspace);
 *   mvb_linear_bwd: x, y, gy, dW, db.
 * The caller must (1) keep those buffers alive and untouched until it has called mvb_side_join(stream), which makes
 * `stream` wait for the pending chain (the Python package parks them, with the call's other buffers, in
 * _lib._deferred["keep"]), and (2) call it before reading any gradient and before a stream capture ends.  Default off:
 * every call joins before it returns.  Deferred or not, with PDL or without, captured or not, the results are the same
 * bits (tests/test_gpu_step_modes.py). */
int mvb_side_join(void *stream);
/* the same for one lane of chains: 0 = convolution weight gradients, 1 = dense-layer weight gradients (mvb_linear_bwd) */
int mvb_side_join_lane(void *stream, int lane);

/* step-engine plumbing: cudaStreamWaitEvent(stream, event, cudaEventWaitExternal).  Legal during stream
 * capture (becomes an external event-wait node): each replay of the captured graph waits for the latest
 * host-side record of `event` - how the one-graph training step waits for the ground-truth H2D copy that
 * main.py:70 issues per batch while the forward pass is already running. */
int mvb_stream_wait_external_event(void *stream, void *event);

/* ---- operator hand-off: COO -> CSR (HOST function) ---------------------------------------
 * Replaces the implicit operator format of the reference: model.py:24-32 `scipy_to_torch_sparse`
 * (uncoalesced COO, int64 / f32), consumed via `_indices()/_values()` at nn/pool.py:19 and
 * models/cheb_VAE.py:118, and the (edge_index, norm) pair of nn/conv.py:541-555.
 * Builds CSR of P (transpose == 0: out rows = P rows) or of P^T (transpose != 0: out rows =
 * P columns) by a STABLE counting sort, so entries of one output row keep their COO order;
 * duplicates are kept (they sum).  n_out_rows may exceed the largest index (empty rows):
 * this is how the 20-node operator acts on a 4998-vertex tensor (models/cheb_VAE.py:288).
 * rowptr has n_out_rows+1 entries; colidx / vals have nnz entries.  HOST pointers. */
int mvb_csr_from_coo_host(int64_t n_out_rows, int64_t n_out_cols, int64_t nnz,
                          const int64_t *coo_row, const int64_t *coo_col, const float *coo_val,
                          int transpose, int32_t *rowptr, int32_t *colidx, float *vals);

/* ---- A1: sparse propagate  (nn/conv.py:242-331 MessagePassing.propagate = index_select
 *          :199-200, message :579-581, scatter-add :363-364) -------------------------------
 * y[r, :] = alpha * sum_{j in row r} vals[j] * x[colidx[j], :]  +  beta * z[r, :]  +  w[r, :]
 * x: [n_src_rows, ncols] (every colidx < n_src_rows), y/z/w: [n_rows, ncols]; z and w may be NULL; y may alias z or w
 * (each row only reads its own z/w row) but must not alias x.  The 16-byte vector path is used
 * when ncols % 4 == 0 and all pointers are 16-byte aligned, else a scalar path. */
int mvb_spmm(int n_rows, int n_src_rows, const int32_t *rowptr, const int32_t *colidx, const float *vals,
             const float *x, float *y, const float *z, const float *w, float alpha, float beta,
             int64_t ncols, void *stream);

/* ---- A5/A6: mesh pooling  (nn/pool.py:13-23 SurfacePool.forward; models/cheb_cls.py:22-27 Pool)
 * forward : y[M, B*F] = P x[N, B*F]      with CSR(P)   (n_out_rows = M)
 * backward: dx[N, B*F] = P^T dy[M, B*F]  with CSR(P^T) (n_out_rows = N)  - no atomics. */
int mvb_pool_fwd(int n_out_rows, int n_in_rows, const int32_t *rowptr, const int32_t *colidx, const float *vals,
                 const float *x, float *y, int64_t ncols, void *stream);
int mvb_pool_bwd(int n_in_rows, int n_out_rows, const int32_t *rowptr_t, const int32_t *colidx_t,
                 const float *vals_t, const float *dy, float *dx, int64_t ncols, void *stream);

/* ---- A3: Chebyshev convolution forward  (nn/conv.py:557-577 ChebConv_batch.forward; the PyG
 *          ChebConv used at models/cheb_cls.py:95 is the same operator with W_k = lins[k].weight^T)
 * T_0 = x, T_1 = L x, T_k = 2 L T_{k-1} - T_{k-2};  y = sum_k T_k W_k (+ bias) (ReLU if relu != 0;
 * the reference applies F.relu at the call site, models/cheb_VAE.py:264,285).
 * x [N,B,Fin]; weight [K,Fin,Fout]; bias [Fout] or NULL; y [N,B,Fout].
 * CSR (rowptr/colidx/vals) is L_hat with N rows; rows without entries are legal.
 * n_active (0..N): the caller's promise that rows >= n_active have no entries and that no entry
 * references a column >= n_active (pass N when unknown).  Those rows have the closed form
 * T_k = cos(k pi/2) x, so they are contracted once with sum_k cos(k pi/2) W_k instead of running
 * the recurrence - the reference's output layer applies the 20-vertex operator to the
 * 4998-vertex mesh (models/cheb_VAE.py:288) and is 99.6 % such rows.
 * basis [(K-1), n_active, B, Fin] receives T_1..T_{K-1} of the active prefix (saved for the
 * backward pass; may be NULL when K == 1 or n_active == 0).
 * nnz: number of CSR entries (rowptr[N]), or -1 if unknown; lets the fused coarse-level
 * recurrence kernel copy the operator into shared memory. */
int mvb_cheb_fwd(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr,
                 const int32_t *colidx, const float *vals, const float *x, const float *weight,
                 const float *bias, int relu, float *basis, float *y, void *stream);

/* ---- A13: Chebyshev convolution backward (autograd of nn/conv.py:557-577) ------------------
 * Two algebraically equal forms (L acts on vertices, W on features, so they commute):
 *   basis form  : dW_k = T_k^T G ; G_{K-1} = G W_{K-1}^T ; G_k = G W_k^T + 2 L^T G_{k+1} - G_{k+2} ;
 *                 dX = G W_0^T + L^T G_1 - G_2          (what autograd does to the reference code;
 *                 needs the forward basis T_1..T_{K-1});
 *   adjoint form: S_0 = G, S_1 = L^T G, S_k = 2 L^T S_{k-1} - S_{k-2} ; dW_k = x^T S_k ;
 *                 dX = sum_k S_k W_k^T                  (the forward kernels run on G; `basis` unused).
 * G = dY, masked by y_for_relu > 0 when the forward ran with relu != 0 (pass the forward output).
 * mvb_cheb_bwd_uses_basis(Fin, Fout, need_dx) tells which form mvb_cheb_bwd takes (1 = basis form:
 * the caller must keep `basis` from the forward call; 0 = adjoint form: `basis` may be NULL and the
 * forward planes need not be kept).  The adjoint form is chosen when dx is wanted and
 * Fout <= 1.2 Fin (less plane traffic, no reverse recurrence).
 * CSR arguments are L^T (for the symmetric L_hat of nn/conv.py:541-555 this equals L).
 * dx may be NULL (first encoder layer: the input needs no gradient), dbias may be NULL.
 * dweight [K,Fin,Fout] and dbias [Fout] are OVERWRITTEN (deterministic ordered reductions, no
 * atomics).  workspace: mvb_cheb_bwd_workspace_bytes(...) bytes, 16-byte aligned.
 * Width limit: the weight gradient is one reduction [M x n] over the rows, M = K*Fin (+1 for the bias) and n = Fout in
 * the basis form, M = K*Fout and n = Fin in the adjoint form.  The tensor cores take it when M <= 128 and n <= 32 (16-
 * or 4-wide planes with K <= 6 / 8, 32-wide with K <= 3); the FFMA reduction holds ceil(M/4) * ceil(n/4) <= 512
 * register tiles.  Beyond both, mvb_cheb_bwd returns MVB_EINVAL ("wgrad: K*Fin x Fout ... too large") instead of launching it:
 * at K = 6 a 32 -> 48 layer (49 x 12 tiles), 48 -> 32 (48 x 12) or 48 -> 48 (72 x 12) - e.g. num_conv_filters
 * 16, 32, 48, 48, 48 trains no further than its first backward pass.  The forward pass has no such limit there. */
int mvb_cheb_bwd_uses_basis(int Fin, int Fout, int need_dx);
size_t mvb_cheb_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int n_active,
                                    int need_dx);
int mvb_cheb_bwd(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr_t,
                 const int32_t *colidx_t, const float *vals_t, const float *x, const float *basis,
                 const float *weight, const float *y_for_relu, const float *dy, float *dx,
                 float *dweight, float *dbias, void *workspace, size_t workspace_bytes,
                 void *stream);

/* ---- A13b: gradient with respect to the operator values (nn/conv.py:557-581 with a `norm` that requires grad) -------
 * An operator whose values change every step (computed from learned edge weights) keeps its pattern: CSR(L) and
 * CSR(L^T) are built once, with perm[nnz] / perm_t[nnz] mapping each CSR(L) / CSR(L^T) slot to its COO entry (the
 * stable counting sort of mvb_csr_from_coo_host: a stable argsort of the COO rows, resp. columns).
 * mvb_csr_values: vals[j] = coo_vals[perm[j]], vals_t[j] = coo_vals[perm_t[j]] - one launch, enqueue only (capturable).
 *
 * mvb_cheb_bwd_op: everything mvb_cheb_bwd returns in the basis form - dx, dweight, dbias are the same bits - plus
 *   d_coo_vals[e] = <G_1[r], T_0[c]> + 2 sum_{k=2}^{K-1} <G_k[r], T_{k-1}[c]>   (<a,b>: sum over the B*Fin entries of a
 *   vertex row; G_k = dloss/dT_k of the basis form's reverse recurrence; (r, c) = (edge_index[1][e], edge_index[0][e]))
 * OVERWRITTEN in COO order, deterministic (one store per entry, no atomics); all zero when K == 1.  Duplicate entries
 * each receive the full value.  Always the basis form (the caller keeps `basis` from mvb_cheb_fwd whatever
 * mvb_cheb_bwd_uses_basis says); the weight-gradient branch is joined before the call returns - it is never deferred
 * (mvb_side_join has nothing to wait for).
 * rowptr / colidx / perm: CSR(L) (the edge gradient); rowptr_t / colidx_t / vals_t: CSR(L^T) (the reverse recurrence).
 * n_active as for mvb_cheb_fwd: every entry must lie in the active prefix.  dx may be NULL, dbias may be NULL.
 * workspace: mvb_cheb_bwd_op_workspace_bytes(...) bytes, 16-byte aligned. */
int mvb_csr_values(int nnz, const int32_t *perm, const int32_t *perm_t, const float *coo_vals, float *vals, float *vals_t,
                   void *stream);
size_t mvb_cheb_bwd_op_workspace_bytes(int N, int B, int Fin, int Fout, int K, int n_active);
int mvb_cheb_bwd_op(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr,
                    const int32_t *colidx, const int32_t *perm, const int32_t *rowptr_t, const int32_t *colidx_t,
                    const float *vals_t, const float *x, const float *basis, const float *weight,
                    const float *y_for_relu, const float *dy, float *dx, float *dweight, float *dbias,
                    float *d_coo_vals, void *workspace, size_t workspace_bytes, void *stream);

/* ---- A9: reparameterisation  (models/cheb_VAE.py:309-319) ----------------------------------
 * z = eps * exp(0.5 * logvar) + mu  on n = B*Z elements; eps is supplied by the caller (the
 * reference draws it with the CPU generator, :316).  Backward: dmu = dz, dlogvar = dz*eps*0.5*std. */
int mvb_vae_reparam_fwd(int64_t n, const float *mu, const float *logvar, const float *eps,
                        float *z, void *stream);
int mvb_vae_reparam_bwd(int64_t n, const float *logvar, const float *eps, const float *dz,
                        float *dmu, float *dlogvar, void *stream);

/* ---- A10/A11: loss epilogue  (models/cheb_VAE.py:321-346 loss_function; logpdf.py:7-8 KLD,
 *          :22-23 gaussian_nll, :24-28 softclip) -----------------------------------------------
 * recon  [N,B,recon_ld] fp32 VERTEX-MAJOR (the decoder output as the kernels produce it): recon_ld >= C
 *        floats per (vertex, mesh) entry, the first C are the reconstruction (the 3-channel output layer
 *        writes entries padded to 4 floats: passing it with recon_ld = 4 saves the slice copy);
 * x_gt   [B,N,C] mesh-major as main.py:70 delivers it, fp64 (x_is_f64 != 0; data.py:107) or fp32
 *        (inference.py:87);  mu/logvar [B,Z];  y_hat [B,ncls] softmax;  y [B,ncls] int64 one-hot;
 * log_sigma = softclip(1, -6) = 1.0009117 by default (models/cheb_VAE.py:328-329).
 * Outputs: loss[1] (fp64; mean_b(kld + rec - 2 log sum_c(y_hat*y))), kld[B] fp32, rec[B] fp64,
 * correct[1] int64, dnll [N,B,recon_ld] fp32 = (recon - x_gt)/sigma^2, zero in the padding (saved for
 * backward).
 * Arithmetic is fp64 when x_gt is fp64 (as torch type promotion makes the reference do),
 * per-element fp32 with fp64 accumulation otherwise.  Deterministic (fixed-order reductions).
 * Entry width: 8 vertices x 32 meshes of C x_gt values and recon_ld floats must fit 48 KB of shared memory - C = recon_ld
 * up to 16 with fp64 x_gt, 24 with fp32; a wider entry returns MVB_EINVAL ("C too large").  No alignment is required of
 * recon, x_gt or dnll (16-byte aligned buffers take the vector paths).
 * workspace: mvb_vae_loss_workspace_bytes(B, N) bytes. */
size_t mvb_vae_loss_workspace_bytes(int B, int N);
int mvb_vae_loss_fwd(int B, int N, int C, int Z, int ncls, const float *recon, int recon_ld, const void *x_gt,
                     int x_is_f64, const float *mu, const float *logvar, const float *y_hat,
                     const int64_t *y, float log_sigma, double *loss, float *kld, double *rec,
                     int64_t *correct, float *dnll, void *workspace, size_t workspace_bytes,
                     void *stream);
/* gloss: DEVICE pointer to the fp64 upstream gradient of `loss` (a scalar).  C here is the entry width of
 * dnll (the recon_ld of the forward call).
 * d_recon[N,B,C] = gloss/B * dnll ; d_mu = gloss/B * mu ; d_logvar = gloss/B * 0.5 (exp(logvar) - 1);
 * d_yhat[b,c] = gloss/B * (-2) * y[b,c] / sum_c(y_hat*y). Any output pointer may be NULL. */
int mvb_vae_loss_bwd(int B, int N, int C, int Z, int ncls, const float *dnll, const float *mu,
                     const float *logvar, const float *y_hat, const int64_t *y,
                     const double *gloss, float *d_recon, float *d_mu, float *d_logvar,
                     float *d_yhat, void *stream);

/* sigma-VAE decoder likelihood (Rybkin et al., "Simple and Effective VAE Training with Calibrated Decoders"): the same
 * loss with a decoder log sigma that is computed on the device instead of passed by the host.  With
 * sc(t) = -6 + softplus(t + 6), n = N*C and SSE = sum_b SSE_b the batch's squared error sum_(b,v,c) (recon - x_gt)^2:
 *   sigma_mode MVB_SIGMA_OPTIMAL: log sigma = sc(0.5 log(SSE / (B n)))  (the gradient flows through sigma);
 *   sigma_mode MVB_SIGMA_LEARNED: log sigma = sc(*s_param), s_param a DEVICE fp32 scalar (a parameter);
 *   rec[b] = 0.5 SSE_b / sigma^2 + n (log sigma + 0.5 log(2 pi)), fp64 arithmetic after the per-element squares
 *   (fp64 squares of differences taken in fp64 when x_gt is fp64, in fp32 otherwise).
 * Arguments and other outputs as mvb_vae_loss_fwd, except dnll = recon - x_gt UNSCALED (zero in the padding).
 * sigma_state: 8 fp64 of device memory written by the forward call, read by the backward call:
 *   [0] log sigma, [1] sigma^-2, [2] SSE, [3] sc'(t) = sigmoid(t + 6), [4] coef (below),
 *   [5] d(sum_b rec_b)/dt = (B n - SSE sigma^-2) sc'(t), [6..7] unused.
 * A perfect reconstruction (SSE = 0) under the optimal sigma gives t = -inf: log sigma = -6, sc' = 0, finite results.
 * No host round trip, no atomics: capturable, and bit-reproducible run to run.  The fixed-sigma entry points above are
 * unaffected. */
#define MVB_SIGMA_OPTIMAL 1
#define MVB_SIGMA_LEARNED 2
int mvb_vae_loss_sigma_fwd(int B, int N, int C, int Z, int ncls, const float *recon, int recon_ld, const void *x_gt,
                           int x_is_f64, const float *mu, const float *logvar, const float *y_hat, const int64_t *y,
                           int sigma_mode, const float *s_param, double *sigma_state, double *loss, float *kld,
                           double *rec, int64_t *correct, float *dnll, void *workspace, size_t workspace_bytes,
                           void *stream);
/* d_recon = gloss/B * coef * dnll with coef = sigma^-2 (learned) or sigma^-2 + (B n - SSE sigma^-2) sc'/SSE (optimal,
 * SSE > 0; sigma^-2 when SSE = 0); d_mu, d_logvar, d_yhat as mvb_vae_loss_bwd; d_s (fp32 scalar, learned sigma) =
 * gloss/B * (B n - SSE sigma^-2) sc'(s), written (not accumulated): it may point into a flat gradient buffer.  C is the
 * entry width of dnll.  Any output pointer may be NULL. */
int mvb_vae_loss_sigma_bwd(int B, int N, int C, int Z, int ncls, const float *dnll, const double *sigma_state,
                           const float *mu, const float *logvar, const float *y_hat, const int64_t *y,
                           const double *gloss, float *d_recon, float *d_mu, float *d_logvar, float *d_yhat,
                           float *d_s, void *stream);

/* ---- importance-weighted estimate of the held-out log-likelihood log p(x | y) (no counterpart in the reference) ----
 * With S samples z_(b,s) ~ q(z | x_b, y_b) per mesh and n = N*C:
 *   log w_(b,s) = log p(x_b | z_(b,s), y_b) - (log q(z_(b,s) | x_b, y_b) - log p(z_(b,s)))
 *   log p(x | z) = -SSE / (2 sigma^2) - n (log sigma + 0.5 log(2 pi)),  log p(x_b | y_b) ~ log mean_s exp(log w_(b,s)).
 * Densities are those of the coordinates the model sees (z-scored).  All sums fp64 in a fixed order; no atomics, no
 * host synchronisation: capturable and bit-reproducible run to run.
 *
 * mvb_iw_sample: mu, logvar [B,Z] fp32 (the heads at eval, z = mu there), eps [B,S,Z] fp32 N(0, I) from the caller,
 *   y [B,C] int64 one-hot.  Writes the decoder input zcat [B*S, C+Z] fp32, mesh-major (row b*S + s = cat(y_b, z)) with
 *   z = eps * exp(0.5 logvar) + mu in fp32 as mvb_vae_reparam_fwd computes it, and
 *   log_r [B*S] fp64 = sum_j (-eps_j^2/2 - logvar_j/2 + z_j^2/2) = log q(z | x, y) - log p(z). */
int mvb_iw_sample(int B, int S, int Z, int C, const float *mu, const float *logvar, const float *eps, const int64_t *y,
                  float *zcat, double *log_r, void *stream);
/* mvb_iw_log_weights: one chunk of S samples per mesh.  recon [N, B*S, recon_ld] fp32 VERTEX-MAJOR (the decoder output
 *   of mvb_iw_sample's zcat: column b*S + s), x_gt [B,N,C] mesh-major fp64 (x_is_f64 != 0) or fp32, log_sigma a DEVICE
 *   fp64 scalar, log_r [B*S] fp64 of the same chunk.  SSE per reconstruction as mvb_vae_loss_sigma_fwd sums it (the
 *   same partial kernel: fp64 squares of differences taken in x_gt's precision), then
 *   log_w[b*S_total + s0 + s] = log p(x_b | z) - log_r[b*S + s]   for s < S  (log_w [B, S_total] fp64, s0 + S <= S_total).
 *   Entry width limits as mvb_vae_loss_fwd; B*S at most 65535*32 = 2097120 reconstructions per call (MVB_EINVAL beyond).
 *   workspace: mvb_iw_log_weights_workspace_bytes(B, S, N) bytes. */
size_t mvb_iw_log_weights_workspace_bytes(int B, int S, int N);
int mvb_iw_log_weights(int B, int S, int N, int C, const float *recon, int recon_ld, const void *x_gt, int x_is_f64,
                       const double *log_sigma, const double *log_r, int S_total, int s0, double *log_w, void *workspace,
                       size_t workspace_bytes, void *stream);
/* mvb_iw_reduce: log_w [B,S] fp64 -> per mesh (fp64 [B]) with m = max_s log w and e_s = exp(log w_s - m):
 *   log_px = m + log sum_s e_s - log S ;  elbo = (1/S) sum_s log w_s ;  ess = (sum_s e_s)^2 / sum_s e_s^2.
 *   log_w_out [B,S] (may be NULL): a copy of log_w for the caller. */
int mvb_iw_reduce(int B, int S, const double *log_w, double *log_px, double *elbo, double *ess, double *log_w_out, void *stream);

/* ---- logpdf.py drop-ins used when the reference's own loss_function runs unchanged ----------
 * KLD (logpdf.py:7-8): out[b] = -0.5 sum_j (1 + logvar - mu^2 - exp(logvar)); bwd as above.
 * gaussian_nll (logpdf.py:22-23), elementwise on n values with scalar log_sigma:
 *   out = 0.5 ((x - mu)/exp(log_sigma))^2 + log_sigma + 0.5 log(2 pi); out/x are fp64 when
 *   x_is_f64 != 0 else fp32; mu (the reconstruction) is fp32.  d_mu = g * (mu - x)/sigma^2. */
int mvb_kld_fwd(int B, int Z, const float *mu, const float *logvar, float *out, void *stream);
int mvb_kld_bwd(int B, int Z, const float *mu, const float *logvar, const float *gout,
                float *d_mu, float *d_logvar, void *stream);
int mvb_gaussian_nll_fwd(int64_t n, const float *mu, const void *x, int x_is_f64, float log_sigma,
                         void *out, void *stream);
int mvb_gaussian_nll_bwd(int64_t n, const float *mu, const void *x, int x_is_f64, float log_sigma,
                         const void *gout, float *d_mu, void *stream);
/* gaussian_nll with log_sigma a DEVICE scalar, fp64 (ls_is_f64 != 0) or fp32 (a learned or batch-derived sigma, read
 * without a host sync): sigma = exp(log_sigma) in the scalar's precision, as torch forms log_sigma.exp() (the fp32 exp
 * correctly rounded), then converted to the arithmetic's precision (that of x).  The backward pass also returns
 * d_log_sigma[0] (fp64) = sum_i g_i (1 - ((x_i - mu_i)/sigma)^2) from per-block partials and an ordered sum:
 * deterministic.  workspace: mvb_gaussian_nll_sigma_workspace_bytes(n) bytes. */
int mvb_gaussian_nll_sigma_fwd(int64_t n, const float *mu, const void *x, int x_is_f64, const void *log_sigma,
                               int ls_is_f64, void *out, void *stream);
size_t mvb_gaussian_nll_sigma_workspace_bytes(int64_t n);
int mvb_gaussian_nll_sigma_bwd(int64_t n, const float *mu, const void *x, int x_is_f64, const void *log_sigma,
                               int ls_is_f64, const void *gout, float *d_mu, double *d_log_sigma, void *workspace,
                               size_t workspace_bytes, void *stream);

/* ---- input hand-off: mesh-major batch -> zero-padded vertex-major planes --------------------
 * out[n, b, 0:Cp] = (x[b, n, 0:C], 0...)   x [B,N,C] as the loader delivers it (models/cheb_VAE.py:195-200
 * reshape), out [N,B,Cp] with Cp >= C (4 for the 3-channel meshes): the layout every kernel works in.  C <= 8; no
 * alignment is required (a 16-byte aligned out takes the vector stores when C = 3, Cp = 4). */
int mvb_pack_vertex_major(int B, int N, int C, int Cp, const float *x, float *out, void *stream);

/* ---- next row f3: per-batch reconstruction error  (main.py:88-93, :139-146; inference.py:100-127)
 * recon_mesh = out * std + mean (fp32) ; recon_mesh = bmm(recon_mesh * s, R) + m (fp64) ;
 * diff = sqrt(((recon_mesh - gt_mesh)^2).sum(-1)) ; mean_err[b] = diff.mean(-1), max_err[b] = diff.max(-1).
 * recon [N,B,ld] fp32 vertex-major with ld >= 3 floats per (vertex, mesh) entry (the decoder output as
 * the kernels produce it, padded to 4); mean/std [N,3] fp32 (norm.npz); s [B], R [B,3,3], m [B,3] fp64
 * (Procrustes scale / rotation / translation, utils.py:58-156); gt [B,N,3] original meshes, fp64 (gt_is_f64 != 0)
 * or fp32 as the loader collates them (data.py:133 torch.Tensor(points)) - read without a conversion pass.
 * The reference copies the [B,N,3] reconstruction to the host for this every batch.
 * Optional outputs (NULL = not wanted): vertex_err [B,N] fp32 = diff itself (evaluate() returns the
 * concatenated per-vertex errors, main.py:146-148); mesh_out [B,N,3] fp32 = the back-transformed mesh
 * (what evaluate(vis=True) / inference.py:131-140 write as OBJ files).  gt may be NULL when only
 * mesh_out is wanted (the sex-changed mesh of main.py:162-164 has no ground truth): errors are 0 then. */
size_t mvb_recon_error_workspace_bytes(int B, int N);
int mvb_recon_error(int B, int N, int ld, const float *recon, const float *mean, const float *std, const double *s,
                    const double *R, const double *m, const void *gt, int gt_is_f64, double *mean_err, double *max_err,
                    float *vertex_err, float *mesh_out, void *workspace, size_t workspace_bytes, void *stream);

/* ---- next row f3: epoch statistics on the device  (main.py:60-65, 83-86, 93, 96; :135-137) ------
 * acc[0] += loss * B; acc[1] += sum_b kld[b]; acc[2] += sum_b rec[b]; acc[3] += sum_b mean_err[b] (if given);
 * acc[4] += correct (if given); acc[5] += B.   acc: 8 fp64 device accumulators, zeroed by the caller per epoch
 * and read once at its end (the reference synchronises three times per batch, main.py:83-85).  With
 * kld.mean()*B == sum kld etc. these are exactly the running totals of main.py.  loss: fp64 or fp32 scalar,
 * rec: fp64 or fp32 [B] (as mvb_vae_loss_fwd returns them), correct: int64 scalar. */
int mvb_epoch_meter_add(int B, const void *loss, int loss_is_f64, const float *kld, const void *rec, int rec_is_f64,
                        const int64_t *correct, const double *mean_err, double *acc, void *stream);

/* ---- next row f2: fused Adam on a flat parameter buffer  (main.py:251 torch.optim.Adam(lr,
 *          weight_decay), L2-style decay; main.py:81 optimizer.step()) --------------------------
 * step: DEVICE int64 counter, incremented by one inside the call (graph-capturable, no host state).
 * g <- g*grad_scale + wd*p ; m <- b1 m + (1-b1) g ; v <- b2 v + (1-b2) g^2 ;
 * p <- p - lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps).   grad_scale = 1/world_size folds the
 * data-parallel gradient average into the update. */
int mvb_adam_step(int64_t n, float *p, const float *g, float *m, float *v, int64_t *step, float lr,
                  float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                  void *stream);
/* The same update with the hyper-parameters in DEVICE memory, hyper[6] = {lr, beta1, beta2, eps, weight_decay,
 * grad_scale}: a captured step follows main.py's per-epoch learning-rate schedule (main.py:266-269 rewrites
 * optimizer.param_groups[..]['lr']) and a restored optimizer state without re-capture. */
int mvb_adam_step_hp(int64_t n, float *p, const float *g, float *m, float *v, int64_t *step, const float *hyper,
                     void *stream);

/* ---- data parallel (new; the reference is single device): gradient exchange fused with the optimizer -------------
 * One process per GPU; every rank keeps its flat fp32 gradient buffer and a 256-byte signal pad (zero at creation) in
 * memory that its peers on the node have mapped (NVLink / NVSwitch peer access: torch symmetric memory, CUDA IPC, ... -
 * the pointers are handed in as HOST arrays of `world` device pointers, entry `rank` = the local buffer).
 *   mvb_dp_begin        at the head of a step, before anything writes the local gradient buffer: opens a new epoch once
 *                       every peer has finished reading that buffer in the previous one (`channels` = how many exchanges a
 *                       step makes, 1 or 2; every step must then use exactly the channels 0..channels-1 once each).
 *   mvb_dp_reduce_adam  instead of all-reduce + mvb_adam_step_hp, for the elements [offset, offset + n) of the flat buffers
 *                       (a gradient bucket; offset, n multiples of 4): tells the peers the local gradient is complete, waits
 *                       for theirs, sums grads[0..world-1] in rank order (bit-identical on every rank, no atomics) straight
 *                       out of the peers' memory and applies Adam (hyper as in mvb_adam_step_hp; fold 1/world into
 *                       hyper[5]) to the local replica of p / m / v in the same pass; grad_sum_out (or NULL) receives the
 *                       summed gradient.  tick = 1: the step counter is incremented first (the first exchange of a step).
 *                       Two buckets on two channels may be in flight at once (the early one on a side stream under the
 *                       rest of the backward pass); max_ctas > 0 caps the grid of such a background launch.
 * p / m / v, grad_sum_out and every rank's gradient buffer must be 16-byte aligned (MVB_EALIGN otherwise).
 * state: mvb_dp_state_bytes() of LOCAL device memory, zero at creation (uint32 words: [0] epoch, [1] number of waits that
 * gave up after ~30 s because a peer never signalled - the results are then invalid; a healthy run keeps it 0).  Every
 * rank must issue the same sequence of begin / reduce calls.  Enqueue-only and CUDA-graph capturable (signals are epoch
 * numbers that only grow). */
int mvb_dp_max_world(void);
size_t mvb_dp_pad_bytes(void);
size_t mvb_dp_state_bytes(void);
int mvb_dp_begin(int world, int rank, int channels, void *const *pads, void *state, void *stream);
int mvb_dp_reduce_adam(int world, int rank, int channel, int64_t offset, int64_t n, float *p, void *const *grads, float *m, float *v,
                       float *grad_sum_out, int64_t *step, int tick, const float *hyper, void *const *pads, void *state,
                       int max_ctas, void *stream);

/* ---- A3 + A5 fused on the step-by-step path: Chebyshev convolution + row selection -------------------------------
 * (the encoder loop body  x = relu(cheb[i](x, L)); x = pool(x, D)  models/cheb_VAE.py:264-265, at the levels too large
 *  for the mesh-resident kernels: level 0 of the template; D is a row selection, mesh_operations.py:72-85.)
 * y_sel [n_sel,B,Fout] = act(conv(x))[sel]: only the rows D keeps (1/4) are contracted and written.  basis as for
 * mvb_cheb_fwd ((K-1) planes [N,B,Fin], all rows - kept for the backward pass).
 * mvb_cheb_sel_bwd: dW / db of such a layer when its input needs NO gradient (the first encoder layer: the basis form
 * dW_k = T_k^T G, db = 1^T G, G = dy_sel * [y_sel > 0] reduced over the selected rows only - G is zero elsewhere).
 * mvb_cheb_sel_supported: 1 for the plane widths of the tensor-core kernels (Fin 4 / 16 / 32, Fout % 4 == 0, <= 32), else 0 -
 * the caller then composes mvb_cheb_fwd + mvb_pool_fwd.  sel[n_sel]: distinct conv rows (see mvb_cheb_layer_fwd). */
int mvb_cheb_sel_supported(int N, int B, int Fin, int Fout, int K, int n_sel);
int mvb_cheb_sel_fwd(int N, int B, int Fin, int Fout, int K, int nnz, const int32_t *rowptr, const int32_t *colidx,
                     const float *vals, const float *x, const float *weight, const float *bias, int relu, int n_sel,
                     const int32_t *sel, float *basis, float *y_sel, void *stream);
size_t mvb_cheb_sel_bwd_workspace_bytes(int Fin, int Fout, int K);
int mvb_cheb_sel_bwd(int N, int B, int Fin, int Fout, int K, const float *x, const float *basis, const float *y_sel_for_relu,
                     const float *dy_sel, int n_sel, const int32_t *sel, float *dweight, float *dbias, void *workspace,
                     size_t workspace_bytes, void *stream);

/* ---- A12 fused: one whole encoder / decoder layer of a COARSE level per launch ---------------
 * (models/cheb_VAE.py:264-265  x = relu(cheb[i](x, L)); x = pool(x, D)   and
 *  models/cheb_VAE.py:284-285  x = pool(x, U); x = relu(cheb_dec[i](x, L)) ).
 * One thread block per mesh keeps the layer in shared memory: optional up-sampling prologue
 * T_0 = U x, the recurrence, the contraction with bias / ReLU, and an optional row-selection
 * epilogue (only the rows that D keeps are contracted and written).
 *   x [n_in,B,Fin] (n_in == N unless U [N x n_in] is given), y [n_out,B,Fout] (n_out == N unless
 *   sel[n_out] is given: output row r is conv row sel[r] - D is such a selection,
 *   mesh_operations.py:72-85: one 1.0 per row).  The entries of sel must be distinct (the kernels invert the map); a D
 *   that selects a vertex twice is a plain sparse product: mvb_pool_* after the convolution.  The same holds for the sel
 *   of mvb_cheb_sel_*.
 * Two implementations behind the same entry points: the tensor-core mesh kernels (csrc/mvb_mesh_tc.cu: 16 / 32-wide
 *   features, up to 1280 vertices - levels 1-3 of the template; a cluster of 1-2 CTAs per mesh keeps the basis planes
 *   in shared memory in the UMMA operand layout and contracts them with tcgen05.mma into TMEM accumulators) and the
 *   FFMA mesh kernels (csrc/mvb_layer.cu: Fin and Fout of 4, 8, 16, 32 or 64 - a power-of-two number of 4-wide quads -
 *   and a few hundred vertices).
 * mvb_cheb_layer_supported: 1 when one of them covers the level in both directions, else 0 - the caller then uses
 *   mvb_pool_* + mvb_cheb_*.
 * Backward: nothing but x and y is kept from the forward pass (the basis is recomputed in shared
 *   memory).  dweight / dbias OVERWRITTEN; dx [n_in,B,Fin] may be NULL.  L^T / U^T as in
 *   mvb_cheb_bwd / mvb_pool_bwd.  workspace: mvb_cheb_layer_bwd_workspace_bytes(N, B, Fin, Fout, K, has_up = U given)
 *   (per-mesh partials summed in mesh order by a second kernel, or the S_k planes of the adjoint form for the
 *   streaming weight-gradient reduction: deterministic either way). */
int mvb_cheb_layer_supported(int N, int B, int Fin, int Fout, int K, int L_nnz, int n_in, int U_nnz, int n_out);
int mvb_cheb_layer_fwd(int N, int B, int Fin, int Fout, int K, const int32_t *L_rowptr, const int32_t *L_colidx,
                       const float *L_vals, int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx,
                       const float *U_vals, int U_nnz, int n_out, const int32_t *sel, const float *x,
                       const float *weight, const float *bias, int relu, float *y, void *stream);
size_t mvb_cheb_layer_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up);
int mvb_cheb_layer_bwd(int N, int B, int Fin, int Fout, int K, const int32_t *L_rowptr, const int32_t *L_colidx,
                       const float *L_vals, const int32_t *Lt_rowptr, const int32_t *Lt_colidx, const float *Lt_vals,
                       int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx, const float *U_vals,
                       const int32_t *Ut_rowptr, const int32_t *Ut_colidx, const float *Ut_vals, int U_nnz, int n_out,
                       const int32_t *sel, const float *x, const float *weight, const float *y_for_relu,
                       const float *dy, float *dx, float *dweight, float *dbias, void *workspace,
                       size_t workspace_bytes, void *stream);

/* ---- the same loop body at the levels that do NOT fit shared memory (level 0: 4998 vertices) ----
 * pool(U) -> ChebConv_batch -> ReLU, models/cheb_VAE.py:284-285 (nn/conv.py:557-577, nn/pool.py:13-23), as ONE
 * persistent launch per direction (csrc/mvb_stream_tc.cu): every CTA owns a block of rows x a slab of 8 / 16 meshes (tiles of
 * 128 (vertex, mesh) pairs), produces each basis plane T_k for them with the arithmetic of mvb_spmm, hands the tile to tcgen05.mma through a
 * shared-memory ring while it is still on chip (accumulators of all its tiles in TMEM across the K steps) and meets
 * the other CTAs at a grid-wide barrier between steps - the basis is never re-read for the contraction.
 *   x [n_in,B,16] (n_in == N unless U [N x n_in] is given), weight [K,16,16], y [N,B,16]; 16-wide features, K <= 8,
 *   no row selection; mvb_cheb_stream_supported says whether (N, B) is covered (opt-in: mvb_tune "stream_tc=1"; B a
 *   multiple of 8, at least ~76 k (vertex, mesh) pairs, and few enough that a CTA's accumulators fit TMEM: B <= ~112 at
 *   4998 vertices) - otherwise use mvb_pool_* + mvb_cheb_*.
 * Backward (adjoint form): G = dY*[y>0] and db, S_k = T_k(L^T) G, dT_0 = sum_k S_k W_k^T, dX = U^T dT_0 in the same
 *   launch; dW through the streaming weight-gradient reduction (on the deferred side chain with mvb_tune
 *   "defer_wgrad=1").  dweight / dbias OVERWRITTEN; dx may be NULL.  Workspaces: *_workspace_bytes; 16-byte aligned. */
int mvb_cheb_stream_supported(int N, int B, int Fin, int Fout, int K, int n_in, int has_up, int n_out);
size_t mvb_cheb_stream_fwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up);
int mvb_cheb_stream_fwd(int N, int B, int Fin, int Fout, int K, const int32_t *L_rowptr, const int32_t *L_colidx,
                        const float *L_vals, int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx,
                        const float *U_vals, int U_nnz, const float *x, const float *weight, const float *bias, int relu,
                        float *y, void *workspace, size_t workspace_bytes, void *stream);
size_t mvb_cheb_stream_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up);
int mvb_cheb_stream_bwd(int N, int B, int Fin, int Fout, int K, const int32_t *Lt_rowptr, const int32_t *Lt_colidx,
                        const float *Lt_vals, int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx,
                        const float *U_vals, const int32_t *Ut_rowptr, const int32_t *Ut_colidx, const float *Ut_vals,
                        int U_nnz, const float *x, const float *weight, const float *y_for_relu, const float *dy, float *dx,
                        float *dweight, float *dbias, void *workspace, size_t workspace_bytes, void *stream);

/* ---- next row f2: the dense bottleneck between the two mesh pyramids ------------------------
 * (models/cheb_VAE.py:149-168 layer definitions; :270-272 enc_lin; :253-258 classifier; :206-221
 *  z heads + reparameterisation; :276-281 dec_lin / dec_lin_2 - torch.nn.Linear + F.relu +
 *  nn.Dropout in the reference, ~60 ATen/cuBLAS launches per training step.)
 *
 * mvb_linear_fwd:  y = dropout_p(relu?(x W^T + bias)),  x logical [M,K], W [N,K] row-major
 *   (torch.nn.Linear.weight), bias [N] or NULL, y logical [M,N].
 *   x_vm_f / y_vm_f: 0 = the matrix is row-major; F > 0 = it is a VERTEX-MAJOR activation
 *   [K/F, M, F] (resp. [N/F, M, F]) - what x.reshape(B, -1) / x.reshape(B, -1, F) of the reference
 *   (models/cheb_VAE.py:270, :281) mean for the [vertices, B, F] buffers of the mesh kernels, so no
 *   transpose copy is made on either side of the bottleneck.
 *   Dropout (p_drop in [0,1), 0 = off / eval mode): inverted dropout with a Philox4x32-10 mask
 *   keyed by (seed, offset, m*N + n), offset = offset_host + (offset_dev ? *offset_dev : 0); the
 *   device term lets a captured CUDA graph draw a fresh mask on every replay.
 * mvb_linear_bwd:  gp = gy * [y > 0]/(1 - p_drop) (relu != 0: y is the forward OUTPUT, a clamped
 *   or dropped unit has y == 0) or gp = gy (relu == 0; p_drop must be 0);
 *   dW [N,K] = gp^T x, db [N] = column sums of gp (may be NULL), dx = gp W in the layout of x (may
 *   be NULL).  y and gy share the layout y_vm_f.  All three are OVERWRITTEN; fixed summation
 *   order, no atomics. */
int mvb_linear_fwd(int M, int K, int N, const float *x, int x_vm_f, const float *W, const float *bias,
                   int relu, float p_drop, uint64_t seed, const int64_t *offset_dev, int64_t offset_host,
                   float *y, int y_vm_f, void *stream);
int mvb_linear_bwd(int M, int K, int N, const float *x, int x_vm_f, const float *W, const float *y,
                   const float *gy, int y_vm_f, int relu, float p_drop, float *dx, float *dW, float *db,
                   void *stream);
/* mvb_vae_heads_fwd: the three heads on h [B,H] (the encoder code after enc_lin):
 *   y_hat [B,C]  = softmax(dropout_p(h) Wc^T + bc)                  models/cheb_VAE.py:253-258
 *   mu, logvar [B,Z] = cat(y, h) Wm^T + bm, cat(y, h) Wv^T + bv     :206-212  (Wm, Wv: [Z, C+H])
 *   z [B,Z]      = mu + eps * exp(logvar/2), or mu when eps == NULL  :215-221, :309-319
 *   zcat [B,C+Z] = cat(y, z)                                         :223
 *   y_onehot [B,C] int64 (main.py:71).  The classifier's dropout is the SECOND mask on h (quirk 8):
 *   a Philox4x32-10 mask keyed by (seed, offset, b*H + j), b the row within the call, offset as for
 *   mvb_linear_fwd - so the first rows of a large call get the mask of a smaller call.
 *   Shapes: any B, H, Z >= 1, C <= 32 (the softmax is one warp's), B*H < 2^32 (the mask counter).
 *   One-launch kernels where the C + 2Z weight rows (forward) or the batch's small gradients
 *   (backward) fit one block's shared memory (at H = 512, Z = 16, C = 2: any B forward, B <= 278
 *   backward), tiled kernels elsewhere; both sum in the same order, so the results are the same bits.
 * mvb_vae_heads_bwd: from the upstream gradients of the five outputs (any may be NULL = zero) to
 *   g_h [B,H] and the six parameter gradients (OVERWRITTEN); same (p_drop, seed, offset) as the
 *   forward call so that the mask is regenerated, not stored.  No workspace, no atomics. */
int mvb_vae_heads_fwd(int B, int H, int Z, int C, const float *h, const int64_t *y_onehot, const float *eps,
                      const float *Wc, const float *bc, const float *Wm, const float *bm, const float *Wv,
                      const float *bv, float p_drop, uint64_t seed, const int64_t *offset_dev,
                      int64_t offset_host, float *y_hat, float *mu, float *logvar, float *z, float *zcat,
                      void *stream);
int mvb_vae_heads_bwd(int B, int H, int Z, int C, const float *h, const int64_t *y_onehot, const float *eps,
                      const float *Wc, const float *Wm, const float *Wv, const float *y_hat,
                      const float *logvar, float p_drop, uint64_t seed, const int64_t *offset_dev,
                      int64_t offset_host, const float *g_yhat, const float *g_mu, const float *g_logvar,
                      const float *g_z, const float *g_zcat, float *g_h, float *dWc, float *dbc, float *dWm,
                      float *dbm, float *dWv, float *dbv, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MVB_H_ */
