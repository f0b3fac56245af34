// CSR SpMM over vertex-major activations: the B200 replacement of the reference's
// gather / scale / scatter_add propagate (nn/conv.py:199-200, :579-581, :363-364) and of the
// recurrence arithmetic `2 * prop - Tx_0` (nn/conv.py:569).
//
//   y[r,:] = alpha * sum_j vals[j] * x[colidx[j],:] + beta * z[r,:] + w[r,:]
//
// One thread owns one 16-byte column quad of one output row; consecutive threads walk the
// B*F columns of a row first, so every neighbour gather is a run of fully coalesced 512-byte
// warp requests.  Nothing is materialised per edge (the reference materialises [E,B,F]).
// Roofline: HBM/L2 bandwidth; algorithmic bytes = (2 or 3)*N*ncols*4 + CSR (SURVEY.md 8(d)).
#include "mvb_internal.cuh"

namespace mvb {

__device__ __forceinline__ float4 ldg4(const float4 *p) { return __ldg(p); }

__device__ __forceinline__ void fma4(float4 &acc, float v, const float4 &x) {
    acc.x = fmaf(v, x.x, acc.x);
    acc.y = fmaf(v, x.y, acc.y);
    acc.z = fmaf(v, x.z, acc.z);
    acc.w = fmaf(v, x.w, acc.w);
}

// 2-D thread mapping: threadIdx.x walks the column quads of a row (coalesced), threadIdx.y the rows
// of the block - no integer division anywhere; IdxT = uint32_t whenever the tensors have fewer than
// 2^31 quads (always, in practice), so that address arithmetic is a single 32-bit multiply-add.
// (The first version computed row = idx / nc4 in 64-bit arithmetic per thread: ncu showed 226
// instructions per thread and an issue-bound kernel - see profiles/README.md.)
template <bool HAS_Z, bool HAS_W, typename IdxT>
__global__ void __launch_bounds__(1024)
spmm_v4_kernel(int n_rows, const int32_t *__restrict__ rowptr, const int32_t *__restrict__ colidx,
               const float *__restrict__ vals, const float4 *__restrict__ x, float4 *y,
               const float4 *z, const float4 *w, float alpha, float beta, int nc4, int chunk) {
    pdl_trigger();
    pdl_wait();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nc4) return;
    // a block walks `chunk` CONSECUTIVE rows of its column slab (blockDim.y rows at a time): the mesh
    // operators are banded, so the x rows gathered by one row group are gathered again by the next
    // ones and stay in L1 - the slab is narrow enough (blockDim.x * 16 bytes per row) for the sliding
    // window of every resident block to fit
    const int r_end = min(n_rows, (int)(blockIdx.y + 1) * chunk);
    for (int r = blockIdx.y * chunk + threadIdx.y; r < r_end; r += blockDim.y) {
        const int s = __ldg(rowptr + r), e = __ldg(rowptr + r + 1);
        const IdxT idx = (IdxT)r * (IdxT)nc4 + (IdxT)c;
        float4 zz = make_float4(0.f, 0.f, 0.f, 0.f), ww = zz;
        if (HAS_Z) zz = __ldcs(z + idx);             // independent of the gathers: issue first; streaming (read once)
        if (HAS_W) ww = __ldcs(w + idx);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int j = s;
        // 4 independent gathers in flight per thread (mean degree is 6)
        for (; j + 4 <= e; j += 4) {
            const int c0 = __ldg(colidx + j), c1 = __ldg(colidx + j + 1);
            const int c2 = __ldg(colidx + j + 2), c3 = __ldg(colidx + j + 3);
            const float v0 = __ldg(vals + j), v1 = __ldg(vals + j + 1);
            const float v2 = __ldg(vals + j + 2), v3 = __ldg(vals + j + 3);
            const float4 x0 = ldg4(x + ((IdxT)c0 * (IdxT)nc4 + (IdxT)c));
            const float4 x1 = ldg4(x + ((IdxT)c1 * (IdxT)nc4 + (IdxT)c));
            const float4 x2 = ldg4(x + ((IdxT)c2 * (IdxT)nc4 + (IdxT)c));
            const float4 x3 = ldg4(x + ((IdxT)c3 * (IdxT)nc4 + (IdxT)c));
            fma4(acc, v0, x0);
            fma4(acc, v1, x1);
            fma4(acc, v2, x2);
            fma4(acc, v3, x3);
        }
        for (; j < e; ++j) {
            const int c0 = __ldg(colidx + j);
            const float v0 = __ldg(vals + j);
            fma4(acc, v0, ldg4(x + ((IdxT)c0 * (IdxT)nc4 + (IdxT)c)));
        }
        float4 o = make_float4(alpha * acc.x, alpha * acc.y, alpha * acc.z, alpha * acc.w);
        if (HAS_Z) {
            o.x = fmaf(beta, zz.x, o.x);
            o.y = fmaf(beta, zz.y, o.y);
            o.z = fmaf(beta, zz.z, o.z);
            o.w = fmaf(beta, zz.w, o.w);
        }
        if (HAS_W) {
            o.x += ww.x;
            o.y += ww.y;
            o.z += ww.z;
            o.w += ww.w;
        }
        y[idx] = o;
    }
}

__global__ void __launch_bounds__(256)
spmm_scalar_kernel(int n_rows, const int32_t *__restrict__ rowptr,
                   const int32_t *__restrict__ colidx, const float *__restrict__ vals,
                   const float *__restrict__ x, float *y, const float *z, const float *w,
                   float alpha, float beta, int64_t ncols) {
    const int64_t total = (int64_t)n_rows * ncols;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(idx / ncols);
        const int64_t c = idx - (int64_t)r * ncols;
        const int s = __ldg(rowptr + r), e = __ldg(rowptr + r + 1);
        float acc = 0.f;
        for (int j = s; j < e; ++j)
            acc = fmaf(__ldg(vals + j), __ldg(x + (int64_t)__ldg(colidx + j) * ncols + c), acc);
        float o = alpha * acc;
        if (z) o = fmaf(beta, z[idx], o);
        if (w) o += w[idx];
        y[idx] = o;
    }
}

// ---------------------------------------------------------------------------------------------
// Fused Chebyshev recurrence for the coarse levels.  The recurrence couples all vertices but is
// independent per (mesh, feature) column, so a CTA that owns a slab of CS4 column quads for ALL N
// vertices can run every step k = 1..K-1 out of shared memory (two N x slab buffers, T_k written
// in place over T_{k-2}) with a block barrier between steps instead of a kernel launch: one launch
// per layer instead of K-1, x read once, each T_k written once.  N <= ~3000 fits (levels 1-4 of the
// template: 1250 / 313 / 79 / 20 vertices).  The reverse recurrence of the backward pass
// (G_k = P_k + 2 L^T G_{k+1} - G_{k+2}) is fused the same way.  Summation order per row is the CSR
// order, as in the step-by-step kernels: results are bit-identical to them.
// ---------------------------------------------------------------------------------------------
// CSR entries as (column, value) pairs: one 8-byte shared (or global) load per neighbour instead of two
// 4-byte ones - the recurrence kernels are bound by shared-memory wavefronts (16 different rows per warp
// make every CSR read a 16-address access)
template <int CS4>
__device__ __forceinline__ float4 row_gather(const float4 *__restrict__ src, const int2 *ce, int s, int e, int cl) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = s;
    for (; j + 2 <= e; j += 2) {
        const int2 ea = ce[j], eb = ce[j + 1];
        const float4 xa = src[ea.x * CS4 + cl];
        const float4 xb = src[eb.x * CS4 + cl];
        fma4(acc, __int_as_float(ea.y), xa);
        fma4(acc, __int_as_float(eb.y), xb);
    }
    if (j < e) {
        const int2 ea = ce[j];
        fma4(acc, __int_as_float(ea.y), src[ea.x * CS4 + cl]);
    }
    return acc;
}

// copy the CSR of the level into shared memory (after the two activation buffers): row pointers and
// packed (column, value) entries.  The launcher guarantees that it fits.
__device__ __forceinline__ void stage_csr(int N, int nnz, const int32_t *__restrict__ rowptr,
                                          const int32_t *__restrict__ colidx, const float *__restrict__ vals,
                                          void *dst, const int32_t *&rp, const int2 *&ce) {
    int32_t *srp = reinterpret_cast<int32_t *>(dst);
    int2 *sce = reinterpret_cast<int2 *>(srp + ((N + 1 + 3) & ~3));
    g2s_copy<4>(srp, rowptr, N + 1, threadIdx.x, blockDim.x);
    for (int base = 0; base < nnz; base += 8 * blockDim.x) {
        int c[8];
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = base + u * blockDim.x + threadIdx.x;
            if (i < nnz) {
                c[u] = __ldg(colidx + i);
                v[u] = __ldg(vals + i);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = base + u * blockDim.x + threadIdx.x;
            if (i < nnz) sce[i] = make_int2(c[u], __float_as_int(v[u]));
        }
    }
    rp = srp;
    ce = sce;
}

template <int CS4>
__global__ void __launch_bounds__(1024)
cheb_recur_fwd_kernel(int N, int K, const int32_t *__restrict__ g_rowptr, const int32_t *__restrict__ g_colidx,
                      const float *__restrict__ g_vals, const float4 *__restrict__ x, float4 *__restrict__ basis,
                      int nc4, int nnz_smem) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ float4 sbuf[];
    float4 *cur = sbuf;                  // T_{k-1}
    float4 *old = sbuf + (size_t)N * CS4;  // T_{k-2}, overwritten by T_k
    const int32_t *rowptr;
    const int2 *ce;
    stage_csr(N, nnz_smem, g_rowptr, g_colidx, g_vals, sbuf + (size_t)2 * N * CS4, rowptr, ce);
    const int tid = threadIdx.x;
    const int cl = tid % CS4, rl = tid / CS4;
    const int RPP = blockDim.x / CS4;
    const int c = blockIdx.x * CS4 + cl;
    const bool col_ok = c < nc4;
    const int64_t plane = (int64_t)N * nc4;
    for (int r = rl; r < N; r += 8 * RPP) {        // 8 independent row loads in flight per thread
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int rr = r + u * RPP;
            v[u] = (col_ok && rr < N) ? __ldg(x + (int64_t)rr * nc4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int rr = r + u * RPP;
            if (rr < N) cur[rr * CS4 + cl] = v[u];
        }
    }
    __syncthreads();
    for (int k = 1; k < K; ++k) {
        float4 *outp = basis + (int64_t)(k - 1) * plane;
        for (int r = rl; r < N; r += RPP) {
            const int s = rowptr[r], e = rowptr[r + 1];
            const float4 acc = row_gather<CS4>(cur, ce, s, e, cl);
            float4 o;
            if (k == 1) {
                o = make_float4(1.f * acc.x, 1.f * acc.y, 1.f * acc.z, 1.f * acc.w);
            } else {
                const float4 zz = old[r * CS4 + cl];
                o.x = fmaf(-1.f, zz.x, 2.f * acc.x);
                o.y = fmaf(-1.f, zz.y, 2.f * acc.y);
                o.z = fmaf(-1.f, zz.z, 2.f * acc.z);
                o.w = fmaf(-1.f, zz.w, 2.f * acc.w);
            }
            old[r * CS4 + cl] = o;
            if (col_ok) outp[(int64_t)r * nc4 + c] = o;
        }
        __syncthreads();
        float4 *t = cur;
        cur = old;
        old = t;
    }
}

// P: K planes [N, nc4] (P_k = dY W_k^T); dx = P_0 + L^T G_1 - G_2 with G_{K-1} = P_{K-1},
// G_k = P_k + 2 L^T G_{k+1} - G_{k+2}.  CSR arguments are L^T.  Requires K >= 2.
template <int CS4>
__global__ void __launch_bounds__(1024)
cheb_recur_bwd_kernel(int N, int K, const int32_t *__restrict__ g_rowptr, const int32_t *__restrict__ g_colidx,
                      const float *__restrict__ g_vals, const float4 *__restrict__ P, float4 *__restrict__ dx,
                      int nc4, int nnz_smem) {
    extern __shared__ float4 sbuf[];
    float4 *g1 = sbuf;                   // G_{k+1}
    float4 *g2 = sbuf + (size_t)N * CS4;   // G_{k+2}, overwritten by G_k
    const int32_t *rowptr;
    const int2 *ce;
    stage_csr(N, nnz_smem, g_rowptr, g_colidx, g_vals, sbuf + (size_t)2 * N * CS4, rowptr, ce);
    const int tid = threadIdx.x;
    const int cl = tid % CS4, rl = tid / CS4;
    const int RPP = blockDim.x / CS4;
    const int c = blockIdx.x * CS4 + cl;
    const bool col_ok = c < nc4;
    const int64_t plane = (int64_t)N * nc4;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    {
        const float4 *pl = P + (int64_t)(K - 1) * plane;
        for (int r = rl; r < N; r += 8 * RPP) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int rr = r + u * RPP;
                v[u] = (col_ok && rr < N) ? __ldg(pl + (int64_t)rr * nc4 + c) : zero;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int rr = r + u * RPP;
                if (rr < N) g1[rr * CS4 + cl] = v[u];
            }
        }
    }
    __syncthreads();
    for (int k = K - 2; k >= 0; --k) {
        const float4 *pk = P + (int64_t)k * plane;
        const bool has_g2 = (k + 2 <= K - 1);
        const float alpha = (k == 0) ? 1.f : 2.f;
        float4 pvr[8];                                   // P_k of this thread's first 8 rows: all loads in flight at once
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int rr = rl + u * RPP;
            pvr[u] = (col_ok && rr < N) ? __ldg(pk + (int64_t)rr * nc4 + c) : zero;
        }
        int it = 0;
        for (int r = rl; r < N; r += RPP, ++it) {
            float4 pv;
            if (it < 8) {
                pv = zero;
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (u == it) pv = pvr[u];
            } else {
                pv = col_ok ? __ldg(pk + (int64_t)r * nc4 + c) : zero;
            }
            const int s = rowptr[r], e = rowptr[r + 1];
            const float4 acc = row_gather<CS4>(g1, ce, s, e, cl);
            float4 o = make_float4(alpha * acc.x, alpha * acc.y, alpha * acc.z, alpha * acc.w);
            if (has_g2) {
                const float4 zz = g2[r * CS4 + cl];
                o.x = fmaf(-1.f, zz.x, o.x);
                o.y = fmaf(-1.f, zz.y, o.y);
                o.z = fmaf(-1.f, zz.z, o.z);
                o.w = fmaf(-1.f, zz.w, o.w);
            }
            o.x += pv.x;
            o.y += pv.y;
            o.z += pv.z;
            o.w += pv.w;
            if (k == 0) {
                if (col_ok) dx[(int64_t)r * nc4 + c] = o;
            } else {
                g2[r * CS4 + cl] = o;
            }
        }
        __syncthreads();
        float4 *t = g1;
        g1 = g2;
        g2 = t;
    }
}

static int g_recur_fused = 1;
void set_recur_fused(int v) { g_recur_fused = v != 0; }
constexpr int RECUR_NT = 1024;         // threads per block of the fused recurrences

static bool recur_shape(int N, int nnz, int64_t ncols, const void *a, const void *b, int *cs4, size_t *smem, int *nnz_smem) {
    if (!g_recur_fused || N < 1 || ncols % 4 != 0 || !aligned16(a) || !aligned16(b)) return false;
    const int nc4 = (int)(ncols / 4);
    int c = 2;                                   // 32-byte rows: whole sectors, >= 2 CTAs per SM at level 1
    if (nc4 % 2 != 0) c = 1;
    size_t bytes = (size_t)2 * N * c * sizeof(float4);
    if (bytes > 200 * 1024 && c == 2) {
        c = 1;
        bytes = (size_t)2 * N * c * sizeof(float4);
    }
    if (bytes > 110 * 1024) return false;        // level 0 (4998 vertices) stays on the step-by-step kernels
    // one block per SM at most: beyond a single wave the L2-resident step-by-step launches win
    // (scripts/recur_ab.py: level 1, 256 meshes: 136 us stepwise vs 167 us fused; 64 meshes: 67 vs 54)
    if ((nc4 + c - 1) / c > num_sms()) return false;
    *cs4 = c;
    if (nnz < 0) return false;                   // the operator is staged in shared memory: its size must be known
    const size_t csr = ((size_t)((N + 1 + 3) & ~3) + 2 * (size_t)((nnz + 3) & ~3)) * 4;
    if (bytes + csr > 200 * 1024) return false;
    bytes += csr;
    *nnz_smem = nnz;
    *smem = bytes;
    return true;
}

// fused multi-step recurrences: 1 = handled, 0 = shape not supported (use the step kernels), < 0 = error
static int launch_cheb_recur_fwd(int N, int nnz, int K, const int32_t *rowptr, const int32_t *colidx, const float *vals,
                          const float *x, float *basis, int64_t ncols, cudaStream_t st) {
    int cs4, nnz_smem;
    size_t smem;
    if (K < 2 || !recur_shape(N, nnz, ncols, x, basis, &cs4, &smem, &nnz_smem)) return 0;
    const int nc4 = (int)(ncols / 4);
    const int grid = (nc4 + cs4 - 1) / cs4;
    static DevFlags optin1, optin2;
    cudaError_t e = cudaSuccess;
    if (cs4 == 2) {
        if (smem_optin(cheb_recur_fwd_kernel<2>, 200 * 1024, optin2, "cheb_recur_fwd_kernel")) e = cudaErrorInvalidValue;
        if (e == cudaSuccess)
            launch_pdl(cheb_recur_fwd_kernel<2>, dim3(grid), dim3(RECUR_NT), smem, st, N, K, rowptr, colidx, vals, (const float4 *)x, (float4 *)basis, nc4, nnz_smem);
    } else {
        if (smem_optin(cheb_recur_fwd_kernel<1>, 200 * 1024, optin1, "cheb_recur_fwd_kernel")) e = cudaErrorInvalidValue;
        if (e == cudaSuccess)
            launch_pdl(cheb_recur_fwd_kernel<1>, dim3(grid), dim3(RECUR_NT), smem, st, N, K, rowptr, colidx, vals, (const float4 *)x, (float4 *)basis, nc4, nnz_smem);
    }
    if (e != cudaSuccess) return set_err(MVB_ECUDA, "cheb_recur_fwd: %s", cudaGetErrorString(e));
    int rc = check_launch("mvb cheb_recur_fwd");
    return rc ? rc : 1;
}

static int launch_cheb_recur_bwd(int N, int nnz, int K, const int32_t *rowptr_t, const int32_t *colidx_t, const float *vals_t,
                          const float *P, float *dx, int64_t ncols, cudaStream_t st) {
    int cs4, nnz_smem;
    size_t smem;
    if (K < 2 || !recur_shape(N, nnz, ncols, P, dx, &cs4, &smem, &nnz_smem)) return 0;
    const int nc4 = (int)(ncols / 4);
    const int grid = (nc4 + cs4 - 1) / cs4;
    static DevFlags optin1, optin2;
    cudaError_t e = cudaSuccess;
    if (cs4 == 2) {
        if (smem_optin(cheb_recur_bwd_kernel<2>, 200 * 1024, optin2, "cheb_recur_bwd_kernel")) e = cudaErrorInvalidValue;
        if (e == cudaSuccess)
            cheb_recur_bwd_kernel<2><<<grid, RECUR_NT, smem, st>>>(N, K, rowptr_t, colidx_t, vals_t, (const float4 *)P, (float4 *)dx, nc4, nnz_smem);
    } else {
        if (smem_optin(cheb_recur_bwd_kernel<1>, 200 * 1024, optin1, "cheb_recur_bwd_kernel")) e = cudaErrorInvalidValue;
        if (e == cudaSuccess)
            cheb_recur_bwd_kernel<1><<<grid, RECUR_NT, smem, st>>>(N, K, rowptr_t, colidx_t, vals_t, (const float4 *)P, (float4 *)dx, nc4, nnz_smem);
    }
    if (e != cudaSuccess) return set_err(MVB_ECUDA, "cheb_recur_bwd: %s", cudaGetErrorString(e));
    int rc = check_launch("mvb cheb_recur_bwd");
    return rc ? rc : 1;
}

int launch_cheb_recurrence(int n, int nnz, int K, const int32_t *rowptr, const int32_t *colidx, const float *vals,
                           const float *t0, float *planes, int64_t ncols, cudaStream_t st) {
    if (K < 2) return MVB_OK;
    const int fused = launch_cheb_recur_fwd(n, nnz, K, rowptr, colidx, vals, t0, planes, ncols, st);
    if (fused) return fused < 0 ? fused : MVB_OK;
    const int64_t plane = (int64_t)n * ncols;
    for (int k = 1; k < K; ++k) {
        float *tk = planes + (int64_t)(k - 1) * plane;
        const float *tkm1 = (k == 1) ? t0 : planes + (int64_t)(k - 2) * plane;
        const float *tkm2 = (k == 1) ? nullptr : (k == 2 ? t0 : planes + (int64_t)(k - 3) * plane);
        const int rc = launch_spmm(n, n, rowptr, colidx, vals, tkm1, tk, tkm2, nullptr, k == 1 ? 1.f : 2.f, -1.f, ncols, st);
        if (rc) return rc;
    }
    return MVB_OK;
}

int launch_cheb_recurrence_bwd(int n, int nnz, int K, const int32_t *rowptr_t, const int32_t *colidx_t, const float *vals_t,
                               float *P, float *dx, int64_t ncols, cudaStream_t st, bool keep_planes) {
    const int64_t plane = (int64_t)n * ncols;
    if (K == 1) {
        if (!dx) return MVB_OK;
        const cudaError_t e = cudaMemcpyAsync(dx, P, (size_t)plane * sizeof(float), cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return set_err(MVB_ECUDA, "cheb_bwd: memcpy: %s", cudaGetErrorString(e));
        return MVB_OK;
    }
    if (!keep_planes) {
        const int fused = launch_cheb_recur_bwd(n, nnz, K, rowptr_t, colidx_t, vals_t, P, dx, ncols, st);
        if (fused) return fused < 0 ? fused : MVB_OK;
    }
    for (int k = K - 2; k >= (dx ? 0 : 1); --k) {
        float *pk = P + (int64_t)k * plane;
        const float *gk1 = P + (int64_t)(k + 1) * plane;
        const float *gk2 = (k + 2 <= K - 1) ? P + (int64_t)(k + 2) * plane : nullptr;
        float *dst = (k == 0) ? dx : pk;
        const int rc = launch_spmm(n, n, rowptr_t, colidx_t, vals_t, gk1, dst, gk2, pk, k == 0 ? 1.f : 2.f, -1.f, ncols, st);
        if (rc) return rc;
    }
    return MVB_OK;
}

int launch_spmm(int n_rows, int n_src_rows, const int32_t *rowptr, const int32_t *colidx, const float *vals,
                const float *x, float *y, const float *z, const float *w, float alpha, float beta,
                int64_t ncols, cudaStream_t st) {
    if (n_rows == 0 || ncols == 0) return MVB_OK;
    const bool vec = (ncols % 4 == 0) && aligned16(x) && aligned16(y) && (!z || aligned16(z)) &&
                     (!w || aligned16(w));
    const int threads = 256;
    // enough CTAs for every SM to hold its full complement of resident warps; grid-stride beyond
    const int64_t max_blocks = (int64_t)num_sms() * 8 * 4;
    if (vec) {
        const int nc4 = (int)(ncols / 4);
        const float4 *x4 = reinterpret_cast<const float4 *>(x);
        float4 *y4 = reinterpret_cast<float4 *>(y);
        const float4 *z4 = reinterpret_cast<const float4 *>(z);
        const float4 *w4 = reinterpret_cast<const float4 *>(w);
        // block = TX column quads x (threads / TX) rows; every block walks `chunk` CONSECUTIVE rows of its
        // 512-byte column slab (the operators are banded: L1 serves the repeated neighbour rows).
        // The grid is ONE WAVE: exactly as many blocks as the GPU holds at once, each with an equal share of
        // the rows.  The kernel is latency-bound, so a trailing partial wave costs as much as a full one:
        // at 64 meshes the 64-row chunks gave 632 blocks = 2.13 waves and 17.3 us, 296 blocks of 136 rows
        // give 14.7 us (0.54 -> 0.64 of the HBM peak; profiles/README.md).
        int tx = 32, chunk = 0, nthreads = 256;
        if (nc4 >= 32) {
            const int gx1 = (nc4 + tx - 1) / tx;
            for (nthreads = 1024; nthreads >= 256; nthreads >>= 1) {
                const int gy1 = num_sms() * (2048 / nthreads) / gx1;
                if (gy1 < 1) continue;
                chunk = (n_rows + gy1 - 1) / gy1;
                if (chunk >= 4 * (nthreads / tx) || nthreads == 256) break;     // >= 4 rows per warp, else smaller blocks
            }
            if (nthreads < 256) {            // more slabs than block slots (> 1184 slabs): several waves of 32-row chunks
                nthreads = 256;
                chunk = 0;
            }
        } else {                             // narrow planes: 256-thread blocks of at most 16 column quads, 32-row chunks
            tx = 16;
            while (tx > nc4 && tx > 1) tx >>= 1;
        }
        const dim3 block(tx, nthreads / tx);
        if (chunk <= 0) chunk = 32;
        if (chunk < (int)block.y) chunk = block.y;
        const int64_t gy = ((int64_t)n_rows + chunk - 1) / chunk;
        const int64_t gx = (nc4 + tx - 1) / tx;
        if (gy > 65535) return set_err(MVB_EINVAL, "spmm: too many row chunks");
        const dim3 grid((unsigned)gx, (unsigned)gy);
        const int64_t max_rows = n_rows > n_src_rows ? n_rows : n_src_rows;
        const bool idx32 = max_rows * nc4 < (1LL << 31);
#define MVB_SPMM_LAUNCH(HZ, HW)                                                                                         \
    do {                                                                                                                \
        if (idx32)                                                                                                      \
            launch_pdl(spmm_v4_kernel<HZ, HW, uint32_t>, grid, block, 0, st, n_rows, rowptr, colidx, vals, x4, y4, z4, w4, alpha, beta, nc4, chunk); \
        else                                                                                                            \
            launch_pdl(spmm_v4_kernel<HZ, HW, int64_t>, grid, block, 0, st, n_rows, rowptr, colidx, vals, x4, y4, z4, w4, alpha, beta, nc4, chunk);  \
    } while (0)
        if (z && w)
            MVB_SPMM_LAUNCH(true, true);
        else if (z)
            MVB_SPMM_LAUNCH(true, false);
        else if (w)
            MVB_SPMM_LAUNCH(false, true);
        else
            MVB_SPMM_LAUNCH(false, false);
#undef MVB_SPMM_LAUNCH
    } else {
        int64_t blocks = ((int64_t)n_rows * ncols + threads - 1) / threads;
        if (blocks > max_blocks) blocks = max_blocks;
        spmm_scalar_kernel<<<(unsigned)blocks, threads, 0, st>>>(n_rows, rowptr, colidx, vals, x, y, z, w, alpha, beta, ncols);
    }
    return check_launch("mvb_spmm");
}

}  // namespace mvb
