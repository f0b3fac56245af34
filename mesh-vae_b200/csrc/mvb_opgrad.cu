// Gradient of the Chebyshev convolution with respect to the values of its operator (the `norm` of
// ChebConv_batch.forward, nn/conv.py:557-581, when it is computed from learned edge weights).
//
// The pattern of L (CSR(L), CSR(L^T)) is built once on the host; the values change every step.  perm / perm_t map
// each CSR slot to its COO entry, so the values of both orientations are one gather from the COO tensor
// (mvb_csr_values), and the gradient is written straight back in COO order.
//
// With G^_k = dloss/dT_k (plane k of the basis-form backward's reverse recurrence, k >= 1):
//   d_coo[e] = <G^_1[r], T_0[c]> + 2 sum_{k=2}^{K-1} <G^_k[r], T_{k-1}[c]>     (r, c) = CSR(L) position of entry e
// a sampled dense-dense product: the rows gathered are the neighbours the SpMM gathers.
#include "mvb_internal.cuh"

namespace mvb {

__global__ void __launch_bounds__(256)
csr_values_kernel(int nnz, const int32_t *__restrict__ perm, const int32_t *__restrict__ perm_t,
                  const float *__restrict__ coo_vals, float *__restrict__ vals, float *__restrict__ vals_t) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += gridDim.x * blockDim.x) {
        vals[j] = __ldg(coo_vals + __ldg(perm + j));
        vals_t[j] = __ldg(coo_vals + __ldg(perm_t + j));
    }
}

int launch_csr_values(int nnz, const int32_t *perm, const int32_t *perm_t, const float *coo_vals, float *vals,
                      float *vals_t, cudaStream_t st) {
    if (nnz == 0) return MVB_OK;
    const int64_t blocks = ((int64_t)nnz + 255) / 256;
    const int grid = (int)(blocks < (int64_t)num_sms() * 8 ? blocks : (int64_t)num_sms() * 8);
    csr_values_kernel<<<grid, 256, 0, st>>>(nnz, perm, perm_t, coo_vals, vals, vals_t);
    return check_launch("mvb csr_values");
}

constexpr int EDGE_BATCH = 8;      // CSR entries of a row whose dot products one pass accumulates (mean degree ~6)

__device__ __forceinline__ float dot4(const float4 &a, const float4 &b, float acc) {
    acc = fmaf(a.x, b.x, acc);
    acc = fmaf(a.y, b.y, acc);
    acc = fmaf(a.z, b.z, acc);
    return fmaf(a.w, b.w, acc);
}

// One warp owns one CSR(L) row r.  For a batch of up to EDGE_BATCH entries it walks k = 1..K-1 in ascending order and
// the ncols columns of a vertex row in 32-lane chunks (16-byte loads when VEC): the G^_k[r] chunk is loaded once and
// dotted with the gathered T_{k-1}[c] chunk of every entry.  The per-lane sums are reduced by a fixed xor butterfly and
// each entry's value is stored once, at its COO position: no atomics, the same bits on every run.
template <bool VEC>
__global__ void __launch_bounds__(256)
cheb_edge_grad_kernel(int n_rows, int64_t ncols, int K, const int32_t *__restrict__ rowptr,
                      const int32_t *__restrict__ colidx, const int32_t *__restrict__ perm, const float *__restrict__ x,
                      const float *__restrict__ basis, const float *__restrict__ G, float *__restrict__ d_coo) {
    const int r = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= n_rows) return;
    const int s = __ldg(rowptr + r), e = __ldg(rowptr + r + 1);
    const int64_t plane = (int64_t)n_rows * ncols;
    for (int j0 = s; j0 < e; j0 += EDGE_BATCH) {
        const int cnt = min(EDGE_BATCH, e - j0);
        int col[EDGE_BATCH];
        float acc[EDGE_BATCH];
#pragma unroll
        for (int u = 0; u < EDGE_BATCH; ++u) {
            col[u] = __ldg(colidx + j0 + (u < cnt ? u : 0));
            acc[u] = 0.f;
        }
        for (int k = 1; k < K; ++k) {
            const float *g = G + (int64_t)k * plane + (int64_t)r * ncols;
            const float *t = (k == 1) ? x : basis + (int64_t)(k - 2) * plane;
            const float coef = (k == 1) ? 1.f : 2.f;
            if (VEC) {
                const int64_t nc4 = ncols >> 2;
                const float4 *g4 = reinterpret_cast<const float4 *>(g);
                for (int64_t q = lane; q < nc4; q += 32) {
                    float4 gv = __ldg(g4 + q);
                    gv = make_float4(coef * gv.x, coef * gv.y, coef * gv.z, coef * gv.w);
#pragma unroll
                    for (int u = 0; u < EDGE_BATCH; ++u)
                        if (u < cnt) acc[u] = dot4(gv, __ldg(reinterpret_cast<const float4 *>(t + (int64_t)col[u] * ncols) + q), acc[u]);
                }
            } else {
#pragma unroll 1
                for (int64_t q = lane; q < ncols; q += 32) {
                    const float gv = coef * __ldg(g + q);
#pragma unroll
                    for (int u = 0; u < EDGE_BATCH; ++u)
                        if (u < cnt) acc[u] = fmaf(gv, __ldg(t + (int64_t)col[u] * ncols + q), acc[u]);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < EDGE_BATCH; ++u) {
            float v = acc[u];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == u && u < cnt) d_coo[__ldg(perm + j0 + u)] = v;
        }
    }
}

int launch_cheb_edge_grad(int n_rows, int64_t ncols, int K, const int32_t *rowptr, const int32_t *colidx,
                          const int32_t *perm, const float *x, const float *basis, const float *G, float *d_coo,
                          cudaStream_t st) {
    if (n_rows == 0) return MVB_OK;
    const int64_t blocks = ((int64_t)n_rows * 32 + 255) / 256;
    const bool vec = ncols % 4 == 0 && aligned16(x) && aligned16(G) && (K <= 2 || aligned16(basis));
    if (vec)
        cheb_edge_grad_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(n_rows, ncols, K, rowptr, colidx, perm, x, basis, G, d_coo);
    else
        cheb_edge_grad_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(n_rows, ncols, K, rowptr, colidx, perm, x, basis, G, d_coo);
    return check_launch("mvb cheb_edge_grad");
}

}  // namespace mvb

using namespace mvb;

extern "C" int mvb_csr_values(int nnz, const int32_t *perm, const int32_t *perm_t, const float *coo_vals, float *vals,
                              float *vals_t, void *stream) {
    MVB_REQUIRE(nnz >= 0, "csr_values: nnz=%d < 0", nnz);
    MVB_REQUIRE(nnz == 0 || (perm && perm_t && coo_vals && vals && vals_t), "csr_values: null pointer");
    return launch_csr_values(nnz, perm, perm_t, coo_vals, vals, vals_t, (cudaStream_t)stream);
}
