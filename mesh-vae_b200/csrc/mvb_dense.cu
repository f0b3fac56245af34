// The dense bottleneck of cheb_VAE between the two mesh pyramids (SURVEY.md 8(f) row f2):
//   enc_lin -> ReLU -> dropout                                  models/cheb_VAE.py:270-272
//   dropout -> classifier_layer -> softmax                      models/cheb_VAE.py:253-258
//   cat(y, h) -> z_mean / z_log_var -> reparameterize -> cat    models/cheb_VAE.py:206-221, 309-319
//   dec_lin -> ReLU -> dropout -> dec_lin_2 -> ReLU -> dropout  models/cheb_VAE.py:276-281
// In the reference these are ~60 tiny ATen / cuBLAS launches per training step (GEMMs with M = the
// mesh batch, bias adds, clamps, dropouts, cats, softmax and their backward): latency, not work.
// Here: one launch per Linear (bias + ReLU + dropout in the epilogue, input / output read or written
// directly in the vertex-major layout of the neighbouring pool), one launch for all three heads, and
// one launch per backward (dW, db and dx together).  Strict fp32 FFMA, fixed summation order (k
// ascending), no atomics: deterministic.  Dropout masks come from a counter-based generator
// (Philox4x32-10) keyed by (seed, step offset, element), so the backward pass regenerates them
// instead of storing them and a captured CUDA graph draws fresh masks on every replay (the offset
// is read from device memory).
#include "mvb_internal.cuh"

namespace mvb {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += W0;
        k.y += W1;
    }
    return c;
}

// Bernoulli(1 - p) keep decision of logical element `idx` for (seed, offset)
__device__ __forceinline__ bool drop_keep(uint64_t seed, uint64_t offset, uint32_t idx, float p) {
    const uint4 r = philox4x32_10(make_uint4(idx >> 2, 0u, (uint32_t)offset, (uint32_t)(offset >> 32)),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t l = idx & 3u;
    const uint32_t v = l == 0 ? r.x : (l == 1 ? r.y : (l == 2 ? r.z : r.w));
    return (float)(v >> 8) * (1.f / 16777216.f) >= p;
}

// element (m, k) of a logical [M, K] matrix: row-major (vmf == 0) or vertex-major [K/vmf, M, vmf]
__device__ __forceinline__ int64_t lin_index(int m, int k, int M, int K, int vmf) {
    return vmf ? ((int64_t)(k / vmf) * M + m) * vmf + (k % vmf) : (int64_t)m * K + k;
}

__device__ __forceinline__ float gp_value(float gy, float yv, int relu, float scale) {
    return relu ? (yv > 0.f ? gy * scale : 0.f) : gy * scale;
}

// Staging uses cp.async (mvb_internal.cuh): the first version of these kernels (register staging, 3
// integer divisions per element) spent 80 us in enc_lin's forward, 95 % of it address arithmetic and
// serialised latencies (profiles/README.md).

// A logical [R, C] matrix in global memory: element (r, c) at base + r*rs + (c / f)*cso + c % f.
// Row-major [R, C]: rs = C, f = INT_MAX.  Vertex-major [C/f, R, f]: rs = f, cso = R*f.
struct MatView {
    const float *base;
    int64_t rs, cso;
    int f;
};
__device__ __forceinline__ MatView mat_view(const float *p, int R, int C, int vmf) {
    MatView v;
    v.base = p;
    if (vmf) { v.rs = vmf; v.cso = (int64_t)R * vmf; v.f = vmf; }
    else { v.rs = C; v.cso = 0; v.f = 0x7fffffff; }
    return v;
}
__device__ __forceinline__ int64_t mat_off(const MatView &v, int r, int c) { return (int64_t)r * v.rs + (int64_t)(c / v.f) * v.cso + (c % v.f); }

// stage the tile rows [r0, r0 + tile_rows) x columns [c0, c0 + tile_cols) of `v` into dst[tile_rows][ld];
// rows >= valid_rows / columns >= valid_cols (tile-relative) are zero-filled.  tile_cols % VEC == 0 and, for
// VEC == 4, valid_cols % 4 == 0.  Wide tiles: a warp walks a row (column offsets computed once per
// thread); narrow tiles: flattened index.
template <int VEC>
__device__ __forceinline__ void stage_async(float *dst, int ld, int tile_rows, int valid_rows, int tile_cols, int valid_cols,
                                            const MatView &v, int r0, int c0, int tid, int nthreads) {
    const int ncg = tile_cols / VEC;
    if (ncg >= 32) {
        const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
        for (int cg = lane; cg < ncg; cg += 32) {
            const int c = cg * VEC;
            const bool cv = c < valid_cols;
            const int64_t coff = cv ? (int64_t)((c0 + c) / v.f) * v.cso + ((c0 + c) % v.f) : 0;
            for (int r = warp; r < tile_rows; r += nwarps) {
                const bool ok = cv && r < valid_rows;
                cp_async<VEC>(dst + r * ld + c, ok ? v.base + (int64_t)(r0 + r) * v.rs + coff : v.base, ok);
            }
        }
    } else if ((ncg & (ncg - 1)) == 0 && v.f == 0x7fffffff) {       // narrow row-major tile, power-of-two groups: no divisions
        const int lg = 31 - __clz(ncg);
        for (int i = tid; i < tile_rows * ncg; i += nthreads) {
            const int r = i >> lg, c = (i & (ncg - 1)) * VEC;
            const bool ok = r < valid_rows && c < valid_cols;
            cp_async<VEC>(dst + r * ld + c, ok ? v.base + (int64_t)(r0 + r) * v.rs + c0 + c : v.base, ok);
        }
    } else {
        for (int i = tid; i < tile_rows * ncg; i += nthreads) {
            const int r = i / ncg, c = (i - r * ncg) * VEC;
            const bool ok = r < valid_rows && c < valid_cols;
            cp_async<VEC>(dst + r * ld + c, ok ? v.base + mat_off(v, r0 + r, c0 + c) : v.base, ok);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// forward: y = dropout(relu(x W^T + b)).  Block tile 64 rows x 8 outputs, the whole K extent (in
// chunks of KC <= 640) staged in shared memory.
// ---------------------------------------------------------------------------------------------
// (32 rows per block: at 64 meshes the grid is 2 x N/8 = 128-160 blocks on 148 SMs and a block stages half the
// activation tile - the staging of x, not the arithmetic, is what a block's time goes into)
constexpr int LF_TM = 32, LF_TN = 8, LF_RPT = LF_TM / 32;      // rows per thread: 256 threads = 8 outputs x 32 row groups

template <int VEC>
__global__ void __launch_bounds__(256)
linear_fwd_kernel(int M, int K, int N, const float *__restrict__ x, int x_vmf, const float *__restrict__ W,
                  const float *__restrict__ bias, int relu, float p, uint64_t seed, const int64_t *off_dev,
                  int64_t off_host, float *__restrict__ y, int y_vmf, int KC) {
    pdl_trigger();
    extern __shared__ float4 dsm4[];
    float *xs = reinterpret_cast<float *>(dsm4);     // [LF_TM][LD]
    const int LD = KC + 4;
    float *ws = xs + LF_TM * LD;                      // [LF_TN][LD]
    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * LF_TM, n0 = blockIdx.x * LF_TN;
    const int rows = min(LF_TM, M - m0), cols = min(LF_TN, N - n0);
    const int n = tid % LF_TN, r0 = (tid / LF_TN) * LF_RPT;
    const MatView xv = mat_view(x, M, K, x_vmf), wv = mat_view(W, N, K, 0);
    float acc0 = 0.f, acc1 = 0.f;
    for (int k0 = 0; k0 < K; k0 += KC) {
        const int kc = min(KC, K - k0);
        const int kc4 = (kc + 3) & ~3;
        if (k0) __syncthreads();
        stage_async<VEC>(ws, LD, LF_TN, cols, kc4, kc, wv, n0, k0, tid, 256);
        if (k0 == 0) pdl_wait();          // the first weight tile is in flight before the previous kernel has finished; x is its output
        stage_async<VEC>(xs, LD, LF_TM, rows, kc4, kc, xv, m0, k0, tid, 256);
        cp_async_wait_all();
        __syncthreads();
        const float4 *w4 = reinterpret_cast<const float4 *>(ws + n * LD);
        const float4 *a4 = reinterpret_cast<const float4 *>(xs + r0 * LD);
        const float4 *b4 = reinterpret_cast<const float4 *>(xs + (r0 + LF_RPT - 1) * LD);
#pragma unroll 4
        for (int k = 0; k < (kc4 >> 2); ++k) {
            const float4 w = w4[k], a = a4[k];
            acc0 = fmaf(a.x, w.x, acc0); acc0 = fmaf(a.y, w.y, acc0); acc0 = fmaf(a.z, w.z, acc0); acc0 = fmaf(a.w, w.w, acc0);
            if (LF_RPT == 2) {
                const float4 b = b4[k];
                acc1 = fmaf(b.x, w.x, acc1); acc1 = fmaf(b.y, w.y, acc1); acc1 = fmaf(b.z, w.z, acc1); acc1 = fmaf(b.w, w.w, acc1);
            }
        }
    }
    if (n >= cols) return;
    const float bv = bias ? __ldg(bias + n0 + n) : 0.f;
    const uint64_t off = (uint64_t)(off_host + (off_dev ? *off_dev : 0));
    const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
#pragma unroll
    for (int u = 0; u < LF_RPT; ++u) {
        const int r = r0 + u;
        if (r >= rows) break;
        float v = (u ? acc1 : acc0) + bv;
        if (relu) v = fmaxf(v, 0.f);
        if (p > 0.f) v = drop_keep(seed, off, (uint32_t)((m0 + r) * N + n0 + n), p) ? v * scale : 0.f;
        y[lin_index(m0 + r, n0 + n, M, N, y_vmf)] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// backward: gp = gy * [y > 0] / (1 - p)  (ReLU + dropout: a dropped or clamped unit has y == 0),
//   dW[N,K] = gp^T x, db[N] = 1^T gp, dx[M,K] = gp W.   One launch, two block roles:
//   role A (blockIdx < nA): a 64 x 64 tile of dW (and db when it owns k-tile 0), m reduced in order;
//   role B: a 32-row x 16-column tile of dx, n reduced in order (chunks of nc_b <= 640).
// gy and y tiles are staged raw with cp.async and combined in shared memory.
// ---------------------------------------------------------------------------------------------
constexpr int BW_TN = 64, BW_TK = 64, BW_LA = 68, BW_TMB = 32, BW_TKX = 16;

template <int VN, int VK>      // cp.async width of the N-indexed arrays (gy, y) and of the K-indexed ones (x, W)
__global__ void __launch_bounds__(256)
linear_bwd_kernel(int M, int K, int N, const float *__restrict__ x, int x_vmf, const float *__restrict__ W,
                  const float *__restrict__ y, const float *__restrict__ gy, int y_vmf, int relu, float scale,
                  float *__restrict__ dx, float *__restrict__ dW, float *__restrict__ db, int nA, int k_tiles, int nc_b) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ float4 dsm4[];
    float *sm = reinterpret_cast<float *>(dsm4);
    const int tid = threadIdx.x;
    const MatView xv = mat_view(x, M, K, x_vmf), gv = mat_view(gy, M, N, y_vmf), yv = mat_view(y, M, N, y_vmf);
    if ((int)blockIdx.x < nA) {
        // ---- role A: dW tile ----
        const int nt = blockIdx.x / k_tiles, kt = blockIdx.x - nt * k_tiles;
        const int n0 = nt * BW_TN, k0 = kt * BW_TK;
        const int ncols = min(BW_TN, N - n0), kcols = min(BW_TK, K - k0);
        float *gps = sm;                          // [64][BW_LA]  gy, then gp
        float *ys = sm + 64 * BW_LA;              // [64][BW_LA]
        float *xs = sm + 2 * 64 * BW_LA;          // [64][BW_LA]
        const int nq = tid / 16, kq = tid % 16;   // outputs n = 4 nq.., k = 4 kq..
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        float dbacc = 0.f;
        for (int m0 = 0; m0 < M; m0 += 64) {
            const int rows = min(64, M - m0);
            if (m0) __syncthreads();
            stage_async<VN>(gps, BW_LA, 64, rows, BW_TN, ncols, gv, m0, n0, tid, 256);
            if (relu) stage_async<VN>(ys, BW_LA, 64, rows, BW_TN, ncols, yv, m0, n0, tid, 256);
            stage_async<VK>(xs, BW_LA, 64, rows, BW_TK, kcols, xv, m0, k0, tid, 256);
            cp_async_wait_all();
            __syncthreads();
            for (int i = tid; i < 64 * BW_TN; i += 256) {
                const int r = i / BW_TN, c = i % BW_TN;            // BW_TN is a compile-time power of two
                gps[r * BW_LA + c] = gp_value(gps[r * BW_LA + c], relu ? ys[r * BW_LA + c] : 1.f, relu, scale);
            }
            __syncthreads();
            for (int m = 0; m < rows; ++m) {
                const float4 g = *reinterpret_cast<const float4 *>(gps + m * BW_LA + 4 * nq);
                const float4 xx = *reinterpret_cast<const float4 *>(xs + m * BW_LA + 4 * kq);
                const float gg[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    acc[i][0] = fmaf(gg[i], xx.x, acc[i][0]); acc[i][1] = fmaf(gg[i], xx.y, acc[i][1]);
                    acc[i][2] = fmaf(gg[i], xx.z, acc[i][2]); acc[i][3] = fmaf(gg[i], xx.w, acc[i][3]);
                }
            }
            if (db && kt == 0 && tid < BW_TN)
                for (int m = 0; m < rows; ++m) dbacc += gps[m * BW_LA + tid];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int nn = n0 + 4 * nq + i;
            if (nn < N)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int k = k0 + 4 * kq + j;
                    if (k < K) dW[(int64_t)nn * K + k] = acc[i][j];
                }
        }
        if (db && kt == 0 && tid < BW_TN && n0 + tid < N) db[n0 + tid] = dbacc;
        return;
    }
    // ---- role B: dx tile ----
    const int bi = blockIdx.x - nA;
    const int kxt = (K + BW_TKX - 1) / BW_TKX;
    const int mt = bi / kxt, kt = bi - mt * kxt;
    const int m0 = mt * BW_TMB, k0 = kt * BW_TKX;
    const int rows = min(BW_TMB, M - m0);
    const int kcols = min(BW_TKX, K - k0);
    const int LG = nc_b + 4;
    float *gps = sm;                              // [32][LG]
    float *ys = sm + BW_TMB * LG;                 // [32][LG]
    float *wt = sm + 2 * BW_TMB * LG;             // [nc_b][BW_TKX]
    const MatView wv = mat_view(W, N, K, 0);
    const int m = tid / 8, kp = tid % 8;          // outputs (m, k = 2 kp, 2 kp + 1)
    float acc0 = 0.f, acc1 = 0.f;
    for (int nc0 = 0; nc0 < N; nc0 += nc_b) {
        const int nc = min(nc_b, N - nc0);
        const int nc4 = (nc + 3) & ~3;
        if (nc0) __syncthreads();
        stage_async<VN>(gps, LG, BW_TMB, rows, nc4, nc, gv, m0, nc0, tid, 256);
        if (relu) stage_async<VN>(ys, LG, BW_TMB, rows, nc4, nc, yv, m0, nc0, tid, 256);
        stage_async<VK>(wt, BW_TKX, nc4, nc, BW_TKX, kcols, wv, nc0, k0, tid, 256);
        cp_async_wait_all();
        __syncthreads();
        for (int r = tid >> 5; r < BW_TMB; r += 8)                  // a warp per row: no divisions
            for (int c = (tid & 31) * 4; c < nc4; c += 128) {
                float4 g = *reinterpret_cast<float4 *>(gps + r * LG + c);
                if (relu) {
                    const float4 yy = *reinterpret_cast<const float4 *>(ys + r * LG + c);
                    g.x = gp_value(g.x, yy.x, 1, scale); g.y = gp_value(g.y, yy.y, 1, scale);
                    g.z = gp_value(g.z, yy.z, 1, scale); g.w = gp_value(g.w, yy.w, 1, scale);
                } else {
                    g.x *= scale; g.y *= scale; g.z *= scale; g.w *= scale;
                }
                *reinterpret_cast<float4 *>(gps + r * LG + c) = g;
            }
        __syncthreads();
        const float4 *g4 = reinterpret_cast<const float4 *>(gps + m * LG);
        for (int q = 0; q < (nc4 >> 2); ++q) {
            const float4 g = g4[q];
            const float2 w0 = *reinterpret_cast<const float2 *>(wt + (4 * q + 0) * BW_TKX + 2 * kp);
            const float2 w1 = *reinterpret_cast<const float2 *>(wt + (4 * q + 1) * BW_TKX + 2 * kp);
            const float2 w2 = *reinterpret_cast<const float2 *>(wt + (4 * q + 2) * BW_TKX + 2 * kp);
            const float2 w3 = *reinterpret_cast<const float2 *>(wt + (4 * q + 3) * BW_TKX + 2 * kp);
            acc0 = fmaf(g.x, w0.x, acc0); acc1 = fmaf(g.x, w0.y, acc1);
            acc0 = fmaf(g.y, w1.x, acc0); acc1 = fmaf(g.y, w1.y, acc1);
            acc0 = fmaf(g.z, w2.x, acc0); acc1 = fmaf(g.z, w2.y, acc1);
            acc0 = fmaf(g.w, w3.x, acc0); acc1 = fmaf(g.w, w3.y, acc1);
        }
    }
    if (m < rows) {
        const int k = k0 + 2 * kp;
        if (k < K) dx[lin_index(m0 + m, k, M, K, x_vmf)] = acc0;
        if (k + 1 < K) dx[lin_index(m0 + m, k + 1, M, K, x_vmf)] = acc1;
    }
}

// ---------------------------------------------------------------------------------------------
// the three heads on h [B,H]:  y_hat = softmax(dropout(h) Wc^T + bc);  [mu | logvar] =
// cat(y, h) [Wm | Wv]^T + [bm | bv];  z_ = mu + eps * exp(logvar / 2) (or mu when eps == NULL);
// zcat = cat(y, z_).   One block per mesh; the C + 2Z weight rows are staged in shared memory with
// cp.async (one exposed latency), then a warp per output (dot product of length C + H).
// ---------------------------------------------------------------------------------------------
constexpr int HEADS_MAX_OUT = 96;     // C + 2 Z

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// stage the rows of the three weight matrices as one [C + 2Z][ldw] table: row o < C is Wc[o] at
// columns [C, C + H) (columns [0, C) zero), rows >= C are Wm / Wv rows (C + H columns)
__device__ __forceinline__ void stage_head_weights(float *wsm, int ldw, int H, int Z, int C, const float *Wc,
                                                   const float *Wm, const float *Wv, int tid, int nthreads) {
    const int nout = C + 2 * Z, W_ = C + H;
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
    for (int o = warp; o < nout; o += nwarps) {
        const float *src = o < C ? Wc + (int64_t)o * H - C : (o - C < Z ? Wm + (int64_t)(o - C) * W_ : Wv + (int64_t)(o - C - Z) * W_);
        for (int j = lane; j < W_; j += 32) {
            const bool ok = !(o < C && j < C);
            cp_async<1>(wsm + o * ldw + j, ok ? src + j : Wm, ok);
        }
    }
}

__global__ void __launch_bounds__(256)
vae_heads_fwd_kernel(int B, int H, int Z, int C, const float *__restrict__ h, const int64_t *__restrict__ yoh,
                     const float *__restrict__ eps, const float *__restrict__ Wc, const float *__restrict__ bc,
                     const float *__restrict__ Wm, const float *__restrict__ bm, const float *__restrict__ Wv,
                     const float *__restrict__ bv, float p, uint64_t seed, const int64_t *off_dev, int64_t off_host,
                     float *__restrict__ y_hat, float *__restrict__ mu, float *__restrict__ logvar,
                     float *__restrict__ z_, float *__restrict__ zcat) {
    pdl_trigger();
    extern __shared__ float4 dsm4[];
    const int ldw = C + H + 1;
    float *hs = reinterpret_cast<float *>(dsm4);   // [C + H]   cat(y, h) row
    float *hd = hs + (C + H);                      // [C + H]   (0, dropout(h)) row (classifier input)
    float *wsm = hd + (C + H);                     // [C + 2Z][ldw]
    __shared__ float outs[HEADS_MAX_OUT];
    const int b = blockIdx.x, tid = threadIdx.x;
    stage_head_weights(wsm, ldw, H, Z, C, Wc, Wm, Wv, tid, blockDim.x);      // weights: in flight before the previous kernel has finished
    pdl_wait();
    const uint64_t off = (uint64_t)(off_host + (off_dev ? *off_dev : 0));
    const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
    for (int j = tid; j < C + H; j += blockDim.x) {
        if (j < C) {
            hs[j] = (float)yoh[(int64_t)b * C + j];
            hd[j] = 0.f;
        } else {
            const float v = __ldg(h + (int64_t)b * H + j - C);
            hs[j] = v;
            hd[j] = (p > 0.f) ? (drop_keep(seed, off, (uint32_t)(b * H + j - C), p) ? v * scale : 0.f) : v;
        }
    }
    cp_async_wait_all();
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
    const int nout = C + 2 * Z;
    for (int o = warp; o < nout; o += nwarps) {
        const float *in = o < C ? hd : hs;
        const float *w = wsm + o * ldw;
        float s = 0.f;
        for (int j = lane; j < C + H; j += 32) s = fmaf(in[j], w[j], s);
        s = warp_sum(s);
        if (lane == 0) outs[o] = s + (o < C ? __ldg(bc + o) : (o - C < Z ? __ldg(bm + o - C) : __ldg(bv + o - C - Z)));
    }
    __syncthreads();
    if (tid == 0) {          // softmax over C classes (C is 2 in the reference)
        float mx = outs[0];
        for (int c = 1; c < C; ++c) mx = fmaxf(mx, outs[c]);
        float den = 0.f;
        for (int c = 0; c < C; ++c) den += expf(outs[c] - mx);
        for (int c = 0; c < C; ++c) y_hat[(int64_t)b * C + c] = expf(outs[c] - mx) / den;
    }
    if (tid < Z) {
        const float m = outs[C + tid], lv = outs[C + Z + tid];
        mu[(int64_t)b * Z + tid] = m;
        logvar[(int64_t)b * Z + tid] = lv;
        const float zz = eps ? fmaf(__ldg(eps + (int64_t)b * Z + tid), expf(0.5f * lv), m) : m;
        z_[(int64_t)b * Z + tid] = zz;
        zcat[(int64_t)b * (C + Z) + C + tid] = zz;
    }
    if (tid >= 32 && tid < 32 + C) zcat[(int64_t)b * (C + Z) + tid - 32] = (float)yoh[(int64_t)b * C + tid - 32];
}

// gradient of the C + 2Z pre-activations of mesh b from the upstream gradients
//   gs[0..C)      = softmax backward of g_yhat
//   gs[C..C+Z)    = g_mu + g_z                       (z_ = mu + eps * std)
//   gs[C+Z..C+2Z) = g_logvar + g_z * eps * std / 2
__device__ __forceinline__ float heads_small_grad(int o, int b, int Z, int C, const float *y_hat, const float *logvar,
                                                  const float *eps, const float *g_yhat, const float *g_mu,
                                                  const float *g_logvar, const float *g_z, const float *g_zcat) {
    if (o < C) {
        float dot = 0.f;
        if (!g_yhat) return 0.f;
        for (int c = 0; c < C; ++c) dot = fmaf(g_yhat[(int64_t)b * C + c], y_hat[(int64_t)b * C + c], dot);
        return y_hat[(int64_t)b * C + o] * (g_yhat[(int64_t)b * C + o] - dot);
    }
    const int i = (o - C) % Z;
    float gz = 0.f;
    if (g_z) gz += g_z[(int64_t)b * Z + i];
    if (g_zcat) gz += g_zcat[(int64_t)b * (C + Z) + C + i];
    if (o - C < Z) return (g_mu ? g_mu[(int64_t)b * Z + i] : 0.f) + gz;
    float g = g_logvar ? g_logvar[(int64_t)b * Z + i] : 0.f;
    if (eps) g = fmaf(gz * eps[(int64_t)b * Z + i], 0.5f * expf(0.5f * logvar[(int64_t)b * Z + i]), g);
    return g;
}

// The small per-mesh inputs of the heads' backward pass (upstream gradients, y_hat, logvar, eps) for rows
// [rb0, rb0 + nr) staged in shared memory with cp.async, so that heads_small_grad reads shared memory
// instead of chasing ~6 dependent global loads per element.
struct SmallIn {
    const float *y_hat, *logvar, *eps, *g_yhat, *g_mu, *g_logvar, *g_z, *g_zcat;
};
__device__ __forceinline__ const float *stage_small(float *&cursor, const float *src, int64_t first, int n, int tid, int nthreads) {
    if (!src) return nullptr;
    float *dst = cursor;
    cursor += (n + 3) & ~3;
    cp_async_words(dst, src + first, n, tid, nthreads);
    return dst;
}
__device__ __forceinline__ SmallIn stage_small_inputs(float *buf, int rb0, int nr, int Z, int C, const SmallIn &g, int tid, int nthreads) {
    SmallIn s;
    float *cur = buf;
    s.y_hat = stage_small(cur, g.y_hat, (int64_t)rb0 * C, nr * C, tid, nthreads);
    s.logvar = stage_small(cur, g.logvar, (int64_t)rb0 * Z, nr * Z, tid, nthreads);
    s.eps = stage_small(cur, g.eps, (int64_t)rb0 * Z, nr * Z, tid, nthreads);
    s.g_yhat = stage_small(cur, g.g_yhat, (int64_t)rb0 * C, nr * C, tid, nthreads);
    s.g_mu = stage_small(cur, g.g_mu, (int64_t)rb0 * Z, nr * Z, tid, nthreads);
    s.g_logvar = stage_small(cur, g.g_logvar, (int64_t)rb0 * Z, nr * Z, tid, nthreads);
    s.g_z = stage_small(cur, g.g_z, (int64_t)rb0 * Z, nr * Z, tid, nthreads);
    s.g_zcat = stage_small(cur, g.g_zcat, (int64_t)rb0 * (C + Z), nr * (C + Z), tid, nthreads);
    return s;
}
__host__ __device__ inline int small_in_words(int nr, int Z, int C) { return nr * (2 * C + 5 * Z + (C + Z)) + 32; }

// blocks [0, nbg): g_h of HB_ROWS meshes each (weights staged once per block).  blocks [nbg, nbg + ntile):
// a 32-column tile of the three weight gradients (column C + H is the bias), batch reduced in order.
constexpr int HB_ROWS = 2, HB_MAXO = 12;     // HB_MAXO = ceil(HEADS_MAX_OUT / 8)

__global__ void __launch_bounds__(256)
vae_heads_bwd_kernel(int B, int H, int Z, int C, const float *__restrict__ h, const int64_t *__restrict__ yoh,
                     const float *__restrict__ Wc, const float *__restrict__ Wm, const float *__restrict__ Wv, SmallIn gin,
                     float p, uint64_t seed, const int64_t *off_dev, int64_t off_host, float *__restrict__ g_h,
                     float *__restrict__ dWc, float *__restrict__ dbc, float *__restrict__ dWm, float *__restrict__ dbm,
                     float *__restrict__ dWv, float *__restrict__ dbv, int nbg) {
    pdl_trigger();
    extern __shared__ float4 dsm4[];
    float *sm = reinterpret_cast<float *>(dsm4);
    const int tid = threadIdx.x;
    const int nout = C + 2 * Z;
    const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
    if ((int)blockIdx.x < nbg) {
        const int ldw = C + H + 1;
        float *wsm = sm;                               // [nout][ldw]
        float *gs = sm + nout * ldw;                   // [HB_ROWS][nout]
        float *small = gs + ((HB_ROWS * nout + 3) & ~3);
        const int b0 = blockIdx.x * HB_ROWS;
        const int nr = min(HB_ROWS, B - b0);
        stage_head_weights(wsm, ldw, H, Z, C, Wc, Wm, Wv, tid, blockDim.x);      // weights: in flight before the previous kernel has finished
        pdl_wait();
        const uint64_t off = (uint64_t)(off_host + (off_dev ? *off_dev : 0));
        const SmallIn si = stage_small_inputs(small, b0, nr, Z, C, gin, tid, blockDim.x);
        cp_async_wait_all();
        __syncthreads();
        for (int i = tid; i < HB_ROWS * nout; i += blockDim.x) {
            const int bl = i / nout;
            gs[i] = bl < nr ? heads_small_grad(i % nout, bl, Z, C, si.y_hat, si.logvar, si.eps, si.g_yhat, si.g_mu, si.g_logvar, si.g_z, si.g_zcat) : 0.f;
        }
        __syncthreads();
        for (int i = tid; i < HB_ROWS * H; i += blockDim.x) {
            const int bl = i / H, j = i - bl * H;
            const int b = b0 + bl;
            if (b >= B) break;
            const float *g = gs + bl * nout;
            float a = 0.f;
            for (int c = 0; c < C; ++c) a = fmaf(g[c], wsm[c * ldw + C + j], a);
            if (p > 0.f) a = drop_keep(seed, off, (uint32_t)(b * H + j), p) ? a * scale : 0.f;
            for (int o = C; o < nout; ++o) a = fmaf(g[o], wsm[o * ldw + C + j], a);
            g_h[(int64_t)b * H + j] = a;
        }
        return;
    }
    // ---- weight gradients ----
    pdl_wait();
    const uint64_t off = (uint64_t)(off_host + (off_dev ? *off_dev : 0));
    float *gs = sm;                                    // [B][nout]
    float *ht = sm + B * nout;                         // [B][33]: columns j0..j0+31 of cat(y, h, 1)
    float *hdt = ht + B * 33;                          // same, with the classifier's dropout mask
    float *small = hdt + ((B * 33 + 3) & ~3);
    const int j0 = ((int)blockIdx.x - nbg) * 32;
    const SmallIn si = stage_small_inputs(small, 0, B, Z, C, gin, tid, blockDim.x);
    for (int i = tid; i < B * 32; i += blockDim.x) {       // the h tile (plain loads, independent of the cp.async group)
        const int b = i >> 5, j = j0 + (i & 31);
        float in = 0.f, ind = 0.f;
        if (j == C + H) in = ind = 1.f;
        else if (j < C) in = (float)yoh[(int64_t)b * C + j];
        else if (j < C + H) {
            in = __ldg(h + (int64_t)b * H + j - C);
            ind = (p > 0.f) ? (drop_keep(seed, off, (uint32_t)(b * H + j - C), p) ? in * scale : 0.f) : in;
        }
        ht[b * 33 + (i & 31)] = in;
        hdt[b * 33 + (i & 31)] = ind;
    }
    cp_async_wait_all();
    __syncthreads();
    for (int i = tid; i < B * nout; i += blockDim.x) {
        const int b = i / nout, o = i - b * nout;
        gs[i] = heads_small_grad(o, b, Z, C, si.y_hat, si.logvar, si.eps, si.g_yhat, si.g_mu, si.g_logvar, si.g_z, si.g_zcat);
    }
    __syncthreads();
    const int jl = tid & 31, og = tid >> 5;           // 8 output groups: o = og, og + 8, ...
    const int j = j0 + jl;                            // column of cat(y, h, 1)
    if (j > C + H) return;
    float acc[HB_MAXO];
#pragma unroll
    for (int t = 0; t < HB_MAXO; ++t) acc[t] = 0.f;
    for (int b = 0; b < B; ++b) {
        const float in = ht[b * 33 + jl], ind = hdt[b * 33 + jl];
        const float *g = gs + b * nout;
#pragma unroll
        for (int t = 0; t < HB_MAXO; ++t) {
            const int o = og + 8 * t;
            if (o < nout) acc[t] = fmaf(g[o], o < C ? ind : in, acc[t]);
        }
    }
#pragma unroll
    for (int t = 0; t < HB_MAXO; ++t) {
        const int o = og + 8 * t;
        if (o >= nout) break;
        if (o < C) {
            if (j == C + H) dbc[o] = acc[t];
            else if (j >= C) dWc[(int64_t)o * H + j - C] = acc[t];
        } else {
            const int i = (o - C) % Z;
            const bool is_mu = (o - C) < Z;
            if (j == C + H) (is_mu ? dbm : dbv)[i] = acc[t];
            else (is_mu ? dWm : dWv)[(int64_t)i * (C + H) + j] = acc[t];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// The heads at any B, H and Z (C <= 32).  The one-launch kernels above stage all C + 2Z weight rows (forward) or the
// whole batch's small gradients (backward) in one block's shared memory, which bounds H, Z and B.  These kernels
// tile instead, and keep the summation order of the one-launch kernels, so a mesh's results are bit-identical
// whichever pair computed them.
//   forward: a block is HT_MESH meshes (a warp each) x one output tile: tile 0 holds the C classifier logits (the
//   softmax stays in the epilogue), tile t >= 1 holds mu and logvar of the latents [16 (t-1), 16 t) (the
//   reparameterisation and zcat stay in the epilogue).  The C + H inputs stream through shared memory in chunks of
//   HT_KC columns; lane l sums the columns j = l (mod 32) in ascending order, then warp_sum - the order of
//   vae_heads_fwd_kernel.
// ---------------------------------------------------------------------------------------------
constexpr int HT_MESH = 8, HT_OUT = 32, HT_ZT = HT_OUT / 2, HT_KC = 128, HT_BC = 32;

__global__ void __launch_bounds__(256)
vae_heads_fwd_tiled_kernel(int B, int H, int Z, int C, const float *__restrict__ h, const int64_t *__restrict__ yoh,
                           const float *__restrict__ eps, const float *__restrict__ Wc, const float *__restrict__ bc,
                           const float *__restrict__ Wm, const float *__restrict__ bm, const float *__restrict__ Wv,
                           const float *__restrict__ bv, float p, uint64_t seed, const int64_t *off_dev, int64_t off_host,
                           float *__restrict__ y_hat, float *__restrict__ mu, float *__restrict__ logvar,
                           float *__restrict__ z_, float *__restrict__ zcat) {
    pdl_trigger();
    pdl_wait();
    __shared__ float xs[HT_MESH][HT_KC];          // inputs: cat(y, h) rows, or (0, dropout(h)) for the classifier tile
    __shared__ float ws[HT_OUT][HT_KC];           // weight rows of the tile's outputs (zero past the valid ones)
    __shared__ float outs[HT_MESH][HT_OUT];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b0 = blockIdx.x * HT_MESH;
    const bool cls = blockIdx.y == 0;
    const int z0 = ((int)blockIdx.y - 1) * HT_ZT;
    const int K = C + H;
    const uint64_t off = (uint64_t)(off_host + (off_dev ? *off_dev : 0));
    const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
    float acc[HT_OUT];
#pragma unroll
    for (int o = 0; o < HT_OUT; ++o) acc[o] = 0.f;
    for (int k0 = 0; k0 < K; k0 += HT_KC) {
        if (k0) __syncthreads();
        for (int i = tid; i < HT_MESH * HT_KC; i += 256) {
            const int r = i / HT_KC, jj = i % HT_KC, j = k0 + jj, b = b0 + r;
            float v = 0.f;
            if (b < B && j < K) {
                if (j < C) v = cls ? 0.f : (float)yoh[(int64_t)b * C + j];
                else {
                    v = __ldg(h + (int64_t)b * H + j - C);
                    if (cls && p > 0.f) v = drop_keep(seed, off, (uint32_t)b * (uint32_t)H + (uint32_t)(j - C), p) ? v * scale : 0.f;
                }
            }
            xs[r][jj] = v;
        }
        for (int i = tid; i < HT_OUT * HT_KC; i += 256) {
            const int o = i / HT_KC, jj = i % HT_KC, j = k0 + jj;
            float w = 0.f;
            if (j < K) {
                if (cls) {
                    if (o < C && j >= C) w = __ldg(Wc + (int64_t)o * H + j - C);
                } else {
                    const int zi = z0 + o % HT_ZT;
                    if (zi < Z) w = __ldg((o < HT_ZT ? Wm : Wv) + (int64_t)zi * K + j);
                }
            }
            ws[o][jj] = w;
        }
        __syncthreads();
        const int kc = min(HT_KC, K - k0);
        for (int jj = lane; jj < kc; jj += 32) {
            const float x = xs[warp][jj];
#pragma unroll
            for (int o = 0; o < HT_OUT; ++o) acc[o] = fmaf(x, ws[o][jj], acc[o]);
        }
    }
    float s = 0.f;                                 // lane o: output o of the tile for mesh b0 + warp
#pragma unroll
    for (int o = 0; o < HT_OUT; ++o) {
        const float t = warp_sum(acc[o]);
        if (lane == o) s = t;
    }
    const int b = b0 + warp;
    if (b >= B) return;                            // warp-uniform, and no block barrier follows
    if (cls) {
        const float v = lane < C ? s + __ldg(bc + lane) : 0.f;
        outs[warp][lane] = v;
        __syncwarp();
        if (lane < C) {                            // softmax in the order of vae_heads_fwd_kernel
            float mx = outs[warp][0];
            for (int c = 1; c < C; ++c) mx = fmaxf(mx, outs[warp][c]);
            float den = 0.f;
            for (int c = 0; c < C; ++c) den += expf(outs[warp][c] - mx);
            y_hat[(int64_t)b * C + lane] = expf(v - mx) / den;
            zcat[(int64_t)b * (C + Z) + lane] = (float)yoh[(int64_t)b * C + lane];
        }
    } else {
        const int zi = z0 + lane % HT_ZT;
        const float v = s + (zi < Z ? __ldg((lane < HT_ZT ? bm : bv) + zi) : 0.f);
        const float lv = __shfl_down_sync(0xffffffffu, v, HT_ZT);
        if (lane < HT_ZT && zi < Z) {
            mu[(int64_t)b * Z + zi] = v;
            logvar[(int64_t)b * Z + zi] = lv;
            const float zz = eps ? fmaf(__ldg(eps + (int64_t)b * Z + zi), expf(0.5f * lv), v) : v;
            z_[(int64_t)b * Z + zi] = zz;
            zcat[(int64_t)b * (C + Z) + C + zi] = zz;
        }
    }
}

// backward.  Blocks [0, nwt): a tile of HT_OUT outputs x 32 columns of cat(y, h, 1) (column C + H is the bias) of the
// weight gradients.  The block walks the batch in chunks of HT_BC meshes, recomputing their small gradients
// (heads_small_grad), and a thread sums over b in ascending order - the order of vae_heads_bwd_kernel, with no batch
// limit and no workspace.  Blocks [nwt, ..): g_h of HT_MESH meshes x 32 columns, a thread per element summing the
// C + 2Z outputs in ascending order in chunks ([0, C), then 32 at a time), the classifier's dropout mask applied
// after its C terms.
__global__ void __launch_bounds__(256)
vae_heads_bwd_tiled_kernel(int B, int H, int Z, int C, const float *__restrict__ h, const int64_t *__restrict__ yoh,
                           const float *__restrict__ Wc, const float *__restrict__ Wm, const float *__restrict__ Wv,
                           SmallIn gin, float p, uint64_t seed, const int64_t *off_dev, int64_t off_host,
                           float *__restrict__ g_h, float *__restrict__ dWc, float *__restrict__ dbc, float *__restrict__ dWm,
                           float *__restrict__ dbm, float *__restrict__ dWv, float *__restrict__ dbv, int nwt, int ncol_t) {
    pdl_trigger();
    pdl_wait();
    __shared__ float sm[3][HT_BC][33];
    const int tid = threadIdx.x, jl = tid & 31, tw = tid >> 5;
    const int nout = C + 2 * Z;
    const uint64_t off = (uint64_t)(off_host + (off_dev ? *off_dev : 0));
    const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
    if ((int)blockIdx.x < nwt) {
        // ---- weight gradients: outputs o0 + tw + 8 t (t < 4) at column j ----
        float(*gs)[33] = sm[0];                    // [HT_BC][HT_OUT]  small gradients of the chunk
        float(*ht)[33] = sm[1];                    // [HT_BC][32]      columns j0.. of cat(y, h, 1)
        float(*hdt)[33] = sm[2];                   // same, with the classifier's dropout mask
        const int ot = blockIdx.x / ncol_t, ct = blockIdx.x - ot * ncol_t;
        const int o0 = ot * HT_OUT, j0 = ct * 32, j = j0 + jl;
        float acc[HT_OUT / 8] = {0.f, 0.f, 0.f, 0.f};
        for (int c0 = 0; c0 < B; c0 += HT_BC) {
            const int nb = min(HT_BC, B - c0);
            if (c0) __syncthreads();
#pragma unroll
            for (int i = tid; i < HT_BC * 32; i += 256) {
                const int r = i >> 5, o = o0 + (i & 31), jj = j0 + (i & 31), b = c0 + r;
                gs[r][i & 31] = (r < nb && o < nout) ? heads_small_grad(o, b, Z, C, gin.y_hat, gin.logvar, gin.eps, gin.g_yhat,
                                                                         gin.g_mu, gin.g_logvar, gin.g_z, gin.g_zcat) : 0.f;
                float in = 0.f, ind = 0.f;
                if (r < nb) {
                    if (jj == C + H) in = ind = 1.f;
                    else if (jj < C) in = (float)yoh[(int64_t)b * C + jj];
                    else if (jj < C + H) {
                        in = __ldg(h + (int64_t)b * H + jj - C);
                        ind = (p > 0.f) ? (drop_keep(seed, off, (uint32_t)b * (uint32_t)H + (uint32_t)(jj - C), p) ? in * scale : 0.f) : in;
                    }
                }
                ht[r][i & 31] = in;
                hdt[r][i & 31] = ind;
            }
            __syncthreads();
            for (int r = 0; r < nb; ++r) {
                const float in = ht[r][jl], ind = hdt[r][jl];
#pragma unroll
                for (int t = 0; t < HT_OUT / 8; ++t) acc[t] = fmaf(gs[r][tw + 8 * t], o0 + tw + 8 * t < C ? ind : in, acc[t]);
            }
        }
        if (j > C + H) return;
#pragma unroll
        for (int t = 0; t < HT_OUT / 8; ++t) {
            const int o = o0 + tw + 8 * t;
            if (o >= nout) break;
            if (o < C) {
                if (j == C + H) dbc[o] = acc[t];
                else if (j >= C) dWc[(int64_t)o * H + j - C] = acc[t];
            } else {
                const int i = (o - C) % Z;
                const bool is_mu = (o - C) < Z;
                if (j == C + H) (is_mu ? dbm : dbv)[i] = acc[t];
                else (is_mu ? dWm : dWv)[(int64_t)i * (C + H) + j] = acc[t];
            }
        }
        return;
    }
    // ---- g_h of mesh b at column j ----
    float(*gs)[33] = sm[0];                        // [HT_MESH][32]  small gradients of the output chunk
    float(*wt)[33] = sm[1];                        // [32][32]       weight rows of the chunk, columns j0.. of h
    const int bi = (int)blockIdx.x - nwt;
    const int hts = (H + 31) / 32;
    const int mt = bi / hts, jt = bi - mt * hts;
    const int b0 = mt * HT_MESH, j0 = jt * 32;
    const int b = b0 + tw, j = j0 + jl;
    float a = 0.f;
    for (int o0 = 0; o0 < nout;) {
        const int n = o0 == 0 ? C : min(32, nout - o0);
        if (o0) __syncthreads();
        {
            const int r = tid >> 5, oo = tid & 31;           // HT_MESH x 32 = 256 threads
            gs[r][oo] = (oo < n && b0 + r < B) ? heads_small_grad(o0 + oo, b0 + r, Z, C, gin.y_hat, gin.logvar, gin.eps, gin.g_yhat,
                                                                  gin.g_mu, gin.g_logvar, gin.g_z, gin.g_zcat) : 0.f;
        }
#pragma unroll
        for (int i = tid; i < 32 * 32; i += 256) {
            const int oo = i >> 5, col = j0 + (i & 31), o = o0 + oo;
            float w = 0.f;
            if (oo < n && col < H)
                w = __ldg(o < C ? Wc + (int64_t)o * H + col
                                : (o - C < Z ? Wm + (int64_t)(o - C) * (C + H) : Wv + (int64_t)(o - C - Z) * (C + H)) + C + col);
            wt[oo][i & 31] = w;
        }
        __syncthreads();
        for (int oo = 0; oo < n; ++oo) a = fmaf(gs[tw][oo], wt[oo][jl], a);
        if (o0 == 0 && p > 0.f && b < B && j < H) a = drop_keep(seed, off, (uint32_t)b * (uint32_t)H + (uint32_t)j, p) ? a * scale : 0.f;
        o0 += n;
    }
    if (b < B && j < H) g_h[(int64_t)b * H + j] = a;
}

}  // namespace mvb

using namespace mvb;

extern "C" int mvb_linear_fwd(int M, int K, int N, const float *x, int x_vm_f, const float *W, const float *bias,
                              int relu, float p_drop, uint64_t seed, const int64_t *offset_dev, int64_t offset_host,
                              float *y, int y_vm_f, void *stream) {
    MVB_REQUIRE(M > 0 && K > 0 && N > 0 && x && W && y, "linear_fwd: bad arguments");
    MVB_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "linear_fwd: dropout p=%f outside [0,1)", p_drop);
    MVB_REQUIRE((x_vm_f == 0 || K % x_vm_f == 0) && (y_vm_f == 0 || N % y_vm_f == 0), "linear_fwd: vertex-major width does not divide the feature count");
    MVB_REQUIRE((int64_t)M * N < (1LL << 32), "linear_fwd: M*N exceeds the dropout counter range");
    const int K4 = (K + 3) & ~3;
    const int KC = K4 < 640 ? K4 : 640;
    const bool vec = (K % 4 == 0) && (x_vm_f == 0 || x_vm_f % 4 == 0) && aligned16(x) && aligned16(W);
    const size_t smem = (size_t)(LF_TM + LF_TN) * (KC + 4) * sizeof(float);
    static DevFlags granted4, granted1;
    int rc = vec ? smem_optin(linear_fwd_kernel<4>, smem, granted4, "linear_fwd") : smem_optin(linear_fwd_kernel<1>, smem, granted1, "linear_fwd");
    if (rc) return rc;
    dim3 grid((N + LF_TN - 1) / LF_TN, (M + LF_TM - 1) / LF_TM);
    if (vec)
        launch_pdl(linear_fwd_kernel<4>, grid, dim3(256), smem, (cudaStream_t)stream, M, K, N, x, x_vm_f, W, bias, relu, p_drop, seed, offset_dev, offset_host, y, y_vm_f, KC);
    else
        launch_pdl(linear_fwd_kernel<1>, grid, dim3(256), smem, (cudaStream_t)stream, M, K, N, x, x_vm_f, W, bias, relu, p_drop, seed, offset_dev, offset_host, y, y_vm_f, KC);
    return check_launch("mvb_linear_fwd");
}

extern "C" int mvb_linear_bwd(int M, int K, int N, const float *x, int x_vm_f, const float *W, const float *y,
                              const float *gy, int y_vm_f, int relu, float p_drop, float *dx, float *dW, float *db,
                              void *stream) {
    MVB_REQUIRE(M > 0 && K > 0 && N > 0 && x && W && gy && dW && (!relu || y), "linear_bwd: bad arguments");
    MVB_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "linear_bwd: dropout p=%f outside [0,1)", p_drop);
    MVB_REQUIRE(relu || p_drop == 0.f, "linear_bwd: dropout without ReLU is not recoverable from y");
    MVB_REQUIRE((x_vm_f == 0 || K % x_vm_f == 0) && (y_vm_f == 0 || N % y_vm_f == 0), "linear_bwd: vertex-major width does not divide the feature count");
    const int k_tiles = (K + BW_TK - 1) / BW_TK;
    const int nA = ((N + BW_TN - 1) / BW_TN) * k_tiles;
    const int nB = dx ? ((K + BW_TKX - 1) / BW_TKX) * ((M + BW_TMB - 1) / BW_TMB) : 0;
    const int N4 = (N + 3) & ~3;
    const int nc_b = N4 < 640 ? N4 : 640;
    const size_t smA = (size_t)3 * 64 * BW_LA * sizeof(float);
    const size_t smB = (size_t)(2 * BW_TMB * (nc_b + 4) + nc_b * BW_TKX) * sizeof(float);
    const size_t smem = nB ? (smA > smB ? smA : smB) : smA;
    const bool vn = (N % 4 == 0) && (y_vm_f == 0 || y_vm_f % 4 == 0) && aligned16(gy) && (!relu || aligned16(y));
    const bool vk = (K % 4 == 0) && (x_vm_f == 0 || x_vm_f % 4 == 0) && aligned16(x) && aligned16(W);
    static DevFlags granted[4];
    const float scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
    int rc;
#define MVB_LBWD(VN_, VK_, SLOT)                                                                                             \
    do {                                                                                                                     \
        rc = smem_optin(linear_bwd_kernel<VN_, VK_>, smem, granted[SLOT], "linear_bwd");                                     \
        if (rc) return rc;                                                                                                   \
        launch_pdl(linear_bwd_kernel<VN_, VK_>, dim3(nA + nB), dim3(256), smem, (cudaStream_t)stream, M, K, N, x, x_vm_f, W, y, gy, y_vm_f, relu, \
                                                                                  scale, dx, dW, db, nA, k_tiles, nc_b);     \
    } while (0)
    // Deferred mode (step engine, mvb_tune "defer_wgrad=1"): the input-gradient tiles (role B) are what the backward
    // pass waits for - they are launched alone on the caller's stream, and the weight / bias gradient tiles (role A) go
    // to the deferred side chain (joined by mvb_side_join before the optimizer).  Otherwise one launch with both roles.
    SideChain side((cudaStream_t)stream, (dx && nB) ? 1 : -1, false);
#define MVB_LBWD_SPLIT(VN_, VK_, SLOT)                                                                                        \
    do {                                                                                                                     \
        rc = smem_optin(linear_bwd_kernel<VN_, VK_>, smem, granted[SLOT], "linear_bwd");                                     \
        if (rc) return rc;                                                                                                   \
        launch_pdl(linear_bwd_kernel<VN_, VK_>, dim3(nB), dim3(256), smem, (cudaStream_t)stream, M, K, N, x, x_vm_f, W, y, gy, y_vm_f, relu,      \
                                                                             scale, dx, dW, db, 0, k_tiles, nc_b);           \
        rc = check_launch("mvb_linear_bwd dx");                                                                              \
        if (rc) return rc;                                                                                                   \
        launch_pdl(linear_bwd_kernel<VN_, VK_>, dim3(nA), dim3(256), smem, side.stream(), M, K, N, x, x_vm_f, W, y, gy, y_vm_f, relu, scale,     \
                                                             nullptr, dW, db, nA, k_tiles, nc_b);                            \
        return check_launch("mvb_linear_bwd dW");                                                                            \
    } while (0)
    if (side.deferred()) {
        if (vn && vk) MVB_LBWD_SPLIT(4, 4, 0);
        else if (vn) MVB_LBWD_SPLIT(4, 1, 1);
        else if (vk) MVB_LBWD_SPLIT(1, 4, 2);
        else MVB_LBWD_SPLIT(1, 1, 3);
    }
#undef MVB_LBWD_SPLIT
    if (vn && vk) MVB_LBWD(4, 4, 0);
    else if (vn) MVB_LBWD(4, 1, 1);
    else if (vk) MVB_LBWD(1, 4, 2);
    else MVB_LBWD(1, 1, 3);
#undef MVB_LBWD
    return check_launch("mvb_linear_bwd");
}

extern "C" int mvb_vae_heads_fwd(int B, int H, int Z, int C, const float *h, const int64_t *y_onehot, const float *eps,
                                 const float *Wc, const float *bc, const float *Wm, const float *bm, const float *Wv,
                                 const float *bv, float p_drop, uint64_t seed, const int64_t *offset_dev,
                                 int64_t offset_host, float *y_hat, float *mu, float *logvar, float *z, float *zcat,
                                 void *stream) {
    MVB_REQUIRE(B > 0 && H > 0 && Z > 0 && C > 0 && h && y_onehot && Wc && bc && Wm && bm && Wv && bv && y_hat && mu &&
                    logvar && z && zcat, "vae_heads_fwd: bad arguments");
    MVB_REQUIRE(C <= 32, "vae_heads_fwd: C=%d classes, at most 32 supported", C);
    MVB_REQUIRE((int64_t)B * H < (1LL << 32), "vae_heads_fwd: B*H exceeds the dropout counter range");
    MVB_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "vae_heads_fwd: dropout p=%f outside [0,1)", p_drop);
    const size_t smem = (2 * (size_t)(C + H) + (size_t)(C + 2 * Z) * (C + H + 1)) * sizeof(float);
    if (C + 2 * Z > HEADS_MAX_OUT || smem > 220 * 1024) {        // the weights do not fit one block: the tiled kernel
        launch_pdl(vae_heads_fwd_tiled_kernel, dim3((B + HT_MESH - 1) / HT_MESH, 1 + (Z + HT_ZT - 1) / HT_ZT), dim3(256), 0,
                   (cudaStream_t)stream, B, H, Z, C, h, y_onehot, eps, Wc, bc, Wm, bm, Wv, bv, p_drop, seed, offset_dev,
                   offset_host, y_hat, mu, logvar, z, zcat);
        return check_launch("mvb_vae_heads_fwd");
    }
    static DevFlags granted;
    int rc = smem_optin(vae_heads_fwd_kernel, smem, granted, "vae_heads_fwd");
    if (rc) return rc;
    launch_pdl(vae_heads_fwd_kernel, dim3(B), dim3(256), smem, (cudaStream_t)stream, B, H, Z, C, h, y_onehot, eps, Wc, bc, Wm, bm, Wv, bv, p_drop,
                                                                  seed, offset_dev, offset_host, y_hat, mu, logvar, z, zcat);
    return check_launch("mvb_vae_heads_fwd");
}

extern "C" int mvb_vae_heads_bwd(int B, int H, int Z, int C, const float *h, const int64_t *y_onehot, const float *eps,
                                 const float *Wc, const float *Wm, const float *Wv, const float *y_hat,
                                 const float *logvar, float p_drop, uint64_t seed, const int64_t *offset_dev,
                                 int64_t offset_host, const float *g_yhat, const float *g_mu, const float *g_logvar,
                                 const float *g_z, const float *g_zcat, float *g_h, float *dWc, float *dbc, float *dWm,
                                 float *dbm, float *dWv, float *dbv, void *stream) {
    MVB_REQUIRE(B > 0 && H > 0 && Z > 0 && C > 0 && h && y_onehot && Wc && Wm && Wv && y_hat && logvar && g_h && dWc &&
                    dbc && dWm && dbm && dWv && dbv, "vae_heads_bwd: bad arguments");
    MVB_REQUIRE(C <= 32, "vae_heads_bwd: C=%d classes, at most 32 supported", C);
    MVB_REQUIRE((int64_t)B * H < (1LL << 32), "vae_heads_bwd: B*H exceeds the dropout counter range");
    MVB_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "vae_heads_bwd: dropout p=%f outside [0,1)", p_drop);
    const int nout = C + 2 * Z;
    const int ntile = (C + H + 1 + 31) / 32;
    SmallIn gin;
    gin.y_hat = y_hat; gin.logvar = logvar; gin.eps = eps; gin.g_yhat = g_yhat; gin.g_mu = g_mu; gin.g_logvar = g_logvar;
    gin.g_z = g_z; gin.g_zcat = g_zcat;
    const size_t smA = ((size_t)nout * (C + H + 1) + HB_ROWS * nout + 4 + small_in_words(HB_ROWS, Z, C)) * sizeof(float);
    const size_t smB = ((size_t)B * (nout + 2 * 33 + 2 * C + 5 * Z + C + Z) + 4 + 32) * sizeof(float);   // small_in_words(B, Z, C)
    const size_t smem = smA > smB ? smA : smB;
    if (nout > HEADS_MAX_OUT || smem > 220 * 1024) {    // the weights or the batch do not fit one block: the tiled kernel
        const int nwt = ((nout + HT_OUT - 1) / HT_OUT) * ntile;
        const int64_t nblk = (int64_t)nwt + (int64_t)((B + HT_MESH - 1) / HT_MESH) * ((H + 31) / 32);
        MVB_REQUIRE(nblk < (1LL << 31), "vae_heads_bwd: B=%d H=%d needs too many blocks", B, H);
        launch_pdl(vae_heads_bwd_tiled_kernel, dim3((unsigned)nblk), dim3(256), 0, (cudaStream_t)stream, B, H, Z, C, h, y_onehot,
                   Wc, Wm, Wv, gin, p_drop, seed, offset_dev, offset_host, g_h, dWc, dbc, dWm, dbm, dWv, dbv, nwt, ntile);
        return check_launch("mvb_vae_heads_bwd");
    }
    static DevFlags granted;
    int rc = smem_optin(vae_heads_bwd_kernel, smem, granted, "vae_heads_bwd");
    if (rc) return rc;
    const int nbg = (B + HB_ROWS - 1) / HB_ROWS;
    launch_pdl(vae_heads_bwd_kernel, dim3(nbg + ntile), dim3(256), smem, (cudaStream_t)stream, B, H, Z, C, h, y_onehot, Wc, Wm, Wv, gin, p_drop, seed,
                                                                            offset_dev, offset_host, g_h, dWc, dbc, dWm, dbm, dWv,
                                                                            dbv, nbg);
    return check_launch("mvb_vae_heads_bwd");
}
