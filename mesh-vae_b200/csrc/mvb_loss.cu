// VAE loss epilogue and the small elementwise pieces around the latent code
// (models/cheb_VAE.py:309-346, logpdf.py:7-8,22-28) as fused, deterministic CUDA kernels.
//
// The reconstruction arrives VERTEX-MAJOR [N,B,C] (as the decoder kernels write it) while the
// ground truth arrives mesh-major [B,N,C] (fp64 in training, main.py:70 / data.py:107): the
// forward kernel stages a (32 vertices x 32 meshes) tile of each through shared memory so both
// global reads are coalesced, emits (recon - x)/sigma^2 for the backward pass in the same sweep
// and reduces the NLL per mesh with a fixed-order warp reduction -> per-(vertex-chunk, mesh)
// partials -> ordered final sum.  No atomics anywhere, bit-reproducible run to run.
// The sigma-VAE variants (optimal and learned decoder sigma) share the partial kernel: it then sums the squared error per
// mesh and keeps recon - x unscaled, and their finalize kernel derives log sigma on the device from the batch's error or
// from a parameter (no host round trip: a captured step follows new inputs and Adam's updates of the parameter).
// The importance-weighted log-likelihood estimate (mvb_iw_*) shares it too: S reconstructions per ground-truth mesh.
// Roofline: HBM; algorithmic bytes = N*B*C*(4 + sizeof(x) + 4).
#include "mvb_internal.cuh"

namespace mvb {

#define MVB_HALF_LOG_2PI 0.91893853320467274178

template <typename XT>
struct AccT { typedef float type; };
template <>
struct AccT<double> { typedef double type; };

// SSE = false: partial = sum of the NLL terms, dnll = (recon - x)/sigma^2 (the reference's constant sigma);
// SSE = true: partial = sum of (recon - x)^2 (fp64 squares), dnll = recon - x (sigma is not known yet).
// B counts the reconstructions (columns of recon); S of them share one ground truth: column j is compared with mesh j / S
// of xgt (S = 1: the loss epilogue; S > 1: the importance samples of mvb_iw_log_weights), and the block loads each
// ground-truth row it needs once.  dnll = NULL: no dnll is written.
template <typename XT, bool SSE>
__global__ void __launch_bounds__(256)
vae_rec_partial_kernel(int B, int N, int C, int ld, int VCH, int BCH, int S, const float *__restrict__ recon,
                       const XT *__restrict__ xgt, float log_sigma, float sigma,
                       double *__restrict__ partial, float *__restrict__ dnll) {
    pdl_trigger();
    pdl_wait();
    typedef typename AccT<XT>::type AT;
    extern __shared__ double smem_d[];
    XT *Xs = reinterpret_cast<XT *>(smem_d);                     // [BCH][VCH*C]
    float *Rs = reinterpret_cast<float *>(Xs + (size_t)BCH * VCH * C);  // [VCH][BCH*ld]  (ld >= C floats per entry)
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int v0 = blockIdx.x * VCH, b0 = blockIdx.y * BCH;
    const int nv = min(VCH, N - v0), nb = min(BCH, B - b0);
    const int m0 = b0 / S, nm = (b0 + nb - 1) / S - m0 + 1;     // the ground-truth meshes of the block's columns
    const int rw = nb * ld; // contiguous run per vertex in recon (entries of ld floats, the first C are data)
    const int xw = nv * C;  // contiguous run per mesh in x_gt
    // both tiles through cp.async: every element of the block's two tiles is in flight at once (one exposed
    // latency instead of one per batch of register loads); a warp walks one contiguous run at a time
    {
        const int warp_ = tid >> 5, lane_ = tid & 31, nwarps_ = nthreads >> 5;
        for (int v = warp_; v < nv; v += nwarps_) {
            const float *src = recon + ((int64_t)(v0 + v) * B + b0) * ld;
            float *dst = Rs + v * (BCH * ld);
            if ((rw & 3) == 0 && ((BCH * ld) & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
                for (int e = 4 * lane_; e < rw; e += 128) cp_async<4>(dst + e, src + e);      // 16-byte pieces (padded entries)
            } else {
                for (int e = lane_; e < rw; e += 32) cp_async<1>(dst + e, src + e);
            }
        }
        for (int b = warp_; b < nm; b += nwarps_) {
            const XT *src = xgt + ((int64_t)(m0 + b) * N + v0) * C;
            XT *dst = Xs + b * (VCH * C);
            constexpr int PER16 = 16 / (int)sizeof(XT);
            if ((xw % PER16) == 0 && ((VCH * C) % PER16) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
                for (int e = PER16 * lane_; e < xw; e += 32 * PER16) {
                    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + e);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src + e) : "memory");
                }
                continue;
            }
            for (int e = lane_; e < xw; e += 32) {
                if (sizeof(XT) == 8) {
                    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + e);
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(src + e) : "memory");
                } else {
                    cp_async<1>(dst + e, src + e);
                }
            }
        }
        cp_async_wait_all();
    }
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
    const AT sg = (AT)sigma;
    const AT inv_sg = (AT)1 / sg, inv_sg2 = (AT)1 / (sg * sg);     // two multiplies per element instead of two (fp64) divisions
    const AT cst = (AT)log_sigma + (AT)MVB_HALF_LOG_2PI;
    for (int b = warp; b < nb; b += nwarps) {
        const XT *xs = Xs + ((b0 + b) / S - m0) * (VCH * C);
        double s = 0.0;
        for (int e = lane; e < xw; e += 32) {
            const int v = e / C, c = e - v * C;
            float *rp = Rs + v * (BCH * ld) + b * ld + c;
            const AT d = (AT)(*rp) - (AT)xs[e];   // recon - x
            if constexpr (SSE) {
                s = fma((double)d, (double)d, s);
                *rp = (float)d;
            } else {
                const AT t = d * inv_sg;
                const AT nll = (AT)0.5 * t * t + cst;
                s += (double)nll;
                *rp = (float)(d * inv_sg2);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
        if (lane == 0) partial[(int64_t)blockIdx.x * B + b0 + b] = s;
    }
    if (!dnll) return;
    __syncthreads();
    // padded mesh coordinates: one 16-byte entry per (vertex, mesh), pad lane zeroed (an offset view of dnll: scalar path)
    if (ld == 4 && C == 3 && (reinterpret_cast<uintptr_t>(dnll) & 15) == 0) {
        for (int i = tid; i < nv * nb; i += nthreads) {
            const int v = i / nb, b = i - v * nb;
            float4 r = *reinterpret_cast<const float4 *>(Rs + v * (BCH * 4) + b * 4);
            r.w = 0.f;
            *reinterpret_cast<float4 *>(dnll + ((int64_t)(v0 + v) * B + b0 + b) * 4) = r;
        }
        return;
    }
    for (int i = tid; i < nv * rw; i += nthreads) {
        const int v = i / rw, rem = i - v * rw;
        const float val = (ld == C || rem % ld < C) ? Rs[v * (BCH * ld) + rem] : 0.f;      // padding entries carry no gradient
        dnll[((int64_t)(v0 + v) * B + b0) * ld + rem] = val;
    }
}

// log sigma = sc(t) = -6 + softplus(t + 6) and sc'(t) = sigmoid(t + 6), both from exp(-|t + 6|): finite for every t,
// t = -inf (a perfect reconstruction under the optimal sigma) included, where they are -6 and 0
__device__ __forceinline__ void softclip_m6(double t, double &log_sigma, double &dsc) {
    const double u = t + 6.0, e = exp(-fabs(u));
    log_sigma = -6.0 + fmax(u, 0.0) + log1p(e);
    dsc = (u >= 0.0 ? 1.0 : e) / (1.0 + e);
}

// SIGMA = false: the reference's constant sigma (the partials are NLL sums).  SIGMA = true: the partials are squared
// errors; after phase 1 the block sums the per-mesh SSE_b in a fixed order, derives log sigma (sigma_mode 1: optimal,
// from the batch's SSE; 2: learned, sc(*s_param)) and writes the state the backward pass reads, then phase 2 turns
// SSE_b into rec_b = SSE_b / (2 sigma^2) + n_elem (log sigma + log(2 pi)/2).
template <bool SIGMA>
__global__ void __launch_bounds__(1024)
vae_loss_finalize_kernel(int B, int Z, int ncls, int nchunks, const double *__restrict__ partial,
                         const float *__restrict__ mu, const float *__restrict__ logvar,
                         const float *__restrict__ y_hat, const int64_t *__restrict__ y,
                         double *loss, float *kld, double *rec, int64_t *correct,
                         int sigma_mode, double n_elem, const float *__restrict__ s_param, double *sigma_state) {
    pdl_trigger();
    pdl_wait();
    __shared__ double s_sum[1024];
    __shared__ int s_cnt[1024];
    __shared__ double s_sig[2];
    const int tid = threadIdx.x;
    double lsum = 0.0;
    int lcnt = 0;
    // phase 1: a warp per mesh sums the vertex-chunk partials (lane-strided, four independent loads in flight per
    // lane, fixed shuffle tree); 32 warps: two meshes per warp at 64 meshes instead of eight
    const int wid = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
    for (int b = wid; b < B; b += nw) {
        double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
        int ch = lane;
        for (; ch + 96 < nchunks; ch += 128) {
            r0 += partial[(int64_t)ch * B + b];
            r1 += partial[(int64_t)(ch + 32) * B + b];
            r2 += partial[(int64_t)(ch + 64) * B + b];
            r3 += partial[(int64_t)(ch + 96) * B + b];
        }
        for (; ch < nchunks; ch += 32) r0 += partial[(int64_t)ch * B + b];
        double r = (r0 + r1) + (r2 + r3);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) r += __shfl_xor_sync(0xffffffffu, r, off);
        if (lane == 0) rec[b] = r;
    }
    __syncthreads();
    if constexpr (SIGMA) {
        double e = 0.0;
        for (int b = tid; b < B; b += blockDim.x) e += rec[b];
        s_sum[tid] = e;
        __syncthreads();
        for (int off = blockDim.x >> 1; off > 0; off >>= 1) {
            if (tid < off) s_sum[tid] += s_sum[tid + off];
            __syncthreads();
        }
        if (tid == 0) {
            const double sse = s_sum[0], bn = (double)B * n_elem;
            const double t = sigma_mode == 1 ? (sse > 0.0 ? 0.5 * log(sse / bn) : -INFINITY) : (double)*s_param;
            double ls, dsc;
            softclip_m6(t, ls, dsc);
            const double inv_s2 = exp(-2.0 * ls);
            const double g_t = (bn - sse * inv_s2) * dsc;         // d(sum_b rec_b)/dt
            sigma_state[0] = ls;
            sigma_state[1] = inv_s2;
            sigma_state[2] = sse;
            sigma_state[3] = dsc;
            // d(sum_b rec_b)/d(recon - x) = coef (recon - x): the optimal sigma adds its own dependence on the error
            // (dt/d(recon - x) = (recon - x)/SSE); a zero SSE has t = -inf and sc' = 0, so nothing is added
            sigma_state[4] = (sigma_mode == 1 && sse > 0.0) ? inv_s2 + g_t / sse : inv_s2;
            sigma_state[5] = g_t;
            s_sig[0] = ls;
            s_sig[1] = inv_s2;
        }
        __syncthreads();
    }
    // phase 2: 16 lanes per mesh for the per-mesh terms (the latent sums are lane-strided + a fixed xor tree; a single
    // thread per mesh walked 2 Z dependent global loads)
    constexpr int G = 16;
    const int sub = tid & (G - 1);
    for (int b0 = 0; b0 < B; b0 += blockDim.x / G) {
        const int b = b0 + tid / G;
        const bool ok = b < B;
        float k = 0.f;
        if (ok)
            for (int j = sub; j < Z; j += G) {
                const float m = mu[b * Z + j], lv = logvar[b * Z + j];
                k += 1.f + lv - m * m - expf(lv);
            }
#pragma unroll
        for (int off = G / 2; off > 0; off >>= 1) k += __shfl_xor_sync(0xffffffffu, k, off);
        if (!ok || sub != 0) continue;
        double r = rec[b];
        if constexpr (SIGMA) {
            r = 0.5 * r * s_sig[1] + n_elem * (s_sig[0] + MVB_HALF_LOG_2PI);
            rec[b] = r;
        }
        k *= -0.5f;
        kld[b] = k;
        float q = 0.f;
        int am_h = 0, am_y = 0;
        float best_h = y_hat[b * ncls];
        int64_t best_y = y[b * ncls];
        for (int c = 0; c < ncls; ++c) {
            const float h = y_hat[b * ncls + c];
            const int64_t yy = y[b * ncls + c];
            q += h * (float)yy;
            if (h > best_h) { best_h = h; am_h = c; }
            if (yy > best_y) { best_y = yy; am_y = c; }
        }
        const float logqy = logf(q);
        lsum += (double)k + r - (double)(2.f * logqy);
        lcnt += (am_h == am_y) ? 1 : 0;
    }
    s_sum[tid] = lsum;
    s_cnt[tid] = lcnt;
    __syncthreads();
    for (int off = blockDim.x >> 1; off > 0; off >>= 1) {
        if (tid < off) {
            s_sum[tid] += s_sum[tid + off];
            s_cnt[tid] += s_cnt[tid + off];
        }
        __syncthreads();
    }
    if (tid == 0) {
        *loss = s_sum[0] / (double)B;
        *correct = (int64_t)s_cnt[0];
    }
}

// COEF: the sigma-VAE backward, dst = (gloss/B * coef) src with coef from the forward pass's sigma state
template <bool COEF>
__global__ void scale_by_gloss_kernel(int64_t n, const float *__restrict__ src,
                                      const double *__restrict__ gloss, double inv_b, const double *__restrict__ coef, float *dst) {
    const float s = COEF ? (float)(*gloss * inv_b * *coef) : (float)(*gloss * inv_b);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = s * src[i];
}

template <bool COEF>
__global__ void scale4_by_gloss_kernel(int64_t n4, const float4 *__restrict__ src,
                                       const double *__restrict__ gloss, double inv_b, const double *__restrict__ coef, float4 *dst) {
    pdl_trigger();
    pdl_wait();
    const float s = COEF ? (float)(*gloss * inv_b * *coef) : (float)(*gloss * inv_b);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = __ldg(src + i);
        dst[i] = make_float4(s * v.x, s * v.y, s * v.z, s * v.w);
    }
}

__global__ void vae_loss_bwd_small_kernel(int B, int Z, int ncls, const float *__restrict__ mu,
                                          const float *__restrict__ logvar,
                                          const float *__restrict__ y_hat,
                                          const int64_t *__restrict__ y,
                                          const double *__restrict__ gloss, float *d_mu,
                                          float *d_logvar, float *d_yhat, const double *__restrict__ d_t, float *d_s) {
    pdl_trigger();
    pdl_wait();
    const float s = (float)(*gloss / (double)B);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (d_s && i == 0) *d_s = (float)(*gloss / (double)B * *d_t);        // learned sigma: gloss/B * d(sum_b rec_b)/ds
    if (i < B * Z) {
        if (d_mu) d_mu[i] = s * mu[i];
        if (d_logvar) d_logvar[i] = s * 0.5f * (expf(logvar[i]) - 1.f);
    }
    if (d_yhat && i < B) {
        float q = 0.f;
        for (int c = 0; c < ncls; ++c) q += y_hat[i * ncls + c] * (float)y[i * ncls + c];
        for (int c = 0; c < ncls; ++c) d_yhat[i * ncls + c] = s * (-2.f) * (float)y[i * ncls + c] / q;
    }
}

// ---- input hand-off: [B,N,C] mesh-major -> [N,B,Cp] vertex-major, zero padded (one pass instead of transpose copy,
// fill and padded copy) -------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pack_vertex_major_kernel(int B, int N, int C, int Cp, const float *__restrict__ x, float *__restrict__ out) {
    pdl_trigger();
    pdl_wait();
    // block = 32 vertices x 8 meshes through shared memory: reads coalesced along a mesh's vertices, writes along
    // a vertex's meshes
    __shared__ float tile[8][32 * 8 + 1];
    const int v0 = blockIdx.x * 32, b0 = blockIdx.y * 8;
    const int nv = min(32, N - v0), nb = min(8, B - b0);
    if (C == 3 && Cp == 4 && nv == 32 && nb == 8 && blockDim.x == 256 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        // the mesh coordinates: 96 contiguous floats per mesh in, one float4 entry per (vertex, mesh) out, no divisions
        const int t = threadIdx.x;
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int i = t + u * 256, b = i / 96, rem = i - b * 96;
            tile[b][rem] = __ldg(x + ((int64_t)(b0 + b) * N + v0) * 3 + rem);
        }
        __syncthreads();
        const int v = t >> 3, b = t & 7;
        const float4 o = make_float4(tile[b][3 * v], tile[b][3 * v + 1], tile[b][3 * v + 2], 0.f);
        *reinterpret_cast<float4 *>(out + ((int64_t)(v0 + v) * B + b0 + b) * 4) = o;
        return;
    }
    for (int i = threadIdx.x; i < nb * nv * C; i += blockDim.x) {
        const int b = i / (nv * C), rem = i - b * (nv * C);
        tile[b][rem] = __ldg(x + ((int64_t)(b0 + b) * N + v0) * C + rem);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nv * nb * Cp; i += blockDim.x) {
        const int v = i / (nb * Cp), rem = i - v * (nb * Cp);
        const int b = rem / Cp, c = rem - b * Cp;
        out[((int64_t)(v0 + v) * B + b0) * Cp + rem] = c < C ? tile[b][v * C + c] : 0.f;
    }
}

// ---- next row f3: per-batch reconstruction error of the training / evaluation loops ---------------
// main.py:88-93, :139-146, inference.py:100-127:  recon_mesh = out.cpu() * std + mean (fp32);
// recon_mesh = bmm(recon_mesh * s, R) + m (fp64: s, R, m come from the Procrustes alignment as float64);
// diff = sqrt(((recon_mesh - gt_mesh)**2).sum(-1)) -> .mean(-1), .max(-1) per mesh.
// The reference moves the whole [B,N,3] reconstruction to the host for this every batch; here it is one
// pass over the vertex-major reconstruction on the device, per-(vertex chunk, mesh) partial sums / maxima
// and an ordered final reduction.
template <typename GtT>
__global__ void __launch_bounds__(256)
recon_error_partial_kernel(int B, int N, int ld, const float *__restrict__ recon, const float *__restrict__ mean,
                           const float *__restrict__ stdv, const double *__restrict__ sc, const double *__restrict__ R,
                           const double *__restrict__ m, const GtT *__restrict__ gt, double *__restrict__ psum,
                           double *__restrict__ pmax, float *__restrict__ vertex_err, float *__restrict__ mesh_out) {
    __shared__ double s_sum[256], s_max[256];
    const int b = blockIdx.y, tid = threadIdx.x;
    const int v = blockIdx.x * 256 + tid;
    double err = 0.0;
    if (v < N) {
        const float *rp = recon + ((int64_t)v * B + b) * ld;
        const double s = sc[b];
        double p[3], q[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) p[c] = (double)__fadd_rn(__fmul_rn(rp[c], stdv[v * 3 + c]), mean[v * 3 + c]) * s;
        const double *Rb = R + (int64_t)b * 9;
#pragma unroll
        for (int j = 0; j < 3; ++j) q[j] = p[0] * Rb[j] + p[1] * Rb[3 + j] + p[2] * Rb[6 + j] + m[(int64_t)b * 3 + j];
        if (mesh_out) {                 // the back-transformed mesh itself (OBJ output of evaluate(vis) / inference.py)
            float *o = mesh_out + ((int64_t)b * N + v) * 3;
            o[0] = (float)q[0];
            o[1] = (float)q[1];
            o[2] = (float)q[2];
        }
        if (gt) {
            const GtT *g = gt + ((int64_t)b * N + v) * 3;
            const double d0 = q[0] - (double)g[0], d1 = q[1] - (double)g[1], d2 = q[2] - (double)g[2];
            err = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
            if (vertex_err) vertex_err[(int64_t)b * N + v] = (float)err;
        }
    }
    s_sum[tid] = err;
    s_max[tid] = err;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (tid < off) {
            s_sum[tid] += s_sum[tid + off];
            s_max[tid] = fmax(s_max[tid], s_max[tid + off]);
        }
        __syncthreads();
    }
    if (tid == 0) {
        psum[(int64_t)blockIdx.x * B + b] = s_sum[0];
        pmax[(int64_t)blockIdx.x * B + b] = s_max[0];
    }
}

__global__ void recon_error_finalize_kernel(int B, int N, int nchunks, const double *__restrict__ psum,
                                            const double *__restrict__ pmax, double *mean_err, double *max_err) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double s = 0.0, mx = 0.0;
    for (int ch = 0; ch < nchunks; ++ch) {
        s += psum[(int64_t)ch * B + b];
        mx = fmax(mx, pmax[(int64_t)ch * B + b]);
    }
    mean_err[b] = s / (double)N;
    max_err[b] = mx;
}

// epoch statistics of the train / evaluate loops (main.py:83-86, :93, :135-137) kept on the device: one launch per
// batch adds the batch's sums into 8 fp64 accumulators; the loop reads them ONCE per epoch instead of three
// `.cpu()` synchronisations + a [B,N,3] read-back per batch.  acc = [loss*B, kld_sum, rec_sum, err_sum, correct, count, 0, 0]
template <typename RecT>
__global__ void __launch_bounds__(256)
epoch_meter_kernel(int B, const double *__restrict__ loss, const float *__restrict__ loss32, const float *__restrict__ kld,
                   const RecT *__restrict__ rec, const int64_t *__restrict__ correct, const double *__restrict__ mean_err,
                   double *acc) {
    __shared__ double sh[3][256];
    const int tid = threadIdx.x;
    double k = 0.0, r = 0.0, e = 0.0;
    for (int b = tid; b < B; b += 256) {          // fixed order: deterministic sums
        k += (double)kld[b];
        r += (double)rec[b];
        if (mean_err) e += mean_err[b];
    }
    sh[0][tid] = k;
    sh[1][tid] = r;
    sh[2][tid] = e;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (tid < off) {
            sh[0][tid] += sh[0][tid + off];
            sh[1][tid] += sh[1][tid + off];
            sh[2][tid] += sh[2][tid + off];
        }
        __syncthreads();
    }
    if (tid == 0) {
        const double l = loss ? *loss : (double)*loss32;
        acc[0] += l * (double)B;
        acc[1] += sh[0][0];
        acc[2] += sh[1][0];
        acc[3] += sh[2][0];
        if (correct) acc[4] += (double)*correct;
        acc[5] += (double)B;
    }
}

// ---- reparameterisation ----------------------------------------------------------------------
__global__ void reparam_fwd_kernel(int64_t n, const float *__restrict__ mu,
                                   const float *__restrict__ logvar, const float *__restrict__ eps,
                                   float *z) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) z[i] = fmaf(eps[i], expf(0.5f * logvar[i]), mu[i]);
}
__global__ void reparam_bwd_kernel(int64_t n, const float *__restrict__ logvar,
                                   const float *__restrict__ eps, const float *__restrict__ dz,
                                   float *dmu, float *dlogvar) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const float g = dz[i];
        if (dmu) dmu[i] = g;
        if (dlogvar) dlogvar[i] = g * eps[i] * 0.5f * expf(0.5f * logvar[i]);
    }
}

// ---- logpdf drop-ins ---------------------------------------------------------------------------
__global__ void kld_fwd_kernel(int B, int Z, const float *__restrict__ mu,
                               const float *__restrict__ logvar, float *out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float k = 0.f;
    for (int j = 0; j < Z; ++j) {
        const float m = mu[b * Z + j], lv = logvar[b * Z + j];
        k += 1.f + lv - m * m - expf(lv);
    }
    out[b] = -0.5f * k;
}
__global__ void kld_bwd_kernel(int B, int Z, const float *__restrict__ mu,
                               const float *__restrict__ logvar, const float *__restrict__ gout,
                               float *d_mu, float *d_logvar) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * Z) return;
    const float g = gout[i / Z];
    if (d_mu) d_mu[i] = g * mu[i];
    if (d_logvar) d_logvar[i] = g * 0.5f * (expf(logvar[i]) - 1.f);
}

// log sigma read from device memory (fp64 when ls_f64, else fp32) and sigma = its exp as torch forms log_sigma.exp(): in
// the scalar's own precision (the fp32 exp correctly rounded from fp64), then converted to the arithmetic's type
template <typename AT>
__device__ __forceinline__ void device_sigma(const void *ls_dev, int ls_f64, AT &ls, AT &sg) {
    const double l = ls_f64 ? *reinterpret_cast<const double *>(ls_dev) : (double)*reinterpret_cast<const float *>(ls_dev);
    ls = (AT)l;
    sg = ls_f64 ? (AT)exp(l) : (AT)(float)exp(l);
}

// ls_dev: log sigma from device memory (device_sigma); NULL: log_sigma / sigma from the host
template <typename XT>
__global__ void nll_fwd_kernel(int64_t n, const float *__restrict__ mu, const XT *__restrict__ x,
                               float log_sigma, float sigma, const void *__restrict__ ls_dev, int ls_f64, XT *out) {
    typedef typename AccT<XT>::type AT;
    AT ls = (AT)log_sigma, sg = (AT)sigma;
    if (ls_dev) device_sigma(ls_dev, ls_f64, ls, sg);
    const AT cst = ls + (AT)MVB_HALF_LOG_2PI;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const AT t = ((AT)x[i] - (AT)mu[i]) / sg;
        out[i] = (XT)((AT)0.5 * t * t + cst);
    }
}
template <typename XT>
__global__ void nll_bwd_kernel(int64_t n, const float *__restrict__ mu, const XT *__restrict__ x,
                               float sigma, const XT *__restrict__ gout, float *d_mu) {
    typedef typename AccT<XT>::type AT;
    const AT sg2 = (AT)sigma * (AT)sigma;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        d_mu[i] = (float)((AT)gout[i] * ((AT)mu[i] - (AT)x[i]) / sg2);
}

// gaussian_nll backward with a device log sigma: d_mu as nll_bwd_kernel, and per-block partials of
// d log_sigma = sum_i g_i (1 - ((x_i - mu_i)/sigma)^2) (fp64, fixed grid-stride order and tree) for an ordered finalize
template <typename XT>
__global__ void __launch_bounds__(256)
nll_sigma_bwd_kernel(int64_t n, const float *__restrict__ mu, const XT *__restrict__ x, const void *__restrict__ ls_dev,
                     int ls_f64, const XT *__restrict__ gout, float *d_mu, double *__restrict__ partial) {
    typedef typename AccT<XT>::type AT;
    __shared__ double sh[256];
    AT ls, sg;
    device_sigma(ls_dev, ls_f64, ls, sg);
    const AT sg2 = sg * sg;
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const AT g = (AT)gout[i], d = (AT)x[i] - (AT)mu[i];
        d_mu[i] = (float)(-g * d / sg2);
        const double t = (double)(d / sg);
        acc += (double)g * (1.0 - t * t);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}

__global__ void __launch_bounds__(256) ordered_sum_kernel(int n, const double *__restrict__ partial, double *out) {
    __shared__ double sh[256];
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) acc += partial[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if (threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0];
}

// ---- importance-weighted log-likelihood estimate: log p(x | y) from S posterior samples per mesh ---------------------
// a warp per (mesh b, sample s) row r = b S + s: the decoder input zcat[r] = cat(y_b, z) with z the expression of
// reparam_fwd_kernel, and log r = log q(z | x, y) - log p(z) = sum_j (-eps_j^2/2 - logvar_j/2 + z_j^2/2) in fp64 (the
// 0.5 log(2 pi) terms cancel), lane-strided with a fixed xor tree
__global__ void __launch_bounds__(256)
iw_sample_kernel(int B, int S, int Z, int C, const float *__restrict__ mu, const float *__restrict__ logvar,
                 const float *__restrict__ eps, const int64_t *__restrict__ y, float *__restrict__ zcat, double *__restrict__ log_r) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= (int64_t)B * S) return;
    const int64_t b = r / S;
    const float *m = mu + b * Z, *lv = logvar + b * Z, *e = eps + r * Z;
    float *out = zcat + r * (C + Z);
    for (int c = lane; c < C; c += 32) out[c] = (float)y[b * C + c];
    double acc = 0.0;
    for (int j = lane; j < Z; j += 32) {
        const float ej = e[j], lj = lv[j];
        const float z = fmaf(ej, expf(0.5f * lj), m[j]);
        out[C + j] = z;
        const double ed = ej, zd = z;
        acc += 0.5 * (zd * zd - ed * ed) - 0.5 * (double)lj;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) log_r[r] = acc;
}

// a warp per reconstruction j = b S + s: SSE_j = the ordered sum of the vertex-chunk partials (the order of
// vae_loss_finalize_kernel's phase 1), log p(x_b | z_j) = -SSE_j / (2 sigma^2) - n (log sigma + 0.5 log(2 pi)) with log sigma
// read from device memory, log w = log p - log r, written to column s0 + s of row b of log_w [B, S_total]
__global__ void __launch_bounds__(256)
iw_log_weights_finalize_kernel(int BS, int S, int S_total, int s0, int nchunks, double n_elem, const double *__restrict__ partial,
                               const double *__restrict__ log_sigma, const double *__restrict__ log_r, double *__restrict__ log_w) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= BS) return;
    double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
    int ch = lane;
    for (; ch + 96 < nchunks; ch += 128) {
        r0 += partial[(int64_t)ch * BS + j];
        r1 += partial[(int64_t)(ch + 32) * BS + j];
        r2 += partial[(int64_t)(ch + 64) * BS + j];
        r3 += partial[(int64_t)(ch + 96) * BS + j];
    }
    for (; ch < nchunks; ch += 32) r0 += partial[(int64_t)ch * BS + j];
    double sse = (r0 + r1) + (r2 + r3);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, off);
    if (lane == 0) {
        const double ls = *log_sigma;
        const double log_px_z = -(0.5 * sse * exp(-2.0 * ls)) - n_elem * (ls + MVB_HALF_LOG_2PI);
        const int b = j / S, s = j - b * S;
        log_w[(int64_t)b * S_total + s0 + s] = log_px_z - log_r[j];
    }
}

// a warp per mesh over its S log-weights (lane-strided, fixed xor trees; the max is exact in any order):
// log_px = max + log sum_s exp(log w - max) - log S, elbo = mean_s log w, ess = (sum e)^2 / sum e^2 with e = exp(log w - max)
__global__ void __launch_bounds__(256)
iw_reduce_kernel(int B, int S, const double *__restrict__ log_w, double *__restrict__ log_px, double *__restrict__ elbo,
                 double *__restrict__ ess, double *__restrict__ log_w_out) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const double *w = log_w + (int64_t)b * S;
    double mx = -INFINITY, sum = 0.0;
    for (int s = lane; s < S; s += 32) {
        const double v = w[s];
        mx = fmax(mx, v);
        sum += v;
        if (log_w_out) log_w_out[(int64_t)b * S + s] = v;
    }
    double e1 = 0.0, e2 = 0.0;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        sum += __shfl_xor_sync(0xffffffffu, sum, off);
    }
    for (int s = lane; s < S; s += 32) {
        const double t = exp(w[s] - mx);
        e1 += t;
        e2 += t * t;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        e1 += __shfl_xor_sync(0xffffffffu, e1, off);
        e2 += __shfl_xor_sync(0xffffffffu, e2, off);
    }
    if (lane == 0) {
        log_px[b] = mx + log(e1) - log((double)S);
        elbo[b] = sum / (double)S;
        ess[b] = e1 * e1 / e2;
    }
}

static inline unsigned ew_grid(int64_t n, int threads) {
    int64_t b = (n + threads - 1) / threads;
    const int64_t cap = (int64_t)num_sms() * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

static void loss_tiles(int C, int ld, size_t xsize, int &VCH, int &BCH, size_t &smem) {
    VCH = 32;
    BCH = 32;
    smem = (size_t)VCH * BCH * (C * xsize + ld * 4);
    while (smem > 48 * 1024 && VCH > 1) {
        VCH /= 2;
        smem = (size_t)VCH * BCH * (C * xsize + ld * 4);
    }
}

}  // namespace mvb

using namespace mvb;

extern "C" size_t mvb_vae_loss_workspace_bytes(int B, int N) {
    // worst case VCH = 1 never happens for C <= 12; size for VCH >= 8 chunks, generous and tiny
    const size_t nch = (size_t)(N + 7) / 8;
    return nch * (size_t)B * sizeof(double);
}

extern "C" int mvb_vae_loss_fwd(int B, int N, int C, int Z, int ncls, const float *recon, int recon_ld,
                                const void *x_gt, int x_is_f64, const float *mu,
                                const float *logvar, const float *y_hat, const int64_t *y,
                                float log_sigma, double *loss, float *kld, double *rec,
                                int64_t *correct, float *dnll, void *workspace,
                                size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(B > 0 && N > 0 && C > 0 && Z > 0 && ncls > 0, "vae_loss_fwd: bad sizes");
    MVB_REQUIRE(recon_ld >= C, "vae_loss_fwd: recon_ld=%d < C=%d", recon_ld, C);
    MVB_REQUIRE(recon && x_gt && mu && logvar && y_hat && y && loss && kld && rec && correct && dnll && workspace,
                "vae_loss_fwd: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    int VCH, BCH;
    size_t smem;
    loss_tiles(C, recon_ld, x_is_f64 ? 8 : 4, VCH, BCH, smem);
    MVB_REQUIRE(VCH >= 8, "vae_loss_fwd: C=%d too large", C);
    const int nch = (N + VCH - 1) / VCH;
    if ((size_t)nch * B * sizeof(double) > workspace_bytes)
        return set_err(MVB_EWORKSPACE, "vae_loss_fwd: workspace %zu < %zu", workspace_bytes, (size_t)nch * B * sizeof(double));
    dim3 grid(nch, (B + BCH - 1) / BCH);
    const float sigma = expf(log_sigma);
    double *partial = reinterpret_cast<double *>(workspace);
    if (x_is_f64)
        launch_pdl(vae_rec_partial_kernel<double, false>, dim3(grid), dim3(256), smem, st, B, N, C, recon_ld, VCH, BCH, 1, recon, (const double *)x_gt, log_sigma, sigma, partial, dnll);
    else
        launch_pdl(vae_rec_partial_kernel<float, false>, dim3(grid), dim3(256), smem, st, B, N, C, recon_ld, VCH, BCH, 1, recon, (const float *)x_gt, log_sigma, sigma, partial, dnll);
    int rc = check_launch("mvb_vae_loss_fwd partial");
    if (rc) return rc;
    launch_pdl(vae_loss_finalize_kernel<false>, dim3(1), dim3(1024), 0, st, B, Z, ncls, nch, partial, mu, logvar, y_hat, y, loss, kld, rec,
               correct, 0, 0.0, (const float *)nullptr, (double *)nullptr);
    return check_launch("mvb_vae_loss_fwd finalize");
}

extern "C" int mvb_vae_loss_bwd(int B, int N, int C, int Z, int ncls, const float *dnll,
                                const float *mu, const float *logvar, const float *y_hat,
                                const int64_t *y, const double *gloss, float *d_recon, float *d_mu,
                                float *d_logvar, float *d_yhat, void *stream) {
    MVB_REQUIRE(B > 0 && N > 0 && C > 0 && gloss, "vae_loss_bwd: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    if (d_recon) {
        MVB_REQUIRE(dnll, "vae_loss_bwd: dnll is null");
        const int64_t n = (int64_t)N * B * C;
        if (n % 4 == 0 && aligned16(dnll) && aligned16(d_recon))
            launch_pdl(scale4_by_gloss_kernel<false>, dim3(ew_grid(n / 4, 256)), dim3(256), 0, st, n / 4, (const float4 *)dnll, gloss, 1.0 / B,
                       (const double *)nullptr, (float4 *)d_recon);
        else
            scale_by_gloss_kernel<false><<<ew_grid(n, 256), 256, 0, st>>>(n, dnll, gloss, 1.0 / B, nullptr, d_recon);
        int rc = check_launch("mvb_vae_loss_bwd recon");
        if (rc) return rc;
    }
    if (d_mu || d_logvar || d_yhat) {
        MVB_REQUIRE(mu && logvar && y_hat && y, "vae_loss_bwd: null latent pointers");
        const int n = B * (Z > 1 ? Z : 1);
        launch_pdl(vae_loss_bwd_small_kernel, dim3((n + 127) / 128), dim3(128), 0, st, B, Z, ncls, mu, logvar, y_hat, y, gloss, d_mu, d_logvar, d_yhat,
                   (const double *)nullptr, (float *)nullptr);
        return check_launch("mvb_vae_loss_bwd latent");
    }
    return MVB_OK;
}

extern "C" int mvb_vae_loss_sigma_fwd(int B, int N, int C, int Z, int ncls, const float *recon, int recon_ld,
                                      const void *x_gt, int x_is_f64, const float *mu, const float *logvar,
                                      const float *y_hat, const int64_t *y, int sigma_mode, const float *s_param,
                                      double *sigma_state, double *loss, float *kld, double *rec, int64_t *correct,
                                      float *dnll, void *workspace, size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(B > 0 && N > 0 && C > 0 && Z > 0 && ncls > 0, "vae_loss_sigma_fwd: bad sizes");
    MVB_REQUIRE(recon_ld >= C, "vae_loss_sigma_fwd: recon_ld=%d < C=%d", recon_ld, C);
    MVB_REQUIRE(sigma_mode == MVB_SIGMA_OPTIMAL || sigma_mode == MVB_SIGMA_LEARNED, "vae_loss_sigma_fwd: sigma_mode=%d", sigma_mode);
    MVB_REQUIRE(sigma_mode != MVB_SIGMA_LEARNED || s_param, "vae_loss_sigma_fwd: learned sigma without s_param");
    MVB_REQUIRE(recon && x_gt && mu && logvar && y_hat && y && sigma_state && loss && kld && rec && correct && dnll && workspace,
                "vae_loss_sigma_fwd: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    int VCH, BCH;
    size_t smem;
    loss_tiles(C, recon_ld, x_is_f64 ? 8 : 4, VCH, BCH, smem);
    MVB_REQUIRE(VCH >= 8, "vae_loss_sigma_fwd: C=%d too large", C);
    const int nch = (N + VCH - 1) / VCH;
    if ((size_t)nch * B * sizeof(double) > workspace_bytes)
        return set_err(MVB_EWORKSPACE, "vae_loss_sigma_fwd: workspace %zu < %zu", workspace_bytes, (size_t)nch * B * sizeof(double));
    dim3 grid(nch, (B + BCH - 1) / BCH);
    double *partial = reinterpret_cast<double *>(workspace);
    if (x_is_f64)
        launch_pdl(vae_rec_partial_kernel<double, true>, dim3(grid), dim3(256), smem, st, B, N, C, recon_ld, VCH, BCH, 1, recon, (const double *)x_gt, 0.f, 1.f, partial, dnll);
    else
        launch_pdl(vae_rec_partial_kernel<float, true>, dim3(grid), dim3(256), smem, st, B, N, C, recon_ld, VCH, BCH, 1, recon, (const float *)x_gt, 0.f, 1.f, partial, dnll);
    int rc = check_launch("mvb_vae_loss_sigma_fwd partial");
    if (rc) return rc;
    launch_pdl(vae_loss_finalize_kernel<true>, dim3(1), dim3(1024), 0, st, B, Z, ncls, nch, partial, mu, logvar, y_hat, y, loss, kld, rec,
               correct, sigma_mode, (double)N * C, s_param, sigma_state);
    return check_launch("mvb_vae_loss_sigma_fwd finalize");
}

extern "C" int mvb_vae_loss_sigma_bwd(int B, int N, int C, int Z, int ncls, const float *dnll, const double *sigma_state,
                                      const float *mu, const float *logvar, const float *y_hat, const int64_t *y,
                                      const double *gloss, float *d_recon, float *d_mu, float *d_logvar, float *d_yhat,
                                      float *d_s, void *stream) {
    MVB_REQUIRE(B > 0 && N > 0 && C > 0 && gloss && sigma_state, "vae_loss_sigma_bwd: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const double *coef = sigma_state + 4, *d_t = sigma_state + 5;
    if (d_recon) {
        MVB_REQUIRE(dnll, "vae_loss_sigma_bwd: dnll is null");
        const int64_t n = (int64_t)N * B * C;
        if (n % 4 == 0 && aligned16(dnll) && aligned16(d_recon))
            launch_pdl(scale4_by_gloss_kernel<true>, dim3(ew_grid(n / 4, 256)), dim3(256), 0, st, n / 4, (const float4 *)dnll, gloss, 1.0 / B, coef,
                       (float4 *)d_recon);
        else
            scale_by_gloss_kernel<true><<<ew_grid(n, 256), 256, 0, st>>>(n, dnll, gloss, 1.0 / B, coef, d_recon);
        int rc = check_launch("mvb_vae_loss_sigma_bwd recon");
        if (rc) return rc;
    }
    if (d_mu || d_logvar || d_yhat || d_s) {
        MVB_REQUIRE(mu && logvar && y_hat && y, "vae_loss_sigma_bwd: null latent pointers");
        const int n = B * (Z > 1 ? Z : 1);
        launch_pdl(vae_loss_bwd_small_kernel, dim3((n + 127) / 128), dim3(128), 0, st, B, Z, ncls, mu, logvar, y_hat, y, gloss, d_mu, d_logvar, d_yhat,
                   d_t, d_s);
        return check_launch("mvb_vae_loss_sigma_bwd latent");
    }
    return MVB_OK;
}

extern "C" int mvb_vae_reparam_fwd(int64_t n, const float *mu, const float *logvar,
                                   const float *eps, float *z, void *stream) {
    MVB_REQUIRE(n >= 0 && mu && logvar && eps && z, "reparam_fwd: bad arguments");
    if (n == 0) return MVB_OK;
    reparam_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, mu, logvar, eps, z);
    return check_launch("mvb_vae_reparam_fwd");
}

extern "C" int mvb_vae_reparam_bwd(int64_t n, const float *logvar, const float *eps,
                                   const float *dz, float *dmu, float *dlogvar, void *stream) {
    MVB_REQUIRE(n >= 0 && logvar && eps && dz, "reparam_bwd: bad arguments");
    if (n == 0) return MVB_OK;
    reparam_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, logvar, eps, dz, dmu, dlogvar);
    return check_launch("mvb_vae_reparam_bwd");
}

extern "C" int mvb_kld_fwd(int B, int Z, const float *mu, const float *logvar, float *out, void *stream) {
    MVB_REQUIRE(B > 0 && Z > 0 && mu && logvar && out, "kld_fwd: bad arguments");
    kld_fwd_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(B, Z, mu, logvar, out);
    return check_launch("mvb_kld_fwd");
}

extern "C" int mvb_kld_bwd(int B, int Z, const float *mu, const float *logvar, const float *gout,
                           float *d_mu, float *d_logvar, void *stream) {
    MVB_REQUIRE(B > 0 && Z > 0 && mu && logvar && gout, "kld_bwd: bad arguments");
    kld_bwd_kernel<<<(B * Z + 127) / 128, 128, 0, (cudaStream_t)stream>>>(B, Z, mu, logvar, gout, d_mu, d_logvar);
    return check_launch("mvb_kld_bwd");
}

extern "C" int mvb_gaussian_nll_fwd(int64_t n, const float *mu, const void *x, int x_is_f64,
                                    float log_sigma, void *out, void *stream) {
    MVB_REQUIRE(n >= 0 && mu && x && out, "gaussian_nll_fwd: bad arguments");
    if (n == 0) return MVB_OK;
    const float sigma = expf(log_sigma);
    if (x_is_f64)
        nll_fwd_kernel<double><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(n, mu, (const double *)x, log_sigma, sigma, nullptr, 0, (double *)out);
    else
        nll_fwd_kernel<float><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(n, mu, (const float *)x, log_sigma, sigma, nullptr, 0, (float *)out);
    return check_launch("mvb_gaussian_nll_fwd");
}

extern "C" int mvb_gaussian_nll_bwd(int64_t n, const float *mu, const void *x, int x_is_f64,
                                    float log_sigma, const void *gout, float *d_mu, void *stream) {
    MVB_REQUIRE(n >= 0 && mu && x && gout && d_mu, "gaussian_nll_bwd: bad arguments");
    if (n == 0) return MVB_OK;
    const float sigma = expf(log_sigma);
    if (x_is_f64)
        nll_bwd_kernel<double><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(n, mu, (const double *)x, sigma, (const double *)gout, d_mu);
    else
        nll_bwd_kernel<float><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(n, mu, (const float *)x, sigma, (const float *)gout, d_mu);
    return check_launch("mvb_gaussian_nll_bwd");
}

extern "C" int mvb_gaussian_nll_sigma_fwd(int64_t n, const float *mu, const void *x, int x_is_f64, const void *log_sigma,
                                          int ls_is_f64, void *out, void *stream) {
    MVB_REQUIRE(n >= 0 && mu && x && log_sigma && out, "gaussian_nll_sigma_fwd: bad arguments");
    if (n == 0) return MVB_OK;
    if (x_is_f64)
        nll_fwd_kernel<double><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(n, mu, (const double *)x, 0.f, 1.f, log_sigma, ls_is_f64,
                                                                                   (double *)out);
    else
        nll_fwd_kernel<float><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(n, mu, (const float *)x, 0.f, 1.f, log_sigma, ls_is_f64,
                                                                                  (float *)out);
    return check_launch("mvb_gaussian_nll_sigma_fwd");
}

extern "C" size_t mvb_gaussian_nll_sigma_workspace_bytes(int64_t n) { return (size_t)ew_grid(n, 256) * sizeof(double); }

extern "C" int mvb_gaussian_nll_sigma_bwd(int64_t n, const float *mu, const void *x, int x_is_f64, const void *log_sigma,
                                          int ls_is_f64, const void *gout, float *d_mu, double *d_log_sigma, void *workspace,
                                          size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(n >= 0 && mu && x && log_sigma && gout && d_mu && d_log_sigma && workspace, "gaussian_nll_sigma_bwd: bad arguments");
    const unsigned grid = ew_grid(n, 256);
    MVB_REQUIRE(workspace_bytes >= (size_t)grid * sizeof(double), "gaussian_nll_sigma_bwd: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    double *partial = reinterpret_cast<double *>(workspace);
    if (x_is_f64)
        nll_sigma_bwd_kernel<double><<<grid, 256, 0, st>>>(n, mu, (const double *)x, log_sigma, ls_is_f64, (const double *)gout, d_mu, partial);
    else
        nll_sigma_bwd_kernel<float><<<grid, 256, 0, st>>>(n, mu, (const float *)x, log_sigma, ls_is_f64, (const float *)gout, d_mu, partial);
    int rc = check_launch("mvb_gaussian_nll_sigma_bwd");
    if (rc) return rc;
    ordered_sum_kernel<<<1, 256, 0, st>>>((int)grid, partial, d_log_sigma);
    return check_launch("mvb_gaussian_nll_sigma_bwd sum");
}

extern "C" size_t mvb_recon_error_workspace_bytes(int B, int N) { return (size_t)2 * ((N + 255) / 256) * B * sizeof(double); }

extern "C" int mvb_recon_error(int B, int N, int ld, const float *recon, const float *mean, const float *std, const double *s,
                               const double *R, const double *m, const void *gt, int gt_is_f64, double *mean_err, double *max_err,
                               float *vertex_err, float *mesh_out, void *workspace, size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(B > 0 && N > 0 && ld >= 3 && recon && mean && std && s && R && m && mean_err && max_err && workspace,
                "recon_error: bad arguments");
    MVB_REQUIRE(gt || mesh_out, "recon_error: neither a ground truth nor a mesh output");
    const int nch = (N + 255) / 256;
    MVB_REQUIRE(workspace_bytes >= mvb_recon_error_workspace_bytes(B, N), "recon_error: workspace too small");
    double *psum = reinterpret_cast<double *>(workspace);
    double *pmax = psum + (size_t)nch * B;
    cudaStream_t st = (cudaStream_t)stream;
    if (gt_is_f64)
        mvb::recon_error_partial_kernel<double><<<dim3(nch, B), 256, 0, st>>>(B, N, ld, recon, mean, std, s, R, m, (const double *)gt, psum, pmax, vertex_err, mesh_out);
    else
        mvb::recon_error_partial_kernel<float><<<dim3(nch, B), 256, 0, st>>>(B, N, ld, recon, mean, std, s, R, m, (const float *)gt, psum, pmax, vertex_err, mesh_out);
    int rc = mvb::check_launch("mvb_recon_error partial");
    if (rc) return rc;
    mvb::recon_error_finalize_kernel<<<(B + 127) / 128, 128, 0, st>>>(B, N, nch, psum, pmax, mean_err, max_err);
    return mvb::check_launch("mvb_recon_error finalize");
}

extern "C" int mvb_epoch_meter_add(int B, const void *loss, int loss_is_f64, const float *kld, const void *rec, int rec_is_f64,
                                   const int64_t *correct, const double *mean_err, double *acc, void *stream) {
    MVB_REQUIRE(B > 0 && loss && kld && rec && acc, "epoch_meter_add: bad arguments");
    const double *l64 = loss_is_f64 ? (const double *)loss : nullptr;
    const float *l32 = loss_is_f64 ? nullptr : (const float *)loss;
    if (rec_is_f64)
        mvb::epoch_meter_kernel<double><<<1, 256, 0, (cudaStream_t)stream>>>(B, l64, l32, kld, (const double *)rec, correct, mean_err, acc);
    else
        mvb::epoch_meter_kernel<float><<<1, 256, 0, (cudaStream_t)stream>>>(B, l64, l32, kld, (const float *)rec, correct, mean_err, acc);
    return mvb::check_launch("mvb_epoch_meter_add");
}

extern "C" int mvb_iw_sample(int B, int S, int Z, int C, const float *mu, const float *logvar, const float *eps, const int64_t *y,
                             float *zcat, double *log_r, void *stream) {
    MVB_REQUIRE(B > 0 && S > 0 && Z > 0 && C > 0, "iw_sample: bad sizes B=%d S=%d Z=%d C=%d", B, S, Z, C);
    MVB_REQUIRE(mu && logvar && eps && y && zcat && log_r, "iw_sample: null pointer");
    const int64_t rows = (int64_t)B * S;
    MVB_REQUIRE(rows <= (int64_t)1 << 30, "iw_sample: B*S=%lld too large", (long long)rows);
    mvb::launch_pdl(mvb::iw_sample_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, (cudaStream_t)stream, B, S, Z, C, mu, logvar,
                    eps, y, zcat, log_r);
    return mvb::check_launch("mvb_iw_sample");
}

extern "C" size_t mvb_iw_log_weights_workspace_bytes(int B, int S, int N) { return mvb_vae_loss_workspace_bytes(B * S, N); }

extern "C" int mvb_iw_log_weights(int B, int S, int N, int C, const float *recon, int recon_ld, const void *x_gt, int x_is_f64,
                                  const double *log_sigma, const double *log_r, int S_total, int s0, double *log_w, void *workspace,
                                  size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(B > 0 && S > 0 && N > 0 && C > 0, "iw_log_weights: bad sizes B=%d S=%d N=%d C=%d", B, S, N, C);
    MVB_REQUIRE(recon_ld >= C, "iw_log_weights: recon_ld=%d < C=%d", recon_ld, C);
    MVB_REQUIRE(s0 >= 0 && S_total >= s0 + S, "iw_log_weights: columns [%d, %d) outside [0, %d)", s0, s0 + S, S_total);
    MVB_REQUIRE(recon && x_gt && log_sigma && log_r && log_w && workspace, "iw_log_weights: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    int VCH, BCH;
    size_t smem;
    mvb::loss_tiles(C, recon_ld, x_is_f64 ? 8 : 4, VCH, BCH, smem);
    MVB_REQUIRE(VCH >= 8, "iw_log_weights: C=%d too large", C);
    // the partial kernel's grid.y walks the B*S reconstructions in tiles of BCH (at most 65535 tiles)
    MVB_REQUIRE(((int64_t)B * S + BCH - 1) / BCH <= 65535, "iw_log_weights: B*S=%lld reconstructions per call, at most %d: decode fewer "
                "samples at a time", (long long)B * S, 65535 * BCH);
    const int BS = B * S;
    const int nch = (N + VCH - 1) / VCH;
    if ((size_t)nch * BS * sizeof(double) > workspace_bytes)
        return mvb::set_err(MVB_EWORKSPACE, "iw_log_weights: workspace %zu < %zu", workspace_bytes, (size_t)nch * BS * sizeof(double));
    dim3 grid(nch, (BS + BCH - 1) / BCH);
    double *partial = reinterpret_cast<double *>(workspace);
    if (x_is_f64)
        mvb::launch_pdl(mvb::vae_rec_partial_kernel<double, true>, grid, dim3(256), smem, st, BS, N, C, recon_ld, VCH, BCH, S, recon,
                        (const double *)x_gt, 0.f, 1.f, partial, (float *)nullptr);
    else
        mvb::launch_pdl(mvb::vae_rec_partial_kernel<float, true>, grid, dim3(256), smem, st, BS, N, C, recon_ld, VCH, BCH, S, recon,
                        (const float *)x_gt, 0.f, 1.f, partial, (float *)nullptr);
    int rc = mvb::check_launch("mvb_iw_log_weights partial");
    if (rc) return rc;
    mvb::launch_pdl(mvb::iw_log_weights_finalize_kernel, dim3((unsigned)((BS + 7) / 8)), dim3(256), 0, st, BS, S, S_total, s0, nch,
                    (double)N * C, (const double *)partial, log_sigma, log_r, log_w);
    return mvb::check_launch("mvb_iw_log_weights finalize");
}

extern "C" int mvb_iw_reduce(int B, int S, const double *log_w, double *log_px, double *elbo, double *ess, double *log_w_out,
                             void *stream) {
    MVB_REQUIRE(B > 0 && S > 0 && log_w && log_px && elbo && ess, "iw_reduce: bad arguments");
    mvb::launch_pdl(mvb::iw_reduce_kernel, dim3((unsigned)((B + 7) / 8)), dim3(256), 0, (cudaStream_t)stream, B, S, log_w, log_px, elbo,
                    ess, log_w_out);
    return mvb::check_launch("mvb_iw_reduce");
}

extern "C" int mvb_pack_vertex_major(int B, int N, int C, int Cp, const float *x, float *out, void *stream) {
    MVB_REQUIRE(B > 0 && N > 0 && C > 0 && Cp >= C && C <= 8 && x && out, "pack_vertex_major: bad arguments");
    mvb::launch_pdl(mvb::pack_vertex_major_kernel, dim3((N + 31) / 32, (B + 7) / 8), dim3(256), 0, (cudaStream_t)stream, B, N, C, Cp, x, out);
    return mvb::check_launch("mvb_pack_vertex_major");
}
