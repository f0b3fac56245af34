// Dense per-row contractions of the Chebyshev convolution, FP32 FFMA path (strict 1e-4 parity):
//
//  * contract_kernel : out[row, :] = act( [T_0 | T_1 | ... | T_{K-1}][row, :] . W + bias )
//      forward  : K input planes of width Fin, W = weight[K*Fin, Fout]      (nn/conv.py:559,566,571,575)
//      backward : 1 input plane (dY, width Fout), W = weight^T [Fout, K*Fin], K output planes
//                 P_k = dY W_k^T  (autograd of the K matmuls)
//  * wgrad_kernel    : dW[K*Fin, Fout] = [T_0|...|T_{K-1}]^T dY, db = 1^T dY, reduced over the
//      N*B rows with a fixed tile->CTA map and an ordered second pass (deterministic, no atomics).
//
// Both stage a tile of rows in shared memory with fully coalesced 16-byte loads (a tile of R
// consecutive (vertex, mesh) rows of one plane is one contiguous R*Fin*4-byte run in the
// vertex-major layout), rows padded to a stride == 4 (mod 32) words so the 128-bit shared loads
// of 8 consecutive rows hit 32 distinct banks.  Each thread owns a TR x 4 (resp. 4 x 4) register
// tile.  Roofline: reads K*u, writes o (SURVEY.md 8(d)); at 6.9 FLOP/B the FFMA pipe, not HBM,
// is the practical bound - the tcgen05 kind::tf32 variant is the planned replacement.
#include "mvb_internal.cuh"

namespace mvb {

static inline int round4(int v) { return (v + 3) & ~3; }
static inline int pad_ld(int m4) {  // smallest ld >= m4 with ld % 32 == 4
    int ld = (m4 / 32) * 32 + 4;
    while (ld < m4) ld += 32;
    return ld;
}

// Stage nr rows of all input planes into Ts[r*LD + p*in_w + i]; plane 0 optionally masked.
__device__ __forceinline__ void stage_planes(float *Ts, int LD, int64_t rows, int64_t row0, int nr,
                                             int in_planes, int in_w, const float *in0,
                                             const float *in_rest, const float *mask, bool vec,
                                             int tid, int nthreads) {
    for (int p = 0; p < in_planes; ++p) {
        const float *src = (p == 0 ? in0 : in_rest + (int64_t)(p - 1) * rows * in_w) + row0 * in_w;
        const float *msk = (p == 0 && mask) ? mask + row0 * in_w : nullptr;
        if (vec) {
            const int q4 = in_w >> 2;
            const int n4 = nr * q4;
            const float4 *s4 = reinterpret_cast<const float4 *>(src);
            const float4 *m4 = reinterpret_cast<const float4 *>(msk);
            for (int base = 0; base < n4; base += 4 * nthreads) {      // 4 independent loads in flight
                float4 v[4], mk[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = base + u * nthreads + tid;
                    if (i < n4) {
                        v[u] = __ldg(s4 + i);
                        if (msk) mk[u] = __ldg(m4 + i);
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = base + u * nthreads + tid;
                    if (i < n4) {
                        const int r = i / q4, q = i - r * q4;
                        if (msk) {
                            v[u].x = mk[u].x > 0.f ? v[u].x : 0.f;
                            v[u].y = mk[u].y > 0.f ? v[u].y : 0.f;
                            v[u].z = mk[u].z > 0.f ? v[u].z : 0.f;
                            v[u].w = mk[u].w > 0.f ? v[u].w : 0.f;
                        }
                        *reinterpret_cast<float4 *>(Ts + r * LD + p * in_w + 4 * q) = v[u];
                    }
                }
            }
        } else {
            const int n = nr * in_w;
            for (int base = 0; base < n; base += 4 * nthreads) {
                float v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = base + u * nthreads + tid;
                    if (i < n) {
                        v[u] = __ldg(src + i);
                        if (msk) v[u] = __ldg(msk + i) > 0.f ? v[u] : 0.f;
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = base + u * nthreads + tid;
                    if (i < n) {
                        const int r = i / in_w, q = i - r * in_w;
                        Ts[r * LD + p * in_w + q] = v[u];
                    }
                }
            }
        }
    }
}

template <int TR>
__global__ void __launch_bounds__(512, 1)
contract_kernel(ContractArgs a, int M, int Nn, int M4, int N4, int LD, int R, int NT,
                int in_vec, int out_vec) {
    extern __shared__ float4 smem4[];
    float *Ws = reinterpret_cast<float *>(smem4);  // [M4][N4]
    float *Ts = Ws + M4 * N4;                      // [R][LD]
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int RG = R / TR;
    const int ni = tid % NT, rg = tid / NT;

    // W tile; with w_fold = K > 1 the K weight blocks are folded with the Chebyshev values at 0,
    // c_k = cos(k pi/2) = 1,0,-1,0,...: rows of the operator without entries see sum_k c_k W_k
    const int nfold = a.w_fold > 1 ? a.w_fold : 1;
    for (int base = 0; base < M4 * N4; base += 4 * nthreads) {          // 4 independent loads in flight
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * nthreads + tid;
            v[u] = 0.f;
            if (i < M4 * N4) {
                const int m = i / N4, n = i - m * N4;
                if (m < M && n < Nn) {
                    if (a.w_transposed == 2) {      // per-plane transposed: W[k][n][o], m = k*in_w + o
                        const int k = m / a.in_w, o = m - k * a.in_w;
                        v[u] = __ldg(a.wmat + ((int64_t)k * Nn + n) * a.in_w + o);
                    } else {
                        for (int k = 0; k < nfold; k += 2) {
                            const float wv = a.w_transposed ? __ldg(a.wmat + ((int64_t)k * Nn + n) * M + m)
                                                            : __ldg(a.wmat + ((int64_t)k * M + m) * Nn + n);
                            v[u] += (k & 2) ? -wv : wv;
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * nthreads + tid;
            if (i < M4 * N4) Ws[i] = v[u];
        }
    }
    if (M4 > M) {
        const int padw = M4 - M;
        for (int i = tid; i < R * padw; i += nthreads) Ts[(i / padw) * LD + M + (i % padw)] = 0.f;
    }
    float bv[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.bias) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (4 * ni + j < Nn) bv[j] = __ldg(a.bias + 4 * ni + j);
    }

    const int64_t ntiles = (a.rows + R - 1) / R;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t row0 = t * R;
        const int nr = (int)((a.rows - row0) < R ? (a.rows - row0) : R);
        __syncthreads();
        stage_planes(Ts, LD, a.rows, row0, nr, a.in_planes, a.in_w, a.in0, a.in_rest, a.mask,
                     in_vec != 0, tid, nthreads);
        __syncthreads();

        float acc[TR][4];
#pragma unroll
        for (int j = 0; j < TR; ++j) {
            acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
        }
        const float *wp = Ws + 4 * ni;
        const float *tp = Ts + rg * LD;
#pragma unroll 2
        for (int m0 = 0; m0 < M4; m0 += 4) {
            const float4 w0 = *reinterpret_cast<const float4 *>(wp + (m0 + 0) * N4);
            const float4 w1 = *reinterpret_cast<const float4 *>(wp + (m0 + 1) * N4);
            const float4 w2 = *reinterpret_cast<const float4 *>(wp + (m0 + 2) * N4);
            const float4 w3 = *reinterpret_cast<const float4 *>(wp + (m0 + 3) * N4);
#pragma unroll
            for (int j = 0; j < TR; ++j) {
                const float4 tv = *reinterpret_cast<const float4 *>(tp + j * RG * LD + m0);
                acc[j][0] = fmaf(tv.x, w0.x, acc[j][0]);
                acc[j][1] = fmaf(tv.x, w0.y, acc[j][1]);
                acc[j][2] = fmaf(tv.x, w0.z, acc[j][2]);
                acc[j][3] = fmaf(tv.x, w0.w, acc[j][3]);
                acc[j][0] = fmaf(tv.y, w1.x, acc[j][0]);
                acc[j][1] = fmaf(tv.y, w1.y, acc[j][1]);
                acc[j][2] = fmaf(tv.y, w1.z, acc[j][2]);
                acc[j][3] = fmaf(tv.y, w1.w, acc[j][3]);
                acc[j][0] = fmaf(tv.z, w2.x, acc[j][0]);
                acc[j][1] = fmaf(tv.z, w2.y, acc[j][1]);
                acc[j][2] = fmaf(tv.z, w2.z, acc[j][2]);
                acc[j][3] = fmaf(tv.z, w2.w, acc[j][3]);
                acc[j][0] = fmaf(tv.w, w3.x, acc[j][0]);
                acc[j][1] = fmaf(tv.w, w3.y, acc[j][1]);
                acc[j][2] = fmaf(tv.w, w3.z, acc[j][2]);
                acc[j][3] = fmaf(tv.w, w3.w, acc[j][3]);
            }
        }

        const int n0 = 4 * ni;
#pragma unroll
        for (int j = 0; j < TR; ++j) {
            const int rl = rg + j * RG;
            if (rl >= nr) continue;
            const int64_t row = row0 + rl;
            float o[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                o[q] = acc[j][q] + bv[q];
                if (a.relu) o[q] = o[q] > 0.f ? o[q] : 0.f;
            }
            if (out_vec) {
                const int p = n0 / a.out_w, jj = n0 - p * a.out_w;
                float *dst = a.out + ((int64_t)p * a.rows + row) * a.out_w + jj;
                *reinterpret_cast<float4 *>(dst) = make_float4(o[0], o[1], o[2], o[3]);
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int n = n0 + q;
                    if (n < Nn) {
                        const int p = n / a.out_w, jj = n - p * a.out_w;
                        a.out[((int64_t)p * a.rows + row) * a.out_w + jj] = o[q];
                    }
                }
            }
        }
    }
}

template <int TR>
static int launch_contract_t(const ContractArgs &a, int M, int Nn, int M4, int N4, int LD, int R,
                             int NT, int in_vec, int out_vec, int grid, int threads, size_t smem,
                             cudaStream_t st) {
    static DevFlags optin;
    {
        const int rc_attr = smem_optin(contract_kernel<TR>, 200 * 1024, optin, "contract");
        if (rc_attr) return rc_attr;
    }
    contract_kernel<TR><<<grid, threads, smem, st>>>(a, M, Nn, M4, N4, LD, R, NT, in_vec, out_vec);
    return check_launch("mvb contract");
}

int launch_contract(const ContractArgs &a, cudaStream_t st) {
    if (a.rows == 0) return MVB_OK;
    {   // tensor-core (tcgen05, 3xTF32) path for the 16/32-wide planes; FFMA below for everything else
        const int rc = launch_contract_tc(a, st);
        if (rc != 0) return rc < 0 ? rc : MVB_OK;
    }
    const int M = a.in_planes * a.in_w, Nn = a.out_planes * a.out_w;
    MVB_REQUIRE(M > 0 && Nn > 0, "contract: empty shape");
    MVB_REQUIRE(!a.row_sel, "contract: a row selection needs the tensor-core path (see mvb_cheb_sel_supported)");
    const int M4 = round4(M), N4 = round4(Nn), LD = pad_ld(M4), NT = N4 / 4;
    int TR = 4, R = 128;
    while ((R / TR) * NT > 512 && R > 32) R /= 2;
    MVB_REQUIRE((R / TR) * NT <= 512, "contract: output width %d too large", Nn);
    size_t smem = ((size_t)M4 * N4 + (size_t)R * LD) * sizeof(float);
    while (smem > 200 * 1024 && R > 8) {
        R /= 2;
        smem = ((size_t)M4 * N4 + (size_t)R * LD) * sizeof(float);
    }
    MVB_REQUIRE(smem <= 200 * 1024, "contract: K*Fin x Fout = %d x %d does not fit shared memory", M, Nn);
    if (R < 4 * TR) TR = 1;
    if ((R / TR) * NT < 128 && TR == 4) TR = 2;
    if ((R / TR) * NT < 128 && TR == 2) TR = 1;
    const int threads = (R / TR) * NT;
    const int in_vec = (a.in_w % 4 == 0) && aligned16(a.in0) && (a.in_planes == 1 || aligned16(a.in_rest)) &&
                       (!a.mask || aligned16(a.mask));
    const int out_vec = (a.out_w % 4 == 0) && aligned16(a.out);
    const int64_t ntiles = (a.rows + R - 1) / R;
    int64_t grid = ntiles;
    const int64_t cap = (int64_t)num_sms() * 4;
    if (grid > cap) grid = cap;
    switch (TR) {
        case 4: return launch_contract_t<4>(a, M, Nn, M4, N4, LD, R, NT, in_vec, out_vec, (int)grid, threads, smem, st);
        case 2: return launch_contract_t<2>(a, M, Nn, M4, N4, LD, R, NT, in_vec, out_vec, (int)grid, threads, smem, st);
        default: return launch_contract_t<1>(a, M, Nn, M4, N4, LD, R, NT, in_vec, out_vec, (int)grid, threads, smem, st);
    }
}

// ---------------------------------------------------------------------------------------------
// weight / bias gradient
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512)
wgrad_kernel(WgradArgs a, int M, int has_bias, int M4, int N4, int LDT, int R, int MT, int NT,
             int ngroups, int in_vec, int dy_vec) {
    extern __shared__ float4 smem4[];
    float *Ts = reinterpret_cast<float *>(smem4);  // [R][LDT]
    float *Ds = Ts + R * LDT;                      // [R][N4]
    float *red = Ds + R * N4;                      // [ngroups][M4*N4]
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int G = MT * NT;
    const int g = tid / G, tg = tid - g * G;
    const int mi = tg / NT, ni = tg - mi * NT;

    // constant columns of the T tile: the "ones" column that yields db, then zero padding
    {
        const int padw = M4 - M;
        for (int i = tid; i < R * padw; i += nthreads) {
            const int r = i / padw, c = M + (i - r * padw);
            Ts[r * LDT + c] = (has_bias && c == M) ? 1.f : 0.f;
        }
        const int padn = N4 - a.n_out;
        for (int i = tid; i < R * padn; i += nthreads) Ds[(i / padn) * N4 + a.n_out + (i % padn)] = 0.f;
    }

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    const int64_t ntiles = (a.rows + R - 1) / R;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t row0 = t * R;
        const int nr = (int)((a.rows - row0) < R ? (a.rows - row0) : R);
        __syncthreads();
        stage_planes(Ts, LDT, a.rows, row0, nr, a.in_planes, a.in_w, a.in0, a.in_rest, nullptr,
                     in_vec != 0, tid, nthreads);
        stage_planes(Ds, N4, a.rows, row0, nr, 1, a.n_out, a.dy, nullptr, a.mask, dy_vec != 0, tid,
                     nthreads);
        __syncthreads();
        if (g < ngroups) {
            for (int r = g; r < nr; r += ngroups) {
                const float4 tv = *reinterpret_cast<const float4 *>(Ts + r * LDT + 4 * mi);
                const float4 dv = *reinterpret_cast<const float4 *>(Ds + r * N4 + 4 * ni);
                acc[0][0] = fmaf(tv.x, dv.x, acc[0][0]);
                acc[0][1] = fmaf(tv.x, dv.y, acc[0][1]);
                acc[0][2] = fmaf(tv.x, dv.z, acc[0][2]);
                acc[0][3] = fmaf(tv.x, dv.w, acc[0][3]);
                acc[1][0] = fmaf(tv.y, dv.x, acc[1][0]);
                acc[1][1] = fmaf(tv.y, dv.y, acc[1][1]);
                acc[1][2] = fmaf(tv.y, dv.z, acc[1][2]);
                acc[1][3] = fmaf(tv.y, dv.w, acc[1][3]);
                acc[2][0] = fmaf(tv.z, dv.x, acc[2][0]);
                acc[2][1] = fmaf(tv.z, dv.y, acc[2][1]);
                acc[2][2] = fmaf(tv.z, dv.z, acc[2][2]);
                acc[2][3] = fmaf(tv.z, dv.w, acc[2][3]);
                acc[3][0] = fmaf(tv.w, dv.x, acc[3][0]);
                acc[3][1] = fmaf(tv.w, dv.y, acc[3][1]);
                acc[3][2] = fmaf(tv.w, dv.z, acc[3][2]);
                acc[3][3] = fmaf(tv.w, dv.w, acc[3][3]);
            }
        }
    }
    // ordered cross-group reduction, then one partial [M4*N4] per CTA
    if (g < ngroups) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) red[(size_t)g * M4 * N4 + (4 * mi + i) * N4 + 4 * ni + j] = acc[i][j];
    }
    __syncthreads();
    float *part = a.partials + (size_t)blockIdx.x * M4 * N4;
    for (int i = tid; i < M4 * N4; i += nthreads) {
        float s = 0.f;
        for (int q = 0; q < ngroups; ++q) s += red[(size_t)q * M4 * N4 + i];
        part[i] = s;
    }
}

// Ordered final reduction of the per-CTA partials.  Thread (tx, ty) of a 32 x 8 block sums
// partials ty, ty+8, ... of output element blockIdx.x*32 + tx (coalesced over tx); the 8 partial
// sums are then added in fixed order -> bit-reproducible.  Optional second partial set B holds
// S = x^T dY over the operator's EMPTY rows ([Fin+1, n_out], single plane): there T_k = c_k x, so
// dW_k += c_k S with c_k = cos(k pi/2)  (models/cheb_VAE.py:288 quirk path).
// a_tr != 0: partial set A comes from the adjoint-basis backward, [S_0|..|S_{K-1}]^T x, stored
// [K*fout][N4A] with N4A = round4(fin): element (k*fin + i, o) of dW is A[(k*fout + o)][i]; the bias
// gradient then comes from the column-sum kernel, not from a "ones" row of A.
__global__ void __launch_bounds__(1024)
wgrad_finalize_kernel(const float *__restrict__ partA, int nA, int M4A, const float *__restrict__ partB,
                      int nB, int M4B, int fin, int M, int n_out, int N4, int a_tr, int N4A, float *dweight,
                      float *dbias) {
    pdl_trigger();
    pdl_wait();
    // 32 outputs x 32 partial lanes per block: ~10 partials per thread instead of ~40 (each a dependent L2 round trip)
    __shared__ float red[32][33];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int total = (M + (dbias ? 1 : 0)) * n_out;
    const int i = blockIdx.x * 32 + tx;
    float s = 0.f;
    if (i < total) {
        const int m = i / n_out, n = i - m * n_out;
        const int k = m / fin;
        if (a_tr) {
            if (m < M) {
                const size_t off = (size_t)(k * n_out + n) * N4A + (m - k * fin);
                for (int p = ty; p < nA; p += 32) s += partA[(size_t)p * M4A * N4A + off];
            }
        } else {
            for (int p = ty; p < nA; p += 32) s += partA[(size_t)p * M4A * N4 + m * N4 + n];
        }
        if (nB > 0) {
            const int mb = (m < M) ? (m - k * fin) : fin;          // bias row of B sits at index fin
            const float c = (m < M) ? ((k & 1) ? 0.f : ((k & 2) ? -1.f : 1.f)) : 1.f;
            if (c != 0.f) {
                float sb = 0.f;
                for (int p = ty; p < nB; p += 32) sb += partB[(size_t)p * M4B * N4 + mb * N4 + n];
                s += c * sb;
            }
        }
    }
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && i < total) {
        float t = red[0][tx];
#pragma unroll
        for (int q = 1; q < 32; ++q) t += red[q][tx];
        const int m = i / n_out, n = i - m * n_out;
        if (m < M)
            dweight[(size_t)m * n_out + n] = t;
        else
            dbias[n] = t;
    }
}

// G = dY * [y > 0] (optional write) and per-block column sums of G (for db): rows x ncol, ncol % 4 == 0.
// Block = 256 threads = (ncol/4 column quads) x row lanes, a fixed chunk of rows per block; the
// per-block partial sums are added in block order by colsum_finalize_kernel: deterministic.
__global__ void __launch_bounds__(256)
mask_colsum_kernel(int64_t rows, int nq, const float4 *__restrict__ dy, const float4 *__restrict__ y,
                   float4 *__restrict__ g, float4 *__restrict__ part, int64_t rows_per_block) {
    pdl_trigger();
    pdl_wait();
    __shared__ float4 red[256];
    const int tid = threadIdx.x;
    const int q = tid % nq, rl = tid / nq, nrl = 256 / nq;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
    const int64_t r1 = (r0 + rows_per_block < rows) ? r0 + rows_per_block : rows;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rl < nrl)
        for (int64_t r = r0 + rl; r < r1; r += nrl) {
            float4 v = __ldg(dy + r * nq + q);
            if (y) {
                const float4 m = __ldg(y + r * nq + q);
                v.x = m.x > 0.f ? v.x : 0.f; v.y = m.y > 0.f ? v.y : 0.f; v.z = m.z > 0.f ? v.z : 0.f; v.w = m.w > 0.f ? v.w : 0.f;
                if (g) g[r * nq + q] = v;
            }
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
    red[tid] = s;
    __syncthreads();
    if (part && tid < nq) {
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int l = 0; l < nrl; ++l) {
            const float4 v = red[l * nq + tid];
            t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
        }
        part[(int64_t)blockIdx.x * nq + tid] = t;
    }
}

// db[c] = sum over the blocks' partials, one warp per column: lane l adds partials l, l+32, ... in
// order, then a fixed shuffle tree - deterministic, and ~nblocks/32 dependent loads instead of nblocks
__global__ void __launch_bounds__(256)
colsum_finalize_kernel(int nblocks, int ncol, const float *__restrict__ part, float *__restrict__ db) {
    pdl_trigger();
    pdl_wait();
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= ncol) return;
    float s = 0.f;
    for (int b = lane; b < nblocks; b += 32) s += part[(int64_t)b * ncol + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) db[c] = s;
}

int mask_colsum_blocks(int64_t rows) {
    int64_t nb = (rows + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 2;
    if (nb > cap) nb = cap;
    return (int)(nb < 1 ? 1 : nb);
}

// g (may be NULL when y is NULL: then G is dy itself), db (may be NULL), part: mask_colsum_blocks(rows)*ncol floats
int launch_mask_colsum(int64_t rows, int ncol, const float *dy, const float *y, float *g, float *db, float *part,
                       cudaStream_t st) {
    if (rows <= 0) return MVB_OK;
    if (!y && !db) return MVB_OK;
    MVB_REQUIRE(ncol % 4 == 0 && ncol <= 1024 && aligned16(dy) && (!y || aligned16(y)) && (!g || aligned16(g)) && aligned16(part),
                "mask_colsum: %d columns / alignment not supported", ncol);
    const int nb = mask_colsum_blocks(rows);
    const int64_t rpb = (rows + nb - 1) / nb;
    launch_pdl(mask_colsum_kernel, dim3(nb), dim3(256), 0, st, rows, ncol / 4, (const float4 *)dy, (const float4 *)y, (float4 *)g,
                                           db ? (float4 *)part : nullptr, rpb);
    int rc = check_launch("mvb mask_colsum");
    if (rc || !db) return rc;
    launch_pdl(colsum_finalize_kernel, dim3((ncol + 7) / 8), dim3(256), 0, st, nb, ncol, part, db);
    return check_launch("mvb colsum finalize");
}

static void wgrad_shape(int M, int n_out, int has_bias, int &M4, int &N4, int &LDT, int &MT, int &NT,
                        int &ngroups, int &R) {
    M4 = round4(M + (has_bias ? 1 : 0));
    N4 = round4(n_out);
    LDT = pad_ld(M4);
    MT = M4 / 4;
    NT = N4 / 4;
    const int G = MT * NT;
    ngroups = 256 / G;
    if (ngroups < 1) ngroups = 1;
    if (ngroups > 16) ngroups = 16;
    R = 64;
}

static int wgrad_grid(int64_t rows, int R) {
    int64_t ntiles = (rows + R - 1) / R;
    int64_t cap = (int64_t)num_sms() * 2;
    return (int)(ntiles < cap ? (ntiles < 1 ? 1 : ntiles) : cap);
}

size_t wgrad_partial_bytes(int M, int n_out) {
    int M4, N4, LDT, MT, NT, ng, R;
    wgrad_shape(M, n_out, 1, M4, N4, LDT, MT, NT, ng, R);
    return (size_t)num_sms() * 2 * M4 * N4 * sizeof(float);
}

// phase 1: per-CTA partials of [T_0|..|T_{P-1}|1]^T dY over a.rows rows; returns the number of
// partial blocks written and their row count M4 through nparts / m4_out
int launch_wgrad_partials(const WgradArgs &a, int has_bias, int *nparts, int *m4_out, cudaStream_t st) {
    const int M = a.in_planes * a.in_w;
    int M4, N4, LDT, MT, NT, ngroups, R;
    wgrad_shape(M, a.n_out, has_bias, M4, N4, LDT, MT, NT, ngroups, R);
    *m4_out = M4;
    *nparts = 0;
    if (a.rows <= 0) return MVB_OK;
    {
        const int rc = launch_wgrad_tc(a, has_bias, M4, N4, nparts, st);
        if (rc != 0) return rc < 0 ? rc : MVB_OK;
    }
    MVB_REQUIRE(!a.row_sel, "wgrad: a row selection needs the tensor-core path (see mvb_cheb_sel_supported)");
    const int G = MT * NT;
    MVB_REQUIRE(G <= 512, "wgrad: K*Fin x Fout = %d x %d too large for the register-tiled reduction", M, a.n_out);
    const int threads = G * ngroups;
    const int grid = wgrad_grid(a.rows, R);
    MVB_REQUIRE((size_t)grid * M4 * N4 * sizeof(float) <= a.partial_bytes, "wgrad: workspace too small");
    const size_t smem = ((size_t)R * LDT + (size_t)R * N4 + (size_t)ngroups * M4 * N4) * sizeof(float);
    MVB_REQUIRE(smem <= 200 * 1024, "wgrad: shared memory %zu too large", smem);
    static DevFlags optin;
    {
        const int rc_attr = smem_optin(wgrad_kernel, 200 * 1024, optin, "wgrad");
        if (rc_attr) return rc_attr;
    }
    const int in_vec = (a.in_w % 4 == 0) && aligned16(a.in0) && (a.in_planes == 1 || aligned16(a.in_rest));
    const int dy_vec = (a.n_out % 4 == 0) && aligned16(a.dy) && (!a.mask || aligned16(a.mask));
    wgrad_kernel<<<grid, threads, smem, st>>>(a, M, has_bias, M4, N4, LDT, R, MT, NT, ngroups, in_vec, dy_vec);
    *nparts = grid;
    return check_launch("mvb wgrad");
}

// ---------------------------------------------------------------------------------------------
// Closed-form rows (operator rows without entries: T_k = cos(k pi/2) x, api.cu) with narrow planes.
// The reference's output layer (16 -> 3 features, 99.6 % of its rows closed-form, models/cheb_VAE.py:288)
// is pure streaming: 80 bytes per row.  The 128-row tensor-core tiles spend their time in per-tile
// set-up there (31-39 us for 25 MB, in-graph timeline); these three FFMA kernels are bandwidth-bound.
//   Wf = sum_k cos(k pi/2) W_k  [Fin x Fout]  folded in shared memory at block start.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void fold_weights(float *Wf, const float *__restrict__ w, int K, int Fin, int Fout, int tid, int nthreads) {
    for (int i = tid; i < Fin * Fout; i += nthreads) {
        float v = 0.f;
        for (int k = 0; k < K; k += 2) {
            const float wv = __ldg(w + (int64_t)k * Fin * Fout + i);
            v += (k & 2) ? -wv : wv;
        }
        Wf[i] = v;
    }
}

// out[row, :] = act(x[row, :] Wf + b);  thread = (row, output quad)
__global__ void __launch_bounds__(256)
fold_rows_fwd_kernel(int64_t rows, int K, int Fin, int Fout, const float *__restrict__ x, const float *__restrict__ w,
                     const float *__restrict__ bias, int relu, float *__restrict__ out) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ float4 smem4[];
    float *Wf = reinterpret_cast<float *>(smem4);
    fold_weights(Wf, w, K, Fin, Fout, threadIdx.x, blockDim.x);
    __syncthreads();
    const int oq = Fout >> 2, iq = Fin >> 2;
    const int64_t total = rows * oq;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = t / oq;
        const int q = (int)(t - row * oq);
        const float4 *xr = reinterpret_cast<const float4 *>(x + row * Fin);
        float4 acc = bias ? __ldg(reinterpret_cast<const float4 *>(bias) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i4 = 0; i4 < iq; ++i4) {
            const float4 xv = __ldg(xr + i4);
            const float4 w0 = *reinterpret_cast<const float4 *>(Wf + (4 * i4 + 0) * Fout + 4 * q);
            const float4 w1 = *reinterpret_cast<const float4 *>(Wf + (4 * i4 + 1) * Fout + 4 * q);
            const float4 w2 = *reinterpret_cast<const float4 *>(Wf + (4 * i4 + 2) * Fout + 4 * q);
            const float4 w3 = *reinterpret_cast<const float4 *>(Wf + (4 * i4 + 3) * Fout + 4 * q);
            acc.x = fmaf(xv.x, w0.x, fmaf(xv.y, w1.x, fmaf(xv.z, w2.x, fmaf(xv.w, w3.x, acc.x))));
            acc.y = fmaf(xv.x, w0.y, fmaf(xv.y, w1.y, fmaf(xv.z, w2.y, fmaf(xv.w, w3.y, acc.y))));
            acc.z = fmaf(xv.x, w0.z, fmaf(xv.y, w1.z, fmaf(xv.z, w2.z, fmaf(xv.w, w3.z, acc.z))));
            acc.w = fmaf(xv.x, w0.w, fmaf(xv.y, w1.w, fmaf(xv.z, w2.w, fmaf(xv.w, w3.w, acc.w))));
        }
        if (relu) { acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f); }
        reinterpret_cast<float4 *>(out + row * Fout)[q] = acc;
    }
}

// dx[row, :] = g[row, :] Wf^T;  thread = (row, input quad)
__global__ void __launch_bounds__(256)
fold_rows_dx_kernel(int64_t rows, int K, int Fin, int Fout, const float *__restrict__ g, const float *__restrict__ w,
                    float *__restrict__ dx) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ float4 smem4[];
    float *Wf = reinterpret_cast<float *>(smem4);
    fold_weights(Wf, w, K, Fin, Fout, threadIdx.x, blockDim.x);
    __syncthreads();
    const int oq = Fout >> 2, iq = Fin >> 2;
    const int64_t total = rows * iq;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = t / iq;
        const int q = (int)(t - row * iq);
        const float4 *gr = reinterpret_cast<const float4 *>(g + row * Fout);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int o4 = 0; o4 < oq; ++o4) {
            const float4 gv = __ldg(gr + o4);
            const float4 w0 = *reinterpret_cast<const float4 *>(Wf + (4 * q + 0) * Fout + 4 * o4);
            const float4 w1 = *reinterpret_cast<const float4 *>(Wf + (4 * q + 1) * Fout + 4 * o4);
            const float4 w2 = *reinterpret_cast<const float4 *>(Wf + (4 * q + 2) * Fout + 4 * o4);
            const float4 w3 = *reinterpret_cast<const float4 *>(Wf + (4 * q + 3) * Fout + 4 * o4);
            acc.x = fmaf(gv.x, w0.x, fmaf(gv.y, w0.y, fmaf(gv.z, w0.z, fmaf(gv.w, w0.w, acc.x))));
            acc.y = fmaf(gv.x, w1.x, fmaf(gv.y, w1.y, fmaf(gv.z, w1.z, fmaf(gv.w, w1.w, acc.y))));
            acc.z = fmaf(gv.x, w2.x, fmaf(gv.y, w2.y, fmaf(gv.z, w2.z, fmaf(gv.w, w2.w, acc.z))));
            acc.w = fmaf(gv.x, w3.x, fmaf(gv.y, w3.y, fmaf(gv.z, w3.z, fmaf(gv.w, w3.w, acc.w))));
        }
        reinterpret_cast<float4 *>(dx + row * Fin)[q] = acc;
    }
}

// S = x^T g over `rows` rows as per-block partials in the layout of the generic weight-gradient partials
// ([M4][N4], M4 = round4(Fin), N4 = round4(Fout)); thread = (4x4 block of S, row lane), rows strided over
// lanes and blocks in a fixed pattern, ordered reduction over the lanes: deterministic.
__global__ void __launch_bounds__(256)
fold_rows_wgrad_kernel(int64_t rows, int Fin, int Fout, const float *__restrict__ x, const float *__restrict__ g,
                       float *__restrict__ partials) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ float4 smem4[];
    float *red = reinterpret_cast<float *>(smem4);     // [lanes][nblk * 16]
    const int iq = Fin >> 2, oq = Fout >> 2, nblk = iq * oq;
    const int lanes = blockDim.x / nblk;
    const int blk = threadIdx.x % nblk, lane = threadIdx.x / nblk;
    const int bi = blk % iq, bo = blk / iq;
    float4 c0 = make_float4(0.f, 0.f, 0.f, 0.f), c1 = c0, c2 = c0, c3 = c0;
    if (lane < lanes)
        for (int64_t r = (int64_t)blockIdx.x * lanes + lane; r < rows; r += (int64_t)gridDim.x * lanes) {
            const float4 xv = __ldg(reinterpret_cast<const float4 *>(x + r * Fin) + bi);
            const float4 gv = __ldg(reinterpret_cast<const float4 *>(g + r * Fout) + bo);
            c0.x = fmaf(xv.x, gv.x, c0.x); c0.y = fmaf(xv.x, gv.y, c0.y); c0.z = fmaf(xv.x, gv.z, c0.z); c0.w = fmaf(xv.x, gv.w, c0.w);
            c1.x = fmaf(xv.y, gv.x, c1.x); c1.y = fmaf(xv.y, gv.y, c1.y); c1.z = fmaf(xv.y, gv.z, c1.z); c1.w = fmaf(xv.y, gv.w, c1.w);
            c2.x = fmaf(xv.z, gv.x, c2.x); c2.y = fmaf(xv.z, gv.y, c2.y); c2.z = fmaf(xv.z, gv.z, c2.z); c2.w = fmaf(xv.z, gv.w, c2.w);
            c3.x = fmaf(xv.w, gv.x, c3.x); c3.y = fmaf(xv.w, gv.y, c3.y); c3.z = fmaf(xv.w, gv.z, c3.z); c3.w = fmaf(xv.w, gv.w, c3.w);
        }
    if (lane < lanes) {
        float *d = red + ((size_t)lane * nblk + blk) * 16;
        *reinterpret_cast<float4 *>(d) = c0; *reinterpret_cast<float4 *>(d + 4) = c1;
        *reinterpret_cast<float4 *>(d + 8) = c2; *reinterpret_cast<float4 *>(d + 12) = c3;
    }
    __syncthreads();
    float *part = partials + (size_t)blockIdx.x * Fin * Fout;       // M4 = Fin, N4 = Fout (both multiples of 4)
    for (int e = threadIdx.x; e < nblk * 16; e += blockDim.x) {
        float s = 0.f;
        for (int l = 0; l < lanes; ++l) s += red[(size_t)l * nblk * 16 + e];
        const int bk = e >> 4, m = (e >> 2) & 3, c = e & 3;
        part[(4 * (bk % iq) + m) * Fout + 4 * (bk / iq) + c] = s;
    }
}

static bool fold_ok(int K, int Fin, int Fout, const void *a, const void *b, const void *c) {
    return K >= 1 && Fin % 4 == 0 && Fout % 4 == 0 && Fin <= 64 && Fout <= 64 && (Fin / 4) * (Fout / 4) <= 64 &&
           (Fin <= 8 || Fout <= 8) && aligned16(a) && aligned16(b) && (!c || aligned16(c));
}
static int fold_grid(int64_t threads) {
    int64_t g = (threads + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 8;
    return (int)(g > cap ? cap : (g < 1 ? 1 : g));
}

int launch_fold_fwd(int64_t rows, int K, int Fin, int Fout, const float *x, const float *w, const float *bias, int relu,
                    float *out, cudaStream_t st) {
    if (fold_ok(K, Fin, Fout, x, out, bias)) {
        launch_pdl(fold_rows_fwd_kernel, dim3(fold_grid(rows * (Fout / 4))), dim3(256), (size_t)Fin * Fout * 4, st, rows, K, Fin, Fout, x, w, bias, relu, out);
        return check_launch("mvb fold_rows_fwd");
    }
    ContractArgs a{};
    a.rows = rows;
    a.in_planes = 1;
    a.in_w = Fin;
    a.in0 = x;
    a.wmat = w;
    a.w_fold = K;
    a.bias = bias;
    a.relu = relu;
    a.out_planes = 1;
    a.out_w = Fout;
    a.out = out;
    return launch_contract(a, st);
}
int launch_fold_dx(int64_t rows, int K, int Fin, int Fout, const float *g, const float *w, float *dx, cudaStream_t st) {
    if (fold_ok(K, Fin, Fout, g, dx, nullptr)) {
        launch_pdl(fold_rows_dx_kernel, dim3(fold_grid(rows * (Fin / 4))), dim3(256), (size_t)Fin * Fout * 4, st, rows, K, Fin, Fout, g, w, dx);
        return check_launch("mvb fold_rows_dx");
    }
    ContractArgs a{};
    a.rows = rows;
    a.in_planes = 1;
    a.in_w = Fout;
    a.in0 = g;
    a.wmat = w;
    a.w_transposed = 1;
    a.w_fold = K;
    a.out_planes = 1;
    a.out_w = Fin;
    a.out = dx;
    return launch_contract(a, st);
}
// partials: at least wgrad_partial_bytes(Fin, Fout); *nparts blocks of [*m4][Fout] are written
int launch_fold_wgrad(int64_t rows, int Fin, int Fout, const float *x, const float *g, float *partials, size_t partial_bytes,
                      int *nparts, int *m4, cudaStream_t st) {
    if (fold_ok(1, Fin, Fout, x, g, partials)) {
        const int nblk = (Fin / 4) * (Fout / 4);
        const int lanes = 256 / nblk;
        int64_t grid = (rows + (int64_t)lanes * 16 - 1) / ((int64_t)lanes * 16);      // >= 16 rows per lane
        const int64_t cap = (int64_t)num_sms() * 2;
        if (grid > cap) grid = cap;
        if (grid < 1) grid = 1;
        if ((size_t)grid * Fin * Fout * sizeof(float) <= partial_bytes) {
            launch_pdl(fold_rows_wgrad_kernel, dim3((unsigned)grid), dim3(256), (size_t)lanes * nblk * 16 * 4, st, rows, Fin, Fout, x, g, partials);
            const int rc = check_launch("mvb fold_rows_wgrad");
            if (rc) return rc;
            *nparts = (int)grid;
            *m4 = Fin;
            return MVB_OK;
        }
    }
    WgradArgs a{};
    a.rows = rows;
    a.in_planes = 1;
    a.in_w = Fin;
    a.in0 = x;
    a.dy = g;
    a.n_out = Fout;
    a.partials = partials;
    a.partial_bytes = partial_bytes;
    return launch_wgrad_partials(a, 0, nparts, m4, st);
}

// phase 2: dweight [M, n_out] (M = K*fin), dbias [n_out] or null.  a_transposed: see the kernel.
int launch_wgrad_finalize(const float *partA, int nA, int M4A, const float *partB, int nB, int M4B,
                          int fin, int M, int n_out, float *dweight, float *dbias, cudaStream_t st, int a_transposed) {
    const int total = (M + (dbias ? 1 : 0)) * n_out;
    const int N4 = round4(n_out);
    launch_pdl(wgrad_finalize_kernel, dim3((total + 31) / 32), dim3(32, 32), 0, st, partA, nA, M4A, partB, nB, M4B, fin, M, n_out,
               N4, a_transposed, round4(fin), dweight, dbias);
    return check_launch("mvb wgrad finalize");
}

}  // namespace mvb
