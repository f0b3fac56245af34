// tcgen05 (5th-gen tensor core) versions of the two dense contractions of the Chebyshev convolution.
//
//   tc_rowgemm_kernel : out[row, :] = act( A[row, :] . Bm + bias ),  A = K planes of width Fin
//                       (forward, nn/conv.py:559-575) or one plane dY of width Fout (backward
//                       P_k = dY W_k^T); 128 rows per tile = the M of one UMMA, N = Fout (or K*Fin),
//                       accumulators in TMEM, read back with tcgen05.ld for the bias/ReLU epilogue.
//   tc_wgrad_kernel   : dW[K*Fin, Fout] (+ db) = [T_0|..|T_{K-1}|1]^T dY : the feature index is the
//                       M of the UMMA (MN-major A straight from the vertex-major tile), rows of the
//                       activation are the K dimension, one TMEM accumulator per CTA over all its
//                       tiles, per-CTA partials + the ordered finalize kernel (deterministic).
//
// Precision: kind::tf32 alone would break the 1e-4 parity gate (10-bit mantissa), so both kernels
// run the error-compensated 3xTF32 scheme: every fp32 operand is split while it is staged into
// shared memory, hi = x & 0xffffe000 (exactly representable in tf32), lo = x - hi (exact in fp32),
// and D += A_hi B_hi + A_lo B_hi + A_hi B_lo  (dropped term ~2^-22).  Tensor throughput is >20x what
// these HBM-bound contractions need, so the 3x MMA count is free.
//
// Operands are staged global -> registers -> shared directly into the canonical SWIZZLE_64B / SWIZZLE_128B layouts the UMMA
// shared-memory descriptors expect: a tile row is 64 B (Fin = 16) or 128 B (Fin = 32) and its
// 16-byte chunk index is XORed with address bits [7,9) / [7,10), which also makes the staging
// stores bank-conflict free.
#include "mvb_internal.cuh"
#include "mvb_tcgen05.cuh"

namespace mvb {

static int g_tc_enabled = 1;
void set_tc_enabled(int v) { g_tc_enabled = v; }
int tc_enabled() { return g_tc_enabled; }

// ---------------------------------------------------------------------------------------------
// row GEMM:  out = act(A . Bm + bias)
// ---------------------------------------------------------------------------------------------
struct TcRowArgs {
    int64_t rows;
    int in_planes, in_w;
    const float *in0, *in_rest, *mask;
    const float *wmat;
    int w_transposed, w_fold;
    int nn_true, nn16;            // real and padded (multiple of 16) output width
    const float *bias;
    int relu;
    int out_w;                    // width of one output plane (nn_true = out_planes * out_w)
    float *out;
    int tmem_cols;
    int tile_w;                   // floats per staged tile row (16 or 32)
    int tile_planes;              // number of staged tiles (= in_planes, 1 for 4-wide planes)
    const int32_t *row_sel;       // optional input-row selection (ContractArgs)
    int sel_group;
    int64_t plane_rows;           // rows of one input plane (== rows without a selection)
};

// input row of output row r under a row selection: row_sel[r / group] * group + r % group
__device__ __forceinline__ int64_t sel_row(const int32_t *row_sel, int group, int64_t r) {
    const int64_t m = r / group;
    return (int64_t)__ldg(row_sel + m) * group + (r - m * group);
}

// B operand: Bt[n][kd] (n = output column, kd = logical K index p*in_w + i), K-major, swizzled like A,
// hi/lo split.  kd maps to (tile plane, column) = (kd / tile_w, kd % tile_w) - for 4-wide planes
// there is a single tile plane.  Loads are issued four at a time (the weights are L2/L1 resident).
__device__ __forceinline__ void stage_b_operand(const TcRowArgs &a, char *Bhi, char *Blo, int b_plane, int row_bytes,
                                                int tid, int nthreads) {
    const int Kd = a.in_planes * a.in_w;
    const int nfold = a.w_fold > 1 ? a.w_fold : 1;
    const int total = a.nn16 * Kd;
    for (int base = 0; base < total; base += 4 * nthreads) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * nthreads + tid;
            v[u] = 0.f;
            if (i < total) {
                const int n = i / Kd, kd = i - n * Kd;
                if (n < a.nn_true) {
                    if (a.w_transposed == 2) {      // per-plane transposed: W[k][n][o], kd = k*in_w + o
                        const int k = kd / a.in_w, o = kd - k * a.in_w;
                        v[u] = __ldg(a.wmat + ((int64_t)k * a.nn_true + n) * a.in_w + o);
                    } else {
                        for (int k = 0; k < nfold; k += 2) {
                            const float wv = a.w_transposed ? __ldg(a.wmat + ((int64_t)k * a.nn_true + n) * Kd + kd)
                                                            : __ldg(a.wmat + ((int64_t)k * Kd + kd) * a.nn_true + n);
                            v[u] += (k & 2) ? -wv : wv;
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * nthreads + tid;
            if (i < total) {
                const int n = i / Kd, kd = i - n * Kd;
                float h, l;
                split_tf32(v[u], h, l);
                const int p = kd / a.tile_w, c = kd - p * a.tile_w;
                const uint32_t off = (uint32_t)(p * b_plane) + swz_off(n, c >> 2, row_bytes) + (uint32_t)((c & 3) << 2);
                *reinterpret_cast<float *>(Bhi + off) = h;
                *reinterpret_cast<float *>(Blo + off) = l;
            }
        }
    }
}

// all MMAs of one 128-row tile: for every tile plane and 8-wide K slice, the three 3xTF32 terms
__device__ __forceinline__ void issue_row_mmas(uint32_t tmem_base, char *Ahi, char *Alo, char *Bhi, char *Blo,
                                               int planes, int a_plane, int b_plane, int kslices, uint32_t sbo,
                                               uint32_t layout_type, uint32_t idesc, uint32_t acc) {
    for (int p = 0; p < planes; ++p) {
        for (int j = 0; j < kslices; ++j) {
            const uint64_t ah = make_desc(smem_u32(Ahi + p * a_plane) + j * 32, 16, sbo, layout_type);
            const uint64_t al = make_desc(smem_u32(Alo + p * a_plane) + j * 32, 16, sbo, layout_type);
            const uint64_t bh = make_desc(smem_u32(Bhi + p * b_plane) + j * 32, 16, sbo, layout_type);
            const uint64_t bl = make_desc(smem_u32(Blo + p * b_plane) + j * 32, 16, sbo, layout_type);
            umma_tf32(tmem_base, al, bh, idesc, acc);     // small terms first
            umma_tf32(tmem_base, ah, bl, idesc, 1);
            umma_tf32(tmem_base, ah, bh, idesc, 1);
            acc = 1;
        }
    }
}

// epilogue of one tile: TMEM -> registers -> bias / ReLU -> global (thread = row, 16 columns per pass)
__device__ __forceinline__ void row_epilogue(const TcRowArgs &a, uint32_t tmem_base, int warp, int row, int nr,
                                             int64_t row0) {
    for (int n0 = 0; n0 < a.nn16; n0 += 16) {
        float v[16];
        tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)n0, v);
        if (row < nr && n0 < a.nn_true) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                if (a.bias && n0 + j < a.nn_true) v[j] += __ldg(a.bias + n0 + j);
                if (a.relu) v[j] = v[j] > 0.f ? v[j] : 0.f;
            }
            const int64_t grow = row0 + row;
            if (a.nn_true - n0 >= 16 && (a.out_w & 15) == 0) {
                const int p = n0 / a.out_w, jj = n0 - p * a.out_w;
                float4 *dst = reinterpret_cast<float4 *>(a.out + ((int64_t)p * a.rows + grow) * a.out_w + jj);
                dst[0] = make_float4(v[0], v[1], v[2], v[3]);
                dst[1] = make_float4(v[4], v[5], v[6], v[7]);
                dst[2] = make_float4(v[8], v[9], v[10], v[11]);
                dst[3] = make_float4(v[12], v[13], v[14], v[15]);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int n = n0 + j;
                    if (n < a.nn_true) {
                        const int p = n / a.out_w, jj = n - p * a.out_w;
                        a.out[((int64_t)p * a.rows + grow) * a.out_w + jj] = v[j];
                    }
                }
            }
        }
    }
}

// W = 16 / 32: planar layout, one swizzled tile per input plane, staged PG planes at a time ("plane
//              groups": the accumulator stays in TMEM across the groups of a tile).  The next group's rows
//              are prefetched into registers while the current group's MMAs run.  Small groups keep the
//              shared-memory footprint low enough for 3-4 resident CTAs per SM, whose phases (global loads
//              in flight / register->shared commit / MMA / epilogue) then overlap - with all 6 planes of
//              the forward contraction staged at once only ONE 128-thread CTA fitted per SM and the
//              kernel ran at 2.7 TB/s (profiles/README.md).
// W = 4      : all NP planes share one tile row (PG = NP).
template <int W, int NP, int PG>
__global__ void __launch_bounds__(128)
tc_rowgemm_kernel(TcRowArgs a) {
    extern __shared__ __align__(1024) char smem_raw[];
    char *smem = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    constexpr bool ONE_TILE = (W == 4);              // 4-wide planes: all NP planes share one tile row
    constexpr int Q4 = W / 4;
    constexpr int NPR = PG;                          // planes prefetched into registers (one group)
    constexpr int NPL = ONE_TILE ? 1 : PG;           // staged A tiles
    constexpr int NPB = ONE_TILE ? 1 : NP;           // staged B tiles (all planes, once)
    constexpr int NG = ONE_TILE ? 1 : NP / PG;
    static_assert(ONE_TILE || NP % PG == 0, "plane groups must divide the plane count");
    constexpr int NV = NPR * Q4;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wt = ONE_TILE ? a.tile_w : W;
    const int row_bytes = wt * 4;
    const int R = 128;
    const int a_plane = R * row_bytes;
    const int b_plane = a.nn16 * row_bytes;
    char *Ahi = smem;
    char *Alo = Ahi + NPL * a_plane;
    char *Bhi = Alo + NPL * a_plane;
    char *Blo = Bhi + NPB * b_plane;
    uint64_t *bar = reinterpret_cast<uint64_t *>(Blo + NPB * b_plane);
    uint32_t *slot = reinterpret_cast<uint32_t *>(bar + 1);

    pdl_trigger();
    if (warp == 0) tmem_alloc(slot, (uint32_t)a.tmem_cols);
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_barrier_init();
    }
    if (ONE_TILE) {             // padding columns of the shared tile row must be finite zeros in A and B
        for (int i = tid; i < (2 * a_plane + 2 * b_plane) / 16; i += blockDim.x)
            reinterpret_cast<float4 *>(Ahi)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncthreads();
    }
    stage_b_operand(a, Bhi, Blo, b_plane, row_bytes, tid, blockDim.x);          // weights: no kernel of the step writes them
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_wait();          // the planes are the previous kernels' output
    const uint32_t tmem_base = *slot;
    const uint32_t idesc = make_idesc(128, a.nn16, 0, 0);
    const uint32_t layout_type = (row_bytes == 128) ? 2u : 4u;
    const uint32_t sbo = 8u * row_bytes;
    const int kslices = ONE_TILE ? (a.in_planes * a.in_w + 7) / 8 : W / 8;
    const int row = warp * 32 + lane;                 // D row (TMEM lane) this thread reads back
    uint32_t phase = 0;
    const int64_t ntiles = (a.rows + R - 1) / R;

    float4 pre[NV];
    float4 prem[Q4];
    // tile-invariant part of a thread's pieces (row within the tile, swizzled shared-memory offset): computed once
    int srow[Q4];
    uint32_t soff[Q4];
#pragma unroll
    for (int j = 0; j < Q4; ++j) {
        const int i = j * 128 + tid;
        srow[j] = i / Q4;
        soff[j] = swz_off(srow[j], i - srow[j] * Q4, row_bytes);
    }
    // global -> registers for plane group g of the tile starting at row0
    auto prefetch = [&](int64_t row0, int g) {
        const int nr = (int)((a.rows - row0) < R ? (a.rows - row0) : R);
#pragma unroll
        if (a.row_sel) {          // selected rows: the pieces of a tile row stay contiguous, the rows are gathered
            int64_t src[Q4];
#pragma unroll
            for (int j = 0; j < Q4; ++j) src[j] = (srow[j] < nr) ? sel_row(a.row_sel, a.sel_group, row0 + srow[j]) : 0;
#pragma unroll
            for (int pp = 0; pp < NPR; ++pp) {
                const int p = g * NPR + pp;
                const float4 *b4 = reinterpret_cast<const float4 *>(p == 0 ? a.in0 : a.in_rest + (int64_t)(p - 1) * a.plane_rows * (Q4 * 4));
#pragma unroll
                for (int j = 0; j < Q4; ++j) {
                    const int i = j * 128 + tid;
                    pre[pp * Q4 + j] = (srow[j] < nr) ? __ldg(b4 + src[j] * Q4 + (i - srow[j] * Q4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        } else {
#pragma unroll
        for (int pp = 0; pp < NPR; ++pp) {
            const int p = g * NPR + pp;
            const float4 *s4 = reinterpret_cast<const float4 *>((p == 0 ? a.in0 : a.in_rest + (int64_t)(p - 1) * a.rows * (Q4 * 4)) + row0 * (Q4 * 4));
#pragma unroll
            for (int j = 0; j < Q4; ++j) {
                pre[pp * Q4 + j] = (srow[j] < nr) ? __ldg(s4 + j * 128 + tid) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        }
        if (a.mask && g == 0) {
            const float4 *m4 = reinterpret_cast<const float4 *>(a.mask + row0 * (Q4 * 4));
#pragma unroll
            for (int j = 0; j < Q4; ++j) {
                prem[j] = (srow[j] < nr) ? __ldg(m4 + j * 128 + tid) : make_float4(1.f, 1.f, 1.f, 1.f);
            }
        }
    };
    // registers -> hi/lo swizzled shared tiles
    auto commit = [&](int g) {
#pragma unroll
        for (int p = 0; p < NPR; ++p) {
#pragma unroll
            for (int j = 0; j < Q4; ++j) {
                float4 v = pre[p * Q4 + j];
                if (p == 0 && g == 0 && a.mask) {
                    v.x = prem[j].x > 0.f ? v.x : 0.f;
                    v.y = prem[j].y > 0.f ? v.y : 0.f;
                    v.z = prem[j].z > 0.f ? v.z : 0.f;
                    v.w = prem[j].w > 0.f ? v.w : 0.f;
                }
                float4 h, l;
                split4(v, h, l);
                const uint32_t off = ONE_TILE ? swz_off(srow[j], p * Q4 + (j * 128 + tid - srow[j] * Q4), row_bytes)
                                              : (uint32_t)(p * a_plane) + soff[j];
                *reinterpret_cast<float4 *>(Ahi + off) = h;
                *reinterpret_cast<float4 *>(Alo + off) = l;
            }
        }
    };
    int64_t t = blockIdx.x;
    if (t < ntiles) prefetch(t * R, 0);
    for (; t < ntiles; t += gridDim.x) {
        const int64_t row0 = t * R;
        const int nr = (int)((a.rows - row0) < R ? (a.rows - row0) : R);
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            commit(g);
            fence_proxy_async();
            tc_fence_before();
            __syncthreads();
            if (tid == 0) {
                tc_fence_after();
                issue_row_mmas(tmem_base, Ahi, Alo, Bhi + g * NPL * b_plane, Blo + g * NPL * b_plane, NPL, a_plane, b_plane, kslices, sbo,
                               layout_type, idesc, g > 0 ? 1u : 0u);
                umma_commit(bar);
            }
            // the next group's rows are in flight during the MMAs (and, for the last group, the epilogue)
            if (g + 1 < NG) prefetch(row0, g + 1);
            else if (t + gridDim.x < ntiles) prefetch((t + gridDim.x) * R, 0);
            mbar_wait(bar, phase);
            phase ^= 1;
            tc_fence_after();
        }
        row_epilogue(a, tmem_base, warp, row, nr, row0);
        tc_fence_before();   // order this tile's TMEM reads before the barrier that precedes the next MMA
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)a.tmem_cols);
}

static int pow2_cols(int n) {
    int c = 32;
    while (c < n) c <<= 1;
    return c;
}

template <int W, int NP, int PG = NP>
static int launch_rowgemm_t(const TcRowArgs &t, unsigned grid, size_t smem, cudaStream_t st) {
    static DevFlags optin;
    {
        const int rc_attr = smem_optin(tc_rowgemm_kernel<W, NP, PG>, 200 * 1024, optin, "tc_rowgemm");
        if (rc_attr) return rc_attr;
    }
    launch_pdl(tc_rowgemm_kernel<W, NP, PG>, dim3(grid), dim3(128), smem, st, t);
    return check_launch("mvb tc_rowgemm");
}

// returns 1 if the tensor-core path took the call, 0 if the shape is not supported (caller falls
// back to the FFMA kernel), < 0 on error
int launch_contract_tc(const ContractArgs &a, cudaStream_t st) {
    if (!g_tc_enabled) return 0;
    const int w = a.in_w;
    const int Kd = a.in_planes * w;
    const int nn_true = a.out_planes * a.out_w;
    const int nn16 = (nn_true + 15) & ~15;
    if (nn16 > 256 || a.rows < 128) return 0;
    const bool planar = (w == 16 && a.in_planes <= 6) || (w == 32 && a.in_planes <= 3) || (w == 4 && a.in_planes <= 8);
    const bool vec_ok = aligned16(a.in0) && (a.in_planes == 1 || aligned16(a.in_rest)) && (!a.mask || aligned16(a.mask));
    if (!(planar && vec_ok) || !aligned16(a.out)) return 0;
    if (a.row_sel && (a.mask || a.sel_group < 1)) return 0;
    TcRowArgs t;
    t.row_sel = a.row_sel;
    t.sel_group = a.sel_group;
    t.plane_rows = a.row_sel ? a.plane_rows : a.rows;
    t.rows = a.rows;
    t.in_planes = a.in_planes;
    t.in_w = w;
    t.in0 = a.in0;
    t.in_rest = a.in_rest;
    t.mask = a.mask;
    t.wmat = a.wmat;
    t.w_transposed = a.w_transposed;
    t.w_fold = a.w_fold;
    t.nn_true = nn_true;
    t.nn16 = nn16;
    t.bias = a.bias;
    t.relu = a.relu;
    t.out_w = a.out_w;
    t.out = a.out;
    t.tmem_cols = pow2_cols(nn16);
    t.tile_w = (w == 4) ? (Kd <= 16 ? 16 : 32) : w;
    t.tile_planes = (w == 4) ? 1 : a.in_planes;
    // plane groups (A tiles staged at a time): 2 of 4-6 planes for 16-wide planes, 1 of 2-3 for 32-wide
    int pg = t.tile_planes;
    if (w == 16 && (a.in_planes == 4 || a.in_planes == 6)) pg = 2;
    else if (w == 32 && a.in_planes >= 2) pg = 1;
    const size_t smem = 1024 + (size_t)pg * (2 * 128 * t.tile_w * 4) + (size_t)t.tile_planes * (2 * nn16 * t.tile_w * 4) + 64;
    if (smem > 200 * 1024) return 0;
    const int64_t ntiles = (a.rows + 127) / 128;
    // CTAs per SM: shared memory and TMEM (512 columns) permitting
    int per_sm = (int)((220 * 1024) / smem);
    if (per_sm > 512 / t.tmem_cols) per_sm = 512 / t.tmem_cols;
    if (per_sm > 4) per_sm = 4;
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)num_sms() * per_sm;
    if (grid > ntiles) grid = ntiles;
    int rc;
    if (w == 4) {
        switch (a.in_planes) {
            case 1: rc = launch_rowgemm_t<4, 1>(t, (unsigned)grid, smem, st); break;
            case 2: rc = launch_rowgemm_t<4, 2>(t, (unsigned)grid, smem, st); break;
            case 3: rc = launch_rowgemm_t<4, 3>(t, (unsigned)grid, smem, st); break;
            case 4: rc = launch_rowgemm_t<4, 4>(t, (unsigned)grid, smem, st); break;
            case 5: rc = launch_rowgemm_t<4, 5>(t, (unsigned)grid, smem, st); break;
            case 6: rc = launch_rowgemm_t<4, 6>(t, (unsigned)grid, smem, st); break;
            case 7: rc = launch_rowgemm_t<4, 7>(t, (unsigned)grid, smem, st); break;
            default: rc = launch_rowgemm_t<4, 8>(t, (unsigned)grid, smem, st); break;
        }
    } else if (w == 16) {
        switch (a.in_planes) {
            case 1: rc = launch_rowgemm_t<16, 1>(t, (unsigned)grid, smem, st); break;
            case 2: rc = launch_rowgemm_t<16, 2>(t, (unsigned)grid, smem, st); break;
            case 3: rc = launch_rowgemm_t<16, 3>(t, (unsigned)grid, smem, st); break;
            case 4: rc = launch_rowgemm_t<16, 4, 2>(t, (unsigned)grid, smem, st); break;
            case 5: rc = launch_rowgemm_t<16, 5>(t, (unsigned)grid, smem, st); break;
            default: rc = launch_rowgemm_t<16, 6, 2>(t, (unsigned)grid, smem, st); break;
        }
    } else {
        switch (a.in_planes) {
            case 1: rc = launch_rowgemm_t<32, 1>(t, (unsigned)grid, smem, st); break;
            case 2: rc = launch_rowgemm_t<32, 2, 1>(t, (unsigned)grid, smem, st); break;
            default: rc = launch_rowgemm_t<32, 3, 1>(t, (unsigned)grid, smem, st); break;
        }
    }
    return rc ? rc : 1;
}

// ---------------------------------------------------------------------------------------------
// weight gradient on tensor cores
// ---------------------------------------------------------------------------------------------
// Both operands are consumed MN-major (the contiguous index of the staged tile - the feature - is
// the M / N of the MMA, the activation row is K).  For 32-bit operands the only MN-major shared
// memory layout UMMA accepts is SWIZZLE_128B_BASE32B (layout type 1): rows of 128 bytes = 32
// features, K atoms of 4 rows (stride byte offset = 512), MN blocks of 32 features at the leading
// byte offset, and a 32-byte-granular swizzle (cute Swizzle<2,5,2> on the byte address): the
// 32-byte unit index (address bits [5,7)) ^= row & 3 (address bits [7,9)).
// Logical feature column of plane p, feature f is p*in_w + f (= the dW row index k*Fin + fi); the
// "ones" column that yields the bias gradient sits at column K*Fin.
struct TcWgradArgs {
    int64_t rows;
    int in_planes, in_w;
    const float *in0, *in_rest;
    const float *dy, *mask;
    int n_out, n16;                // Fout and its padding to the MMA N (16 or 32)
    int has_bias;
    int M4, N4;                    // partial block layout [M4][N4] expected by the finalize kernel
    float *partials;
    int tmem_cols;
    const int32_t *row_sel;        // optional selection of the T rows (WgradArgs); dy / mask are dense over the selected rows
    int sel_group;
    int64_t plane_rows;
};

// byte offset of logical (row r, feature column col) in a BASE32B tile made of 32-column blocks of blk bytes
__device__ __forceinline__ uint32_t b32_off(int r, int col, int blk) {
    const int b = col >> 5, c = (col & 31) >> 2;
    return (uint32_t)(b * blk + r * 128 + (((c >> 1) ^ (r & 3)) << 5) + ((c & 1) << 4) + ((col & 3) << 2));
}

// NPF planes of width 4*Q4 floats (4, 16 or 32), Fout % 4 == 0: vector staging with register prefetch
constexpr int WG_NT = 256;      // 8 warps: all of them stage tiles, warps 0-3 own the TMEM lanes of the epilogue (ncu: the
                                // 128-thread version was paced by its own instruction stream at 8 warps per SM)
template <int NPF, int Q4>
__global__ void __launch_bounds__(WG_NT)
tc_wgrad_kernel(TcWgradArgs a) {
    extern __shared__ __align__(1024) char smem_raw[];
    char *smem = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    constexpr int W = 4 * Q4;                          // plane width
    constexpr int LPT = (64 * Q4 + WG_NT - 1) / WG_NT; // float4 loads per thread per plane per 64-row tile
    constexpr int DJ = 512 / WG_NT;                    // dY pieces per thread (up to 64 rows x 8 quads)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int R = 64;                                  // activation rows (= UMMA K extent) per tile
    const int blk = R * 128;                           // one 32-feature block of the T tile: 8 KB
    char *Thi = smem;                                  // 4 blocks = 128 feature columns
    char *Tlo = Thi + 4 * blk;
    char *Dhi = Tlo + 4 * blk;                         // dY tile, rows of 128 B
    char *Dlo = Dhi + blk;
    uint64_t *bar = reinterpret_cast<uint64_t *>(Dlo + blk);
    uint32_t *slot = reinterpret_cast<uint32_t *>(bar + 1);

    pdl_trigger();
    if (warp == 0) tmem_alloc(slot, (uint32_t)a.tmem_cols);
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_barrier_init();
    }
    // zero everything once (unused feature columns, padding of dY rows), then the ones column
    for (int i = tid; i < (10 * blk) / 16; i += blockDim.x)
        reinterpret_cast<float4 *>(Thi)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    if (a.has_bias) {
        const int col = a.in_planes * a.in_w;
        for (int r = tid; r < R; r += blockDim.x) *reinterpret_cast<float *>(Thi + b32_off(r, col, blk)) = 1.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_wait();          // shared-memory and TMEM set-up above; the planes / dY are the previous kernels' output
    const uint32_t tmem_base = *slot;
    // N-STACKING (Fout <= 16): the lo parts of dY go into columns 16..31 of the same 128-byte B rows, so ONE MMA with
    // N = 32 yields A.[B_hi | B_lo]; two MMAs per K step (A_hi, A_lo) instead of three give all four hi/lo products, the
    // epilogue adds the two column halves.  These MMAs cost the same whatever N is (the M = 128 operand is streamed from
    // shared memory per instruction), and their count paces the kernel.
    const bool nstack = a.n16 == 16;
    const uint32_t idesc = make_idesc(128, nstack ? 32 : a.n16, 1, 1);
    const int64_t ntiles = (a.rows + R - 1) / R;
    const int dq4 = a.n_out >> 2;                      // float4 chunks per dY row

    // register prefetch DEPTH tiles ahead.  Depth 3 for the narrow planes (10 KB per tile) measured no faster than depth 1
    // (43.3 vs 42.7 us): the kernel is paced by the MMA instruction stream, not by memory latency - see N-stacking below
    constexpr int DEPTH = 1;
    float4 pre[DEPTH][LPT * NPF];
    float4 pred[DEPTH][DJ], prem[DEPTH][DJ];
    // everything about a thread's pieces of a tile that does not depend on the tile - row, shared-memory offsets,
    // validity - is computed once: the per-tile code is then loads, the hi/lo split and stores (ncu: 11.2 M warp
    // instructions for 4998 narrow tiles before, two integer divisions and a swizzle computation per piece per tile)
    // 16-wide planes (4 quads per row): a warp's 32 pieces are 8 rows x 4 quads.  In this row-major lane order the 8 lanes
    // of a quarter warp (2 rows x 4 quads) hit only TWO of the four 32-byte units of the BASE32B swizzle - every 16-byte
    // store is a 2-way bank conflict (ncu r02b: 47 % of the shared wavefronts of tc_wgrad<6,4>).  A conflict-free lane
    // order measured no faster (bench.py, 0.9209 / 0.9389 against 0.9181 / 0.9182 ms per step): the stores do not pace
    // the kernel.
    int trow[LPT];                       // row of T piece j within the tile, -1 = no piece
    int tidx[LPT];                       // its quad index inside the tile (row * Q4 + quad)
    uint32_t toff[NPF][LPT];
#pragma unroll
    for (int j = 0; j < LPT; ++j) {
        const int i = j * WG_NT + tid;
        tidx[j] = i;
        trow[j] = (i < 64 * Q4) ? i / Q4 : -1;
#pragma unroll
        for (int p = 0; p < NPF; ++p) toff[p][j] = trow[j] >= 0 ? b32_off(trow[j], p * W + (i - trow[j] * Q4) * 4, blk) : 0u;
    }
    int drow[DJ], didx[DJ];
    uint32_t doff[DJ], doff_lo[DJ];
#pragma unroll
    for (int j = 0; j < DJ; ++j) {
        const int i = j * WG_NT + tid;
        didx[j] = i;
        drow[j] = (i < R * dq4) ? i / dq4 : -1;
        const int q = drow[j] >= 0 ? i - drow[j] * dq4 : 0;
        doff[j] = drow[j] >= 0 ? b32_off(drow[j], q * 4, blk) : 0u;
        doff_lo[j] = drow[j] >= 0 ? b32_off(drow[j], 16 + q * 4, blk) : 0u;       // N-stacked position of the lo part
    }
    auto prefetch = [&](const int d, int64_t row0) {
        const int nr = (int)((a.rows - row0) < R ? (a.rows - row0) : R);
        if (a.row_sel) {
            int64_t src[LPT];
#pragma unroll
            for (int j = 0; j < LPT; ++j) src[j] = (trow[j] >= 0 && trow[j] < nr) ? sel_row(a.row_sel, a.sel_group, row0 + trow[j]) : 0;
#pragma unroll
            for (int p = 0; p < NPF; ++p) {
                const float4 *b4 = reinterpret_cast<const float4 *>(p == 0 ? a.in0 : a.in_rest + (int64_t)(p - 1) * a.plane_rows * W);
#pragma unroll
                for (int j = 0; j < LPT; ++j) {
                    const int i = tidx[j];
                    pre[d][p * LPT + j] = (trow[j] >= 0 && trow[j] < nr) ? __ldg(b4 + src[j] * Q4 + (i - trow[j] * Q4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        } else {
#pragma unroll
        for (int p = 0; p < NPF; ++p) {
            const float4 *s4 = reinterpret_cast<const float4 *>((p == 0 ? a.in0 : a.in_rest + (int64_t)(p - 1) * a.rows * W) + row0 * W);
#pragma unroll
            for (int j = 0; j < LPT; ++j)
                pre[d][p * LPT + j] = (trow[j] >= 0 && trow[j] < nr) ? __ldg(s4 + tidx[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        }
        const float4 *d4 = reinterpret_cast<const float4 *>(a.dy + row0 * a.n_out);
        const float4 *m4 = reinterpret_cast<const float4 *>(a.mask ? a.mask + row0 * a.n_out : nullptr);
#pragma unroll
        for (int j = 0; j < DJ; ++j) {
            const bool ok = drow[j] >= 0 && drow[j] < nr;
            pred[d][j] = ok ? __ldg(d4 + didx[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (a.mask) prem[d][j] = ok ? __ldg(m4 + didx[j]) : make_float4(1.f, 1.f, 1.f, 1.f);
        }
    };
    auto commit = [&](const int d) {
#pragma unroll
        for (int p = 0; p < NPF; ++p) {
#pragma unroll
            for (int j = 0; j < LPT; ++j) {
                if (trow[j] >= 0) {
                    float4 h, l;
                    split4(pre[d][p * LPT + j], h, l);
                    *reinterpret_cast<float4 *>(Thi + toff[p][j]) = h;
                    *reinterpret_cast<float4 *>(Tlo + toff[p][j]) = l;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < DJ; ++j) {
            if (drow[j] >= 0) {
                float4 v = pred[d][j];
                if (a.mask) {
                    v.x = prem[d][j].x > 0.f ? v.x : 0.f;
                    v.y = prem[d][j].y > 0.f ? v.y : 0.f;
                    v.z = prem[d][j].z > 0.f ? v.z : 0.f;
                    v.w = prem[d][j].w > 0.f ? v.w : 0.f;
                }
                float4 h, l;
                split4(v, h, l);
                *reinterpret_cast<float4 *>(Dhi + doff[j]) = h;
                if (nstack)
                    *reinterpret_cast<float4 *>(Dhi + doff_lo[j]) = l;
                else
                    *reinterpret_cast<float4 *>(Dlo + doff[j]) = l;
            }
        }
    };
    uint32_t acc = 0, phase = 0;
    bool pending = false;
    int64_t t = blockIdx.x;
#pragma unroll
    for (int d = 0; d < DEPTH; ++d)
        if (t + (int64_t)d * gridDim.x < ntiles) prefetch(d, (t + (int64_t)d * gridDim.x) * R);
    while (t < ntiles) {
#pragma unroll
        for (int d = 0; d < DEPTH; ++d) {          // static register slots: the tile loop is unrolled DEPTH times
            if (t >= ntiles) continue;
            if (pending) {   // the previous tile's MMAs must have finished reading shared memory
                mbar_wait(bar, phase);
                phase ^= 1;
            }
            commit(d);
            fence_proxy_async();
            tc_fence_before();
            __syncthreads();
            if (tid == 0) {
                tc_fence_after();
                for (int ks = 0; ks < R / 8; ++ks) {          // 8 activation rows per MMA = two 4-row K atoms
                    const uint64_t ah = make_desc(smem_u32(Thi) + ks * 1024, blk, 512, 1u);
                    const uint64_t al = make_desc(smem_u32(Tlo) + ks * 1024, blk, 512, 1u);
                    const uint64_t bh = make_desc(smem_u32(Dhi) + ks * 1024, blk, 512, 1u);
                    const uint64_t bl = make_desc(smem_u32(Dlo) + ks * 1024, blk, 512, 1u);
                    umma_tf32(tmem_base, al, bh, idesc, acc);
                    if (!nstack) umma_tf32(tmem_base, ah, bl, idesc, 1);
                    umma_tf32(tmem_base, ah, bh, idesc, 1);
                    acc = 1;
                }
                umma_commit(bar);
            }
            pending = true;
            const int64_t nx = t + (int64_t)DEPTH * gridDim.x;
            if (nx < ntiles) prefetch(d, nx * R);     // overlaps this and the next DEPTH-1 tiles
            t += gridDim.x;
        }
    }
    if (pending) {
        mbar_wait(bar, phase);
        phase ^= 1;
    }
    tc_fence_after();
    // D[m = feature (or bias row)][n = fo] -> per-CTA partial block [M4][N4]
    const int m = warp * 32 + lane;
    float *part = a.partials + (size_t)blockIdx.x * a.M4 * a.N4;
    for (int n0 = 0; warp < 4 && n0 < a.n16; n0 += 16) {      // TMEM lanes 0..127 belong to warps 0..3
        float v[16];
        tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)n0, v);
        if (nstack) {                       // + A.B_lo from the upper column half
            float v2[16];
            tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + 16u, v2);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] += v2[j];
        }
        if (m < a.M4) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if (n0 + j < a.N4) part[m * a.N4 + n0 + j] = pending ? v[j] : 0.f;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)a.tmem_cols);
}

template <int NPF, int Q4>
static int launch_wgrad_t(const TcWgradArgs &t, unsigned grid, size_t smem, cudaStream_t st) {
    static DevFlags optin;
    {
        const int rc_attr = smem_optin(tc_wgrad_kernel<NPF, Q4>, 200 * 1024, optin, "tc_wgrad");
        if (rc_attr) return rc_attr;
    }
    launch_pdl(tc_wgrad_kernel<NPF, Q4>, dim3(grid), dim3(WG_NT), smem, st, t);
    return check_launch("mvb tc_wgrad");
}

// returns 1 if taken, 0 if unsupported, < 0 on error.  Partial layout matches the FFMA wgrad kernel.
int launch_wgrad_tc(const WgradArgs &a, int has_bias, int M4, int N4, int *nparts, cudaStream_t st) {
    if (!g_tc_enabled) return 0;
    const int M = a.in_planes * a.in_w;
    if (M + (has_bias ? 1 : 0) > 128 || M4 > 128 || a.n_out > 32 || a.rows < 256) return 0;
    const bool fast = ((a.in_w == 16 && a.in_planes <= 6) || (a.in_w == 4 && a.in_planes <= 8) || (a.in_w == 32 && a.in_planes <= 3)) &&
                      (a.n_out % 4 == 0) && aligned16(a.in0) &&
                      (a.in_planes == 1 || aligned16(a.in_rest)) && aligned16(a.dy) && (!a.mask || aligned16(a.mask));
    if (!fast || (a.row_sel && a.sel_group < 1)) return 0;
    TcWgradArgs t;
    t.row_sel = a.row_sel;
    t.sel_group = a.sel_group;
    t.plane_rows = a.row_sel ? a.plane_rows : a.rows;
    t.rows = a.rows;
    t.in_planes = a.in_planes;
    t.in_w = a.in_w;
    t.in0 = a.in0;
    t.in_rest = a.in_rest;
    t.dy = a.dy;
    t.mask = a.mask;
    t.n_out = a.n_out;
    t.n16 = (a.n_out + 15) & ~15;
    t.has_bias = has_bias;
    t.M4 = M4;
    t.N4 = N4;
    t.partials = a.partials;
    t.tmem_cols = 32;
    const size_t smem = 1024 + 10 * 64 * 128 + 64;
    const int64_t ntiles = (a.rows + 63) / 64;
    int64_t grid = (int64_t)num_sms() * 2;
    if (grid > ntiles) grid = ntiles;
    if ((size_t)grid * M4 * N4 * sizeof(float) > a.partial_bytes) return set_err(MVB_EWORKSPACE, "tc_wgrad: workspace too small");
    int rc;
    if (a.in_w == 32) {
        switch (a.in_planes) {
            case 1: rc = launch_wgrad_t<1, 8>(t, (unsigned)grid, smem, st); break;
            case 2: rc = launch_wgrad_t<2, 8>(t, (unsigned)grid, smem, st); break;
            default: rc = launch_wgrad_t<3, 8>(t, (unsigned)grid, smem, st); break;
        }
    } else if (a.in_w == 16) {
        switch (a.in_planes) {
            case 1: rc = launch_wgrad_t<1, 4>(t, (unsigned)grid, smem, st); break;
            case 2: rc = launch_wgrad_t<2, 4>(t, (unsigned)grid, smem, st); break;
            case 3: rc = launch_wgrad_t<3, 4>(t, (unsigned)grid, smem, st); break;
            case 4: rc = launch_wgrad_t<4, 4>(t, (unsigned)grid, smem, st); break;
            case 5: rc = launch_wgrad_t<5, 4>(t, (unsigned)grid, smem, st); break;
            default: rc = launch_wgrad_t<6, 4>(t, (unsigned)grid, smem, st); break;
        }
    } else {
        switch (a.in_planes) {
            case 1: rc = launch_wgrad_t<1, 1>(t, (unsigned)grid, smem, st); break;
            case 2: rc = launch_wgrad_t<2, 1>(t, (unsigned)grid, smem, st); break;
            case 3: rc = launch_wgrad_t<3, 1>(t, (unsigned)grid, smem, st); break;
            case 4: rc = launch_wgrad_t<4, 1>(t, (unsigned)grid, smem, st); break;
            case 5: rc = launch_wgrad_t<5, 1>(t, (unsigned)grid, smem, st); break;
            case 6: rc = launch_wgrad_t<6, 1>(t, (unsigned)grid, smem, st); break;
            case 7: rc = launch_wgrad_t<7, 1>(t, (unsigned)grid, smem, st); break;
            default: rc = launch_wgrad_t<8, 1>(t, (unsigned)grid, smem, st); break;
        }
    }
    if (rc) return rc;
    *nparts = (int)grid;
    return 1;
}

}  // namespace mvb

extern "C" int mvb_set_tensor_cores(int enable) {
    const int old = mvb::tc_enabled();
    mvb::set_tc_enabled(enable ? 1 : 0);
    return old;
}
