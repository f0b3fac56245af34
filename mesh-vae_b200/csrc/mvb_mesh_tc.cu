// Mesh-resident Chebyshev layers with the basis contracted on the tensor cores (tcgen05 + TMEM).
//
// One layer of the reference's encoder / decoder loop
//     x = relu(cheb[i](x, L)); x = pool(x, D)                models/cheb_VAE.py:264-265
//     x = pool(x, U);          x = relu(cheb_dec[i](x, L))   models/cheb_VAE.py:284-285
// (ChebConv_batch.forward nn/conv.py:557-577, SurfacePool nn/pool.py:13-23) as ONE launch for every level whose
// planes fit shared memory (1250 / 313 / 79 vertices of the template).  One mesh is owned by a cluster of C = 1 or
// 2 CTAs; CTA c holds the feature columns [c*WL, (c+1)*WL) (WL = Fin / C = 8, 16 or 32) of ALL N vertices:
//
//   * the recurrence T_k = 2 L T_{k-1} - T_{k-2} is independent per feature column, so it runs entirely out of
//     shared memory with no traffic between the CTAs: two planes [N][WL] (T_k is written in place over T_{k-2}),
//     the operator staged as packed (column, value) pairs, one block barrier per step;
//   * the planes ARE the tensor-core operands: they are kept in the canonical K-major SWIZZLE_32B/64B/128B layout
//     of the UMMA shared-memory descriptors (row = vertex = M index, WL features = K index), so after the barrier of
//     step k one thread issues  D[128 x Fout] += T_k[tile] . W_k[c*WL .. , :]  for every 128-vertex tile straight from
//     the plane, accumulators in TMEM (N/128 tiles x Fout columns), while the other warps already compute T_{k+1};
//   * fp32 accuracy through the 3xTF32 split (mvb_tc.cu): kind::tf32 reads only the upper 19 bits of an operand, so
//     the raw fp32 plane is the `hi` operand as it stands and only lo = x - trunc(x) is written to a third plane;
//   * prologue: T_0 = x or T_0 = U x (the barycentric up-sampling, 3 entries per row, from the staged coarse rows);
//     epilogue: TMEM -> registers -> bias / ReLU -> only the rows the down-sampling D keeps are written;
//   * C = 2: each CTA holds a K-split partial of the contraction; the halves are exchanged through distributed
//     shared memory (the partner's output-column half is stored into its buffer) between two cluster barriers.
//
// Summation order of the recurrence is the CSR order with the same fmaf sequence as the step kernels
// (mvb_spmm.cu), so the basis is bit-identical to theirs; the contraction differs from the FFMA path by the
// 3xTF32 rounding (<= 2e-6 relative, tests/test_gpu_layer.py).  No atomics: deterministic.
#include "mvb_internal.cuh"
#include "mvb_tcgen05.cuh"

namespace mvb {

// threads per CTA: the recurrence is a chain of shared-memory latencies, but every step also ends in a block barrier and the
// gathers share one LSU pipe - same-box A/B of the whole step (scripts/trace_step.py): 1024 threads 923 us, 896: 907, 768: 906-908,
// 640: 914, 512: 921; every mesh launch is 1-4 us shorter at 768 than at 1024
constexpr int MT_NT = 768;
constexpr int MT_NC = MT_NT - 32;    // ... of which the last warp only issues the MMAs (and so never delays a step)
constexpr int MT_ISSUER = MT_NC;     // thread that issues tcgen05.mma / tcgen05.commit

struct MeshTcArgs {
    int N, B, Fin, Fout, K;
    const int32_t *Lrp, *Lci; const float *Lv; int Lnnz;          // CSR(L) [N x N] (forward) / CSR(L^T) (backward)
    int n_in;                                                     // rows of x (== N without U)
    const int32_t *Urp, *Uci; const float *Uv;                    // CSR(U) [N x n_in] or NULL
    int n_out; const int32_t *sel;                                // output row r = conv row sel[r]; NULL: identity
    const float *x, *w, *bias;
    int relu;
    float *out;
    int C;                                                        // CTAs per mesh
    int tiles;                                                    // ceil(N / 128)
    int tmem_cols;
    // shared-memory offsets (bytes from the 1024-aligned base)
    int o_pa, o_pb, o_lo, o_lo2, o_bhi, o_blo, o_rp, o_ce, o_inv, o_bar, total;      // o_lo2 == o_lo: single lo plane
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_f4(uint32_t addr, const float4 &v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- shared memory through 32-bit shared-space addresses: the planes are reached through run-time offsets and swapped
// pointers, for which the compiler falls back to GENERIC loads (LD.E: ncu showed every gather waiting on the long
// scoreboard, 45 us per level-1 layer); explicit ld.shared / st.shared keeps them on the LDS / STS path ----
__device__ __forceinline__ float4 lds4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts4(uint32_t a, const float4 &v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ int2 lds_i2(uint32_t a) {
    int2 v;
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_i2(uint32_t a, int x, int y) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ int lds_i(uint32_t a) {
    int v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds_f(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_i(uint32_t a, int v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_f(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }

// Swizzled byte offset of 16-byte chunk q of row r: r*RB + ((q ^ x(r)) << 4) with x(r) = the row bits the UMMA swizzle
// mode XORs in.  As r*RB has no bits below 5 + log2(WL/8), this is (r*RB | x(r) << 4) ^ (q << 4): the row part is
// precomputed per operator entry (row_code), the quad part per thread.
template <int WL>
__device__ __forceinline__ uint32_t row_code(int r) {
    constexpr int RB = WL * 4;
    const int x = (RB == 128) ? (r & 7) : (RB == 64 ? ((r >> 1) & 3) : ((r >> 2) & 1));
    return (uint32_t)(r * RB) | (uint32_t)(x << 4);
}
template <int WL>
__device__ __forceinline__ uint32_t swz(int r, int q) { return row_code<WL>(r) ^ (uint32_t)(q << 4); }

__device__ __forceinline__ void fma4m(float4 &a, float s, const float4 &x) {
    a.x = fmaf(s, x.x, a.x); a.y = fmaf(s, x.y, a.y); a.z = fmaf(s, x.z, a.z); a.w = fmaf(s, x.w, a.w);
}

// sum_j vals[j] * src[col[j]][quad] over the staged CSR row [s, e): entries are (row_code(col), value) pairs; the fmaf
// order is the CSR order of the step kernels (mvb_spmm.cu), four gathers in flight
__device__ __forceinline__ float4 gather_rc(uint32_t src, uint32_t ce, int s, int e, uint32_t qs) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = s;
    for (; j + 4 <= e; j += 4) {
        const int2 e0 = lds_i2(ce + 8u * j), e1 = lds_i2(ce + 8u * j + 8u), e2 = lds_i2(ce + 8u * j + 16u), e3 = lds_i2(ce + 8u * j + 24u);
        const float4 x0 = lds4(src + ((uint32_t)e0.x ^ qs)), x1 = lds4(src + ((uint32_t)e1.x ^ qs));
        const float4 x2 = lds4(src + ((uint32_t)e2.x ^ qs)), x3 = lds4(src + ((uint32_t)e3.x ^ qs));
        fma4m(acc, __int_as_float(e0.y), x0);
        fma4m(acc, __int_as_float(e1.y), x1);
        fma4m(acc, __int_as_float(e2.y), x2);
        fma4m(acc, __int_as_float(e3.y), x3);
    }
    if (j + 2 <= e) {
        const int2 e0 = lds_i2(ce + 8u * j), e1 = lds_i2(ce + 8u * j + 8u);
        const float4 x0 = lds4(src + ((uint32_t)e0.x ^ qs)), x1 = lds4(src + ((uint32_t)e1.x ^ qs));
        fma4m(acc, __int_as_float(e0.y), x0);
        fma4m(acc, __int_as_float(e1.y), x1);
        j += 2;
    }
    if (j < e) {
        const int2 e0 = lds_i2(ce + 8u * j);
        fma4m(acc, __int_as_float(e0.y), lds4(src + ((uint32_t)e0.x ^ qs)));
    }
    return acc;
}

__device__ __forceinline__ float4 lo_of(const float4 &v) {
    float4 h, l;
    split4(v, h, l);
    return l;
}

// operator into shared memory: rows[v] = (start, end) of row v, entries (row_code(column), value)
template <int WL>
__device__ __forceinline__ void stage_operator(const MeshTcArgs &a, uint32_t rows, uint32_t ce, int tid) {
    for (int v = tid; v < a.N; v += MT_NT) sts_i2(rows + 8u * v, __ldg(a.Lrp + v), __ldg(a.Lrp + v + 1));
    for (int base = 0; base < a.Lnnz; base += 4 * MT_NT) {
        int cc[4];
        float vv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * MT_NT + tid;
            if (i < a.Lnnz) { cc[u] = __ldg(a.Lci + i); vv[u] = __ldg(a.Lv + i); }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * MT_NT + tid;
            if (i < a.Lnnz) sts_i2(ce + 8u * i, (int)row_code<WL>(cc[u]), __float_as_int(vv[u]));
        }
    }
}

// one recurrence step out of shared memory: old <- alpha * L cur - [k >= 2] old (and its lo part); `bar` / `phase`:
// the MMAs issued after the previous step still read `lo` (and, one step earlier, `old`) - wait before the first store
template <int WL>
__device__ __forceinline__ void recur_step(uint32_t cur, uint32_t old, uint32_t plo, uint32_t rows, uint32_t ce, int N, int k,
                                           uint64_t *bar, uint32_t phase, bool wait_mma, int tid, float *gout, int64_t gstride) {
    constexpr int QL = WL / 4;
    bool waited = !wait_mma;
    for (int i = tid; i < N * QL; i += MT_NC) {
        if (tid >= MT_NC) break;            // the issuer warp
        const int v = i / QL, q = i % QL;
        const int2 se = lds_i2(rows + 8u * v);
        const uint32_t qs = (uint32_t)(q << 4);
        const float4 acc = gather_rc(cur, ce, se.x, se.y, qs);
        const uint32_t off = row_code<WL>(v) ^ qs;
        float4 o;
        if (k == 1) {
            o = make_float4(1.f * acc.x, 1.f * acc.y, 1.f * acc.z, 1.f * acc.w);
        } else {
            const float4 z = lds4(old + off);
            o.x = fmaf(-1.f, z.x, 2.f * acc.x); o.y = fmaf(-1.f, z.y, 2.f * acc.y);
            o.z = fmaf(-1.f, z.z, 2.f * acc.z); o.w = fmaf(-1.f, z.w, 2.f * acc.w);
        }
        if (!waited) {
            mbar_wait(bar, phase);
            waited = true;
        }
        sts4(old + off, o);
        sts4(plo + off, lo_of(o));
        if (gout) *reinterpret_cast<float4 *>(gout + (int64_t)v * gstride + 4 * q) = o;
    }
    if (!waited) mbar_wait(bar, phase);
}

// all MMAs of recurrence step k: every 128-row tile of the plane against W_k's rows of this CTA (3xTF32).  Issued by
// ONE thread of the warp that takes no part in the recurrence (MT_ISSUER): the descriptors of a step differ only in
// their 14-bit start-address field, so the per-tile work is a 64-bit add per operand.
template <int WL>
__device__ __forceinline__ void issue_step_mmas(const MeshTcArgs &a, uint32_t tmem_base, uint32_t plane, uint32_t lo,
                                                uint32_t bhi, uint32_t blo, int k, int ncols_acc, uint32_t idesc) {
    constexpr int RB = WL * 4;
    constexpr uint32_t LT = (RB == 128) ? 2u : (RB == 64 ? 4u : 6u);
    constexpr uint32_t SBO = 8u * RB;
    const uint32_t b_tile = (uint32_t)(ncols_acc * RB);
    const uint64_t ah0 = make_desc(plane, 16, SBO, LT), al0 = make_desc(lo, 16, SBO, LT);
    const uint64_t bh0 = make_desc(bhi + k * b_tile, 16, SBO, LT), bl0 = make_desc(blo + k * b_tile, 16, SBO, LT);
    for (int t = 0; t < a.tiles; ++t) {
        const uint32_t d = tmem_base + (uint32_t)(t * ncols_acc);
#pragma unroll
        for (int j = 0; j < WL / 8; ++j) {
            const uint64_t ao = (uint64_t)((t * 128 * RB + j * 32) >> 4), bo = (uint64_t)((j * 32) >> 4);
            umma_tf32(d, al0 + ao, bh0 + bo, idesc, (k > 0 || j > 0) ? 1u : 0u);     // small terms first
            umma_tf32(d, ah0 + ao, bl0 + bo, idesc, 1u);
            umma_tf32(d, ah0 + ao, bh0 + bo, idesc, 1u);
        }
    }
}

// 16-column TMEM chunks [lo, hi) that cover the columns [c0, c0 + H) of a W-column accumulator
__device__ __forceinline__ int chunk_lo(int c0) { return c0 & ~15; }
__device__ __forceinline__ int chunk_hi(int c0, int H, int W) { const int e = (c0 + H + 15) & ~15; return e < W ? e : W; }

// T_0 = U x through the coarse rows staged (unswizzled, [n_in][FL floats]) at `tmp`; U's entries are read from global
// memory (used once).  Row arithmetic of the pooling SpMM: 1.f * sum_j v_j x_j in CSR order.
__device__ __forceinline__ float4 upsample_row(const MeshTcArgs &a, uint32_t tmp, int v, int q, int FQ) {
    const int s = __ldg(a.Urp + v), e = __ldg(a.Urp + v + 1);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = s; j < e; ++j) fma4m(acc, __ldg(a.Uv + j), lds4(tmp + (uint32_t)((__ldg(a.Uci + j) * FQ + q) * 16)));
    return make_float4(1.f * acc.x, 1.f * acc.y, 1.f * acc.z, 1.f * acc.w);
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
template <int WL>
__global__ void __launch_bounds__(MT_NT, 1)
cheb_mesh_tc_fwd_kernel(const MeshTcArgs a) {
    extern __shared__ __align__(1024) char mt_smem_raw[];
    const uint32_t sm = (smem_u32(mt_smem_raw) + 1023u) & ~1023u;
    constexpr int RB = WL * 4, QL = WL / 4;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = (a.C > 1) ? (int)cluster_ctarank() : 0;
    const int b = (a.C > 1) ? blockIdx.x / a.C : blockIdx.x;
    const int N = a.N, Fin = a.Fin, Fout = a.Fout, K = a.K;
    const uint32_t pa = sm + a.o_pa, pb = sm + a.o_pb, plo = sm + a.o_lo, plo2 = sm + a.o_lo2;
    const bool lo2 = a.o_lo2 != a.o_lo;                  // lo parts of odd steps in their own plane
    const uint32_t bhi = sm + a.o_bhi, blo = sm + a.o_blo;
    const uint32_t rows = sm + a.o_rp, ce = sm + a.o_ce, inv = sm + a.o_inv;
    char *smg = mt_smem_raw + (sm - smem_u32(mt_smem_raw));       // generic view of the aligned base (barrier, TMEM slot)
    uint64_t *bar = reinterpret_cast<uint64_t *>(smg + a.o_bar);
    uint32_t *slot = reinterpret_cast<uint32_t *>(bar + 2);            // bar[0]: commits of even steps (all steps without lo2), bar[1]: odd

    pdl_trigger();
    if (warp == 0) tmem_alloc(slot, (uint32_t)a.tmem_cols);
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_barrier_init();
    }
    stage_operator<WL>(a, rows, ce, tid);
    // ---- B operands: Bt_k[n][kd] = W_k[c*WL + kd][n], K-major, swizzled like the planes, hi / lo ----
    for (int i = tid; i < K * WL * Fout; i += MT_NT) {
        const int n = i % Fout, kk = i / Fout;
        const int kd = kk % WL, k = kk / WL;
        const float wv = __ldg(a.w + ((int64_t)k * Fin + c * WL + kd) * Fout + n);
        float h, l;
        split_tf32(wv, h, l);
        const uint32_t off = (uint32_t)(k * Fout * RB) + swz<WL>(n, kd >> 2) + (uint32_t)((kd & 3) << 2);
        sts_f(bhi + off, h);
        sts_f(blo + off, l);
    }
    if (a.sel) {
        for (int v = tid; v < N; v += MT_NT) sts_i(inv + 4u * v, -1);
    }
    pdl_wait();          // everything above reads only the operator and the weights; x is the previous kernel's output
    // ---- T_0 into plane A (+ its lo part) ----
    const int64_t xrow = (int64_t)a.B * Fin;               // floats between consecutive vertices of one mesh
    const float *xb = a.x + (int64_t)b * Fin + c * WL;
    if (a.Urp) {
        // coarse rows of this mesh (unswizzled [n_in][WL]) into plane B, then T_0 = U x
        for (int base = 0; base < a.n_in * QL; base += 4 * MT_NT) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = base + u * MT_NT + tid;
                if (i < a.n_in * QL) v[u] = __ldg(reinterpret_cast<const float4 *>(xb + (int64_t)(i / QL) * xrow) + (i % QL));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = base + u * MT_NT + tid;
                if (i < a.n_in * QL) sts4(pb + (uint32_t)i * 16u, v[u]);
            }
        }
        __syncthreads();
        for (int i = tid; i < N * QL; i += MT_NT) {
            const int v = i / QL, q = i % QL;
            const float4 o = upsample_row(a, pb, v, q, QL);
            const uint32_t off = swz<WL>(v, q);
            sts4(pa + off, o);
            sts4(plo + off, lo_of(o));
        }
    } else {
        for (int base = 0; base < N * QL; base += 4 * MT_NT) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = base + u * MT_NT + tid;
                if (i < N * QL) v[u] = __ldg(reinterpret_cast<const float4 *>(xb + (int64_t)(i / QL) * xrow) + (i % QL));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = base + u * MT_NT + tid;
                if (i < N * QL) {
                    const uint32_t off = swz<WL>(i / QL, i % QL);
                    sts4(pa + off, v[u]);
                    sts4(plo + off, lo_of(v[u]));
                }
            }
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (a.sel) {
        for (int r = tid; r < a.n_out; r += MT_NT) sts_i(inv + 4u * (uint32_t)__ldg(a.sel + r), r);
    }
    const uint32_t tmem_base = *slot;
    const uint32_t idesc = make_idesc(128, Fout, 0, 0);
    if (tid == MT_ISSUER) {
        issue_step_mmas<WL>(a, tmem_base, pa, plo, bhi, blo, 0, Fout, idesc);
        umma_commit(bar);
    }
    // ---- recurrence steps: T_k into `old` (over T_{k-2}), its MMAs overlap the next step.  Before its first store a
    // thread waits for the MMAs that still read what it overwrites: those of step k-1 (single lo plane), or - with the
    // second lo plane - only those of step k-2, committed to the barrier of this step's parity ----
    uint32_t cur = pa, old = pb;
    for (int k = 1; k < K; ++k) {
        const uint32_t lo_k = (lo2 && (k & 1)) ? plo2 : plo;
        uint64_t *bar_w = lo2 ? bar + (k & 1) : bar;
        const uint32_t par_w = lo2 ? (uint32_t)(((k >> 1) + 1) & 1) : (uint32_t)((k - 1) & 1);
        recur_step<WL>(cur, old, lo_k, rows, ce, N, k, bar_w, par_w, !(lo2 && k < 2), tid, nullptr, 0);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (tid == MT_ISSUER) {
            tc_fence_after();
            issue_step_mmas<WL>(a, tmem_base, old, lo_k, bhi, blo, k, Fout, idesc);
            umma_commit(lo2 ? bar + (k & 1) : bar);
        }
        const uint32_t t = cur; cur = old; old = t;
    }
    const int kl = K - 1;          // the last commit (tcgen05.commit tracks every MMA issued before it)
    mbar_wait(lo2 ? bar + (kl & 1) : bar, lo2 ? (uint32_t)((kl >> 1) & 1) : (uint32_t)(kl & 1));
    tc_fence_after();

    // ---- epilogue: TMEM -> registers -> bias / ReLU -> the rows D keeps ----
    const int quarter = warp & 3, group = warp >> 2;            // a warp reads TMEM lanes [32 (warp % 4), +32)
    constexpr int NG = MT_NT / 128;
    if (a.C == 1) {
        for (int t = group; t < a.tiles; t += NG) {
            const int row = t * 128 + quarter * 32 + lane;
            const int ro = (row < N) ? (a.sel ? lds_i(inv + 4u * row) : row) : -1;
            for (int n0 = 0; n0 < Fout; n0 += 16) {
                float v[16];
                tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * Fout + n0), v);
                if (ro >= 0) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        if (a.bias) v[j] += __ldg(a.bias + n0 + j);
                        if (a.relu) v[j] = fmaxf(v[j], 0.f);
                    }
                    float4 *dst = reinterpret_cast<float4 *>(a.out + ((int64_t)ro * a.B + b) * Fout + n0);
                    dst[0] = make_float4(v[0], v[1], v[2], v[3]);
                    dst[1] = make_float4(v[4], v[5], v[6], v[7]);
                    dst[2] = make_float4(v[8], v[9], v[10], v[11]);
                    dst[3] = make_float4(v[12], v[13], v[14], v[15]);
                }
            }
        }
    } else {
        // K-split partials: this CTA finalises the output columns [c*H, (c+1)*H), H = Fout / 2.  Phase A: the partner's
        // column half of every row goes into ITS buffer theirs[row][H] (over the dead plane B) through DSMEM; phase B
        // (after the cluster barrier): own half from TMEM + the partner's contribution -> bias / ReLU -> global.
        const int H = Fout >> 1, HQ = H >> 2;
        const uint32_t theirs = pb;
        cluster_sync_all();                      // the partner's MMAs no longer read its planes
        const uint32_t theirs_remote = map_to_cta(theirs, (uint32_t)(c ^ 1));
        const int ps = (c ^ 1) * H;              // first column of the partner's half
        for (int t = group; t < a.tiles; t += NG) {
            const int row = t * 128 + quarter * 32 + lane;
            for (int n0 = chunk_lo(ps); n0 < chunk_hi(ps, H, Fout); n0 += 16) {
                float v[16];
                tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * Fout + n0), v);
                if (row < N) {
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const int col = n0 + 4 * j4 - ps;                    // column inside the partner's half
                        if (col >= 0 && col < H)
                            st_cluster_f4(theirs_remote + (uint32_t)((row * HQ + (col >> 2)) * 16),
                                          make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]));
                    }
                }
            }
        }
        cluster_sync_all();                      // both halves are in place
        for (int t = group; t < a.tiles; t += NG) {
            const int row = t * 128 + quarter * 32 + lane;
            const int ro = (row < N) ? (a.sel ? lds_i(inv + 4u * row) : row) : -1;
            for (int n0 = chunk_lo(c * H); n0 < chunk_hi(c * H, H, Fout); n0 += 16) {
                float v[16];
                tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * Fout + n0), v);
                if (ro >= 0) {
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const int col = n0 + 4 * j4 - c * H;                 // column inside this CTA's half
                        if (col < 0 || col >= H) continue;
                        const float4 o = lds4(theirs + (uint32_t)((row * HQ + (col >> 2)) * 16));
                        float4 r = make_float4(v[4 * j4] + o.x, v[4 * j4 + 1] + o.y, v[4 * j4 + 2] + o.z, v[4 * j4 + 3] + o.w);
                        const int gc = c * H + col;
                        if (a.bias) {
                            r.x += __ldg(a.bias + gc); r.y += __ldg(a.bias + gc + 1); r.z += __ldg(a.bias + gc + 2); r.w += __ldg(a.bias + gc + 3);
                        }
                        if (a.relu) { r.x = fmaxf(r.x, 0.f); r.y = fmaxf(r.y, 0.f); r.z = fmaxf(r.z, 0.f); r.w = fmaxf(r.w, 0.f); }
                        *reinterpret_cast<float4 *>(a.out + ((int64_t)ro * a.B + b) * Fout + gc) = r;
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)a.tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// backward (adjoint form, mvb_api.cu): G = dY * [y > 0] scattered to the rows D keeps, S_k = T_k(L^T) G on
// Fout-wide planes, dX = sum_k S_k W_k^T contracted tile by tile on the tensor cores, [U^T epilogue].  The planes
// S_0..S_{K-1} (and T_0 = U x when the layer has an up-sampling prologue) go to global memory for the
// weight-gradient reduction dW_k = T_0^T S_k, whose long dimension (the rows) is the K of the MMA: it stays a
// streaming kernel over all meshes (tc_wgrad_kernel, one MMA per 8 rows for all k at once) - inside a per-mesh CTA
// it would be paced by its own MMA count.  db: per-mesh column sums of G, summed over the meshes in order.
// ---------------------------------------------------------------------------------------------
struct MeshTcBwdArgs {
    MeshTcArgs m;                       // N, B, Fin, Fout, K, CSR(L^T) in Lrp/Lci/Lv, U (for T_0), sel, x, w; out = dx or NULL
    const int32_t *Utrp, *Utci; const float *Utv;       // CSR(U^T) [n_in x N] (dx through the up-sampling)
    const float *dy, *y;                // [n_out, B, Fout]; y == NULL: no ReLU mask
    float *S;                           // [K][N][B][Fout]
    float *T0;                          // [N][B][Fin] (only with U)
    float *dbp;                         // [B][Fout] or NULL
    int o_red;                          // shared-memory offset of the column-sum scratch
};

template <int WL>
__global__ void __launch_bounds__(MT_NT, 1)
cheb_mesh_tc_bwd_kernel(const MeshTcBwdArgs g) {
    extern __shared__ __align__(1024) char mt_smem_raw[];
    const uint32_t sm = (smem_u32(mt_smem_raw) + 1023u) & ~1023u;
    const MeshTcArgs &a = g.m;
    constexpr int RB = WL * 4, QL = WL / 4;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = (a.C > 1) ? (int)cluster_ctarank() : 0;
    const int b = (a.C > 1) ? blockIdx.x / a.C : blockIdx.x;
    const int N = a.N, Fin = a.Fin, Fout = a.Fout, K = a.K;
    const uint32_t pa = sm + a.o_pa, pb = sm + a.o_pb, plo = sm + a.o_lo, plo2 = sm + a.o_lo2;
    const bool lo2 = a.o_lo2 != a.o_lo;                  // lo parts of odd steps in their own plane
    const uint32_t bhi = sm + a.o_bhi, blo = sm + a.o_blo;
    const uint32_t rows = sm + a.o_rp, ce = sm + a.o_ce, inv = sm + a.o_inv, red = sm + g.o_red;
    char *smg = mt_smem_raw + (sm - smem_u32(mt_smem_raw));
    uint64_t *bar = reinterpret_cast<uint64_t *>(smg + a.o_bar);
    uint32_t *slot = reinterpret_cast<uint32_t *>(bar + 2);            // bar[0]: commits of even steps (all steps without lo2), bar[1]: odd

    pdl_trigger();
    if (warp == 0) tmem_alloc(slot, (uint32_t)a.tmem_cols);
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_barrier_init();
    }
    stage_operator<WL>(a, rows, ce, tid);
    // B operands of dX += S_k W_k^T: Bt_k[n = fi][kd = fo - c*WL] = W_k[fi][fo]
    for (int i = tid; i < K * Fin * WL; i += MT_NT) {
        const int kd = i % WL, kk = i / WL;
        const int n = kk % Fin, k = kk / Fin;
        const float wv = __ldg(a.w + ((int64_t)k * Fin + n) * Fout + c * WL + kd);
        float h, l;
        split_tf32(wv, h, l);
        const uint32_t off = (uint32_t)(k * Fin * RB) + swz<WL>(n, kd >> 2) + (uint32_t)((kd & 3) << 2);
        sts_f(bhi + off, h);
        sts_f(blo + off, l);
    }
    for (int v = tid; v < N; v += MT_NT) sts_i(inv + 4u * v, a.sel ? -1 : v);
    pdl_wait();          // operator, weights and shared-memory set-up above; x / dy / y and every global write below
    // ---- T_0 = U x of this CTA's share of the input features, straight to global (operand of the weight gradient) ----
    if (a.Urp && g.T0) {
        const int FL = Fin / a.C, FQ = FL >> 2;
        const float *xb = a.x + (int64_t)b * Fin + c * FL;
        const int64_t xrow = (int64_t)a.B * Fin;
        for (int i = tid; i < a.n_in * FQ; i += MT_NT)
            sts4(pb + (uint32_t)i * 16u, __ldg(reinterpret_cast<const float4 *>(xb + (int64_t)(i / FQ) * xrow) + (i % FQ)));
        __syncthreads();
        for (int i = tid; i < N * FQ; i += MT_NT) {
            const int v = i / FQ, q = i % FQ;
            *reinterpret_cast<float4 *>(g.T0 + ((int64_t)v * a.B + b) * Fin + c * FL + 4 * q) = upsample_row(a, pb, v, q, FQ);
        }
    }
    __syncthreads();
    if (a.sel) {
        for (int r = tid; r < a.n_out; r += MT_NT) sts_i(inv + 4u * (uint32_t)__ldg(a.sel + r), r);
        __syncthreads();
    }
    // ---- S_0 = G ----
    const int64_t plane_g = (int64_t)N * a.B * Fout;           // floats per S plane in global memory
    const int64_t grow = (int64_t)a.B * Fout;
    {
        const float *dyb = g.dy + (int64_t)b * Fout + c * WL;
        const float *yb = g.y ? g.y + (int64_t)b * Fout + c * WL : nullptr;
        for (int i = tid; i < N * QL; i += MT_NT) {
            const int v = i / QL, q = i % QL;
            const int r = lds_i(inv + 4u * v);
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r >= 0) {
                o = __ldg(reinterpret_cast<const float4 *>(dyb + (int64_t)r * grow) + q);
                if (yb) {
                    const float4 yv = __ldg(reinterpret_cast<const float4 *>(yb + (int64_t)r * grow) + q);
                    o.x = yv.x > 0.f ? o.x : 0.f; o.y = yv.y > 0.f ? o.y : 0.f;
                    o.z = yv.z > 0.f ? o.z : 0.f; o.w = yv.w > 0.f ? o.w : 0.f;
                }
            }
            const uint32_t off = swz<WL>(v, q);
            sts4(pa + off, o);
            sts4(plo + off, lo_of(o));
            *reinterpret_cast<float4 *>(g.S + ((int64_t)v * a.B + b) * Fout + c * WL + 4 * q) = o;
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *slot;
    const uint32_t idesc = make_idesc(128, Fin, 0, 0);
    if (tid == MT_ISSUER) {
        issue_step_mmas<WL>(a, tmem_base, pa, plo, bhi, blo, 0, Fin, idesc);
        umma_commit(bar);
    }
    // db partial of this mesh: column sums of G in a fixed order (rows strided over NP parts, parts summed in order)
    if (g.dbp) {
        constexpr int NP = MT_NT / WL;
        const int col = tid % WL, part = tid / WL;
        float s = 0.f;
        for (int v = part; v < N; v += NP) s += lds_f(pa + swz<WL>(v, col >> 2) + (uint32_t)((col & 3) << 2));
        sts_f(red + 4u * (uint32_t)(part * WL + col), s);
        __syncthreads();
        if (tid < WL) {
            float t = 0.f;
            for (int p = 0; p < NP; ++p) t += lds_f(red + 4u * (uint32_t)(p * WL + tid));
            g.dbp[(int64_t)b * Fout + c * WL + tid] = t;
        }
    }
    uint32_t cur = pa, old = pb;
    for (int k = 1; k < K; ++k) {
        const uint32_t lo_k = (lo2 && (k & 1)) ? plo2 : plo;
        uint64_t *bar_w = lo2 ? bar + (k & 1) : bar;
        const uint32_t par_w = lo2 ? (uint32_t)(((k >> 1) + 1) & 1) : (uint32_t)((k - 1) & 1);
        recur_step<WL>(cur, old, lo_k, rows, ce, N, k, bar_w, par_w, !(lo2 && k < 2), tid,
                       g.S + (int64_t)k * plane_g + (int64_t)b * Fout + c * WL, grow);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (tid == MT_ISSUER) {
            tc_fence_after();
            issue_step_mmas<WL>(a, tmem_base, old, lo_k, bhi, blo, k, Fin, idesc);
            umma_commit(lo2 ? bar + (k & 1) : bar);
        }
        const uint32_t t = cur; cur = old; old = t;
    }
    {
        const int kl = K - 1;
        mbar_wait(lo2 ? bar + (kl & 1) : bar, lo2 ? (uint32_t)((kl >> 1) & 1) : (uint32_t)(kl & 1));
    }
    tc_fence_after();

    if (a.out) {
        // dT_0: this CTA finalises the input-feature columns [c*H, (c+1)*H), H = Fin / C.  C = 2: the partner's half of
        // the K-split partial goes into ITS buffer theirs[row][H] through DSMEM (phase A); phase B adds own half (TMEM)
        // and the partner's contribution; with an up-sampling prologue the sum is kept in shared memory for U^T.
        const int quarter = warp & 3, group = warp >> 2;
        constexpr int NG = MT_NT / 128;
        const int H = Fin / a.C, HQ = H >> 2;
        const uint32_t mine = pa, theirs = pb;
        if (a.C > 1) {
            cluster_sync_all();
            const uint32_t theirs_remote = map_to_cta(theirs, (uint32_t)(c ^ 1));
            const int ps = (c ^ 1) * H;
            for (int t = group; t < a.tiles; t += NG) {
                const int row = t * 128 + quarter * 32 + lane;
                for (int n0 = chunk_lo(ps); n0 < chunk_hi(ps, H, Fin); n0 += 16) {
                    float v[16];
                    tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * Fin + n0), v);
                    if (row < N) {
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4) {
                            const int col = n0 + 4 * j4 - ps;
                            if (col >= 0 && col < H)
                                st_cluster_f4(theirs_remote + (uint32_t)((row * HQ + (col >> 2)) * 16),
                                              make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]));
                        }
                    }
                }
            }
            cluster_sync_all();
        } else {
            __syncthreads();
        }
        for (int t = group; t < a.tiles; t += NG) {
            const int row = t * 128 + quarter * 32 + lane;
            for (int n0 = chunk_lo(c * H); n0 < chunk_hi(c * H, H, Fin); n0 += 16) {
                float v[16];
                tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * Fin + n0), v);
                if (row < N) {
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const int col = n0 + 4 * j4 - c * H;
                        if (col < 0 || col >= H) continue;
                        const uint32_t off = (uint32_t)((row * HQ + (col >> 2)) * 16);
                        float4 r = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
                        if (a.C > 1) {
                            const float4 o = lds4(theirs + off);
                            r.x += o.x; r.y += o.y; r.z += o.z; r.w += o.w;
                        }
                        if (g.Utrp) sts4(mine + off, r);
                        else *reinterpret_cast<float4 *>(a.out + ((int64_t)row * a.B + b) * Fin + c * H + col) = r;
                    }
                }
            }
        }
        if (g.Utrp) {
            __syncthreads();
            for (int i = tid; i < a.n_in * HQ; i += MT_NT) {
                const int ci = i / HQ, qh = i % HQ;
                const int s = __ldg(g.Utrp + ci), e = __ldg(g.Utrp + ci + 1);
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int j = s; j < e; ++j)
                    fma4m(acc, __ldg(g.Utv + j), lds4(mine + (uint32_t)((__ldg(g.Utci + j) * HQ + qh) * 16)));
                *reinterpret_cast<float4 *>(a.out + ((int64_t)ci * a.B + b) * Fin + c * H + 4 * qh) =
                    make_float4(1.f * acc.x, 1.f * acc.y, 1.f * acc.z, 1.f * acc.w);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)a.tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int g_mesh_tc = 1;            // 0: the FFMA mesh-resident kernels of mvb_layer.cu (A/B runs)
static int g_mesh_tc_c = 0;          // 0: automatic cluster size, 1 / 2: forced
void set_mesh_tc(int enable, int c) { g_mesh_tc = enable ? 1 : 0; g_mesh_tc_c = (c == 1 || c == 2) ? c : 0; }

static int pow2_cols_m(int n) {
    int c = 32;
    while (c < n) c <<= 1;
    return c;
}
static int al(int v, int a) { return (v + a - 1) / a * a; }

// fills the layout for (N, Fin, Fout, K, nnz) with C CTAs per mesh; false when it does not fit
static bool mesh_tc_layout(MeshTcArgs &a, int width_in, int width_acc, int C) {
    if (width_in % C) return false;
    const int WL = width_in / C;
    if (WL != 8 && WL != 16 && WL != 32) return false;
    if (width_acc != 16 && width_acc != 32) return false;
    if (C == 2 && (width_acc / 2) % 8) return false;
    a.C = C;
    a.tiles = (a.N + 127) / 128;
    if (a.tiles * width_acc > 512) return false;
    a.tmem_cols = pow2_cols_m(a.tiles * width_acc);
    const int RB = WL * 4;
    const int rows = a.n_in > a.tiles * 128 ? a.n_in : a.tiles * 128;
    int plane = al(rows * RB, 1024);
    if (C == 2) {                                   // the exchange buffers [N][width_acc / 2] alias the planes
        const int ex = al(a.N * (width_acc / 2) * 4, 1024);
        if (ex > plane) plane = ex;
    }
    int o = 0;
    a.o_pa = o; o += plane;
    a.o_pb = o; o += plane;
    a.o_lo = o; o += plane;
    a.o_bhi = o; o += al(a.K * width_acc * RB, 1024);
    a.o_blo = o; o += al(a.K * width_acc * RB, 1024);
    a.o_rp = o; o += al(a.N * 8, 16);
    a.o_ce = o; o += al(a.Lnnz * 8, 16);
    a.o_inv = o; o += al(a.N * 4, 16);
    a.o_bar = o; o += 32;
    // a second lo plane (lo parts of even / odd steps apart) when there is room: a step then only waits for the MMAs
    // issued TWO steps earlier - never in practice - instead of the ones issued just before it
    a.o_lo2 = a.o_lo;
    if ((size_t)o + plane + 4096 + 1024 <= 227 * 1024) {
        o = al(o, 1024);
        a.o_lo2 = o; o += plane;
    }
    a.total = o;
    return (size_t)a.total + 1024 <= 227 * 1024;
}

template <int WL>
static int launch_mesh_fwd_t(const MeshTcArgs &a, cudaStream_t st) {
    static DevFlags optin;
    int rc = smem_optin(cheb_mesh_tc_fwd_kernel<WL>, 227 * 1024, optin, "cheb_mesh_tc_fwd");
    if (rc) return rc;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(a.B * a.C));
    cfg.blockDim = dim3(MT_NT);
    cfg.dynamicSmemBytes = (size_t)a.total + 1024;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)a.C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, cheb_mesh_tc_fwd_kernel<WL>, a);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(MVB_ECUDA, "cheb_mesh_tc_fwd: launch: %s", cudaGetErrorString(e));
    }
    return check_launch("mvb cheb_mesh_tc_fwd");
}

// cluster size for a layer whose recurrence planes are `width_in` wide: two CTAs per mesh while that keeps every
// SM busy (or when one CTA cannot hold the mesh), else one
static int pick_mesh_c(MeshTcArgs &a, int width_in, int width_acc) {
    MeshTcArgs t1 = a, t2 = a;
    const bool ok1 = mesh_tc_layout(t1, width_in, width_acc, 1);
    const bool ok2 = mesh_tc_layout(t2, width_in, width_acc, 2);
    int c = 0;
    if (g_mesh_tc_c == 1) c = ok1 ? 1 : 0;
    else if (g_mesh_tc_c == 2) c = ok2 ? 2 : 0;
    else if (ok2 && (!ok1 || a.B * 2 <= num_sms() + num_sms() / 2)) c = 2;
    else if (ok1) c = 1;
    else if (ok2) c = 2;
    if (c == 1) a = t1;
    else if (c == 2) a = t2;
    return c;
}

// 1 = the tensor-core mesh kernel covers this layer
int mesh_tc_fwd_supported(int N, int B, int Fin, int Fout, int K, int Lnnz, int n_in, int n_out) {
    if (!g_mesh_tc || N < 1 || B < 1 || K < 1 || K > 16 || Lnnz < 0) return 0;
    MeshTcArgs a{};
    a.N = N; a.B = B; a.Fin = Fin; a.Fout = Fout; a.K = K; a.Lnnz = Lnnz; a.n_in = n_in; a.n_out = n_out;
    return pick_mesh_c(a, Fin, Fout) ? 1 : 0;
}

// returns 1 = launched, 0 = shape not covered (caller uses the FFMA mesh kernel), < 0 = error
int launch_mesh_tc_fwd(int N, int B, int Fin, int Fout, int K, const int32_t *Lrp, const int32_t *Lci, const float *Lv, int Lnnz,
                       int n_in, const int32_t *Urp, const int32_t *Uci, const float *Uv, int n_out, const int32_t *sel,
                       const float *x, const float *w, const float *bias, int relu, float *y, cudaStream_t st) {
    if (!g_mesh_tc || K > 16) return 0;
    MeshTcArgs a{};
    a.N = N; a.B = B; a.Fin = Fin; a.Fout = Fout; a.K = K;
    a.Lrp = Lrp; a.Lci = Lci; a.Lv = Lv; a.Lnnz = Lnnz;
    a.n_in = n_in; a.Urp = Urp; a.Uci = Uci; a.Uv = Uv;
    a.n_out = n_out; a.sel = sel;
    a.x = x; a.w = w; a.bias = bias; a.relu = relu; a.out = y;
    const int c = pick_mesh_c(a, Fin, Fout);
    if (!c) return 0;
    int rc;
    switch (Fin / c) {
        case 8: rc = launch_mesh_fwd_t<8>(a, st); break;
        case 16: rc = launch_mesh_fwd_t<16>(a, st); break;
        default: rc = launch_mesh_fwd_t<32>(a, st); break;
    }
    return rc ? rc : 1;
}


template <int WL>
static int launch_mesh_bwd_t(const MeshTcBwdArgs &g, cudaStream_t st) {
    static DevFlags optin;
    int rc = smem_optin(cheb_mesh_tc_bwd_kernel<WL>, 227 * 1024, optin, "cheb_mesh_tc_bwd");
    if (rc) return rc;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(g.m.B * g.m.C));
    cfg.blockDim = dim3(MT_NT);
    cfg.dynamicSmemBytes = (size_t)g.m.total + 1024;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)g.m.C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, cheb_mesh_tc_bwd_kernel<WL>, g);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(MVB_ECUDA, "cheb_mesh_tc_bwd: launch: %s", cudaGetErrorString(e));
    }
    return check_launch("mvb cheb_mesh_tc_bwd");
}

// layout of the backward kernel: recurrence planes are Fout wide, accumulators Fin wide; + the column-sum scratch
static int pick_mesh_c_bwd(MeshTcBwdArgs &g, int has_up) {
    MeshTcArgs &a = g.m;
    const int c = pick_mesh_c(a, a.Fout, a.Fin);
    if (!c) return 0;
    if (has_up) {                  // T_0 staging: n_in rows of Fin / C floats in one plane
        const int plane = a.o_pb - a.o_pa;
        if (a.n_in * (a.Fin / c) * 4 > plane || (a.Fin / c) % 4) return 0;
    }
    g.o_red = a.total;
    a.total += MT_NT * 4;
    if ((size_t)a.total + 1024 > 227 * 1024) return 0;
    return c;
}

// weight-gradient plane groups: tc_wgrad takes at most 128 feature rows (planes x Fout) per launch
static int wgrad_group(int K, int Fout) {
    const int cap = 128 / Fout > 0 ? 128 / Fout : 1;
    const int ngroups = (K + cap - 1) / cap;
    return (K + ngroups - 1) / ngroups;
}

int mesh_tc_bwd_supported(int N, int B, int Fin, int Fout, int K, int Lnnz, int n_in, int n_out, int has_up) {
    if (!g_mesh_tc || N < 1 || B < 1 || K < 1 || K > 16 || Lnnz < 0 || (int64_t)N * B < 256) return 0;
    MeshTcBwdArgs g{};
    g.m.N = N; g.m.B = B; g.m.Fin = Fin; g.m.Fout = Fout; g.m.K = K; g.m.Lnnz = Lnnz; g.m.n_in = n_in; g.m.n_out = n_out;
    return pick_mesh_c_bwd(g, has_up) ? 1 : 0;
}

// Workspace of the backward layer: S_0..S_{K-1}, T_0 (with up-sampling), the db partials, then the weight-gradient
// partials of each plane group.  A launch has at most 16 groups (K <= 16); the size query measures any K.
struct MeshBwdWs {
    float *S, *T0, *dbp;
    float *part[16];
    size_t part_bytes[16];
};
static MeshBwdWs mesh_bwd_ws(WsCarve &c, int N, int B, int Fin, int Fout, int K, int has_up) {
    MeshBwdWs w{};
    w.S = c.take<float>((size_t)K * N * B * Fout * sizeof(float));
    if (has_up) w.T0 = c.take<float>((size_t)N * B * Fin * sizeof(float));
    w.dbp = c.take<float>((size_t)B * Fout * sizeof(float));
    const int grp = wgrad_group(K, Fout);
    for (int g = 0, k0 = 0; k0 < K; ++g, k0 += grp) {
        const size_t bytes = align_up(wgrad_partial_bytes((K - k0 < grp ? K - k0 : grp) * Fout, Fin), 256);
        float *p = c.take<float>(bytes);
        if (g < 16) {
            w.part[g] = p;
            w.part_bytes[g] = bytes;
        }
    }
    return w;
}

size_t mesh_tc_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up) {
    WsCarve c;
    mesh_bwd_ws(c, N, B, Fin, Fout, K, has_up);
    return c.off;
}

// returns 1 = handled, 0 = shape not covered, < 0 = error.  Lt*: CSR(L^T); U* / Ut*: CSR(U), CSR(U^T) or NULL
int launch_mesh_tc_bwd(int N, int B, int Fin, int Fout, int K, const int32_t *Ltrp, const int32_t *Ltci, const float *Ltv, int Lnnz,
                       int n_in, const int32_t *Urp, const int32_t *Uci, const float *Uv, const int32_t *Utrp, const int32_t *Utci,
                       const float *Utv, int n_out, const int32_t *sel, const float *x, const float *w, const float *y_for_relu,
                       const float *dy, float *dx, float *dweight, float *dbias, void *workspace, size_t workspace_bytes,
                       cudaStream_t st) {
    if (!g_mesh_tc || K > 16 || (int64_t)N * B < 256) return 0;
    MeshTcBwdArgs g{};
    MeshTcArgs &a = g.m;
    a.N = N; a.B = B; a.Fin = Fin; a.Fout = Fout; a.K = K;
    a.Lrp = Ltrp; a.Lci = Ltci; a.Lv = Ltv; a.Lnnz = Lnnz;
    a.n_in = n_in; a.Urp = Urp; a.Uci = Uci; a.Uv = Uv;
    a.n_out = n_out; a.sel = sel;
    a.x = x; a.w = w; a.out = dx;
    const int has_up = Urp != nullptr;
    const int c = pick_mesh_c_bwd(g, has_up);
    if (!c) return 0;
    WsCarve carve{reinterpret_cast<char *>(workspace)};
    const MeshBwdWs ws = mesh_bwd_ws(carve, N, B, Fin, Fout, K, has_up);
    if (workspace_bytes < carve.off) return set_err(MVB_EWORKSPACE, "cheb_layer_bwd: workspace %zu < %zu", workspace_bytes, carve.off);
    g.S = ws.S;
    g.T0 = ws.T0;
    g.dbp = dbias ? ws.dbp : nullptr;
    g.Utrp = has_up ? Utrp : nullptr; g.Utci = Utci; g.Utv = Utv;
    g.dy = dy; g.y = y_for_relu;
    int rc;
    switch (Fout / c) {
        case 8: rc = launch_mesh_bwd_t<8>(g, st); break;
        case 16: rc = launch_mesh_bwd_t<16>(g, st); break;
        default: rc = launch_mesh_bwd_t<32>(g, st); break;
    }
    if (rc) return rc;
    // db and dW off the critical path: on the deferred side chain when the step engine has switched it on
    SideChain side(st, 0, false);
    const cudaStream_t ws_st = side.stream();
    if (dbias) {
        rc = launch_layer_finalize(B, 0, Fout, nullptr, g.dbp, nullptr, dbias, ws_st);
        if (rc) return rc;
    }
    // dW_k[i][o] = sum_rows T_0[row][i] S_k[row][o]: streaming tensor-core reduction over all meshes, plane groups
    const int64_t rows = (int64_t)N * B;
    const int grp = wgrad_group(K, Fout);
    for (int gi = 0, k0 = 0; k0 < K; ++gi, k0 += grp) {
        const int np = K - k0 < grp ? K - k0 : grp;
        WgradArgs wa{};
        wa.rows = rows;
        wa.in_planes = np;
        wa.in_w = Fout;
        wa.in0 = g.S + (int64_t)k0 * rows * Fout;
        wa.in_rest = g.S + (int64_t)(k0 + 1) * rows * Fout;
        wa.dy = has_up ? g.T0 : x;
        wa.n_out = Fin;
        wa.partials = ws.part[gi];
        wa.partial_bytes = ws.part_bytes[gi];
        int nA = 0, m4A = 0;
        rc = launch_wgrad_partials(wa, 0, &nA, &m4A, ws_st);
        if (rc) return rc;
        rc = launch_wgrad_finalize(wa.partials, nA, m4A, nullptr, 0, 0, Fin, np * Fin, Fout, dweight + (int64_t)k0 * Fin * Fout, nullptr,
                                   ws_st, 1);
        if (rc) return rc;
    }
    return 1;
}

}  // namespace mvb
