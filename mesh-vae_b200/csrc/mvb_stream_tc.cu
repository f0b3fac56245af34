// Row-streaming fused Chebyshev layer for the levels that do NOT fit shared memory (level 0: 4998 vertices).
//
//     x = pool(x, U);  x = relu(cheb_dec[i](x, L))          models/cheb_VAE.py:284-285
//     (ChebConv_batch.forward nn/conv.py:557-577, SurfacePool nn/pool.py:13-23)
//
// ONE persistent launch per direction instead of pool + (K-1) SpMM steps + contraction (+ mask/column-sum + U^T pool
// in backward).  The (vertex, mesh) pairs of the vertex-major tensor - 16-float rows - are cut into 128-pair tiles
// (= the M of one UMMA); CTA c owns `tiles_per_cta` consecutive tiles for the whole kernel (one CTA per SM, every CTA
// resident: 2499 tiles = 147 x 17 at 64 meshes).  Per recurrence step k
//
//   * 31 compute warps produce T_k = 2 L T_{k-1} - T_{k-2} for the CTA's pairs exactly as the step kernel does
//     (mvb_spmm.cu: one thread = one 16-byte quad, CSR order, same fmaf sequence - bit-identical basis), with the
//     CTA's band of the operator staged once in shared memory as (premultiplied row offset, value) pairs;
//   * the quad is stored to global memory (the neighbours of other CTAs gather it in step k+1) AND into a ring of
//     shared-memory stages in the canonical K-major SWIZZLE_64B UMMA layout, together with its lo = x - trunc(x) part;
//   * when the 16 warp-items of a tile have arrived on the stage's mbarrier, one thread of the 32nd warp issues
//     D[tile] += T_k[tile] . W_k (3xTF32: lo.hi + hi.lo + hi.hi) with tcgen05.mma; the accumulators of all the CTA's
//     tiles stay in TMEM (tiles_per_cta x 16 columns) across the K steps; tcgen05.commit frees the stage;
//   * a grid-wide barrier (one atomic per CTA, acquire/release fences as in cooperative groups' grid sync) separates
//     the steps.
//
// So the basis never returns from HBM for the contraction: per layer the traffic is the recurrence itself.  Forward:
// prologue T_0 = U x (3 entries per row) computed in step 0, epilogue TMEM -> bias / ReLU -> y; the last plane is never
// written.  Backward (adjoint form, mvb_api.cu): step 0 computes G = dY * [y > 0] (+ per-CTA column sums for db), the
// planes S_k = T_k(L^T) G go to global memory for the streaming weight-gradient reduction (tc_wgrad_kernel) as does
// T_0 = U x, dT_0 = sum_k S_k W_k^T comes out of TMEM, and after one more grid barrier dX = U^T dT_0 is gathered.
// No atomics on data: deterministic.
#include "mvb_internal.cuh"
#include "mvb_tcgen05.cuh"

namespace mvb {

constexpr int ST_NT_MAX = 1024;        // threads per CTA (template parameter NT; 768 / 544 measured slower); the last warp issues the MMAs
constexpr int ST_NS = 4;               // stages of the operand ring (one 128-pair tile each: 8 KB hi + 8 KB lo)
constexpr int ST_STAGE = 16384;
constexpr int ST_ECAP = 4096;          // staged operator entries per CTA
constexpr int ST_RCAP = 592;           // staged rows per CTA

struct StreamArgs {
    int N, B, K, Nacc;                                            // Nacc: accumulator width (Fout forward, Fin backward)
    const int32_t *Lrp, *Lci; const float *Lv;                    // CSR(L) forward / CSR(L^T) backward
    int n_in;
    const int32_t *Urp, *Uci; const float *Uv;                    // CSR(U) [N x n_in] or NULL
    const int32_t *Utrp, *Utci; const float *Utv;                 // backward: CSR(U^T) [n_in x N] or NULL
    const float *x;                                               // [n_in, B, 16]
    const float *w;                                               // [K][Fin][Fout]
    const float *bias; int relu;
    float *out;                                                   // forward y [N,B,Nacc]; backward dx [n_in,B,Nacc] or NULL
    const float *dy, *y;                                          // backward: [N,B,16]; y == NULL: no ReLU mask
    float *planes;                                                // forward: 3 rotating planes; backward: S [K][N][B][16]
    float *T0;                                                    // backward with U: T_0 = U x [N,B,16] (weight-gradient operand)
    float *dT0;                                                   // backward with U and dx: [N,B,Nacc]
    float *dbp;                                                   // backward: [grid][16] column sums of G, or NULL
    unsigned int *ctr;                                            // grid barrier counter, zero at launch
    // decomposition: CTA (row block rb, mesh slab) owns rows [rb*RP, +RP) x meshes [slab*SW, +SW); a tile (the M of one
    // UMMA) is 128/SW consecutive rows x the SW meshes of the slab
    int SW;                                                       // 8 or 16 meshes per slab (template parameter of the kernel)
    int RP;                                                       // rows per CTA (a multiple of 128/SW)
    int nslabs;                                                   // B / SW
    int tiles_per_cta;
    int64_t pairs;                                                // N * B
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float4 ldg_plain4(const float4 *p) {           // coherent load (data written earlier in this kernel)
    float4 v;
    asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ldg_stream4(const float4 *p) {          // coherent, read once: keep L1 for the gathered rows
    float4 v;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fma4s(float4 &a, float s, const float4 &x) {
    a.x = fmaf(s, x.x, a.x); a.y = fmaf(s, x.y, a.y); a.z = fmaf(s, x.z, a.z); a.w = fmaf(s, x.w, a.w);
}

// all CTAs of the grid: every global store before the barrier is visible to every load after it
__device__ __forceinline__ void grid_barrier(unsigned int *ctr, unsigned int target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(ctr, 1u);
        unsigned int v;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
        } while (v < target);
        __threadfence();
    }
    __syncthreads();
}

template <bool BWD, int ST_NT, int SW>
__global__ void __launch_bounds__(ST_NT, 1)
cheb_stream_tc_kernel(const StreamArgs a) {
    constexpr int ST_NW = ST_NT / 32 - 1;                          // producer warps
    extern __shared__ __align__(1024) char st_smem_raw[];
    const uint32_t sm = (smem_u32(st_smem_raw) + 1023u) & ~1023u;
    char *smg = st_smem_raw + (sm - smem_u32(st_smem_raw));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int K = a.K, B = a.B, Nacc = a.Nacc, N = a.N;
    // ---- shared memory: stages | B hi | B lo | rows | entries | column-sum scratch | barriers ----
    const uint32_t stages = sm;
    const uint32_t bhi = stages + ST_NS * ST_STAGE;
    const uint32_t b_bytes = (uint32_t)(K * Nacc * 64);
    const uint32_t blo = bhi + ((b_bytes + 1023u) & ~1023u);
    char *g_rp = smg + (blo - sm) + ((b_bytes + 1023u) & ~1023u);
    int2 *row_s = reinterpret_cast<int2 *>(g_rp);                             // [ST_RCAP] (start, end) into ent_s
    int2 *ent_s = row_s + ST_RCAP;                                            // [ST_ECAP] (row offset in float4 units, value)
    float4 *red = reinterpret_cast<float4 *>(ent_s + ST_ECAP);                // [ST_NW * 32] (backward)
    uint64_t *full = reinterpret_cast<uint64_t *>(reinterpret_cast<char *>(red) + (BWD ? ST_NW * 32 * 16 : 0));
    uint64_t *empty = full + ST_NS;
    uint64_t *done = empty + ST_NS;
    uint32_t *slot = reinterpret_cast<uint32_t *>(done + 1);

    const int cta = blockIdx.x;
    const int rb = cta / a.nslabs, slab = cta - rb * a.nslabs;
    const int R0 = rb * a.RP;
    const int my_rows = min(a.RP, N - R0);
    constexpr int rpt = 128 / SW;                                     // rows per tile
    const int my_tiles = (my_rows + rpt - 1) / rpt;
    const int n_witems = my_tiles * 16;                           // warp-items: 32 quads = 512 contiguous bytes (SW = 4: 2 x 256)
    const int nq = B * 4;                                         // quads per row

    const int tmem_need = a.tiles_per_cta * Nacc;
    const int tmem_cols = tmem_need <= 32 ? 32 : (tmem_need <= 64 ? 64 : (tmem_need <= 128 ? 128 : (tmem_need <= 256 ? 256 : 512)));
    if (warp == 0) tmem_alloc(slot, (uint32_t)tmem_cols);
    if (tid == 0) {
        for (int s = 0; s < ST_NS; ++s) {
            mbar_init(full + s, 16);
            mbar_init(empty + s, 1);
        }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    // ---- the CTA's band of the operator ----
    const int e_first = __ldg(a.Lrp + R0);
    for (int i = tid; i < my_rows; i += ST_NT) row_s[i] = make_int2(__ldg(a.Lrp + R0 + i) - e_first, __ldg(a.Lrp + R0 + i + 1) - e_first);
    {
        const int n_ent = __ldg(a.Lrp + R0 + my_rows) - e_first;
        for (int i = tid; i < n_ent && i < ST_ECAP; i += ST_NT)
            ent_s[i] = make_int2(__ldg(a.Lci + e_first + i) * nq, __float_as_int(__ldg(a.Lv + e_first + i)));
    }
    // ---- B operands, K-major SWIZZLE_64B, hi / lo.  forward: Bt_k[n = fo][kd = fi] = W_k[fi][fo];
    //      backward (dT_0 += S_k W_k^T): Bt_k[n = fi][kd = fo] = W_k[fi][fo] ----
    for (int i = tid; i < K * 16 * Nacc; i += ST_NT) {
        const int kd = i & 15, n = (i >> 4) % Nacc, k = (i >> 4) / Nacc;
        const float wv = BWD ? __ldg(a.w + ((int64_t)k * Nacc + n) * 16 + kd) : __ldg(a.w + ((int64_t)k * 16 + kd) * Nacc + n);
        float h, l;
        split_tf32(wv, h, l);
        const uint32_t off = (uint32_t)(k * Nacc * 64) + swz_off(n, kd >> 2, 64) + (uint32_t)((kd & 3) << 2);
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(bhi + off), "f"(h) : "memory");
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(blo + off), "f"(l) : "memory");
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *slot;
    const uint32_t idesc = make_idesc(128, Nacc, 0, 0);
    const int64_t plane4 = a.pairs * 4;                   // float4 quads per plane
    float4 *planes4 = reinterpret_cast<float4 *>(a.planes);
    const bool has_u = a.Urp != nullptr;
    float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);         // backward: this thread's column sums of G

    // ---- lane geometry (fixed for the whole kernel): a warp-item is one row x 8 meshes (sub-slab `sub` of the slab) ----
    constexpr int SH = SW == 16 ? 1 : 0;                  // log2(sub-slabs per row)
    const int q = lane & 3, l3 = lane >> 2;               // quad of the 16 features, mesh within the sub-slab
    const int mq_lane = slab * SW * 4 + lane;             // + sub * 32: quad within the row
    // pair index inside a tile: pr = rit * SW + sub * 8 + l3; its SWIZZLE_64B offset is rit * SW * 64 + sub * 512 + a lane constant
    const uint32_t soff_lane = (uint32_t)(l3 * 64 + ((q ^ ((l3 >> 1) & 3)) << 4));

    // one item into the stage of its tile (hi = the raw fp32 value: kind::tf32 reads its upper 19 bits) + arrive
    auto stage_item = [&](const float4 &o, int k, int rowl, int sub) {
        const int t = rowl >> (4 - SH);
        const int seq = k * my_tiles + t, s = seq % ST_NS;
        if (seq >= ST_NS) mbar_wait(empty + s, (uint32_t)(((seq / ST_NS) - 1) & 1));
        float4 h, l;
        split4(o, h, l);
        const uint32_t off = stages + s * ST_STAGE + (uint32_t)((rowl & ((16 >> SH) - 1)) * (SW * 64) + sub * 512) + soff_lane;
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(off), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w) : "memory");
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(off + 8192u), "f"(l.x), "f"(l.y), "f"(l.z), "f"(l.w) : "memory");
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(full + s);
    };

    unsigned int bar_no = 0;
    for (int k = 0; k < K; ++k) {
        if (warp == ST_NW) {
            // ---- MMA issuer: tile by tile as the stages fill ----
            if (lane == 0) {
                for (int t = 0; t < my_tiles; ++t) {
                    const int seq = k * my_tiles + t, s = seq % ST_NS;
                    mbar_wait(full + s, (uint32_t)((seq / ST_NS) & 1));
                    tc_fence_after();
                    const uint32_t hi = stages + s * ST_STAGE, lo = hi + 8192;
                    const uint32_t d = tmem_base + (uint32_t)(t * Nacc);
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const uint64_t ah = make_desc(hi + j * 32, 16, 512, 4u), al = make_desc(lo + j * 32, 16, 512, 4u);
                        const uint64_t bh = make_desc(bhi + k * Nacc * 64 + j * 32, 16, 512, 4u);
                        const uint64_t bl = make_desc(blo + k * Nacc * 64 + j * 32, 16, 512, 4u);
                        umma_tf32(d, al, bh, idesc, (k > 0 || j > 0) ? 1u : 0u);      // small terms first
                        umma_tf32(d, ah, bl, idesc, 1u);
                        umma_tf32(d, ah, bh, idesc, 1u);
                    }
                    umma_commit(empty + s);
                }
                if (k == K - 1) umma_commit(done);
            }
            __syncwarp();
        } else if (k == 0) {
            // ---- step 0: T_0 = x or U x (forward), G = dY * [y > 0] (backward; + T_0 = U x for the weight gradient) ----
            float4 *dst = BWD ? planes4 : (has_u ? planes4 : nullptr);
            for (int g = warp; g < n_witems; g += ST_NW) {
                const int sub = g & ((1 << SH) - 1), rowl = g >> SH;
                float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                if (rowl < my_rows) {
                    const int r = R0 + rowl, mq = mq_lane + sub * 32;
                    const int e4 = r * nq + mq;
                    if (BWD) {
                        o = __ldg(reinterpret_cast<const float4 *>(a.dy) + e4);
                        if (a.y) {
                            const float4 yv = __ldg(reinterpret_cast<const float4 *>(a.y) + e4);
                            o.x = yv.x > 0.f ? o.x : 0.f; o.y = yv.y > 0.f ? o.y : 0.f;
                            o.z = yv.z > 0.f ? o.z : 0.f; o.w = yv.w > 0.f ? o.w : 0.f;
                        }
                        cs.x += o.x; cs.y += o.y; cs.z += o.z; cs.w += o.w;
                    }
                    if (has_u && (!BWD || a.T0)) {
                        // T_0 = U x: the pooling SpMM's arithmetic (1.f * sum_j v_j x_j in CSR order)
                        const int s = __ldg(a.Urp + r), e = __ldg(a.Urp + r + 1);
                        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                        const float4 *x4 = reinterpret_cast<const float4 *>(a.x) + mq;
                        for (int j = s; j < e; ++j) fma4s(acc, __ldg(a.Uv + j), __ldg(x4 + __ldg(a.Uci + j) * nq));
                        const float4 u = make_float4(1.f * acc.x, 1.f * acc.y, 1.f * acc.z, 1.f * acc.w);
                        if (BWD) reinterpret_cast<float4 *>(a.T0)[e4] = u;
                        else o = u;
                    } else if (!BWD) {
                        o = __ldg(reinterpret_cast<const float4 *>(a.x) + e4);
                    }
                    if (dst) dst[e4] = o;
                }
                stage_item(o, 0, rowl, sub);
            }
        } else {
            // ---- steps k >= 1: warp-items in row order (the 31 warps form a window that slides down the CTA's rows, so the
            // rows they gather stay in L1 as in the step kernel) ----
            const float4 *src, *old = nullptr;
            float4 *dst = nullptr;
            if (!BWD) {
                src = (k == 1 && !has_u) ? reinterpret_cast<const float4 *>(a.x) : planes4 + (int64_t)((k - 1) % 3) * plane4;
                if (k >= 2) old = (k == 2 && !has_u) ? reinterpret_cast<const float4 *>(a.x) : planes4 + (int64_t)((k - 2) % 3) * plane4;
                if (k < K - 1) dst = planes4 + (int64_t)(k % 3) * plane4;               // the last plane is never gathered
            } else {
                src = planes4 + (int64_t)(k - 1) * plane4;
                if (k >= 2) old = planes4 + (int64_t)(k - 2) * plane4;
                dst = planes4 + (int64_t)k * plane4;
            }
            const float alpha = k == 1 ? 1.f : 2.f;
            for (int g = warp; g < n_witems; g += ST_NW) {
                const int sub = g & ((1 << SH) - 1), rowl = g >> SH;
                float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                if (rowl < my_rows) {
                    const int mq = mq_lane + sub * 32;
                    const int e4 = (R0 + rowl) * nq + mq;
                    float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (old) z = ldg_stream4(old + e4);
                    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                    const float4 *sq = src + mq;
                    const int2 se = row_s[rowl];
                    int j = se.x;
                    const int e = se.y;
                    if (e <= ST_ECAP) {
                        for (; j + 4 <= e; j += 4) {
                            const int2 e0 = ent_s[j], e1 = ent_s[j + 1], e2 = ent_s[j + 2], e3 = ent_s[j + 3];
                            const float4 x0 = ldg_plain4(sq + e0.x), x1 = ldg_plain4(sq + e1.x);
                            const float4 x2 = ldg_plain4(sq + e2.x), x3 = ldg_plain4(sq + e3.x);
                            fma4s(acc, __int_as_float(e0.y), x0);
                            fma4s(acc, __int_as_float(e1.y), x1);
                            fma4s(acc, __int_as_float(e2.y), x2);
                            fma4s(acc, __int_as_float(e3.y), x3);
                        }
                        if (j + 2 <= e) {
                            const int2 e0 = ent_s[j], e1 = ent_s[j + 1];
                            const float4 x0 = ldg_plain4(sq + e0.x), x1 = ldg_plain4(sq + e1.x);
                            fma4s(acc, __int_as_float(e0.y), x0);
                            fma4s(acc, __int_as_float(e1.y), x1);
                            j += 2;
                        }
                        if (j < e) {
                            const int2 e0 = ent_s[j];
                            fma4s(acc, __int_as_float(e0.y), ldg_plain4(sq + e0.x));
                        }
                    } else {                     // (a band with more entries than the staging area holds)
                        for (j += e_first; j < e + e_first; ++j) fma4s(acc, __ldg(a.Lv + j), ldg_plain4(sq + __ldg(a.Lci + j) * nq));
                    }
                    // k == 1: 1.f * acc; k >= 2: fmaf(-1, z, 2 * acc) - the step kernel's arithmetic (z = 0 when k == 1)
                    o.x = alpha * acc.x; o.y = alpha * acc.y; o.z = alpha * acc.z; o.w = alpha * acc.w;
                    if (old) {
                        o.x = fmaf(-1.f, z.x, o.x); o.y = fmaf(-1.f, z.y, o.y);
                        o.z = fmaf(-1.f, z.z, o.z); o.w = fmaf(-1.f, z.w, o.w);
                    }
                    if (dst) dst[e4] = o;
                }
                stage_item(o, k, rowl, sub);
            }
        }
        if (k < K - 1) {
            ++bar_no;
            grid_barrier(a.ctr, bar_no * gridDim.x);
        }
    }
    // ---- every MMA done ----
    mbar_wait(done, 0);
    tc_fence_after();
    const int quarter = warp & 3, group = warp >> 2;
    float *eout = BWD ? (a.Utrp ? a.dT0 : a.out) : a.out;
    if (eout && warp < (ST_NT / 128) * 4) {
        // TMEM lane pr of tile t = (row in tile, mesh in slab): pr = rit * SW + mesh
        const int pr = quarter * 32 + lane;
        const int rit = pr / SW, mesh = slab * SW + (pr - rit * SW);
        for (int t = group; t < my_tiles; t += ST_NT / 128) {
            const int rowl = t * rpt + rit;
            for (int n0 = 0; n0 < Nacc; n0 += 16) {
                float v[16];
                tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * Nacc + n0), v);
                if (rowl < my_rows) {
                    if (!BWD) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            if (a.bias) v[j] += __ldg(a.bias + n0 + j);
                            if (a.relu) v[j] = fmaxf(v[j], 0.f);
                        }
                    }
                    float4 *dst = reinterpret_cast<float4 *>(eout + ((int64_t)(R0 + rowl) * B + mesh) * Nacc + n0);
                    dst[0] = make_float4(v[0], v[1], v[2], v[3]);
                    dst[1] = make_float4(v[4], v[5], v[6], v[7]);
                    dst[2] = make_float4(v[8], v[9], v[10], v[11]);
                    dst[3] = make_float4(v[12], v[13], v[14], v[15]);
                }
            }
        }
    }
    if (BWD) {
        if (a.dbp) {
            // column sums of G over this CTA's block in a fixed order: per-thread sums -> 8 parts per column -> in order
            if (warp < ST_NW) red[tid] = cs;
            __syncthreads();
            float *redf = reinterpret_cast<float *>(red);
            float part = 0.f;
            const int col = tid & 15, pt = tid >> 4;             // threads 0..127: column, part
            if (tid < 128) {
                const int qq = col >> 2;
                for (int u = 0; u < ST_NW; ++u) part += redf[(qq + 4 * (pt * ST_NW + u)) * 4 + (col & 3)];
            }
            __syncthreads();
            if (tid < 128) redf[pt * 16 + col] = part;
            __syncthreads();
            if (tid < 16) {
                float s = 0.f;
                for (int u = 0; u < 8; ++u) s += redf[u * 16 + tid];
                a.dbp[(int64_t)cta * 16 + tid] = s;
            }
        }
        if (a.Utrp && a.out) {
            // dX = U^T dT_0 (the pooling SpMM's arithmetic) once every CTA's dT_0 tiles are in global memory
            ++bar_no;
            grid_barrier(a.ctr, bar_no * gridDim.x);
            const int64_t items = (int64_t)a.n_in * B * (Nacc / 4);
            const int nqa = B * (Nacc / 4);
            const float4 *d4 = reinterpret_cast<const float4 *>(a.dT0);
            for (int64_t i = (int64_t)cta * ST_NT + tid; i < items; i += (int64_t)gridDim.x * ST_NT) {
                const int ci = (int)(i / nqa), mqa = (int)(i - (int64_t)ci * nqa);
                const int s = __ldg(a.Utrp + ci), e = __ldg(a.Utrp + ci + 1);
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                int j = s;
                for (; j + 4 <= e; j += 4) {
                    const float4 x0 = ldg_plain4(d4 + (int64_t)__ldg(a.Utci + j) * nqa + mqa), x1 = ldg_plain4(d4 + (int64_t)__ldg(a.Utci + j + 1) * nqa + mqa);
                    const float4 x2 = ldg_plain4(d4 + (int64_t)__ldg(a.Utci + j + 2) * nqa + mqa), x3 = ldg_plain4(d4 + (int64_t)__ldg(a.Utci + j + 3) * nqa + mqa);
                    fma4s(acc, __ldg(a.Utv + j), x0);
                    fma4s(acc, __ldg(a.Utv + j + 1), x1);
                    fma4s(acc, __ldg(a.Utv + j + 2), x2);
                    fma4s(acc, __ldg(a.Utv + j + 3), x3);
                }
                for (; j < e; ++j) fma4s(acc, __ldg(a.Utv + j), ldg_plain4(d4 + (int64_t)__ldg(a.Utci + j) * nqa + mqa));
                reinterpret_cast<float4 *>(a.out)[i] = make_float4(1.f * acc.x, 1.f * acc.y, 1.f * acc.z, 1.f * acc.w);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int g_stream_tc = 0;            // opt-in (mvb_tune stream_tc=1): at 64 meshes the launch is at time parity with the step-by-step
                                       // kernels it replaces (fwd 103 vs 108 us, bwd 122 vs 122 us in the captured step) but holds every SM, so
                                       // the deferred weight-gradient chains no longer overlap it: 944 vs 911 us per step (profiles/README.md)
static int g_stream_sw = 16;           // meshes per slab (mvb_tune stream_tc=enable,sw; 0: the decomposition with the least work per CTA)
void set_stream_tc(int v, int sw) {
    g_stream_tc = v ? 1 : 0;
    if (sw == 0 || sw == 8 || sw == 16) g_stream_sw = sw;
}

struct StreamPlan {
    int grid, SW, RP, nslabs, tiles_per_cta;
    size_t smem;
};

static bool stream_plan_sw(int N, int B, int sw, int sms, StreamPlan *pl) {
    if (B % sw) return false;
    const int nslabs = B / sw, rpt = 128 / sw;
    const int nrb_max = sms / nslabs;
    if (nrb_max < 1) return false;
    int rp = (N + nrb_max - 1) / nrb_max;
    rp = (rp + rpt - 1) / rpt * rpt;
    if (rp > ST_RCAP || (rp / rpt) * 16 > 512) return false;       // staged rows; accumulators of a CTA's tiles must fit TMEM
    pl->SW = sw; pl->RP = rp; pl->nslabs = nslabs; pl->tiles_per_cta = rp / rpt;
    pl->grid = (N + rp - 1) / rp * nslabs;
    return true;
}

static bool stream_plan(int N, int B, int Fin, int Fout, int K, int n_in, int has_up, int n_out, bool bwd, StreamPlan *pl) {
    if (!g_stream_tc || !tc_enabled()) return false;
    if (Fin != 16 || Fout != 16 || K < 1 || K > 8 || N < 1 || B < 1) return false;
    if (n_out != N) return false;                                  // no row selection
    if (!has_up && n_in != N) return false;
    const int64_t pairs = (int64_t)N * B;
    if (pairs < 148 * 128 * 4) return false;                       // small levels: the mesh-resident kernels
    if (pairs * 4 * 2 >= ((int64_t)1 << 31)) return false;         // 32-bit quad offsets within a plane
    const int sms = num_sms();
    bool ok = false;
    if (g_stream_sw) {
        ok = stream_plan_sw(N, B, g_stream_sw, sms, pl);
    }
    if (!ok) {
        const int cand[2] = {16, 8};
        int64_t best = 0;
        for (int c = 0; c < 2; ++c) {
            StreamPlan t;
            if (!stream_plan_sw(N, B, cand[c], sms, &t)) continue;
            const int64_t cost = (int64_t)t.RP * t.SW;
            if (!ok || cost < best) { *pl = t; best = cost; ok = true; }
        }
    }
    if (!ok) return false;
    const size_t b_bytes = ((size_t)K * 16 * 64 + 1023) / 1024 * 1024;
    pl->smem = 1024 + (size_t)ST_NS * ST_STAGE + 2 * b_bytes + (size_t)ST_RCAP * 8 + (size_t)ST_ECAP * 8 + (bwd ? ST_NT_MAX * 16 : 0) +
               (2 * ST_NS + 1) * 8 + 48;
    return pl->smem <= 227 * 1024;
}

int stream_tc_supported(int N, int B, int Fin, int Fout, int K, int n_in, int has_up, int n_out) {
    StreamPlan pl;
    return stream_plan(N, B, Fin, Fout, K, n_in, has_up, n_out, true, &pl) ? 1 : 0;
}

// Workspaces: a 256-byte block of tile counters, then the [N][B][16] planes (multiples of 64 bytes, packed without
// padding).  Forward: three planes.  Backward: S_0..S_{K-1}, with up-sampling T_0 and dT_0, then the db partials and
// the weight-gradient partials.
struct StreamWs {
    unsigned int *ctr;
    float *planes, *T0, *dT0, *dbp, *part;
    size_t part_bytes;
};
static StreamWs stream_fwd_ws(WsCarve &c, int N, int B) {
    StreamWs w{};
    w.ctr = c.take<unsigned int>(256);
    w.planes = c.take<float>(3 * (size_t)N * B * 16 * sizeof(float), 64);
    return w;
}
static StreamWs stream_bwd_ws(WsCarve &c, int N, int B, int K, int has_up) {
    const size_t plane = (size_t)N * B * 16 * sizeof(float);
    StreamWs w{};
    w.ctr = c.take<unsigned int>(256);
    w.planes = c.take<float>((size_t)K * plane, 64);
    if (has_up) {
        w.T0 = c.take<float>(plane, 64);
        w.dT0 = c.take<float>(plane, 64);
    }
    w.dbp = c.take<float>((size_t)num_sms() * 16 * sizeof(float));
    w.part_bytes = align_up(wgrad_partial_bytes(K * 16, 16), 256);
    w.part = c.take<float>(w.part_bytes);
    return w;
}

template <bool BWD, int NT, int SW>
static int launch_stream_kernel(const StreamArgs &a, const StreamPlan &pl, cudaStream_t st) {
    static DevFlags optin;
    int rc = smem_optin(cheb_stream_tc_kernel<BWD, NT, SW>, 227 * 1024, optin, "cheb_stream_tc");
    if (rc) return rc;
    cheb_stream_tc_kernel<BWD, NT, SW><<<pl.grid, NT, pl.smem, st>>>(a);
    return check_launch("mvb cheb_stream_tc");
}

template <bool BWD>
static int launch_stream_t(const StreamArgs &a, const StreamPlan &pl, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(a.ctr, 0, 256, st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(MVB_ECUDA, "cheb_stream_tc: memset: %s", cudaGetErrorString(e));
    }
    if (pl.SW == 16) return launch_stream_kernel<BWD, ST_NT_MAX, 16>(a, pl, st);
    return launch_stream_kernel<BWD, ST_NT_MAX, 8>(a, pl, st);
}

// returns 1 = launched, 0 = shape not covered, < 0 = error
int launch_stream_tc_fwd(int N, int B, int Fin, int Fout, int K, const int32_t *Lrp, const int32_t *Lci, const float *Lv, int n_in,
                         const int32_t *Urp, const int32_t *Uci, const float *Uv, int n_out, const int32_t *sel, const float *x,
                         const float *w, const float *bias, int relu, float *y, void *workspace, size_t workspace_bytes, cudaStream_t st) {
    StreamPlan pl;
    if (sel || !stream_plan(N, B, Fin, Fout, K, n_in, Urp != nullptr, n_out, false, &pl)) return 0;
    WsCarve c{reinterpret_cast<char *>(workspace)};
    const StreamWs ws = stream_fwd_ws(c, N, B);
    if (workspace_bytes < c.off) return set_err(MVB_EWORKSPACE, "cheb_stream_fwd: workspace %zu < %zu", workspace_bytes, c.off);
    StreamArgs a{};
    a.N = N; a.B = B; a.K = K; a.Nacc = Fout;
    a.Lrp = Lrp; a.Lci = Lci; a.Lv = Lv;
    a.n_in = n_in; a.Urp = Urp; a.Uci = Uci; a.Uv = Uv;
    a.x = x; a.w = w; a.bias = bias; a.relu = relu; a.out = y;
    a.ctr = ws.ctr;
    a.planes = ws.planes;
    a.SW = pl.SW; a.RP = pl.RP; a.nslabs = pl.nslabs; a.tiles_per_cta = pl.tiles_per_cta;
    a.pairs = (int64_t)N * B;
    const int rc = launch_stream_t<false>(a, pl, st);
    return rc ? rc : 1;
}

int launch_stream_tc_bwd(int N, int B, int Fin, int Fout, int K, const int32_t *Ltrp, const int32_t *Ltci, const float *Ltv, int n_in,
                         const int32_t *Urp, const int32_t *Uci, const float *Uv, const int32_t *Utrp, const int32_t *Utci,
                         const float *Utv, int n_out, const int32_t *sel, const float *x, const float *w, const float *y_for_relu,
                         const float *dy, float *dx, float *dweight, float *dbias, void *workspace, size_t workspace_bytes,
                         cudaStream_t st) {
    StreamPlan pl;
    const int has_up = Urp != nullptr;
    if (sel || !stream_plan(N, B, Fin, Fout, K, n_in, has_up, n_out, true, &pl)) return 0;
    WsCarve c{reinterpret_cast<char *>(workspace)};
    const StreamWs ws = stream_bwd_ws(c, N, B, K, has_up);
    if (workspace_bytes < c.off) return set_err(MVB_EWORKSPACE, "cheb_stream_bwd: workspace %zu < %zu", workspace_bytes, c.off);
    StreamArgs a{};
    a.N = N; a.B = B; a.K = K; a.Nacc = Fin;
    a.Lrp = Ltrp; a.Lci = Ltci; a.Lv = Ltv;
    a.n_in = n_in; a.Urp = Urp; a.Uci = Uci; a.Uv = Uv;
    a.Utrp = (has_up && dx) ? Utrp : nullptr; a.Utci = Utci; a.Utv = Utv;
    a.x = x; a.w = w; a.out = dx;
    a.dy = dy; a.y = y_for_relu;
    a.ctr = ws.ctr;
    a.planes = ws.planes;
    a.T0 = ws.T0;
    a.dT0 = ws.dT0;
    a.dbp = dbias ? ws.dbp : nullptr;
    a.SW = pl.SW; a.RP = pl.RP; a.nslabs = pl.nslabs; a.tiles_per_cta = pl.tiles_per_cta;
    a.pairs = (int64_t)N * B;
    int rc = launch_stream_t<true>(a, pl, st);
    if (rc) return rc;
    // db and dW off the critical path (deferred side chain when the step engine has switched it on)
    SideChain side(st, 0, false);
    const cudaStream_t ws_st = side.stream();
    if (dbias) {
        rc = launch_layer_finalize(pl.grid, 0, 16, nullptr, a.dbp, nullptr, dbias, ws_st);
        if (rc) return rc;
    }
    WgradArgs wa{};
    wa.rows = (int64_t)N * B;
    wa.in_planes = K;
    wa.in_w = 16;
    wa.in0 = a.planes;
    wa.in_rest = a.planes + (int64_t)N * B * 16;
    wa.dy = has_up ? a.T0 : x;
    wa.n_out = Fin;
    wa.partials = ws.part;
    wa.partial_bytes = ws.part_bytes;
    int nA = 0, m4A = 0;
    rc = launch_wgrad_partials(wa, 0, &nA, &m4A, ws_st);
    if (rc) return rc;
    rc = launch_wgrad_finalize(wa.partials, nA, m4A, nullptr, 0, 0, Fin, K * Fin, Fout, dweight, nullptr, ws_st, 1);
    if (rc) return rc;
    return 1;
}

}  // namespace mvb

// ---------------------------------------------------------------------------------------------
// C ABI (include/mvb.h)
// ---------------------------------------------------------------------------------------------
extern "C" int mvb_cheb_stream_supported(int N, int B, int Fin, int Fout, int K, int n_in, int has_up, int n_out) {
    return mvb::stream_tc_supported(N, B, Fin, Fout, K, n_in, has_up, n_out);
}

extern "C" size_t mvb_cheb_stream_fwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up) {
    (void)Fin; (void)Fout; (void)K; (void)has_up;
    mvb::WsCarve c;
    mvb::stream_fwd_ws(c, N, B);
    return c.off;
}

extern "C" int mvb_cheb_stream_fwd(int N, int B, int Fin, int Fout, int K, const int32_t *L_rowptr, const int32_t *L_colidx,
                                   const float *L_vals, int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx,
                                   const float *U_vals, int U_nnz, const float *x, const float *weight, const float *bias, int relu,
                                   float *y, void *workspace, size_t workspace_bytes, void *stream) {
    (void)L_nnz; (void)U_nnz;
    MVB_REQUIRE(L_rowptr && L_colidx && L_vals && x && weight && y && workspace, "cheb_stream_fwd: null pointer");
    MVB_REQUIRE(U_rowptr || n_in == N, "cheb_stream_fwd: n_in=%d != N=%d without an up-sampling operator", n_in, N);
    if (!mvb::aligned16(x) || !mvb::aligned16(y) || !mvb::aligned16(workspace)) return mvb::set_err(MVB_EALIGN, "cheb_stream_fwd: x / y / workspace must be 16-byte aligned");
    const int rc = mvb::launch_stream_tc_fwd(N, B, Fin, Fout, K, L_rowptr, L_colidx, L_vals, n_in, U_rowptr, U_colidx, U_vals, N, nullptr, x,
                                             weight, bias, relu, y, workspace, workspace_bytes, (cudaStream_t)stream);
    if (rc < 0) return rc;
    if (rc == 0) return mvb::set_err(MVB_EINVAL, "cheb_stream_fwd: shape N=%d B=%d Fin=%d Fout=%d K=%d not supported (see mvb_cheb_stream_supported)", N, B, Fin, Fout, K);
    return MVB_OK;
}

extern "C" size_t mvb_cheb_stream_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up) {
    (void)Fin; (void)Fout;
    mvb::WsCarve c;
    mvb::stream_bwd_ws(c, N, B, K, has_up);
    return c.off;
}

extern "C" int mvb_cheb_stream_bwd(int N, int B, int Fin, int Fout, int K, const int32_t *Lt_rowptr, const int32_t *Lt_colidx,
                                   const float *Lt_vals, int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx,
                                   const float *U_vals, const int32_t *Ut_rowptr, const int32_t *Ut_colidx, const float *Ut_vals,
                                   int U_nnz, const float *x, const float *weight, const float *y_for_relu, const float *dy, float *dx,
                                   float *dweight, float *dbias, void *workspace, size_t workspace_bytes, void *stream) {
    (void)L_nnz; (void)U_nnz;
    MVB_REQUIRE(Lt_rowptr && Lt_colidx && Lt_vals && x && weight && dy && dweight && workspace, "cheb_stream_bwd: null pointer");
    MVB_REQUIRE(U_rowptr || n_in == N, "cheb_stream_bwd: n_in != N without an up-sampling operator");
    MVB_REQUIRE(!U_rowptr || !dx || Ut_rowptr, "cheb_stream_bwd: dx requested without U^T");
    if (!mvb::aligned16(x) || !mvb::aligned16(dy) || (y_for_relu && !mvb::aligned16(y_for_relu)) || (dx && !mvb::aligned16(dx)) || !mvb::aligned16(workspace))
        return mvb::set_err(MVB_EALIGN, "cheb_stream_bwd: tensors must be 16-byte aligned");
    const int rc = mvb::launch_stream_tc_bwd(N, B, Fin, Fout, K, Lt_rowptr, Lt_colidx, Lt_vals, n_in, U_rowptr, U_colidx, U_vals, Ut_rowptr,
                                             Ut_colidx, Ut_vals, N, nullptr, x, weight, y_for_relu, dy, dx, dweight, dbias, workspace,
                                             workspace_bytes, (cudaStream_t)stream);
    if (rc < 0) return rc;
    if (rc == 0) return mvb::set_err(MVB_EINVAL, "cheb_stream_bwd: shape N=%d B=%d Fin=%d Fout=%d K=%d not supported", N, B, Fin, Fout, K);
    return MVB_OK;
}
