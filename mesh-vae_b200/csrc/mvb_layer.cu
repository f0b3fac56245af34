// Mesh-resident Chebyshev layers for the coarse levels of the mesh pyramid.
//
// At the coarse levels (313 / 79 / 20 vertices of the template, SURVEY.md 8 shapes table) one mesh's
// planes are a few tens of KB: the whole layer of the reference's encoder / decoder loop
//     x = relu(cheb[i](x, L)); x = pool(x, D)          models/cheb_VAE.py:264-265
//     x = pool(x, U);          x = relu(cheb_dec[i](x, L))   models/cheb_VAE.py:284-285
// fits in the shared memory of ONE block per mesh.  The step-by-step path spends 30-90 us per such
// layer and direction in 4-6 launches whose cost is latency and per-block set-up, not bytes (in-graph
// timeline, profiles/README.md); here a layer is one launch:
//   forward : [U prologue] -> T_0..T_{K-1} in shared memory (ping-pong) -> out += T_k W_k (4x4 register
//             tiles, FFMA fp32) -> bias, ReLU -> [row-selection epilogue: only the rows D keeps are
//             contracted and written]
//   backward: G = dY * [y > 0]; pass 1 recomputes T_k (nothing is saved by the forward pass except
//             its input and output) and reduces dW_k = T_k^T G, db = 1^T G per mesh; pass 2 runs the
//             reverse recurrence G_k = G W_k^T + 2 L^T G_{k+1} - G_{k+2} in the same buffers and
//             applies U^T; a second tiny kernel sums the per-mesh partials in mesh order.
// No atomics, fixed summation orders: deterministic.  Arithmetic per row is the same sequence as the
// step kernels (alpha * sum_j v_j x_j, then fma(-1, T_{k-2}, .)).
#include "mvb_internal.cuh"

namespace mvb {

struct LayerArgs {
    int N, B, Fin, Fout, K;
    const int32_t *Lrp, *Lci; const float *Lv; int Lnnz;          // CSR(L)  [N x N]
    const int32_t *Ltrp, *Ltci; const float *Ltv;                 // CSR(L^T) (backward)
    int n_in;                                                     // rows of x (== N without U)
    const int32_t *Urp, *Uci; const float *Uv; int Unnz;          // CSR(U)  [N x n_in] or NULL
    const int32_t *Utrp, *Utci; const float *Utv;                 // CSR(U^T) [n_in x N] (backward)
    int n_out; const int32_t *sel;                                // output row r = conv row sel[r]; NULL: identity
    const float *x, *w, *bias, *y, *dy;
    int relu;
    float *out;                                                   // forward: y; backward: dx (may be NULL)
    float *dwp, *dbp;                                             // backward: per-mesh partials [B][K*Fin*Fout], [B][Fout]
    int splits;                                                   // forward: blocks per mesh (output columns split)
};

constexpr int LY_MAXT = 3;
constexpr int LY_NT = 512;          // threads per block: 16 warps hide the shared-memory latencies of the tile loops

__host__ __device__ inline int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

__host__ __device__ inline int r4(int n) { return (n + 3) & ~3; }

struct LayerSmem {        // offsets in 4-byte words
    int tA, tB, G, W, red, csr, ucsr, inv, total;
};
__host__ __device__ inline LayerSmem layer_smem(int N, int Fin, int Fout, int K, int Lnnz, int n_in, int Unnz, int n_out,
                                                bool backward, int fin_local) {
    LayerSmem s;
    const int LDT = fin_local + 4;
    const int rows = N > n_in ? N : n_in;
    int o = 0;
    s.tA = o; o += rows * LDT;
    s.tB = o; o += rows * LDT;
    s.G = o; if (backward) o += n_out * (Fout + 4);
    s.W = o; o += K * Fin * Fout;
    if (backward) {           // dW partials: one per row split, or one per warp when a warp's lanes share blocks (shuffle-reduced)
        const int nblk = (fin_local / 4) * (Fout / 4);
        s.red = o; o += (nblk >= 32 ? LY_NT : (LY_NT / 32) * nblk) * 16;
    } else {
        s.red = o;
    }
    s.csr = o; o += r4(N + 1) + 2 * r4(Lnnz);
    s.ucsr = o; if (Unnz > 0) o += r4((N > n_in ? N : n_in) + 1) + 2 * r4(Unnz);
    s.inv = o; if (backward) o += r4(N);
    s.total = o;
    return s;
}

// CSR into shared memory: row pointers by cp.async, entries as packed (column, value) pairs - one 8-byte load per
// neighbour in the gather loops instead of two 4-byte ones.  Visible after the caller's next wait + __syncthreads.
__device__ __forceinline__ void stage_csr_async(float *smem, int nrows, int nnz, const int32_t *rp, const int32_t *ci,
                                                const float *v, const int32_t *&srp, const int2 *&sce, int tid) {
    int32_t *a = reinterpret_cast<int32_t *>(smem);
    int2 *b = reinterpret_cast<int2 *>(a + r4(nrows + 1));
    cp_async_words(a, rp, nrows + 1, tid, LY_NT);
    for (int base = 0; base < nnz; base += 4 * LY_NT) {          // 8 independent loads in flight per thread
        int c[4];
        float w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * LY_NT + tid;
            if (i < nnz) { c[u] = __ldg(ci + i); w[u] = __ldg(v + i); }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * LY_NT + tid;
            if (i < nnz) b[i] = make_int2(c[u], __float_as_int(w[u]));
        }
    }
    srp = a; sce = b;
}

__device__ __forceinline__ float4 ld4s(const float *p) { return *reinterpret_cast<const float4 *>(p); }
__device__ __forceinline__ void st4s(float *p, const float4 &v) { *reinterpret_cast<float4 *>(p) = v; }
__device__ __forceinline__ void fma4s(float4 &a, float s, const float4 &x) {
    a.x = fmaf(s, x.x, a.x); a.y = fmaf(s, x.y, a.y); a.z = fmaf(s, x.z, a.z); a.w = fmaf(s, x.w, a.w);
}

// dst[v][q] = sum_j vals[j] * src[colidx[j]][q]  for the rows of a CSR held in shared memory
__device__ __forceinline__ float4 gather_row(const float *src, int LDT, const int2 *ce, int s, int e, int q) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = s;
    for (; j + 2 <= e; j += 2) {
        const int2 ea = ce[j], eb = ce[j + 1];
        const float4 xa = ld4s(src + ea.x * LDT + 4 * q), xb = ld4s(src + eb.x * LDT + 4 * q);
        fma4s(acc, __int_as_float(ea.y), xa);
        fma4s(acc, __int_as_float(eb.y), xb);
    }
    if (j < e) {
        const int2 ea = ce[j];
        fma4s(acc, __int_as_float(ea.y), ld4s(src + ea.x * LDT + 4 * q));
    }
    return acc;
}

// one recurrence step in shared memory: old <- alpha * L cur - [k >= 2] old   (row arithmetic of the step kernels)
__device__ __forceinline__ void recur_step(float *cur, float *old, int N, int lqf, int LDT, const int32_t *rp, const int2 *ce,
                                           int k, int tid) {
    for (int i = tid; i < (N << lqf); i += LY_NT) {
        const int v = i >> lqf, q = i & ((1 << lqf) - 1);
        const float4 acc = gather_row(cur, LDT, ce, rp[v], rp[v + 1], q);
        float4 o;
        if (k == 1) {
            o = make_float4(1.f * acc.x, 1.f * acc.y, 1.f * acc.z, 1.f * acc.w);
        } else {
            const float4 z = ld4s(old + v * LDT + 4 * q);
            o.x = fmaf(-1.f, z.x, 2.f * acc.x); o.y = fmaf(-1.f, z.y, 2.f * acc.y);
            o.z = fmaf(-1.f, z.z, 2.f * acc.z); o.w = fmaf(-1.f, z.w, 2.f * acc.w);
        }
        st4s(old + v * LDT + 4 * q, o);
    }
}

// load this mesh's rows of a vertex-major tensor [rows, B, F] into dst[rows][LD] (16-byte copies)
// (columns [c0, c0 + 4 << lq) of rows that are Ftot floats wide)
__device__ __forceinline__ void stage_mesh_rows(float *dst, int LD, const float *src, int rows, int B, int b, int Ftot, int c0, int lq,
                                                int tid) {
    for (int i = tid; i < (rows << lq); i += LY_NT) {
        const int r = i >> lq, q = i & ((1 << lq) - 1);
        cp_async<4>(dst + r * LD + 4 * q, src + ((int64_t)r * B + b) * Ftot + c0 + 4 * q);
    }
}

// T_0 of this mesh in tA (through the U prologue when there is one); returns with the block synchronised
__device__ __forceinline__ void stage_t0(const LayerArgs &a, float *sm, const LayerSmem &S, int b, int tid, int c0, int lqf) {
    const int LDT = (4 << lqf) + 4;
    float *tA = sm + S.tA, *tB = sm + S.tB;
    if (a.Urp) {
        const int32_t *urp;
        const int2 *uce;
        stage_csr_async(sm + S.ucsr, a.N, a.Unnz, a.Urp, a.Uci, a.Uv, urp, uce, tid);
        stage_mesh_rows(tB, LDT, a.x, a.n_in, a.B, b, a.Fin, c0, lqf, tid);
        cp_async_wait_all();
        __syncthreads();
        for (int i = tid; i < (a.N << lqf); i += LY_NT) {
            const int v = i >> lqf, q = i & ((1 << lqf) - 1);
            st4s(tA + v * LDT + 4 * q, gather_row(tB, LDT, uce, urp[v], urp[v + 1], q));
        }
    } else {
        stage_mesh_rows(tA, LDT, a.x, a.N, a.B, b, a.Fin, c0, lqf, tid);
        cp_async_wait_all();
    }
    __syncthreads();
}

// One register tile of the contraction: acc[j] += T[row_j][:] . W_k[:, 4 cq .. 4 cq + 3] for the NJ valid rows of the
// tile (rows are valid as a prefix; tiles of the last row groups are partial - the kernels are issue-bound, so rows
// that do not exist must not be computed: at 79 vertices three of four tile rows would be padding)
template <int NJ>
__device__ __forceinline__ void contract_tile(const float *T, int LDT, const int *rows, const float *Wk, int Fout, int QF,
                                              float4 *acc) {
    const float *r[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) r[j] = T + rows[j] * LDT;
    for (int i4 = 0; i4 < QF; ++i4) {
        const float4 w0 = ld4s(Wk + (4 * i4 + 0) * Fout), w1 = ld4s(Wk + (4 * i4 + 1) * Fout);
        const float4 w2 = ld4s(Wk + (4 * i4 + 2) * Fout), w3 = ld4s(Wk + (4 * i4 + 3) * Fout);
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const float4 av = ld4s(r[j] + 4 * i4);
            fma4s(acc[j], av.x, w0); fma4s(acc[j], av.y, w1); fma4s(acc[j], av.z, w2); fma4s(acc[j], av.w, w3);
        }
    }
}

// One register tile of P_k = G W_k^T (backward): p[j] = G[row_j][:] . Wt_k[:, 4 pq .. 4 pq + 3], Wt[k][o][i] in shared memory
template <int NJ>
__device__ __forceinline__ void pk_tile(const float *G, int LDG, const int *rows, const float *Wk, int Fin, int CQ, float4 *p) {
#pragma unroll
    for (int j = 0; j < NJ; ++j) p[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int o4 = 0; o4 < CQ; ++o4) {
        const float *wo = Wk + 4 * o4 * Fin;
        const float4 t0 = ld4s(wo), t1 = ld4s(wo + Fin), t2 = ld4s(wo + 2 * Fin), t3 = ld4s(wo + 3 * Fin);
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const float4 g = ld4s(G + rows[j] * LDG + 4 * o4);
            p[j].x = fmaf(g.x, t0.x, fmaf(g.y, t1.x, fmaf(g.z, t2.x, fmaf(g.w, t3.x, p[j].x))));
            p[j].y = fmaf(g.x, t0.y, fmaf(g.y, t1.y, fmaf(g.z, t2.y, fmaf(g.w, t3.y, p[j].y))));
            p[j].z = fmaf(g.x, t0.z, fmaf(g.y, t1.z, fmaf(g.z, t2.z, fmaf(g.w, t3.z, p[j].z))));
            p[j].w = fmaf(g.x, t0.w, fmaf(g.y, t1.w, fmaf(g.z, t2.w, fmaf(g.w, t3.w, p[j].w))));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LY_NT)
cheb_layer_fwd_kernel(LayerArgs a, LayerSmem S) {
    extern __shared__ float4 lsm4[];
    float *sm = reinterpret_cast<float *>(lsm4);
    const int tid = threadIdx.x, b = blockIdx.x;
    const int Fin = a.Fin, Fout = a.Fout, K = a.K, N = a.N;
    const int LDT = Fin + 4, QF = Fin >> 2, lqf = ilog2(QF);
    float *Ws = sm + S.W;
    const int32_t *lrp;
    const int2 *lce;
    for (int i = tid; i < (K * Fin * Fout) >> 2; i += LY_NT) cp_async<4>(Ws + 4 * i, a.w + 4 * i);
    stage_csr_async(sm + S.csr, N, a.Lnnz, a.Lrp, a.Lci, a.Lv, lrp, lce, tid);
    stage_t0(a, sm, S, b, tid, 0, lqf);          // waits for every copy issued so far

    // contraction tiles: thread = (column quad cq, row group rg); tile t holds rows rg + j*NRG + t*4*NRG
    const int CQl = (Fout >> 2) / a.splits;           // column quads of this block
    const int lcql = ilog2(CQl);
    const int cq = blockIdx.y * CQl + (tid & (CQl - 1)), rg = tid >> lcql, NRG = LY_NT >> lcql;
    int rr[LY_MAXT][4];
#pragma unroll
    for (int t = 0; t < LY_MAXT; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = rg + j * NRG + t * 4 * NRG;
            rr[t][j] = r < a.n_out ? (a.sel ? __ldg(a.sel + r) : r) : -1;
        }
    float4 acc[LY_MAXT][4];
#pragma unroll
    for (int t = 0; t < LY_MAXT; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[t][j] = make_float4(0.f, 0.f, 0.f, 0.f);

    int nj[LY_MAXT];                                  // valid rows of each tile (a prefix of its 4 rows)
#pragma unroll
    for (int t = 0; t < LY_MAXT; ++t) nj[t] = (rr[t][0] >= 0) + (rr[t][1] >= 0) + (rr[t][2] >= 0) + (rr[t][3] >= 0);
    auto contract = [&](const float *T, int k) {
        const float *Wk = Ws + k * Fin * Fout + 4 * cq;
#pragma unroll
        for (int t = 0; t < LY_MAXT; ++t) {
            if (nj[t] == 4) contract_tile<4>(T, LDT, rr[t], Wk, Fout, QF, acc[t]);
            else if (nj[t] == 3) contract_tile<3>(T, LDT, rr[t], Wk, Fout, QF, acc[t]);
            else if (nj[t] == 2) contract_tile<2>(T, LDT, rr[t], Wk, Fout, QF, acc[t]);
            else if (nj[t] == 1) contract_tile<1>(T, LDT, rr[t], Wk, Fout, QF, acc[t]);
        }
    };

    float *cur = sm + S.tA, *old = sm + S.tB;
    contract(cur, 0);
    for (int k = 1; k < K; ++k) {
        recur_step(cur, old, N, lqf, LDT, lrp, lce, k, tid);
        __syncthreads();
        contract(old, k);
        float *t = cur; cur = old; old = t;
    }
    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.bias) bv = make_float4(__ldg(a.bias + 4 * cq), __ldg(a.bias + 4 * cq + 1), __ldg(a.bias + 4 * cq + 2), __ldg(a.bias + 4 * cq + 3));
#pragma unroll
    for (int t = 0; t < LY_MAXT; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = rg + j * NRG + t * 4 * NRG;
            if (r < a.n_out) {
                float4 v = acc[t][j];
                v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
                if (a.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                *reinterpret_cast<float4 *>(a.out + ((int64_t)r * a.B + b) * Fout + 4 * cq) = v;
            }
        }
}

// ---------------------------------------------------------------------------------------------
// backward.  grid = (B, splits): block (b, s) owns the input-feature quads [s*QFl, (s+1)*QFl) of mesh
// b - the recurrences are independent per feature column, dW_k rows and dx columns of different
// splits are disjoint, so the splits share nothing but the (re-staged) G and W.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LY_NT)
cheb_layer_bwd_kernel(LayerArgs a, LayerSmem S) {
    extern __shared__ float4 lsm4[];
    float *sm = reinterpret_cast<float *>(lsm4);
    const int tid = threadIdx.x, b = blockIdx.x;
    const int Fin = a.Fin, Fout = a.Fout, K = a.K, N = a.N;
    const int QFl = (Fin >> 2) / a.splits, lqf = ilog2(QFl);      // local input-feature quads
    const int q0 = blockIdx.y * QFl, c0 = 4 * q0;                 // first local quad / feature
    const int LDT = 4 * QFl + 4, LDG = Fout + 4, CQ = Fout >> 2, lcq = ilog2(CQ);
    float *Ws = sm + S.W, *G = sm + S.G, *red = sm + S.red;
    int32_t *inv = reinterpret_cast<int32_t *>(sm + S.inv);
    const int32_t *lrp;
    const int2 *lce;
    // W is only read by the P_k tiles of pass 2, four input features at a time: staged TRANSPOSED, Wt[k][o][i], so that
    // the lanes of a warp (consecutive input-feature quads) read consecutive 16-byte pieces - the [k][i][o] layout put
    // them 4 * Fout words apart, on the same banks (ncu: 16 wavefronts per load instead of 1-4)
    if (a.out)
        for (int i = tid; i < K * Fin * Fout; i += LY_NT) {
            const int o = i % Fout, ki = i / Fout;                  // i = (k * Fin + in) * Fout + o
            const int in = ki % Fin, k = ki / Fin;
            Ws[(k * Fout + o) * Fin + in] = __ldg(a.w + i);
        }
    // a.out == NULL: weight gradient only (pass 1)
    stage_csr_async(sm + S.csr, N, a.Lnnz, a.Lrp, a.Lci, a.Lv, lrp, lce, tid);
    stage_mesh_rows(G, LDG, a.dy, a.n_out, a.B, b, Fout, 0, lcq, tid);
    for (int v = tid; v < N; v += LY_NT) inv[v] = a.sel ? -1 : v;
    stage_t0(a, sm, S, b, tid, c0, lqf);
    if (a.sel)
        for (int r = tid; r < a.n_out; r += LY_NT) inv[__ldg(a.sel + r)] = r;
    if (a.relu)                                              // G = dY * [y > 0]
        for (int i = tid; i < (a.n_out << lcq); i += LY_NT) {
            const int r = i >> lcq, q = i & (CQ - 1);
            const float4 yv = __ldg(reinterpret_cast<const float4 *>(a.y + ((int64_t)r * a.B + b) * Fout + 4 * q));
            float4 g = ld4s(G + r * LDG + 4 * q);
            g.x = yv.x > 0.f ? g.x : 0.f; g.y = yv.y > 0.f ? g.y : 0.f; g.z = yv.z > 0.f ? g.z : 0.f; g.w = yv.w > 0.f ? g.w : 0.f;
            st4s(G + r * LDG + 4 * q, g);
        }
    __syncthreads();

    // ---- pass 1: dW_k = T_k^T G (this block's rows of dW_k), db = 1^T G ----
    const int NBLK = QFl * CQ, lnb = lqf + lcq;        // 4x4 blocks of this split's part of one dW_k
    const int RS = LY_NT >> lnb;                       // row splits
    const int blk = tid & (NBLK - 1), rs = tid >> lnb;
    const int iq = blk & (QFl - 1), oq = blk >> lqf;
    float *dwp = a.dwp + (int64_t)b * K * Fin * Fout;
    auto wgrad = [&](const float *T, int k) {
        float4 c0_ = make_float4(0.f, 0.f, 0.f, 0.f), c1 = c0_, c2 = c0_, c3 = c0_;
        for (int r = rs; r < a.n_out; r += RS) {
            const int v = a.sel ? __ldg(a.sel + r) : r;
            const float4 t = ld4s(T + v * LDT + 4 * iq), g = ld4s(G + r * LDG + 4 * oq);
            fma4s(c0_, t.x, g); fma4s(c1, t.y, g); fma4s(c2, t.z, g); fma4s(c3, t.w, g);
        }
        // lanes of a warp that hold the same 4x4 block (NBLK < 32): fixed xor tree first, one partial per warp
        for (int off = NBLK; off < 32; off <<= 1) {
            c0_.x += __shfl_xor_sync(0xffffffffu, c0_.x, off); c0_.y += __shfl_xor_sync(0xffffffffu, c0_.y, off);
            c0_.z += __shfl_xor_sync(0xffffffffu, c0_.z, off); c0_.w += __shfl_xor_sync(0xffffffffu, c0_.w, off);
            c1.x += __shfl_xor_sync(0xffffffffu, c1.x, off); c1.y += __shfl_xor_sync(0xffffffffu, c1.y, off);
            c1.z += __shfl_xor_sync(0xffffffffu, c1.z, off); c1.w += __shfl_xor_sync(0xffffffffu, c1.w, off);
            c2.x += __shfl_xor_sync(0xffffffffu, c2.x, off); c2.y += __shfl_xor_sync(0xffffffffu, c2.y, off);
            c2.z += __shfl_xor_sync(0xffffffffu, c2.z, off); c2.w += __shfl_xor_sync(0xffffffffu, c2.w, off);
            c3.x += __shfl_xor_sync(0xffffffffu, c3.x, off); c3.y += __shfl_xor_sync(0xffffffffu, c3.y, off);
            c3.z += __shfl_xor_sync(0xffffffffu, c3.z, off); c3.w += __shfl_xor_sync(0xffffffffu, c3.w, off);
        }
        const bool per_warp = NBLK < 32;
        const int nparts = per_warp ? LY_NT / 32 : RS;
        __syncthreads();                      // red is free (the previous k's reduction has been read)
        if (!per_warp || (tid & 31) < NBLK) {
            float *dst = red + ((per_warp ? (tid >> 5) : rs) * NBLK + blk) * 16;
            st4s(dst, c0_); st4s(dst + 4, c1); st4s(dst + 8, c2); st4s(dst + 12, c3);
        }
        __syncthreads();
        for (int e = tid; e < NBLK * 16; e += LY_NT) {          // ordered sum over the partials
            float s = 0.f;
            for (int p = 0; p < nparts; ++p) s += red[p * NBLK * 16 + e];
            const int bk = e >> 4, m = (e >> 2) & 3, c = e & 3;
            const int i = c0 + 4 * (bk & (QFl - 1)) + m, o = 4 * (bk >> lqf) + c;
            dwp[((int64_t)k * Fin + i) * Fout + o] = s;
        }
    };
    float *cur = sm + S.tA, *old = sm + S.tB;
    wgrad(cur, 0);
    for (int k = 1; k < K; ++k) {
        recur_step(cur, old, N, lqf, LDT, lrp, lce, k, tid);
        __syncthreads();
        wgrad(old, k);
        float *t = cur; cur = old; old = t;
    }
    if (a.dbp && blockIdx.y == 0 && tid < Fout) {
        float s = 0.f;
        for (int r = 0; r < a.n_out; ++r) s += G[r * LDG + tid];
        a.dbp[(int64_t)b * Fout + tid] = s;
    }
    if (!a.out) return;
    __syncthreads();

    // ---- pass 2: reverse recurrence in the same buffers ----
    stage_csr_async(sm + S.csr, N, a.Lnnz, a.Ltrp, a.Ltci, a.Ltv, lrp, lce, tid);      // L^T replaces L
    const int32_t *utrp = nullptr;
    const int2 *utce = nullptr;
    if (a.Utrp) stage_csr_async(sm + S.ucsr, a.n_in, a.Unnz, a.Utrp, a.Utci, a.Utv, utrp, utce, tid);
    // P_k tiles: thread = (local input-feature quad pq, row group rg) over the n_out rows that carry gradient
    const int pq = tid & (QFl - 1), rg = tid >> lqf, NRG = LY_NT >> lqf;
    int rr[LY_MAXT][4];
#pragma unroll
    for (int t = 0; t < LY_MAXT; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = rg + j * NRG + t * 4 * NRG;
            rr[t][j] = r < a.n_out ? r : -1;
        }
    // dst[v] = P_k[v] - [sub] dst[v] on the rows with gradient (v = sel[r]); other rows are handled by the gather pass
    auto add_pk = [&](float *dst, int k, bool sub) {
        const float *Wk = Ws + k * Fin * Fout + 4 * (q0 + pq);          // Wt[k][o][4 (q0 + pq) .. + 3]
#pragma unroll
        for (int t = 0; t < LY_MAXT; ++t) {
            if (rr[t][0] < 0) break;
            float4 p[4];
            const int njt = 1 + (rr[t][1] >= 0) + (rr[t][2] >= 0) + (rr[t][3] >= 0);
            if (njt == 4) pk_tile<4>(G, LDG, rr[t], Wk, Fin, CQ, p);
            else if (njt == 3) pk_tile<3>(G, LDG, rr[t], Wk, Fin, CQ, p);
            else if (njt == 2) pk_tile<2>(G, LDG, rr[t], Wk, Fin, CQ, p);
            else pk_tile<1>(G, LDG, rr[t], Wk, Fin, CQ, p);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (rr[t][j] < 0) continue;
                const int v = a.sel ? __ldg(a.sel + rr[t][j]) : rr[t][j];
                float *d = dst + v * LDT + 4 * pq;
                if (sub) {
                    const float4 z = ld4s(d);
                    p[j].x -= z.x; p[j].y -= z.y; p[j].z -= z.z; p[j].w -= z.w;
                }
                st4s(d, p[j]);
            }
        }
    };
    float *g1 = sm + S.tA, *g2 = sm + S.tB;
    // G_{K-1} = P_{K-1}: zero the rows without gradient, then the tiles
    if (a.sel)
        for (int i = tid; i < (N << lqf); i += LY_NT) {
            const int v = i >> lqf, q = i & (QFl - 1);
            if (inv[v] < 0) st4s(g1 + v * LDT + 4 * q, make_float4(0.f, 0.f, 0.f, 0.f));
        }
    add_pk(g1, K - 1, false);
    cp_async_wait_all();
    __syncthreads();
    for (int k = K - 2; k >= 0; --k) {
        const bool has_g2 = (k + 2 <= K - 1);
        const float alpha = (k == 0) ? 1.f : 2.f;
        add_pk(g2, k, has_g2);                // rows with gradient: g2 <- P_k - G_{k+2}
        __syncthreads();
        for (int i = tid; i < (N << lqf); i += LY_NT) {
            const int v = i >> lqf, q = i & (QFl - 1);
            const float4 acc = gather_row(g1, LDT, lce, lrp[v], lrp[v + 1], q);
            float4 base = ld4s(g2 + v * LDT + 4 * q);
            if (inv[v] < 0) {                 // row without gradient: P_k = 0
                if (has_g2) { base.x = -base.x; base.y = -base.y; base.z = -base.z; base.w = -base.w; }
                else base = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            float4 o;
            o.x = fmaf(alpha, acc.x, base.x); o.y = fmaf(alpha, acc.y, base.y);
            o.z = fmaf(alpha, acc.z, base.z); o.w = fmaf(alpha, acc.w, base.w);
            st4s(g2 + v * LDT + 4 * q, o);
        }
        __syncthreads();
        float *t = g1; g1 = g2; g2 = t;
    }
    // g1 = dT_0 (this split's feature columns)
    if (a.Utrp) {
        for (int i = tid; i < (a.n_in << lqf); i += LY_NT) {
            const int c = i >> lqf, q = i & (QFl - 1);
            const float4 v = gather_row(g1, LDT, utce, utrp[c], utrp[c + 1], q);
            *reinterpret_cast<float4 *>(a.out + ((int64_t)c * a.B + b) * Fin + c0 + 4 * q) = v;
        }
    } else {
        for (int i = tid; i < (N << lqf); i += LY_NT) {
            const int v = i >> lqf, q = i & (QFl - 1);
            *reinterpret_cast<float4 *>(a.out + ((int64_t)v * a.B + b) * Fin + c0 + 4 * q) = ld4s(g1 + v * LDT + 4 * q);
        }
    }
}

// ordered sum of the per-mesh partials: dst[j] = sum_b part[b][j].  Block = 32 outputs x 8 mesh lanes (each lane sums
// every 8th mesh, then a fixed-order sum over the lanes): B/8 dependent L2 round trips per thread instead of B.
__global__ void __launch_bounds__(256)
layer_finalize_kernel(int B, int nw, int nb, const float *__restrict__ dwp, const float *__restrict__ dbp,
                      float *__restrict__ dw, float *__restrict__ db) {
    pdl_trigger();
    pdl_wait();
    __shared__ float red[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int j = blockIdx.x * 32 + tx;
    float s = 0.f;
    if (j < nw) {
        for (int b = ty; b < B; b += 8) s += __ldg(dwp + (int64_t)b * nw + j);
    } else if (db && j - nw < nb) {
        for (int b = ty; b < B; b += 8) s += __ldg(dbp + (int64_t)b * nb + (j - nw));
    }
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0) {
        float t = red[0][tx];
#pragma unroll
        for (int q = 1; q < 8; ++q) t += red[q][tx];
        if (j < nw) dw[j] = t;
        else if (db && j - nw < nb) db[j - nw] = t;
    }
}

static bool pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

// blocks per mesh: as many as keep every SM busy when the batch is small, while a block keeps >= `min_q` quads
// (one block per SM: two feature splits per mesh of the backward pass at 64 meshes.  Sizing it for two blocks per SM - 4
// splits, kernel capped at 64 registers - measured 157 us against 149 us for the four backward layers of a step: the
// per-block instruction count does not shrink with the split.  Running the dW and dX halves of the backward layer as two
// concurrent kernels measured 63 us for the pair against 59 us for the single kernel at level 2: both halves saturate
// the same shared-memory pipe; profiles/README.md)
static int pick_splits(int B, int quads, int min_q) {
    int s = 1;
    while (B * s * 2 <= num_sms() + num_sms() / 2 && quads / (s * 2) >= min_q) s *= 2;
    return s;
}

static int layer_check(int N, int B, int Fin, int Fout, int K, int Lnnz, int n_in, int Unnz, int n_out, bool backward,
                       LayerSmem *S_out, int *splits_out) {
    if (N <= 0 || B <= 0 || K <= 0 || n_in <= 0 || n_out <= 0 || Lnnz < 0) return 0;
    if (Fin % 4 || Fout % 4 || Fin > 64 || Fout > 64) return 0;
    const int QF = Fin / 4, CQ = Fout / 4;
    if (!pow2(QF) || !pow2(CQ)) return 0;
    // forward splits the output columns (each split redoes the cheap recurrence), backward the input features
    // (the backward splits redo nothing - the recurrences are per feature column)
    const int splits = backward ? pick_splits(B, QF, 1) : pick_splits(B, CQ, 2);
    const int ql = (backward ? QF : CQ) / splits;                 // local tile-column quads
    if (n_out > LY_MAXT * 4 * (LY_NT / ql)) return 0;
    if (backward && (QF / splits) * CQ > LY_NT) return 0;
    const LayerSmem S = layer_smem(N, Fin, Fout, K, Lnnz, n_in, Unnz, n_out, backward, backward ? Fin / splits : Fin);
    if ((size_t)S.total * 4 > 200 * 1024) return 0;
    if (S_out) *S_out = S;
    if (splits_out) *splits_out = splits;
    return 1;
}

int launch_layer_finalize(int B, int nw, int nb, const float *dwp, const float *dbp, float *dw, float *db, cudaStream_t st) {
    if (nw + nb <= 0) return MVB_OK;
    launch_pdl(layer_finalize_kernel, dim3((nw + nb + 31) / 32), dim3(256), 0, st, B, nw, nb, dwp, dbp, dw, db);
    return check_launch("mvb layer finalize");
}

}  // namespace mvb

using namespace mvb;


extern "C" int mvb_cheb_layer_supported(int N, int B, int Fin, int Fout, int K, int L_nnz, int n_in, int U_nnz, int n_out) {
    // every layer has two implementations: the tensor-core mesh kernels (mvb_mesh_tc.cu; 16 / 32-wide features,
    // up to 1280 vertices) and the FFMA mesh kernels of this file (4, 8, 16, 32 or 64 features in and out - a power-of-two
    // number of quads, layer_check - and levels of a few hundred vertices)
    const bool fwd = mesh_tc_fwd_supported(N, B, Fin, Fout, K, L_nnz, n_in, n_out) ||
                     layer_check(N, B, Fin, Fout, K, L_nnz, n_in, U_nnz, n_out, false, nullptr, nullptr);
    const bool bwd = mesh_tc_bwd_supported(N, B, Fin, Fout, K, L_nnz, n_in, n_out, U_nnz > 0) ||
                     layer_check(N, B, Fin, Fout, K, L_nnz, n_in, U_nnz, n_out, true, nullptr, nullptr);
    return fwd && bwd;
}

// workspace of the FFMA backward kernel: per-mesh dW partials [B][K*Fin*Fout], then per-mesh db partials [B][Fout]
static float *layer_bwd_ws(WsCarve &c, int B, int Fin, int Fout, int K, float **dbp) {
    float *dwp = c.take<float>((size_t)B * K * Fin * Fout * sizeof(float), sizeof(float));
    *dbp = c.take<float>((size_t)B * Fout * sizeof(float), sizeof(float));
    return dwp;
}

// one buffer serves whichever kernel runs: the tensor-core layer (mesh_tc_bwd_workspace_bytes) or the FFMA one
extern "C" size_t mvb_cheb_layer_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up) {
    WsCarve c;
    float *dbp;
    layer_bwd_ws(c, B, Fin, Fout, K, &dbp);
    const size_t tc = mesh_tc_bwd_workspace_bytes(N, B, Fin, Fout, K, has_up);
    return c.off > tc ? c.off : tc;
}

extern "C" int mvb_cheb_layer_fwd(int N, int B, int Fin, int Fout, int K, const int32_t *L_rowptr, const int32_t *L_colidx,
                                  const float *L_vals, int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx,
                                  const float *U_vals, int U_nnz, int n_out, const int32_t *sel, const float *x,
                                  const float *weight, const float *bias, int relu, float *y, void *stream) {
    MVB_REQUIRE(L_rowptr && x && weight && y, "cheb_layer_fwd: null pointer");
    MVB_REQUIRE(U_rowptr || n_in == N, "cheb_layer_fwd: n_in=%d != N=%d without an up-sampling operator", n_in, N);
    MVB_REQUIRE(sel || n_out == N, "cheb_layer_fwd: n_out=%d != N=%d without a row selection", n_out, N);
    if (aligned16(x) && aligned16(weight) && aligned16(y)) {
        const int tc = launch_mesh_tc_fwd(N, B, Fin, Fout, K, L_rowptr, L_colidx, L_vals, L_nnz, n_in, U_rowptr, U_colidx, U_vals,
                                          n_out, sel, x, weight, bias, relu, y, (cudaStream_t)stream);
        if (tc != 0) return tc < 0 ? tc : MVB_OK;
    }
    LayerSmem S;
    int splits = 1;
    if (!layer_check(N, B, Fin, Fout, K, L_nnz, n_in, U_rowptr ? U_nnz : 0, n_out, false, &S, &splits))
        return set_err(MVB_EINVAL, "cheb_layer_fwd: shape N=%d Fin=%d Fout=%d K=%d not supported (see mvb_cheb_layer_supported)", N, Fin, Fout, K);
    if (!aligned16(x) || !aligned16(weight) || !aligned16(y)) return set_err(MVB_EALIGN, "cheb_layer_fwd: x / weight / y must be 16-byte aligned");
    LayerArgs a{};
    a.N = N; a.B = B; a.Fin = Fin; a.Fout = Fout; a.K = K;
    a.Lrp = L_rowptr; a.Lci = L_colidx; a.Lv = L_vals; a.Lnnz = L_nnz;
    a.n_in = n_in; a.Urp = U_rowptr; a.Uci = U_colidx; a.Uv = U_vals; a.Unnz = U_rowptr ? U_nnz : 0;
    a.n_out = n_out; a.sel = sel;
    a.x = x; a.w = weight; a.bias = bias; a.relu = relu; a.out = y;
    a.splits = splits;
    static DevFlags optin;
    const size_t smem = (size_t)S.total * 4;
    if (smem > 48 * 1024) {
        const int rc_attr = smem_optin(cheb_layer_fwd_kernel, 200 * 1024, optin, "cheb_layer_fwd");
        if (rc_attr) return rc_attr;
    }
    cheb_layer_fwd_kernel<<<dim3(B, splits), LY_NT, smem, (cudaStream_t)stream>>>(a, S);
    return check_launch("mvb_cheb_layer_fwd");
}

extern "C" int mvb_cheb_layer_bwd(int N, int B, int Fin, int Fout, int K, const int32_t *L_rowptr, const int32_t *L_colidx,
                                  const float *L_vals, const int32_t *Lt_rowptr, const int32_t *Lt_colidx, const float *Lt_vals,
                                  int L_nnz, int n_in, const int32_t *U_rowptr, const int32_t *U_colidx, const float *U_vals,
                                  const int32_t *Ut_rowptr, const int32_t *Ut_colidx, const float *Ut_vals, int U_nnz, int n_out,
                                  const int32_t *sel, const float *x, const float *weight, const float *y_for_relu,
                                  const float *dy, float *dx, float *dweight, float *dbias, void *workspace,
                                  size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(L_rowptr && Lt_rowptr && x && weight && dy && dweight && workspace, "cheb_layer_bwd: null pointer");
    MVB_REQUIRE(U_rowptr || n_in == N, "cheb_layer_bwd: n_in != N without an up-sampling operator");
    MVB_REQUIRE(!U_rowptr || !dx || Ut_rowptr, "cheb_layer_bwd: dx requested without U^T");
    MVB_REQUIRE(sel || n_out == N, "cheb_layer_bwd: n_out != N without a row selection");
    if (aligned16(x) && aligned16(weight) && aligned16(dy) && (!y_for_relu || aligned16(y_for_relu)) && (!dx || aligned16(dx)) && aligned16(workspace)) {
        const int tc = launch_mesh_tc_bwd(N, B, Fin, Fout, K, Lt_rowptr, Lt_colidx, Lt_vals, L_nnz, n_in, U_rowptr, U_colidx, U_vals,
                                          Ut_rowptr, Ut_colidx, Ut_vals, n_out, sel, x, weight, y_for_relu, dy, dx, dweight, dbias,
                                          workspace, workspace_bytes, (cudaStream_t)stream);
        if (tc != 0) return tc < 0 ? tc : MVB_OK;
    }
    LayerSmem S;
    int splits = 1;
    if (!layer_check(N, B, Fin, Fout, K, L_nnz, n_in, U_rowptr ? U_nnz : 0, n_out, true, &S, &splits))
        return set_err(MVB_EINVAL, "cheb_layer_bwd: shape N=%d Fin=%d Fout=%d K=%d not supported", N, Fin, Fout, K);
    if (!aligned16(x) || !aligned16(weight) || !aligned16(dy) || (y_for_relu && !aligned16(y_for_relu)) || (dx && !aligned16(dx)))
        return set_err(MVB_EALIGN, "cheb_layer_bwd: tensors must be 16-byte aligned");
    WsCarve c{reinterpret_cast<char *>(workspace)};
    float *dbp;
    float *dwp = layer_bwd_ws(c, B, Fin, Fout, K, &dbp);
    if (workspace_bytes < c.off) return set_err(MVB_EWORKSPACE, "cheb_layer_bwd: workspace %zu < %zu", workspace_bytes, c.off);
    LayerArgs a{};
    a.N = N; a.B = B; a.Fin = Fin; a.Fout = Fout; a.K = K;
    a.Lrp = L_rowptr; a.Lci = L_colidx; a.Lv = L_vals; a.Lnnz = L_nnz;
    a.Ltrp = Lt_rowptr; a.Ltci = Lt_colidx; a.Ltv = Lt_vals;
    a.n_in = n_in; a.Urp = U_rowptr; a.Uci = U_colidx; a.Uv = U_vals; a.Unnz = U_rowptr ? U_nnz : 0;
    a.Utrp = U_rowptr ? Ut_rowptr : nullptr; a.Utci = Ut_colidx; a.Utv = Ut_vals;
    a.n_out = n_out; a.sel = sel;
    a.x = x; a.w = weight; a.y = y_for_relu; a.dy = dy; a.relu = y_for_relu != nullptr; a.out = dx;
    a.dwp = dwp;
    a.dbp = dbp;
    a.splits = splits;
    static DevFlags optin;
    const size_t smem = (size_t)S.total * 4;
    if (smem > 48 * 1024) {
        const int rc_attr = smem_optin(cheb_layer_bwd_kernel, 200 * 1024, optin, "cheb_layer_bwd");
        if (rc_attr) return rc_attr;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int nw = K * Fin * Fout, nb = dbias ? Fout : 0;
    cheb_layer_bwd_kernel<<<dim3(B, splits), LY_NT, smem, st>>>(a, S);
    const int rc = check_launch("mvb_cheb_layer_bwd");
    if (rc) return rc;
    return launch_layer_finalize(B, nw, nb, a.dwp, a.dbp, dweight, dbias, st);
}
