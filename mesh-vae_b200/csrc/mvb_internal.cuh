// Internal helpers shared by the libmvb_sm100a translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "mvb.h"

namespace mvb {

// thread-local last-error text (mvb_last_error)
char *err_buf();
int set_err(int code, const char *fmt, ...);

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Bump carver over a caller's workspace: every piece starts at an `align`-aligned offset and spans a whole number of
// `align` units.  One function per entry point describes its workspace with it: the *_workspace_bytes query runs that
// function with base == nullptr (it only measures, every pointer is NULL) and the launch runs it on the caller's buffer,
// so the two cannot disagree.
struct WsCarve {
    char *base = nullptr;
    size_t off = 0;
    template <class T>
    T *take(size_t bytes, size_t align = 256) {
        off = align_up(off, align);
        T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += align_up(bytes, align);
        return p;
    }
};

#define MVB_REQUIRE(cond, ...)                          \
    do {                                                \
        if (!(cond)) return mvb::set_err(MVB_EINVAL, __VA_ARGS__); \
    } while (0)

// after a kernel launch: report launch-configuration errors without synchronising
void count_launch();
inline int check_launch(const char *what) {
    count_launch();
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(MVB_ECUDA, "%s: %s", what, cudaGetErrorString(e));
    }
    return MVB_OK;
}

int num_sms();  // multiprocessor count of the CURRENT device, cached per device (148 on B200)
int pdl_enabled();   // mvb_tune pdl=0/1: launch the kernels that have a pdl_wait() with the programmatic-serialization attribute

// Function attributes (the opt-in for > 48 KB of dynamic shared memory) are per DEVICE: a process that drives several
// GPUs must set them on each.  DevFlags keeps one bit / one size per device ordinal for a call site.
inline int device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        dev = 0;
    }
    return (dev >= 0 && dev < 64) ? dev : 0;
}
struct DevFlags {
    size_t granted[64] = {0};
};
template <typename KernelT>
inline int smem_optin(KernelT kernel, size_t bytes, DevFlags &f, const char *what) {
    if (bytes <= 48 * 1024) return MVB_OK;          // the default limit: no opt-in needed
    const int d = device_slot();
    if (bytes <= f.granted[d]) return MVB_OK;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(MVB_ECUDA, "%s: cudaFuncSetAttribute(%zu bytes): %s", what, bytes, cudaGetErrorString(e));
    }
    f.granted[d] = bytes;
    return MVB_OK;
}

#ifdef __CUDACC__
// Programmatic dependent launch (PDL): a kernel launched with the stream-serialization attribute may start while its
// predecessor in the stream is still running - as soon as every CTA of the predecessor has executed pdl_trigger() (or
// exited) - and runs its prologue (TMEM allocation, barrier init, operator / weight staging: data that no kernel of the
// step writes) until pdl_wait(), which returns once the predecessor grid has completed and its writes are visible.
// EVERYTHING that reads or writes a tensor of the step must come after pdl_wait().  Both are no-ops in an ordinary launch.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// launch with the programmatic-serialization attribute (kernels that begin with pdl_trigger() / pdl_wait())
template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);          // errors surface through check_launch()
}

// global -> shared copy with U independent loads in flight per thread.  A plain
// `for (i = tid; i < n; i += nthreads) dst[i] = src[i];` serialises on the load->store dependency
// (one global-memory latency per iteration); small launch-latency-bound kernels spent most of their
// time in such loops (profiles/README.md, B = 4 launch list).
template <int U, typename T>
__device__ __forceinline__ void g2s_copy(T *dst, const T *__restrict__ src, int n, int tid, int nthreads) {
    for (int base = 0; base < n; base += U * nthreads) {
        T v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * nthreads + tid;
            if (i < n) v[u] = __ldg(src + i);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * nthreads + tid;
            if (i < n) dst[i] = v[u];
        }
    }
}

// cp.async (global -> shared without a register round trip): every copy of a tile is in flight at
// once, so staging costs ONE exposed memory latency instead of one per batch of register loads.
// VEC = 4: 16-byte copies (both addresses 16-byte aligned); VEC = 1: 4-byte copies.  !valid: the
// destination is zero-filled (src-size 0) and the source is not dereferenced.
template <int VEC>
__device__ __forceinline__ void cp_async(void *smem_dst, const void *gsrc, bool valid = true) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    const int sz = valid ? 4 * VEC : 0;
    if (VEC == 4)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory"); }
// n 4-byte words global -> shared (any alignment)
__device__ __forceinline__ void cp_async_words(void *dst, const void *src, int n, int tid, int nthreads) {
    for (int i = tid; i < n; i += nthreads) cp_async<1>(reinterpret_cast<char *>(dst) + 4 * i, reinterpret_cast<const char *>(src) + 4 * i);
}
#endif

// ---- launchers implemented in the .cu files ------------------------------------------------
int launch_spmm(int n_rows, int n_src_rows, const int32_t *rowptr, const int32_t *colidx, const float *vals,
                const float *x, float *y, const float *z, const float *w, float alpha, float beta,
                int64_t ncols, cudaStream_t st);

// Chebyshev recurrence T_1 = L t0, T_k = 2 L T_{k-1} - T_{k-2} (k < K) into planes[k-1] (n * ncols floats each): one
// fused launch when the level fits shared memory, else one SpMM launch per step.
int launch_cheb_recurrence(int n, int nnz, int K, const int32_t *rowptr, const int32_t *colidx, const float *vals,
                           const float *t0, float *planes, int64_t ncols, cudaStream_t st);
// its reverse: in place on the K planes P (G_k overwrites P_k), G_{K-1} = P_{K-1}, G_k = P_k + 2 L^T G_{k+1} - G_{k+2}
// (k >= 1), dx = P_0 + L^T G_1 - G_2 (dx = P_0 when K == 1); CSR(L^T) in rowptr_t / colidx_t / vals_t.
// keep_planes: G_1..G_{K-1} must be left in P for the caller (the step kernels: the fused kernel keeps them in shared
// memory); dx may then be NULL, and the last step is skipped.
int launch_cheb_recurrence_bwd(int n, int nnz, int K, const int32_t *rowptr_t, const int32_t *colidx_t, const float *vals_t,
                               float *P, float *dx, int64_t ncols, cudaStream_t st, bool keep_planes = false);

// mvb_opgrad.cu: vals[j] = coo_vals[perm[j]], vals_t[j] = coo_vals[perm_t[j]]
int launch_csr_values(int nnz, const int32_t *perm, const int32_t *perm_t, const float *coo_vals, float *vals,
                      float *vals_t, cudaStream_t st);
// d_coo[perm[j]] = <G_1[r], T_0[c]> + 2 sum_{k=2}^{K-1} <G_k[r], T_{k-1}[c]> for CSR(L) entry j = (r, c), r < n_rows;
// G: K planes [n_rows, ncols] (plane k = G_k, k >= 1), T_0 = x, T_k = basis plane k-1.  K >= 2.
int launch_cheb_edge_grad(int n_rows, int64_t ncols, int K, const int32_t *rowptr, const int32_t *colidx,
                          const int32_t *perm, const float *x, const float *basis, const float *G, float *d_coo,
                          cudaStream_t st);

// Generic small-matrix contraction over the rows of vertex-major activations:
//   out[p_out][row][j] = act( sum_{p_in,i} in[p_in][row][i] * Wm[p_in*in_w + i][p_out*out_w + j] + bias )
// in plane 0 = in0, planes 1.. = in_rest + (p-1)*rows*in_w.  Wm is [M, Nn] row-major in global
// memory, or [Nn, M] row-major when w_transposed == 1, or - w_transposed == 2 - the weight tensor
// [in_planes][Nn][in_w] itself read as sum_k S_k W_k^T (the adjoint-basis backward).  mask (optional, same layout as plane 0 of the
// input): input values of plane 0 are zeroed where mask <= 0 (fused ReLU backward).
struct ContractArgs {
    int64_t rows;
    int in_planes, in_w;
    const float *in0, *in_rest;
    const float *mask;
    const float *wmat;
    int w_transposed;
    int w_fold;           // > 1: fold that many weight blocks with c_k = cos(k pi/2) (empty-row closed form)
    const float *bias;
    int relu;
    int out_planes, out_w;
    float *out;
    // optional row selection (the down-sampling D folded into the contraction, models/cheb_VAE.py:264-265): output row
    // r = m * sel_group + b reads input row row_sel[m] * sel_group + b of every plane; planes are plane_rows rows long.
    // Tensor-core path only (launch_contract_tc); NULL = all rows in order.
    const int32_t *row_sel;
    int sel_group;
    int64_t plane_rows;
};
int launch_contract(const ContractArgs &a, cudaStream_t st);

// dW/db reduction:  dwm[m][n] = sum_rows tcat[row][m] * dy[row][n],  db[n] = sum_rows dy[row][n]
// tcat planes as above (K planes of width Fin), dy [rows, Fout] (optionally masked by mask > 0).
// Deterministic: fixed tile->CTA assignment, per-CTA partials in workspace, ordered final sum.
struct WgradArgs {
    int64_t rows;
    int in_planes, in_w;
    const float *in0, *in_rest;
    const float *dy;
    const float *mask;
    int n_out;            // Fout
    float *partials;      // workspace
    size_t partial_bytes;
    // optional row selection for the tcat planes (dy / mask are dense over the selected rows): see ContractArgs
    const int32_t *row_sel;
    int sel_group;
    int64_t plane_rows;
};
size_t wgrad_partial_bytes(int M, int n_out);
int launch_wgrad_partials(const WgradArgs &a, int has_bias, int *nparts, int *m4_out, cudaStream_t st);
int launch_wgrad_finalize(const float *partA, int nA, int M4A, const float *partB, int nB, int M4B,
                          int fin, int M, int n_out, float *dweight, float *dbias, cudaStream_t st, int a_transposed = 0);
// G = dY * [y > 0] (g written only when y != NULL) and db = column sums of G (when db != NULL)
int mask_colsum_blocks(int64_t rows);
int launch_mask_colsum(int64_t rows, int ncol, const float *dy, const float *y, float *g, float *db, float *part,
                       cudaStream_t st);

// closed-form rows (operator rows without entries): narrow FFMA kernels where they cover the shape, else the generic
// contraction / weight-gradient kernels with w_fold = K
int launch_fold_fwd(int64_t rows, int K, int Fin, int Fout, const float *x, const float *w, const float *bias, int relu,
                    float *out, cudaStream_t st);
int launch_fold_dx(int64_t rows, int K, int Fin, int Fout, const float *g, const float *w, float *dx, cudaStream_t st);
int launch_fold_wgrad(int64_t rows, int Fin, int Fout, const float *x, const float *g, float *partials, size_t partial_bytes,
                      int *nparts, int *m4, cudaStream_t st);

// tcgen05 paths (mvb_tc.cu): return 1 = handled, 0 = shape unsupported (use FFMA), < 0 = error
int launch_contract_tc(const ContractArgs &a, cudaStream_t st);
int tc_enabled();
int launch_wgrad_tc(const WgradArgs &a, int has_bias, int M4, int N4, int *nparts, cudaStream_t st);

// setters behind mvb_tune (mvb_api.cu)
void set_recur_fused(int v);
void set_mesh_tc(int enable, int c);
void set_stream_tc(int v, int sw);
void set_pdl(int v);

// mesh-resident tensor-core layers (mvb_mesh_tc.cu): 1 = handled / supported, 0 = shape not covered, < 0 = error
int mesh_tc_fwd_supported(int N, int B, int Fin, int Fout, int K, int Lnnz, int n_in, int n_out);
int mesh_tc_bwd_supported(int N, int B, int Fin, int Fout, int K, int Lnnz, int n_in, int n_out, int has_up);
size_t mesh_tc_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int has_up);
int launch_mesh_tc_fwd(int N, int B, int Fin, int Fout, int K, const int32_t *Lrp, const int32_t *Lci, const float *Lv, int Lnnz,
                       int n_in, const int32_t *Urp, const int32_t *Uci, const float *Uv, int n_out, const int32_t *sel,
                       const float *x, const float *w, const float *bias, int relu, float *y, cudaStream_t st);
int launch_mesh_tc_bwd(int N, int B, int Fin, int Fout, int K, const int32_t *Ltrp, const int32_t *Ltci, const float *Ltv, int Lnnz,
                       int n_in, const int32_t *Urp, const int32_t *Uci, const float *Uv, const int32_t *Utrp, const int32_t *Utci,
                       const float *Utv, int n_out, const int32_t *sel, const float *x, const float *w, const float *y_for_relu,
                       const float *dy, float *dx, float *dweight, float *dbias, void *workspace, size_t workspace_bytes,
                       cudaStream_t st);
// ordered sum over the meshes of per-mesh partials (mvb_layer.cu): dw[j] = sum_b dwp[b][j], db likewise
int launch_layer_finalize(int B, int nw, int nb, const float *dwp, const float *dbp, float *dw, float *db, cudaStream_t st);

// A side chain: kernels that need what the caller's stream `st` has enqueued so far - construct the guard after the
// chain's producer kernel - but that nothing later on `st` reads before the call returns (weight gradients).  stream()
// is where to enqueue the chain:
//   - while mvb_tune "defer_wgrad=1" is on and lane >= 0: a deferred lane (mvb_api.cu; lane 0 = convolution weight
//     gradients, lane 1 = dense-layer weight gradients).  The destructor records the chain's end; mvb_side_join joins it.
//   - otherwise, with `local`: the calling thread's side stream.  The destructor joins it into `st`.
//   - otherwise (or when no side stream can be had): `st` itself.
// The destructor runs on every exit path: a captured graph must not end forked.
struct SideLane;
class SideChain {
  public:
    SideChain(cudaStream_t st, int lane, bool local);
    ~SideChain();
    SideChain(const SideChain &) = delete;
    SideChain &operator=(const SideChain &) = delete;
    cudaStream_t stream() const { return stream_; }
    bool deferred() const { return deferred_; }

  private:
    cudaStream_t st_, stream_;
    SideLane *lane_ = nullptr;
    bool deferred_ = false;
};

}  // namespace mvb
