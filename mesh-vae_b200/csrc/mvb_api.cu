// C-ABI entry points: library info, the host COO->CSR hand-off, SpMM / pooling wrappers and the
// Chebyshev convolution forward / backward compositions.  See include/mvb.h for the contract and
// the reference symbols (file:line) each entry point replaces.
#include <stdarg.h>
#include <stdlib.h>
#include <atomic>
#include <mutex>
#include <vector>
#include "mvb_internal.cuh"

namespace mvb {

static thread_local char g_err[512] = {0};
char *err_buf() { return g_err; }
int set_err(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

int num_sms() {
    static int cached[64] = {0};
    const int d = device_slot();
    if (cached[d] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d) == cudaSuccess && n > 0)
            cached[d] = n;
        else {
            cudaGetLastError();
            cached[d] = 148;
        }
    }
    return cached[d];
}

}  // namespace mvb

using namespace mvb;

namespace mvb {
static int g_pdl = 1;
int pdl_enabled() { return g_pdl; }
void set_pdl(int v) { g_pdl = v ? 1 : 0; }
}  // namespace mvb

extern "C" int mvb_version(void) { return MVB_VERSION; }
extern "C" int mvb_sm_arch(void) { return 100; }
extern "C" const char *mvb_last_error(void) { return err_buf(); }
extern "C" int64_t mvb_launch_count(void) { return (int64_t)mvb::launch_count(); }


extern "C" int mvb_device_cc(void) {
    int dev = 0, major = 0, minor = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(MVB_ECUDA, "mvb_device_cc: %s", cudaGetErrorString(e));
    }
    return major * 10 + minor;
}

// ---------------------------------------------------------------------------------------------
// host: stable counting sort COO -> CSR (of P or of P^T)
// ---------------------------------------------------------------------------------------------
extern "C" int mvb_csr_from_coo_host(int64_t n_out_rows, int64_t n_out_cols, int64_t nnz,
                                     const int64_t *coo_row, const int64_t *coo_col,
                                     const float *coo_val, int transpose, int32_t *rowptr,
                                     int32_t *colidx, float *vals) {
    MVB_REQUIRE(n_out_rows >= 0 && n_out_cols >= 0 && nnz >= 0, "csr_from_coo: negative size");
    MVB_REQUIRE(n_out_rows < INT32_MAX && n_out_cols < INT32_MAX && nnz < INT32_MAX, "csr_from_coo: sizes exceed int32");
    MVB_REQUIRE(rowptr && (nnz == 0 || (coo_row && coo_col && coo_val && colidx && vals)), "csr_from_coo: null pointer");
    const int64_t *r = transpose ? coo_col : coo_row;
    const int64_t *c = transpose ? coo_row : coo_col;
    for (int64_t i = 0; i <= n_out_rows; ++i) rowptr[i] = 0;
    for (int64_t e = 0; e < nnz; ++e) {
        if (r[e] < 0 || r[e] >= n_out_rows || c[e] < 0 || c[e] >= n_out_cols)
            return set_err(MVB_EINVAL, "csr_from_coo: entry %lld = (%lld,%lld) outside [%lld,%lld]", (long long)e,
                           (long long)r[e], (long long)c[e], (long long)n_out_rows, (long long)n_out_cols);
        rowptr[r[e] + 1]++;
    }
    for (int64_t i = 0; i < n_out_rows; ++i) rowptr[i + 1] += rowptr[i];
    std::vector<int32_t> cursor(rowptr, rowptr + n_out_rows);
    for (int64_t e = 0; e < nnz; ++e) {
        const int32_t pos = cursor[r[e]]++;
        colidx[pos] = (int32_t)c[e];
        vals[pos] = coo_val[e];
    }
    return MVB_OK;
}

// ---------------------------------------------------------------------------------------------
// SpMM / pooling
// ---------------------------------------------------------------------------------------------
extern "C" int mvb_spmm(int n_rows, int n_src_rows, const int32_t *rowptr, const int32_t *colidx, const float *vals,
                        const float *x, float *y, const float *z, const float *w, float alpha,
                        float beta, int64_t ncols, void *stream) {
    MVB_REQUIRE(n_rows >= 0 && ncols >= 0, "spmm: negative size");
    MVB_REQUIRE(rowptr && x && y, "spmm: null pointer");
    MVB_REQUIRE(x != y, "spmm: y must not alias x");
    return launch_spmm(n_rows, n_src_rows, rowptr, colidx, vals, x, y, z, w, alpha, beta, ncols, (cudaStream_t)stream);
}

extern "C" int mvb_pool_fwd(int n_out_rows, int n_in_rows, const int32_t *rowptr, const int32_t *colidx,
                            const float *vals, const float *x, float *y, int64_t ncols, void *stream) {
    MVB_REQUIRE(n_out_rows >= 0 && ncols >= 0 && rowptr && x && y, "pool_fwd: bad arguments");
    return launch_spmm(n_out_rows, n_in_rows, rowptr, colidx, vals, x, y, nullptr, nullptr, 1.f, 0.f, ncols, (cudaStream_t)stream);
}

extern "C" int mvb_pool_bwd(int n_in_rows, int n_out_rows, const int32_t *rowptr_t, const int32_t *colidx_t,
                            const float *vals_t, const float *dy, float *dx, int64_t ncols, void *stream) {
    MVB_REQUIRE(n_in_rows >= 0 && ncols >= 0 && rowptr_t && dy && dx, "pool_bwd: bad arguments");
    return launch_spmm(n_in_rows, n_out_rows, rowptr_t, colidx_t, vals_t, dy, dx, nullptr, nullptr, 1.f, 0.f, ncols, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Chebyshev convolution
// ---------------------------------------------------------------------------------------------
// n_active: rows >= n_active of L have no entries and no entry references a column >= n_active
// (n_active == N for an ordinary operator).  For the empty rows the recurrence has the closed form
// T_k = c_k x, c_k = cos(k pi/2), so they collapse to ONE plane with the folded weight
// sum_k c_k W_k; only the first n_active vertices (a contiguous prefix in the vertex-major layout)
// run the SpMM recurrence.  This is what makes the reference's output layer - the 20-vertex
// operator applied to the 4998-vertex mesh, models/cheb_VAE.py:288 - a streaming pass.
extern "C" int mvb_cheb_fwd(int N, int B, int Fin, int Fout, int K, int n_active, int nnz,
                            const int32_t *rowptr, const int32_t *colidx, const float *vals,
                            const float *x, const float *weight, const float *bias, int relu,
                            float *basis, float *y, void *stream) {
    MVB_REQUIRE(N > 0 && B > 0 && Fin > 0 && Fout > 0 && K > 0, "cheb_fwd: bad sizes N=%d B=%d Fin=%d Fout=%d K=%d", N, B, Fin, Fout, K);
    MVB_REQUIRE(n_active >= 0 && n_active <= N, "cheb_fwd: n_active=%d outside [0,%d]", n_active, N);
    MVB_REQUIRE(x && weight && y && (K == 1 || n_active == 0 || (basis && rowptr)), "cheb_fwd: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_active > 0) {
        // recurrence: T_1 = L x ; T_k = 2 L T_{k-1} - T_{k-2}     (nn/conv.py:564, 568-569)
        int rc = launch_cheb_recurrence(n_active, nnz, K, rowptr, colidx, vals, x, basis, (int64_t)B * Fin, st);
        if (rc) return rc;
        ContractArgs a{};
        a.rows = (int64_t)n_active * B;
        a.in_planes = K;
        a.in_w = Fin;
        a.in0 = x;
        a.in_rest = basis;
        a.wmat = weight;
        a.bias = bias;
        a.relu = relu;
        a.out_planes = 1;
        a.out_w = Fout;
        a.out = y;
        rc = launch_contract(a, st);
        if (rc) return rc;
    }
    if (n_active < N) {
        const int64_t off = (int64_t)n_active * B;
        return launch_fold_fwd((int64_t)(N - n_active) * B, K, Fin, Fout, x + off * Fin, weight, bias, relu, y + off * Fout, st);
    }
    return MVB_OK;
}

// ---------------------------------------------------------------------------------------------
// Chebyshev convolution followed by a row selection (the encoder loop body at the levels that do not fit a
// mesh-resident kernel: x = relu(cheb[i](x, L)); x = pool(x, D), models/cheb_VAE.py:264-265, D = one 1.0 per row,
// mesh_operations.py:72-85).  Only the rows D keeps are contracted and written (1/4 of them at every level), and the
// backward pass - the basis form for a layer whose input needs no gradient, i.e. the first encoder layer - reduces
// dW / db over those rows only: dY is zero everywhere else.  Tensor-core kernels only (4 / 16 / 32-wide planes).
// ---------------------------------------------------------------------------------------------
static bool sel_shape_ok(int N, int B, int Fin, int Fout, int K, int n_sel) {
    if (!tc_enabled() || N < 1 || B < 1 || K < 1 || n_sel < 1 || n_sel > N) return false;
    if (!((Fin == 4 && K <= 8) || (Fin == 16 && K <= 6) || (Fin == 32 && K <= 3))) return false;     // planar layouts of tc_rowgemm / tc_wgrad
    if (Fout % 4 || Fout > 32 || (int64_t)n_sel * B < 256) return false;
    if (K * Fin + 1 > 128) return false;
    return true;
}

extern "C" int mvb_cheb_sel_supported(int N, int B, int Fin, int Fout, int K, int n_sel) {
    return sel_shape_ok(N, B, Fin, Fout, K, n_sel) ? 1 : 0;
}

extern "C" int mvb_cheb_sel_fwd(int N, int B, int Fin, int Fout, int K, int nnz, const int32_t *rowptr, const int32_t *colidx,
                                const float *vals, const float *x, const float *weight, const float *bias, int relu, int n_sel,
                                const int32_t *sel, float *basis, float *y_sel, void *stream) {
    MVB_REQUIRE(sel_shape_ok(N, B, Fin, Fout, K, n_sel), "cheb_sel_fwd: shape N=%d B=%d Fin=%d Fout=%d K=%d n_sel=%d not supported", N, B, Fin,
                Fout, K, n_sel);
    MVB_REQUIRE(x && weight && y_sel && sel && (K == 1 || (basis && rowptr)), "cheb_sel_fwd: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = launch_cheb_recurrence(N, nnz, K, rowptr, colidx, vals, x, basis, (int64_t)B * Fin, st);
    if (rc) return rc;
    ContractArgs a{};
    a.rows = (int64_t)n_sel * B;
    a.in_planes = K;
    a.in_w = Fin;
    a.in0 = x;
    a.in_rest = basis;
    a.wmat = weight;
    a.bias = bias;
    a.relu = relu;
    a.out_planes = 1;
    a.out_w = Fout;
    a.out = y_sel;
    a.row_sel = sel;
    a.sel_group = B;
    a.plane_rows = (int64_t)N * B;
    rc = launch_contract_tc(a, st);
    if (rc < 0) return rc;
    if (rc == 0) return set_err(MVB_EINVAL, "cheb_sel_fwd: the tensor-core contraction does not cover this call (alignment?)");
    return MVB_OK;
}

// workspace of mvb_cheb_sel_bwd: the weight-gradient partials
static float *cheb_sel_bwd_ws(WsCarve &c, int Fin, int Fout, int K) { return c.take<float>(wgrad_partial_bytes(K * Fin, Fout)); }

extern "C" size_t mvb_cheb_sel_bwd_workspace_bytes(int Fin, int Fout, int K) {
    WsCarve c;
    cheb_sel_bwd_ws(c, Fin, Fout, K);
    return c.off;
}

extern "C" int mvb_cheb_sel_bwd(int N, int B, int Fin, int Fout, int K, const float *x, const float *basis,
                                const float *y_sel_for_relu, const float *dy_sel, int n_sel, const int32_t *sel, float *dweight,
                                float *dbias, void *workspace, size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(sel_shape_ok(N, B, Fin, Fout, K, n_sel), "cheb_sel_bwd: shape not supported");
    MVB_REQUIRE(x && dy_sel && sel && dweight && workspace && (K == 1 || basis), "cheb_sel_bwd: null pointer");
    WsCarve c{reinterpret_cast<char *>(workspace)};
    WgradArgs wa{};
    wa.partials = cheb_sel_bwd_ws(c, Fin, Fout, K);
    wa.partial_bytes = c.off;
    if (workspace_bytes < c.off) return set_err(MVB_EWORKSPACE, "cheb_sel_bwd: workspace %zu < %zu", workspace_bytes, c.off);
    cudaStream_t st = (cudaStream_t)stream;
    wa.rows = (int64_t)n_sel * B;
    wa.in_planes = K;
    wa.in_w = Fin;
    wa.in0 = x;
    wa.in_rest = basis;
    wa.dy = dy_sel;
    wa.mask = y_sel_for_relu;
    wa.n_out = Fout;
    wa.row_sel = sel;
    wa.sel_group = B;
    wa.plane_rows = (int64_t)N * B;
    int nA = 0, m4A = 0;
    int rc = launch_wgrad_partials(wa, dbias != nullptr, &nA, &m4A, st);
    if (rc) return rc;
    return launch_wgrad_finalize(wa.partials, nA, m4A, nullptr, 0, 0, Fin, K * Fin, Fout, dweight, dbias, st);
}

// ---------------------------------------------------------------------------------------------
// Side chains (SideChain, mvb_internal.cuh).  A non-deferred chain that runs beside the caller's stream (the
// weight-gradient branch of mvb_cheb_bwd) uses the calling thread's own side stream and is joined before the call
// returns: the two branches overlap, and in a captured CUDA graph they become parallel branches.
// Deferred chains: the weight-gradient reduction of a layer (10-20 us) is not on the critical path of the backward pass:
// nothing reads dW / db before the optimizer.  In deferred mode (mvb_tune "defer_wgrad=1", switched on by the step
// engine around its backward pass) such a chain is forked onto a per-device lane stream (the chains of successive layers
// queue up there, each started by an event on the caller's stream once its producer kernel has been enqueued) and
// joined back only by mvb_side_join - so they fill the idle SMs / memory bandwidth under the following layers'
// latency-bound kernels; in a captured CUDA graph they form a parallel branch.
// The deferred state is per device and process-wide (autograd runs backward functions on its own thread).
// ---------------------------------------------------------------------------------------------
namespace mvb {
struct SideLane {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    bool tried = false, ok = false, pending = false;
};

// Creation is not a stream operation: legal while another stream is capturing only in relaxed mode, so it happens
// during the (uncaptured) warm-up calls; when it fails the lane is never used and the chain runs on the caller's stream.
static SideLane *open_lane(SideLane &s, int priority) {
    if (!s.tried) {
        s.tried = true;
        if (cudaStreamCreateWithPriority(&s.stream, cudaStreamNonBlocking, priority) == cudaSuccess &&
            cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) == cudaSuccess)
            s.ok = true;
        else
            cudaGetLastError();
    }
    return s.ok ? &s : nullptr;
}

// make the lane wait for what `st` has enqueued so far
static bool fork_lane(SideLane *s, cudaStream_t st) {
    if (!s) return false;
    if (cudaEventRecord(s->fork, st) != cudaSuccess || cudaStreamWaitEvent(s->stream, s->fork, 0) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return true;
}

constexpr int LAZY_SLOTS = 4;       // slot 1 = lane 1 (dense-layer weight gradients); slots 0, 2, 3 = lane 0 (convolution weight gradients:
                                    // successive chains go round robin over CONV_LANES of them, so that chains can overlap each other)
static SideLane g_lazy[64][LAZY_SLOTS];
constexpr int CONV_LANES = 3;       // same-box A/B (bench.py, 300 steps, second pass): 1 lane 0.9197 ms per step, 2: 0.9152, 3: 0.9116,
                                    // 4: 0.9109, 5: 0.9111, 7: 0.9109 - the chains queued behind each other in the tail of the
                                    // backward pass (the last layers' reductions) now run side by side
static int g_conv_next[64] = {0};
static const int kConvSlot[CONV_LANES] = {0, 2, 3};
static std::mutex g_lazy_mu;
static int g_defer_wgrad = 0;
void set_defer_wgrad(int v) { g_defer_wgrad = v ? 1 : 0; }

static SideLane *lazy_side(int slot) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    // LOWEST priority: when a chain and a kernel of the caller's stream are ready together (the input-gradient
    // contraction next to the weight-gradient reduction of the same layer), the block scheduler serves the caller's
    // kernel first - the chain takes what is left (a captured graph keeps the priority as a kernel-node attribute)
    int least = 0, greatest = 0;
    SideLane &s = g_lazy[dev][slot & (LAZY_SLOTS - 1)];
    if (!s.tried && cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess) {
        least = 0;
        cudaGetLastError();
    }
    return open_lane(s, least);
}

// make `st` wait for a pending chain (if any)
static void lazy_join_locked(SideLane *s, cudaStream_t st) {
    if (s && s->pending) {
        cudaStreamWaitEvent(st, s->join, 0);
        s->pending = false;
    }
}

SideChain::SideChain(cudaStream_t st, int lane, bool local) : st_(st), stream_(st) {
    if (lane >= 0 && g_defer_wgrad) {
        std::lock_guard<std::mutex> lk(g_lazy_mu);
        int slot = 1;
        if (lane == 0) {
            int dev = 0;
            if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
            slot = kConvSlot[g_conv_next[dev]];
            g_conv_next[dev] = (g_conv_next[dev] + 1) % CONV_LANES;
        }
        SideLane *s = lazy_side(slot);
        if (fork_lane(s, st)) {
            lane_ = s;
            stream_ = s->stream;
            deferred_ = true;
            return;
        }
    }
    if (local) {
        static thread_local SideLane t_side;
        SideLane *s = open_lane(t_side, 0);
        if (fork_lane(s, st)) {
            lane_ = s;
            stream_ = s->stream;
        }
    }
}

// deferred: record the chain's end (a lane is in order: the latest record covers every earlier chain) for mvb_side_join;
// local: join into the caller's stream now
SideChain::~SideChain() {
    if (!lane_) return;
    if (deferred_) {
        std::lock_guard<std::mutex> lk(g_lazy_mu);
        cudaEventRecord(lane_->join, lane_->stream);
        lane_->pending = true;
        if (!g_defer_wgrad) lazy_join_locked(lane_, st_);
    } else {
        cudaEventRecord(lane_->join, lane_->stream);
        cudaStreamWaitEvent(st_, lane_->join, 0);
    }
}
}  // namespace mvb

extern "C" int mvb_side_join(void *stream) {
    std::lock_guard<std::mutex> lk(mvb::g_lazy_mu);
    for (int slot = 0; slot < mvb::LAZY_SLOTS; ++slot) mvb::lazy_join_locked(mvb::lazy_side(slot), (cudaStream_t)stream);
    return MVB_OK;
}

// join only the chains of one lane (1 = the dense layers' weight gradients: the data-parallel engine reduces their
// bucket while the convolution chains of lane 0 are still running)
extern "C" int mvb_side_join_lane(void *stream, int lane) {
    std::lock_guard<std::mutex> lk(mvb::g_lazy_mu);
    if (lane == 1) {
        mvb::lazy_join_locked(mvb::lazy_side(1), (cudaStream_t)stream);
    } else {
        for (int c = 0; c < mvb::CONV_LANES; ++c) mvb::lazy_join_locked(mvb::lazy_side(mvb::kConvSlot[c]), (cudaStream_t)stream);
    }
    return MVB_OK;
}

// Two algebraically equal forms of the backward pass (L acts on vertices, W on features: they commute):
//   basis form  : dW_k = T_k(L x)^T G,  dX = sum_k T_k(L^T) (G W_k^T)      - needs the forward basis T_k,
//                 K planes P_k = G W_k^T and a reverse recurrence on Fin-wide planes;
//   adjoint form: S_k = T_k(L^T) G,  dW_k = x^T S_k,  dX = sum_k S_k W_k^T - the FORWARD kernels run on G
//                 (recurrence on Fout-wide planes, one contraction), nothing saved by the forward pass.
// Plane traffic is ~(32 Fin + 2 Fout) vs ~(27 Fout + 2 Fin) plane-widths: the adjoint form is used when
// the input gradient is wanted and Fout <= 1.2 Fin (every 16->16 layer of the reference model; the
// first encoder layer, which needs no dX, keeps the basis form: its basis is only 3-4 columns wide).
static bool adjoint_form(int Fin, int Fout, int need_dx) { return need_dx && 25 * Fout <= 30 * Fin && Fout % 4 == 0; }

// workspace of the basis form: weight-gradient partials of the active prefix and of the empty rows, then (with dX or
// the operator gradient: need_planes) the K planes P_k = dY W_k^T
struct ChebBwdBasisWs {
    float *partA, *partB, *P;
    size_t partA_bytes, partB_bytes;
};
static ChebBwdBasisWs cheb_bwd_basis_ws(WsCarve &c, int N, int B, int Fin, int Fout, int K, int n_active, int need_planes) {
    ChebBwdBasisWs w{};
    w.partA_bytes = align_up(wgrad_partial_bytes(K * Fin, Fout), 256);
    w.partA = c.take<float>(w.partA_bytes);
    if (n_active < N) {
        w.partB_bytes = align_up(wgrad_partial_bytes(Fin, Fout), 256);
        w.partB = c.take<float>(w.partB_bytes);
    }
    if (need_planes) w.P = c.take<float>((size_t)K * n_active * B * Fin * sizeof(float));
    return w;
}

// workspace of the adjoint form: weight-gradient partials (active prefix, empty rows), the column-sum partials of db,
// G = dY * [y > 0] and S_1..S_{K-1}
struct ChebBwdAdjointWs {
    float *partA, *partB, *colpart, *G, *S;
    size_t partA_bytes, partB_bytes;
};
static ChebBwdAdjointWs cheb_bwd_adjoint_ws(WsCarve &c, int N, int B, int Fin, int Fout, int K, int n_active) {
    ChebBwdAdjointWs w{};
    w.partA_bytes = align_up(wgrad_partial_bytes(K * Fout, Fin), 256);
    w.partA = c.take<float>(w.partA_bytes);
    if (n_active < N) {
        w.partB_bytes = align_up(wgrad_partial_bytes(Fin, Fout), 256);
        w.partB = c.take<float>(w.partB_bytes);
    }
    w.colpart = c.take<float>((size_t)mask_colsum_blocks((int64_t)N * B) * Fout * sizeof(float));
    w.G = c.take<float>((size_t)N * B * Fout * sizeof(float));
    w.S = c.take<float>((size_t)(K > 1 ? K - 1 : 0) * n_active * B * Fout * sizeof(float));
    return w;
}

extern "C" int mvb_cheb_bwd_uses_basis(int Fin, int Fout, int need_dx) { return adjoint_form(Fin, Fout, need_dx) ? 0 : 1; }

extern "C" size_t mvb_cheb_bwd_workspace_bytes(int N, int B, int Fin, int Fout, int K, int n_active, int need_dx) {
    WsCarve c;
    if (adjoint_form(Fin, Fout, need_dx))
        cheb_bwd_adjoint_ws(c, N, B, Fin, Fout, K, n_active);
    else
        cheb_bwd_basis_ws(c, N, B, Fin, Fout, K, n_active, need_dx);
    return c.off;
}

static int cheb_bwd_adjoint(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr_t,
                            const int32_t *colidx_t, const float *vals_t, const float *x, const float *weight,
                            const float *y_for_relu, const float *dy, float *dx, float *dweight, float *dbias, char *ws,
                            cudaStream_t st);

// CSR(L) with its COO permutation and the COO gradient it is written to: the operator gradient of mvb_cheb_bwd_op
struct OpGradArgs {
    const int32_t *rowptr, *colidx, *perm;
    float *d_coo_vals;
};
static int cheb_bwd_basis(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr_t,
                          const int32_t *colidx_t, const float *vals_t, const float *x, const float *basis,
                          const float *weight, const float *y_for_relu, const float *dy, float *dx, float *dweight,
                          float *dbias, const OpGradArgs *og, char *ws, cudaStream_t st);

extern "C" int mvb_cheb_bwd(int N, int B, int Fin, int Fout, int K, int n_active, int nnz,
                            const int32_t *rowptr_t, const int32_t *colidx_t, const float *vals_t,
                            const float *x, const float *basis, const float *weight,
                            const float *y_for_relu, const float *dy, float *dx, float *dweight,
                            float *dbias, void *workspace, size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(N > 0 && B > 0 && Fin > 0 && Fout > 0 && K > 0, "cheb_bwd: bad sizes");
    MVB_REQUIRE(n_active >= 0 && n_active <= N, "cheb_bwd: n_active=%d outside [0,%d]", n_active, N);
    const bool adj = adjoint_form(Fin, Fout, dx != nullptr);
    MVB_REQUIRE(x && weight && dy && dweight && workspace && (adj || K == 1 || n_active == 0 || basis), "cheb_bwd: null pointer");
    MVB_REQUIRE(!dx || K == 1 || n_active == 0 || rowptr_t, "cheb_bwd: dx requested without L^T");
    if (!aligned16(workspace)) return set_err(MVB_EALIGN, "cheb_bwd: workspace not 16-byte aligned");
    const size_t need = mvb_cheb_bwd_workspace_bytes(N, B, Fin, Fout, K, n_active, dx != nullptr);
    if (workspace_bytes < need) return set_err(MVB_EWORKSPACE, "cheb_bwd: workspace %zu < %zu", workspace_bytes, need);
    cudaStream_t st = (cudaStream_t)stream;
    if (adj) {
        if (!aligned16(dy) || (y_for_relu && !aligned16(y_for_relu)))
            return set_err(MVB_EALIGN, "cheb_bwd: dy / y must be 16-byte aligned");
        return cheb_bwd_adjoint(N, B, Fin, Fout, K, n_active, nnz, rowptr_t, colidx_t, vals_t, x, weight, y_for_relu, dy, dx,
                                dweight, dbias, reinterpret_cast<char *>(workspace), st);
    }
    return cheb_bwd_basis(N, B, Fin, Fout, K, n_active, nnz, rowptr_t, colidx_t, vals_t, x, basis, weight, y_for_relu, dy, dx,
                          dweight, dbias, nullptr, reinterpret_cast<char *>(workspace), st);
}

// The operator gradient needs G_k = dloss/dT_k, which only the basis form's reverse recurrence produces: this entry point
// always takes the basis form, whatever mvb_cheb_bwd_uses_basis says, and runs its weight-gradient branch beside the
// caller's stream, joined before it returns (never deferred).
extern "C" size_t mvb_cheb_bwd_op_workspace_bytes(int N, int B, int Fin, int Fout, int K, int n_active) {
    WsCarve c;
    cheb_bwd_basis_ws(c, N, B, Fin, Fout, K, n_active, 1);
    return c.off;
}

extern "C" int mvb_cheb_bwd_op(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr,
                               const int32_t *colidx, const int32_t *perm, const int32_t *rowptr_t, const int32_t *colidx_t,
                               const float *vals_t, const float *x, const float *basis, const float *weight,
                               const float *y_for_relu, const float *dy, float *dx, float *dweight, float *dbias,
                               float *d_coo_vals, void *workspace, size_t workspace_bytes, void *stream) {
    MVB_REQUIRE(N > 0 && B > 0 && Fin > 0 && Fout > 0 && K > 0 && nnz >= 0, "cheb_bwd_op: bad sizes");
    MVB_REQUIRE(n_active >= 0 && n_active <= N, "cheb_bwd_op: n_active=%d outside [0,%d]", n_active, N);
    MVB_REQUIRE(x && weight && dy && dweight && workspace && (nnz == 0 || d_coo_vals), "cheb_bwd_op: null pointer");
    MVB_REQUIRE(K == 1 || n_active == 0 || (basis && rowptr && colidx && perm && rowptr_t && colidx_t && vals_t),
                "cheb_bwd_op: null operator or basis pointer");
    if (!aligned16(workspace)) return set_err(MVB_EALIGN, "cheb_bwd_op: workspace not 16-byte aligned");
    const size_t need = mvb_cheb_bwd_op_workspace_bytes(N, B, Fin, Fout, K, n_active);
    if (workspace_bytes < need) return set_err(MVB_EWORKSPACE, "cheb_bwd_op: workspace %zu < %zu", workspace_bytes, need);
    const OpGradArgs og{rowptr, colidx, perm, d_coo_vals};
    return cheb_bwd_basis(N, B, Fin, Fout, K, n_active, nnz, rowptr_t, colidx_t, vals_t, x, basis, weight, y_for_relu, dy, dx,
                          dweight, dbias, &og, reinterpret_cast<char *>(workspace), (cudaStream_t)stream);
}

static int cheb_bwd_basis(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr_t,
                          const int32_t *colidx_t, const float *vals_t, const float *x, const float *basis,
                          const float *weight, const float *y_for_relu, const float *dy, float *dx, float *dweight,
                          float *dbias, const OpGradArgs *og, char *ws, cudaStream_t st) {
    const int64_t rows_act = (int64_t)n_active * B;
    const int64_t rows_in = (int64_t)(N - n_active) * B;
    WsCarve c{ws};
    const ChebBwdBasisWs w = cheb_bwd_basis_ws(c, N, B, Fin, Fout, K, n_active, dx != nullptr || og != nullptr);
    const int has_bias = dbias != nullptr;
    int rc, nA = 0, m4A = 0, nB = 0, m4B = 0;

    // The weight-gradient branch (partials + ordered finalize) and the input-gradient branch
    // (P_k, reverse recurrence) are independent: fork the former onto a side stream so that the two
    // overlap (and become parallel branches of a captured CUDA graph), join before returning.
    SideChain side(st, -1, dx != nullptr || og != nullptr);
    const cudaStream_t wst = side.stream();

    // dW_k = T_k^T dY, db = 1^T dY over the active prefix ...
    WgradArgs wa{};
    wa.rows = rows_act;
    wa.in_planes = K;
    wa.in_w = Fin;
    wa.in0 = x;
    wa.in_rest = basis;
    wa.dy = dy;
    wa.mask = y_for_relu;
    wa.n_out = Fout;
    wa.partials = w.partA;
    wa.partial_bytes = w.partA_bytes;
    rc = launch_wgrad_partials(wa, has_bias, &nA, &m4A, wst);
    if (rc) return rc;
    // ... plus S = x^T dY over the empty rows (dW_k += c_k S)
    if (rows_in > 0) {
        WgradArgs wb{};
        wb.rows = rows_in;
        wb.in_planes = 1;
        wb.in_w = Fin;
        wb.in0 = x + rows_act * Fin;
        wb.dy = dy + rows_act * Fout;
        wb.mask = y_for_relu ? y_for_relu + rows_act * Fout : nullptr;
        wb.n_out = Fout;
        wb.partials = w.partB;
        wb.partial_bytes = w.partB_bytes;
        rc = launch_wgrad_partials(wb, has_bias, &nB, &m4B, wst);
        if (rc) return rc;
    }
    rc = launch_wgrad_finalize(w.partA, nA, m4A, w.partB, nB, m4B, Fin, K * Fin, Fout, dweight, dbias, wst);
    if (rc || !(dx || og)) return rc;

    if (rows_act > 0) {
        // P_k = dY W_k^T for all k in one pass (plane k of the workspace)
        ContractArgs a{};
        a.rows = rows_act;
        a.in_planes = 1;
        a.in_w = Fout;
        a.in0 = dy;
        a.mask = y_for_relu;
        a.wmat = weight;          // [K*Fin, Fout] row-major == [Nn, M] -> transposed view
        a.w_transposed = 1;
        a.out_planes = K;
        a.out_w = Fin;
        a.out = w.P;
        rc = launch_contract(a, st);
        if (rc) return rc;
        // reverse recurrence, in place on the P planes: dX = sum_k T_k(L^T) P_k; for the operator gradient the planes
        // G_k = dloss/dT_k (k >= 1) stay in P
        rc = launch_cheb_recurrence_bwd(n_active, nnz, K, rowptr_t, colidx_t, vals_t, w.P, dx, (int64_t)B * Fin, st, og != nullptr);
        if (rc) return rc;
    }
    if (og) {
        // d_coo[e] = <G_1[r], T_0[c]> + 2 sum_{k>=2} <G_k[r], T_{k-1}[c]>; every entry lies in the active prefix
        if (K > 1 && rows_act > 0) {
            rc = launch_cheb_edge_grad(n_active, (int64_t)B * Fin, K, og->rowptr, og->colidx, og->perm, x, basis, w.P, og->d_coo_vals, st);
        } else if (nnz > 0) {
            const cudaError_t e = cudaMemsetAsync(og->d_coo_vals, 0, (size_t)nnz * sizeof(float), st);
            rc = e == cudaSuccess ? MVB_OK : set_err(MVB_ECUDA, "cheb_bwd_op: memset: %s", cudaGetErrorString(e));
        }
        if (rc) return rc;
    }
    if (rows_in > 0 && dx) {
        // empty rows: dX = dY (sum_k c_k W_k)^T
        ContractArgs a{};
        a.rows = rows_in;
        a.in_planes = 1;
        a.in_w = Fout;
        a.in0 = dy + rows_act * Fout;
        a.mask = y_for_relu ? y_for_relu + rows_act * Fout : nullptr;
        a.wmat = weight;
        a.w_transposed = 1;
        a.w_fold = K;
        a.out_planes = 1;
        a.out_w = Fin;
        a.out = dx + rows_act * Fin;
        rc = launch_contract(a, st);
        if (rc) return rc;
    }
    return MVB_OK;
}

static int cheb_bwd_adjoint(int N, int B, int Fin, int Fout, int K, int n_active, int nnz, const int32_t *rowptr_t,
                            const int32_t *colidx_t, const float *vals_t, const float *x, const float *weight,
                            const float *y_for_relu, const float *dy, float *dx, float *dweight, float *dbias, char *ws,
                            cudaStream_t st) {
    const int64_t rows_act = (int64_t)n_active * B, rows_in = (int64_t)(N - n_active) * B, rows_all = (int64_t)N * B;
    WsCarve c{ws};
    const ChebBwdAdjointWs w = cheb_bwd_adjoint_ws(c, N, B, Fin, Fout, K, n_active);
    // G = dY * [y > 0] over ALL rows, db = column sums of G
    const float *G = y_for_relu ? w.G : dy;
    int rc = launch_mask_colsum(rows_all, Fout, dy, y_for_relu, y_for_relu ? w.G : nullptr, dbias, w.colpart, st);
    if (rc) return rc;
    // S_k = T_k(L^T) G on the active prefix: the forward recurrence kernels with CSR(L^T)
    if (n_active > 0) {
        rc = launch_cheb_recurrence(n_active, nnz, K, rowptr_t, colidx_t, vals_t, G, w.S, (int64_t)B * Fout, st);
        if (rc) return rc;
    }
    // weight-gradient branch on a side stream, input-gradient contraction on the main stream.  Deferred mode (step
    // engine): the branch is joined lazily - nothing reads dW before the optimizer - so the contraction that the next
    // layer waits for no longer shares the memory system with it; otherwise forked and joined within this call.
    SideChain side(st, 0, true);
    const cudaStream_t wst = side.stream();
    // the input-gradient contraction is launched FIRST (the next layer waits for it; in deferred mode the
    // weight-gradient chain behind it then only takes the block slots it leaves free)
    if (rows_act > 0) {      // dX = sum_k S_k W_k^T
        ContractArgs a{};
        a.rows = rows_act;
        a.in_planes = K;
        a.in_w = Fout;
        a.in0 = G;
        a.in_rest = w.S;
        a.wmat = weight;
        a.w_transposed = 2;
        a.out_planes = 1;
        a.out_w = Fin;
        a.out = dx;
        rc = launch_contract(a, st);
        if (rc) return rc;
    }
    if (rows_in > 0) {       // empty rows: dX = G (sum_k c_k W_k)^T
        rc = launch_fold_dx(rows_in, K, Fin, Fout, G + rows_act * Fout, weight, dx + rows_act * Fin, st);
        if (rc) return rc;
    }
    int nA = 0, m4A = 0, nB = 0, m4B = 0;
    if (rows_act > 0) {      // A = [S_0|..|S_{K-1}]^T x   ([K*Fout, Fin]; dW_k[i][o] = A[k*Fout + o][i])
        WgradArgs wa{};
        wa.rows = rows_act;
        wa.in_planes = K;
        wa.in_w = Fout;
        wa.in0 = G;
        wa.in_rest = w.S;
        wa.dy = x;
        wa.n_out = Fin;
        wa.partials = w.partA;
        wa.partial_bytes = w.partA_bytes;
        rc = launch_wgrad_partials(wa, 0, &nA, &m4A, wst);
        if (rc) return rc;
    }
    if (rows_in > 0) {       // empty rows of the operator: S = x^T G, dW_k += cos(k pi/2) S
        rc = launch_fold_wgrad(rows_in, Fin, Fout, x + rows_act * Fin, G + rows_act * Fout, w.partB, w.partB_bytes, &nB, &m4B, wst);
        if (rc) return rc;
    }
    return launch_wgrad_finalize(w.partA, nA, m4A, w.partB, nB, m4B, Fin, K * Fin, Fout, dweight, nullptr, wst, 1);
}

// Make `stream` wait for the LATEST record of `event` at execution time.  With cudaEventWaitExternal the call is
// legal while `stream` is being captured and becomes an external event-wait node: every replay of the graph then
// waits for whatever the host recorded on the event last (the step engine's ground-truth H2D copy).
extern "C" int mvb_stream_wait_external_event(void *stream, void *event) {
    MVB_REQUIRE(event != nullptr, "stream_wait_external_event: null event");
    cudaError_t e = cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)event, cudaEventWaitExternal);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(MVB_ECUDA, "stream_wait_external_event: %s", cudaGetErrorString(e));
    }
    return MVB_OK;
}

// ---------------------------------------------------------------------------------------------
// run-time switches (tests, the step engine): NOT part of the operator API.  spec = "key=a[,b];key=..."
//   mesh_tc=e,c        tensor-core mesh layers on/off, CTAs per mesh (0 = automatic)
//   fused_recurrence=0|1  one-launch Chebyshev recurrence for the levels that fit shared memory off / on
//   stream_tc=e,sw     row-streaming fused level-0 layers (mvb_cheb_stream_*) on/off, meshes per slab (8 / 16, 0 = least work per CTA)
//   pdl=0|1            programmatic dependent launch of the step's kernels (default on; the engine switches it off for N > 1)
//   defer_wgrad=0|1    weight-gradient chains of the mesh layers joined lazily (engine only; see mvb_side_join)
// ---------------------------------------------------------------------------------------------
extern "C" int mvb_tune(const char *spec) {
    MVB_REQUIRE(spec != nullptr, "mvb_tune: null spec");
    const char *p = spec;
    while (*p) {
        char key[32];
        int n = 0, v[2] = {0, 0}, nv = 0;
        while (*p && *p != '=' && *p != ';' && n < 31) key[n++] = *p++;
        key[n] = 0;
        if (*p == '=') {
            ++p;
            while (nv < 2) {
                char *end = nullptr;
                v[nv] = (int)strtol(p, &end, 10);
                if (end == p) break;
                ++nv;
                p = end;
                if (*p == ',') ++p; else break;
            }
        }
        while (*p && *p != ';') ++p;
        if (*p == ';') ++p;
        if (!strcmp(key, "mesh_tc")) set_mesh_tc(v[0], v[1]);
        else if (!strcmp(key, "fused_recurrence")) set_recur_fused(v[0]);
        else if (!strcmp(key, "stream_tc")) set_stream_tc(v[0], nv > 1 ? v[1] : -1);
        else if (!strcmp(key, "pdl")) set_pdl(v[0]);
        else if (!strcmp(key, "defer_wgrad")) set_defer_wgrad(v[0]);
        else if (key[0]) return set_err(MVB_EINVAL, "mvb_tune: unknown key '%s'", key);
    }
    return MVB_OK;
}
