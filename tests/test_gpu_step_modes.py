"""The training step's launch modes against the serial path, bit for bit, and its gradients against float64.

Every step of TrainEngine runs backward with four mechanisms the kernel tests leave off: deferred weight-gradient chains
(mvb_tune "defer_wgrad=1": the dW / db reductions of the deferring entry points run on low-priority lane streams and
are joined once, by mvb_side_join), gradient sinks (the backward kernels write into views of one flat buffer),
programmatic dependent launch (PDL) and CUDA-graph capture.  include/mvb.h promises that pdl and defer_wgrad change only
how kernels are launched and joined.  This module holds them to that:

  1. each deferring entry point (mvb_cheb_bwd in the adjoint form, mvb_cheb_layer_bwd on the tensor-core mesh kernels,
     mvb_cheb_stream_bwd, mvb_linear_bwd with dx) in an autograd graph of at least five deferring layers - the three
     convolution lanes wrap around, chains queue behind each other and later layers run while earlier chains are
     pending - gives the same bits serial (no deferral, no PDL), deferred with PDL, and captured in a CUDA graph and
     replayed; the serial result meets the float64 reference of tests/operator_cases.py;
  2. while a chain is pending, every buffer it reads or writes (per the C sources) lies in a tensor that
     functional._park_or_join has parked in _lib._deferred["keep"] - a deterministic audit - and NaN-filled
     allocations of the freed temporaries' sizes do not change a bit (that part depends on timing);
  3. the whole engine (graph, deferral, PDL) against a serial engine: the same gradients, losses and parameters;
  4. the serial engine's step against the oracle model in float64, with the device's ReLU decisions: rel_err < 1e-4 and
     elem_err <= 1 for the loss, the outputs and every gradient at the benchmark batch.

Not covered here: the data-parallel paths (dp.PeerBuffers, the one-graph step that joins only lane 1 after the first
part of the backward pass) need two GPUs."""
import copy

import numpy as np
import pytest
import torch

from oracle import mesh_vae_oracle as O
from tests import operator_cases as C
from tests.helpers import OPERATORS_NPZ, elem_err, rel_err, seeded_state_dict

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOL = 1e-4
FLIP = 1e-5            # a ReLU decision may differ from the reference only within FLIP * max|pre-activation| of zero
DEFAULTS = "mesh_tc=1,0;stream_tc=0,16;fused_recurrence=1;pdl=1;defer_wgrad=0"
MAX_ERR = {}           # part -> largest rel_err seen (printed at the end of the module with pytest -s)
AUDITED = {}           # entry point -> deferred calls audited


@pytest.fixture(scope="module")
def mvb():
    import meshvae_b200
    assert meshvae_b200._lib.lib.mvb_device_cc() == 100, "these kernels are built for sm_100a only"
    yield meshvae_b200
    print("\nlargest rel_err per part: " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(MAX_ERR.items())))
    print("deferred calls audited: " + ", ".join(f"{k} {v}" for k, v in sorted(AUDITED.items())))


def _restore(mvb):
    mvb._lib.defer_side_chains(False)
    mvb._lib.side_join()
    mvb._lib.tune(DEFAULTS)
    mvb._lib.lib.mvb_set_tensor_cores(1)


def _note(part, e):
    MAX_ERR[part] = max(MAX_ERR.get(part, 0.0), e)


def _gate(part, what, dev, ref):
    d = dev.detach().double().cpu() if isinstance(dev, torch.Tensor) else torch.from_numpy(np.asarray(dev, np.float64))
    r = ref.detach().double().cpu() if isinstance(ref, torch.Tensor) else torch.from_numpy(np.asarray(ref, np.float64))
    e = rel_err(d, r)
    _note(part, e)
    assert e < TOL, f"{part} {what}: rel_err {e:.3e}"
    ee = elem_err(d, r)
    assert ee <= 1.0, f"{part} {what}: elem_err {ee:.3f}"


# ---------------------------------------------------------------------------------------------
# part 2: the parking audit.  functional.lib is wrapped in a recorder that notes, for each backward call of a deferring
# entry point, the buffers its pending chain reads or writes; functional._park_or_join is wrapped so that, right after
# a call has parked its tensors (and before any join), each of those pointers is checked against the storages in
# _lib._deferred["keep"], and NaN-filled tensors of the sizes of the call's temporaries are allocated on the main stream.
# ---------------------------------------------------------------------------------------------
def _chain_buffers(name, a):
    """[(what, pointer, bytes)] of what the deferred chain of one call reads or writes, read off the C sources:
    mvb_cheb_bwd, adjoint form (csrc/mvb_api.cu cheb_bwd_adjoint): workspace (G, S_k, partials), x, dweight, and dy
        itself when there is no ReLU (G = dy); db is reduced on the caller's stream
    mvb_cheb_layer_bwd (csrc/mvb_mesh_tc.cu launch_mesh_tc_bwd) and mvb_cheb_stream_bwd (csrc/mvb_stream_tc.cu
        launch_stream_tc_bwd): workspace (S_k, T_0, db partials, dW partials), x when there is no U prologue, dweight,
        dbias
    mvb_linear_bwd with dx (csrc/mvb_dense.cu): x, y, gy, dW, db
    The bytes size the NaN-filled allocations after the call; an entry without a pointer ("(dy)") only sizes one.
    -> None when the call does not defer"""
    f4 = 4
    if name == "mvb_cheb_bwd":
        n, b, fin, fout = a[0], a[1], a[2], a[3]
        x, y, dy, dx, dw, ws, ws_bytes = a[10], a[13], a[14], a[15], a[16], a[18], a[19]
        if dx is None or _Recorder.real.mvb_cheb_bwd_uses_basis(fin, fout, 1):
            return None
        out = [("workspace", ws, ws_bytes), ("x", x, n * b * fin * f4), ("dweight", dw, 0)]
        if y is None:
            out.append(("dy", dy, n * b * fout * f4))
        return out
    if name == "mvb_cheb_layer_bwd":
        n, b, fin, fout = a[0], a[1], a[2], a[3]
        n_in, urp, n_out = a[12], a[13], a[20]
        x, dw, db, ws, ws_bytes = a[22], a[27], a[28], a[29], a[30]
        out = [("workspace", ws, ws_bytes), ("dweight", dw, 0), ("dbias", db, 0)]
        if urp is None:
            out.append(("x", x, n_in * b * fin * f4))
        return out + [("(dy)", None, n_out * b * fout * f4)]
    if name == "mvb_cheb_stream_bwd":
        n, b, fin, fout = a[0], a[1], a[2], a[3]
        n_in, urp = a[9], a[10]
        x, dw, db, ws, ws_bytes = a[17], a[22], a[23], a[24], a[25]
        out = [("workspace", ws, ws_bytes), ("dweight", dw, 0), ("dbias", db, 0)]
        if urp is None:
            out.append(("x", x, n_in * b * fin * f4))
        return out + [("(dy)", None, n * b * fout * f4)]
    if name == "mvb_linear_bwd":
        m, k, n = a[0], a[1], a[2]
        x, y, gy, dx, dw, db = a[3], a[6], a[7], a[11], a[12], a[13]
        if dx is None:
            return None
        return [("x", x, m * k * f4), ("y", y, m * n * f4), ("gy", gy, m * n * f4), ("dW", dw, 0), ("db", db, 0)]
    return None


class _Recorder:
    """stands in for functional.lib: the four deferring backward entry points are recorded, everything else passes"""
    NAMES = ("mvb_cheb_bwd", "mvb_cheb_layer_bwd", "mvb_cheb_stream_bwd", "mvb_linear_bwd")
    real = None

    def __init__(self, lib, deferred):
        _Recorder.real = lib
        self._deferred = deferred
        self.last = None
        self.pressure = []
        self.audited = {}

    def __getattr__(self, name):
        fn = getattr(_Recorder.real, name)
        if name not in self.NAMES:
            return fn

        def call(*args):
            rc = fn(*args)
            self.last = (name, _chain_buffers(name, args)) if self._deferred["on"] else None
            return rc
        return call


@pytest.fixture
def audit(mvb, monkeypatch):
    Fn, L = mvb.functional, mvb._lib
    rec = _Recorder(L.lib, L._deferred)
    real_park, real_join = Fn._park_or_join, L.side_join

    def park(ctx, tensors):
        n0 = len(L._deferred["keep"])
        real_park(ctx, tensors)
        last, rec.last = rec.last, None
        if last is None or last[1] is None or len(L._deferred["keep"]) == n0:
            return                     # not deferred, or joined at once (a gradient that goes back to autograd)
        name, bufs = last
        spans = []
        for group in L._deferred["keep"]:
            for t in group:
                if t is not None and t.numel():
                    s = t.untyped_storage()
                    spans.append((s.data_ptr(), s.data_ptr() + s.nbytes()))
        for what, p, _ in bufs:
            if p:
                assert any(lo <= p < hi for lo, hi in spans), f"{name}: {what} is read by the pending chain but not parked"
        rec.audited[name] = rec.audited.get(name, 0) + 1
        AUDITED[name] = AUDITED.get(name, 0) + 1
        if not torch.cuda.is_current_stream_capturing():
            # the memory a missed park would have freed goes to the next allocation of the same size class
            for _, _, nbytes in bufs:
                if nbytes:
                    rec.pressure.append(torch.full((nbytes // 4 + 1,), float("nan"), device=DEV))

    def join(lane=None):
        real_join(lane)
        if lane is None:
            assert not L._deferred["keep"], "side_join left tensors parked"
            rec.pressure.clear()

    monkeypatch.setattr(Fn, "lib", rec)
    monkeypatch.setattr(Fn, "_park_or_join", park)
    monkeypatch.setattr(L, "side_join", join)
    yield rec


# ---------------------------------------------------------------------------------------------
# part 1: graphs of deferring layers, serial / deferred / captured
# ---------------------------------------------------------------------------------------------
N_SMALL = 300
SMALL_OPS = {
    "irr": lambda: C.irregular(N_SMALL, seed=1, hubs=3, hub_deg=(200, 290), isolated=9, dups=30, loops=12),
    "irr2": lambda: C.irregular(N_SMALL, seed=41, dups=10, loops=5, isolated=3),
    "tail": lambda: C.irregular(N_SMALL, seed=5, n_active=241, dups=10, loops=5, isolated=4),
    "up": lambda: C.upsample(N_SMALL, 75, seed=6),
    "up2": lambda: C.upsample(N_SMALL, 75, seed=7, max_per_row=3),
    "down": lambda: C.selection(N_SMALL, 75, seed=8),
}
BIG_OPS = {
    "dir0": lambda: C.directed(0, seed=8, both=False),
    "rel0": lambda: C.relabelled(0, seed=10),
    "up": lambda: C.upsample(4998, 1250, seed=11, max_per_row=3),
    "up2": lambda: C.upsample(4998, 1250, seed=12, max_per_row=3),
    "down": lambda: C.selection(4998, 1250, seed=13),
}
# layer specs: ("conv", L, fin, fout, K, relu, bias) - cheb_conv;  ("layer", L, U, D, fin, fout, K, bias) - cheb_layer with
# ReLU (the fused kernels' layers);  ("pool", P);  ("linear", fin, fout, p) - fused Linear + ReLU + dropout, with bias
CHAINS = {
    # the adjoint form: 16 -> 16, 32 -> 32, 32 -> 16, with and without ReLU (the chain then reads dY), K = 1 / 6 / 8, and
    # an isolated tail (n_active < N: the chain folds the closed-form rows with launch_fold_wgrad).  The 16 -> 32 layer
    # takes the basis form, which joins its weight-gradient branch before it returns.
    "adjoint": ("small", (N_SMALL, 16), [
        ("conv", "irr", 16, 16, 6, True, True), ("conv", "irr2", 16, 16, 1, False, True),
        ("conv", "irr", 16, 32, 3, True, True), ("conv", "irr2", 32, 32, 8, True, False),
        ("conv", "tail", 32, 32, 6, False, True), ("conv", "irr", 32, 16, 8, True, True),
        ("conv", "tail", 16, 16, 8, False, True)]),
    # the tensor-core mesh layers: with a U prologue (the chain reads T_0 from the workspace) and without (it reads x),
    # with and without bias, K = 9 and 16 (several weight-gradient plane groups on the chain)
    "mesh": ("small", (75, 16), [
        ("layer", "irr", "up", None, 16, 16, 9, True), ("layer", "irr2", None, None, 16, 16, 16, False),
        ("layer", "irr", None, "down", 16, 16, 9, True), ("layer", "irr2", "up2", None, 16, 16, 16, False),
        ("layer", "irr", None, None, 16, 16, 9, True), ("layer", "irr2", None, None, 16, 16, 16, True)]),
    # the row-streaming layers of level 0, dec (U prologue) and plain
    "stream": ("big", (1250, 16), [
        ("layer", "dir0", "up", None, 16, 16, 6, True), ("layer", "rel0", None, None, 16, 16, 8, False),
        ("pool", "down"),
        ("layer", "rel0", "up2", None, 16, 16, 3, True), ("layer", "dir0", None, None, 16, 16, 6, True),
        ("layer", "rel0", None, None, 16, 16, 6, False)]),
    # the dense layers: dx, ReLU and dropout 0.2 (their dW / db tiles are the chains of lane 1)
    "linear": ("dense", (96,), [("linear", 96, 128, 0.2), ("linear", 128, 64, 0.2), ("linear", 64, 160, 0.2),
                                ("linear", 160, 96, 0.2), ("linear", 96, 128, 0.2)]),
}
DEFERRING = {"adjoint": ("mvb_cheb_bwd", 6), "mesh": ("mvb_cheb_layer_bwd", 6), "stream": ("mvb_cheb_stream_bwd", 5),
             "linear": ("mvb_linear_bwd", 5)}
PART1 = ([("adjoint", "", b) for b in (1, 3, 64, 300)] +
         [("mesh", m, b) for m in ("mesh_tc=1,1", "mesh_tc=1,2") for b in (1, 3, 64, 300)] +
         [("stream", m, 64) for m in ("stream_tc=1,8", "stream_tc=1,16")] +
         [("linear", "", b) for b in (1, 3, 64, 300)])


def _f32(a):
    return np.asarray(a, np.float32).astype(np.float64)


class _Graph:
    """the layers of one CHAINS entry on the device (parameters with gradient sinks into one flat buffer) and on the
    host (the same fp32 values in float64, the operators as float64 CSR)"""

    def __init__(self, mvb, chain, b, seed):
        kind, in_shape, specs = CHAINS[chain]
        self.mvb, self.specs, self.b = mvb, specs, b
        Fn = mvb.functional
        ops = {"small": SMALL_OPS, "big": BIG_OPS}.get(kind, {})
        used = {s[1] for s in specs if s[0] in ("conv", "layer")} | {s[2] for s in specs if s[0] == "layer"} | \
               {s[3] for s in specs if s[0] == "layer"} | {s[1] for s in specs if s[0] == "pool"}
        self.ops = {k: ops[k]() for k in used if k is not None}
        self.dev_ops = {}
        for k, op in self.ops.items():
            if op.n_rows == op.n_cols and not k.startswith(("up", "down")):
                ei, norm = op.edges()
                self.dev_ops[k] = mvb.operators.from_edges(ei.to(DEV), norm.to(DEV), op.n_rows, DEV)
            else:
                self.dev_ops[k] = mvb.operators.from_sparse(op.sparse().to(DEV), DEV)
        rng = np.random.default_rng(seed)
        host, self.params = [], []
        for s in specs:
            if s[0] == "conv":
                _, _, fin, fout, k, _, bias = s
            elif s[0] == "layer":
                _, _, _, _, fin, fout, k, bias = s
            elif s[0] == "linear":
                _, fin, fout, _ = s
                w = _f32(rng.standard_normal((fout, fin)) / np.sqrt(fin))
                host.append((w, _f32(rng.standard_normal(fout) * 0.1)))
                continue
            else:
                host.append((None, None))
                continue
            host.append((_f32(rng.standard_normal((k, fin, fout)) * 0.1), _f32(rng.standard_normal(fout) * 0.1) if bias else None))
        self.host = host
        dev = [(None if w is None else torch.tensor(w, dtype=torch.float32, device=DEV).requires_grad_(True),
                None if bb is None else torch.tensor(bb, dtype=torch.float32, device=DEV).requires_grad_(True)) for w, bb in host]
        flat_params = [p for pair in dev for p in pair if p is not None]
        offsets, n = mvb.dp.flat_layout(flat_params, 32)
        self.flat = torch.zeros(n, device=DEV)
        views = mvb.dp.flat_views(self.flat, flat_params, offsets)
        for p, v in zip(flat_params, views):
            p._mvb_grad_sink = v                 # as engine.TrainEngine installs them
        self.sinks = {id(p): v for p, v in zip(flat_params, views)}
        self.dev = dev
        shape = (in_shape[0], b, in_shape[1]) if len(in_shape) == 2 else (b, in_shape[0])
        self.x_host = _f32(rng.standard_normal(shape))
        self.x = torch.tensor(self.x_host, dtype=torch.float32, device=DEV).requires_grad_(True)
        self.rng_off = torch.zeros((), dtype=torch.int64, device=DEV)
        for s in specs:          # the adjoint form wherever the specs above say so (Fout <= 1.2 Fin)
            if s[0] == "conv":
                assert bool(Fn.lib.mvb_cheb_bwd_uses_basis(s[2], s[3], 1)) == (s[3] > 1.2 * s[2]), s

    def forward(self, x):
        """-> (output, [device output of every layer])"""
        Fn = self.mvb.functional
        h, outs = x, []
        for i, (s, (w, bb)) in enumerate(zip(self.specs, self.dev)):
            if s[0] == "conv":
                h = Fn.cheb_conv(h, w, bb, self.dev_ops[s[1]], s[5])
            elif s[0] == "layer":
                lo, uo = self.dev_ops[s[1]], self.dev_ops.get(s[2])
                do = self.dev_ops.get(s[3])
                h = Fn.cheb_layer(h, w, bb, lo, uo, do, relu=True)
            elif s[0] == "pool":
                h = Fn.pool(h, self.dev_ops[s[1]])
            else:
                h = Fn.linear(h, w, bb, relu=True, p=s[3], rng=(0x5EED + 977 * i, self.rng_off, 3))
            outs.append(h)
        return h, outs

    def layer_kinds(self):
        """the fused-layer kind (mesh / stream) each cheb_layer spec takes under the current switches"""
        Fn = self.mvb.functional
        kinds, n_in = [], self.x.shape[0]
        for s in self.specs:
            if s[0] == "layer":
                lo, uo, do = self.dev_ops[s[1]], self.dev_ops.get(s[2]), self.dev_ops.get(s[3])
                kinds.append(Fn._fused_layer_kind(lo.n_rows, self.b, s[4], s[5], s[6], lo, uo, do))
        return kinds

    def run(self, gy, x=None):
        """forward + backward through autograd -> (y, [layer outputs], dx); the weight gradients go into the sinks"""
        x = self.x if x is None else x
        y, outs = self.forward(x)
        dx, = torch.autograd.grad(y, [x], gy)
        return y, outs, dx


def _reference(g: _Graph, outs_dev, gy):
    """float64 forward and backward of the graph with the device's ReLU (and dropout) decisions -> (outputs, dx,
    [(dW, db)])"""
    h = g.x_host
    saved, ref_outs = [], []
    for s, (w, bb), yd in zip(g.specs, g.host, outs_dev):
        yd = yd.detach().double().cpu().numpy()
        if s[0] == "pool":
            saved.append(None)
            h = C.pool_ref(h, g.ops[s[1]].csr)
            ref_outs.append(h)
            continue
        if s[0] == "linear":
            pre = h @ w.T + bb
            keep = yd > 0
            assert np.all(pre[keep] > -FLIP * np.abs(pre).max()), "a kept output has a negative pre-activation"
            scale = 1.0 / (1.0 - s[3]) if s[3] > 0 else 1.0
            mask = keep * scale
            saved.append((h, mask))
            h = pre * mask
        else:
            L = g.ops[s[1]].csr
            U = g.ops[s[2]].csr if s[0] == "layer" and s[2] is not None else None
            D = g.ops[s[3]].csr if s[0] == "layer" and s[3] is not None else None
            pre, t0 = C.cheb_ref_fwd(h, L, w, bb, U)
            if D is not None:
                pre = C.pool_ref(pre, D)
            relu = s[0] == "layer" or s[5]
            if relu:
                mask = (yd > 0).astype(np.float64)
                flips = mask != (pre > 0)
                assert np.all(np.abs(pre[flips]) <= FLIP * np.abs(pre).max()), "a ReLU decision differs from the reference"
            else:
                mask = np.ones_like(pre)
            saved.append((t0, mask, L, U, D))
            h = pre * mask
        ref_outs.append(h)
    g_ = gy.detach().double().cpu().numpy()
    grads = []
    for s, (w, bb), sv in zip(reversed(g.specs), reversed(g.host), reversed(saved)):
        if s[0] == "pool":
            g_ = C.pool_ref_bwd(g_, g.ops[s[1]].csr)
            grads.append((None, None))
            continue
        if s[0] == "linear":
            xin, mask = sv
            gm = g_ * mask
            grads.append((gm.T @ xin, gm.sum(0)))
            g_ = gm @ w
            continue
        t0, mask, L, U, D = sv
        gm = g_ * mask
        if D is not None:
            gm = C.pool_ref_bwd(gm, D)
        g_, dw, db = C.cheb_ref_bwd(gm, t0, L, w, U)
        grads.append((dw, db if bb is not None else None))
    return ref_outs, g_, grads[::-1]


def _grads(g: _Graph):
    return [tuple(None if p is None else g.sinks[id(p)].clone() for p in pair) for pair in g.dev]


@pytest.mark.parametrize("chain,mode,b", PART1, ids=[f"{c}-{m.replace('=', '').replace(',', '_') or 'auto'}-B{b}" for c, m, b in PART1])
def test_deferred_and_captured_backward_are_bit_identical_to_serial(mvb, audit, chain, mode, b):
    L = mvb._lib
    g = _Graph(mvb, chain, b, seed=b * 31 + len(chain))
    try:
        if mode:
            L.tune(mode)
        kinds = g.layer_kinds()
        if chain == "mesh":
            assert kinds == ["mesh"] * 6, kinds
        if chain == "stream":
            assert kinds == ["stream"] * 5, kinds
        y0, _ = g.forward(g.x)
        gy = torch.tensor(_f32(np.random.default_rng(b + 7).standard_normal(tuple(y0.shape))), dtype=torch.float32, device=DEV)
        del y0
        results = {}

        # (a) serial: every chain joined within its call, no programmatic dependent launch
        L.defer_side_chains(False)
        L.tune("pdl=0")
        g.flat.fill_(float("nan"))
        y, outs, dx = g.run(gy)
        torch.cuda.synchronize()
        results["serial"] = (y.detach().clone(), dx.clone(), _grads(g))
        serial_outs = [o.detach().clone() for o in outs]
        del y, outs, dx

        # (b) what the engine runs: deferred chains (audited), PDL, one join at the end
        L.tune("pdl=1")
        L.defer_side_chains(True)
        g.flat.fill_(float("nan"))
        n_audit = audit.audited.get(DEFERRING[chain][0], 0)
        y, outs, dx = g.run(gy)
        L.side_join()
        torch.cuda.synchronize()
        results["deferred"] = (y.detach().clone(), dx.clone(), _grads(g))
        assert audit.audited.get(DEFERRING[chain][0], 0) - n_audit == DEFERRING[chain][1], audit.audited
        del y, outs, dx

        # (c) (b) captured in a CUDA graph (the lane streams exist: (b) ran uncaptured) and replayed twice.  Warm-up and
        # capture on one stream, with an input leaf first used there: autograd then has no other stream to wait for
        graph = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            xc = g.x.detach().clone().requires_grad_(True)
            y, outs, dx = g.run(gy, xc)
            L.side_join()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        del y, outs, dx
        with torch.cuda.graph(graph, stream=s):
            y, outs, dx = g.run(gy, xc)
            L.side_join()
        for r in range(2):
            g.flat.fill_(float("nan"))
            dx.fill_(float("nan"))
            y.detach().fill_(float("nan"))
            graph.replay()
            torch.cuda.synchronize()
            results[f"replay{r}"] = (y.detach().clone(), dx.clone(), _grads(g))
        L.defer_side_chains(False)
        del graph
    finally:
        _restore(mvb)

    ya, dxa, ga = results["serial"]
    for m, (yb, dxb, gb) in results.items():
        assert torch.equal(ya, yb), f"{m}: output"
        assert torch.equal(dxa, dxb), f"{m}: dx"
        for i, (pa, pb) in enumerate(zip(ga, gb)):
            for what, ta, tb in (("dW", pa[0], pb[0]), ("db", pa[1], pb[1])):
                if ta is not None:
                    assert torch.equal(ta, tb), f"{m}: layer {i} {what}"

    # the serial result against float64
    ref_outs, dx_ref, grads_ref = _reference(g, serial_outs, gy)
    part = "1 " + chain
    for i, (o, r) in enumerate(zip(serial_outs, ref_outs)):
        _gate(part, f"layer {i} output", o, r)
    _gate(part, "dx", dxa, dx_ref)
    for i, ((dw, db), (rw, rb)) in enumerate(zip(ga, grads_ref)):
        if dw is not None:
            _gate(part, f"layer {i} dW", dw, rw)
        if db is not None:
            _gate(part, f"layer {i} db", db, rb)


# ---------------------------------------------------------------------------------------------
# part 3: the whole engine, default (graph, deferral, PDL) against serial (eager, no deferral, no PDL)
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ops():
    return O.load_operators(OPERATORS_NPZ)


ENGINE_CONFIGS = {"default": {}, "orders87163_widths8_24": dict(polygon_order=[8, 7, 1, 6, 3], num_conv_filters=[8, 8, 24, 24, 24],
                                                                 num_classes=3, num_style=8)}


def _config(name, dropout):
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    cfg.update(ENGINE_CONFIGS[name])
    cfg["dropout"] = dropout
    return cfg


def _net(mvb, ops, cfg, seed=11):
    A, D, U, nn_ = ops
    net = mvb.cheb_VAE(3, copy.deepcopy(cfg), [d.to(DEV) for d in D], [u.to(DEV) for u in U], [a.to(DEV) for a in A], nn_,
                       model=cfg["model"])
    net.load_state_dict(seeded_state_dict(net, seed))
    return net.to(DEV)


def _batch(b, n, classes, z, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, n, 3, generator=g)
    y = torch.arange(b)[torch.randperm(b, generator=g)] % classes
    return x, y, torch.randn(b, z, generator=g)


def _engine_run(mvb, ops, cfg, b, steps, serial, monkeypatch):
    """-> (losses, flat_g after step 0, flat_p after the last step)"""
    from meshvae_b200.engine import TrainEngine
    L = mvb._lib
    real = L.defer_side_chains
    try:
        if serial:
            L.tune("pdl=0")
            monkeypatch.setattr(L, "defer_side_chains", lambda on: real(False))
        net = _net(mvb, ops, cfg)
        eng = TrainEngine(net, b, lr=1e-3, weight_decay=5e-4, use_graph=not serial)
        eng.capture(warmup=1)
        losses, g0 = [], None
        for s in range(steps):
            x, y, eps = _batch(b, ops[3][0], cfg["num_classes"], cfg["num_style"], 900 + s)
            losses.append(eng.step(x.pin_memory(), x.double().pin_memory(), y.pin_memory(), eps_host=eps.pin_memory()))
            if s == 0:
                g0 = eng.opt.flat_g.clone()
        torch.cuda.synchronize()
        return losses, g0, eng.opt.flat_p.clone()
    finally:
        monkeypatch.setattr(L, "defer_side_chains", real)
        _restore(mvb)


PART3 = ([("default", b, p, 3) for b in (1, 3, 64, 300) for p in (0.0, 0.2)] + [("default", 512, 0.0, 1)] +
         [("orders87163_widths8_24", 16, 0.2, 3)])


@pytest.mark.parametrize("name,b,p,steps", PART3, ids=[f"{n}-B{b}-p{p}" for n, b, p, _ in PART3])
def test_engine_default_step_is_bit_identical_to_serial(mvb, ops, audit, monkeypatch, name, b, p, steps):
    cfg = _config(name, p)
    n0 = dict(audit.audited)
    la, ga, pa = _engine_run(mvb, ops, cfg, b, steps, False, monkeypatch)
    for ep in ("mvb_cheb_bwd", "mvb_linear_bwd") + (("mvb_cheb_layer_bwd",) if name == "default" else ()):
        assert audit.audited.get(ep, 0) > n0.get(ep, 0), f"the default engine deferred no {ep} call"
    lb, gb, pb = _engine_run(mvb, ops, cfg, b, steps, True, monkeypatch)
    assert all(np.isfinite(v) for v in la), la
    assert la == lb, (la, lb)
    assert torch.equal(ga, gb), "step-0 gradients differ"
    assert torch.equal(pa, pb), f"parameters differ after {steps} steps"


# ---------------------------------------------------------------------------------------------
# part 4: the serial engine's step 0 against the oracle in float64, with the device's ReLU decisions
# ---------------------------------------------------------------------------------------------
class _MaskedF:
    """stands in for torch.nn.functional inside the oracle: relu multiplies by the next recorded device mask"""

    def __init__(self, masks):
        self.masks = list(masks)
        self.flips = []

    def __getattr__(self, name):
        return getattr(torch.nn.functional, name)

    def relu(self, t):
        m, rows = self.masks.pop(0)
        pre = t.detach()
        own = (pre > 0).double()
        if rows is not None:        # encoder site: the device saw only the rows D keeps (the others get no gradient)
            full = own.clone()
            full[:, rows] = m
            sel_pre, sel_m, sel_own = pre[:, rows], m, own[:, rows]
        else:
            full, sel_pre, sel_m, sel_own = m, pre, m, own
        flips = sel_m != sel_own
        bound = FLIP * float(sel_pre.abs().max())
        worst = float(sel_pre[flips].abs().max()) if bool(flips.any()) else 0.0
        self.flips.append((int(flips.sum()), worst, bound))
        return t * full


@pytest.mark.parametrize("b", [64, 300])
def test_engine_step_matches_float64_with_device_relu_decisions(mvb, ops, monkeypatch, b):
    from meshvae_b200.engine import TrainEngine
    Fn, L = mvb.functional, mvb._lib
    cfg = _config("default", 0.0)
    A, D, U, nn_ = ops
    x, y, eps = _batch(b, nn_[0], cfg["num_classes"], cfg["num_style"], 4242 + b)
    rec = {"on": False, "sites": [], "heads": None}
    real = L.defer_side_chains
    try:
        L.tune("pdl=0")
        monkeypatch.setattr(L, "defer_side_chains", lambda on: real(False))
        net = _net(mvb, ops, cfg, seed=7)
        real_layer, real_linear, real_heads = net._layer, Fn.linear, Fn.vae_heads

        def layer(h, conv, lvl, up=None, down=None):
            out = real_layer(h, conv, lvl, up=up, down=down)
            if rec["on"]:
                rec["sites"].append((out.detach().double().cpu(), down))
            return out

        def linear(h, *a, **kw):
            out = real_linear(h, *a, **kw)
            if rec["on"]:
                o = out.detach()
                o = o.permute(1, 0, 2).reshape(o.shape[1], -1) if kw.get("y_vm_f") else o
                rec["sites"].append((o.double().cpu(), None))
            return out

        def heads(*a, **kw):
            out = real_heads(*a, **kw)
            if rec["on"]:
                rec["heads"] = [t.detach().double().cpu() for t in out[:4]]
            return out
        monkeypatch.setattr(net, "_layer", layer)
        monkeypatch.setattr(Fn, "linear", linear)
        monkeypatch.setattr(Fn, "vae_heads", heads)
        eng = TrainEngine(net, b, lr=1e-3, weight_decay=5e-4, use_graph=False)
        eng.capture(warmup=1)
        rec["on"] = True
        loss = eng.step(x.pin_memory(), x.double().pin_memory(), y.pin_memory(), eps_host=eps.pin_memory())
        rec["on"] = False
        torch.cuda.synchronize()
        dev = {"loss": torch.tensor(loss, dtype=torch.float64), "recon": eng.recon.double().cpu(), "kld": eng.kld.double().cpu(),
               "rec": eng.rec.double().cpu()}
        names = {id(p): n for n, p in net.named_parameters()}
        grads = {names[id(p)]: v.detach().double().cpu() for p, v in zip(eng.opt.params, eng.opt.grad_views)}
    finally:
        monkeypatch.setattr(L, "defer_side_chains", real)
        _restore(mvb)
    assert len(rec["sites"]) == 11, len(rec["sites"])

    # the masks, in the oracle's call order: 4 encoder convolutions, enc_lin, dec_lin, dec_lin_2, 4 decoder convolutions
    masks = []
    for out, down in rec["sites"]:
        m = (out > 0).double()
        if down is not None:
            idx = down._indices().cpu()
            order = torch.argsort(idx[0])
            rows = idx[1][order]
            assert rows.numel() == out.shape[1]
            masks.append((m, rows))
        else:
            masks.append((m, None))
    mf = _MaskedF(masks)
    ref = O.OracleChebVAE(3, cfg, D, U, A, nn_)
    ref.load_state_dict(seeded_state_dict(ref, 7))
    ref.double()
    ref.train()
    monkeypatch.setattr(O, "F", mf)
    y_hot = torch.nn.functional.one_hot(y, cfg["num_classes"]).double()
    lo, co, ro, (ko, reco, zo), yho = ref(x.double(), x.double(), y_hot, m_type="train", eps=eps.double())
    lo.backward()
    monkeypatch.undo()
    assert not mf.masks, "the oracle used fewer ReLU sites than the device"
    for i, (n, worst, bound) in enumerate(mf.flips):
        assert worst <= bound, f"ReLU site {i}: {n} decisions differ, the largest pre-activation {worst:.3e} > {bound:.3e}"
    print(f"\nB={b}: ReLU decisions that differ from the oracle's own, per site: {[n for n, _, _ in mf.flips]}")

    part = f"4 B{b}"
    _gate(part, "loss", dev["loss"], lo)
    _gate(part, "recon", dev["recon"], ro)
    _gate(part, "kld", dev["kld"], ko)
    _gate(part, "rec", dev["rec"], reco)
    y_hat, mu, logvar, z_ = rec["heads"]
    for what, a, r in (("y_hat", y_hat, yho), ("z", z_, zo)):
        _gate(part, what, a, r)
    po = dict(ref.named_parameters())
    worst = {}
    for name, gv in grads.items():
        r = po[name].grad
        assert r is not None, name
        worst[name] = rel_err(gv, r)
        _gate(part + " grad", name, gv, r)
    print(f"B={b}: largest gradient rel_err {max(worst.values()):.2e} ({max(worst, key=worst.get)})")
