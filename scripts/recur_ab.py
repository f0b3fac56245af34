"""A/B the fused coarse-level recurrence kernel against the step-by-step SpMM launches on the level-1 / 2 operators, L2-warm and
cold."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import meshvae_b200 as mvb
import bench
dev = torch.device("cuda:0")
_, net, A, nn_ = bench.build_model(dev)
L = mvb._lib
flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
for lvl, B, F in [(1, 64, 16), (1, 64, 32), (2, 64, 16), (1, 256, 16)]:
    n = nn_[lvl]
    ei, norm = mvb.ChebConv_batch.norm(A[lvl]._indices(), n)
    op = mvb.operators.from_edges(ei, norm, n, dev)
    x = torch.randn(n, B, F, device=dev)
    w = torch.randn(6, F, 16, device=dev) * 0.1
    ref = None
    for fused in (0, 1):
        L.tune(f"fused_recurrence={fused}")
        basis = torch.empty(5, n, B, F, device=dev); y = torch.empty(n, B, 16, device=dev)
        ms = {}
        for cold in (True, False):
            t = []
            for i in range(13):
                if cold: flush.fill_(float(i))
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0 = L.lib.mvb_launch_count()
                s.record()
                L.check(L.lib.mvb_cheb_fwd(n, B, F, 16, 6, n, op.nnz, L.ptr(op.rowptr), L.ptr(op.colidx), L.ptr(op.vals), L.ptr(x), L.ptr(w), None, 0, L.ptr(basis), L.ptr(y), L.stream_ptr()))
                e.record(); e.synchronize()
                if i >= 3: t.append(s.elapsed_time(e))
            ms[cold] = sum(t) / len(t) * 1e3
        if ref is None: ref = basis.clone()
        print(f"lvl{lvl} B{B} F{F} fused={fused} ({L.lib.mvb_launch_count()-c0} launches): recurrence+contraction cold {ms[True]:6.1f} us  warm {ms[False]:6.1f} us  identical={torch.equal(basis, ref)}")
L.tune(f"fused_recurrence={1}")
