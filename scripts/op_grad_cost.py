"""Cost of the gradient with respect to the operator values: the backward pass of a level-0 ChebConv_batch 16 -> 16,
K = 6, B = 64 on the template operator with a frozen `norm` (adjoint form, no operator gradient) and with a learned one
(basis form + cheb_edge_grad_kernel), timed with CUDA events in alternating blocks, plus cheb_edge_grad_kernel alone
(torch.profiler, a separate pass) and its achieved bytes/s.

    python scripts/op_grad_cost.py --out DIR [--blocks 10 --iters 50]

Writes DIR/op_grad_cost.json with the card's name and power limit read in the same run.  The operands (~40 MB) fit the
126 MB L2: the numbers are L2-warm, as in a training step where the forward pass has just written them."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import meshvae_b200 as mvb  # noqa: E402
from oracle import mesh_vae_oracle as O  # noqa: E402
from tests.helpers import OPERATORS_NPZ  # noqa: E402

B, F, K = 64, 16, 6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def edge_grad_bytes(n_active, nnz):
    """compulsory traffic of cheb_edge_grad_kernel: G_1..G_{K-1} and T_0..T_{K-2} once each, rowptr, colidx, perm and
    the gradient; and the gathered traffic (each entry reads its neighbour's T rows: served by L2 / L1 after the first)"""
    plane = n_active * B * F * 4
    csr = (n_active + 1) * 4 + nnz * 4 * 2
    compulsory = 2 * (K - 1) * plane + csr + nnz * 4
    gathered = (K - 1) * (n_active * B * F * 4 + nnz * B * F * 4) + csr + nnz * 4
    return compulsory, gathered


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    dev = torch.device("cuda:0")
    A, _, _, nn_ = O.load_operators(OPERATORS_NPZ)
    n = nn_[0]
    ei, norm0 = mvb.ChebConv_batch.norm(A[0]._indices().to(dev), n)
    torch.manual_seed(0)
    conv = mvb.ChebConv_batch(F, F, K).to(dev)
    conv.fuse_relu = True
    x = torch.randn(B, n, F, device=dev).requires_grad_(True)
    gy = torch.randn(B, n, F, device=dev)
    learned = norm0.clone().requires_grad_(True)
    arms = {"frozen": (conv(x, ei, norm0), [x, conv.weight, conv.bias]),
            "learned": (conv(x, ei, learned), [x, conv.weight, conv.bias, learned])}

    def bwd(arm):
        y, inputs = arms[arm]
        return torch.autograd.grad(y, inputs, gy, retain_graph=True)

    for arm in arms:                                   # warm-up: workspaces, side stream, allocator
        for _ in range(5):
            bwd(arm)
    torch.cuda.synchronize()
    times = {arm: [] for arm in arms}
    for _ in range(a.blocks):
        for arm in arms:
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(a.iters):
                bwd(arm)
            e.record()
            e.synchronize()
            times[arm].append(s.elapsed_time(e) * 1e3 / a.iters)

    prof_iters = 50
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(prof_iters):
            bwd("learned")
        torch.cuda.synchronize()
    ka = [e for e in prof.key_averages() if "cheb_edge_grad_kernel" in e.key]
    launches = sum(e.count for e in ka)
    edge_mean = sum(e.device_time_total for e in ka) / launches if launches else None
    pat = mvb.operators.pattern_from_edges(ei, n, dev)
    compulsory, gathered = edge_grad_bytes(pat.n_active, pat.nnz)
    res = {
        "case": {"level": 0, "vertices": n, "nnz": pat.nnz, "B": B, "Fin": F, "Fout": F, "K": K, "relu": True, "dx": True},
        "card": card(),
        "backward_us": {arm: {"median": statistics.median(t), "min": min(t), "max": max(t), "blocks": t}
                        for arm, t in times.items()},
        "edge_grad_kernel": {
            "launches_seen": launches, "mean_us": edge_mean,
            "compulsory_bytes": compulsory, "gathered_bytes": gathered,
            "compulsory_GBps": compulsory / edge_mean / 1e3 if edge_mean else None,
            "gathered_GBps": gathered / edge_mean / 1e3 if edge_mean else None},
    }
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "op_grad_cost.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "backward_us"}, indent=1))
    print({arm: round(statistics.median(t), 2) for arm, t in times.items()}, "us per backward (median of blocks)")


if __name__ == "__main__":
    main()
