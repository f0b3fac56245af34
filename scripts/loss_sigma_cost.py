"""Cost of the sigma-VAE decoder variances in the training step: the captured TrainEngine step (default config, B = 64,
dropout 0.2, fp64 ground truth) with the reference's constant sigma, the optimal sigma and the learned sigma, timed with
CUDA events in alternating blocks of graph replays on inputs already on the device, plus the loss kernels of each mode
(torch.profiler, a separate pass).

    python scripts/loss_sigma_cost.py --out DIR [--blocks 10 --iters 50]

Writes DIR/loss_sigma_cost.json with the card's name and power limit read in the same run."""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import meshvae_b200 as mvb  # noqa: E402
from meshvae_b200.engine import TrainEngine  # noqa: E402
from oracle import mesh_vae_oracle as O  # noqa: E402
from tests.helpers import OPERATORS_NPZ, seeded_state_dict  # noqa: E402

B = 64
MODES = ("fixed", "optimal", "learned")
LOSS_KERNELS = ("vae_rec_partial_kernel", "vae_loss_finalize_kernel", "scale4_by_gloss_kernel", "scale_by_gloss_kernel",
                "vae_loss_bwd_small_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def engine(mode, ops, dev):
    A, D, U, nn_ = ops
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    net = mvb.cheb_VAE(3, cfg, [d.to(dev) for d in D], [u.to(dev) for u in U], [a.to(dev) for a in A], nn_)
    net.load_state_dict(seeded_state_dict(net, 7))
    net = net.to(dev)
    net.set_decoder_sigma(mode)
    eng = TrainEngine(net, B)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, nn_[0], 3, generator=g)
    eng.capture()
    eng.step(x.pin_memory(), x.double().pin_memory(), (torch.arange(B) % 2).pin_memory(),
             eps_host=torch.randn(B, net.z, generator=g).pin_memory())
    torch.cuda.synchronize()
    return eng


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    dev = torch.device("cuda:0")
    ops = O.load_operators(OPERATORS_NPZ)
    engines = {m: engine(m, ops, dev) for m in MODES}
    for eng in engines.values():                      # warm-up of every graph
        for _ in range(10):
            eng.device_step()
    torch.cuda.synchronize()
    times = {m: [] for m in MODES}
    for _ in range(a.blocks):
        for m in MODES:
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(a.iters):
                engines[m].device_step()
            e.record()
            e.synchronize()
            times[m].append(s.elapsed_time(e) * 1e3 / a.iters)
    kernels = {}
    for m in MODES:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                engines[m].device_step()
            torch.cuda.synchronize()
        kernels[m] = {e.key: {"count": e.count, "mean_us": e.device_time_total / e.count}
                      for e in prof.key_averages() if any(k in e.key for k in LOSS_KERNELS) and e.count}
    res = {"case": {"B": B, "vertices": ops[3][0], "dropout": O.DEFAULT_CONFIG["dropout"], "x_gt": "fp64", "graph": True},
           "card": card(),
           "step_us": {m: {"median": statistics.median(t), "min": min(t), "max": max(t), "blocks": t} for m, t in times.items()},
           "loss_kernels": kernels,
           "log_sigma_last_step": {m: float(engines[m].log_sigma) for m in MODES}}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "loss_sigma_cost.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "step_us"}, indent=1))
    print({m: round(statistics.median(t), 2) for m, t in times.items()}, "us per step (median of blocks)")


if __name__ == "__main__":
    main()
