"""Time mvb_vae_heads_fwd / mvb_vae_heads_bwd (the fused VAE heads) with CUDA events at the shapes of
tests/test_gpu_heads_shapes.py, dropout 0.2, all five upstream gradients present.  Each timing is a loop of --iters
back-to-back calls on one stream between two events (warmed up first), reported as microseconds per call; the
inputs stay in L2 between calls, as they do inside a training step.  Prints one JSON object (with the card's name
and power limit) and, with --out, writes it there too.

    python scripts/heads_shapes.py [--iters 200] [--out heads_shapes.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = [(64, 512, 16, 2), (256, 512, 16, 2),                                   # the default config: one-launch kernels
          (1, 512, 16, 2), (257, 512, 16, 2), (512, 512, 16, 2), (1000, 512, 16, 2),
          (64, 512, 48, 2), (64, 512, 64, 2), (300, 1024, 128, 2),
          (64, 1562, 16, 2), (64, 4096, 256, 3), (7, 100, 5, 10)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        out = "unknown"
    return {"name": name, "power_limit": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--p", type=float, default=0.2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import meshvae_b200
    L = meshvae_b200._lib
    assert torch.cuda.is_available() and L.lib.mvb_device_cc() == 100, "needs a B200 (sm_100a)"
    dev = torch.device("cuda:0")
    rows = []
    for b, hd, z, c in SHAPES:
        g = torch.Generator(device="cpu").manual_seed(1)
        t = lambda *s: torch.randn(*s, generator=g).to(dev)      # noqa: E731
        h, eps = t(b, hd), t(b, z)
        y = torch.nn.functional.one_hot(torch.randint(0, c, (b,), generator=g), c).to(dev)
        wc, bc, wm, bm, wv, bv = t(c, hd) / hd ** 0.5, t(c), t(z, c + hd) / (c + hd) ** 0.5, t(z), t(z, c + hd) / (c + hd) ** 0.5, t(z)
        y_hat, mu, lv, zz, zcat = (torch.empty(b, n, device=dev) for n in (c, z, z, z, c + z))
        ups = [t(b, c), t(b, z), t(b, z), t(b, z), t(b, c + z)]
        g_h = torch.empty_like(h)
        dws = [torch.empty_like(w) for w in (wc, bc, wm, bm, wv, bv)]
        P = L.ptr

        def fwd():
            L.check(L.lib.mvb_vae_heads_fwd(b, hd, z, c, P(h), P(y), P(eps), P(wc), P(bc), P(wm), P(bm), P(wv), P(bv), args.p, 5, None,
                                            1, P(y_hat), P(mu), P(lv), P(zz), P(zcat), L.stream_ptr()), "fwd")

        def bwd():
            L.check(L.lib.mvb_vae_heads_bwd(b, hd, z, c, P(h), P(y), P(eps), P(wc), P(wm), P(wv), P(y_hat), P(lv), args.p, 5, None, 1,
                                            *[P(u) for u in ups], P(g_h), *[P(d) for d in dws], L.stream_ptr()), "bwd")

        row = {"B": b, "H": hd, "Z": z, "C": c}
        for name, fn in (("fwd_us", fwd), ("bwd_us", bwd)):
            for _ in range(10):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            row[name] = round(e0.elapsed_time(e1) * 1e3 / args.iters, 2)
        rows.append(row)
    res = {"what": "mvb_vae_heads_fwd / _bwd, us per call (CUDA events, back-to-back calls, L2-warm)", "p_drop": args.p,
           "iters": args.iters, "card": card(), "rows": rows}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
