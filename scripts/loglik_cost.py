"""Cost of the importance-weighted log-likelihood estimate, cheb_VAE.log_likelihood (default config, B = 64 meshes, fp64
ground truth, the constant decoder sigma), at S = 1, 16 and 128 samples per mesh with a sample_chunk that keeps the
decoder batch near 2048 meshes:

  * the time per call and the meshes x samples per second, and the time of the decoder alone on the same batches, CUDA
    events around blocks of calls after a warm-up, the three S and the two kinds alternating block by block;
  * in a separate pass under torch.profiler, with programmatic dependent launch off (a kernel launched early would count
    its wait for the previous one), the device time of the three new kernels (iw_sample_kernel, the SSE partial kernel
    vae_rec_partial_kernel and iw_log_weights_finalize_kernel of mvb_iw_log_weights, iw_reduce_kernel) against that of
    all the call's kernels and of the decoder alone.

    python scripts/loglik_cost.py --out DIR [--blocks 10 --iters 5]

Writes DIR/loglik_cost.json with the card's name and power limit read in the same run."""
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
import torch.nn.functional as F  # noqa: E402

import meshvae_b200 as mvb  # noqa: E402
from oracle import mesh_vae_oracle as O  # noqa: E402
from tests.helpers import OPERATORS_NPZ, seeded_state_dict  # noqa: E402

B = 64
SAMPLES = (1, 16, 128)
DECODER_BATCH = 2048
IW_KERNELS = ("iw_sample_kernel", "vae_rec_partial_kernel", "iw_log_weights_finalize_kernel", "iw_reduce_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def pdl_at_start():
    """the PDL switch as the process started: on, unless MVB_TUNE (applied when the package is imported) turned it off"""
    on = 1
    for item in os.environ.get("MVB_TUNE", "").split(";"):
        key, _, val = item.partition("=")
        if key.strip() == "pdl" and val.strip():
            on = int(val.split(",")[0])
    return on


def chunk_for(s):
    return max(1, min(s, DECODER_BATCH // B))


def device_times(fn, reps):
    """kernel name -> (launches, total device us) over `reps` calls of fn under torch.profiler"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    return {e.key: (e.count, e.self_device_time_total) for e in prof.key_averages() if e.count and e.self_device_time_total > 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--iters", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    dev = torch.device("cuda:0")
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    net = mvb.cheb_VAE(3, cfg, [d.to(dev) for d in D], [u.to(dev) for u in U], [a_.to(dev) for a_ in A], nn_)
    net.load_state_dict(seeded_state_dict(net, 7))
    net = net.to(dev).eval()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, nn_[0], 3, generator=g).to(dev)
    x_gt = x.double()
    y = F.one_hot(torch.arange(B) % 2, 2).to(dev)
    gen = torch.Generator(device=dev).manual_seed(0)

    def call(s):
        return net.log_likelihood(x, x_gt, y, s, chunk_for(s), gen)

    def decode(s):
        """the decoder on the batches of call(s): (S / chunk) decodes of B * chunk meshes"""
        c = chunk_for(s)
        zcat = torch.cat([y.float(), torch.zeros(B, net.z, device=dev)], 1).repeat_interleave(c, 0)
        with torch.no_grad():
            for s0 in range(0, s, c):
                net.decoder(zcat[:B * min(c, s - s0)])
                net._recon_padded = None

    for s in SAMPLES:                                   # warm-up of every shape
        for _ in range(3):
            call(s)
            decode(s)
    torch.cuda.synchronize()
    times = {(k, s): [] for k in ("call", "decoder") for s in SAMPLES}
    for _ in range(a.blocks):
        for s in SAMPLES:
            for k, fn in (("call", call), ("decoder", decode)):
                st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                st.record()
                for _ in range(a.iters):
                    fn(s)
                en.record()
                en.synchronize()
                times[(k, s)].append(st.elapsed_time(en) / a.iters)

    profile = {}
    mvb._lib.tune("pdl=0")
    try:
        for s in SAMPLES:
            c = chunk_for(s)
            reps = 5
            k_call = device_times(lambda: call(s), reps)
            k_dec = device_times(lambda: decode(s), reps)
            iw = {k: {"launches": n, "us_per_call": t / reps} for k, (n, t) in k_call.items() if any(w in k for w in IW_KERNELS)}
            iw_us = sum(v["us_per_call"] for v in iw.values())
            call_us = sum(t for _, t in k_call.values()) / reps
            dec_us = sum(t for _, t in k_dec.values()) / reps
            profile[s] = {"sample_chunk": c, "decoder_batch": B * c, "iw_kernels": iw, "iw_kernels_us": iw_us,
                          "all_kernels_us": call_us, "decoder_alone_us": dec_us,
                          "iw_share_of_call": iw_us / call_us, "iw_vs_decoder": iw_us / dec_us}
    finally:
        mvb._lib.tune(f"pdl={pdl_at_start()}")

    res = {"case": {"B": B, "vertices": nn_[0], "x_gt": "fp64", "sigma": "fixed", "decoder_batch_target": DECODER_BATCH,
                    "blocks": a.blocks, "iters": a.iters},
           "card": card(),
           "call_ms": {s: {"median": statistics.median(t), "min": min(t), "max": max(t), "sample_chunk": chunk_for(s),
                           "mesh_samples_per_s": B * s / (statistics.median(t) * 1e-3),
                           "decoder_alone_median": statistics.median(times[("decoder", s)]), "blocks": t,
                           "decoder_blocks": times[("decoder", s)]}
                       for (k, s), t in times.items() if k == "call"},
           "profile": profile}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "loglik_cost.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))
    for s in SAMPLES:
        c, p = res["call_ms"][s], profile[s]
        print(f"S={s:4d} chunk={c['sample_chunk']:3d}: {c['median']:.3f} ms/call ({c['min']:.3f}-{c['max']:.3f}), "
              f"{c['mesh_samples_per_s']:.0f} mesh-samples/s, decoder alone {c['decoder_alone_median']:.3f} ms; profiled "
              f"(PDL off): new kernels {p['iw_kernels_us']:.1f} us of {p['all_kernels_us']:.1f} us kernel time "
              f"({100 * p['iw_share_of_call']:.2f} %), decoder alone {p['decoder_alone_us']:.1f} us; "
              + ", ".join(f"{k.split('(')[0].split(' ')[-1]} {v['us_per_call']:.1f}" for k, v in p['iw_kernels'].items()))


if __name__ == "__main__":
    main()
