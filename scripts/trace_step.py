"""In-graph kernel timeline of one training step (torch.profiler / CUPTI on a graph replay): true
durations with warm caches and concurrency, plus the idle gaps between kernels on the critical path.
  python scripts/trace_step.py [--batch 64] > gpurun_out/trace.txt"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bench  # noqa: E402
from torch.profiler import profile, ProfilerActivity  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=64)
a = ap.parse_args()
# under torchrun (WORLD_SIZE > 1): the data-parallel step of rank 0
world = int(os.environ.get("WORLD_SIZE", "1"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
dev = torch.device("cuda", local)
mvb, net, A, nn_ = bench.build_model(dev)
# switches for A/B runs: MVB_TUNE="fused_recurrence=0;mesh_tc=0" (include/mvb.h: mvb_tune)
if os.environ.get("MVB_TUNE"):
    mvb._lib.tune(os.environ["MVB_TUNE"])
from meshvae_b200.engine import TrainEngine  # noqa: E402
eng = TrainEngine(net, a.batch)
eng.capture(warmup=3)
g = torch.Generator().manual_seed(1)
x = torch.randn(a.batch, nn_[0], 3, generator=g).pin_memory()
eng.step(x, x.double().pin_memory(), torch.randint(0, 2, (a.batch,), generator=g))
for _ in range(5):
    eng.device_step()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
    for _ in range(3):
        eng.device_step()
    torch.cuda.synchronize()
evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
evs.sort(key=lambda e: e.time_range.start)
# split into replays by the adam kernel
steps, cur = [], []
_seen_reduce = False
for e in evs:
    cur.append(e)
    last = "dp_reduce_adam" if world > 1 and eng.peer is not None else "adam"
    if (last == "adam" and ("adam_kernel" in e.name or "adam_hp_kernel" in e.name)) or (
            last != "adam" and last in e.name and (not eng.split or _seen_reduce)):
        _seen_reduce = False
        steps.append(cur)
        cur = []
    elif "dp_reduce_adam" in e.name:
        _seen_reduce = True
if world > 1 and int(os.environ.get("RANK", "0")) != 0:
    torch.cuda.synchronize()
    dist.barrier()
    sys.exit(0)
st = steps[1] if len(steps) > 1 else steps[0]
t0 = st[0].time_range.start
end_prev = t0
tot_busy = 0.0
print(f"# {len(st)} kernels in the replay; columns: start_us dur_us gap_before_us name")
agg = {}
for e in st:
    s, d = e.time_range.start - t0, e.time_range.end - e.time_range.start
    gap = e.time_range.start - end_prev
    end_prev = max(end_prev, e.time_range.end)
    name = e.name.replace("void ", "")[:70]
    print(f"{s:9.1f} {d:7.1f} {gap:7.1f}  {name}")
    k = name.split("(")[0][:60]
    agg.setdefault(k, [0, 0.0])
    agg[k][0] += 1
    agg[k][1] += d
print(f"# step span {end_prev - t0:.1f} us")
print("# per-kernel totals (in-graph durations)")
for k, (n, d) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    print(f"# {d:8.1f} us {n:3d}  {k}")
if world > 1:
    torch.cuda.synchronize()
    dist.barrier()
