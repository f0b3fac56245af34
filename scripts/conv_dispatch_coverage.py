"""Which Chebyshev-convolution kernel instantiations the polygon-order / filter-width tests reach.

Runs the kernel-level cases of tests/test_gpu_conv_orders.py (step path, row selection) and the K grids of
tests/test_gpu_operators.py (mesh-resident layers, streaming layer, fused recurrence, run-to-run determinism) once under
torch.profiler with CUDA activities, prints every tc_rowgemm_kernel / tc_wgrad_kernel / cheb_mesh_tc_* /
cheb_stream_tc_kernel instantiation, FFMA contraction / reduction / mesh-layer kernel and fold kernel it saw with its
launch count, and lists the instantiations compiled into libmvb_sm100a.so (cuobjdump -symbols | cu++filt) that never ran.

    python scripts/conv_dispatch_coverage.py [--out FILE] [--cuda-home /usr/local/cuda]

Exit status 0 whatever the coverage; 1 if a test failed."""
import argparse
import os
import re
import subprocess
import sys
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FAMILIES = ("tc_rowgemm_kernel", "tc_wgrad_kernel", "cheb_mesh_tc_fwd_kernel", "cheb_mesh_tc_bwd_kernel",
            "cheb_stream_tc_kernel", "contract_kernel", "wgrad_kernel", "wgrad_finalize_kernel", "cheb_layer_fwd_kernel",
            "cheb_layer_bwd_kernel", "fold_rows_fwd_kernel", "fold_rows_dx_kernel", "fold_rows_wgrad_kernel")
TESTS = ["tests/test_gpu_conv_orders.py::test_cheb_conv_orders_and_widths",
         "tests/test_gpu_conv_orders.py::test_cheb_conv_sel_orders",
         "tests/test_gpu_operators.py::test_cheb_layer",
         "tests/test_gpu_operators.py::test_cheb_stream",
         "tests/test_gpu_operators.py::test_fused_recurrence_is_bit_identical_on_other_operators",
         "tests/test_gpu_operators.py::test_bit_identical_run_to_run"]
_NAME = re.compile(r"mvb::(\w+)\s*(<[^>]*>)?")


def key(demangled: str):
    """'void mvb::tc_wgrad_kernel<(int)2, (int)4>(mvb::TcWgradArgs)' and the profiler's 'void mvb::tc_wgrad_kernel<2, 4>(...)'
    -> 'tc_wgrad_kernel<2,4>'; None for kernels outside FAMILIES"""
    m = _NAME.search(demangled)
    if not m or m.group(1) not in FAMILIES:
        return None
    args = m.group(2) or ""
    args = re.sub(r"\((?:int|bool|unsigned int)\)", "", args).replace("false", "0").replace("true", "1").replace(" ", "")
    return m.group(1) + args


def compiled(lib_path: str, cuda_home: str):
    syms = subprocess.run([os.path.join(cuda_home, "bin", "cuobjdump"), "-symbols", lib_path], check=True,
                          capture_output=True, text=True).stdout
    names = [ln.split()[-1] for ln in syms.splitlines() if "STT_FUNC" in ln and "STO_ENTRY" in ln]
    dem = subprocess.run([os.path.join(cuda_home, "bin", "cu++filt")], input="\n".join(names), check=True,
                         capture_output=True, text=True).stdout
    return sorted({k for k in (key(d) for d in dem.splitlines()) if k})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--cuda-home", default=os.environ.get("CUDA_HOME", "/usr/local/cuda"))
    args = ap.parse_args()
    import pytest
    import torch
    from torch.profiler import ProfilerActivity, profile
    import meshvae_b200
    lib_path = meshvae_b200._lib.lib._name
    built = compiled(lib_path, args.cuda_home)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc = pytest.main(["-q", "-m", "gpu", "-p", "no:cacheprovider", *[os.path.join(ROOT, t) for t in TESTS]])
        torch.cuda.synchronize()
    seen = Counter()
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            k = key(e.name)
            if k:
                seen[k] += 1
    lines = [f"library: {lib_path}", f"device: {torch.cuda.get_device_name(0)}", f"tests: exit status {int(rc)}", "",
             "launches per instantiation (seen under the profiler):"]
    lines += [f"  {n:8d}  {k}" for k, n in sorted(seen.items())]
    never = [k for k in built if k not in seen]
    lines += ["", f"compiled into the library: {len(built)}, ran: {len(built) - len(never)}, never ran: {len(never)}"]
    lines += [f"  never ran: {k}" for k in never]
    extra = sorted(k for k in seen if k not in built)
    if extra:
        lines += [f"  seen but not found among the library's symbols: {k}" for k in extra]
    report = "\n".join(lines)
    print(report)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(report + "\n")
    return 0 if int(rc) == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
