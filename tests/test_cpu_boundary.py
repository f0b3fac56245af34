"""CPU-only checks of the boundary: the C-ABI library loads and exports every symbol include/mvb.h
declares, the host COO->CSR routine is right, the module mirrors expose the reference's API surface
and state-dict contract, and the product path fails loudly (no CPU fallback)."""
import copy
import os
import re
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from tests.helpers import ROOT, OPERATORS_NPZ
import meshvae_b200 as mvb
from meshvae_b200 import _lib
from meshvae_b200.operators import csr_from_coo_host
from oracle import mesh_vae_oracle as O


def test_library_exports_every_header_symbol():
    hdr = open(os.path.join(ROOT, "include", "mvb.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(mvb_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(_lib.lib, name), name
    assert _lib.lib.mvb_version() == 100
    assert _lib.lib.mvb_sm_arch() == 100


def test_tune_takes_only_the_implementation_switches():
    """mvb_tune only sets host-side switches (no GPU needed).  The kernel variants and tuning knobs that were measured and
    not adopted are gone: their keys are rejected like any unknown key, so none of them comes back unnoticed."""
    retired = ["tc_tma", "wgrad_perm", "background_div", "tc_tuning", "tc_balance", "layer_tuning", "spmm_shape",
               "spmm_mode", "stream_nt", "conv_lanes", "overlap", "mesh_dbg"]
    try:
        for key in retired:
            with pytest.raises(_lib.MvbError, match="unknown key"):
                _lib.tune(f"{key}=1")
        for spec in ("mesh_tc=1,2", "fused_recurrence=0", "stream_tc=1,8", "pdl=0", "defer_wgrad=1"):
            _lib.tune(spec)
    finally:
        _lib.tune("mesh_tc=1,0;fused_recurrence=1;stream_tc=0,16;pdl=1;defer_wgrad=0")


def test_only_sm100a_code_is_embedded():
    import subprocess
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "--list-elf", mvb.build.LIB], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


def test_csr_from_coo_host_matches_scipy_and_keeps_order():
    d = np.load(OPERATORS_NPZ)
    for name in ("A0", "D1", "U0", "U3", "A4"):
        r, c, v = d[f"{name}_row"], d[f"{name}_col"], d[f"{name}_val"]
        m, n = (int(s) for s in d[f"{name}_shape"])
        for transpose in (False, True):
            rp, ci, vv = csr_from_coo_host(r, c, v, m, n, transpose)
            ref = sp.coo_matrix((v, (r, c)), shape=(m, n))
            ref = (ref.T if transpose else ref).tocsr()
            got = sp.csr_matrix((vv, ci, rp), shape=ref.shape)
            assert abs(got - ref).max() == 0
            assert rp[-1] == len(v)
    # stable: duplicates and explicit zeros are kept, in COO order inside a row
    r = np.array([1, 0, 1, 1]); c = np.array([2, 0, 2, 0]); v = np.array([1.0, 0.0, 3.0, 4.0], dtype=np.float32)
    rp, ci, vv = csr_from_coo_host(r, c, v, 3, 3)
    assert rp.tolist() == [0, 1, 4, 4] and ci.tolist() == [0, 2, 2, 0] and vv.tolist() == [0.0, 1.0, 3.0, 4.0]
    # coarse operator on a bigger tensor: trailing empty rows (quirk 1)
    rp, ci, vv = csr_from_coo_host(d["A4_row"], d["A4_col"], d["A4_val"], 4998, 4998)
    assert rp.shape == (4999,) and rp[20] == rp[-1] == 96
    with pytest.raises(_lib.MvbError):
        csr_from_coo_host(np.array([5]), np.array([0]), np.array([1.0]), 3, 3)


def test_state_dict_contract_and_api_surface():
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    cfg = copy.deepcopy(O.DEFAULT_CONFIG)
    net = mvb.cheb_VAE(3, cfg, D, U, A, nn_, model=cfg["model"])
    ref = O.OracleChebVAE(3, copy.deepcopy(O.DEFAULT_CONFIG), D, U, A, nn_)
    assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == \
           {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert "cheb_dec.4.bias" not in net.state_dict() and net.cheb_dec[-1].bias is None
    assert sum(p.numel() for p in net.parameters()) == 712642
    for attr in ("encoder", "decoder", "classifier", "sample", "reparameterize", "loss_function", "forward",
                 "A_edge_index", "A_norm", "pool", "cheb", "cheb_dec"):
        assert hasattr(net, attr)
    conv = mvb.ChebConv_batch(3, 16, 6)
    assert tuple(conv.weight.shape) == (6, 3, 16) and tuple(conv.bias.shape) == (16,)
    assert conv.in_channels == 3 and conv.out_channels == 16 and conv.normalization is None
    ei, nrm = mvb.ChebConv_batch.norm(A[2]._indices(), nn_[2])
    ei_o, nrm_o = O.cheb_norm(A[2]._indices(), nn_[2])
    assert torch.equal(ei, ei_o) and torch.equal(nrm, nrm_o)
    cfg2 = copy.deepcopy(O.DEFAULT_CONFIG)
    gcn = mvb.cheb_GCN(6, cfg2, D, U, A, nn_)
    assert cfg2["num_conv_filters"][0] == 6                       # in-place mutation kept (quirk 9)
    ref_g = O.OracleChebGCN(6, copy.deepcopy(O.DEFAULT_CONFIG), D, U, A, nn_)
    assert {k: tuple(v.shape) for k, v in gcn.state_dict().items()} == \
           {k: tuple(v.shape) for k, v in ref_g.state_dict().items()}


def test_no_cpu_fallback():
    A, D, U, nn_ = O.load_operators(OPERATORS_NPZ)
    conv = mvb.ChebConv_batch(3, 16, 6)
    ei, nrm = mvb.ChebConv_batch.norm(A[4]._indices(), nn_[4])
    with pytest.raises(mvb.MvbError):
        conv(torch.randn(2, 20, 3), ei, nrm)
    with pytest.raises(mvb.MvbError):
        mvb.SurfacePool()(torch.randn(2, 79, 8), D[3])
    with pytest.raises(mvb.MvbError):
        mvb.logpdf.KLD(torch.randn(2, 16), torch.randn(2, 16))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mesh-vae_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f
