"""ctypes binding of libmvb_sm100a.so (the C ABI declared in include/mvb.h).

There is no CPU fallback: if the library is missing it is built with nvcc, and if that fails the
import raises.  Every compute call goes through `check()`, which raises MvbError with the
library's own message on a non-zero return code."""
import ctypes
import os
from ctypes import c_int, c_int64, c_uint64, c_float, c_void_p, c_size_t, c_char_p

from . import build as _build

_vp = c_void_p


class MvbError(RuntimeError):
    pass


def _load():
    if os.environ.get("MVB_LIB"):          # A/B runs against another build of the same sources (scripts/): never built on the fly
        return ctypes.CDLL(os.environ["MVB_LIB"])
    path = _build.LIB
    if not os.path.exists(path) or _build._stale():
        try:
            path = _build.build()
        except Exception as e:  # noqa: BLE001
            if not os.path.exists(_build.LIB):
                raise MvbError(f"libmvb_sm100a.so is missing and could not be built: {e}") from e
            path = _build.LIB
    return ctypes.CDLL(path)


lib = _load()

# name -> (restype, argtypes)   -- mirrors include/mvb.h one to one
SIGNATURES = {
    "mvb_version": (c_int, []),
    "mvb_sm_arch": (c_int, []),
    "mvb_last_error": (c_char_p, []),
    "mvb_device_cc": (c_int, []),
    "mvb_launch_count": (c_int64, []),
    "mvb_set_tensor_cores": (c_int, [c_int]),
    "mvb_tune": (c_int, [c_char_p]),
    "mvb_side_join": (c_int, [_vp]),
    "mvb_side_join_lane": (c_int, [_vp, c_int]),
    "mvb_stream_wait_external_event": (c_int, [_vp, _vp]),
    "mvb_csr_from_coo_host": (c_int, [c_int64, c_int64, c_int64, _vp, _vp, _vp, c_int, _vp, _vp, _vp]),
    "mvb_spmm": (c_int, [c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_float, c_float, c_int64, _vp]),
    "mvb_pool_fwd": (c_int, [c_int, c_int, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "mvb_pool_bwd": (c_int, [c_int, c_int, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "mvb_cheb_fwd": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp, c_int, _vp, _vp, _vp]),
    "mvb_cheb_bwd_uses_basis": (c_int, [c_int, c_int, c_int]),
    "mvb_cheb_bwd_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "mvb_cheb_bwd": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                             _vp, c_size_t, _vp]),
    "mvb_csr_values": (c_int, [c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvb_cheb_bwd_op_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "mvb_cheb_bwd_op": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _vp, _vp, _vp, _vp, c_size_t, _vp]),
    "mvb_vae_reparam_fwd": (c_int, [c_int64, _vp, _vp, _vp, _vp, _vp]),
    "mvb_vae_reparam_bwd": (c_int, [c_int64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvb_vae_loss_workspace_bytes": (c_size_t, [c_int, c_int]),
    "mvb_pack_vertex_major": (c_int, [c_int, c_int, c_int, c_int, _vp, _vp, _vp]),
    "mvb_vae_loss_fwd": (c_int, [c_int, c_int, c_int, c_int, c_int, _vp, c_int, _vp, c_int, _vp, _vp, _vp, _vp, c_float,
                                 _vp, _vp, _vp, _vp, _vp, _vp, c_size_t, _vp]),
    "mvb_vae_loss_bwd": (c_int, [c_int, c_int, c_int, c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvb_vae_loss_sigma_fwd": (c_int, [c_int] * 5 + [_vp, c_int, _vp, c_int] + [_vp] * 4 + [c_int] + [_vp] * 8 + [c_size_t, _vp]),
    "mvb_vae_loss_sigma_bwd": (c_int, [c_int] * 5 + [_vp] * 13),
    "mvb_iw_sample": (c_int, [c_int] * 4 + [_vp] * 7),
    "mvb_iw_log_weights_workspace_bytes": (c_size_t, [c_int] * 3),
    "mvb_iw_log_weights": (c_int, [c_int] * 4 + [_vp, c_int, _vp, c_int, _vp, _vp, c_int, c_int, _vp, _vp, c_size_t, _vp]),
    "mvb_iw_reduce": (c_int, [c_int, c_int] + [_vp] * 6),
    "mvb_kld_fwd": (c_int, [c_int, c_int, _vp, _vp, _vp, _vp]),
    "mvb_kld_bwd": (c_int, [c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvb_gaussian_nll_fwd": (c_int, [c_int64, _vp, _vp, c_int, c_float, _vp, _vp]),
    "mvb_gaussian_nll_bwd": (c_int, [c_int64, _vp, _vp, c_int, c_float, _vp, _vp, _vp]),
    "mvb_gaussian_nll_sigma_fwd": (c_int, [c_int64, _vp, _vp, c_int, _vp, c_int, _vp, _vp]),
    "mvb_gaussian_nll_sigma_workspace_bytes": (c_size_t, [c_int64]),
    "mvb_gaussian_nll_sigma_bwd": (c_int, [c_int64, _vp, _vp, c_int, _vp, c_int, _vp, _vp, _vp, _vp, c_size_t, _vp]),
    "mvb_cheb_sel_supported": (c_int, [c_int] * 6),
    "mvb_cheb_sel_fwd": (c_int, [c_int] * 6 + [_vp] * 6 + [c_int, c_int] + [_vp] * 4),
    "mvb_cheb_sel_bwd_workspace_bytes": (c_size_t, [c_int] * 3),
    "mvb_cheb_sel_bwd": (c_int, [c_int] * 5 + [_vp] * 4 + [c_int] + [_vp] * 4 + [c_size_t, _vp]),
    "mvb_cheb_layer_supported": (c_int, [c_int] * 9),
    "mvb_cheb_layer_fwd": (c_int, [c_int] * 5 + [_vp, _vp, _vp, c_int, c_int, _vp, _vp, _vp, c_int, c_int, _vp, _vp, _vp, _vp, c_int, _vp, _vp]),
    "mvb_cheb_layer_bwd_workspace_bytes": (c_size_t, [c_int] * 6),
    "mvb_cheb_layer_bwd": (c_int, [c_int] * 5 + [_vp] * 6 + [c_int, c_int] + [_vp] * 6 + [c_int, c_int] + [_vp] * 9 + [c_size_t, _vp]),
    "mvb_cheb_stream_supported": (c_int, [c_int] * 8),
    "mvb_cheb_stream_fwd_workspace_bytes": (c_size_t, [c_int] * 6),
    "mvb_cheb_stream_fwd": (c_int, [c_int] * 5 + [_vp, _vp, _vp, c_int, c_int, _vp, _vp, _vp, c_int, _vp, _vp, _vp, c_int, _vp, _vp,
                                    c_size_t, _vp]),
    "mvb_cheb_stream_bwd_workspace_bytes": (c_size_t, [c_int] * 6),
    "mvb_cheb_stream_bwd": (c_int, [c_int] * 5 + [_vp, _vp, _vp, c_int, c_int] + [_vp] * 6 + [c_int] + [_vp] * 8 + [c_size_t, _vp]),
    "mvb_linear_fwd": (c_int, [c_int, c_int, c_int, _vp, c_int, _vp, _vp, c_int, c_float, c_uint64, _vp, c_int64, _vp, c_int, _vp]),
    "mvb_linear_bwd": (c_int, [c_int, c_int, c_int, _vp, c_int, _vp, _vp, _vp, c_int, c_int, c_float, _vp, _vp, _vp, _vp]),
    "mvb_vae_heads_fwd": (c_int, [c_int, c_int, c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_float, c_uint64, _vp,
                                  c_int64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvb_vae_heads_bwd": (c_int, [c_int, c_int, c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_float, c_uint64, _vp,
                                  c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvb_recon_error_workspace_bytes": (c_size_t, [c_int, c_int]),
    "mvb_recon_error": (c_int, [c_int, c_int, c_int] + [_vp] * 7 + [c_int] + [_vp] * 4 + [_vp, c_size_t, _vp]),
    "mvb_epoch_meter_add": (c_int, [c_int, _vp, c_int, _vp, _vp, c_int, _vp, _vp, _vp, _vp]),
    "mvb_adam_step": (c_int, [c_int64, _vp, _vp, _vp, _vp, _vp, c_float, c_float, c_float, c_float, c_float, c_float,
                              _vp]),
    "mvb_adam_step_hp": (c_int, [c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvb_dp_max_world": (c_int, []),
    "mvb_dp_pad_bytes": (c_size_t, []),
    "mvb_dp_state_bytes": (c_size_t, []),
    "mvb_dp_begin": (c_int, [c_int, c_int, c_int, _vp, _vp, _vp]),
    "mvb_dp_reduce_adam": (c_int, [c_int, c_int, c_int, c_int64, c_int64, _vp, _vp, _vp, _vp, _vp, _vp, c_int, _vp, _vp, _vp, c_int, _vp]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here == header/library mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return (lib.mvb_last_error() or b"").decode()


def check(rc: int, what: str = ""):
    if rc != 0:
        raise MvbError(f"{what or 'mvb call'} failed (code {rc}): {last_error()}")


def tune(spec: str):
    """run-time switches (include/mvb.h: mvb_tune), e.g. tune("fused_recurrence=0;mesh_tc=1,2")"""
    check(lib.mvb_tune(spec.encode()), "mvb_tune")


if os.environ.get("MVB_TUNE"):          # A/B runs of the switches (tests, bench, scripts alike)
    tune(os.environ["MVB_TUNE"])


# Deferred side chains (include/mvb.h: mvb_side_join): while on, the tensors a chain still reads are parked here until
# the join, so that the caching allocator cannot hand their memory to a later kernel of the main stream
_deferred = {"on": False, "keep": []}


def defer_side_chains(on: bool):
    _deferred["on"] = bool(on)
    tune(f"defer_wgrad={1 if on else 0}")


def side_join(lane=None):
    """make the current stream wait for the pending side chains (of one lane, or of all: the parked tensors are then
    released)"""
    if lane is None:
        check(lib.mvb_side_join(stream_ptr()), "mvb_side_join")
        _deferred["keep"].clear()
    else:
        check(lib.mvb_side_join_lane(stream_ptr(), int(lane)), "mvb_side_join_lane")


def ptr(t):
    """device (or host) pointer of a tensor, None -> NULL"""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
