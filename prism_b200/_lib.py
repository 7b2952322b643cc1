"""ctypes binding of libprism_b200.so -- mirrors include/prism_b200.h one-to-one.

There is no CPU fallback: if the CUDA library cannot be found or built, importing a
product code path raises.  (The CPU oracle lives under oracle/ and is never imported
from this package.)
"""
import ctypes as C
import os

from . import build as _build

_LIB = None


class PbError(RuntimeError):
    pass


class pb_per_state(C.Structure):
    _fields_ = [
        ("len", C.c_longlong), ("seq", C.c_longlong), ("max_priority", C.c_float), ("p_sum", C.c_float),
        ("p_min", C.c_float), ("status", C.c_int), ("batch_max", C.c_float), ("owned_lo", C.c_int),
        ("owned_n", C.c_int), ("pad", C.c_int * 5),
    ]


class pb_tree(C.Structure):
    _fields_ = [
        ("sum", C.c_void_p), ("min", C.c_void_p), ("owner", C.c_void_p), ("counters", C.c_void_p),
        ("state", C.c_void_p),
        ("capacity", C.c_longlong), ("size", C.c_longlong), ("alpha", C.c_float), ("eps_f32", C.c_float),
        ("eps_f64", C.c_double), ("weight_eps_in_denominator", C.c_int), ("default_priority_fp64", C.c_int),
    ]


class pb_store(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p), ("aux_obs", C.c_void_p), ("action", C.c_void_p), ("reward", C.c_void_p),
        ("done", C.c_void_p), ("trunc", C.c_void_p), ("slot_seq", C.c_void_p), ("next_link", C.c_void_p),
        ("prev_link", C.c_void_p), ("size", C.c_longlong), ("aux_size", C.c_longlong), ("obs_elems", C.c_int),
        ("obs_dtype", C.c_int), ("obs_scale", C.c_int), ("frame_stack", C.c_int), ("n_step", C.c_int),
        ("pad", C.c_int), ("gamma", C.c_double),
    ]


# numpy view of pb_step_meta (64 bytes per staged step)
STEP_META_DTYPE = [("seq", "<i8"), ("prev_link", "<i8"), ("next_link", "<i8"), ("aux_row", "<i8"),
                   ("patch_slot", "<i8"), ("patch_val", "<i8"), ("reward", "<f4"), ("action", "<i4"),
                   ("done", "u1"), ("trunc", "u1"), ("pad", "u1", (6,))]

assert C.sizeof(pb_per_state) == 64

PB_PEER_MAX = 8


class pb_peer_group(C.Structure):
    _fields_ = [("world", C.c_int), ("rank", C.c_int),
                ("grad", C.c_void_p * PB_PEER_MAX), ("reduced", C.c_void_p * PB_PEER_MAX),
                ("flags", C.c_void_p * PB_PEER_MAX), ("norm_parts", C.c_void_p * PB_PEER_MAX),
                ("state", C.c_void_p * PB_PEER_MAX), ("epoch", C.c_void_p), ("status", C.c_void_p),
                ("timeout_ns", C.c_ulonglong), ("grad_stride", C.c_longlong)]


_P = C.c_void_p
_LL = C.c_longlong
_I = C.c_int
_F = C.c_float
_TREE = C.POINTER(pb_tree)
_STORE = C.POINTER(pb_store)
_PEER = C.POINTER(pb_peer_group)

# name -> argtypes (every function returns int unless listed in _RESTYPES)
SIGNATURES = {
    "pb_abi_version": [],
    "pb_error_string": [_I],
    "pb_launch_count": [],
    "pb_event_create": [C.POINTER(C.c_void_p)],
    "pb_event_destroy": [_P],
    "pb_event_record": [_P, _P],
    "pb_event_synchronize": [_P],
    "pb_stream_wait_event": [_P, _P],
    "pb_copy_h2d_async": [_P, _P, _LL, _P],
    "pb_staged_copy_submit": [_P, _P, _P, _P, _LL, _P, _P],
    "pb_copy_d2h_async": [_P, _P, _LL, _P],
    "pb_copy_d2d_async": [_P, _P, _LL, _P],
    "pb_tree_layout": [_LL, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong),
                       C.POINTER(C.c_longlong), C.POINTER(C.c_int)],
    "pb_tree_init": [_TREE, _P],
    "pb_tree_export": [_TREE, _P, _P, _P],
    "pb_tree_trace": [_I, _P, _I],
    "pb_gemm_trace": [_I, _P, _I],
    "pb_tree_sample_batches": [_TREE, _LL, _LL, _P, _I, _F, _P, _P, _P, _P],
    "pb_tree_build": [_TREE, _P, _LL, _P],
    "pb_tree_stats": [_TREE, _P],
    "pb_tree_set_leaves": [_TREE, _LL, _P, _P, _I, _P],
    "pb_tree_update_priority": [_TREE, _LL, _P, _P, _I, _P],
    "pb_tree_extend": [_TREE, _LL, _P, _P],
    "pb_tree_scan": [_TREE, _LL, _P, _P, _P],
    "pb_tree_sample": [_TREE, _LL, _P, _I, _F, _P, _P, _P, _P],
    "pb_tree_sample_global": [_TREE, _I, _I, _P, _LL, _P, _F, _P, _P, _P, _P],
    "pb_store_extend_plan": [_LL, _LL, _I, _LL, _LL, _P, _P, _P, _P, _P, _P],
    "pb_store_scatter": [_STORE, _LL, _P, _P, _P, _P],
    "pb_select_copy_f64": [_P, _P, _P, _P, _LL, _LL, _P],
    "pb_store_scatter_dbuf": [_STORE, _LL, _P, _P, _P, _P, _P, _P, _P, _P],
    "pb_store_gather": [_STORE, _LL, _P, _P, _P, _P, _P, _P, _P, _P],
    "pb_store_nstep": [_STORE, _LL, _P, _P, _P, _P, _P, _P, _P],
    "pb_iqn_cos_basis": [_LL, _I, _P, _P, _P],
    "pb_iqn_qh_loss": [_I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _F, _F, _P, _F, _P, _P, _P],
    "pb_ens_q_loss": [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _F, _P, _F, _P, _P, _P],
    "pb_ens_q_loss_total": [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _F, _P, _F, _P, _P, _P, _F, _P, _P, _P, _P, _P],
    "pb_ids_select": [_I, _I, _I, _I, _P, _P, _F, _F, _F, _P, _P, _P],
    "pb_iqn_qh_loss_sq": [_I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _F, _F, _P, _F, _P, _P, _P, _I],
    "pb_ens_q_loss_sq": [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _F, _P, _F, _P, _P, _P, _I],
    "pb_ens_q_loss_total_sq": [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _F, _P, _F, _P, _P, _P, _F, _P, _P, _P, _P, _P,
                               _I],
    "pb_ids_select_sq": [_I, _I, _I, _I, _P, _P, _F, _F, _F, _P, _P, _P, _I],
    "pb_value_squash": [_LL, _P, _P, _I, _I, _P],
    "pb_greedy_select": [_I, _I, _I, _P, _P, _P],
    "pb_adam_clip_step": [_LL, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _P],
    "pb_adam_fused_max_n": [],
    "pb_adam_fused_step": [_I, _P, _F, _LL, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _P],
    "pb_pack_grads": [_I, _P, _F, _P, _P, _P, _P, _P],
    "pb_pack_grads_parity": [_I, _P, _F, _P, _P, _LL, _P, _P, _P, _P],
    "pb_grad_sumsq": [_LL, _P, _P, _P, _P, _P],
    "pb_adam_clip_apply": [_LL, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _I, _P, _P],
    "pb_opt_fused_max_n": [_I],
    "pb_opt_fused_step": [_I, _I, _P, _F, _LL, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _P],
    "pb_opt_clip_apply": [_I, _LL, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _I, _P, _P],
    "pb_loss_combine": [_I, _P, _P, _P, _F, _P, _P, _P, _P],
    "pb_conv3x3_relu_supported": [_I, _I, _I, _I],
    "pb_conv3x3_relu_fwd": [_I, _I, _I, _I, _I, _P, _P, _P, _P, _P],
    "pb_conv3x3_relu_bwd_groups": [_I],
    "pb_conv3x3_relu_bwd": [_I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P],
    "pb_linear_fwd": [_I, _I, _I, _I, _P, _LL, _P, _P, _I, _P, _P],
    "pb_peer_alloc": [_LL, C.POINTER(C.c_void_p)],
    "pb_peer_free": [_P],
    "pb_peer_preload": [],
    "pb_optimizer_preload": [],
    "pb_peer_export": [_P, _P],
    "pb_peer_open": [_P, C.POINTER(C.c_void_p)],
    "pb_peer_close": [_P],
    "pb_peer_barrier": [_PEER, _P],
    "pb_peer_state_allgather": [_PEER, _P, _P, _P],
    "pb_peer_slice": [_LL, _I],
    "pb_peer_reduce_scatter": [_PEER, _LL, _P, _P, _P],
    "pb_peer_pull_sum": [_PEER, _LL, _P, _P, C.POINTER(C.c_int), _P],
    "pb_peer_adam": [_PEER, _LL, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _P],
    "pb_peer_allreduce_adam_max_n": [],
    "pb_peer_allreduce_adam": [_PEER, _LL, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _P],
    "pb_peer_allreduce_opt_max_n": [_I],
    "pb_peer_allreduce_opt": [_I, _PEER, _LL, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _P],
    "pb_peer_opt": [_I, _PEER, _LL, _P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _P],
    "pb_peer_state_put": [_PEER, _P, _P],
    "pb_peer_trace": [_I, _P, _I],
    "pb_tree_sample_global_peer": [_TREE, _PEER, _LL, _P, _F, _P, _P, _P, _P],
    "pb_uniform_init": [_P, _LL, _LL, _I, _P],
    "pb_uniform_extend": [_P, _LL, _LL, _P],
    "pb_uniform_sample": [_P, _LL, _P, _I, _P, _P, _P],
    "pb_uniform_sample_global": [_P, _I, _I, _P, _LL, _P, _P, _P, _P, _P],
    "pb_uniform_sample_global_peer": [_P, _PEER, _LL, _P, _P, _P, _P, _P],
    "pb_layer_norm_supported": [_LL, _I],
    "pb_layer_norm_bwd_blocks": [_LL, _I],
    "pb_layer_norm_fwd": [_LL, _I, _F, _P, _P, _P, _P, _P, _P, _P],
    "pb_layer_norm_bwd": [_LL, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "pb_layer_norm_grouped_fwd": [_I, _LL, _LL, _I, _F, _P, _P, _P, _P, _P, _P, _P],
    "pb_layer_norm_grouped_bwd_blocks": [_I, _LL, _I],
    "pb_layer_norm_grouped_bwd": [_I, _LL, _LL, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "pb_narrow_linear_supported": [_LL, _I, _I],
    "pb_narrow_linear_bwd_blocks": [_LL],
    "pb_narrow_linear_fwd": [_I, _LL, _I, _I, _P, _LL, _P, _P, _P, _P],
    "pb_narrow_linear_bwd": [_I, _LL, _I, _I, _P, _LL, _P, _P, _P, _P, _P, _P, _P],
    "pb_narrow_linear_bwd_reduce": [_I, _LL, _I, _I, _P, _P, _P, _P],
    "pb_sum_heads": [_I, _LL, _P, _P, _P],
    "pb_iqn_draw_cos_basis": [_LL, _I, _P, _P, _P, _P],
    "pb_relu_bwd_bias_strips": [_LL],
    "pb_relu_bwd_bias": [_I, _LL, _I, _P, _P, _P, _P, _P, _P],
    "pb_theil_chunks": [_LL],
    "pb_theil_fwd": [_I, _I, _I, _P, _P, _P, _P, _P],
    "pb_theil_bwd": [_I, _I, _I, _P, _P, _P, _P, _P],
    "pb_iqn_phi_bwd": [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P],
    "pb_tc_gemm_supported": [_I, _I, _I, _LL, _LL, _LL],
    "pb_tc_gemm": [_I, _I, _I, _I, _I, _P, _I, _LL, _LL, _P, _I, _LL, _LL, _P, _LL, _I, _P, _I, _LL, _P, _LL, _LL, _P, _LL, _I, _P],
    "pb_linear_fwd_tc_supported": [_I, _I, _I],
    "pb_linear_fwd_tc": [_I, _I, _I, _I, _P, _LL, _P, _P, _I, _P, _P],
    "pb_linear_bwd_input": [_I, _I, _I, _I, _P, _P, _P, _I, _P, _P],
    "pb_linear_bwd_weight": [_I, _I, _I, _I, _P, _P, _P, _LL, _P, _P, _P],
    "pb_stamp_time": [_P, _P],
    "pb_store_stage_block": [_LL, _LL, _I, _LL, _LL, _LL, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P],
    "pb_wire_unpack_numbers": [_P, _LL, _P, _LL, _P],
    "pb_wire_array_header": [_LL, _P, _P],
    "pb_wire_pack_numbers": [_P, _I, _LL, _P, _LL, _P],
    "pb_wire_index_timesteps": [_P, _LL, _LL, _P, _P],
}
_RESTYPES = {"pb_error_string": C.c_char_p, "pb_launch_count": C.c_longlong, "pb_peer_slice": C.c_longlong,
             "pb_peer_allreduce_adam_max_n": C.c_longlong, "pb_adam_fused_max_n": C.c_longlong,
             "pb_opt_fused_max_n": C.c_longlong, "pb_peer_allreduce_opt_max_n": C.c_longlong}

# update rules of the pb_opt_* / pb_peer_*_opt entries (include/prism_b200.h)
PB_OPT_ADAM, PB_OPT_RMSPROP, PB_OPT_RMSPROP_CENTERED, PB_OPT_SGD = 0, 1, 2, 3
# value squashing kinds of the *_sq entries and pb_value_squash, and the obs_look_further epsilon (include/prism_b200.h)
PB_SQUASH_NONE, PB_SQUASH_OBS_LOOK_FURTHER, PB_SQUASH_SYMLOG = 0, 1, 2
PB_SQUASH_OLF_EPS = 1e-2

PB_E_POOL = -4
ABI_VERSION = 2


def lib_path():
    return _build.LIB_PATH


def load():
    """Load (building first if needed) libprism_b200.so.  Raises if unavailable."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.build()
    if not os.path.exists(path):
        raise PbError("libprism_b200.so missing at %s and could not be built" % path)
    lib = C.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = ABI drift, fail loudly
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    if lib.pb_abi_version() != ABI_VERSION:
        raise PbError("libprism_b200.so ABI version mismatch")
    _LIB = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().pb_error_string(rc).decode()
        raise PbError("%s failed: %s (code %d)" % (what or "libprism_b200 call", msg, rc))


def ptr(t):
    """Raw device/host pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def cur_stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def launch_count():
    return int(load().pb_launch_count())


def require_cuda(t, name="tensor"):
    if not t.is_cuda:
        raise PbError("%s must live on a CUDA device: libprism_b200 has no CPU path" % name)
