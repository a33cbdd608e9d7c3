"""ctypes binding of liblcrec_b200.so (the C ABI declared in include/lcrec_b200.h).

No CPU fallback: if the library is missing or the device is not an sm_100 GPU, every operator
raises.  Build the library with ``python -m lcrec_b200.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblcrec_b200.so")

i32, i64, f64 = C.c_int32, C.c_int64, C.c_double
vp = C.c_void_p
pp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); mirrors include/lcrec_b200.h one to one
SIGNATURES = {
    "lcrec_version": (C.c_int, []),
    "lcrec_strerror": (C.c_char_p, [C.c_int]),
    "lcrec_last_error": (C.c_char_p, []),
    "lcrec_device_check": (C.c_int, []),
    "lcrec_launch_count": (i64, []),
    "lcrec_mlp_create": (C.c_int, [C.c_int, C.POINTER(i32), pp, pp, C.c_int, vp, pp]),
    "lcrec_mlp_update": (C.c_int, [vp, pp, pp, vp]),
    "lcrec_mlp_destroy": (C.c_int, [vp]),
    "lcrec_mlp_workspace_bytes": (i64, [vp, i64]),
    "lcrec_mlp_forward": (C.c_int, [vp, vp, i64, vp, pp, vp, i64, vp]),
    "lcrec_mlp_forward_ex": (C.c_int, [vp, vp, C.c_int, i64, vp, pp, vp, i64, vp]),
    "lcrec_mlp_set_acc_chunk": (C.c_int, [vp, C.c_int]),
    "lcrec_mlp_set_variant": (C.c_int, [vp, C.c_int]),
    "lcrec_mlp_set_engine": (C.c_int, [vp, C.c_int]),
    "lcrec_mlp_set_trace": (C.c_int, [vp, vp]),
    "lcrec_pair_set_cluster_cap": (C.c_int, [C.c_int]),
    "lcrec_mlp_in_dim": (C.c_int, [vp]),
    "lcrec_mlp_out_dim": (C.c_int, [vp]),
    "lcrec_linear_workspace_bytes": (i64, [i64, C.c_int, C.c_int]),
    "lcrec_linear_forward": (C.c_int, [vp, i64, C.c_int, vp, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, i64, vp]),
    "lcrec_rq_quantize": (C.c_int, [vp, i64, C.c_int, C.c_int, pp, C.POINTER(i32), C.c_int, C.c_int, vp, vp, vp, vp, vp]),
    "lcrec_vq_distances": (C.c_int, [vp, i64, C.c_int, vp, C.c_int, vp, vp]),
    "lcrec_sinkhorn_workspace_bytes": (i64, [i64, C.c_int]),
    "lcrec_sinkhorn_dense": (C.c_int, [vp, i64, C.c_int, f64, C.c_int, vp, vp, vp, vp, i64, vp]),
    "lcrec_sinkhorn_dense_argmax_workspace_bytes": (i64, [i64, C.c_int]),
    "lcrec_sinkhorn_dense_argmax": (C.c_int, [vp, i64, C.c_int, f64, C.c_int, vp, vp, vp, i64, vp]),
    "lcrec_sinkhorn_set_dense_cluster": (C.c_int, [C.c_int]),
    "lcrec_sinkhorn_set_wide": (C.c_int, [C.c_int]),
    "lcrec_sinkhorn_dist_symmetric_bytes": (i64, [C.c_int]),
    "lcrec_sinkhorn_dense_dist": (C.c_int, [vp, i64, i64, C.c_int, f64, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.c_uint64,
                                            vp, i64, vp]),
    "lcrec_center_distances": (C.c_int, [vp, i64, C.c_int, vp, vp, vp, i64, vp]),
    "lcrec_sinkhorn_groups_workspace_bytes": (i64, [i64, C.c_int]),
    "lcrec_sinkhorn_groups": (C.c_int, [vp, C.c_int, vp, C.c_int, vp, vp, vp, i64, i64, f64, C.c_int, vp, C.c_int,
                                        C.c_int, vp, vp, i64, vp]),
    "lcrec_sinkhorn_groups_part": (C.c_int, [vp, C.c_int, vp, C.c_int, vp, vp, vp, i64, i64, f64, C.c_int, vp, C.c_int,
                                             C.c_int, C.c_int, C.c_int, vp, vp, i64, vp]),
    "lcrec_linear_backward_workspace_bytes": (i64, [i64, C.c_int, C.c_int]),
    "lcrec_linear_backward": (C.c_int, [vp, vp, vp, vp, i64, C.c_int, C.c_int, vp, vp, vp, vp, i64, vp]),
    "lcrec_mlp_backward_workspace_bytes": (i64, [vp, i64]),
    "lcrec_mlp_backward": (C.c_int, [vp, pp, vp, pp, vp, i64, vp, pp, pp, vp, i64, vp]),
    "lcrec_rq_set_tc_mode": (C.c_int, [C.c_int]),
    "lcrec_sinkhorn_groups_ex": (C.c_int, [vp, C.c_int, vp, C.c_int, vp, vp, vp, i64, i64, i64, f64, C.c_int, vp, C.c_int,
                                           C.c_int, C.c_int, C.c_int, vp, vp, i64, vp]),
    "lcrec_sinkhorn_set_mode": (C.c_int, [C.c_int]),
    "lcrec_collisions_workspace_bytes": (i64, [i64]),
    "lcrec_collisions": (C.c_int, [vp, i64, C.c_int, C.POINTER(i32), vp, vp, vp, vp, i64, vp]),
    "lcrec_sort_codes": (C.c_int, [vp, i64, C.c_int, C.POINTER(i32), vp, vp, vp, i64, vp]),
    "lcrec_prefix_segments": (C.c_int, [vp, i64, C.c_int, C.POINTER(i32), vp, vp, vp, vp, i64, vp]),
    "lcrec_segment_collisions_workspace_bytes": (i64, [i64]),
    "lcrec_collisions_in_segments": (C.c_int, [vp, i64, C.c_int, C.c_int, vp, vp, vp, i64, vp, vp, vp, vp, i64, vp]),
    "lcrec_collisions_in_segments_active": (C.c_int, [vp, i64, C.c_int, C.c_int, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp,
                                                      i64, vp]),
    "lcrec_profile_enable": (C.c_int, [C.c_int]),
    "lcrec_profile_collect": (C.c_int, [C.POINTER(C.c_double), C.POINTER(i64)]),
    "lcrec_indexer_create": (C.c_int, [vp, C.c_int, C.c_int, pp, C.POINTER(i32), f64, C.c_int, i64, i64, pp]),
    "lcrec_indexer_destroy": (C.c_int, [vp]),
    "lcrec_indexer_run_device": (C.c_int, [vp, vp, i64, C.c_int, vp, C.POINTER(i64), vp]),
    "lcrec_indexer_run_host": (C.c_int, [vp, vp, i64, C.c_int, vp, C.POINTER(i64), vp]),
    "lcrec_indexer_pass0": (C.c_int, [vp, vp, i64, i64, vp]),
    "lcrec_indexer_run_device_ex": (C.c_int, [vp, vp, C.c_int, i64, C.c_int, vp, C.POINTER(i64), vp]),
    "lcrec_indexer_run_host_ex": (C.c_int, [vp, vp, C.c_int, i64, C.c_int, vp, C.POINTER(i64), vp]),
    "lcrec_indexer_pass0_ex": (C.c_int, [vp, vp, C.c_int, i64, i64, vp]),
    "lcrec_indexer_pass0_host_ex": (C.c_int, [vp, vp, C.c_int, i64, i64, i64, vp]),
    "lcrec_indexer_round": (C.c_int, [vp, i64, C.POINTER(i64), vp]),
    "lcrec_indexer_resolve": (C.c_int, [vp, vp, vp, i64, C.c_int, C.POINTER(i64), vp]),
    "lcrec_indexer_set_segments": (C.c_int, [C.c_int]),
    "lcrec_indexer_set_speculative": (C.c_int, [C.c_int]),
    "lcrec_ema_update": (C.c_int, [vp, vp, i64, C.c_int, C.c_int, f64, f64, vp, vp, vp, vp]),
    "lcrec_codebook_usage": (C.c_int, [vp, C.c_int, f64, f64, vp, vp, vp]),
    "lcrec_ema_dist_symmetric_bytes": (i64, [i64, C.c_int]),
    "lcrec_ema_update_dist": (C.c_int, [vp, vp, i64, i64, C.c_int, C.c_int, f64, f64, vp, vp, vp, vp, vp, vp, vp, C.c_int,
                                        C.c_int, i64, C.c_uint64, vp]),
    "lcrec_masked_mean_pool_workspace_bytes": (i64, [i64, i64, C.c_int]),
    "lcrec_masked_mean_pool": (C.c_int, [vp, C.c_int, vp, i64, i64, C.c_int, vp, i64, C.c_int, f64, vp, i64, vp]),
    "lcrec_kmeans_workspace_bytes": (i64, [i64, C.c_int, C.c_int]),
    "lcrec_kmeans_center": (C.c_int, [vp, i64, C.c_int, vp, vp, C.POINTER(f64), vp, i64, vp]),
    "lcrec_kmeans_lloyd": (C.c_int, [vp, i64, C.c_int, vp, C.c_int, C.c_int, f64, vp, vp, C.POINTER(f64), C.POINTER(C.c_int),
                                     vp, i64, vp]),
    "lcrec_rq_train_forward": (C.c_int, [vp, vp, i64, C.c_int, C.c_int, pp, vp, vp, vp, vp, vp]),
    "lcrec_rq_train_backward": (C.c_int, [vp, vp, i64, C.c_int, C.c_int, C.POINTER(i32), vp, vp, f64, vp, pp, vp]),
    "lcrec_adam_workspace_bytes": (i64, [C.c_int, C.POINTER(i64)]),
    "lcrec_adam_clip_step": (C.c_int, [C.c_int, pp, pp, pp, pp, C.POINTER(i64), f64, f64, f64, f64, f64, C.c_int, i64, f64,
                                       C.c_int, vp, vp, i64, vp]),
    "lcrec_adam_hyper": (C.c_int, [f64, f64, f64, f64, i64, C.POINTER(C.c_float)]),
    "lcrec_adam_clip_step_dev": (C.c_int, [C.c_int, pp, pp, pp, pp, C.POINTER(i64), vp, f64, f64, f64, f64, C.c_int, f64,
                                           C.c_int, vp, vp, i64, vp]),
    "lcrec_simple_opt_clip_step": (C.c_int, [C.c_int, C.c_int, pp, pp, pp, C.POINTER(i64), f64, f64, f64, f64, f64, C.c_int, vp, vp, i64, vp]),
    "lcrec_bn_sums_elems": (i64, [C.c_int]),
    "lcrec_bn_splits": (C.c_int, [i64, C.c_int]),
    "lcrec_bn_forward_reduce": (C.c_int, [vp, i64, C.c_int, vp, vp]),
    "lcrec_bn_forward_apply": (C.c_int, [vp, vp, C.c_int, i64, i64, C.c_int, vp, vp, f64, f64, C.c_int, vp, vp, vp, vp, vp, vp]),
    "lcrec_bn_backward_reduce": (C.c_int, [vp, vp, vp, C.c_int, vp, vp, i64, C.c_int, vp, vp]),
    "lcrec_bn_backward_apply": (C.c_int, [vp, vp, vp, C.c_int, vp, C.c_int, i64, i64, C.c_int, vp, vp, vp, vp, vp, vp, vp]),
    "lcrec_recon_loss_workspace_bytes": (i64, [i64]),
    "lcrec_recon_loss": (C.c_int, [vp, vp, i64, C.c_int, vp, vp, i64, vp]),
    "lcrec_recon_loss_backward": (C.c_int, [vp, vp, i64, C.c_int, vp, vp, vp]),
    "lcrec_index_json_workspace_bytes": (i64, [i64]),
    "lcrec_index_json": (C.c_int, [vp, i64, C.c_int, vp, i64, vp, vp, i64, vp]),
    "lcrec_index_json_ex": (C.c_int, [vp, i64, C.c_int, i64, C.c_int, vp, i64, vp, vp, i64, vp]),
    "lcrec_fp64_peak_probe": (C.c_int, [C.POINTER(f64), vp, i64, vp]),
    "lcrec_ddiv_probe": (C.c_int, [vp, vp, i64, vp, vp]),
    "lcrec_sinkhorn_set_col": (C.c_int, [C.c_int]),
    "lcrec_exchange_record_bytes": (i64, [C.c_int, C.c_int]),
    "lcrec_exchange_slab_bytes": (i64, [i64, C.c_int, C.c_int]),
    "lcrec_exchange_workspace_bytes": (i64, [i64, C.c_int]),
    "lcrec_exchange_pack": (C.c_int, [vp, vp, i64, C.c_int, C.c_int, C.POINTER(i32), C.c_int, i64, vp, vp, vp, vp, i64, vp]),
    "lcrec_exchange_unpack": (C.c_int, [vp, C.c_int, i64, C.c_int, C.c_int, vp, vp, i64, vp]),
    "lcrec_exchange_pack_last": (C.c_int, [vp, C.c_int, vp, C.c_int, i64, C.c_int, vp, i64, vp]),
    "lcrec_exchange_scatter_last": (C.c_int, [vp, vp, i64, C.c_int, vp, vp]),
    "lcrec_kmeanspp_workspace_bytes": (i64, [i64, C.c_int]),
    "lcrec_kmeanspp_seed": (C.c_int, [vp, i64, C.c_int, C.c_int, i64, vp, C.c_int, vp, vp, vp, i64, vp]),
    "lcrec_indexer_codes": (vp, [vp]),
    "lcrec_indexer_resid": (vp, [vp]),
}

_lib = None


class LcrecError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"lcrec_b200 error {code}: {message}")
        self.code = code


def load() -> C.CDLL:
    """Load the C-ABI library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built "
            "(python -m lcrec_b200.build).  lcrec_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        lib = load()
        detail = lib.lcrec_last_error().decode(errors="replace")
        kind = lib.lcrec_strerror(rc).decode()
        raise LcrecError(rc, f"{kind}: {detail}")


def ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))(*[C.c_void_p(p) for p in ptrs])
    return arr


def i32_array(vals):
    return (i32 * len(vals))(*[int(v) for v in vals])
