"""ctypes binding of ``csrc/librgcn_b200.so`` (the C ABI declared in ``include/rgcn_b200.h``).

There is NO CPU fallback: if the library is missing or the device is not a B200-class GPU the
product path raises.  (The CPU restatement lives in ``oracle/`` and is test infrastructure.)
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "librgcn_b200.so")

ABI_VERSION = 8          # RGCN_B200_ABI_VERSION of include/rgcn_b200.h

_lock = threading.Lock()
_lib = None

p = C.c_void_p
i32, i64, sz = C.c_int32, C.c_int64, C.c_size_t


class CsrStruct(C.Structure):
    """Mirror of ``rgcn_csr_t`` (include/rgcn_b200.h)."""
    _fields_ = [("rowptr", p), ("idx", p), ("w", p), ("n_rows", i64), ("E", i64), ("R", i32),
                ("n_hubs", i32), ("n_chunks", i32), ("hub_threshold", i32), ("hub_keys", p),
                ("hub_chunk_ptr", p), ("chunk_table", p), ("row_order", p), ("order_chunk_rows", i64)]


PCSR = C.POINTER(CsrStruct)
f32, u32, u64 = C.c_float, C.c_uint32, C.c_uint64


class LayerFwdArgs(C.Structure):
    """Mirror of ``rgcn_layer_fwd_args`` (include/rgcn_b200.h)."""
    _fields_ = [("csr", PCSR), ("x_src", p), ("ld_x_src", i64), ("x_root", p), ("ld_x_root", i64),
                ("d_in", i32), ("d_out", i32), ("relu", i32), ("mode", i32),
                ("weight", p), ("root", p), ("bias", p),
                ("dropout_p", f32), ("dropout_seed", u32), ("dropout_counter", p),
                ("A_hi", p), ("A_lo", p), ("lda", i64), ("out", p), ("ldo", i64),
                ("peer_out_host", p), ("n_peer", i32), ("peer_row0", i64), ("peer_ld", i64),
                ("agg_workspace", p), ("agg_workspace_bytes", sz), ("gemm_workspace", p), ("gemm_workspace_bytes", sz),
                ("w_planes", p), ("w_planes_bytes", sz), ("pipeline", i32),
                ("x_bf16", p), ("ld_x_bf16", i64), ("out_bf16", p), ("ld_out_bf16", i64),
                ("rows", p), ("n_list", i64), ("slot", p), ("dropout_row0", i64)]


class MaskedPlanesOut(C.Structure):
    """Mirror of ``rgcn_masked_planes_out`` (include/rgcn_b200.h)."""
    _fields_ = [("mask", p), ("ld_mask", i64), ("scale", f32), ("hi", p), ("lo", p), ("ldp", i64), ("colsum_partial", p)]


class LayerBwdArgs(C.Structure):
    """Mirror of ``rgcn_layer_bwd_args`` (include/rgcn_b200.h)."""
    _fields_ = [("csr_t", PCSR), ("g_out", p), ("ld_g_out", i64), ("relu_mask", p), ("ld_mask", i64), ("mask_scale", f32),
                ("n_dst", i64), ("d_in", i32), ("d_out", i32), ("mode", i32), ("add_root_term", i32),
                ("weight", p), ("root", p), ("A_hi", p), ("A_lo", p), ("lda", i64),
                ("G_hi", p), ("G_lo", p), ("ldg", i64), ("colsum_partial", p), ("gA", p), ("ld_gA", i64),
                ("g_x", p), ("ld_g_x", i64), ("g_weight", p), ("g_root", p), ("g_bias", p),
                ("agg_workspace", p), ("agg_workspace_bytes", sz), ("gemm_workspace", p), ("gemm_workspace_bytes", sz),
                ("rows", p), ("n_list", i64), ("slot", p), ("Ac_hi", p), ("Ac_lo", p), ("ldac", i64),
                ("next_G", C.POINTER(MaskedPlanesOut)), ("g_ready", i32), ("n_colsum_ready", i32), ("slot_ready", i32),
                ("w_planes", p), ("a_compact", i32), ("csr_fwd", PCSR), ("src_flag", p)]

ADAM_MAX_SEGMENTS = 64   # RGCN_ADAM_MAX_SEGMENTS


class AdamSegment(C.Structure):
    """Mirror of ``rgcn_adam_segment`` (include/rgcn_b200.h)."""
    _fields_ = [("param", p), ("grad", p), ("exp_avg", p), ("exp_avg_sq", p), ("step", p), ("numel", i64),
                ("group", i32)]


class AdamHparams(C.Structure):
    """Mirror of ``rgcn_adam_hparams`` (include/rgcn_b200.h)."""
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("weight_decay", C.c_double), ("decoupled_weight_decay", i32)]


class LinkBatchArgs(C.Structure):
    """Mirror of ``rgcn_link_batch_args`` (include/rgcn_b200.h)."""
    _fields_ = [("pos_head", p), ("pos_tail", p), ("pos_rel", p), ("n_pos", i64), ("num_neg", i32), ("num_rel", i32),
                ("num_nodes", i64), ("seed", u32), ("max_tries", i32), ("counter", p),
                ("heads", p), ("tails", p), ("rels", p), ("labels", p), ("head_prob", p),
                ("filter_keys", p), ("filter_tails", p), ("n_filter", i64),
                ("head_offsets", p), ("head_nodes", p), ("tail_offsets", p), ("tail_nodes", p),
                ("exhausted", p), ("ticket", p)]

# name -> (restype, argtypes); must list every symbol of include/rgcn_b200.h
PROTOTYPES = {
    "rgcn_abi_version": (C.c_int, []),
    "rgcn_last_error": (C.c_int, [C.c_char_p, sz]),
    "rgcn_check_device": (C.c_int, []),
    "rgcn_launch_count": (i64, []),
    "rgcn_probe_gather_sink_floats": (i64, [i32]),
    "rgcn_probe_gather": (C.c_int, [p, i64, i64, i32, p, i64, i32, p, p]),
    "rgcn_csr_build_workspace_bytes": (sz, [i64, i64, i64, i32]),
    "rgcn_csr_build": (C.c_int, [p, p, p, i64, i64, i64, i32, p, p, p, p, p, p, p, p, p, p, sz, p]),
    "rgcn_hub_plan_workspace_bytes": (sz, [i64, i64]),
    "rgcn_hub_plan": (C.c_int, [p, i64, i32, p, p, i64, C.POINTER(i32), C.POINTER(i32), p, sz, p]),
    "rgcn_hub_chunk_table": (C.c_int, [p, p, i32, i32, p, p]),
    "rgcn_aggregate_workspace_bytes": (sz, [PCSR, i32]),
    "rgcn_aggregate_blocks": (i64, [PCSR, i32]),
    "rgcn_aggregate_fwd": (C.c_int, [PCSR, p, i64, i32, p, i32, p, p, i64, i32, p, i64, p, p, i64, p, sz, p]),
    "rgcn_reduce_partials": (C.c_int, [p, i64, i32, p, p]),
    "rgcn_aggregate_bwd": (C.c_int, [PCSR, p, i64, i32, p, i64, p, i64, C.POINTER(MaskedPlanesOut), p, sz, p]),
    "rgcn_aggregate_row_blocks": (i64, [PCSR, i32]),
    "rgcn_aggregate_fwd_rows": (C.c_int, [PCSR, p, i64, i32, p, p, i64, i32, p, i64, i64, i64, i32, p, sz, p]),
    "rgcn_weight_planes_bytes": (sz, [i32, i32]),
    "rgcn_prepare_weights": (C.c_int, [p, i32, p, i32, i32, i32, p, p, p]),
    "rgcn_transform_fwd_w": (C.c_int, [p, p, i64, i32, p, p, i32, i64, i32, p, i64, i32, C.c_float, C.c_uint32, p, i64,
                                       p, i32, i64, i64, p, i64, p]),
    "rgcn_aggregate_fwd_bf16": (C.c_int, [PCSR, p, i64, i32, p, i64, p, i64, i64, i64, i32, p, sz, p]),
    "rgcn_rows_list_build": (C.c_int, [p, p, i64, i64, p, p, p]),
    "rgcn_aggregate_fwd_list": (C.c_int, [PCSR, p, i64, i32, p, p, i64, i32, p, i64, p, i64, p, p, sz, p]),
    "rgcn_aggregate_fwd_bf16_list": (C.c_int, [PCSR, p, i64, i32, p, i64, p, i64, p, i64, p, p, sz, p]),
    "rgcn_transform_fwd_w_rows": (C.c_int, [p, p, i64, i32, p, p, i32, i64, i32, p, i64, i32, p, i64, p, p, i32, i64, i64, p]),
    "rgcn_transform_dgrad_w": (C.c_int, [p, p, i64, i32, p, i32, i64, p, i64, i32, p]),
    "rgcn_aggregate_bwd_rows": (C.c_int, [PCSR, p, i64, i32, p, i32, p, i64, p, i64, C.POINTER(MaskedPlanesOut), p, sz, p]),
    "rgcn_aggregate_bwd_rows_marked": (C.c_int, [PCSR, PCSR, p, i64, p, p, i64, i32, p, i32, p, i64, p, i64, p, sz, p]),
    "rgcn_rows_compact_size": (i64, [i64]),
    "rgcn_rows_compact_blocks": (i64, [i64]),
    "rgcn_rows_compact": (C.c_int, [p, i64, i64, p, p, i64, i32, p, p, i64, p, p, i64, i32, p, p, i64, p, p, i32, i32, p]),
    "rgcn_split_planes_blocks": (i64, [i64, i32]),
    "rgcn_split_planes": (C.c_int, [p, i64, p, i64, i64, i32, p, p, i64, p, C.c_float, p, i64, p]),
    "rgcn_transform_workspace_bytes": (sz, [i64, i32, i32]),
    "rgcn_transform_fwd": (C.c_int, [p, p, i64, i32, i32, p, p, p, i32, i64, i32, p, i64, i32, C.c_float, C.c_uint32, p,
                                     p, i32, i64, i64, p, sz, p]),
    "rgcn_basis_combine": (C.c_int, [p, p, i32, i32, i64, p, p]),
    "rgcn_basis_combine_bwd": (C.c_int, [p, p, p, i32, i32, i64, p, p, p]),
    "rgcn_layer_fwd": (C.c_int, [C.POINTER(LayerFwdArgs), p]),
    "rgcn_layer_bwd": (C.c_int, [C.POINTER(LayerBwdArgs), p]),
    "rgcn_p2p_pull_rows": (C.c_int, [p, i32, i64, i64, p, i64, i64, i32, p, i64, p]),
    "rgcn_p2p_push_rows": (C.c_int, [p, i64, i64, i32, p, i32, i64, i64, p]),
    "rgcn_p2p_reduce_split": (C.c_int, [p, i32, i64, i64, p, i64, p, i64, C.c_float, i64, i32, p, i64, p, p, i64, p, p]),
    "rgcn_p2p_allreduce_flag_bytes": (sz, []),
    "rgcn_p2p_allreduce": (C.c_int, [p, p, p, i32, i32, i64, C.c_float, p, p, p]),
    "rgcn_transform_dgrad": (C.c_int, [p, p, i64, i32, p, i32, p, i32, i64, p, i64, i32, p, sz, p]),
    "rgcn_transform_wgrad": (C.c_int, [p, p, i64, i32, i32, p, p, i64, i32, i64, p, i32, p, p, p, i32, p, sz, p]),
    "rgcn_distmult_fwd": (C.c_int, [p, i64, p, i64, p, p, p, p, p, p, i64, i32, p, p]),
    "rgcn_distmult_bwd": (C.c_int, [p, i64, p, i64, p, p, p, p, p, p, p, i64, i32, p, i64, p, i64, p, p, p]),
    "rgcn_rows_prepare": (C.c_int, [p, i64, p, i64, i32, p, p, i32, p, i64, p]),
    "rgcn_allpairs_scores": (C.c_int, [p, i64, i64, p, i64, p, i64, i32, C.c_float, C.c_float, p, i64, p]),
    "rgcn_allpairs_rank": (C.c_int, [p, i64, i64, p, i64, p, i64, i32, p, p, p, p, p]),
    "rgcn_rank_count": (C.c_int, [p, i64, i64, i64, p, p, p, p, p]),
    "rgcn_scores_diag_w": (C.c_int, [p, p, i64, i32, p, i64, p, p]),
    "rgcn_scores_rank_w": (C.c_int, [p, p, i64, i32, p, i64, i64, p, p, p, p, p]),
    "rgcn_scores_topk_slots": (i32, [i64, i64]),
    "rgcn_scores_topk_w": (C.c_int, [p, p, i64, i32, p, i64, i64, i32, C.c_float, C.c_float, p, p, p, i32, p, p, p]),
    "rgcn_rank_excl_correct": (C.c_int, [p, i64, p, i64, p, i64, p, i32, i64, i64, p, p, p, p, p, p, p, p]),
    "rgcn_scores_rank_excl_w": (C.c_int, [p, p, i64, i32, p, i64, i64, p, p, p, p, p, p, p, p]),
    "rgcn_scores_topk_excl_w": (C.c_int, [p, p, i64, i32, p, i64, i64, i32, C.c_float, C.c_float, p, p, p, i32, p, p,
                                          p, p, p, p]),
    "rgcn_bce_logits_fwd": (C.c_int, [p, p, i64, p, p, p]),
    "rgcn_bce_logits_bwd": (C.c_int, [p, p, i64, p, p, p]),
    "rgcn_link_batch": (C.c_int, [p, p, p, i64, i32, i64, u32, p, p, p, p, p, p]),
    "rgcn_link_batch_ex": (C.c_int, [C.POINTER(LinkBatchArgs), p]),
    "rgcn_link_loss_workspace_bytes": (sz, [i64]),
    "rgcn_link_loss_fwd": (C.c_int, [p, i64, p, p, p, p, p, i64, i32, C.c_float, u32, p, p, p, p, p, i64, i32, p, p, sz, p]),
    "rgcn_link_loss_bwd": (C.c_int, [p, i64, p, p, p, p, p, p, p, p, i64, i32, C.c_float, u32, p, p, i64, p, i32, i64, p]),
    "rgcn_link_bwd_rows_workspace_bytes": (sz, [i64, i32, i32]),
    "rgcn_link_loss_bwd_rows": (C.c_int, [p, i64, p, p, p, p, p, p, p, p, i64, i32, C.c_float, u32, p, i64, i32, p, i64, p,
                                          p, p, p, i32, p, sz, p]),
    "rgcn_check_pairs": (C.c_int, [p, p, p, i64, i64, i32, p, p]),
    "rgcn_adam_workspace_bytes": (sz, [i64, i32]),
    "rgcn_adam_step": (C.c_int, [C.POINTER(AdamSegment), i32, p, i32, C.c_float, p, p, sz, p]),
}


class RGCNLibraryError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RGCNLibraryError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:  # pragma: no cover
                raise RGCNLibraryError(f"{LIB_PATH} does not export {name}; rebuild the library") from e
            fn.restype = res
            fn.argtypes = args
        if lib.rgcn_abi_version() != ABI_VERSION:
            raise RGCNLibraryError("ABI version mismatch between the Python host side and librgcn_b200.so")
        _lib = lib
    return _lib


def last_error() -> str:
    buf = C.create_string_buffer(512)
    load().rgcn_last_error(buf, 512)
    return buf.value.decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RGCNLibraryError(f"{what or 'librgcn_b200'} failed (code {rc}): {last_error()}")
