"""ctypes binding of libsegger_b200.so (the C ABI declared in include/segger_b200.h).

The product path has NO fallback: if the shared library is missing or a call fails this module
raises.  torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_LIB_PATH = Path(__file__).resolve().parent / "csrc" / "libsegger_b200.so"
_lib = None

ACT_NONE, ACT_GELU, ACT_SILU = 0, 1, 2

c_i64, c_i32, c_f32, c_u64, c_sz, c_vp, c_int = (
    C.c_int64, C.c_int32, C.c_float, C.c_uint64, C.c_size_t, C.c_void_p, C.c_int)


class KnnPlan(C.Structure):
    _fields_ = [("xmin", C.c_double), ("ymin", C.c_double), ("cell", C.c_double),
                ("nx", c_i64), ("ny", c_i64), ("n_points", c_i64), ("n_query", c_i64),
                ("k", c_int), ("max_dist", C.c_double)]


# name -> (restype, argtypes); mirrors include/segger_b200.h one to one
_PROTOS = {
    "sgb_version": (c_int, []),
    "sgb_last_error": (C.c_char_p, []),
    "sgb_csr_workspace_bytes": (c_sz, [c_i64]),
    "sgb_csr_build": (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp,
                              c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_gatv2_fwd": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_int,
                              c_int, c_f32, c_f32, c_u64, c_vp, c_int, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "sgb_gatv2_alpha": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_int, c_int,
                                c_f32, c_vp, c_vp, c_vp, c_vp]),
    "sgb_gatv2_bwd_workspace_bytes": (c_sz, [c_i64, c_i64, c_int, c_int]),
    "sgb_gatv2_bwd": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_vp,
                              c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_f32,
                              c_f32, c_u64, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp,
                              c_sz, c_vp]),
    "sgb_dropout_mask": (c_int, [c_u64, c_i64, c_int, c_f32, c_vp, c_vp]),
    "sgb_linear_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "sgb_linear_fwd": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_vp,
                               c_i64, c_int, c_vp, c_sz, c_vp]),
    "sgb_linear_fwd_gather": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_int, c_vp,
                                      c_i64, c_int, c_vp, c_sz, c_vp]),
    "sgb_linear_dgrad": (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int,
                                 c_vp, c_i64, c_vp, c_sz, c_vp]),
    "sgb_linear_wgrad_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64]),
    "sgb_linear_wgrad": (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_int, c_vp,
                                 c_sz, c_vp]),
    "sgb_act_fwd": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_vp]),
    "sgb_act_bwd": (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_vp]),
    "sgb_embedding_fwd": (c_int, [c_vp, c_i64, c_int, c_vp, c_int, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_vp]),
    "sgb_embedding_bwd_workspace_bytes": (c_sz, [c_i64, c_int, c_i64]),
    "sgb_embedding_bwd": (c_int, [c_vp, c_i64, c_vp, c_int, c_i64, c_int, c_i64, c_vp, c_int, c_vp, c_vp, c_sz,
                                  c_vp]),
    "sgb_posfreq_workspace_bytes": (c_sz, [c_i64]),
    "sgb_posfreq_fwd": (c_int, [c_vp, c_i64, c_vp, c_int, c_i64, c_int, c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "sgb_poscheb_fwd": (c_int, [c_vp, c_i64, c_vp, c_int, c_i64, c_int, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "sgb_index_strictly_increasing": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp]),
    "sgb_rows_add": (c_int, [c_vp, c_i64, c_i64, c_vp, c_int, c_i64, c_int, c_vp, c_i64, c_vp]),
    "sgb_triplet_sample": (c_int, [c_vp, c_i64, c_int, c_int] + [c_vp] * 16 + [c_vp]),
    "sgb_loss_workspace_bytes": (c_sz, [c_i64]),
    "sgb_triplet_margin_fwd": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_f32, c_f32,
                                       c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_triplet_self_bwd_supported": (c_int, [c_int]),
    "sgb_triplet_self_bwd": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_int, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp,
                                     c_vp, c_vp, c_vp, c_i64, c_vp]),
    "sgb_triplet_margin_bwd": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_f32, c_f32,
                                       c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "sgb_pair_loss_fwd": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_int, c_int, c_f32, c_vp, c_vp, c_vp,
                                  c_sz, c_vp]),
    "sgb_pair_loss_bwd": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_int, c_int, c_f32, c_vp, c_vp, c_vp,
                                  c_vp, c_vp]),
    "sgb_pip_workspace_bytes": (c_sz, [c_i64, c_i64, c_int, c_int]),
    "sgb_pip_count": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_i64, C.c_double, C.c_double, C.c_double, c_int, c_int, c_vp,
                              c_vp, c_sz, c_vp]),
    "sgb_pip_fill_scratch_bytes": (c_sz, [c_i64]),
    "sgb_pip_fill": (c_int, [c_vp, c_vp, c_i64, c_i64, C.c_double, C.c_double, C.c_double, c_int, c_int, c_i64, c_vp, c_i64,
                             c_vp, c_sz, c_vp, c_sz, c_vp]),
    "sgb_polygon_props": (c_int, [c_vp, c_vp, c_i64, C.c_double, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "sgb_pip_buffered_count": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_i64, C.c_double, C.c_double, C.c_double, c_int,
                                       c_int, c_vp, c_vp, c_sz, c_vp]),
    "sgb_pip_buffered_fill": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, C.c_double, C.c_double, C.c_double, c_int, c_int, c_i64,
                                      c_vp, c_i64, c_vp, c_sz, c_vp, c_sz, c_vp]),
    "sgb_polygon_props_multi": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, C.c_double, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "sgb_pip_multi_count": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, C.c_double, C.c_double, C.c_double,
                                    c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "sgb_pip_multi_fill": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, C.c_double, C.c_double, C.c_double, c_int, c_int,
                                   c_i64, c_vp, c_i64, c_vp, c_sz, c_vp, c_sz, c_vp]),
    "sgb_gatv2_quad_supported": (c_int, [c_int, c_int]),
    "sgb_l2norm_fwd": (c_int, [c_vp, c_i64, c_i64, c_int, c_f32, c_vp, c_i64, c_vp, c_vp]),
    "sgb_l2norm_bwd": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_f32, c_vp, c_i64, c_vp]),
    "sgb_score_argmax": (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_i64, c_i64, c_f32, c_vp,
                                 c_int, c_f32, c_vp, c_vp, c_vp, c_vp]),
    "sgb_knn2d_plan": (c_int, [c_vp, c_int, c_i64, c_vp, c_i64, c_int, C.c_double, C.POINTER(KnnPlan), c_vp, c_vp]),
    "sgb_knn2d_workspace_bytes": (c_sz, [C.POINTER(KnnPlan)]),
    "sgb_knn2d": (c_int, [C.POINTER(KnnPlan), c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_knn2d_ring_plan": (c_int, [c_vp, c_int, c_i64, c_vp, c_i64, c_int, C.c_double, C.POINTER(KnnPlan), c_vp, c_vp]),
    "sgb_knn2d_ring_workspace_bytes": (c_sz, [C.POINTER(KnnPlan)]),
    "sgb_knn2d_ring": (c_int, [C.POINTER(KnnPlan), c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_knn_count_valid": (c_int, [c_vp, c_i64, c_int, c_i64, c_vp, c_vp]),
    "sgb_knn_coo_workspace_bytes": (c_sz, [c_i64]),
    "sgb_knn_count_edges": (c_int, [c_vp, c_i64, c_vp, C.POINTER(c_i64), c_vp, c_sz, c_vp]),
    "sgb_knn_table_to_coo": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_i64, c_i64, c_vp, c_vp]),
    "sgb_select_workspace_bytes": (c_sz, [c_i64]),
    "sgb_mask_select": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_box_select": (c_int, [c_vp, c_int, c_i64, C.POINTER(C.c_double), C.POINTER(C.c_double), c_vp, c_vp, c_vp, c_vp,
                               c_vp, c_sz, c_vp]),
    "sgb_scatter_rank": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_i32, c_vp]),
    "sgb_gather_rows_bytes": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "sgb_edge_subset": (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp,
                                c_sz, c_vp]),
    "sgb_argsort_workspace_bytes": (c_sz, [c_i64]),
    "sgb_argsort_stable": (c_int, [c_vp, c_int, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_invert_permutation": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "sgb_tilecut_nodes": (c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_int, c_vp, c_vp, c_vp, c_vp]),
    "sgb_tilecut_edges": (c_int, [c_vp, c_vp, c_int, c_i64, c_i64, c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_int, c_vp, c_int,
                                  c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "sgb_partition_edges": (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_vp, c_vp, c_int, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp,
                                    c_i64, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_ranges_gather": (c_int, [c_vp, c_i64, c_vp, c_vp, c_int, c_i64, c_vp, c_vp]),
    "sgb_edges_collate": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_i64, c_vp]),
    "sgb_quadtree_max_leaves": (c_i64, [c_i64, c_i64, c_int]),
    "sgb_quadtree_workspace_bytes": (c_sz, [c_i64, c_i64, c_int]),
    "sgb_quadtree_build": (c_int, [c_vp, c_int, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "sgb_quadtree_label": (c_int, [c_vp, c_int, c_i64, c_vp, c_int, c_vp, c_int, c_vp, c_vp]),
    "sgb_quadtree_fit_mask": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_int, c_vp, c_vp]),
    "sgb_batch_vector": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp]),
    "sgb_dedupe_workspace_bytes": (c_sz, [c_i64]),
    "sgb_dedupe_max": (c_int, [c_vp, c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_gene_threshold_workspace_bytes": (c_sz, [c_i64, c_int]),
    "sgb_gene_thresholds": (c_int, [c_vp, c_int, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sgb_compact_predictions": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                        c_sz, c_vp]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)


def lib_path() -> Path:
    return Path(os.environ.get("SEGGER_B200_LIB", _LIB_PATH))


def load():
    """Load (once) and return the ctypes handle.  Raises if the library is absent."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not path.exists():
            raise RuntimeError(
                f"{path} not found: build it with `python -m segger_b200.build` "
                "(segger_b200 has no CPU or eager fallback)")
        lib = C.CDLL(str(path))
        for name, (res, args) in _PROTOS.items():
            fn = getattr(lib, name)   # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().sgb_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libsegger_b200 {what} failed (code {rc}): {msg}")


def ptr(t) -> int | None:
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "segger_b200 kernels run on CUDA tensors only (no CPU fallback); got a tensor on "
                f"{t.device}")
