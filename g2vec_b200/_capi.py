"""ctypes binding of libg2vec_b200.so (the C ABI declared in include/g2vec_b200.h).

There is no CPU fallback: if the library is missing and cannot be built, or a call fails,
a RuntimeError is raised.
"""
import ctypes
import os

from . import build as _build

_lib = None

_vp, _i32, _i64, _u32, _u64, _f32 = (ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32,
                                     ctypes.c_uint64, ctypes.c_float)

# name -> (restype, argtypes); must list every symbol include/g2vec_b200.h declares
SIGNATURES = {
    "g2v_abi_version": (ctypes.c_int, []),
    "g2v_last_error": (ctypes.c_char_p, []),
    "g2v_device_info": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "g2v_launch_count": (_i64, []),
    "g2v_walk_workspace_bytes": (ctypes.c_size_t, []),
    "g2v_walk_launch": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i64, _i32, _u64, _u32, _i64, _i64, _i64,
                                       _vp, _vp, _vp, _vp]),
    "g2v_walk_packed_bytes": (ctypes.c_int, [_i32, _i64, _vp, _vp]),
    "g2v_walk_prepare": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp]),
    "g2v_walk_launch_packed": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i64, _i32, _u64, _u32, _i64, _i64, _i64,
                                              _vp, _vp, _vp, _vp, _vp]),
    "g2v_walk_host": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i64, _i32, _u64, _u32, _i64, _i64, _i64, _vp, _vp]),
    "g2v_cbow_fwdbwd": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _i32, _i32, _i32, _vp]),
    "g2v_cbow_update": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f32, _f32,
                                       _f32, _f32, _i32, _vp, _vp]),
    "g2v_cbow_update_nvl": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _f32, _f32, _f32,
                                           _f32, _i32, _vp, _vp]),
    "g2v_cbow_adam_tick": (ctypes.c_int, [_vp, _f32, _f32, _f32, _vp]),
    "g2v_cbow_eval": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "g2v_cbow_loop_init": (ctypes.c_int, [_vp, _i64, _i32, _vp]),
    "g2v_cbow_loop_attach": (ctypes.c_int, [_vp]),
    "g2v_cbow_loop_begin": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "g2v_cbow_loop_decide": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "g2v_cbow_loop_counters_nvl": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _vp]),
    "g2v_cbow_slab_plan": (ctypes.c_int, [_i32, _i32, _vp]),
    "g2v_cbow_slab_workspace_bytes": (ctypes.c_size_t, [_i64, _i32, _i32]),
    "g2v_cbow_slab_setup": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _i32, _i32, _vp, _vp]),
    "g2v_cbow_fwdbwd_slabs": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _vp, _vp,
                                             _i32, _i32, _i32, _i32, _vp, _vp]),
    "g2v_cbow_eval_slabs": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "g2v_cbow_step_host": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32,
                                          _i32, _i32, _f32, _f32, _f32, _f32, _i32, _vp, _vp]),
    "g2v_cbow_r1_prepare": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _vp]),
    "g2v_cbow_r1_windows": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "g2v_cbow_r1_windows_csc": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                              _i32, _i32, _vp]),
    "g2v_cbow_r1_scratch_bytes": (ctypes.c_size_t, [_i32]),
    "g2v_cbow_r1_update": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f32, _f32,
                                         _f32, _f32, _i32, _vp, _vp]),
    "g2v_pcc_zscore": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp]),
    "g2v_pcc_edge_weights": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _i64, _vp, _vp]),
    "g2v_paths_canonicalise": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _vp]),
    "g2v_paths_mark": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp]),
    "g2v_paths_set_workspace_bytes": (ctypes.c_size_t, [_i64]),
    "g2v_paths_set_select": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    "g2v_paths_set_emit": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _i64, _i64, _vp, _vp, _vp, _vp,
                                          _vp, _vp]),
    "g2v_kmeans_workspace_bytes": (ctypes.c_size_t, [_i32, _i32, _i32]),
    "g2v_kmeans_center": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "g2v_kmeans_dist": (ctypes.c_int, [_vp, _i32, _i32, _vp, _i32, _vp, _vp, _vp]),
    "g2v_kmeans_lloyd_step": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "g2v_post_tscores": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "g2v_post_row_norms": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "g2v_fmt_row_bytes": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _vp]),
    "g2v_fmt_emit": (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "g2v_test_l2_rows": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp]),
    "g2v_test_draws": (ctypes.c_int, [_u64, _u64, _i32, _vp, _vp]),
    "g2v_test_curand_draws": (ctypes.c_int, [_u64, _u64, _i32, _vp, _vp]),
}

OPT_ADAM_TF1, OPT_SGD = 0, 1
REDUCE_SUM, REDUCE_MEAN = 0, 1


def library_path():
    return _build.LIB


def load():
    """Load (building first if stale and nvcc is present) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("G2VEC_B200_LIB") or _build.LIB     # A/B builds of the same ABI (profiles/variants)
    if path == _build.LIB and _build.stale():
        try:
            _build.build_library()
        except Exception as exc:  # no nvcc, or compile error
            if not os.path.exists(path):
                raise RuntimeError(
                    "libg2vec_b200.so is not built and could not be built (%s). Run "
                    "`python -c 'import __graft_entry__ as g; g.build()'`. There is no CPU fallback." % exc)
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.g2v_abi_version() != 2:
        raise RuntimeError("libg2vec_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().g2v_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (rc=%d): %s" % (what, rc, msg))


def launch_count():
    return int(load().g2v_launch_count())
