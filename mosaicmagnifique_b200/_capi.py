"""ctypes binding of include/mosaic_b200.h. Fails loudly when the CUDA library is missing: there is no fallback."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))


class MosaicError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("mosaic_b200 error %d: %s" % (code, msg))
        self.code = code


class CellShapeC(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "size", "row_spacing", "col_spacing", "alt_row_spacing", "alt_col_spacing", "alt_row_offset", "alt_col_offset",
        "alt_col_flip_h", "alt_col_flip_v", "alt_row_flip_h", "alt_row_flip_v")]


class Timings(ctypes.Structure):
    _fields_ = [("preprocess_ms", ctypes.c_double), ("diff_ms", ctypes.c_double), ("select_ms", ctypes.c_double),
                ("total_ms", ctypes.c_double), ("h2d_bytes", ctypes.c_double), ("d2h_bytes", ctypes.c_double),
                ("pixel_diffs", ctypes.c_double), ("pixel_diffs_nominal", ctypes.c_double),
                ("kernel_launches", ctypes.c_int64), ("evaluated_pixel_diffs", ctypes.c_double)]


PROGRESS_FN = ctypes.CFUNCTYPE(None, ctypes.c_int, ctypes.c_void_p)

_lib = None


def library_path():
    return os.environ.get("MOSAIC_B200_LIB", os.path.join(HERE, "libmosaic_b200.so"))


def capi():
    """Loads libmosaic_b200.so and declares every entry point of include/mosaic_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError("libmosaic_b200.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; "
                          "g.build()'` or `make -C mosaicmagnifique_b200/csrc`; there is no CPU fallback" % path)
    L = ctypes.CDLL(path)
    c = ctypes
    vp, i, i64, sz, dbl = c.c_void_p, c.c_int, c.c_int64, c.c_size_t, c.c_double
    u8p, f32p, i64p, i32p, dblp, ip = (c.POINTER(t) for t in (c.c_uint8, c.c_float, c.c_int64, c.c_int32, c.c_double, c.c_int))
    shp = c.POINTER(CellShapeC)
    sig = {
        "mosaic_create": (i, [i, c.POINTER(vp)]),
        "mosaic_destroy": (None, [vp]),
        "mosaic_last_error": (c.c_char_p, [vp]),
        "mosaic_version": (c.c_char_p, []),
        "mosaic_set_main_image": (i, [vp, vp, i, i, sz]),
        "mosaic_set_library": (i, [vp, vp, i64, i]),
        "mosaic_set_colour_difference": (i, [vp, i]),
        "mosaic_set_colour_scheme": (i, [vp, i]),
        "mosaic_set_cell_group": (i, [vp, shp, vp, i, i, i]),
        "mosaic_set_cell_group_ex": (i, [vp, shp, vp, i, i, i, i]),
        "mosaic_host_cell_group_cell": (i, [shp, vp, i, i, i, i, i, i, shp, vp, sz]),
        "mosaic_get_cell_shape": (i, [vp, i, i, shp, vp, sz]),
        "mosaic_set_grid_state": (i, [vp, i, i, i, vp]),
        "mosaic_compute_grid_state": (i, [vp]),
        "mosaic_get_grid_steps": (i, [vp]),
        "mosaic_get_grid_size": (i, [vp, i, ip, ip]),
        "mosaic_set_repeat": (i, [vp, i, i]),
        "mosaic_set_variant_quirk": (i, [vp, i]),
        "mosaic_generate": (i, [vp]),
        "mosaic_get_best_fits": (i, [vp, i, vp, i, i]),
        "mosaic_set_tile_flips": (i, [vp, i]),
        "mosaic_get_best_fit_flips": (i, [vp, i, vp, i, i]),
        "mosaic_set_usage_limit": (i, [vp, i]),
        "mosaic_build_photomosaic": (i, [vp, vp, vp, i, i, sz]),
        "mosaic_get_max_progress": (i, [vp]),
        "mosaic_set_progress_callback": (None, [vp, PROGRESS_FN, vp]),
        "mosaic_cancel": (None, [vp]),
        "mosaic_reset_cancel": (None, [vp]),
        "mosaic_set_keep_differences": (i, [vp, i]),
        "mosaic_get_valid_cell_count": (i64, [vp, i]),
        "mosaic_get_differences": (i, [vp, i, vp, i64, i64]),
        "mosaic_set_report_margins": (i, [vp, i]),
        "mosaic_get_margins": (i, [vp, i, vp, vp, i64]),
        "mosaic_get_timings": (i, [vp, c.POINTER(Timings)]),
        "mosaic_set_shard": (i, [vp, i, i]),
        "mosaic_host_shard_split": (i, [i64, i, i, i, i64p, i64p, i64p]),
        "mosaic_generate_candidates": (i, [vp]),
        "mosaic_get_candidate_count": (i, [vp, i, i64p, i64p, ip]),
        "mosaic_get_candidates_device": (i, [vp, i, c.POINTER(vp), c.POINTER(vp)]),
        "mosaic_select_from_candidates": (i, [vp, i, vp, vp, i]),
        "mosaic_get_candidate_block": (i, [vp, i, c.POINTER(vp), i64p, ip, c.POINTER(sz)]),
        "mosaic_select_from_gathered": (i, [vp, i, vp, i, i64]),
        "mosaic_get_shard_rows": (i, [vp, i, i, ip, ip]),
        "mosaic_set_main_image_rows": (i, [vp, vp, i, i, sz, i, i]),
        "mosaic_set_library_shard": (i, [vp, vp, i64, i64, i64, i, i64]),
        "mosaic_get_library_device": (i, [vp, c.POINTER(vp), ip, i64p]),
        "mosaic_kernel_colour_difference": (i, [i, i, vp, vp, i64, vp]),
        "mosaic_kernel_image_difference_sum": (i, [i, i, vp, vp, i64, vp, i, vp, vp]),
        "mosaic_kernel_prune_bound": (i, [i, vp, i, vp, i64, vp, i, vp, i, vp]),
        "mosaic_kernel_select": (i, [i, vp, i64, vp, i, i, i, i]),
        "mosaic_kernel_topk": (i, [i, vp, i64, i64, i, vp, vp]),
        "mosaic_kernel_bgr_to_lab": (i, [i, vp, i64, vp]),
        "mosaic_kernel_hue_rotate": (i, [i, vp, i, i, c.c_float, vp]),
        "mosaic_kernel_resize_area_u8": (i, [i, vp, i64, i, i, vp]),
        "mosaic_kernel_resize_area_f32": (i, [i, vp, i64, i, i, vp]),
        "mosaic_kernel_microbench": (i, [i, dblp, i]),
        "mosaic_grid_size": (None, [shp, i, i, i, ip, ip]),
        "mosaic_rect_at": (None, [shp, i, i, ip]),
        "mosaic_flip_at": (i, [shp, i, i]),
        "mosaic_host_grid_state": (i, [shp, vp, i, i, i, vp, i, i, sz, i, ip, ip, ip, vp, sz]),
        "mosaic_host_merge_bounds": (i, [vp, i, vp, i]),
        "mosaic_mcs_load": (i, [c.c_char_p, shp, vp, sz, c.c_char_p, sz]),
        "mosaic_mcs_save": (i, [c.c_char_p, shp, vp, c.c_char_p]),
        "mosaic_mil_info": (i, [c.c_char_p, i64p, ip, c.POINTER(sz)]),
        "mosaic_mil_load": (i, [c.c_char_p, vp, sz, c.c_char_p, sz]),
        "mosaic_mil_save": (i, [c.c_char_p, vp, i64, i, c.c_char_p]),
        "mosaic_io_last_error": (c.c_char_p, []),
        "mosaic_host_resize_area_u8": (i, [vp, i, i, i, vp, i, i]),
        "mosaic_host_resize_cubic_u8": (i, [vp, i, i, i, vp, i, i]),
        "mosaic_kernel_resize_cubic_u8": (i, [i, vp, i, i, i, vp, i, i]),
        "mosaic_library_ingest": (i, [i, vp, i, i, sz, i, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    L._signatures = sig
    _lib = L
    return L
