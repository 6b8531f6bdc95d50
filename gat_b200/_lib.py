"""ctypes binding of libgat_b200.so (include/gat_b200.h).

The library is built in-tree by `__graft_entry__.build()` / `make -C gat_b200/csrc`.  There is no
Python or CPU fallback: if the shared library is missing, or no CUDA device is present, the engine
raises instead of computing anything on the host.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GATB_LIB: another build of the same library (kernel tuning experiments), never a different implementation
LIB_PATH = os.environ.get("GATB_LIB") or os.path.join(_HERE, "lib", "libgat_b200.so")

OK = 0
ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_TOO_LARGE, ERR_RANGE = -1, -2, -3, -4, -5

# every symbol include/gat_b200.h declares (tests/test_abi.py checks the .so exports them all)
SYMBOLS = [
    "gatb_version", "gatb_create", "gatb_destroy", "gatb_last_error", "gatb_set_stream",
    "gatb_synchronize", "gatb_launch_count", "gatb_set_batch_size", "gatb_profile", "gatb_profile_read",
    "gatb_annotations_create", "gatb_annotations_create_async", "gatb_annotations_wait",
    "gatb_annotations_destroy", "gatb_count_lists",
    "gatb_sampler_create", "gatb_sampler_destroy", "gatb_sampler_sample_capacity",
    "gatb_sampler_unit_capacity", "gatb_sampler_set_kind", "gatb_sampler_set_shift", "gatb_sampler_place",
    "gatb_sampler_place_units", "gatb_run", "gatb_column_stats", "gatb_column_pvalue", "gatb_compare_stats",
    "gatb_format_counts", "gatb_count_work", "gatb_microbench",
    "gatb_lists_from_rows", "gatb_lists_from_csr", "gatb_lists_restrict", "gatb_lists_collapse", "gatb_lists_select",
    "gatb_lists_info", "gatb_lists_sizes", "gatb_lists_download", "gatb_lists_destroy",
    "gatb_annotations_create_from_lists",
    "gatb_set_output_routes", "gatb_set_route_mode", "gatb_peer_alloc", "gatb_peer_free", "gatb_peer_open", "gatb_peer_close",
    "gatb_colacc_create", "gatb_colacc_set_windows", "gatb_colacc_add", "gatb_colacc_state", "gatb_colacc_merge",
    "gatb_colacc_finish", "gatb_colacc_destroy",
]

COLACC_SUMS, COLACC_HIST = 1, 2


class Route(ctypes.Structure):
    """gatb_route (include/gat_b200.h)"""
    _fields_ = [("base", ctypes.c_void_p), ("plane_stride", ctypes.c_uint64), ("row_stride", ctypes.c_uint64),
                ("row0", ctypes.c_uint64), ("col_begin", ctypes.c_uint32), ("col_end", ctypes.c_uint32)]


class GatB200Error(RuntimeError):
    """error reported by libgat_b200.so"""

    def __init__(self, code, message):
        RuntimeError.__init__(self, "gat_b200 error %i: %s" % (code, message))
        self.code = code


_lib = None


def load():
    """load libgat_b200.so; fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "gat_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C gat_b200/csrc` (there is no CPU fallback)" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    if hasattr(L, "gatb_emulation_marker"):
        raise ImportError("gat_b200: %s is the host-emulated test build of the kernels (tests/emu), not the CUDA "
                          "library -- the engine only runs on the GPU" % LIB_PATH)
    _lib = bind(L)
    return L


def bind(L):
    """declare the C signatures of include/gat_b200.h on a loaded library (load() does; tests/test_emu_parity.py binds
    the emulated test build of the same sources this way, without making it the engine's library)"""
    vp, i32, u32, u64, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_double
    L.gatb_version.restype = i32
    L.gatb_version.argtypes = []
    L.gatb_create.restype = i32
    L.gatb_create.argtypes = [i32, ctypes.POINTER(vp)]
    L.gatb_destroy.restype = None
    L.gatb_destroy.argtypes = [vp]
    L.gatb_last_error.restype = ctypes.c_char_p
    L.gatb_last_error.argtypes = [vp]
    L.gatb_set_stream.restype = i32
    L.gatb_set_stream.argtypes = [vp, vp]
    L.gatb_synchronize.restype = i32
    L.gatb_synchronize.argtypes = [vp]
    L.gatb_launch_count.restype = u64
    L.gatb_launch_count.argtypes = [vp]
    L.gatb_set_batch_size.restype = i32
    L.gatb_set_batch_size.argtypes = [vp, u32]
    L.gatb_profile.restype = i32
    L.gatb_profile.argtypes = [vp, i32]
    L.gatb_profile_read.restype = i32
    L.gatb_profile_read.argtypes = [vp, vp, vp]
    L.gatb_annotations_create.restype = i32
    L.gatb_annotations_create.argtypes = [vp, i32, i32, vp, vp, vp, vp, ctypes.POINTER(vp)]
    L.gatb_annotations_create_async.restype = i32
    L.gatb_annotations_create_async.argtypes = [vp, i32, i32, vp, vp, vp, vp, ctypes.POINTER(vp)]
    L.gatb_annotations_wait.restype = i32
    L.gatb_annotations_wait.argtypes = [vp]
    L.gatb_annotations_destroy.restype = None
    L.gatb_annotations_destroy.argtypes = [vp]
    L.gatb_count_lists.restype = i32
    L.gatb_count_lists.argtypes = [vp, vp, i32, vp, u64, vp, vp, vp, vp, vp]
    L.gatb_sampler_create.restype = i32
    L.gatb_sampler_create.argtypes = [vp, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp, u32, u32, ctypes.POINTER(vp)]
    L.gatb_sampler_destroy.restype = None
    L.gatb_sampler_destroy.argtypes = [vp]
    L.gatb_sampler_sample_capacity.restype = u64
    L.gatb_sampler_sample_capacity.argtypes = [vp]
    L.gatb_sampler_set_kind.restype = i32
    L.gatb_sampler_set_kind.argtypes = [vp, i32]
    L.gatb_sampler_set_shift.restype = i32
    L.gatb_sampler_set_shift.argtypes = [vp, ctypes.c_double, i32]
    L.gatb_sampler_place.restype = i32
    L.gatb_sampler_place.argtypes = [vp, u64, u32, u64, u64, vp, vp, vp, vp, vp]
    L.gatb_sampler_unit_capacity.restype = u64
    L.gatb_sampler_unit_capacity.argtypes = [vp]
    L.gatb_sampler_place_units.restype = i32
    L.gatb_sampler_place_units.argtypes = [vp, u64, u32, u64, u64, vp, vp, vp, vp, vp]
    L.gatb_column_pvalue.restype = i32
    L.gatb_column_pvalue.argtypes = [vp, vp, i32, i32, u64, i32, vp, vp, vp]
    L.gatb_run.restype = i32
    L.gatb_run.argtypes = [vp, vp, i32, vp, u64, u32, u64, u64, vp, vp, i32, vp]
    L.gatb_column_stats.restype = i32
    L.gatb_column_stats.argtypes = [vp, vp, i32, i32, u64, i32, vp, vp, dbl, vp, vp, vp, vp, vp, vp]
    L.gatb_compare_stats.restype = i32
    L.gatb_compare_stats.argtypes = [vp, u64, vp, i32, vp, i32, u64, vp, vp, vp, vp, vp, dbl, vp, vp, vp, vp, vp, vp]
    L.gatb_format_counts.restype = i32
    L.gatb_format_counts.argtypes = [vp, vp, i32, u64, i32, vp, vp, u64]
    L.gatb_count_work.restype = i32
    L.gatb_count_work.argtypes = [vp, vp, u32, vp]
    L.gatb_microbench.restype = i32
    L.gatb_microbench.argtypes = [i32, i32, u64, i32, vp]
    L.gatb_lists_from_rows.restype = i32
    L.gatb_lists_from_rows.argtypes = [vp, u64, vp, vp, vp, u32, i32, ctypes.POINTER(vp)]
    L.gatb_lists_from_csr.restype = i32
    L.gatb_lists_from_csr.argtypes = [vp, u32, vp, vp, vp, ctypes.POINTER(vp)]
    L.gatb_lists_restrict.restype = i32
    L.gatb_lists_restrict.argtypes = [vp, u32, u32, vp, i32, ctypes.POINTER(vp)]
    L.gatb_lists_collapse.restype = i32
    L.gatb_lists_collapse.argtypes = [vp, u32, ctypes.POINTER(vp)]
    L.gatb_lists_select.restype = i32
    L.gatb_lists_select.argtypes = [vp, u32, vp, ctypes.POINTER(vp)]
    L.gatb_lists_info.restype = i32
    L.gatb_lists_info.argtypes = [vp, vp, vp]
    L.gatb_lists_sizes.restype = i32
    L.gatb_lists_sizes.argtypes = [vp, vp, vp]
    L.gatb_lists_download.restype = i32
    L.gatb_lists_download.argtypes = [vp, vp, vp, vp]
    L.gatb_lists_destroy.restype = None
    L.gatb_lists_destroy.argtypes = [vp]
    L.gatb_annotations_create_from_lists.restype = i32
    L.gatb_annotations_create_from_lists.argtypes = [vp, vp, i32, i32, vp, ctypes.POINTER(vp)]
    L.gatb_set_output_routes.restype = i32
    L.gatb_set_output_routes.argtypes = [vp, i32, vp]
    L.gatb_set_route_mode.restype = i32
    L.gatb_set_route_mode.argtypes = [vp, i32]
    L.gatb_peer_alloc.restype = i32
    L.gatb_peer_alloc.argtypes = [vp, u64, ctypes.POINTER(vp), vp]
    L.gatb_peer_free.restype = i32
    L.gatb_peer_free.argtypes = [vp, vp]
    L.gatb_peer_open.restype = i32
    L.gatb_peer_open.argtypes = [vp, vp, ctypes.POINTER(vp)]
    L.gatb_peer_close.restype = i32
    L.gatb_peer_close.argtypes = [vp, vp]
    L.gatb_colacc_create.restype = i32
    L.gatb_colacc_create.argtypes = [vp, i32, u64, vp, vp, ctypes.POINTER(vp)]
    L.gatb_colacc_set_windows.restype = i32
    L.gatb_colacc_set_windows.argtypes = [vp, vp, vp]
    L.gatb_colacc_add.restype = i32
    L.gatb_colacc_add.argtypes = [vp, vp, u64, u64, i32]
    L.gatb_colacc_state.restype = i32
    L.gatb_colacc_state.argtypes = [vp, vp, vp, vp, vp, vp]
    L.gatb_colacc_merge.restype = i32
    L.gatb_colacc_merge.argtypes = [vp, u64, vp, vp, vp, vp]
    L.gatb_colacc_finish.restype = i32
    L.gatb_colacc_finish.argtypes = [vp, dbl, vp, vp, vp, vp, vp, vp, vp]
    L.gatb_colacc_destroy.restype = None
    L.gatb_colacc_destroy.argtypes = [vp]
    return L
