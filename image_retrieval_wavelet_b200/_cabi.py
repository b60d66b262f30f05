"""ctypes binding of ``libb200ret.so`` (C-ABI declared in ``include/b200ret.h``).

There is no CPU fallback: if the shared library is missing the import fails loudly, and every entry point that
needs a device raises when CUDA is unavailable.  torch only supplies ``data_ptr()`` and the current stream.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200RET_LIB") or os.path.join(_HERE, "libb200ret.so")   # override: A/B runs of two builds

OK = 0
ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_WORKSPACE, ERR_ALIGNMENT, ERR_NO_DEVICE = -1, -2, -3, -4, -5, -6
LABELS_OVERLAP, LABELS_EQUAL = 0, 1
RESIZE_BICUBIC, RESIZE_BILINEAR = 0, 1
MAX_CODE_BITS = 256
MAX_LABEL_BITS = 256

c_void_p, c_int, c_ll, c_size_t, c_double = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_size_t, ctypes.c_double


class MapPlan(ctypes.Structure):
    """``b200_map_plan`` (include/b200ret.h)."""
    _fields_ = [
        ("Q", c_int), ("N", c_ll), ("N_total", c_ll), ("B", c_int), ("LW", c_int), ("label_mode", c_int), ("k", c_ll),
        ("bins", c_int), ("T", c_int), ("groups", c_int), ("Qpad", c_int), ("S", c_int), ("seg_len", c_int),
        ("wide", c_int), ("tile", c_int), ("stash", c_int),
        ("off_hist", c_size_t), ("off_tot", c_size_t), ("off_dstar", c_size_t), ("off_psum", c_size_t),
        ("off_phits", c_size_t), ("off_stash_d", c_size_t), ("off_stash_r", c_size_t), ("workspace_bytes", c_size_t),
        ("select", c_int), ("sel_stride", c_int), ("sel_S", c_int), ("sel_seg_len", c_int), ("sel_chunk", c_int),
        ("sel_maxc", c_int), ("smp_S", c_int), ("smp_seg_len", c_int), ("sel_T", c_int), ("smp_rows", c_ll), ("sel_pool_chunks", c_ll),
        ("off_sel_flags", c_size_t), ("off_sel_bound", c_size_t), ("off_sel_count", c_size_t), ("off_sel_table", c_size_t),
        ("off_sel_pool", c_size_t), ("off_smp_codes", c_size_t), ("off_smp_hist", c_size_t),
    ]


# name -> (restype, argtypes); mirrors include/b200ret.h one to one (tests check every symbol exists)
SIGNATURES = {
    "b200_version": (c_int, []),
    "b200_sizeof_map_plan": (c_size_t, []),
    "b200_error_string": (ctypes.c_char_p, [c_int]),
    "b200_last_cuda_error": (ctypes.c_char_p, []),
    "b200_launch_count": (ctypes.c_ulonglong, []),
    "b200_swt2_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200_raw_stack": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b200_swt2_fwd_host": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int]),
    "b200_resize_workspace_bytes": (c_size_t, [c_ll, c_int, c_int, c_int, c_int, c_int]),
    "b200_resize_u8": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "b200_resize_crop_workspace_bytes": (c_size_t, [c_int, c_void_p, c_int, c_int, c_int, c_int]),
    "b200_resize_crop_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t,
                                    c_void_p]),
    "b200_dwt2_workspace_bytes": (c_size_t, [c_ll, c_int, c_int, c_int, c_int]),
    "b200_dwt2_fwd": (c_int, [c_void_p, c_int, c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_size_t,
                              c_void_p]),
    "b200_pack_codes": (c_int, [c_void_p, c_ll, c_int, c_void_p, c_void_p, c_void_p]),
    "b200_pack_labels": (c_int, [c_void_p, c_ll, c_int, c_void_p, c_void_p, c_void_p]),
    "b200_pack_labels_scalar": (c_int, [c_void_p, c_int, c_ll, c_void_p, c_void_p, c_void_p]),
    "b200_bit_counts": (c_int, [c_void_p, c_ll, c_int, c_void_p, c_void_p]),
    "b200_hamming_dist": (c_int, [c_void_p, c_void_p, c_int, c_ll, c_int, c_void_p, c_void_p]),
    "b200_label_relevance": (c_int, [c_void_p, c_void_p, c_int, c_ll, c_int, c_int, c_void_p, c_void_p]),
    "b200_map_plan_init": (c_int, [ctypes.POINTER(MapPlan), c_int, c_ll, c_ll, c_int, c_int, c_int, c_ll]),
    "b200_hamming_hist": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200_hamming_scan": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200_hamming_ap": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_ll, c_void_p]),
    "b200_ap_reduce": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200_ap_finalize": (c_int, [c_void_p, c_void_p, c_int, c_ll, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200_hamming_map": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p]),
    "b200_hamming_map_try": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p]),
    "b200_map_final": (c_int, [c_void_p, c_int, c_void_p, c_int, c_ll, c_void_p, c_void_p]),
    "b200_hamming_map_stage_ms": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200_map_select_status": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p]),
    "b200_hamming_topk": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200_ranked_ap": (c_int, [c_void_p, c_int, c_int, c_ll, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p]),
    "b200_merge_topk": (c_int, [c_void_p, c_void_p, c_int, c_int, c_ll, c_int, c_void_p, c_void_p, c_void_p]),
    "b200_hamming_radius_counts": (c_int, [ctypes.POINTER(MapPlan), c_void_p, c_void_p, c_void_p]),
    "b200_ranked_cumhits": (c_int, [c_void_p, c_int, c_ll, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "b200_curve_accumulate": (c_int, [c_void_p, c_int, c_ll, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200_knn_workspace_bytes": (c_size_t, [c_int, c_ll, c_int, c_int]),
    "b200_knn_topk": (c_int, [c_void_p, c_void_p, c_int, c_ll, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                              c_void_p]),
    "b200_mean_f64": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "b200_comm_create": (c_int, [c_int, c_int, c_size_t, ctypes.POINTER(c_void_p)]),
    "b200_comm_export": (c_int, [c_void_p, c_void_p]),
    "b200_comm_open": (c_int, [c_void_p, c_void_p]),
    "b200_comm_buffer": (c_void_p, [c_void_p, c_int]),
    "b200_comm_bytes": (c_size_t, [c_void_p]),
    "b200_comm_world": (c_int, [c_void_p]),
    "b200_comm_rank": (c_int, [c_void_p]),
    "b200_comm_barrier": (c_int, [c_void_p, c_void_p]),
    "b200_comm_put": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200_comm_put_barrier_final": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, ctypes.c_size_t, c_int, ctypes.c_size_t,
                                            c_void_p, c_void_p]),
    "b200_pack_to_ranks": (c_int, [c_void_p, c_int, c_ll, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "b200_comm_status": (c_int, [c_void_p, ctypes.POINTER(c_int)]),
    "b200_comm_status_word": (c_void_p, [c_void_p]),
    "b200_comm_destroy": (c_int, [c_void_p]),
    "b200_select_topk_f32": (c_int, [c_void_p, c_int, c_ll, c_ll, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b200_maphashing_host_packed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_ll, c_int, c_int, c_int, c_ll, c_void_p,
                                            c_void_p, c_void_p]),
    "b200_maphashing_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_ll, c_int, c_int, c_int, c_ll, c_void_p,
                                     c_void_p, c_void_p, c_void_p]),
}

_lib = None


class B200Error(RuntimeError):
    pass


def load():
    """Load the shared library once.  Raises ImportError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m image_retrieval_wavelet_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback for the B200 hot paths.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.b200_sizeof_map_plan() != ctypes.sizeof(MapPlan):
            raise ImportError(f"{LIB_PATH}: b200_map_plan is {lib.b200_sizeof_map_plan()} bytes, the ctypes mirror {ctypes.sizeof(MapPlan)}: "
                              "rebuild the library (python -m image_retrieval_wavelet_b200.build --force)")
        _lib = lib
    return _lib


def check(rc, what=""):
    """Map a C-ABI status to the Python exception the reference's own code would raise."""
    if rc == OK:
        return
    lib = load()
    msg = f"{what}: {lib.b200_error_string(rc).decode()}" if what else lib.b200_error_string(rc).decode()
    if rc == ERR_INVALID_ARG:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ERR_CUDA:
        raise B200Error(f"{msg}: {lib.b200_last_cuda_error().decode()}")
    raise B200Error(msg)


def code_words(bits):
    return 1 if bits <= 64 else (2 if bits <= 128 else 4)


def label_words(labels):
    return 1 if labels <= 64 else (2 if labels <= 128 else 4)


def launch_count():
    return int(load().b200_launch_count())


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise B200Error("no CUDA device: the B200 hot paths have no CPU fallback")


def stream_ptr():
    import torch

    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device/host pointer of a tensor (None -> NULL)."""
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


class nvtx_range:
    """``with nvtx_range("b200/<what>"):`` — an NVTX range around a host-side phase (Nsight Systems shows it above the kernels
    it launched; SURVEY §5 tracing).  ``B200_NVTX=0`` turns the ranges into no-ops; without torch's NVTX bindings they are
    no-ops too."""

    _on = os.environ.get("B200_NVTX", "1") != "0"

    def __init__(self, name):
        self.name = name
        self.pushed = False

    def __enter__(self):
        if nvtx_range._on:
            try:
                import torch

                torch.cuda.nvtx.range_push(self.name)
                self.pushed = True
            except Exception:
                nvtx_range._on = False
        return self

    def __exit__(self, *exc):
        if self.pushed:
            import torch

            torch.cuda.nvtx.range_pop()
        return False

