"""ctypes binding of libscanpy_b200.so (the C ABI declared in include/scanpy_b200.h).

This is the only module that touches the shared library.  There is NO CPU path: if the
library cannot be loaded, or no sm_100 device is present, every entry point raises.
torch is used here strictly as plumbing: device allocations (torch.empty(device='cuda')),
host<->device copies and the current CUDA stream handle; all arithmetic happens in the .so.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, byref, c_char, c_char_p, c_double, c_float, c_int32, c_int64, c_uint64, c_void_p
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libscanpy_b200.so"
CSRC = _PKG / "csrc"


class B200Error(RuntimeError):
    """Raised for any non-zero status from libscanpy_b200 (message = sb2_last_error())."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"libscanpy_b200 error {code}: {msg}")
        self.code = code


class DeviceInfo(ctypes.Structure):
    _fields_ = [("device", c_int32), ("sm_count", c_int32), ("cc_major", c_int32), ("cc_minor", c_int32),
                ("clock_khz", c_int32), ("mem_clock_khz", c_int32), ("l2_bytes", c_int32),
                ("smem_per_block_optin", c_int32), ("total_mem", c_int64), ("name", c_char * 64)]


class PcaInfo(ctypes.Structure):
    _fields_ = [("iterations", c_int32), ("converged", c_int32), ("max_rel_residual", c_double),
                ("total_var", c_double)]


class KnnInfo(ctypes.Structure):
    _fields_ = [("n_uncertified", c_int64), ("max_norm", c_float), ("pass1_ms", c_float), ("pass1_flops", c_double),
                ("pass1_issued_flops", c_double), ("pass1_tensor", c_int32), ("n_resweep", c_int64)]


class EigsInfo(ctypes.Structure):
    _fields_ = [("restarts", c_int32), ("matvecs", c_int32), ("n_converged", c_int32), ("reserved", c_int32),
                ("max_residual", c_double)]


class LeidenInfo(ctypes.Structure):
    _fields_ = [("passes", c_int32), ("levels", c_int32), ("moves", c_int64)]


# name -> (restype, argtypes); every symbol include/scanpy_b200.h declares must appear here
SIGNATURES = {
    "sb2_version": (c_int32, []),
    "sb2_last_error": (c_char_p, []),
    "sb2_ctx_create": (c_int32, [c_int32, c_void_p, ctypes.c_uint32, POINTER(c_void_p)]),
    "sb2_ctx_destroy": (c_int32, [c_void_p]),
    "sb2_ctx_sync": (c_int32, [c_void_p]),
    "sb2_device_info_get": (c_int32, [c_void_p, POINTER(DeviceInfo)]),
    "sb2_ctx_launch_count": (c_int64, [c_void_p]),
    "sb2_comm_unique_id": (c_int32, [c_void_p]),
    "sb2_comm_init": (c_int32, [c_void_p, c_int32, c_int32, c_void_p]),
    "sb2_comm_allgather": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64]),
    "sb2_comm_allreduce_f64": (c_int32, [c_void_p, c_void_p, c_int64]),
    "sb2_pca_csr_f32": (c_int32, [c_void_p, c_int64, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int32,
                                  c_int32, c_int32, c_double, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, POINTER(PcaInfo)]),
    "sb2_tsvd_csr_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_double,
                                   c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(PcaInfo)]),
    "sb2_pca_stream_accumulate_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sb2_pca_stream_solve_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_double,
                                           c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           POINTER(c_int32), POINTER(PcaInfo)]),
    "sb2_pca_stream_project_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                             c_void_p, c_void_p, c_void_p]),
    "sb2_csr_col_stats": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sb2_spmm_csr": (c_int32, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p]),
    "sb2_spmm_csr_t": (c_int32, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p]),
    "sb2_csr_gram": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sb2_knn_l2_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int64, c_int32, c_void_p,
                                 c_void_p, POINTER(KnnInfo)]),
    "sb2_knn_debug_proposals_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                              c_void_p]),
    "sb2_fuzzy_simplicial_set_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_float, c_float,
                                               c_void_p, c_void_p, c_void_p, c_int64, POINTER(c_int64), c_void_p,
                                               c_void_p]),
    "sb2_knn_connectivities_f64": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int32, c_void_p, c_void_p,
                                             c_void_p, c_int64, POINTER(c_int64)]),
    "sb2_leiden_csr_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_double, c_int32, c_uint64,
                                     c_void_p, POINTER(c_double), POINTER(c_int32), POINTER(LeidenInfo)]),
    "sb2_modularity_csr_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_double, c_void_p,
                                         POINTER(c_double)]),
    "sb2_eigsh_csr_scaled": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32,
                                       c_double, c_int32, c_void_p, c_void_p, c_void_p, POINTER(EigsInfo)]),
    "sb2_transition_scale_f64": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "sb2_umap_spectral_init_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int32, c_uint64, c_void_p]),
    "sb2_umap_layout_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_double, c_double,
                                      c_double, c_double, c_int32, c_uint64, c_void_p]),
    "sb2_group_arc_counts": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "sb2_louvain_csr_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_double, c_uint64,
                                      c_void_p, POINTER(c_double), POINTER(c_int32), POINTER(LeidenInfo)]),
    "sb2_csr_col_stats_rows_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p]),
    "sb2_csr_scale_cols_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                         c_double]),
    "sb2_csr_scale_dense_f64": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_int32, c_double, c_void_p]),
    "sb2_dense_col_stats": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "sb2_dense_scale": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32,
                                  c_double]),
    "sb2_csr_row_sums_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sb2_csr_hiexpr_count_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_double,
                                           c_void_p]),
    "sb2_csr_scale_rows_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "sb2_log1p_f32": (c_int32, [c_void_p, c_int64, c_void_p, c_double]),
    "sb2_csr_col_sums_f32": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int32, c_double, c_void_p,
                                       c_void_p]),
    "sb2_rank_genes_group_stats": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_int32, c_double, c_void_p, c_void_p, c_void_p]),
    "sb2_rank_genes_wilcoxon": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_void_p,
                                          c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
}

RANK_GENES_MAX_GROUPS = 1024  # SB2_RANK_GENES_MAX_GROUPS in include/scanpy_b200.h

_lib = None


def build(force: bool = False) -> Path:
    """Compile the CUDA sources for sm_100a into scanpy_b200/libscanpy_b200.so (in-tree)."""
    srcs = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [_PKG.parent / "include" / "scanpy_b200.h"]
    newest = max(p.stat().st_mtime for p in srcs)
    if force or not LIB_PATH.exists() or LIB_PATH.stat().st_mtime < newest:
        r = subprocess.run(["make", "-C", str(CSRC), "-j8"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("building libscanpy_b200.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    return LIB_PATH


def load():
    """Load the library (never builds implicitly on a GPU box: the .so ships in-tree)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise B200Error(-2, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                "(there is no CPU fallback)")
        lib = ctypes.CDLL(str(LIB_PATH), mode=ctypes.RTLD_GLOBAL if os.name != "nt" else 0)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code: int) -> None:
    if code != 0:
        raise B200Error(code, load().sb2_last_error().decode(errors="replace"))


class Context:
    """Owns an sb2_ctx bound to one CUDA device and (by default) torch's current stream."""

    def __init__(self, device: int | None = None, *, use_torch_stream: bool = True):
        import torch

        if not torch.cuda.is_available():
            raise B200Error(-2, "no CUDA device visible: scanpy_b200 has no CPU path")
        self.lib = load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        torch.cuda.set_device(self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream if use_torch_stream else 0
        h = c_void_p()
        check(self.lib.sb2_ctx_create(self.device, c_void_p(stream), 0 if use_torch_stream else 1, byref(h)))
        self.handle = h
        self.n_ranks, self.rank = 1, 0

    def close(self):
        if getattr(self, "handle", None):
            self.lib.sb2_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        check(self.lib.sb2_ctx_sync(self.handle))

    def device_info(self) -> DeviceInfo:
        info = DeviceInfo()
        check(self.lib.sb2_device_info_get(self.handle, byref(info)))
        return info

    @property
    def launches(self) -> int:
        return int(self.lib.sb2_ctx_launch_count(self.handle))


_default_ctx: dict[int, Context] = {}


def default_context() -> Context:
    import torch

    dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
    ctx = _default_ctx.get(dev)
    if ctx is None:
        ctx = _default_ctx[dev] = Context(dev)
    return ctx


def ptr(t) -> c_void_p:
    """Raw device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return c_void_p(0)
    if hasattr(t, "data_ptr"):
        assert t.is_contiguous()
        return c_void_p(t.data_ptr())
    assert t.flags["C_CONTIGUOUS"]
    return c_void_p(t.ctypes.data)
