"""ctypes binding of `libmdf_b200.so` (C ABI in `include/mdf_b200.h`).

The product path has no CPU implementation: if the shared library has not been built, or no
sm_100 GPU is visible, every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Dict, Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmdf_b200.so")

MDF_OK, MDF_EINVAL, MDF_ECUDA, MDF_ENOMEM, MDF_EUNSUPPORTED, MDF_ENOENT, MDF_EPARSE = 0, -1, -2, -3, -4, -5, -6


class UnsupportedModelError(NotImplementedError):
    """The `.onnx` graph is not one the fused pipeline computes (MDF_EUNSUPPORTED); a RuntimeError, as `predict.pyi:70-72`
    promises for models that cannot be loaded.  There is no fallback executor."""

c_f32p = C.POINTER(C.c_float)
c_i32p = C.POINTER(C.c_int32)
c_u32p = C.POINTER(C.c_uint32)
c_i64p = C.POINTER(C.c_int64)


class ModelDesc(C.Structure):
    _fields_ = [
        ("n_channels", C.c_int), ("lstm_hidden", C.c_int), ("n_lstm", C.c_int),
        ("lstm_W", c_f32p * 4), ("lstm_R", c_f32p * 4), ("lstm_B", c_f32p * 4),
        ("lm_dim", C.c_int), ("aa_W", c_f32p), ("lm_W", c_f32p), ("lm_b", c_f32p),
        ("n_gc", C.c_int), ("gc_dims", C.c_int * 8), ("gc_W", c_f32p * 8), ("gc_b", c_f32p * 8),
        ("gc_activation", C.c_int), ("gc_alpha", C.c_float), ("eps", C.c_float),
        ("fc_dim", C.c_int), ("fc_W", c_f32p), ("fc_b", c_f32p),
        ("n_terms", C.c_int), ("out_W", c_f32p), ("out_b", c_f32p),
    ]


MAX_CONV = 32


class CnnDesc(C.Structure):
    _fields_ = [
        ("n_channels", C.c_int), ("n_conv", C.c_int),
        ("conv_width", C.c_int * MAX_CONV), ("conv_filters", C.c_int * MAX_CONV), ("conv_pad_left", C.c_int * MAX_CONV),
        ("conv_W", c_f32p * MAX_CONV), ("scale", c_f32p), ("shift", c_f32p),
        ("n_terms", C.c_int), ("out_W", c_f32p), ("out_b", c_f32p),
    ]


_lib = None
_lib_lock = threading.Lock()


def lib() -> C.CDLL:
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build the CUDA extension first "
                "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        vp = C.c_void_p
        L.mdf_last_error.restype = C.c_char_p
        L.mdf_version.restype = C.c_int
        L.mdf_ctx_create.argtypes = [C.c_int, vp, C.c_size_t, vp, C.POINTER(vp)]
        L.mdf_ctx_destroy.argtypes = [vp]
        L.mdf_ctx_synchronize.argtypes = [vp]
        L.mdf_ctx_launch_count.argtypes = [vp]
        L.mdf_ctx_launch_count.restype = C.c_int64
        L.mdf_ctx_profile.argtypes = [vp, C.c_int]
        L.mdf_ctx_profile.restype = C.c_int
        L.mdf_ctx_profile_report.argtypes = [vp, C.c_char_p, C.c_size_t]
        L.mdf_ctx_profile_report.restype = C.c_int
        L.mdf_ctx_set_debug_taps.argtypes = [vp, C.c_int]
        L.mdf_ctx_set_debug_taps.restype = C.c_int
        L.mdf_pairwise_sqeuclidean.argtypes = [vp, c_f32p, C.c_int, C.c_int, c_f32p]
        L.mdf_contact_map_dense.argtypes = [vp, c_f32p, C.c_int, C.c_float, c_i32p]
        L.mdf_contact_map_sparse.argtypes = [vp, c_f32p, C.c_int, C.c_float, c_i32p, C.c_int64, c_i64p]
        L.mdf_align_contact_map.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_int, c_i32p, C.c_int64, C.c_int,
                                            c_i32p, C.POINTER(C.c_int)]
        L.mdf_cmap_build_transfer.argtypes = [vp, C.c_int, c_f32p, c_i64p, C.c_char_p, C.c_char_p, c_i64p, c_i64p,
                                              C.c_float, C.c_int, c_u32p, c_i64p, c_i32p, c_i64p]
        L.mdf_model_create.argtypes = [vp, C.POINTER(ModelDesc), C.POINTER(vp)]
        L.mdf_model_destroy.argtypes = [vp]
        L.mdf_model_load.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
        L.mdf_cnn_model_load.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
        L.mdf_onnx_inspect.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]
        L.mdf_onnx_tensor.argtypes = [C.c_char_p, C.c_char_p, c_f32p, C.c_int64, c_i64p]
        L.mdf_onnx_tensor.restype = C.c_int
        ip_ = C.POINTER(C.c_int)
        L.mdf_model_info.argtypes = [vp, ip_, ip_, ip_, ip_, ip_, ip_]
        L.mdf_model_set_engine.argtypes = [vp, C.c_int]
        L.mdf_model_get_engine.argtypes = [vp]
        L.mdf_model_get_engine.restype = C.c_int
        L.mdf_gcn_forward_dense.argtypes = [vp, C.c_char_p, C.c_int, c_i32p, c_f32p]
        L.mdf_gcn_forward_packed.argtypes = [vp, C.c_int, C.c_char_p, c_i64p, c_u32p, c_i64p, c_f32p]
        L.mdf_path_forward.argtypes = [vp, C.c_int, vp, c_i64p, vp, c_i64p, vp, vp, c_i64p,
                                       C.c_float, C.c_int, vp]
        L.mdf_path_submit.argtypes = [vp, C.c_int, vp, c_i64p, vp, c_i64p, vp, vp, c_i64p, C.c_float, C.c_int, vp, C.POINTER(vp)]
        L.mdf_path_submit_ragged.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_float, C.c_int, vp, C.POINTER(vp)]
        L.mdf_path_submit_pairs.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_char_p, C.c_int, C.c_int, C.c_int,
                                            C.c_float, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.POINTER(vp)]
        L.mdf_path_wait.argtypes = [vp]
        for name in ("mdf_path_submit", "mdf_path_submit_ragged", "mdf_path_submit_pairs", "mdf_path_wait"):
            getattr(L, name).restype = C.c_int
        L.mdf_batch_upload.argtypes = [vp, C.c_int, vp, c_i64p, vp, c_i64p, vp, vp, c_i64p, C.POINTER(vp)]
        L.mdf_batch_upload_pairs.argtypes = [vp, C.c_int, vp, c_i64p, vp, c_i64p, vp, c_i64p, vp, C.c_char_p, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(vp)]
        L.mdf_batch_fetch_alignment.argtypes = [vp, vp, vp, vp, vp, vp, vp]
        for name in ("mdf_batch_upload_pairs", "mdf_batch_fetch_alignment"):
            getattr(L, name).restype = C.c_int
        L.mdf_batch_destroy.argtypes = [vp]
        L.mdf_path_run.argtypes = [vp, vp, C.c_float, C.c_int]
        L.mdf_path_run_stages.argtypes = [vp, vp, C.c_float, C.c_int, C.c_int]
        L.mdf_path_run_shared.argtypes = [vp, vp, C.c_float, C.c_int]
        L.mdf_batch_fetch_scores.argtypes = [vp, vp, vp]
        L.mdf_batch_fetch.argtypes = [vp, vp, C.c_int, vp, C.c_size_t]
        L.mdf_batch_invalidate.argtypes = [vp]
        L.mdf_batch_invalidate.restype = C.c_int
        L.mdf_batch_unpack_dense.argtypes = [vp, vp, c_i64p]
        L.mdf_batch_unpack_dense.restype = C.c_int
        L.mdf_batch_scores_device.argtypes = [vp]
        L.mdf_batch_scores_device.restype = vp
        L.mdf_cnn_model_create.argtypes = [vp, C.POINTER(CnnDesc), C.POINTER(vp)]
        L.mdf_cnn_model_destroy.argtypes = [vp]
        L.mdf_cnn_forward.argtypes = [vp, C.c_int, vp, c_i64p, vp]
        L.mdf_cnn_upload.argtypes = [vp, C.c_int, vp, c_i64p]
        L.mdf_cnn_run.argtypes = [vp]
        L.mdf_cnn_fetch.argtypes = [vp, vp, vp]
        L.mdf_cnn_submit_ragged.argtypes = [vp, C.c_int, vp, vp, vp, C.POINTER(vp)]
        L.mdf_pdb_calpha.argtypes = [vp, C.c_size_t, C.c_char, vp, vp, vp, C.c_int, C.POINTER(C.c_int)]
        L.mdf_pdb_calpha_batch.argtypes = [C.c_int, vp, c_i64p, C.c_char, C.c_int, vp, vp, C.c_int64, c_i64p]
        L.mdf_coords_cache_create.argtypes = [C.c_char_p, C.c_int64, vp, vp, vp]
        L.mdf_coords_cache_open.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.mdf_coords_cache_close.argtypes = [vp]
        L.mdf_coords_cache_size.argtypes = [vp]
        L.mdf_coords_cache_size.restype = C.c_int64
        L.mdf_coords_cache_lookup.argtypes = [vp, C.c_int64, vp, vp, vp, c_i64p]
        L.mdf_coords_cache_entry.argtypes = [vp, C.c_int64, C.c_char_p, C.c_size_t, C.POINTER(C.c_int)]
        for name in ("mdf_pdb_calpha", "mdf_pdb_calpha_batch", "mdf_coords_cache_create", "mdf_coords_cache_open", "mdf_coords_cache_close",
                     "mdf_coords_cache_lookup", "mdf_coords_cache_entry"):
            getattr(L, name).restype = C.c_int
        L.mdf_nw_align.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, C.c_char_p, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]
        L.mdf_nw_align.restype = C.c_int
        for name in ("mdf_model_load", "mdf_cnn_model_load", "mdf_onnx_inspect", "mdf_model_info"):
            getattr(L, name).restype = C.c_int
        for name in ("mdf_cnn_model_create", "mdf_cnn_model_destroy", "mdf_cnn_forward", "mdf_cnn_upload", "mdf_cnn_run",
                     "mdf_cnn_fetch", "mdf_cnn_submit_ragged"):
            getattr(L, name).restype = C.c_int
        for name in ("mdf_ctx_create", "mdf_ctx_destroy", "mdf_ctx_synchronize", "mdf_pairwise_sqeuclidean",
                     "mdf_contact_map_dense", "mdf_contact_map_sparse", "mdf_align_contact_map",
                     "mdf_cmap_build_transfer", "mdf_cmap_build_transfer_ragged", "mdf_model_create", "mdf_model_destroy", "mdf_model_set_engine",
                     "mdf_gcn_forward_dense", "mdf_gcn_forward_packed", "mdf_path_forward", "mdf_batch_upload",
                     "mdf_batch_destroy", "mdf_path_run", "mdf_path_run_stages", "mdf_path_run_shared",
                     "mdf_batch_fetch_scores", "mdf_batch_fetch"):
            getattr(L, name).restype = C.c_int
        _lib = L
        return _lib


EXPORTED_SYMBOLS = [
    "mdf_last_error", "mdf_version", "mdf_ctx_create", "mdf_ctx_destroy", "mdf_ctx_synchronize",
    "mdf_ctx_launch_count", "mdf_ctx_profile", "mdf_ctx_profile_report", "mdf_ctx_set_debug_taps", "mdf_pairwise_sqeuclidean", "mdf_contact_map_dense", "mdf_contact_map_sparse",
    "mdf_align_contact_map", "mdf_cmap_build_transfer", "mdf_model_create", "mdf_model_destroy",
    "mdf_model_set_engine", "mdf_model_get_engine", "mdf_gcn_forward_dense", "mdf_gcn_forward_packed", "mdf_path_forward",
    "mdf_batch_upload", "mdf_batch_destroy", "mdf_path_run", "mdf_path_run_stages", "mdf_path_run_shared",
    "mdf_batch_fetch_scores", "mdf_batch_fetch", "mdf_batch_scores_device", "mdf_batch_unpack_dense", "mdf_batch_invalidate",
    "mdf_cnn_model_create", "mdf_cnn_model_destroy", "mdf_cnn_forward", "mdf_cnn_upload", "mdf_cnn_run", "mdf_cnn_fetch",
    "mdf_cnn_submit_ragged",
    "mdf_path_submit", "mdf_path_submit_ragged", "mdf_path_submit_pairs", "mdf_path_wait", "mdf_cmap_build_transfer_ragged",
    "mdf_batch_upload_pairs", "mdf_batch_fetch_alignment",
    "mdf_pdb_calpha", "mdf_pdb_calpha_batch", "mdf_coords_cache_create", "mdf_coords_cache_open", "mdf_coords_cache_close",
    "mdf_coords_cache_size", "mdf_coords_cache_lookup", "mdf_coords_cache_entry",
    "mdf_nw_align",
    "mdf_model_load", "mdf_cnn_model_load", "mdf_onnx_inspect", "mdf_onnx_tensor", "mdf_model_info",
]


def check(rc: int) -> None:
    if rc == MDF_OK:
        return
    msg = (lib().mdf_last_error() or b"").decode("utf-8", "replace")
    if rc == MDF_EINVAL:
        raise ValueError(msg)
    if rc == MDF_ENOMEM:
        raise MemoryError(msg)
    if rc == MDF_EUNSUPPORTED:
        raise UnsupportedModelError(msg)
    if rc == MDF_ENOENT:
        raise FileNotFoundError(msg)
    if rc == MDF_EPARSE:
        raise RuntimeError(msg)
    raise RuntimeError(msg)


_pyhost = None


def pyhost():
    """The CPython glue module `_mdf_pyhost` (csrc/pyhost.c, built in-tree beside libmdf_b200.so): collects the buffer pointers
    of lists of str / ndarray in C and calls the ragged entry points with the GIL released."""
    global _pyhost
    if _pyhost is None:
        import importlib.machinery
        import importlib.util
        import sysconfig
        path = os.path.join(_HERE, "_mdf_pyhost" + sysconfig.get_config_var("EXT_SUFFIX"))
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: build the extension first (python -c 'import __graft_entry__ as g; g.build()')")
        loader = importlib.machinery.ExtensionFileLoader("_mdf_pyhost", path)
        spec = importlib.util.spec_from_loader("_mdf_pyhost", loader)
        mod = importlib.util.module_from_spec(spec)
        loader.exec_module(mod)
        _pyhost = mod
    return _pyhost


def fn_addr(name: str) -> int:
    return C.cast(getattr(lib(), name), C.c_void_p).value


def inspect_onnx(path: str) -> dict:
    """`mdf_onnx_inspect`: what the library recognises in an `.onnx` file (host only, no GPU needed)."""
    import json
    buf = C.create_string_buffer(1 << 16)
    check(lib().mdf_onnx_inspect(os.fsencode(path), buf, len(buf)))
    return json.loads(buf.value.decode())


def onnx_tensor(path: str, role: str) -> np.ndarray:
    """`mdf_onnx_tensor`: the recognised weight playing `role`, flat float32 (host only)."""
    n = C.c_int64(0)
    check(lib().mdf_onnx_tensor(os.fsencode(path), role.encode(), None, 0, C.byref(n)))
    out = np.empty(n.value, np.float32)
    check(lib().mdf_onnx_tensor(os.fsencode(path), role.encode(), fp(out), n.value, C.byref(n)))
    return out


def packed_row_words(L: int) -> int:
    return ((L + 127) // 128) * 4


def fp(a: np.ndarray):
    return a.ctypes.data_as(c_f32p)


def ip(a: np.ndarray):
    return a.ctypes.data_as(c_i32p)


def up(a: np.ndarray):
    return a.ctypes.data_as(c_u32p)


def lp(a: np.ndarray):
    return a.ctypes.data_as(c_i64p)


class Context:
    """One per (process, device): owns the stream and the HBM workspace arena."""

    def __init__(self, device: Optional[int] = None, stream: Optional[int] = None):
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        self.device = device
        h = C.c_void_p()
        check(lib().mdf_ctx_create(device, None, 0, C.c_void_p(stream) if stream else None, C.byref(h)))
        self.handle = h

    def synchronize(self) -> None:
        check(lib().mdf_ctx_synchronize(self.handle))

    @property
    def launch_count(self) -> int:
        return int(lib().mdf_ctx_launch_count(self.handle))

    def profile(self, enable: bool = True) -> None:
        check(lib().mdf_ctx_profile(self.handle, 1 if enable else 0))

    def set_debug_taps(self, enable: bool = True) -> None:
        check(lib().mdf_ctx_set_debug_taps(self.handle, 1 if enable else 0))

    def profile_report(self):
        """[(stage, milliseconds, algorithmic units)] recorded since profile(True)."""
        buf = C.create_string_buffer(1 << 20)
        check(lib().mdf_ctx_profile_report(self.handle, buf, len(buf)))
        out = []
        for line in buf.value.decode().splitlines():
            name, ms, units = line.split("\t")
            out.append((name, float(ms), float(units)))
        return out

    def close(self) -> None:
        if getattr(self, "handle", None):
            lib().mdf_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_contexts: Dict[int, Context] = {}


def default_context(device: Optional[int] = None) -> Context:
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _contexts:
        _contexts[device] = Context(device)
    return _contexts[device]
