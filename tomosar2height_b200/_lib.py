"""ctypes binding of libt2h.so (the C ABI declared in include/t2h.h).

There is no CPU fallback: if the library is missing, or an op is handed a tensor that is not a
contiguous fp32 CUDA tensor, a RuntimeError is raised.
"""
import ctypes
import os
import shutil
import subprocess
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "libt2h.so")
CSRC = os.path.join(_HERE, "csrc")
SOURCES = ["t2h_topology.cu", "t2h_segment.cu", "t2h_sample.cu", "t2h_scene.cu", "t2h_linear.cu", "t2h_blocks.cu",
           "t2h_eval.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]

_p, _i32, _i64, _sz, _f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_double

# name -> argtypes (every function returns int unless listed in _RESTYPE)
SIGNATURES = {
    "t2h_abi_version": [],
    "t2h_status_string": [_i32],
    "t2h_cell_index": [_p, _i64, _i64, _i32, _p, _p],
    "t2h_xy_keys": [_p, _i64, _i64, _i64, _i32, _i32, _p, _p, _p],
    "t2h_xy_keys_ragged": [_p, _i64, _i64, _p, _i32, _i32, _i32, _p, _p, _p],
    "t2h_index_keys": [_p, _i64, _i64, _i64, _p, _p, _p],
    "t2h_sort_workspace_bytes": [_i64],
    "t2h_sort_by_cell": [_p, _i64, _i64, _p, _sz, _p, _p, _p, _p],
    "t2h_gather_rows": [_p, _p, _i64, _i32, _p, _p],
    "t2h_scatter_rows": [_p, _p, _i64, _i32, _p, _p],
    "t2h_seg_workspace_bytes": [_i64, _i64, _i32],
    "t2h_seg_max_fwd": [_p, _i64, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _sz, _p, _p, _p, _p],
    "t2h_seg_max_bwd": [_p, _p, _i64, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p, _sz, _p, _p],
    "t2h_seg_reduce_fwd": [_p, _i64, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _i32, _p, _sz, _p, _p],
    "t2h_seg_broadcast": [_p, _i64, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p],
    "t2h_seg_broadcast_add": [_p, _p, _i64, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p, _p],
    "t2h_seg_mean_fwd": [_p, _i64, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _sz, _p, _p],
    "t2h_seg_mean_bwd": [_p, _i64, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p],
    "t2h_bilinear_sample_fwd": [_p, _i32, _i32, _p, _i64, _p, _p, _i64, _i64, _p, _p],
    "t2h_bilinear_sample_bwd_workspace_bytes": [_i32, _i32, _i64, _i64, _i32],
    "t2h_bilinear_sample_bwd": [_p, _i64, _i32, _i32, _p, _i64, _p, _p, _p, _i64, _i32, _i32, _p, _sz, _p, _p],
    "t2h_tile_count": [_p, _p, _i64, _p, _f64, _p, _p, _p],
    "t2h_tile_write": [_p, _p, _i64, _p, _f64, _f64, _p, _p, _p, _p],
    "t2h_blend_accumulate": [_p, _i32, _i32, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p],
    "t2h_raster_windows": [_p, _i32, _i64, _i64, _p, _p, _i32, _i32, _p, _p, _p, _p],
    "t2h_residual_stats_workspace_bytes": [_i64, _i32],
    "t2h_residual_stats": [_p, _p, _i64, _p, _i32, _i32, _f64, _p, _sz, _p, _p, _p],
    "t2h_upsample_bilinear_fwd": [_p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p],
    "t2h_upsample_bilinear_bwd": [_p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p],
    "t2h_split_tf32": [_p, _i64, _p, _p, _p],
    "t2h_linear_wgrad_workspace_bytes": [_i64, _i32, _i32],
    "t2h_linear_wgrad": [_p, _i64, _p, _i64, _i64, _i32, _i32, _i32, _p, _sz, _p, _i64, _p, _p],
    "t2h_conv3x3_fwd": [_p, _i32, _i32, _i32, _i32, _p, _p, _i32, _p, _i32, _p, _p, _p, _p],
    "t2h_conv3x3_wgrad_workspace_bytes": [_i32, _i32, _i32, _i32, _i32],
    "t2h_conv3x3_wgrad": [_p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _sz, _p, _p, _p],
    "t2h_colsum_workspace_bytes": [_i64, _i32],
    "t2h_colsum": [_p, _i64, _i64, _i32, _p, _sz, _p, _p],
    "t2h_resblock_workspace_bytes": [_i64, _i32, _i32, _i32, _i32, _i32],
    "t2h_resblock_fwd": [_p, _i64, _i32, _p, _i64, _i32, _i64, _p, _p, _i32, _p, _p, _p, _i32, _p, _sz, _p, _i64, _p, _i64, _p],
    "t2h_resblock_bwd": [_p, _i64, _p, _i64, _i32, _p, _i64, _i32, _p, _i64, _i64, _p, _i32, _p, _p, _i32, _p, _sz,
                         _p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p],
    "t2h_comm_mlp_workspace_bytes": [_i64, _i32, _i32],
    "t2h_comm_mlp_fwd": [_p, _i64, _i32, _p, _i64, _i32, _i64, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _i64, _p, _i64, _p],
    "t2h_comm_mlp_bwd": [_p, _i64, _p, _i64, _i32, _p, _i64, _i32, _p, _i64, _i64, _p, _p, _p, _p, _sz,
                         _p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _p],
    "t2h_linear_fwd": [_p, _i64, _i32, _p, _i64, _i32, _i64, _p, _p, _i32, _p, _i32, _p, _i64, _p, _i64, _p, _i64, _p],
    "t2h_linear_wgrad_f16": [_p, _i64, _p, _p, _i64, _p, _i64, _i32, _i32, _i32, _p, _sz, _p, _i64, _p, _p],
    "t2h_conv3x3_fwd_f16": [_p, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _i32, _p, _i32, _p, _p, _p, _p, _p],
    "t2h_conv3x3_wgrad_f16": [_p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _sz, _p, _p, _p],
    "t2h_add_absmax": [_p, _p, _i64, _p, _p, _p],
    "t2h_absmax": [_p, _i64, _i32, _p, _i64, _i32, _i64, _p, _p],
    "t2h_split_f16": [_p, _i64, _p, _p, _p, _p],
    "t2h_linear_fwd_f16": [_p, _i64, _i32, _p, _i64, _i32, _i64, _p, _p, _p, _p, _i32, _p, _i32, _p, _i64, _p, _i64, _p,
                           _i64, _p, _p],
}
_RESTYPE = {"t2h_status_string": ctypes.c_char_p, "t2h_sort_workspace_bytes": _sz,
            "t2h_linear_wgrad_workspace_bytes": _sz, "t2h_colsum_workspace_bytes": _sz,
            "t2h_conv3x3_wgrad_workspace_bytes": _sz, "t2h_bilinear_sample_bwd_workspace_bytes": _sz,
            "t2h_seg_workspace_bytes": _sz, "t2h_resblock_workspace_bytes": _sz,
            "t2h_comm_mlp_workspace_bytes": _sz, "t2h_residual_stats_workspace_bytes": _sz}

_lib = None
_lock = threading.Lock()
launch_count = 0  # kernels-launching C calls made through this binding (bench.py reports it)


def _nvcc() -> str:
    """nvcc from PATH, else from the CUDA toolkit named by CUDA_HOME / CUDA_PATH (default /usr/local/cuda)."""
    home = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    return shutil.which("nvcc") or os.path.join(home, "bin", "nvcc")


def build_library(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libt2h.so (in-tree, next to the package that loads it)."""
    nvcc = _nvcc()
    build_dir = os.path.join(_ROOT, "build")
    os.makedirs(build_dir, exist_ok=True)
    objects = []
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    headers.append(os.path.join(_ROOT, "include", "t2h.h"))
    newest_header = max(os.path.getmtime(h) for h in headers)
    procs = []
    for src in SOURCES:
        src_path = os.path.join(CSRC, src)
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        objects.append(obj)
        if os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src_path), newest_header):
            continue
        cmd = [nvcc, *NVCC_FLAGS, "-I", os.path.join(_ROOT, "include"), "-I", CSRC, "-c", src_path, "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, proc in procs:
        out, _ = proc.communicate()
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    stale = not os.path.exists(LIB_PATH) or any(os.path.getmtime(o) > os.path.getmtime(LIB_PATH) for o in objects)
    if procs or stale:
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH, *objects]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}")
    global _lib
    _lib = None
    return LIB_PATH


def load():
    """dlopen libt2h.so and declare every symbol of include/t2h.h.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the sm_100a extension has not been built "
                "(run `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
            fn.argtypes = argtypes
            fn.restype = _RESTYPE.get(name, ctypes.c_int)
        _lib = lib
    return _lib


_seen = threading.local()  # device of the tensors handed to the pending call


def ptr(t):
    """raw device pointer of a tensor argument (None -> NULL); remembers the tensor's device for ``call``"""
    if t is None:
        return None
    if t.is_cuda:
        _seen.device = t.device.index
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def check(status: int, op: str):
    if status != 0:
        msg = load().t2h_status_string(status).decode()
        raise RuntimeError(f"{op} failed: {msg} (status {status})")


def call(name: str, *args):
    """Invoke a status-returning entry point on the current stream; raise RuntimeError on failure."""
    global launch_count
    launch_count += 1
    # kernels are enqueued on the current stream of the CURRENT device: tensors living elsewhere would be touched by
    # the wrong GPU (and per-device kernel attributes would be missing) -- fail loudly instead
    dev = getattr(_seen, "device", None)
    _seen.device = None
    if dev is not None and dev != torch.cuda.current_device():
        raise RuntimeError(f"{name}: tensors live on cuda:{dev} but the current device is cuda:{torch.cuda.current_device()}; "
                           f"run the model under torch.cuda.device({dev}) (one process per GPU)")
    check(getattr(load(), name)(*args, stream()), name)


def require_cuda_f32(t: torch.Tensor, what: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{what}: expected a CUDA tensor (the B200 path has no CPU fallback)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"{what}: expected float32, got {t.dtype}")
    return t
