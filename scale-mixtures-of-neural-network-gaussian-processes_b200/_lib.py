"""ctypes binding of libsmnngp.so (C-ABI declared in include/smnngp.h) + the in-tree nvcc build.

There is no CPU fallback: if the library cannot be built / loaded every op raises.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsmnngp.so")
SOURCES = ["gram.cu", "chol.cu", "reduce.cu", "api.cu", "stages.cu", "draws.cu", "grad.cu", "peer.cu", "exchange.cu",
           "context.cu", "trtri.cu", "multigpu.cu", "grid_batch.cu",
           "grad_batch.cu", "test_nll_batch.cu", "mixture.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Wno-deprecated-gpu-targets"]

EXPORTS = [
    "smnngp_abi_version", "smnngp_last_error", "smnngp_gram_workspace_bytes", "smnngp_gram_f64",
    "smnngp_nngp_diag_f64", "smnngp_potrf_workspace_bytes", "smnngp_potrf_f64", "smnngp_potrf_trapezoid_f64",
    "smnngp_cov_solve_workspace_bytes", "smnngp_cov_solve_f64",
    "smnngp_lml_workspace_bytes", "smnngp_lml_f64", "smnngp_lml_grad_workspace_bytes", "smnngp_lml_grad_f64",
    "smnngp_lml_grad_host_f64", "smnngp_predict_workspace_bytes", "smnngp_predict_f64", "smnngp_predict_cov_f64",
    "smnngp_test_nll_f64", "smnngp_lml_host_f64", "smnngp_predict_host_f64", "smnngp_test_nll_host_f64",
    "smnngp_host_release", "smnngp_set_panel_width", "smnngp_set_tile_variant", "smnngp_debug_occupancy", "smnngp_set_lookahead", "smnngp_set_fused_panel", "smnngp_set_tail_cols", "smnngp_set_gram_super_rows", "smnngp_set_lookahead_reserve", "smnngp_debug_potf2_clocks",
    "smnngp_sample_f_iid_f64", "smnngp_draw_metrics_f64",
    "smnngp_grid_base_f64", "smnngp_grid_workspace_bytes", "smnngp_grid_point_f64",
    "smnngp_grid_batch_workspace_bytes", "smnngp_grid_batch_f64",
    "smnngp_lml_grad_batch_workspace_bytes", "smnngp_lml_grad_batch_f64",
    "smnngp_test_nll_batch_workspace_bytes", "smnngp_test_nll_batch_f64",
    "smnngp_scale_draws_f64", "smnngp_mixture_nll_f64",
    "smnngp_stage_qtable_f64", "smnngp_stage_gram_f64", "smnngp_stage_factor_diag_f64", "smnngp_stage_trsm_f64",
    "smnngp_stage_update_f64", "smnngp_stage_sumsq_f64", "smnngp_stage_lml_finalize_f64",
    "smnngp_stage_predict_finalize_f64", "smnngp_stage_test_nll_finalize_f64",
    "smnngp_stage_factor_diag_inv_f64", "smnngp_stage_scatter_inverse_f64", "smnngp_stage_signal_f64",
    "smnngp_stage_wait_flags_f64", "smnngp_stage_trsm_scatter_f64", "smnngp_set_peer_wait_mode",
    "smnngp_stage_push_panel_f64",
    "smnngp_peer_alloc", "smnngp_peer_open", "smnngp_peer_close", "smnngp_peer_free",
    "smnngp_instr_reset", "smnngp_instr_launches", "smnngp_instr_updates", "smnngp_dmma_peak_tflops",
    "smnngp_stage_assemble_inverse_f64", "smnngp_stage_update2_f64", "smnngp_stage_trsm_scatter2_f64",
    "smnngp_mg_create", "smnngp_mg_destroy", "smnngp_mg_ipc_handle", "smnngp_mg_region", "smnngp_mg_connect_ipc",
    "smnngp_mg_connect_ptrs", "smnngp_mg_connect_emulated", "smnngp_mg_set_timeout", "smnngp_mg_set_sm_reserve", "smnngp_mg_set_reserve_margin",
    "smnngp_mg_timeline", "smnngp_mg_timeline_read", "smnngp_mg_last_error", "smnngp_mg_layout", "smnngp_lml_mg_f64",
    "smnngp_mg_create_predict", "smnngp_predict_mg_f64", "smnngp_test_nll_mg_f64",
    "smnngp_mg_create_grad", "smnngp_lml_grad_mg_f64",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libsmnngp.so (no CPU fallback exists)")
    return exe


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(_HERE, "..", "include", "smnngp.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into lib/libsmnngp.so (cross-compiles without a GPU).  Safe to call from every
    rank of a torchrun job at once: an exclusive file lock serialises the builders, the staleness check is repeated
    under the lock (only the first rank compiles) and the library is moved into place atomically."""
    if not force and not _stale():
        return LIB_PATH
    import fcntl
    nvcc = _nvcc()
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(_HERE, "build")
    os.makedirs(obj_dir, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():
                return LIB_PATH

            def cc(src):
                obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
                cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("SMNNGP_NVCC_FLAGS", "").split(), "-c",
                       os.path.join(CSRC, src), "-o", obj]
                if verbose:
                    cmd.insert(1, "-Xptxas=-v")
                r = subprocess.run(cmd, capture_output=True, text=True)
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
                if verbose:
                    print(r.stderr)
                return obj

            with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
                objs = list(ex.map(cc, SOURCES))
            tmp = LIB_PATH + f".tmp{os.getpid()}"
            # the -gencode on the link line keeps nvcc's device-link stub at sm_100a too (default: sm_52)
            r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp, *objs,
                                "-lcudart"], capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
            os.replace(tmp, LIB_PATH)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


XLA_LIB_PATH = os.path.join(LIB_DIR, "libsmnngp_xla.so")


def build_xla_shim(force: bool = False) -> str:
    """Compile csrc/xla_ffi_c_shim.c (XLA FFI handlers over the C-ABI, plain-C call-frame level) into
    lib/libsmnngp_xla.so with gcc.  Without jaxlib it is built against the locally re-declared subset of
    xla/ffi/api/c_api.h (csrc/xla_ffi_min/); with SMNNGP_XLA_FFI_INCLUDE=<jaxlib include dir> against the real header."""
    src = os.path.join(CSRC, "xla_ffi_c_shim.c")
    deps = [src, os.path.join(CSRC, "xla_ffi_min", "c_api_subset.h"), os.path.join(_HERE, "..", "include", "smnngp.h")]
    if not force and os.path.exists(XLA_LIB_PATH) and all(os.path.getmtime(d) <= os.path.getmtime(XLA_LIB_PATH) for d in deps):
        return XLA_LIB_PATH
    build()
    cmd = ["gcc", "-O2", "-std=c11", "-Wall", "-Werror", "-fPIC", "-shared", src, "-I", CSRC]
    real = os.environ.get("SMNNGP_XLA_FFI_INCLUDE")
    if real:
        cmd += ["-DSMNNGP_USE_REAL_XLA_FFI", "-I", real]
    tmp = XLA_LIB_PATH + f".tmp{os.getpid()}"
    cmd += ["-L", LIB_DIR, "-lsmnngp", "-Wl,-rpath,$ORIGIN", "-o", tmp]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"gcc failed on xla_ffi_c_shim.c:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, XLA_LIB_PATH)
    return XLA_LIB_PATH


_lib = None

_vp, _i64, _i, _d, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_size_t


def _declare(lib):
    lib.smnngp_abi_version.restype = _i
    lib.smnngp_last_error.restype = C.c_char_p
    lib.smnngp_gram_workspace_bytes.restype = _sz
    lib.smnngp_gram_workspace_bytes.argtypes = [_i64, _i64, _i, _i]
    lib.smnngp_gram_f64.argtypes = [_vp, _vp, _vp, _i64, _i64, _i64, _i, _i, _i, _vp, _i, _i, _vp, _i64, _vp, _sz]
    lib.smnngp_nngp_diag_f64.argtypes = [_vp, _vp, _i64, _i64, _i, _i, _i, _vp, _vp, _vp, _sz]
    lib.smnngp_potrf_workspace_bytes.restype = _sz
    lib.smnngp_potrf_workspace_bytes.argtypes = [_i64]
    lib.smnngp_potrf_f64.argtypes = [_vp, _vp, _i64, _i64, _vp, _vp, _sz]
    lib.smnngp_potrf_trapezoid_f64.argtypes = [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _sz]
    lib.smnngp_cov_solve_workspace_bytes.restype = _sz
    lib.smnngp_cov_solve_workspace_bytes.argtypes = [_i64]
    lib.smnngp_cov_solve_f64.argtypes = [_vp, _vp, _i64, _i64, _vp, _d, _d, _vp, _sz, _vp, _vp]
    lib.smnngp_lml_workspace_bytes.restype = _sz
    lib.smnngp_lml_workspace_bytes.argtypes = [_i64, _i64, _i, _i]
    lib.smnngp_lml_f64.argtypes = [_vp, _vp, _vp, _i64, _i64, _i, _i, _i, _vp, _i, _vp, _sz, _vp, _vp]
    lib.smnngp_lml_grad_workspace_bytes.restype = _sz
    lib.smnngp_lml_grad_workspace_bytes.argtypes = [_i64, _i64, _i, _i]
    lib.smnngp_lml_grad_f64.argtypes = [_vp, _vp, _vp, _i64, _i64, _i, _i, _i, _vp, _i, _vp, _sz, _vp, _vp, _vp]
    lib.smnngp_lml_grad_host_f64.argtypes = [_vp, _vp, _i64, _i64, _i, _i, _i, _vp, _i, _vp, _vp, _vp]
    lib.smnngp_predict_workspace_bytes.restype = _sz
    lib.smnngp_predict_workspace_bytes.argtypes = [_i64, _i64, _i64, _i64, _i, _i]
    lib.smnngp_predict_f64.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i, _i, _i, _vp, _i, _vp, _sz,
                                       _vp, _vp, _vp]
    lib.smnngp_predict_cov_f64.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i, _i, _i, _vp, _i, _vp,
                                           _sz, _vp, _vp, _vp, _i64, _vp]
    lib.smnngp_test_nll_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i, _i, _i, _vp, _i, _d, _d,
                                        _vp, _sz, _vp, _vp, _vp, _vp, _vp]
    lib.smnngp_lml_host_f64.argtypes = [_vp, _vp, _i64, _i64, _i, _i, _i, _vp, _i, _vp, _vp]
    lib.smnngp_predict_host_f64.argtypes = [_vp, _vp, _vp, _i64, _i64, _i64, _i64, _i, _i, _i, _vp, _i, _vp, _vp,
                                            _vp]
    lib.smnngp_test_nll_host_f64.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i, _i, _i, _vp, _i, _d, _d,
                                             _vp, _vp, _vp, _vp]
    lib.smnngp_host_release.restype = None
    lib.smnngp_set_panel_width.restype = None
    lib.smnngp_set_panel_width.argtypes = [_i]
    lib.smnngp_set_tile_variant.restype = None
    lib.smnngp_set_tile_variant.argtypes = [_i]
    lib.smnngp_debug_occupancy.argtypes = [_i]
    lib.smnngp_debug_potf2_clocks.restype = None
    lib.smnngp_debug_potf2_clocks.argtypes = [_vp]
    lib.smnngp_set_lookahead_reserve.restype = None
    lib.smnngp_set_lookahead_reserve.argtypes = [_i, _i]
    lib.smnngp_set_lookahead.restype = None
    lib.smnngp_set_lookahead.argtypes = [_i]
    lib.smnngp_set_fused_panel.restype = None
    lib.smnngp_set_fused_panel.argtypes = [_i]
    lib.smnngp_set_tail_cols.restype = None
    lib.smnngp_set_tail_cols.argtypes = [_i64]
    lib.smnngp_set_gram_super_rows.restype = None
    lib.smnngp_set_gram_super_rows.argtypes = [_i, _i64]
    lib.smnngp_grid_base_f64.argtypes = [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _vp]
    lib.smnngp_grid_workspace_bytes.restype = _sz
    lib.smnngp_grid_workspace_bytes.argtypes = [_i64, _i64, _i, _i]
    lib.smnngp_grid_point_f64.argtypes = [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _i64, _i, _i, _i, _vp, _vp,
                                          _sz, _vp, _vp, _vp, _vp]
    lib.smnngp_grid_batch_workspace_bytes.restype = _sz
    lib.smnngp_grid_batch_workspace_bytes.argtypes = [_i64, _i64, _i, _i, _i64]
    lib.smnngp_grid_batch_f64.argtypes = [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _i64, _i64, _i, _i, _i, _vp,
                                          _vp, _sz, _vp, _vp, _vp, _vp]
    lib.smnngp_lml_grad_batch_workspace_bytes.restype = _sz
    lib.smnngp_lml_grad_batch_workspace_bytes.argtypes = [_i64, _i, _i, _i64]
    lib.smnngp_lml_grad_batch_f64.argtypes = [_vp, _vp, _i64, _vp, _vp, _i64, _i64, _i, _i, _i, _vp, _i, _vp, _sz,
                                              _vp, _vp, _vp]
    lib.smnngp_test_nll_batch_workspace_bytes.restype = _sz
    lib.smnngp_test_nll_batch_workspace_bytes.argtypes = [_i64, _i64, _i, _i, _i64]
    lib.smnngp_test_nll_batch_f64.argtypes = [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i, _i,
                                              _i, _vp, _i, _d, _d, _vp, _sz, _vp, _vp, _vp, _vp, _vp]
    lib.smnngp_scale_draws_f64.argtypes = [_vp, _i, _vp, _i64, _i64, C.c_uint64, _vp]
    lib.smnngp_mixture_nll_f64.argtypes = [_vp, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _i64, _vp, _i64, _i64, _d, _d,
                                           _vp, _vp, _vp, _vp]
    lib.smnngp_sample_f_iid_f64.argtypes = [_vp, _vp, _vp, _i, _i64, _i64, _i64, _vp, _i, C.c_uint64, _vp]
    lib.smnngp_draw_metrics_f64.argtypes = [_vp, _vp, _vp, _i, _vp, _i64, _i64, _i64, _vp, _i, C.c_uint64, _vp, _vp, _vp]
    lib.smnngp_stage_qtable_f64.argtypes = [_vp, _vp, _i64, _i64, _i, _i, _i, _vp, _vp, _i64, _vp, _vp]
    lib.smnngp_stage_gram_f64.argtypes = [_vp, _vp, _i64, _vp, _i64, _i64, _i, _i, _i, _vp, _vp, _i64, _vp, _i64, _vp,
                                          _i, _i, _vp, _i64]
    lib.smnngp_stage_factor_diag_f64.argtypes = [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _i64]
    lib.smnngp_stage_trsm_f64.argtypes = [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp]
    lib.smnngp_stage_update_f64.argtypes = [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _i64, _i, _i64, _i64,
                                            _i64, _i]
    lib.smnngp_stage_sumsq_f64.argtypes = [_vp, _vp, _i64, _vp]
    lib.smnngp_stage_test_nll_finalize_f64.argtypes = [_vp, _vp, _vp, _vp, _i64, _i64, _d, _d, _vp, _i, _vp, _vp, _vp,
                                                       _vp]
    lib.smnngp_stage_predict_finalize_f64.argtypes = [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _vp]
    lib.smnngp_stage_lml_finalize_f64.argtypes = [_vp, _vp, _vp, _i, _i64, _vp, _vp]
    _u64, _u = C.c_uint64, C.c_int
    lib.smnngp_stage_factor_diag_inv_f64.argtypes = [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _i64]
    lib.smnngp_stage_scatter_inverse_f64.argtypes = [_vp, _vp, _i64, _i64, _vp, _i, _i64, _vp, _i64, _u64, _vp]
    lib.smnngp_stage_signal_f64.argtypes = [_vp, _vp, _i, _i64, _u64]
    lib.smnngp_stage_wait_flags_f64.argtypes = [_vp, _vp, _i64, _i, _u64, _d, _vp]
    lib.smnngp_stage_trsm_scatter_f64.argtypes = [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _i, _i,
                                                  _i64, _i64, _i64, _i64, _i64, _vp, _i64, _u64, _vp]
    lib.smnngp_stage_push_panel_f64.argtypes = [_vp, _vp, _i64, _i64, _i64, _i, _i, _i64, _i64, _i64, _vp, _vp, _i64,
                                                _u64]
    lib.smnngp_set_peer_wait_mode.restype = None
    lib.smnngp_set_peer_wait_mode.argtypes = [_i]
    lib.smnngp_peer_alloc.argtypes = [_sz, _vp, _vp]
    lib.smnngp_peer_open.argtypes = [_vp, _vp]
    lib.smnngp_peer_close.argtypes = [_vp]
    lib.smnngp_peer_free.argtypes = [_vp]
    lib.smnngp_stage_assemble_inverse_f64.argtypes = [_vp, _vp, _i64, _i64, _vp, _vp, _i, _i64, _vp, _i64, _u64, _vp]
    lib.smnngp_mg_create.argtypes = [_vp, _i, _i, _i64, _i64]
    lib.smnngp_mg_destroy.argtypes = [_vp]
    lib.smnngp_mg_ipc_handle.argtypes = [_vp, _vp]
    lib.smnngp_mg_region.restype = _vp
    lib.smnngp_mg_region.argtypes = [_vp]
    lib.smnngp_mg_connect_ipc.argtypes = [_vp, _vp]
    lib.smnngp_mg_connect_ptrs.argtypes = [_vp, _vp, _vp]
    lib.smnngp_mg_connect_emulated.argtypes = [_vp]
    lib.smnngp_mg_set_timeout.restype = None
    lib.smnngp_mg_set_timeout.argtypes = [_vp, _d]
    lib.smnngp_mg_set_reserve_margin.restype = None
    lib.smnngp_mg_set_reserve_margin.argtypes = [_vp, _d]
    lib.smnngp_mg_set_sm_reserve.restype = None
    lib.smnngp_mg_set_sm_reserve.argtypes = [_vp, _i]
    lib.smnngp_mg_timeline.restype = None
    lib.smnngp_mg_timeline.argtypes = [_vp, _i]
    lib.smnngp_mg_timeline_read.argtypes = [_vp, _i, _vp, _vp, _vp]
    lib.smnngp_mg_last_error.restype = C.c_char_p
    lib.smnngp_mg_layout.restype = _i64
    lib.smnngp_mg_layout.argtypes = [_i, _i64, _i64, _i64, _i, _vp, _vp]
    lib.smnngp_lml_mg_f64.argtypes = [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp, _i, _i, _vp, _vp]
    lib.smnngp_mg_create_predict.argtypes = [_vp, _i, _i, _i64, _i64, _i64, _i64]
    lib.smnngp_mg_create_grad.argtypes = [_vp, _i, _i, _i64, _i64]
    lib.smnngp_lml_grad_mg_f64.argtypes = [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp, _i, _vp, _vp, _vp]
    lib.smnngp_predict_mg_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp, _i, _vp, _vp, _vp]
    lib.smnngp_test_nll_mg_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp, _i, _d, _d, _vp,
                                           _vp, _vp, _vp]
    lib.smnngp_instr_reset.restype = None
    lib.smnngp_instr_reset.argtypes = [_i]
    lib.smnngp_instr_launches.restype = C.c_longlong
    lib.smnngp_instr_updates.argtypes = [_vp, _vp]
    lib.smnngp_dmma_peak_tflops.restype = _d
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ("smnngp_abi_version",):
            fn.restype = _i


def load():
    """Return the loaded library; builds it on first use when the .so is missing or stale."""
    global _lib
    if _lib is not None:
        return _lib
    path = LIB_PATH
    if _stale():
        path = build()
    lib = C.CDLL(path)
    _declare(lib)
    if lib.smnngp_abi_version() != 1:
        raise RuntimeError("libsmnngp.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().smnngp_last_error().decode()
        raise RuntimeError(f"libsmnngp {what} failed (status {rc}): {msg}")
