"""Build and bind libltgan.so -- the C-ABI shared library declared in include/ltgan.h.

The library is compiled in-tree with nvcc for sm_100a only and loaded with ctypes; there is no
fallback path: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_ROOT = os.path.dirname(_HERE)
_INCLUDE = os.path.join(_ROOT, "include")
# experiments: LTG_LIB_SUFFIX=_x LTG_NVCC_EXTRA="-DFOO=1" builds and loads libltgan_x.so beside the product library
_SUFFIX = os.environ.get("LTG_LIB_SUFFIX", "")
LIB_PATH = os.path.join(_HERE, "libltgan%s.so" % _SUFFIX)

SOURCES = ["runtime.cu", "gemm_ops.cu", "vae_kernels.cu", "adam_kernels.cu", "sampler_kernels.cu", "disc_kernels.cu",
           "topk_kernels.cu", "mid_kernels.cu", "mid_tc.cu", "disc_fused.cu", "peer_kernels.cu", "ingest.cu", "tables.cu"]
HEADERS = ["ltg_common.cuh", "gemm_sm100.cuh"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-I", _INCLUDE]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ for sm_100a and link libltgan.so (no GPU needed: nvcc cross-compiles). Safe to call from
    several processes at once (torchrun ranks): the build runs under an exclusive file lock and the library is moved into place
    atomically; the other ranks find it up to date when they get the lock."""
    srcs = [os.path.join(_CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(_CSRC, h) for h in HEADERS] + [os.path.join(_INCLUDE, "ltgan.h")]

    def fresh():
        return os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= _newest(deps)
    if not force and fresh():
        return LIB_PATH
    import fcntl
    objdir = os.path.join(_HERE, "build" + _SUFFIX)
    os.makedirs(objdir, exist_ok=True)
    with open(os.path.join(objdir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and fresh():
                return LIB_PATH
            return _build_locked(srcs, objdir, force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(srcs, objdir, force, verbose):
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        hdr_deps = [os.path.join(_CSRC, h) for h in HEADERS] + [os.path.join(_INCLUDE, "ltgan.h")]
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= _newest([src] + hdr_deps):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + os.environ.get("LTG_NVCC_EXTRA", "").split() + ["-c", src, "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    tmp = LIB_PATH + ".tmp.%d" % os.getpid()
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


# ---------------------------------------------------------------------------------------------
# ctypes signatures (mirror of include/ltgan.h)
# ---------------------------------------------------------------------------------------------
_P = ctypes.c_void_p
_I = ctypes.c_int
_I64 = ctypes.c_int64
_U64 = ctypes.c_uint64
_U32 = ctypes.c_uint32
_F = ctypes.c_float

SIGNATURES = {
    "ltg_last_error": (ctypes.c_char_p, []),
    "ltg_version": (_I, []),
    "ltg_init": (_I, []),
    "ltg_step_advance": (_I, [_P, _P, _I, _F, _F, _F, _F, _F, _P, _I64, _P, _P]),
    "ltg_step_advance3": (_I, [_P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _I64, _P, _I64, _P, _I64, _P, _P, _P, _P]),
    "ltg_gemm_bf16": (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P, _I, _P, _I, _P, _I, _F, _I, _F, _U64, _U32, _U32, _P, _I,
                           _I, _P, _P, _I, _F, _I64, _P]),
    "ltg_enc_gather_fwd": (_I, [_P, _P, _P, _I, _I, _I64, _P, _P, _F, _U64, _U32, _P, _P, _I, _P, _I, _P, _P, _P, _P, _I, _P, _I, _P]),
    "ltg_enc_gather_partial": (_I, [_P, _P, _I, _I, _I, _I64, _P, _P, _F, _U64, _U32, _P, _P, _P, _I, _P, _P, _I, _P]),
    "ltg_bias_tanh": (_I, [_P, _I, _P, _I, _I, _P, _I, _P]),
    "ltg_enc_coef_scatter": (_I, [_P, _P, _P, _P, _P, _I, _I, _F, _U64, _U32, _P, _P, _I, _P]),
    "ltg_latent_fwd": (_I, [_P, _P, _I, _I64, _F, _U64, _U32, _P, _P, _I, _P, _P, _P]),
    "ltg_latent_bwd": (_I, [_P, _P, _P, _I, _I, _F, _P, _P, _I, _P, _P]),
    "ltg_vae_mid_fwd": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _I64, _F, _U64, _U32, _P, _P, _P, _I, _P, _P, _I, _P, _P]),
    "ltg_vae_mid_bwd": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P]),
    "ltg_vae_mid_fwd_tc": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _I64, _F, _U64, _U32, _P, _P, _P, _I, _P, _P, _I, _P, _P]),
    "ltg_vae_mid_bwd_tc": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P]),
    "ltg_tanh_bwd": (_I, [_P, _I, _I, _I64, _P, _I, _I, _I, _P, _I, _P, _I, _P, _P]),
    "ltg_dec_logits_nblk": (_I, [_I, _I]),
    "ltg_dec_logits_fwd": (_I, [_P, _I, _P, _P, _I, _I, _P, _I, _P, _P]),
    "ltg_dec_row_stats": (_I, [_P, _I, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ltg_dec_probs": (_I, [_P, _I, _P, _I, _I, _P, _I, _P]),
    "ltg_dec_dlogits": (_I, [_P, _I, _P, _P, _P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ltg_adam": (_I, [_P, _P, _P, _P, _I, _I64, _P, _I64, _F, _P, _F, _F, _F, _P]),
    "ltg_enc_wgrad_compact": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _P]),
    "ltg_enc_adam": (_I, [_P, _P, _P, _P, _I, _P, _P, _F, _P, _F, _F, _F, _I, _P]),
    "ltg_sum_partials": (_I, [_P, _I, _I64, _I64, _P, _P]),
    "ltg_enc_coef_clear": (_I, [_P, _P, _I, _P, _I, _P]),
    "ltg_enc_xc_clear": (_I, [_P, _P, _I, _I, _P, _P, _I, _P]),
    "ltg_enc_wgrad_expand": (_I, [_P, _I, _P, _P, _P]),
    "ltg_sample_pairs": (_I, [_P, _I, _I, _I, _I64, _P, _P, _P, _P, _P, _P, _U64, _U32, _P, _P, _P, _P, _P, _I, _P, _P]),
    "ltg_sample_pairs_vals": (_I, [_P, _I, _P, _I, _I, _I64, _P, _P, _P, _P, _P, _P, _U64, _U32, _P, _P, _P, _P, _P, _I, _P, _P]),
    "ltg_dec_row_bwd": (_I, [_P, _I, _P, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ltg_wgrad_adam": (_I, [_P, _I, _P, _I, _I, _I, _I, _P, _P, _P, _P, _I, _I, _I, _P, _F, _P, _F, _F, _F, _P]),
    "ltg_peer_barrier": (_I, [_P, _I, _I, _I, _P, _P]),
    "ltg_peer_allreduce_small": (_I, [_P, _I64, _I, _P, _I, _I, _I, _P, _P]),
    "ltg_peer_reduce": (_I, [_P, _P, _I64, _I64, _I, _P, _P]),
    "ltg_peer_push": (_I, [_P, _I64, _P, _P, _I64, _I, _P]),
    "ltg_adam_peer": (_I, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I, _F, _P, _F, _F, _F, _P]),
    "ltg_enc_adam_peer": (_I, [_P, _P, _P, _P, _P, _I64, _I, _P, _P, _I, _F, _P, _F, _F, _F, _P]),
    "ltg_disc_gather": (_I, [_P, _P, _P, _I, _P, _P, _P]),
    "ltg_disc_fused_supported": (_I, [_I, _I, _I, _I, _I, _I, _I, _I]),
    "ltg_disc_fwd_fused": (_I, [_P, _P, _I, _I, _P, _I, _P, _I, _I, _P, _I, _I, _I, _I, _P, _P, _P, _F, _U64, _U32, _U32, _P, _P, _P, _P, _P, _P, _P, _P,
                                _I, _P]),
    "ltg_disc_fused_set_trace": (_I, [_P]),
    "ltg_disc_head": (_I, [_P, _I, _I, _I, _P, _P, _P, _F, _P, _P, _P, _P, _P, _P]),
    "ltg_topk_metrics": (_I, [_P, _I, _I64, _I, _I, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _P]),
    "ltg_topk_recommend": (_I, [_P, _I64, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P]),
    "ltg_cast_bf16": (_I, [_P, _I64, _P, _I64, _I64, _I64, _P]),
    "ltg_csv_open": (_I, [_P, _P, _P, _I, _P, _P]),
    "ltg_csv_pairs": (_I, [_P, _P, _P]),
    "ltg_csv_to_csr": (_I, [_P, _I64, _I64, _I64, _I, _P, _P, _P, _P]),
    "ltg_csv_close": (_I, [_P]),
    "ltg_cand_sets": (_I, [_P, _P, _I, _P, _P, _I, _P, _I, _P, _P, _P, _I64, _I, _P, _P, _P]),
    "ltg_real_pairs": (_I, [_P, _P, _I, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I64, _I, _P, _P, _P]),
}

_lib = None


def load():
    """Load libltgan.so (building it first if the sources are newer). Raises if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    build()   # no-op when libltgan.so is newer than every source (mtime check), so an edited kernel is never loaded stale
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: loud by design
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class LtgError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = load().ltg_last_error()
        raise LtgError("libltgan call failed (rc=%d): %s" % (rc, msg.decode() if msg else "?"))


def ptr(t):
    """Device (or host) pointer of a torch tensor / numpy array, None -> NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    if hasattr(t, "ctypes"):
        return t.ctypes.data
    return int(t)
