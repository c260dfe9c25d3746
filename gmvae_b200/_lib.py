"""ctypes binding of libgmvae_b200.so (include/gmvae_abi.h).  No CPU fallback: if the shared
library cannot be loaded the import of the product fails loudly."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

MAX_HIDDEN = 8
NAME_LEN = 64
ABI_VERSION = 1
MODEL_IDS = {"vae": 0, "vae_gmp": 1, "gmvae": 2}
OBJECTIVE_IDS = {"reference": 0, "marginal": 1}
PRECISION_IDS = {"fp32": 0, "bf16": 1}


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("model", C.c_int32), ("objective", C.c_int32), ("precision", C.c_int32),
        ("data_size", C.c_int32), ("latent_size", C.c_int32), ("mixture_components", C.c_int32),
        ("num_hidden", C.c_int32), ("hidden_sizes", C.c_int32 * MAX_HIDDEN), ("max_batch", C.c_int32),
        ("sigma_min", C.c_float), ("raw_sigma_bias", C.c_float), ("gen_bias_init", C.c_float),
        ("temperature", C.c_float), ("learning_rate", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
        ("epsilon", C.c_float), ("device", C.c_int32), ("deterministic", C.c_int32), ("reserved", C.c_int32 * 6),
    ]


class ParamDesc(C.Structure):
    _fields_ = [("name", C.c_char * NAME_LEN), ("offset", C.c_int64), ("rows", C.c_int32), ("cols", C.c_int32)]


# every symbol include/gmvae_abi.h declares: name -> (restype, argtypes)
_P, _I, _I64, _F = C.c_void_p, C.c_int, C.c_int64, C.POINTER(C.c_float)
SYMBOLS = {
    "gmvae_create": (_I, [C.POINTER(Config), C.POINTER(_P)]),
    "gmvae_destroy": (None, [_P]),
    "gmvae_param_count": (_I64, [_P]),
    "gmvae_grad_count": (_I64, [_P]),
    "gmvae_num_params": (_I, [_P]),
    "gmvae_param_table": (_I, [_P, C.POINTER(ParamDesc), _I]),
    "gmvae_workspace_bytes": (C.c_size_t, [_P]),
    "gmvae_bind": (_I, [_P, _P, _P, _P, _P, _P, C.c_size_t]),
    "gmvae_params_updated": (_I, [_P, _P]),
    "gmvae_forward_backward": (_I, [_P, _P, _I, _I, _P, _P, _P]),
    "gmvae_finalize_loss": (_I, [_P, _P, _P]),
    "gmvae_adam_step": (_I, [_P, _P]),
    "gmvae_get_step": (_I, [_P, C.POINTER(_I64), _P]),
    "gmvae_set_step": (_I, [_P, _I64, _P]),
    "gmvae_set_seed": (_I, [_P, C.c_uint64]),
    "gmvae_nccl_unique_id": (_I, [C.c_char_p]),
    "gmvae_nccl_init": (_I, [_P, C.c_char_p, _I, _I]),
    "gmvae_allreduce_grads": (_I, [_P, _P]),
    "gmvae_peer_export": (_I, [_P, _I, _I, C.c_char_p]),
    "gmvae_peer_attach": (_I, [_P, C.c_char_p]),
    "gmvae_peer_grads": (_P, [_P]),
    "gmvae_train_step": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "gmvae_step_graph_capture": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "gmvae_step_graph_launch": (_I, [_P, _P]),
    "gmvae_encode": (_I, [_P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "gmvae_decode": (_I, [_P, _P, _I, _P, _P]),
    "gmvae_prior_table": (_I, [_P, _P, _P, _P]),
    "gmvae_condition": (_I, [_P, _I, _P, _P, _I, _P, _P, _P]),
    "gmvae_dist_normal_sample": (_I, [_P, _P, _P, _I64, _P, _P]),
    "gmvae_dist_normal_log_prob": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "gmvae_dist_bernoulli_log_prob": (_I, [_P, _P, _I, _I, _P, _P]),
    "gmvae_dist_bernoulli_mean": (_I, [_P, _I64, _P, _P]),
    "gmvae_dist_relaxed_sample": (_I, [_P, _P, _I, _I, C.c_float, _P, _P]),
    "gmvae_binarize": (_I, [_P, _P, _I64, _P, _I, C.c_uint64, _P, _P]),
    "gmvae_unpack_bits": (_I, [_P, _P, _I, _P, _P]),
    "gmvae_debug_gemm": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P]),
    "gmvae_debug_noise": (_I, [_P, _P, _I64, _P, _I64, _P]),
    "gmvae_debug_chain_trace": (_I, [_P, _P, _I]),
    "gmvae_debug_chain_jobstat": (_I, [_P, _P]),
    "gmvae_debug_chain_jobs": (_I, [_P, C.POINTER(C.c_int), _I]),
    "gmvae_profile_enable": (_I, [_P, _I]),
    "gmvae_profile_read": (_I, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64), _I]),
    "gmvae_launch_count": (_I64, [_P]),
    "gmvae_last_error": (C.c_char_p, []),
    "gmvae_build_info": (C.c_char_p, []),
}

_lib = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Loads (building first if the .so is missing and nvcc is present) the native library."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    # (Re)build when the library is missing or older than a source file -- under a file lock, so that the ranks of one
    # torchrun launch do not race nvcc on the same output.  A stale library with no nvcc around is loaded as it is.
    if _build.needs_build():
        import fcntl
        import shutil
        have_nvcc = os.path.exists(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")) or shutil.which("nvcc")
        if have_nvcc or not os.path.exists(path):
            try:
                with open(path + ".lock", "w") as lk:
                    fcntl.flock(lk, fcntl.LOCK_EX)
                    try:
                        if _build.needs_build():
                            _build.build()
                    finally:
                        fcntl.flock(lk, fcntl.LOCK_UN)
            except Exception as e:  # no nvcc / compile error: the product cannot run
                if not os.path.exists(path):
                    raise RuntimeError(
                        f"libgmvae_b200.so is missing and could not be built ({e}); there is no CPU fallback. "
                        f"Run `python -m gmvae_b200.build`.") from e
                raise
    try:
        import torch  # noqa: F401  (loads the bundled libnccl/libcudart the library links against)
    except Exception:
        pass
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().gmvae_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libgmvae_b200 {what} failed (code {rc}): {msg}")
