"""Loader of the C-ABI CUDA library (csrc/ -> libcrowdnav_b200.so, include/crowdnav_b200.h).

There is NO CPU fallback: `load()` raises when the library is missing or does
not export every symbol the header declares, and every compute entry point
goes through `check()`, which raises with cn_last_error() on failure.
"""
import ctypes as C
import os
import subprocess

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# CROWDNAV_B200_LIB: another build of the same library (A/B timing of kernel variants inside one process launch)
LIB_PATH = os.environ.get("CROWDNAV_B200_LIB") or os.path.join(_HERE, "libcrowdnav_b200.so")

# every function include/crowdnav_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "cn_last_error": (C.c_char_p, []),
    "cn_abi_version": (C.c_int, []),
    "cn_env_state_bytes": (C.c_size_t, [C.POINTER(abi.CnConfig), C.c_int]),
    "cn_env_create": (C.c_int, [C.POINTER(abi.CnConfig), C.c_int, C.c_int, _P, C.c_size_t, C.POINTER(_P)]),
    "cn_env_destroy": (C.c_int, [_P]),
    "cn_env_reset": (C.c_int, [_P, _P, C.POINTER(abi.CnObsOut), _P]),
    "cn_env_step": (C.c_int, [_P, _P, C.POINTER(abi.CnStepOut), C.c_int, _P]),
    "cn_env_set_state": (C.c_int, [_P, C.POINTER(abi.CnStateView), _P]),
    "cn_env_get_state": (C.c_int, [_P, C.POINTER(abi.CnStateView), _P]),
    "cn_env_observe": (C.c_int, [_P, C.POINTER(abi.CnObsOut), _P]),
    "cn_env_render": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P]),
    "cn_env_robot_act": (C.c_int, [_P, C.c_int32, _P, _P]),
    "cn_env_join": (C.c_int, [_P, _P]),
    "cn_env_refill": (C.c_int, [_P, _P]),
    "cn_dsrnn_set_refill_env": (C.c_int, [_P, _P]),
    "cn_dsrnn_set_edge_event": (C.c_int, [_P, _P]),
    "cn_dsrnn_set_edge_image": (C.c_int, [_P, _P, _P, _P, _P]),
    "cn_env_last_launches": (C.c_int, [_P]),
    "cn_dsrnn_create": (C.c_int, [C.POINTER(abi.CnDsrnnWeights), C.c_int, _P, C.POINTER(_P)]),
    "cn_dsrnn_destroy": (C.c_int, [_P]),
    "cn_dsrnn_update_weights": (C.c_int, [_P, C.POINTER(abi.CnDsrnnWeights), _P]),
    "cn_dsrnn_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "cn_dsrnn_forward": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(abi.CnDsrnnIO), C.c_int, _P, C.c_size_t, _P]),
    "cn_dsrnn_last_launches": (C.c_int, [_P]),
    "cn_dsrnn_enable_timing": (C.c_int, [_P, C.c_int]),
    "cn_dsrnn_time_ms": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "cn_env_enable_timing": (C.c_int, [_P, C.c_int]),
    "cn_env_time_ms": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "cn_gru_gates_forward": (C.c_int, [_P] * 11 + [C.c_int, C.c_int, _P]),
    "cn_gru_gates_backward": (C.c_int, [_P] * 12 + [C.c_int, C.c_int, _P]),
    "cn_split_bf16": (C.c_int, [_P, _P, _P, C.c_size_t, _P]),
    "cn_dsrnn_edge_sequence_step": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(abi.CnEdgeSeqStep), _P]),
    "cn_gru_gates_backward_pairs": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, _P]),
    "cn_gemm_bf16x3": (C.c_int, [C.POINTER(abi.CnGemm), C.c_int, _P]),
    "cn_encoder_grad": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, C.c_longlong, _P]),
    "cn_encoder_grad_ordered_workspace_bytes": (C.c_size_t, [C.c_longlong]),
    "cn_encoder_grad_ordered": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, C.c_longlong, _P, C.c_size_t, _P]),
    "cn_gemm_bf16x3_ordered_workspace_bytes": (C.c_int, [C.POINTER(abi.CnGemm), C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_int)]),
    "cn_gemm_bf16x3_ordered": (C.c_int, [C.POINTER(abi.CnGemm), C.c_int, _P, C.c_size_t, _P]),
    "cn_gemm_enable_timing": (C.c_int, [C.c_int]),
    "cn_gemm_time_ms": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "cn_attention_train_forward": (C.c_int, [_P, _P, _P, _P, _P, C.c_float, C.c_int, C.c_int, _P]),
    "cn_attention_train_backward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_float, C.c_int, C.c_int, _P]),
}

_LIB = None


class CrowdNavLibraryError(RuntimeError):
    pass


def build(verbose=False):
    """Compile csrc/ for sm_100a with nvcc (cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], stdout=out)


def load():
    """dlopen libcrowdnav_b200.so and bind every declared symbol; raises if anything is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise CrowdNavLibraryError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise CrowdNavLibraryError(f"{LIB_PATH} does not export {name}") from exc
        fn.restype, fn.argtypes = restype, argtypes
    if lib.cn_abi_version() != abi.ABI_VERSION:
        raise CrowdNavLibraryError("ABI version mismatch: library %d, python %d" % (lib.cn_abi_version(), abi.ABI_VERSION))
    _LIB = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().cn_last_error()
        raise CrowdNavLibraryError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))


def raw_stream(device_index):
    """cudaStream_t of torch's current stream on `device_index` as a c_void_p.  This sits on the host's critical path
    of every step (right after the synchronisation of a train.py-style loop): the raw getter costs ~0.2 us, building a
    torch.cuda.Stream object ~3 us."""
    try:
        return C.c_void_p(_raw_stream(device_index))
    except NameError:
        import torch
        return C.c_void_p(torch.cuda.current_stream(device_index).cuda_stream)


try:
    from torch._C import _cuda_getCurrentRawStream as _raw_stream
except ImportError:      # older / CPU-only torch builds: raw_stream() falls back to torch.cuda.current_stream
    pass
