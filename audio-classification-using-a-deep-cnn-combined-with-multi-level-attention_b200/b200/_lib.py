"""ctypes binding of libvggish_mla_b200.so (include/vggish_mla_b200.h).

The library is the product: if it is missing, or a call fails, we raise — there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# VMB_LIB=<path> loads another build of the library (A/B timing of two builds on one box: tools/ab/*.so)
LIB_PATH = os.environ.get("VMB_LIB") or os.path.join(_HERE, "libvggish_mla_b200.so")

_c_p = C.c_void_p
_ll = C.c_longlong
_int = C.c_int
_sz = C.c_size_t

# name -> (restype, argtypes); mirrors the header one to one.
SIGNATURES = {
    "vmb_last_error": (C.c_char_p, []),
    "vmb_abi_version": (_int, []),
    "vmb_device_arch": (_int, [_int]),
    "vmb_launch_count": (_ll, []),
    "vmb_igemm_pair_enable": (_int, [_int]),
    "vmb_igemm_halo_enable": (_int, [_int]),
    "vmb_mla_fuse_enable": (_int, [_int]),
    "vmb_profile_enable": (_int, [_int]),
    "vmb_profile_collect": (_int, [_c_p, _c_p, _int]),
    "vmb_num_frames": (_ll, [_ll]),
    "vmb_num_examples": (_ll, [_ll]),
    "vmb_logmel": (_int, [_c_p, _ll, _ll, _ll, _ll, _c_p, _c_p]),
    "vmb_logmel_pcm16": (_int, [_c_p, _ll, _ll, _ll, _ll, _c_p, _c_p]),
    "vmb_logmel_cudacore": (_int, [_c_p, _ll, _ll, _ll, _ll, _c_p, _c_p]),
    "vmb_stft_magnitude": (_int, [_c_p, _ll, _c_p, _c_p]),
    "vmb_spec_tiles": (_int, [_c_p, _ll, _int, _int, _int, _c_p, _c_p]),
    "vmb_front_end_tables": (_int, [_c_p, _c_p]),
    "vmb_conv1_relu_pool": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, _c_p]),
    "vmb_conv1_relu_pool_ex": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, _int, _c_p]),
    "vmb_conv1_relu_pool_cudacore": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, _c_p]),
    "vmb_conv3x3_relu": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, _int, _int, _int, _int, _int, _c_p]),
    "vmb_conv3x3_relu_ex": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, _int, _int, _int, _int, _int, _int, _c_p]),
    "vmb_linear_ex": (_int, [_c_p, _c_p, _c_p, _c_p, _int, _int, _ll, _int, _int, _int, _c_p]),
    "vmb_linear": (_int, [_c_p, _c_p, _c_p, _c_p, _int, _int, _ll, _int, _int, _c_p]),
    "vmb_postprocess": (_int, [_c_p, _c_p, _c_p, _c_p, _c_p, _ll, _c_p]),
    "vmb_vggish_create": (_int, [C.POINTER(_c_p), C.POINTER(_c_p), C.POINTER(_c_p), C.POINTER(_c_p),
                                 C.POINTER(_c_p), _c_p]),
    "vmb_vggish_create_ex": (_int, [C.POINTER(_c_p), C.POINTER(_c_p), C.POINTER(_c_p), C.POINTER(_c_p),
                                    C.POINTER(_c_p), _int, _c_p]),
    "vmb_vggish_precision": (_int, [_c_p]),
    "vmb_vggish_saturation": (_int, [_c_p, _int]),
    "vmb_vggish_handle_workspace_bytes": (_sz, [_c_p, _ll]),
    "vmb_vggish_destroy": (None, [_c_p]),
    "vmb_vggish_workspace_bytes": (_sz, [_ll]),
    "vmb_vggish_forward": (_int, [_c_p, _c_p, _ll, _c_p, _c_p, _c_p, _sz, _c_p]),
    "vmb_vggish_fc_train_workspace_bytes": (_sz, [_ll]),
    "vmb_vggish_fc_grad_count": (_ll, []),
    "vmb_vggish_refresh_fc": (_int, [_c_p, C.POINTER(_c_p), C.POINTER(_c_p), _c_p]),
    "vmb_vggish_forward_train": (_int, [_c_p, _c_p, _ll, _c_p, _c_p, _sz, _c_p]),
    "vmb_vggish_fc_backward": (_int, [_c_p, _c_p, _sz, _c_p, _ll, _c_p, _c_p]),
    "vmb_vggish_conv4_2_train_workspace_bytes": (_sz, [_ll]),
    "vmb_vggish_refresh_conv4_2": (_int, [_c_p, _c_p, _c_p, _c_p, _c_p]),
    "vmb_vggish_forward_train_conv4_2": (_int, [_c_p, _c_p, _ll, _c_p, _c_p, _sz, _c_p]),
    "vmb_vggish_conv4_2_backward": (_int, [_c_p, _c_p, _sz, _c_p, _ll, _c_p, _c_p, _c_p]),
    "vmb_mla_create": (_int, [C.POINTER(_c_p), _int, C.POINTER(_int), _int, _int, _int, _int, _c_p, _ll, _c_p]),
    "vmb_mla_destroy": (None, [_c_p]),
    "vmb_mla_num_classes": (_int, [_c_p]),
    "vmb_mla_param_count": (_ll, [_int, C.POINTER(_int), _int, _int, _int, _int]),
    "vmb_mla_forward": (_int, [_c_p, _c_p, _ll, _c_p, _c_p]),
    "vmb_mla_embedded_mapping": (_int, [_c_p, _int, _c_p, _ll, _c_p, _c_p]),
    "vmb_mla_attention": (_int, [_c_p, _int, _c_p, _ll, _c_p, _c_p]),
    "vmb_mla_forward_fp32": (_int, [_c_p, _c_p, _ll, _c_p, _c_p]),
    "vmb_mla_train_param_count": (_ll, [_int, C.POINTER(_int), _int, _int, _int, _int, C.POINTER(_ll)]),
    "vmb_mla_trainer_create": (_int, [C.POINTER(_c_p), _int, C.POINTER(_int), _int, _int, _int, _int, _ll, _c_p]),
    "vmb_mla_trainer_destroy": (None, [_c_p]),
    "vmb_mla_train_step": (_int, [_c_p, _c_p, _c_p, _c_p, _c_p, _ll, C.c_float, C.c_ulonglong, _c_p, _c_p, _c_p, _c_p]),
    "vmb_mla_train_tail_offset": (_ll, [_c_p]),
    "vmb_mla_train_wait_tail": (_int, [_c_p, _c_p]),
    "vmb_mla_train_forward": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, C.c_float, C.c_ulonglong, _c_p, _c_p]),
    "vmb_mla_train_backward": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, C.c_float, C.c_ulonglong, _c_p, _c_p]),
    "vmb_mla_train_backward_dx": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, C.c_float, C.c_ulonglong, _c_p, _c_p, _c_p]),
    "vmb_adam_step": (_int, [_c_p, _c_p, _c_p, _c_p, _ll, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _ll,
                             C.c_float, _c_p]),
    "vmb_dp_slice": (None, [_ll, _int, _int, C.POINTER(_ll), C.POINTER(_ll)]),
    "vmb_dp_create": (_int, [C.POINTER(_c_p), _ll, _int, _int, _c_p]),
    "vmb_dp_connect": (_int, [_c_p, _c_p]),
    "vmb_dp_params": (_c_p, [_c_p]),
    "vmb_dp_grads": (_c_p, [_c_p, _int]),
    "vmb_dp_adam_step": (_int, [_c_p, _int, _c_p, _c_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _ll, _c_p]),
    "vmb_dp_status": (_int, [_c_p]),
    "vmb_dp_disconnect": (None, [_c_p]),
    "vmb_dp_destroy": (None, [_c_p]),
    "vmb_pipeline_workspace_bytes": (_sz, [_ll, _ll]),
    "vmb_pipeline_forward": (_int, [_c_p, _c_p, _c_p, _ll, _ll, _c_p, _c_p, _c_p, _sz, _c_p]),
    "vmb_pipeline_forward_host": (_int, [_c_p, _c_p, _c_p, _ll, _ll, _c_p, _ll, _c_p]),
    "vmb_pipeline_submit_host": (_int, [_c_p, _c_p, _c_p, _ll, _ll, _c_p, _ll, _c_p]),
    "vmb_pipeline_submit_host_pcm16": (_int, [_c_p, _c_p, _c_p, _ll, _ll, _c_p, _ll, _c_p]),
    "vmb_pipeline_forward_pcm16": (_int, [_c_p, _c_p, _c_p, _ll, _ll, _c_p, _c_p, _c_p, _sz, _c_p]),
    "vmb_pipeline_wait_host": (_int, [_c_p, _int]),
}

_lib = None


class B200Error(RuntimeError):
    """A C-ABI call returned non-zero; the message is vmb_last_error()."""


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200Error(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
                "(there is no CPU fallback for this path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def last_error() -> str:
    msg = lib().vmb_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int, what: str) -> None:
    if status != 0:
        raise B200Error(f"{what} failed: {last_error()}")


def ptr(t) -> int:
    """data_ptr of a CUDA tensor (or None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
