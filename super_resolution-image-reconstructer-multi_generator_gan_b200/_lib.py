"""ctypes binding of libsrgan_b200.so (C ABI declared in include/srgan_b200.h).

The library is built in-tree with nvcc for sm_100a (``build()``); there is no fallback path: ``lib()`` raises if the
shared object is missing, and every wrapper raises ``RuntimeError`` with ``srg_last_error()`` on a non-zero return
code (the reference surfaces failures as Python exceptions from torch, SURVEY 8b).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_longlong, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
# SRG_LIB_SO: developer override for same-box A/B runs against an older build of the library (never rebuilt)
SO_PATH = os.environ.get("SRG_LIB_SO") or os.path.join(HERE, "libsrgan_b200.so")
SOURCES = ["conv_gemm.cu", "conv_ops.cu", "vgg_ops.cu", "resample.cu", "trunk_fused.cu", "wgrad_gemm.cu", "elementwise.cu", "peer_sync.cu", "generator.cu", "discriminator.cu", "metrics.cu", "api.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC"]

_lib = None


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build() -> bool:
    if os.environ.get("SRG_LIB_SO"):
        return False
    if not os.path.exists(SO_PATH):
        return True
    so_m = os.path.getmtime(SO_PATH)
    deps = _sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    deps.append(os.path.join(ROOT, "include", "srgan_b200.h"))
    return any(os.path.getmtime(d) > so_m for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into libsrgan_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    if not force and not needs_build():
        return SO_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-o", SO_PATH] + _sources() + ["-ldl"]
    if verbose:
        print(" ".join(cmd))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    return SO_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU or PyTorch fallback for the SR-GAN hot path.")
    L = ctypes.CDLL(SO_PATH)
    _declare(L)
    if L.srg_abi_version() != 1:
        raise RuntimeError("libsrgan_b200.so ABI version mismatch")
    _lib = L
    return L


EXPORTS = {
    # name: (restype, argtypes)
    "srg_abi_version": (c_int, []),
    "srg_last_error": (c_char_p, []),
    "srg_generator_create": (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int]),
    "srg_generator_destroy": (None, [c_void_p]),
    "srg_generator_num_params": (c_int, [c_void_p]),
    "srg_generator_param_elems": (c_int64, [c_void_p]),
    "srg_generator_param_info": (c_int, [c_void_p, c_int, c_char_p, c_int, POINTER(c_int64), POINTER(c_int64),
                                         POINTER(c_int), POINTER(c_int)]),
    "srg_generator_num_buffers": (c_int, [c_void_p]),
    "srg_generator_buffer_elems": (c_int64, [c_void_p]),
    "srg_generator_buffer_info": (c_int, [c_void_p, c_int, c_char_p, c_int, POINTER(c_int64), POINTER(c_int64)]),
    "srg_generator_workspace_bytes": (c_size_t, [c_void_p, c_int]),
    "srg_generator_bind": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int]),
    "srg_generator_set_grads": (c_int, [c_void_p, c_void_p]),
    "srg_generator_pack": (c_int, [c_void_p, c_void_p]),
    "srg_generator_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "srg_generator_backward": (c_int, [c_void_p, c_void_p, c_void_p]),
    "srg_generator_forward_frozen": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "srg_generator_backward_ex": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "srg_generator_tile_halo": (c_int, [c_int, c_int]),
    "srg_generator_forward_tiles": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "srg_generator_forward_frozen_tiles": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                                                   c_void_p]),
    "srg_generator_backward_tiles": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "srg_generator_forward_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "srg_generator_forward_tiles_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                                               c_void_p]),
    "srg_generator_num_tensors": (c_int, [c_void_p]),
    "srg_generator_tensor_info": (c_int, [c_void_p, c_int, c_char_p, c_int, POINTER(c_int64), POINTER(c_int),
                                          POINTER(c_int)]),
    "srg_generator_launch_count": (c_longlong, [c_void_p]),
    "srg_generator_set_keep_grads": (c_int, [c_void_p, c_int]),
    "srg_total_launches": (c_longlong, []),
    "srg_set_conv_variant": (c_int, [c_int]),
    "srg_conv9_rows_window": (c_int, [c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "srg_wgrad_batched_plan": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int),
                                       POINTER(c_int)]),
    "srg_generator_profile_enable": (c_int, [c_void_p, c_int]),
    "srg_generator_profile_read": (c_int, [c_void_p, POINTER(c_double), POINTER(c_longlong)]),
    "srg_bn_stats_rows": (c_int, [c_int64]),
    "srg_bn_stats": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "srg_bn_finalize": (c_int, [c_void_p, c_int, c_double, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_void_p]),
    "srg_bn_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p]),
    "srg_bn_backward_finalize": (c_int, [c_void_p, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p]),
    "srg_bn_backward_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "srg_conv2d_packed_weight_bytes": (c_size_t, [c_int, c_int, c_int]),
    "srg_conv2d_pack_weights": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "srg_conv2d_fprop": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_float,
                                 c_void_p, c_void_p, c_void_p]),
    "srg_conv2d_dgrad": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                 c_void_p]),
    "srg_conv2d_wgrad_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "srg_conv2d_wgrad": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p,
                                 c_void_p]),
    "srg_unfold3x3_rgb": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "srg_fold3x3_rgb": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "srg_maxpool2x2_forward": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "srg_maxpool2x2_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "srg_l1_bf16_scratch_bytes": (c_size_t, []),
    "srg_l1_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_int, c_float, c_int, c_void_p, c_void_p, c_size_t, c_void_p,
                            c_void_p]),
    "srg_resize_plan_ksize": (c_int, [c_int, c_int, c_int]),
    "srg_resize_plan": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p]),
    "srg_resize_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "srg_set_trunk_fused": (c_int, [c_int]),
    "srg_generator_forward_phases": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "srg_generator_backward_phases": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "srg_generators_trunk": (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_void_p]),
    "srg_debug_trunk_prof": (c_int, [POINTER(c_longlong), c_int]),
    "srg_generator_trunk_layers": (c_int, [c_void_p]),
    "srg_generator_trunk_error": (c_int, [c_void_p]),
    "srg_generator_set_allreduce": (c_int, [c_void_p, c_void_p, c_void_p, c_int]),
    "srg_nccl_unique_id": (c_int, [c_void_p]),
    "srg_nccl_comm_create": (c_int, [c_void_p, c_int, c_int, POINTER(c_void_p)]),
    "srg_nccl_comm_destroy": (None, [c_void_p]),
    "srg_nccl_allreduce_f64": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "srg_nccl_allreduce_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "srg_nccl_allreduce_mean_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "srg_generator_use_nccl": (c_int, [c_void_p, c_void_p, c_int]),
    "srg_peer_sync_create": (c_int, [POINTER(c_void_p), c_int, c_int]),
    "srg_peer_sync_handle": (c_int, [c_void_p, c_void_p]),
    "srg_peer_sync_connect": (c_int, [c_void_p, c_void_p]),
    "srg_peer_sync_destroy": (None, [c_void_p]),
    "srg_peer_sync_error": (c_int, [c_void_p]),
    "srg_generator_use_peer_sync": (c_int, [c_void_p, c_void_p]),
    "srg_discriminator_create": (c_int, [POINTER(c_void_p), c_int, c_int, c_int]),
    "srg_discriminator_destroy": (None, [c_void_p]),
    "srg_discriminator_output_hw": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int)]),
    "srg_discriminator_num_params": (c_int, [c_void_p]),
    "srg_discriminator_param_elems": (c_int64, [c_void_p]),
    "srg_discriminator_param_info": (c_int, [c_void_p, c_int, c_char_p, c_int, POINTER(c_int64), POINTER(c_int64),
                                             POINTER(c_int), POINTER(c_int)]),
    "srg_discriminator_workspace_bytes": (c_size_t, [c_void_p, c_int]),
    "srg_discriminator_bind": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int]),
    "srg_discriminator_set_grads": (c_int, [c_void_p, c_void_p]),
    "srg_discriminator_pack": (c_int, [c_void_p, c_void_p]),
    "srg_discriminator_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "srg_discriminator_backward": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "srg_discriminator_num_tensors": (c_int, [c_void_p]),
    "srg_discriminator_tensor_info": (c_int, [c_void_p, c_int, c_char_p, c_int, POINTER(c_int64), POINTER(c_int),
                                              POINTER(c_int)]),
    "srg_recon_loss_scratch_bytes": (c_size_t, []),
    "srg_recon_loss_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "srg_recon_loss_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_float, c_void_p]),
    "srg_tanh_mean": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p,
                              c_float, c_void_p]),
    "srg_point_loss": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p, c_void_p, c_float, c_void_p]),
    "srg_image_enhance": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "srg_mse": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p, c_void_p]),
    "srg_image_metrics_scratch_bytes": (c_size_t, [c_int, c_int, c_int]),
    "srg_image_metrics": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p,
                                  c_void_p]),
    "srg_adam_step_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_float, c_float, c_float,
                                  c_void_p, c_float, c_void_p]),
    "srg_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float,
                              c_int, c_float, c_void_p]),
}


def _declare(L: ctypes.CDLL) -> None:
    for name, (res, args) in EXPORTS.items():
        fn = getattr(L, name)          # AttributeError here == the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().srg_last_error()
        raise RuntimeError(f"libsrgan_b200 {what} failed (code {rc}): {msg.decode() if msg else ''}")


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
