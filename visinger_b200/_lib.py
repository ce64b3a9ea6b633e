"""ctypes binding of the C-ABI library (include/visinger_b200.h).

The library is built IN-TREE with nvcc for sm_100a (`visinger_b200/lib/libvisinger_b200.so`) and
loaded with ctypes: no torch types cross the boundary, only raw device pointers, sizes and the
CUDA stream handle.  PyTorch is used for device memory and streams only.  There is no CPU or
eager fallback: if the library cannot be built or loaded, or a tensor is not on a CUDA device,
the call raises.
"""
from __future__ import annotations

import ctypes
import hashlib
import math
import os
import shutil
import subprocess
import threading
from typing import Dict, Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_LIBDIR = os.path.join(_HERE, "lib")
_LIBPATH = os.path.join(_LIBDIR, "libvisinger_b200.so")
_HEADER = os.path.join(os.path.dirname(_HERE), "include", "visinger_b200.h")
_SOURCES = ["api.cu", "pack.cu", "run_f32.cu", "run_tc.cu", "output.cu", "model.cu"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-diag-suppress", "550"]

PRECISION_FP32 = 0
PRECISION_BF16 = 1
PRECISION_BF16X3 = 2
_PRECISIONS = {"fp32": PRECISION_FP32, "float32": PRECISION_FP32, "bf16": PRECISION_BF16, "bfloat16": PRECISION_BF16,
               "bf16x3": PRECISION_BF16X3}

VSG_MAX_UPS = 8
VSG_MAX_RESBLOCK_KERNELS = 4
VSG_MAX_RESBLOCK_DILATIONS = 4


def precision_code(p) -> int:
    if isinstance(p, int):
        return p
    try:
        return _PRECISIONS[str(p).lower()]
    except KeyError:
        raise ValueError(f"unknown precision {p!r}; use 'fp32', 'bf16' or 'bf16x3'") from None


class VsgConfig(ctypes.Structure):
    _fields_ = [
        ("flow_channels", ctypes.c_int32), ("flow_hidden", ctypes.c_int32), ("flow_kernel_size", ctypes.c_int32),
        ("flow_dilation_rate", ctypes.c_int32), ("flow_n_layers", ctypes.c_int32), ("flow_n_flows", ctypes.c_int32),
        ("flow_gin", ctypes.c_int32),
        ("dec_initial_channel", ctypes.c_int32), ("dec_resblock", ctypes.c_int32), ("dec_n_kernels", ctypes.c_int32),
        ("dec_resblock_kernel_sizes", ctypes.c_int32 * VSG_MAX_RESBLOCK_KERNELS),
        ("dec_n_dilations", ctypes.c_int32 * VSG_MAX_RESBLOCK_KERNELS),
        ("dec_resblock_dilations", (ctypes.c_int32 * VSG_MAX_RESBLOCK_DILATIONS) * VSG_MAX_RESBLOCK_KERNELS),
        ("dec_n_ups", ctypes.c_int32),
        ("dec_upsample_rates", ctypes.c_int32 * VSG_MAX_UPS),
        ("dec_upsample_kernel_sizes", ctypes.c_int32 * VSG_MAX_UPS),
        ("dec_upsample_initial_channel", ctypes.c_int32), ("dec_gin", ctypes.c_int32),
    ]


class VsgEncConfig(ctypes.Structure):
    _fields_ = [("in_channels", ctypes.c_int32), ("out_channels", ctypes.c_int32), ("hidden_channels", ctypes.c_int32),
                ("kernel_size", ctypes.c_int32), ("dilation_rate", ctypes.c_int32), ("n_layers", ctypes.c_int32),
                ("gin_channels", ctypes.c_int32)]


class VsgRelEncConfig(ctypes.Structure):
    _fields_ = [("hidden_channels", ctypes.c_int32), ("filter_channels", ctypes.c_int32), ("n_heads", ctypes.c_int32),
                ("n_layers", ctypes.c_int32), ("kernel_size", ctypes.c_int32), ("window_size", ctypes.c_int32),
                ("gin_channels", ctypes.c_int32)]


class VsgModelConfig(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "ph_dict_size", "pitch_size", "dur_size", "hidden", "filter", "n_heads", "ffn_kernel_size", "window_size",
        "enc_layers", "pitch_predictor_layers", "frame_prior_layers", "use_pos_embed", "use_pitch_embed", "use_spk_id",
        "use_spk_embed", "num_spk", "spk_embed_dim")] + [("hot", VsgConfig)]


class VsgTensor(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("data", ctypes.c_void_p), ("ndim", ctypes.c_int32),
                ("shape", ctypes.c_int64 * 4)]


class VsgDebugConv(ctypes.Structure):
    """Descriptor of vsg_debug_conv_tc (include/visinger_b200.h)."""
    _fields_ = ([(n, ctypes.c_void_p) for n in ("x", "w", "bias", "bcond", "mask", "add0", "add1", "out_raw", "out_act",
                                                "out_f32")] +
                [(n, ctypes.c_int32) for n in ("planes", "mode", "couple_sign", "add0_is_act", "bcond_bs")] +
                [("scale", ctypes.c_float), ("slope", ctypes.c_float)] +
                [(n, ctypes.c_int32) for n in ("B", "Lin", "Cin", "Cout", "k", "dil", "in_off0", "Lq", "out_stride",
                                               "out_phase", "Lout", "x_ld", "x_part_stride", "ld", "part_stride",
                                               "epi_sigs")])


class VsgDebugPair(ctypes.Structure):
    """Descriptor of vsg_debug_pair_tc (include/visinger_b200.h)."""
    _fields_ = ([(n, ctypes.c_void_p) for n in ("xa", "w1", "b1", "w2", "b2", "add0", "add1", "out_raw", "out_act",
                                                "out_f32")] +
                [("add0_is_act", ctypes.c_int32), ("scale", ctypes.c_float)] +
                [(n, ctypes.c_int32) for n in ("B", "L", "C", "k", "d1")])


class VsgDebugConvF32(ctypes.Structure):
    """Descriptor of vsg_debug_conv_f32 (include/visinger_b200.h)."""
    _fields_ = ([(n, ctypes.c_void_p) for n in ("x", "w", "bias", "bcond", "res", "mask", "y", "y2")] +
                [(n, ctypes.c_int64) for n in ("x_bs", "y_bs", "res_bs", "y2_bs")] +
                [(n, ctypes.c_int32) for n in ("x_cs", "y_cs", "res_cs", "y2_cs", "B", "Cin", "Lin", "Cout", "k", "dil",
                                               "in_off0", "pre_lrelu")] +
                [("slope", ctypes.c_float)] +
                [(n, ctypes.c_int32) for n in ("bcond_bs", "mask_bs", "Lq", "out_stride", "out_phase", "Lout", "epi",
                                               "acc_mode")] +
                [("acc_div", ctypes.c_float)] +
                [(n, ctypes.c_int32) for n in ("rs_split", "y2_first", "y2_mask", "couple_sign", "gate_interleave")])


# epilogues of vsg_debug_conv_f32 (csrc/kernels_f32.cuh EPI_*, and the magnitude instantiation)
EPI_F32 = dict(LINEAR=0, GATE=1, RES_SKIP=2, COUPLE=3, MAG=4)
ACC_SET, ACC_ADD, ACC_ADD_DIV = 0, 1, 2

# epilogue images of the convolution kernel (csrc/conv_tc.cuh, EPI_SIG_*), as vsg_debug_conv_tc and vsg_last_launch_images
# number them
EPI_SIG = dict(GENERIC=0, ACT=1, RES_ACT=2, LINEAR=3, X6=4, SUM0=5, SUM1=6, FINAL=7, POST=8, ACT_X3=9, RES_ACT_X3=10,
               SUM0_X3=11, SUM1_X3=12, FINAL_X3=13, MAG=14)
EPI_TC_LINEAR, EPI_TC_GATE, EPI_TC_COUPLE = 0, 1, 2


def _source_files():
    files = [os.path.join(_CSRC, f) for f in sorted(os.listdir(_CSRC)) if f.endswith((".cu", ".cuh", ".h", ".inc"))]
    return files + [_HEADER]


def _source_hash() -> str:
    h = hashlib.sha256()
    for f in _source_files():
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _nvcc() -> Optional[str]:
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else shutil.which("nvcc")


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a into the in-tree shared library (no GPU needed)."""
    os.makedirs(_LIBDIR, exist_ok=True)
    want = _source_hash()
    stamp = _LIBPATH + ".hash"
    if not force and os.path.exists(_LIBPATH) and os.path.exists(stamp) and open(stamp).read().strip() == want:
        return _LIBPATH
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("visinger_b200: libvisinger_b200.so is missing or stale and nvcc was not found; "
                           "there is no fallback path")
    # one nvcc per translation unit, in parallel, then one link: run_tc.cu alone is most of the serial build time
    objdir = os.path.join(os.path.dirname(_HERE), "build", "obj")
    os.makedirs(objdir, exist_ok=True)
    cflags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + cflags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(_CSRC, src)]
        if verbose:
            print(" ".join(cmd), flush=True)
        proc = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, proc

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=len(_SOURCES)) as pool:
        results = list(pool.map(compile_one, _SOURCES))
    for src, _, proc in results:
        if proc.returncode != 0:
            raise RuntimeError(f"visinger_b200: nvcc failed on {src}\n" + proc.stdout + proc.stderr)
        if verbose:
            print(proc.stdout + proc.stderr, flush=True)
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", _LIBPATH + ".tmp"] + [o for _, o, _ in results]
    proc = subprocess.run(link, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("visinger_b200: link failed\n" + proc.stdout + proc.stderr)
    os.replace(_LIBPATH + ".tmp", _LIBPATH)
    with open(stamp, "w") as fh:
        fh.write(want)
    return _LIBPATH


_lib = None
_lock = threading.Lock()


def lib() -> ctypes.CDLL:
    """Load (building first if stale) the C-ABI library.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        # VSG_LIB_OVERRIDE: load another build of the same library (A/B timing of two kernel versions on one GPU box)
        path = os.environ.get("VSG_LIB_OVERRIDE") or build()
        L = ctypes.CDLL(path)
        vp, i32, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t
        L.vsg_abi_version.restype = ctypes.c_int
        L.vsg_last_error.restype = ctypes.c_char_p
        L.vsg_last_launch_count.restype = i32
        L.vsg_pack_create.restype = ctypes.c_int
        L.vsg_pack_create.argtypes = [ctypes.POINTER(VsgConfig), ctypes.POINTER(VsgTensor), i32, ctypes.c_char_p,
                                      ctypes.c_char_p, i32, ctypes.POINTER(vp)]
        L.vsg_pack_destroy.restype = None
        L.vsg_pack_destroy.argtypes = [vp]
        L.vsg_workspace_bytes.restype = sz
        L.vsg_workspace_bytes.argtypes = [vp, i32, i32, i32]
        L.vsg_hop_size.restype = i32
        L.vsg_hop_size.argtypes = [vp]
        L.vsg_prior_sample.restype = ctypes.c_int
        L.vsg_prior_sample.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp]
        L.vsg_flow_forward.restype = ctypes.c_int
        L.vsg_flow_forward.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, sz, vp]
        L.vsg_generator_forward.restype = ctypes.c_int
        L.vsg_generator_forward.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
        L.vsg_infer.restype = ctypes.c_int
        L.vsg_infer.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
        L.vsg_wav_to_int16.restype = ctypes.c_int
        L.vsg_wav_to_int16.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp]
        L.vsg_debug_conv1d_bf16.restype = ctypes.c_int
        L.vsg_debug_conv1d_bf16.argtypes = [vp, vp, vp, vp, vp, ctypes.c_float, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32,
                                            i32]
        L.vsg_last_launch_images.restype = ctypes.c_int
        L.vsg_last_launch_images.argtypes = [vp, i32]
        L.vsg_debug_conv_tc.restype = ctypes.c_int
        L.vsg_debug_conv_tc.argtypes = [ctypes.POINTER(VsgDebugConv), ctypes.POINTER(ctypes.c_int32), i32]
        L.vsg_debug_upsample_tc.restype = ctypes.c_int
        L.vsg_debug_upsample_tc.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32,
                                            ctypes.POINTER(ctypes.c_int32), i32]
        L.vsg_debug_conv_f32.restype = ctypes.c_int
        L.vsg_debug_conv_f32.argtypes = [ctypes.POINTER(VsgDebugConvF32), ctypes.POINTER(ctypes.c_int32), i32]
        L.vsg_debug_conv_f32_plan.restype = ctypes.c_int
        L.vsg_debug_conv_f32_plan.argtypes = [i32, i32, i32, ctypes.POINTER(ctypes.c_int32)]
        L.vsg_debug_upsample_f32.restype = ctypes.c_int
        L.vsg_debug_upsample_f32.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, i32]
        L.vsg_debug_conv_post_f32.restype = ctypes.c_int
        L.vsg_debug_conv_post_f32.argtypes = [vp, vp, i32, i32, i32, ctypes.c_float, i32, i32, i32, vp, ctypes.c_int64, i32]
        L.vsg_debug_cond_f32.restype = ctypes.c_int
        L.vsg_debug_cond_f32.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32]
        L.vsg_set_tc_options.restype = ctypes.c_int
        L.vsg_set_tc_options.argtypes = [i32, i32, i32, i32]
        L.vsg_debug_pair_tc.restype = ctypes.c_int
        L.vsg_debug_pair_tc.argtypes = [ctypes.POINTER(VsgDebugPair), ctypes.POINTER(ctypes.c_int32), i32]
        L.vsg_debug_pair_bf16.restype = ctypes.c_int
        L.vsg_debug_pair_bf16.argtypes = [vp, vp, vp, vp, vp, vp, vp, ctypes.c_float, vp, vp, vp, i32, i32, i32, i32, i32, i32]
        L.vsg_enc_pack_create.restype = ctypes.c_int
        L.vsg_enc_pack_create.argtypes = [ctypes.POINTER(VsgEncConfig), ctypes.POINTER(VsgTensor), i32, ctypes.c_char_p, i32,
                                          ctypes.POINTER(ctypes.c_void_p)]
        L.vsg_posterior_workspace_bytes.restype = ctypes.c_size_t
        L.vsg_posterior_workspace_bytes.argtypes = [vp, i32, i32, i32]
        L.vsg_posterior_forward.restype = ctypes.c_int
        L.vsg_posterior_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, ctypes.c_size_t, vp]
        L.vsg_relenc_pack_create.restype = ctypes.c_int
        L.vsg_relenc_pack_create.argtypes = [ctypes.POINTER(VsgRelEncConfig), ctypes.POINTER(VsgTensor), i32, ctypes.c_char_p,
                                             i32, ctypes.POINTER(ctypes.c_void_p)]
        L.vsg_relenc_workspace_bytes.restype = ctypes.c_size_t
        L.vsg_relenc_workspace_bytes.argtypes = [vp, i32, i32, i32, i32]
        L.vsg_relenc_forward.restype = ctypes.c_int
        L.vsg_relenc_forward.argtypes = [vp, vp, vp, vp, i32, vp, i32, i32, i32, vp, ctypes.c_size_t, vp]
        L.vsg_frame_prior_pack_create.restype = ctypes.c_int
        L.vsg_frame_prior_pack_create.argtypes = L.vsg_relenc_pack_create.argtypes
        L.vsg_frame_prior_workspace_bytes.restype = ctypes.c_size_t
        L.vsg_frame_prior_workspace_bytes.argtypes = [vp, i32, i32, i32]
        L.vsg_frame_prior_forward.restype = ctypes.c_int
        L.vsg_frame_prior_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, ctypes.c_size_t, vp]
        L.vsg_length_regulate.restype = ctypes.c_int
        L.vsg_length_regulate.argtypes = [vp, vp, vp, i32, vp, i32, i32, i32, i32, vp]
        L.vsg_infer_zp.restype = ctypes.c_int
        L.vsg_infer_zp.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, ctypes.c_size_t, vp]
        L.vsg_debug_resblock_bf16.restype = ctypes.c_int
        L.vsg_debug_resblock_bf16.argtypes = [vp, vp, vp, i32, vp, vp, ctypes.c_float, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32]
        L.vsg_debug_set_plan.restype = ctypes.c_int
        L.vsg_debug_set_plan.argtypes = [i32, i32, i32, i32, i32]
        L.vsg_debug_last_ms.restype = ctypes.c_float
        for fn in (L.vsg_debug_attention_bf16, L.vsg_debug_attention_f32):
            fn.restype = ctypes.c_int
            fn.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32]
        L.vsg_debug_attention_split_bf16.restype = ctypes.c_int
        L.vsg_debug_attention_split_bf16.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32]
        L.vsg_debug_layernorm_bf16.restype = ctypes.c_int
        L.vsg_debug_layernorm_bf16.argtypes = [vp, vp, vp, vp, i32, vp, ctypes.c_float, i32, i32, i32, i32]
        L.vsg_model_pack_create.restype = ctypes.c_int
        L.vsg_model_pack_create.argtypes = [ctypes.POINTER(VsgModelConfig), ctypes.POINTER(VsgTensor), i32, ctypes.c_char_p,
                                            i32, ctypes.POINTER(ctypes.c_void_p)]
        L.vsg_model_workspace_bytes.restype = sz
        L.vsg_model_workspace_bytes.argtypes = [vp, i32, i32, i32, i32]
        L.vsg_model_forward.restype = ctypes.c_int
        L.vsg_model_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, sz, vp]
        L.vsg_convert_pack_create.restype = ctypes.c_int
        L.vsg_convert_pack_create.argtypes = [ctypes.POINTER(VsgModelConfig), ctypes.POINTER(VsgTensor), i32,
                                              ctypes.c_char_p, i32, i32, ctypes.POINTER(ctypes.c_void_p)]
        L.vsg_convert_workspace_bytes.restype = sz
        L.vsg_convert_workspace_bytes.argtypes = [vp, i32, i32, i32]
        L.vsg_spectrogram.restype = ctypes.c_int
        L.vsg_spectrogram.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
        L.vsg_model_convert.restype = ctypes.c_int
        L.vsg_model_convert.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
        L.vsg_normal_noise.restype = ctypes.c_int
        L.vsg_normal_noise.argtypes = [vp, vp, i32, i32, i32, vp]
        L.vsg_debug_position_table.restype = ctypes.c_int
        L.vsg_debug_position_table.argtypes = [vp, i32, i32, vp, vp]
        L.vsg_window_context.restype = ctypes.c_int
        L.vsg_window_context.argtypes = [vp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
        L.vsg_window_workspace_bytes.restype = sz
        L.vsg_window_workspace_bytes.argtypes = [vp, i32, i32, i32, i32]
        L.vsg_infer_zp_window.restype = ctypes.c_int
        L.vsg_infer_zp_window.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int64, vp, i32, i32, i32, i32, i32, vp, sz, vp]
        L.vsg_generator_forward_window.restype = ctypes.c_int
        L.vsg_generator_forward_window.argtypes = [vp, vp, vp, vp, ctypes.c_int64, i32, i32, i32, i32, i32, vp, sz, vp]
        L.vsg_convert_window_context.restype = ctypes.c_int
        L.vsg_convert_window_context.argtypes = [vp] + [ctypes.POINTER(ctypes.c_int32)] * 3
        L.vsg_convert_window_input.restype = ctypes.c_int
        L.vsg_convert_window_input.argtypes = [vp, i32, i32, i32, i32, i32, ctypes.POINTER(ctypes.c_int64),
                                               ctypes.POINTER(ctypes.c_int64)]
        L.vsg_convert_window_workspace_bytes.restype = sz
        L.vsg_convert_window_workspace_bytes.argtypes = [vp, i32, i32, i32, i32]
        L.vsg_model_convert_window.restype = ctypes.c_int
        L.vsg_model_convert_window.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ctypes.c_int64, vp, i32, i32, i32,
                                               i32, i32, vp, sz, vp]
        if L.vsg_abi_version() != 1:
            raise RuntimeError("visinger_b200: ABI version mismatch between _lib.py and the shared library")
        _lib = L
        return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().vsg_last_error().decode(errors="replace")
        raise RuntimeError(f"visinger_b200: {what} failed ({rc}): {msg}")


def last_launch_count() -> int:
    return int(lib().vsg_last_launch_count())


def last_launch_images() -> Dict[str, int]:
    """Launches of the convolution kernel per epilogue image (EPI_SIG names) in the most recent call on this thread."""
    out = (ctypes.c_int32 * len(EPI_SIG))()
    check(lib().vsg_last_launch_images(out, len(EPI_SIG)), "vsg_last_launch_images")
    return {name: int(out[i]) for name, i in EPI_SIG.items()}


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"visinger_b200: {name} is on {t.device}; the B200 path has no CPU fallback "
                           "(move the module and its inputs to a CUDA device)")


def as_f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


class Pack:
    """Owner of a VsgPack* (device-resident pre-packed weights)."""

    def __init__(self, cfg: VsgConfig, state_dict: Dict[str, torch.Tensor], flow_prefix: str, dec_prefix: str,
                 device: torch.device):
        self._h = ctypes.c_void_p()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("visinger_b200: weights must live on a CUDA device; there is no CPU fallback")
        L = lib()
        host = {}
        for k, v in state_dict.items():
            if (flow_prefix is not None and k.startswith(flow_prefix)) or \
               (dec_prefix is not None and k.startswith(dec_prefix)):
                host[k] = v.detach().to("cpu", torch.float32).contiguous()
        arr = (VsgTensor * len(host))()
        keep = []
        for i, (k, v) in enumerate(host.items()):
            nm = k.encode()
            keep.append(nm)
            arr[i].name = nm
            arr[i].data = v.data_ptr()
            arr[i].ndim = v.dim()
            for d in range(v.dim()):
                arr[i].shape[d] = v.shape[d]
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = L.vsg_pack_create(ctypes.byref(cfg), arr, len(host), (flow_prefix or "").encode(),
                               (dec_prefix or "").encode(), idx, ctypes.byref(self._h))
        check(rc, "vsg_pack_create")
        self.index = idx
        self.hop = int(L.vsg_hop_size(self._h))

    @property
    def handle(self):
        return self._h

    def workspace_bytes(self, B: int, T: int, precision: int) -> int:
        return int(lib().vsg_workspace_bytes(self._h, B, T, precision))

    def window_context(self):
        """(flow, decoder) context frames each side of a streaming window (vsg_window_context)."""
        cf, cd = ctypes.c_int32(), ctypes.c_int32()
        check(lib().vsg_window_context(self._h, ctypes.byref(cf), ctypes.byref(cd)), "vsg_window_context")
        return int(cf.value), int(cd.value)

    def window_workspace_bytes(self, B: int, T: int, max_frames: int, precision: int) -> int:
        return int(lib().vsg_window_workspace_bytes(self._h, B, T, max_frames, precision))

    def __del__(self):
        try:
            if self._h and _lib is not None:
                _lib.vsg_pack_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass


def _weight_table(host: Dict[str, torch.Tensor]):
    arr = (VsgTensor * len(host))()
    keep = []
    for i, (k, v) in enumerate(host.items()):
        nm = k.encode()
        keep.append(nm)
        arr[i].name = nm
        arr[i].data = v.data_ptr()
        arr[i].ndim = v.dim()
        for d in range(v.dim()):
            arr[i].shape[d] = v.shape[d]
    return arr, keep


class EncPack:
    """Owner of the VsgPack* of a PosteriorEncoder (vsg_enc_pack_create)."""

    def __init__(self, cfg: VsgEncConfig, state_dict: Dict[str, torch.Tensor], prefix: str, device: torch.device):
        self._h = ctypes.c_void_p()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("visinger_b200: weights must live on a CUDA device; there is no CPU fallback")
        host = {k: v.detach().to("cpu", torch.float32).contiguous() for k, v in state_dict.items() if k.startswith(prefix)}
        arr, keep = _weight_table(host)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = lib().vsg_enc_pack_create(ctypes.byref(cfg), arr, len(host), prefix.encode(), idx, ctypes.byref(self._h))
        check(rc, "vsg_enc_pack_create")
        self.index = idx

    @property
    def handle(self):
        return self._h

    def workspace_bytes(self, B: int, T: int, precision: int) -> int:
        return int(lib().vsg_posterior_workspace_bytes(self._h, B, T, precision))

    def __del__(self):
        try:
            if self._h and _lib is not None:
                _lib.vsg_pack_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass


class RelEncPack:
    """Owner of the VsgPack* of a RelativeEncoder (vsg_relenc_pack_create) or, with frame_prior=True, of a whole
    FramePriorNetwork (encoder + proj; vsg_frame_prior_pack_create)."""

    def __init__(self, cfg: VsgRelEncConfig, state_dict: Dict[str, torch.Tensor], prefix: str, device: torch.device,
                 frame_prior: bool = False):
        self._h = ctypes.c_void_p()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("visinger_b200: weights must live on a CUDA device; there is no CPU fallback")
        host = {k: v.detach().to("cpu", torch.float32).contiguous() for k, v in state_dict.items() if k.startswith(prefix)}
        arr, keep = _weight_table(host)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        create = lib().vsg_frame_prior_pack_create if frame_prior else lib().vsg_relenc_pack_create
        rc = create(ctypes.byref(cfg), arr, len(host), prefix.encode(), idx, ctypes.byref(self._h))
        check(rc, "vsg_frame_prior_pack_create" if frame_prior else "vsg_relenc_pack_create")
        self.index = idx

    @property
    def handle(self):
        return self._h

    def workspace_bytes(self, B: int, T: int, g_per_frame: int, precision: int) -> int:
        return int(lib().vsg_relenc_workspace_bytes(self._h, B, T, g_per_frame, precision))

    def __del__(self):
        try:
            if self._h and _lib is not None:
                _lib.vsg_pack_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass


def position_freq(dim: int) -> torch.Tensor:
    """The frequencies of SinusoidalPositionalEmbedding.get_embedding, from the same torch expression (CPU fp32), so that
    the native table is that table: torch's fp32 exp is not correctly rounded."""
    half = dim // 2
    return torch.exp(torch.arange(half, dtype=torch.float) * -(math.log(10000) / (half - 1)))


class ModelPack:
    """Owner of the VsgPack* of a whole VISinger (vsg_model_pack_create): `state_dict` is the model's (reference
    checkpoint keys under `prefix`); the entry `prefix + "embed_positions.freq"` is added from `position_freq`."""

    def __init__(self, cfg: VsgModelConfig, state_dict: Dict[str, torch.Tensor], prefix: str, device: torch.device):
        self._h = ctypes.c_void_p()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("visinger_b200: weights must live on a CUDA device; there is no CPU fallback")
        host = {k: v.detach().to("cpu", torch.float32).contiguous() for k, v in state_dict.items() if k.startswith(prefix)}
        host[prefix + "embed_positions.freq"] = position_freq(cfg.hidden)
        arr, keep = _weight_table(host)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = lib().vsg_model_pack_create(ctypes.byref(cfg), arr, len(host), prefix.encode(), idx, ctypes.byref(self._h))
        check(rc, "vsg_model_pack_create")
        self.cfg = cfg
        self.index = idx
        self.hop = int(lib().vsg_hop_size(self._h))

    @property
    def handle(self):
        return self._h

    def workspace_bytes(self, B: int, T_ph: int, T: int, precision: int) -> int:
        return int(lib().vsg_model_workspace_bytes(self._h, B, T_ph, T, precision))

    def __del__(self):
        try:
            if self._h and _lib is not None:
                _lib.vsg_pack_destroy(self._h)
                self._h = ctypes.c_void_p()
        except Exception:
            pass


class ConvertPack(ModelPack):
    """Owner of the VsgPack* of a whole VISinger with its posterior encoder and linear spectrogram
    (vsg_convert_pack_create): everything a ModelPack holds, plus `prefix + "posterior_encoder.*"` and the DFT basis of
    a periodic Hann window of `win_length` samples."""

    def __init__(self, cfg: VsgModelConfig, state_dict: Dict[str, torch.Tensor], prefix: str, win_length: int,
                 device: torch.device):
        self._h = ctypes.c_void_p()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("visinger_b200: weights must live on a CUDA device; there is no CPU fallback")
        host = {k: v.detach().to("cpu", torch.float32).contiguous() for k, v in state_dict.items() if k.startswith(prefix)}
        host[prefix + "embed_positions.freq"] = position_freq(cfg.hidden)
        arr, keep = _weight_table(host)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = lib().vsg_convert_pack_create(ctypes.byref(cfg), arr, len(host), prefix.encode(), int(win_length), idx,
                                           ctypes.byref(self._h))
        check(rc, "vsg_convert_pack_create")
        self.cfg = cfg
        self.index = idx
        self.hop = int(lib().vsg_hop_size(self._h))
        self.bins = int(host[prefix + "posterior_encoder.pre.weight"].shape[1])
        self.win_length = int(win_length)

    def convert_workspace_bytes(self, B: int, T: int, precision: int) -> int:
        return int(lib().vsg_convert_workspace_bytes(self._h, B, T, precision))

    def convert_window_context(self):
        """(posterior, flow, decoder) context frames each side of a voice-conversion window (vsg_convert_window_context)."""
        cp, cf, cd = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        check(lib().vsg_convert_window_context(self._h, ctypes.byref(cp), ctypes.byref(cf), ctypes.byref(cd)),
              "vsg_convert_window_context")
        return int(cp.value), int(cf.value), int(cd.value)

    def convert_window_input(self, B: int, T: int, t0: int, t1: int, precision: int):
        """(s0, s1): the samples of each utterance's row that window [t0, t1) reads (vsg_convert_window_input)."""
        s0, s1 = ctypes.c_int64(), ctypes.c_int64()
        check(lib().vsg_convert_window_input(self._h, B, T, t0, t1, precision, ctypes.byref(s0), ctypes.byref(s1)),
              "vsg_convert_window_input")
        return int(s0.value), int(s1.value)

    def convert_window_workspace_bytes(self, B: int, T: int, max_frames: int, precision: int) -> int:
        return int(lib().vsg_convert_window_workspace_bytes(self._h, B, T, max_frames, precision))

    def spectrogram(self, wav: torch.Tensor, lengths: torch.Tensor, precision: int) -> torch.Tensor:
        """vsg_spectrogram: wav CUDA fp32 [B, T * hop], lengths CUDA int32 [B] (latent frames) -> fp32 [B, bins, T]."""
        require_cuda(wav, "wav")
        require_cuda(lengths, "lengths")
        B, L = wav.shape
        if L % self.hop or lengths.numel() != B:
            raise RuntimeError(f"expected wav [B, T * {self.hop}] and lengths [B]")
        T = L // self.hop
        w, ln = as_f32c(wav), lengths.to(torch.int32).contiguous()
        spec = torch.empty(B, self.bins, T, dtype=torch.float32, device=wav.device)
        if B == 0 or T == 0:
            return spec
        with torch.cuda.device(wav.device):
            ws = workspace(wav.device, self.convert_workspace_bytes(B, T, precision))
            rc = lib().vsg_spectrogram(self._h, w.data_ptr(), ln.data_ptr(), spec.data_ptr(), B, T, precision,
                                       ws.data_ptr(), ws.numel(), stream_ptr(wav.device))
        check(rc, "vsg_spectrogram")
        return spec


def normal_noise(seeds: torch.Tensor, C: int, T: int) -> torch.Tensor:
    """vsg_normal_noise: seeds CUDA int64 [B] (read as uint64) -> fp32 [B, C, T], element (b, c, t) a function of
    (seeds[b], c, t) only."""
    require_cuda(seeds, "seeds")
    s = seeds.to(torch.int64).contiguous()
    out = torch.empty(s.numel(), C, T, dtype=torch.float32, device=s.device)
    with torch.cuda.device(s.device):
        rc = lib().vsg_normal_noise(s.data_ptr(), out.data_ptr(), s.numel(), C, T, stream_ptr(s.device))
    check(rc, "vsg_normal_noise")
    return out


def debug_position_table(rows: int, dim: int, freq: Optional[torch.Tensor], device) -> torch.Tensor:
    """vsg_debug_position_table: the sinusoidal table [rows, dim] the model call builds (freq None = correctly rounded)."""
    device = torch.device(device)
    fq = as_f32c(freq.to(device)) if freq is not None else None
    out = torch.empty(rows, dim, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        rc = lib().vsg_debug_position_table(fq.data_ptr() if fq is not None else None, rows, dim, out.data_ptr(),
                                            stream_ptr(device))
    check(rc, "vsg_debug_position_table")
    return out


def length_regulate(enc: torch.Tensor, mel2ph: torch.Tensor, pos_table: Optional[torch.Tensor]) -> torch.Tensor:
    """enc [B, H, T_ph] fp32, mel2ph [B, T] int64, pos_table [rows, H] fp32 or None -> [B, H, T]  (vsg_length_regulate)."""
    require_cuda(enc, "enc")
    require_cuda(mel2ph, "mel2ph")
    ec = as_f32c(enc)
    mc = mel2ph.to(torch.int64).contiguous()
    B, H, T_ph = ec.shape
    T = mc.shape[1]
    tab = as_f32c(pos_table) if pos_table is not None else None
    if tab is not None:
        require_cuda(tab, "pos_table")
    y = torch.empty(B, H, T, dtype=torch.float32, device=enc.device)
    if B and T:
        with torch.cuda.device(enc.device):
            rc = lib().vsg_length_regulate(ec.data_ptr(), mc.data_ptr(), tab.data_ptr() if tab is not None else None,
                                           tab.shape[0] if tab is not None else 0, y.data_ptr(), B, H, T_ph, T,
                                           stream_ptr(enc.device))
        check(rc, "vsg_length_regulate")
    return y


_ws_cache: Dict[tuple, torch.Tensor] = {}


def workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Grow-only scratch buffer per (device, stream); allocated through torch's caching allocator."""
    stream = torch.cuda.current_stream(device)
    key = (device.index, stream.cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = None
        _ws_cache.pop(key, None)
        buf = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def release_workspaces() -> None:
    _ws_cache.clear()


def debug_conv1d_bf16(x_bld: torch.Tensor, w: torch.Tensor, bias, dilation: int, flags: int = 0, add0=None,
                      add1=None, scale: float = 1.0, want_bf16: bool = False, want_f32: bool = True, want_raw: bool = True):
    """Per-layer parity hook: one Conv1d (+ fused epilogue) on the tcgen05 kernel.
    x_bld / add0 / add1: CUDA bf16 [B, L, C] channels-last; w: [Cout, Cin, k] fp32 (any device).
    Returns out_f32 [B, L, Cout], or (out_f32, out_raw_bf16, out_act_bf16) when want_bf16."""
    require_cuda(x_bld, "x")
    assert x_bld.dtype == torch.bfloat16 and x_bld.is_contiguous()
    B, Lx, Cin = x_bld.shape
    planes = 3 if (flags & 256) else 2 if (flags & 4) else 1    # split-bf16: [hi | lo] ([hi | mid | lo]) planes per row
    Cin //= planes
    Cout, _, k = w.shape
    wh = w.detach().to("cpu", torch.float32).contiguous()
    bh = bias.detach().to("cpu", torch.float32).contiguous() if bias is not None else None
    dev = x_bld.device
    out = torch.empty(B, Lx, Cout, dtype=torch.float32, device=dev)
    raw = torch.zeros(B, Lx, planes * Cout, dtype=torch.bfloat16, device=dev) if (want_bf16 and want_raw) else None
    act = torch.zeros(B, Lx, planes * Cout, dtype=torch.bfloat16, device=dev) if want_bf16 else None
    for t in (add0, add1):
        assert t is None or (t.is_cuda and t.dtype == torch.bfloat16 and t.is_contiguous())
    torch.cuda.synchronize(dev)
    rc = lib().vsg_debug_conv1d_bf16(x_bld.data_ptr(), wh.data_ptr(), bh.data_ptr() if bh is not None else None,
                                     add0.data_ptr() if add0 is not None else None,
                                     add1.data_ptr() if add1 is not None else None, float(scale),
                                     out.data_ptr() if want_f32 else None,
                                     raw.data_ptr() if raw is not None else None, act.data_ptr() if want_bf16 else None,
                                     B, Lx, Cin, Cout, k, dilation, flags, dev.index or 0)
    check(rc, "vsg_debug_conv1d_bf16")
    return (out, raw, act) if want_bf16 else out


def _ptr(t):
    return t.data_ptr() if t is not None else None


def debug_conv_tc(x, w, bias=None, *, B, Lin, Lq, Lout=None, dil=1, in_off0=None, out_stride=1, out_phase=0, planes=1,
                  mode=EPI_TC_LINEAR, couple_sign=-1, add0_is_act=0, bcond=None, bcond_bs=0, mask=None, add0=None, add1=None,
                  out_raw=None, out_act=None, out_f32=None, scale=1.0, slope=0.1, x_ld=0, x_part_stride=0, ld=0,
                  part_stride=0, epi_sigs=2) -> int:
    """One launch of the convolution kernel through vsg_debug_conv_tc (include/visinger_b200.h).  x, bcond, mask, adds and
    outputs are caller-allocated CUDA tensors (outputs written in place); w [Cout, Cin, k] and bias [Cout] may live anywhere.
    in_off0 defaults to the centred -(k - 1) * dil / 2.  Returns the EPI_SIG_* image the launch ran."""
    require_cuda(x, "x")
    for t in (x, bcond, mask, add0, add1, out_raw, out_act, out_f32):
        assert t is None or (t.is_cuda and t.is_contiguous())
    Cout, Cin, k = w.shape
    wh = w.detach().to("cpu", torch.float32).contiguous()
    bh = bias.detach().to("cpu", torch.float32).contiguous() if bias is not None else None
    d = VsgDebugConv(_ptr(x), wh.data_ptr(), _ptr(bh), _ptr(bcond), _ptr(mask), _ptr(add0), _ptr(add1), _ptr(out_raw),
                     _ptr(out_act), _ptr(out_f32), planes, mode, couple_sign, add0_is_act, bcond_bs, scale, slope, B, Lin,
                     Cin, Cout, k, dil, -((k - 1) * dil // 2) if in_off0 is None else in_off0, Lq, out_stride, out_phase,
                     Lq if Lout is None else Lout, x_ld, x_part_stride, ld, part_stride, epi_sigs)
    img = ctypes.c_int32(-1)
    torch.cuda.synchronize(x.device)
    check(lib().vsg_debug_conv_tc(ctypes.byref(d), ctypes.byref(img), x.device.index or 0), "vsg_debug_conv_tc")
    return int(img.value)


def debug_upsample_tc(x, w, bias, rate: int, flags: int, out_act, out_raw=None, out_f32=None) -> int:
    """The decoder's upsampler through vsg_debug_upsample_tc: x CUDA bf16 (layout per flags), w [Cin, Cout, k] (the
    ConvTranspose1d weight), bias [Cout]; caller-allocated outputs.  Returns the EPI_SIG_* image of the last launch."""
    require_cuda(x, "x")
    for t in (x, out_act, out_raw, out_f32):
        assert t is None or (t.is_cuda and t.is_contiguous())
    Cin, Cout, k = w.shape
    B, Lin = x.shape[-3], x.shape[-2]
    wh = w.detach().to("cpu", torch.float32).contiguous()
    bh = bias.detach().to("cpu", torch.float32).contiguous()
    img = ctypes.c_int32(-1)
    torch.cuda.synchronize(x.device)
    check(lib().vsg_debug_upsample_tc(x.data_ptr(), wh.data_ptr(), bh.data_ptr(), Cin, Cout, rate, k, B, Lin, out_act.data_ptr(),
                                      _ptr(out_raw), _ptr(out_f32), flags, ctypes.byref(img), x.device.index or 0),
          "vsg_debug_upsample_tc")
    return int(img.value)


def debug_conv_f32_plan(Cout: int, k: int, dil: int):
    """vsg_debug_conv_f32_plan (host only): (warps along channels, warps along time, dynamic shared memory bytes), or None
    where the kernel refuses the shape (VSG_EUNSUPPORTED)."""
    out = (ctypes.c_int32 * 3)()
    rc = lib().vsg_debug_conv_f32_plan(Cout, k, dil, out)
    if rc == -4:
        return None
    check(rc, "vsg_debug_conv_f32_plan")
    return int(out[0]), int(out[1]), int(out[2])


def debug_conv_f32(x, w, bias=None, *, B, Cin, Lin, Lq, Lout=None, x_bs=None, x_cs=None, dil=1, in_off0=None,
                   pre_lrelu=0, slope=0.1, bcond=None, bcond_bs=0, out_stride=1, out_phase=0, epi=0, y=None, y_bs=None,
                   y_cs=None, res=None, res_bs=None, res_cs=None, y2=None, y2_bs=None, y2_cs=None, mask=None, mask_bs=None,
                   acc_mode=ACC_SET, acc_div=1.0, rs_split=0, y2_first=0, y2_mask=0, couple_sign=1, gate_interleave=0,
                   check_rc=True):
    """One launch of the fp32 convolution kernel through vsg_debug_conv_f32 (include/visinger_b200.h).  Tensors are flat
    CUDA fp32 buffers addressed through the given strides (outputs written in place); strides default to a dense
    [B, C, L] layout.  w [Cout, Cin, k] and bias [Cout] may live anywhere.  in_off0 defaults to -(k - 1) * dil / 2.
    Returns ((warps along channels, warps along time), rc); raises on an error unless check_rc is False."""
    for t in (x, bcond, res, mask, y, y2):
        assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous())
    Cout, wc, k = w.shape
    assert wc == Cin
    Lout = Lq if Lout is None else Lout
    x_cs = Lin if x_cs is None else x_cs
    x_bs = Cin * x_cs if x_bs is None else x_bs
    ych = Cout // 2 if epi in (1, 4) else (rs_split if epi == 2 else Cout)
    y_cs = Lout if y_cs is None else y_cs
    y_bs = ych * y_cs if y_bs is None else y_bs
    res_cs = Lout if res_cs is None else res_cs
    res_bs = Cout * res_cs if res_bs is None else res_bs
    y2_cs = Lout if y2_cs is None else y2_cs
    y2_bs = (Cout - rs_split) * y2_cs if y2_bs is None else y2_bs
    mask_bs = Lout if mask_bs is None else mask_bs
    wh = w.detach().to("cpu", torch.float32).contiguous()
    bh = bias.detach().to("cpu", torch.float32).contiguous() if bias is not None else None
    d = VsgDebugConvF32(_ptr(x), wh.data_ptr(), _ptr(bh), _ptr(bcond), _ptr(res), _ptr(mask), _ptr(y), _ptr(y2),
                        x_bs, y_bs, res_bs, y2_bs, x_cs, y_cs, res_cs, y2_cs, B, Cin, Lin, Cout, k, dil,
                        -((k - 1) * dil // 2) if in_off0 is None else in_off0, pre_lrelu, slope, bcond_bs, mask_bs, Lq,
                        out_stride, out_phase, Lout, epi, acc_mode, acc_div, rs_split, y2_first, y2_mask, couple_sign,
                        gate_interleave)
    tile = (ctypes.c_int32 * 2)()
    dev = x.device if x is not None else torch.device("cuda", 0)
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
    rc = lib().vsg_debug_conv_f32(ctypes.byref(d), tile, dev.index or 0)
    if check_rc:
        check(rc, "vsg_debug_conv_f32")
    return (int(tile[0]), int(tile[1])), rc


def debug_upsample_f32(x, w, bias, rate: int, y) -> None:
    """The fp32 decoder's upsampler through vsg_debug_upsample_f32: x CUDA fp32 [B, Cin, Lin], w [Cin, Cout, k] (the
    ConvTranspose1d weight) and bias [Cout] anywhere, y CUDA fp32 [B, Cout, Lin * rate] written in place."""
    require_cuda(x, "x")
    for t in (x, y):
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
    Cin, Cout, k = w.shape
    B, _, Lin = x.shape
    wh = w.detach().to("cpu", torch.float32).contiguous()
    bh = bias.detach().to("cpu", torch.float32).contiguous()
    torch.cuda.synchronize(x.device)
    check(lib().vsg_debug_upsample_f32(x.data_ptr(), wh.data_ptr(), bh.data_ptr(), Cin, Cout, rate, k, B, Lin, y.data_ptr(),
                                       x.device.index or 0), "vsg_debug_upsample_f32")


def debug_conv_post_f32(x, w, slope: float, n0: int, n1: int, wav, wav_ld: int) -> None:
    """The fp32 conv_post through vsg_debug_conv_post_f32: x CUDA fp32 [B, C, L], w [C, k] anywhere; samples [n0, n1) of
    utterance b are written to wav (flat CUDA fp32) at b * wav_ld."""
    require_cuda(x, "x")
    assert x.dtype == torch.float32 and x.is_contiguous() and wav.is_cuda and wav.is_contiguous()
    B, C, L = x.shape
    k = w.shape[-1]
    wh = w.detach().to("cpu", torch.float32).reshape(C, k).contiguous()
    torch.cuda.synchronize(x.device)
    check(lib().vsg_debug_conv_post_f32(x.data_ptr(), wh.data_ptr(), C, L, k, float(slope), B, n0, n1, wav.data_ptr(),
                                        int(wav_ld), x.device.index or 0), "vsg_debug_conv_post_f32")


def debug_cond_f32(W, bias, g, out) -> None:
    """The condition GEMV through vsg_debug_cond_f32: W [O, I], bias [O] or None, g [B, I], out [B, O], CUDA fp32."""
    for t in (W, bias, g, out):
        assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous())
    O, I = W.shape
    B = g.shape[0]
    torch.cuda.synchronize(W.device)
    check(lib().vsg_debug_cond_f32(W.data_ptr(), _ptr(bias), g.data_ptr(), out.data_ptr(), O, I, B, W.device.index or 0),
          "vsg_debug_cond_f32")


def debug_pair_bf16(xa_bld: torch.Tensor, w1, b1, w2, b2, d1: int, add0=None, add1=None, scale: float = 1.0,
                    want_f32: bool = True, want_raw: bool = True):
    """Per-layer parity hook of the fused ResBlock1 pair kernel.  xa_bld / add0 / add1: CUDA bf16 [B, L, C];
    returns (out_f32, out_raw_bf16, out_act_bf16)."""
    require_cuda(xa_bld, "xa")
    assert xa_bld.dtype == torch.bfloat16 and xa_bld.is_contiguous()
    B, Lx, C = xa_bld.shape
    k = w1.shape[2]
    h = [t.detach().to("cpu", torch.float32).contiguous() for t in (w1, b1, w2, b2)]
    dev = xa_bld.device
    out = torch.zeros(B, Lx, C, dtype=torch.float32, device=dev) if want_f32 else None
    raw = torch.zeros(B, Lx, C, dtype=torch.bfloat16, device=dev) if want_raw else None
    act = torch.zeros(B, Lx, C, dtype=torch.bfloat16, device=dev)
    torch.cuda.synchronize(dev)
    rc = lib().vsg_debug_pair_bf16(xa_bld.data_ptr(), h[0].data_ptr(), h[1].data_ptr(), h[2].data_ptr(), h[3].data_ptr(),
                                   add0.data_ptr() if add0 is not None else None,
                                   add1.data_ptr() if add1 is not None else None, float(scale),
                                   out.data_ptr() if want_f32 else None,
                                   raw.data_ptr() if raw is not None else None, act.data_ptr(), B, Lx, C, k, d1,
                                   dev.index or 0)
    check(rc, "vsg_debug_pair_bf16")
    return out, raw, act


def debug_pair_tc(xa, w1, b1, w2, b2, d1: int, *, add0=None, add0_is_act=0, add1=None, scale=1.0, out_raw=None,
                  out_act=None, out_f32=None) -> int:
    """The fused ResBlock1 pair through vsg_debug_pair_tc (include/visinger_b200.h).  xa, adds and outputs are
    caller-allocated CUDA tensors [B, L, C] (outputs written in place); w1 / w2 [C, C, k] and b1 / b2 [C] may live anywhere.
    Returns the EPI_SIG_* image of conv2's epilogue."""
    require_cuda(xa, "xa")
    for t in (xa, add0, add1, out_raw, out_act, out_f32):
        assert t is None or (t.is_cuda and t.is_contiguous())
    B, L, C = xa.shape
    k = w1.shape[2]
    h = [t.detach().to("cpu", torch.float32).contiguous() for t in (w1, b1, w2, b2)]
    d = VsgDebugPair(xa.data_ptr(), *[t.data_ptr() for t in h], _ptr(add0), _ptr(add1), _ptr(out_raw), _ptr(out_act),
                     _ptr(out_f32), add0_is_act, scale, B, L, C, k, d1)
    img = ctypes.c_int32(-1)
    torch.cuda.synchronize(xa.device)
    check(lib().vsg_debug_pair_tc(ctypes.byref(d), ctypes.byref(img), xa.device.index or 0), "vsg_debug_pair_tc")
    return int(img.value)


def debug_resblock_bf16(xa_bld: torch.Tensor, ws, bs, dilations, add1=None, scale: float = 1.0, max_mb: int = 0, sets: int = 0,
                        want_raw: bool = True, want_act: bool = True, reps: int = 1, want_f32: bool = True):
    """Per-layer parity hook of the whole-ResBlock1 kernel (csrc/rb_tc.cuh).  xa_bld / add1: CUDA bf16 [B, L, C];
    ws / bs: lists [c1_0, c2_0, c1_1, c2_1, ...] of fp32 [C, C, k] / [C].  Returns (out_f32, out_raw_bf16, out_act_bf16[, ms]).
    sets bit 11 (with bit 8): the row-packed kernel's split-bf16 instantiation -- xa / add1 / raw / act are two-plane
    tensors [B, L, 2 C] (`split_bf16`), out_f32 stays [B, L, C].  (The kernel takes xa / add1 and writes raw as planar
    tensors [2][B, L, C]; the conversion from / to the decoder's rows [hi | lo] happens here.)"""
    require_cuda(xa_bld, "xa")
    assert xa_bld.dtype == torch.bfloat16 and xa_bld.is_contiguous()
    B, Lx, C = xa_bld.shape
    x3 = bool(sets & 2048)
    if x3:
        assert C % 2 == 0
        C //= 2
        xa_bld = torch.stack([xa_bld[..., :C], xa_bld[..., C:]]).contiguous()
        if add1 is not None:
            add1 = torch.stack([add1[..., :C], add1[..., C:]]).contiguous()
    k = ws[0].shape[2]
    n_pairs = len(dilations)
    assert len(ws) == 2 * n_pairs and len(bs) == 2 * n_pairs
    wh = torch.stack([w.detach().to("cpu", torch.float32) for w in ws]).contiguous()
    bh = torch.stack([b.detach().to("cpu", torch.float32) for b in bs]).contiguous()
    dl = (ctypes.c_int32 * n_pairs)(*[int(d) for d in dilations])
    dev = xa_bld.device
    out = torch.zeros(B, Lx, C, dtype=torch.float32, device=dev) if want_f32 else None
    raw = torch.zeros((2, B, Lx, C) if x3 else (B, Lx, C), dtype=torch.bfloat16, device=dev) if want_raw else None
    act = torch.zeros(B, Lx, (2 if x3 else 1) * C, dtype=torch.bfloat16, device=dev) if want_act else None
    assert add1 is None or (add1.is_cuda and add1.dtype == torch.bfloat16 and add1.is_contiguous())
    torch.cuda.synchronize(dev)
    if reps > 1:
        lib().vsg_debug_set_plan(0, 0, -1, -1, reps)
    try:
        rc = lib().vsg_debug_resblock_bf16(xa_bld.data_ptr(), wh.data_ptr(), bh.data_ptr(), n_pairs, dl,
                                           add1.data_ptr() if add1 is not None else None, float(scale),
                                           out.data_ptr() if out is not None else None, raw.data_ptr() if raw is not None else None,
                                           act.data_ptr() if act is not None else None, B, Lx, C, k, int(max_mb), int(sets),
                                           dev.index or 0)
        ms = float(lib().vsg_debug_last_ms()) if reps > 1 else None
    finally:
        if reps > 1:
            lib().vsg_debug_set_plan(0, 0, -1, -1, 1)
    check(rc, "vsg_debug_resblock_bf16")
    if x3 and raw is not None:
        raw = torch.cat([raw[0], raw[1]], dim=-1)
    return (out, raw, act, ms) if reps > 1 else (out, raw, act)


def _debug_attention(name, qkv, mask, ek, ev, n_heads: int, channels_last: bool, *extra):
    require_cuda(qkv, "qkv")
    assert qkv.is_contiguous()
    B, T = (qkv.shape[0], qkv.shape[1]) if channels_last else (qkv.shape[0], qkv.shape[2])
    H = (qkv.shape[2] if channels_last else qkv.shape[1]) // 3
    nrel, dk = ek.shape
    dev = qkv.device
    mask, ek, ev = (as_f32c(t.to(dev)).reshape(-1) for t in (mask, ek, ev))
    assert mask.numel() == B * T and ev.numel() == nrel * dk and nrel % 2 == 1 and H == n_heads * dk
    o = torch.zeros((B, T, H) if channels_last else (B, H, T), dtype=qkv.dtype, device=dev)
    torch.cuda.synchronize(dev)
    rc = getattr(lib(), name)(qkv.data_ptr(), mask.data_ptr(), ek.data_ptr(), ev.data_ptr(), o.data_ptr(), B, T, n_heads, dk,
                              (nrel - 1) // 2, *extra, dev.index or 0)
    check(rc, name)
    return o


def debug_attention_bf16(qkv_btc: torch.Tensor, mask, ek, ev, n_heads: int) -> torch.Tensor:
    """Per-kernel parity hook of the tcgen05 attention kernel (csrc/attn_tc.cuh).  qkv_btc: CUDA bf16 [B, T, 3H]
    (q | k | v, channels-last, as the fused QKV projection writes it); mask [B, T] (or [B, 1, T]); ek / ev: [2w+1, dk]
    fp32.  Returns o: bf16 [B, T, H]."""
    assert qkv_btc.dtype == torch.bfloat16
    return _debug_attention("vsg_debug_attention_bf16", qkv_btc, mask, ek, ev, n_heads, True)


def debug_attention_split_bf16(qkv_btc: torch.Tensor, mask, ek, ev, n_heads: int, key_chunk: int = 0) -> torch.Tensor:
    """Per-kernel parity hook of the split-key attention path (csrc/attn_tc.cuh split mode + combine) at any T: keys in
    chunks of key_chunk frames (a multiple of 128 up to 2048; 0 = 2048, the encoder's choice beyond T = 2048).  Same
    arguments and result as debug_attention_bf16."""
    assert qkv_btc.dtype == torch.bfloat16
    return _debug_attention("vsg_debug_attention_split_bf16", qkv_btc, mask, ek, ev, n_heads, True, int(key_chunk))


def debug_attention_f32(qkv_bct: torch.Tensor, mask, ek, ev, n_heads: int) -> torch.Tensor:
    """Per-kernel parity hook of the fp32 attention kernel (csrc/relenc_f32.cuh).  qkv_bct: CUDA fp32 [B, 3H, T];
    returns o: fp32 [B, H, T]."""
    assert qkv_bct.dtype == torch.float32
    return _debug_attention("vsg_debug_attention_f32", qkv_bct, mask, ek, ev, n_heads, False)


def debug_layernorm_bf16(x_btc: torch.Tensor, gamma, beta, mask, g=None, eps: float = 1e-4) -> torch.Tensor:
    """Per-kernel parity hook of the bf16 encoder's LayerNorm -> + g -> * mask step (csrc/relenc_tc.cuh), on a copy of
    x_btc (CUDA bf16 [B, T, C]); g: None, [B, C] per utterance or [B, C, T] per frame.  Returns the bf16 result."""
    require_cuda(x_btc, "x")
    assert x_btc.dtype == torch.bfloat16
    B, T, C = x_btc.shape
    dev = x_btc.device
    y = x_btc.contiguous().clone()
    gamma, beta, mask = (as_f32c(t.to(dev)) for t in (gamma, beta, mask))
    assert mask.numel() == B * T
    g_t = 0
    if g is not None:
        g = as_f32c(g.to(dev))
        g_t = 1 if g.dim() == 3 else 0
        assert g.shape == ((B, C, T) if g_t else (B, C))
    torch.cuda.synchronize(dev)
    rc = lib().vsg_debug_layernorm_bf16(y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), g.data_ptr() if g is not None else None,
                                        g_t, mask.data_ptr(), float(eps), B, T, C, dev.index or 0)
    check(rc, "vsg_debug_layernorm_bf16")
    return y


def split_bf16(x: torch.Tensor) -> torch.Tensor:
    """[..., C] fp32 -> [..., 2C] bf16 planes [hi | lo] with hi = bf16(x), lo = bf16(x - hi)."""
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.cat([hi, lo], dim=-1).contiguous()


def merge_bf16(x: torch.Tensor) -> torch.Tensor:
    """Inverse view of split_bf16: [..., 2C] bf16 planes -> [..., C] fp32 = hi + lo."""
    C = x.shape[-1] // 2
    return x[..., :C].float() + x[..., C:].float()


def set_tc_options(halo_mode: int = 1, w_resident: int = 1, l2_tensor_mb: int = -1, min_tiles: int = -1) -> None:
    check(lib().vsg_set_tc_options(int(halo_mode), int(w_resident), int(l2_tensor_mb), int(min_tiles)),
          "vsg_set_tc_options")


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream
