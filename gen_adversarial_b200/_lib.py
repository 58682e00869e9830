"""ctypes loader for libga_b200.so (the C-ABI declared in include/ga_b200.h).

The product path has NO fallback: if the shared library is missing or a symbol is absent this module
raises, and every op wrapper in `ops.py` raises RuntimeError when an entry point returns non-zero
(message from `ga_last_error()`), mirroring TORCH_CHECK in the reference's
src/mlvgms_autoencoders/StyleGan_E4E/stylegan2/op/fused_bias_act.cpp:7-9.
"""
from __future__ import annotations

import ctypes
import glob
import os
import re
import subprocess
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT_DIR = os.path.dirname(PKG_DIR)
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libga_b200.so")
HEADER = os.path.join(ROOT_DIR, "include", "ga_b200.h")

GA_F32, GA_BF16 = 0, 1
PRE_NONE, PRE_ELU, PRE_SILU, PRE_AFFINE_SILU, PRE_AFFINE = 0, 1, 2, 3, 4
ACT_NONE, ACT_SILU, ACT_ELU, ACT_RELU, ACT_LRELU_SQRT2, ACT_PRELU = 0, 1, 2, 3, 4, 5
MUL_VALUE, MUL_RELU_MASK, MUL_ELU_FROM_Y, MUL_PRELU_FROM_Y = 0, 1, 2, 3

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


class GaTensor(ctypes.Structure):
    _fields_ = [("data", c_void_p), ("dtype", c_int32), ("n", c_int32), ("h", c_int32), ("w", c_int32), ("c", c_int32)]


class GaConvDesc(ctypes.Structure):
    _fields_ = [("kh", c_int32), ("kw", c_int32), ("stride", c_int32), ("pad", c_int32), ("up", c_int32),
                ("pre_op", c_int32), ("post_act", c_int32),
                ("pre_scale", c_void_p), ("pre_shift", c_void_p), ("weight", c_void_p), ("bias", c_void_p),
                ("tf32", c_int32), ("ktot", c_int32),
                ("mul", c_void_p), ("mul_dtype", c_int32), ("mul_mode", c_int32),
                ("dact_out", c_void_p), ("dact_dtype", c_int32), ("act_after_add", c_int32), ("act_slope", c_void_p),
                ("csum_out", c_void_p)]


def sources():
    return sorted(glob.glob(os.path.join(CSRC_DIR, "*.cu")))


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(CSRC_DIR, "*.cuh")) + [HEADER]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> gen_adversarial_b200/libga_b200.so (in-tree).
    Every .cu is compiled to its own object (in parallel, cached by mtime under csrc/_build/) and linked with nvcc -shared."""
    if not force and not _stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    obj_dir = os.path.join(CSRC_DIR, "_build")
    os.makedirs(obj_dir, exist_ok=True)
    hdr_t = max(os.path.getmtime(d) for d in glob.glob(os.path.join(CSRC_DIR, "*.cuh")) + [HEADER])
    cflags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_t):
            return obj, ""
        cmd = [nvcc] + cflags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
        return obj, res.stderr

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, sources()))
    if verbose:
        print("".join(r[1] for r in results))
    res = subprocess.run([nvcc, "-shared", "-o", LIB_PATH] + [r[0] for r in results], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + res.stdout + res.stderr)
    return LIB_PATH


def declared_symbols():
    """every function name declared in include/ga_b200.h"""
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(ga_[a-z0-9_]+)\s*\(", txt)))


_LIB = None

T = POINTER(GaTensor)
D = POINTER(GaConvDesc)

_PROTOS = {
    "ga_last_error": (c_char_p, []),
    "ga_abi_version": (c_int, []),
    "ga_f32_round_tf32": (c_int, [c_int]),
    "ga_launch_count": (c_int64, [c_int]),
    "ga_seed_salt_set": (c_int, [c_void_p]),
    "ga_seed_salt_bump": (c_int, [c_void_p]),
    "ga_noise_sumsq_parts": (c_int, [c_int]),
    "ga_channel_sum_parts": (c_int, [c_int, c_int]),
    "ga_noise_sumsq": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "ga_noise_sumsq_philox": (c_int, [c_uint64, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "ga_preprocess_image_supported": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "ga_preprocess_image_fwd": (c_int, [c_void_p, c_void_p, c_uint64, c_int64, c_float, c_void_p, c_int, c_int, T, c_void_p, c_void_p]),
    "ga_preprocess_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_int64, c_float, c_void_p, c_int, c_int, T,
                                  c_void_p, c_void_p]),
    "ga_preprocess_bwd": (c_int, [T, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "ga_conv2d_simt": (c_int, [T, D, T, T, c_void_p]),
    "ga_conv2d_tc": (c_int, [T, T, D, T, T, T, c_void_p]),
    "ga_conv2d_tc_csum_supported": (c_int, [T, D, c_int]),
    "ga_conv2d_tc_supported": (c_int, [T, T, D, c_int]),
    "ga_dwconv5x5_fwd": (c_int, [T, c_void_p, c_void_p, c_int, c_int, T, c_void_p]),
    "ga_dwconv5x5_ex": (c_int, [T, T, c_void_p, c_void_p, c_int, c_int, T, T, c_void_p]),
    "ga_channel_sum": (c_int, [T, c_void_p, c_void_p]),
    "ga_affine_act_bwd": (c_int, [T, T, c_void_p, c_void_p, c_int, T, T, c_void_p]),
    "ga_add": (c_int, [T, T, T, c_void_p]),
    "ga_se_residual_bwd": (c_int, [T, T, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float, T, c_void_p]),
    "ga_sumpool2x2": (c_int, [T, T, T, c_void_p]),
    "ga_upsample_bilinear2x_bwd": (c_int, [T, T, c_void_p]),
    "ga_depth_to_space2": (c_int, [T, T, c_void_p]),
    "ga_phase_interleave": (c_int, [T, T, T, c_int, c_void_p, T, c_void_p]),
    "ga_subsample2x_bwd": (c_int, [T, T, c_void_p]),
    "ga_codes_assemble_bwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ga_maxpool3x3s2_bwd": (c_int, [T, T, c_int, T, c_void_p]),
    "ga_avgpool_bwd_relu": (c_int, [T, T, T, c_void_p]),
    "ga_maxpool2x2_bwd": (c_int, [T, T, c_int, T, c_void_p]),
    "ga_latent_mix_bwd": (c_int, [T, T, T, c_void_p, c_uint64, c_int, c_int64, c_void_p, c_float, c_int, T, T, c_void_p]),
    "ga_discmix_mean_bwd": (c_int, [T, c_int, c_void_p, T, T, c_void_p]),
    "ga_se_residual_fwd": (c_int, [T, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float, T, T, T, T,
                                   c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "ga_mbconv_fused_supported": (c_int, [T, c_int]),
    "ga_debug_mbconv_trace": (c_int, [c_void_p]),
    "ga_debug_c3_trace": (c_int, [c_void_p]),
    "ga_tc_halo_enable": (c_int, [c_int]),
    "ga_mbconv_fused": (c_int, [T, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, T, c_void_p]),
    "ga_torgb_fused": (c_int, [T, c_void_p, c_void_p, T, c_void_p, T, c_void_p]),
    "ga_mbconv_fused_bwd": (c_int, [T, c_void_p, c_void_p, T, T, c_void_p, T, c_int, T, c_void_p]),
    "ga_mbconv_fused_ex": (c_int, [T, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, T, c_void_p, T, T, c_void_p]),
    "ga_add_layernorm": (c_int, [T, T, c_void_p, c_void_p, c_float, T, T, c_void_p]),
    "ga_attention_ws_floats": (c_int64, [c_int, c_int, c_int, c_int]),
    "ga_attention": (c_int, [T, c_int, T, c_int, T, c_int, c_int, c_int, c_void_p, T, c_void_p]),
    "ga_codes_assemble": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ga_resize_bilinear": (c_int, [T, c_int, c_int, T, c_void_p]),
    "ga_image_pool_out": (c_int, [T, c_int, c_int, c_int, c_float, c_float, c_void_p, T, c_void_p]),
    "ga_philox_codes": (c_int, [c_uint64, c_int64, c_float, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ga_latent_mix_fwd": (c_int, [T, T, c_void_p, c_uint64, c_int, c_int64, c_void_p, c_float, c_int, T, c_void_p]),
    "ga_latent_level": (c_int, [T, T, T, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_uint64, c_int, c_int64, c_void_p,
                                c_float, c_int, T, T, T, c_void_p]),
    "ga_discmix_mean_fwd": (c_int, [T, c_int, c_void_p, T, c_void_p]),
    "ga_upsample_nearest2x": (c_int, [T, T, c_void_p]),
    "ga_upsample_bilinear2x": (c_int, [T, T, c_void_p]),
    "ga_maxpool2x2": (c_int, [T, T, c_void_p]),
    "ga_cast": (c_int, [T, T, c_void_p]),
    "ga_subsample2x": (c_int, [T, T, c_void_p]),
    "ga_maxpool3x3s2": (c_int, [T, T, c_void_p]),
    "ga_global_avgpool": (c_int, [T, T, c_void_p]),
    "ga_affine_act": (c_int, [T, c_void_p, c_void_p, c_int, T, c_void_p]),
    "ga_nchw_to_nhwc": (c_int, [c_void_p, T, c_float, c_float, c_void_p]),
    "ga_pixelnorm": (c_int, [c_void_p, c_int, c_int, T, c_void_p]),
    "ga_style_demod": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ga_channel_scale": (c_int, [T, c_void_p, T, c_void_p]),
    "ga_styled_bias_act": (c_int, [T, c_int, c_void_p, c_void_p, c_float, c_void_p, c_int, T, c_void_p, c_void_p, T, c_void_p, T, c_void_p]),
    "ga_upfirdn2d": (c_int, [T, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, T, c_void_p]),
    "ga_avgpool_to_nchw": (c_int, [T, c_int, c_int, c_void_p, c_void_p]),
    "ga_latent_lerp": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ga_styled_bias_act_bwd_parts": (c_int, [c_int, c_int]),
    "ga_styled_bias_act_bwd": (c_int, [T, T, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, T,
                                       c_void_p, c_void_p, c_void_p, c_void_p]),
    "ga_style_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ga_latent_lerp_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ga_image_pool_out_bwd": (c_int, [c_void_p, T, c_int, c_int, c_int, c_float, T, c_void_p]),
    "ga_apgd_l2_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_int, c_int, c_void_p]),
    "ga_fgsm_l2_step": (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_void_p]),
    "ga_l2_ball_start": (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_void_p]),
    "ga_pgd_linf_step": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_float, c_int64, c_void_p]),
    "ga_softmax_xent": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
}


def lib():
    """Load (building first if the in-tree .so is missing/stale and nvcc is available)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if _stale():
        build_library()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(L, name, None)
        if fn is None:
            raise RuntimeError(f"libga_b200.so does not export {name}")
        fn.restype = res
        fn.argtypes = args
    if L.ga_abi_version() != 11:
        raise RuntimeError("libga_b200.so ABI version mismatch")
    _LIB = L
    return L


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().ga_last_error().decode(errors="replace")
        raise RuntimeError(f"libga_b200 {what} failed (rc={rc}): {msg}")
