"""ctypes binding of the C-ABI CUDA library (``include/te_b200.h``).

There is no CPU fallback: if ``lib/libte_b200.so`` is missing (and cannot be built with nvcc)
importing this module raises, and every call checks the returned status code.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libte_b200.so")

c_int, c_ll, c_uint, c_void_p, c_char_p, c_float = (ctypes.c_int, ctypes.c_longlong, ctypes.c_uint, ctypes.c_void_p,
                                                    ctypes.c_char_p, ctypes.c_float)


class TeVitConfig(ctypes.Structure):
    """``te_vit_config`` of include/te_b200.h."""
    _fields_ = [("img_size", c_int), ("patch_size", c_int), ("in_chans", c_int), ("num_classes", c_int),
                ("dim", c_int), ("depth", c_int), ("heads", c_int), ("mlp_dim", c_int), ("distilled", c_int),
                ("eps_block", c_float), ("eps_final", c_float)]


class TeBertConfig(ctypes.Structure):
    """``te_bert_config`` of include/te_b200.h."""
    _fields_ = [("vocab_size", c_int), ("max_position", c_int), ("type_vocab", c_int), ("hidden", c_int),
                ("layers", c_int), ("heads", c_int), ("intermediate", c_int), ("num_labels", c_int),
                ("layer_norm_eps", c_float)]


FLAG_ZPLUS_TENSOR_CORES = 1
FLAG_ROLLOUT_FUSED = 2
FLAG_KEEP_ALL_CAMS = 4
FLAG_RELPROP_TO_INPUT = 8
FLAG_GRADIENTS_ONLY = 128
FLAG_LINEAR_TENSOR_CORES = 16
FLAG_ATTN_TENSOR_CORES = 32
FLAG_ZPLUS_BF16 = 64
FLAG_BACKWARD_TF32 = 256
FLAG_RULES_LRP = 512
FLAG_RELPROP_TF32 = 1024
FLAG_ZPLUS_S1_BF16 = 2048
FLAG_LINEAR_F16_SPLIT = 4096
FLAG_ZPLUS_R_F16 = 8192
FLAG_BACKWARD_F16 = 16384
FLAG_TENSOR_CORES = FLAG_ZPLUS_TENSOR_CORES | FLAG_LINEAR_TENSOR_CORES      # the ones that need derived weights
FLAG_ALL_FAST = FLAG_TENSOR_CORES | FLAG_ATTN_TENSOR_CORES | FLAG_ROLLOUT_FUSED
# what bench.py runs by default: updated as faster selections pass the parity tests (tests/test_gpu_parity_full.py)
FLAG_BENCH_DEFAULT = FLAG_ALL_FAST | FLAG_BACKWARD_TF32 | FLAG_RELPROP_TF32 | FLAG_ZPLUS_S1_BF16 | FLAG_LINEAR_F16_SPLIT

_P = c_void_p
_CFG = ctypes.POINTER(TeVitConfig)
_BCFG = ctypes.POINTER(TeBertConfig)

# name -> (restype, argtypes)   — exactly the prototypes of include/te_b200.h
PROTOTYPES = {
    "te_last_error": (c_char_p, []),
    "te_version": (c_int, []),
    "te_kernel_launch_count": (c_ll, []),
    "te_vit_num_weights": (c_int, [_CFG]),
    "te_vit_weight_name": (c_char_p, [_CFG, c_int]),
    "te_vit_weight_numel": (c_ll, [_CFG, c_int]),
    "te_vit_weight_offset": (c_ll, [_CFG, c_int]),
    "te_vit_weight_total": (c_ll, [_CFG]),
    "te_vit_workspace_bytes": (c_ll, [_CFG, c_int]),
    "te_vit_forward": (c_int, [_CFG, _P, _P, _P, c_int, c_uint, _P, _P, c_ll, _P]),
    "te_vit_derived_total": (c_ll, [_CFG]),
    "te_vit_prepare_derived": (c_int, [_CFG, _P, _P, _P]),
    "te_vit_attribute": (c_int, [_CFG, _P, _P, c_int, _P, c_int, c_uint, _P, _P, c_ll, _P]),
    "te_vit_explain": (c_int, [_CFG, _P, _P, _P, c_int, _P, c_int, c_uint, _P, _P, _P, c_ll, _P]),
    "te_vit_tensor": (c_int, [_CFG, c_int, _P, c_char_p, c_int, ctypes.POINTER(_P), ctypes.POINTER(c_ll),
                              ctypes.POINTER(c_ll)]),
    "te_set_option": (c_int, [c_char_p, c_int]),
    "te_vit_relprop_pixels": (c_int, [_CFG, _P, _P, c_int, _P, _P, _P, c_ll, _P]),
    "te_vit_relprop_pixels_ex": (c_int, [_CFG, _P, _P, c_int, c_uint, _P, _P, _P, c_ll, _P]),
    "te_bert_num_weights": (c_int, [_BCFG]),
    "te_bert_weight_name": (c_char_p, [_BCFG, c_int]),
    "te_bert_weight_numel": (c_ll, [_BCFG, c_int]),
    "te_bert_weight_offset": (c_ll, [_BCFG, c_int]),
    "te_bert_weight_total": (c_ll, [_BCFG]),
    "te_bert_derived_total": (c_ll, [_BCFG]),
    "te_bert_prepare_derived": (c_int, [_BCFG, _P, _P, _P]),
    "te_bert_workspace_bytes": (c_ll, [_BCFG, c_int, c_int]),
    "te_bert_forward": (c_int, [_BCFG, _P, _P, _P, _P, c_int, c_int, c_uint, _P, _P, c_ll, _P]),
    "te_bert_attribute": (c_int, [_BCFG, _P, _P, c_int, c_int, _P, c_int, c_uint, _P, _P, c_ll, _P]),
    "te_bert_explain": (c_int, [_BCFG, _P, _P, _P, _P, c_int, c_int, _P, c_int, c_uint, _P, _P, _P, c_ll, _P]),
    "te_bert_tensor": (c_int, [_BCFG, c_int, c_int, _P, c_char_p, c_int, ctypes.POINTER(_P), ctypes.POINTER(c_ll),
                               ctypes.POINTER(c_ll)]),
    "te_linear_relprop": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_uint, _P]),
    "te_linear_relprop_ex": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_uint, _P]),
    "te_add_relprop": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_ll, _P]),
    "te_clone_relprop": (c_int, [_P, _P, _P, _P, _P, c_ll, _P]),
    "te_matmul_av_relprop": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "te_matmul_qk_relprop": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "te_index_select_relprop": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P]),
    "te_patch_embed_relprop_workspace_bytes": (c_ll, [c_int, c_int, c_int, c_int, c_int]),
    "te_patch_embed_relprop": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_ll, _P]),
    "te_relevance_heatmap": (c_int, [_P, c_int, c_int, c_int, _P, _P]),
    "te_head_reduce": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "te_head_region_mean": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "te_rollout_workspace_bytes": (c_ll, [c_int, c_int, c_int]),
    "te_attribution_rollout": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_uint, _P, _P, _P,
                                       c_ll, _P]),
    "te_compute_rollout_attention": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_ll, _P]),
    "te_linear_forward": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "te_linear_forward_ex": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_uint, _P]),
    "te_linear_backward_ex": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_uint, _P]),
    "te_f16_block_split": (c_int, [_P, c_int, c_int, _P, _P, _P, _P]),
    "te_attention_nn": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_float, c_int, c_uint,
                                _P]),
    "te_attention_nk": (c_int, [_P, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_float, c_int,
                                c_uint, _P]),
}

# epilogues of te_attention_nn / te_attention_nk
ATTN_STORE, ATTN_MUL, ATTN_SD, ATTN_SOFTMAX = 0, 1, 2, 3

_lib = None


def load():
    """Load the library, (re)building it first when its source stamp does not match (nvcc available); a stale or
    missing library without nvcc raises.  Raises on any failure — there is no CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    if _build.have_nvcc():
        _build.build()                   # no-op when the source/header stamp matches the built library
    elif not os.path.exists(LIB_PATH):
        raise OSError("%s is missing and nvcc is not available to build it (no CPU fallback)" % LIB_PATH)
    elif not _build.stamp_matches():
        raise OSError("%s is stale: csrc/ or include/te_b200.h changed since it was built and nvcc is not available"
                      % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class TeError(RuntimeError):
    pass


def check(status, what=""):
    if status < 0:
        msg = load().te_last_error()
        raise TeError("%s failed (%d): %s" % (what or "te_b200 call", status, msg.decode() if msg else ""))
    return status


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())
