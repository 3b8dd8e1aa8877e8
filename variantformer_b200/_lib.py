"""ctypes binding of libvf_b200.so (include/vf_b200.h).

The CUDA library is THE implementation: there is no CPU or PyTorch fallback.  If the
shared object is missing (not built) or the device is not a B200-class GPU the import of
any compute entry point raises immediately.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# VF_LIB: a differently compiled build of the SAME library (A/B timing of kernel variants, tools/build_variant.py)
LIB_PATH = os.path.abspath(os.environ["VF_LIB"]) if os.environ.get("VF_LIB") else os.path.join(_HERE, "csrc", "libvf_b200.so")

EPI_BIAS_BF16, EPI_BIAS_GEGLU_BF16, EPI_BIAS_RESID_F32, EPI_BIAS_F32, EPI_BIAS_GELU_BF16 = range(5)

_vp, _i32, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t

# name -> argtypes; every symbol include/vf_b200.h declares (tests assert this list == the header)
SIGNATURES = {
    "vf_last_error": ([], C.c_char_p),
    "vf_abi_version": ([], _i32),
    "vf_launch_count": ([], C.c_ulonglong),
    "vf_attention_build_slots": ([_vp, _vp, _i32, _i32, _vp, _i32], _i32),
    "vf_seq2reg_workspace_bytes": ([_vp, _i64], _sz),
    "vf_seq2reg_forward": ([_vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _i32, _vp, _sz, _vp, _vp], _i32),
    "vf_seq2gene_workspace_bytes": ([_vp, _vp], _sz),
    "vf_seq2gene_forward": ([_vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp], _i32),
    "vf_seq2gene_forward_attn": ([_vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp], _i32),
    "vf_seq2gene_cre_rows": ([_vp, _vp, _vp, _sz, _vp, _i32, _vp, _vp], _i32),
    "vf_device_check": ([_vp], _i32),
    "vf_gemm_bf16": ([_vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp], _i32),
    "vf_gemm_bf16_ln": ([_vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _i32,
                         _vp, _i32, _vp, _i32, C.c_float, _vp, _vp], _i32),
    "vf_rowstats": ([_vp, _i32, _i32, _i32, _vp, _vp, _i32, _vp], _i32),
    "vf_attention_mc_varlen": ([_vp, _i32, _vp, _i32, _vp, _i32, _vp, _i32, _i64, _i64, _vp, _i32, _i32, _i32, _vp,
                                _vp], _i32),
    "vf_cross_attention_probs": ([_vp, _i32, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _i32, _vp, _vp, _i32, _vp], _i32),
    "vf_label_attention": ([_vp, _i32, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _i32, _vp], _i32),
    "vf_layernorm": ([_vp, _i32, _vp, _vp, _i32, _i32, C.c_float, _vp, _i32, _i32, _vp], _i32),
    "vf_window_lengths": ([_vp, _i32, _i32, _vp, _vp], _i32),
    "vf_compact_tokens": ([_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp], _i32),
    "vf_embed_tokens": ([_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp], _i32),
    "vf_masked_meanpool": ([_vp, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _vp], _i32),
    "vf_center_rows": ([_vp, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp], _i32),
    "vf_uncenter_rows": ([_vp, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _i32, _vp], _i32),
    "vf_gather_rows": ([_vp, _i32, _vp, _i32, _vp, _i32, _i32, _vp, _vp, _i32, _vp], _i32),
    "vf_head_out": ([_vp, _i32, _vp, _vp, _i32, _i32, _i32, _vp, _vp], _i32),
    "vf_cast_f32_to_bf16": ([_vp, _vp, _sz, _vp], _i32),
    "vf_forest_predict": ([_vp, _i32, _i32, _i32] + [_vp] * 9 + [_i32, _vp, _vp], _i32),
    "vf_encode_windows": ([_vp] * 13 + [_i32, _i32, _vp, _i64, _vp, _vp, _vp], _i32),
    "vf_encode_windows_edit": ([_vp] * 18 + [_i32, _i32, _vp, _i64, _vp, _vp, _vp, _vp], _i32),
    "vf_encode_windows_edits": ([_vp] * 20 + [_i32, _i32, _vp, _i64, _vp, _vp, _vp, _vp], _i32),
    "vf_encode_windows_overrides": ([_vp] * 16 + [_i32, _i32, _vp, _i64, _vp, _vp, _vp], _i32),
    "vf_window_genotype_keys": ([_vp] * 11 + [_i32, _vp, _vp, _vp, _vp, _vp], _i32),
    "vf_window_genotype_equal": ([_vp] * 11 + [_i32, _vp, _vp, _vp], _i32),
    "vf_window_genotype_keys_edits": ([_vp] * 18 + [_i32, _vp, _vp, _vp, _vp, _vp, _vp], _i32),
    "vf_window_genotype_equal_edits": ([_vp] * 18 + [_i32, _vp, _vp, _vp], _i32),
    "vf_mutate_windows": ([_vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp], _i32),
    "vf_splice_windows": ([_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp], _i32),
    "vf_bpe_tokenize": ([_vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _i64, _vp, _i32, _i32, _vp, _vp, _i64,
                         _i32, _vp], _i32),
}

_lib = None


class VFError(RuntimeError):
    pass


def load():
    """Load the shared library (no device access)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VFError(
            f"{LIB_PATH} not found: build it with `python -m variantformer_b200.csrc.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (args, res) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.argtypes = args
        fn.restype = res
    if lib.vf_abi_version() != 2:
        raise VFError("libvf_b200.so ABI version mismatch")
    _lib = lib
    return lib


_device_ok = False


def lib():
    """Library handle for compute calls: also checks that the current device is sm_100."""
    global _device_ok
    l = load()
    if not _device_ok:
        import torch
        if not torch.cuda.is_available():
            raise VFError("variantformer_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        sms = C.c_int(0)
        check(l.vf_device_check(C.byref(sms)))
        _device_ok = True
    return l


def check(rc: int):
    if rc != 0:
        raise VFError(load().vf_last_error().decode() or f"libvf_b200 error {rc}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream
