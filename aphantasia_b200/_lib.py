"""ctypes binding of libaphb200.so (the C ABI declared in include/aphb200.h).

The product path has NO fallback: if the CUDA library is missing or a call fails, this raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libaphb200.so')

_lib = None

c_f32p = C.c_void_p   # device pointers are passed as integers (tensor.data_ptr())
_SIGS = {
    'aph_version': (C.c_int, []),
    'aph_last_error': (C.c_char_p, []),
    'aph_launch_count': (C.c_int64, []),
    'aph_fft_plan_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int]),
    'aph_fft_plan_destroy': (C.c_int, [C.c_void_p]),
    'aph_synth_fft_fwd': (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_int, C.c_float, C.c_void_p, C.c_int,
                                    c_f32p, C.c_void_p, c_f32p, C.c_void_p]),
    'aph_synth_fft_bwd': (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_void_p, c_f32p, C.c_float, C.c_void_p, C.c_int,
                                    c_f32p, C.c_void_p]),
    'aph_dwt_plan_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    'aph_dwt_plan_destroy': (C.c_int, [C.c_void_p]),
    'aph_dwt_plan_levels': (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p]),
    'aph_synth_dwt_fwd': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int, c_f32p, C.c_void_p, c_f32p, C.c_void_p]),
    'aph_synth_dwt_bwd': (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'aph_pixel_fwd': (C.c_int, [c_f32p, C.c_int64, C.c_float, C.c_int, C.c_void_p, C.c_int, C.c_void_p, c_f32p, C.c_void_p]),
    'aph_pixel_bwd': (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_int64, C.c_float, C.c_int, C.c_void_p, C.c_int, c_f32p, C.c_void_p]),
    'aph_valid_rgb_fwd': (C.c_int, [c_f32p, C.c_int64, C.c_void_p, c_f32p, C.c_void_p]),
    'aph_valid_rgb_bwd': (C.c_int, [c_f32p, c_f32p, C.c_int64, C.c_void_p, c_f32p, C.c_void_p]),
    'aph_sample_fwd': (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_void_p]),
    'aph_sample_fwd_patches': (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_void_p, C.c_int,
                                         C.POINTER(C.c_int), C.c_void_p]),
    'aph_sample_bwd': (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_void_p]),
    'aph_sample_bwd_scaled': (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int, C.c_float, c_f32p, C.c_void_p]),
    'aph_rng_crop_tables': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]),
    'aph_vit_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p]),
    'aph_vit_destroy': (C.c_int, [C.c_void_p]),
    'aph_vit_load_tensor': (C.c_int, [C.c_void_p, C.c_char_p, c_f32p, C.c_int64, C.c_void_p]),
    'aph_vit_finalize': (C.c_int, [C.c_void_p]),
    'aph_vit_fwd': (C.c_int, [C.c_void_p, c_f32p, C.c_int, c_f32p, C.c_int, C.c_void_p]),
    'aph_vit_patch_operand': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'aph_vit_fwd_prepatched': (C.c_int, [C.c_void_p, C.c_int, c_f32p, C.c_int, C.c_void_p]),
    'aph_vit_bwd': (C.c_int, [C.c_void_p, c_f32p, C.c_int, c_f32p, C.c_void_p]),
    'aph_vit_bytes': (C.c_int64, [C.c_void_p]),
    'aph_text_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p]),
    'aph_text_destroy': (C.c_int, [C.c_void_p]),
    'aph_text_load_tensor': (C.c_int, [C.c_void_p, C.c_char_p, c_f32p, C.c_int64, C.c_void_p]),
    'aph_text_finalize': (C.c_int, [C.c_void_p]),
    'aph_text_fwd': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, c_f32p, C.c_void_p]),
    'aph_text_bytes': (C.c_int64, [C.c_void_p]),
    'aph_gemm_bf16_tn': (C.c_int, [C.c_void_p, C.c_void_p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    'aph_gemm_epi_test': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, C.c_void_p, C.c_int, c_f32p, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_int, C.c_void_p]),
    'aph_gemm_variant_launches': (C.c_int64, [C.c_int, C.c_int]),
    'aph_prof_gemm': (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    'aph_sim_fwd': (C.c_int, [c_f32p, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    'aph_derivat_fwd': (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p, c_f32p, C.c_void_p]),
    'aph_derivat_bwd': (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, C.c_void_p]),
    'aph_head_fwd': (C.c_int, [c_f32p, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    'aph_head_bwd': (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, c_f32p, C.c_void_p]),
    'aph_synth_fft_bwd_adam': (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_void_p, c_f32p, C.c_float, C.c_void_p, C.c_int,
                                         c_f32p, c_f32p, c_f32p, c_f32p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    'aph_allreduce_sym': (C.c_int, [C.c_uint64, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    'aph_adam_step': (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p]),
}
EXPORTS = tuple(_SIGS)


class VitConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('patch', 'width', 'layers', 'heads', 'out_dim', 'res', 'max_batch', 'reserved')]


class TextConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('width', 'layers', 'heads', 'ctx', 'vocab', 'out_dim', 'max_batch')]


def lib():
    """Loads libaphb200.so once. Raises (never falls back) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError('aphantasia_b200: %s not built. Run `python -c "import __graft_entry__ as g; g.build()"` '
                               '(or `make -C aphantasia_b200/csrc`). There is no CPU fallback.' % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(l, name)
            f.restype, f.argtypes = res, args
        _lib = l
    return _lib


def check(rc, what):
    if rc != 0:
        raise RuntimeError('%s failed (rc=%d): %s' % (what, rc, lib().aph_last_error().decode('utf-8', 'replace')))


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t, name):
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise RuntimeError('aphantasia_b200: %s must be a CUDA tensor; this implementation has no CPU path' % name)
