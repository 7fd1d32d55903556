"""ctypes binding of libb200imagen.so (include/b200_imagen.h).

The product path has NO fallback: if the shared library is missing or a kernel call
fails, a RuntimeError is raised (never a silent torch/CPU path).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('B200_IMAGEN_LIB') or os.path.join(_HERE, 'csrc', 'libb200imagen.so')   # the override is for A/B runs of two builds

MAX_SRC, MAX_SEG = 4, 24
ACT_NONE, ACT_SILU, ACT_GELU = 0, 1, 2
OUT_BF16, OUT_PIXEL_SHUFFLE, OUT_F32_NCHW, OUT_F32 = 0, 1, 2, 3
IMPL_TCGEN05, IMPL_SIMT_CHECKER = 0, 1
NORM_NONE, NORM_LN, NORM_RMS_FILM_SILU = 0, 1, 2
ABI_VERSION = 2


class Src(C.Structure):
    _fields_ = [('ptr', C.c_void_p), ('C', C.c_int32), ('ld', C.c_int32)]


class Seg(C.Structure):
    _fields_ = [('src', C.c_int32), ('dh', C.c_int32), ('dw', C.c_int32)]


class Epilogue(C.Structure):
    _fields_ = [
        ('bias', C.c_void_p), ('act', C.c_int32), ('out_scale', C.c_float),
        ('residual', C.c_void_p), ('ldr', C.c_int32), ('out_mode', C.c_int32),
        ('out', C.c_void_p), ('ldc', C.c_int32),
        ('out2', C.c_void_p), ('ldc2', C.c_int32), ('split_col', C.c_int32),
        ('rows_per_group', C.c_int32), ('group_stride', C.c_int32), ('row_offset', C.c_int32),
        ('l2_cols', C.c_int32), ('l2_scale', C.c_void_p), ('ps_C', C.c_int32), ('dup_rows', C.c_int32),
        # ABI v2: per-row norms fused into the epilogue (include/b200_imagen.h)
        ('norm1', C.c_int32), ('norm1_g', C.c_void_p), ('norm2', C.c_int32), ('norm2_g', C.c_void_p), ('film', C.c_void_p),
        ('film_ld', C.c_int32), ('rows_per_sample', C.c_int32), ('out_norm', C.c_void_p), ('ld_norm', C.c_int32),
    ]


class TimeRowJob(C.Structure):
    _fields_ = [('table', C.c_void_p), ('dst', C.c_void_p), ('sample_stride', C.c_int64),
                ('rows', C.c_int32), ('width', C.c_int32)]


class DdpmCoef(C.Structure):
    _fields_ = [(n, C.c_float) for n in ('sigma', 'alpha', 'inv_alpha_clamped', 'alpha_next', 'c', 'noise_std', 'pad0', 'pad1')]


class EdmCoef(C.Structure):
    _fields_ = [(n, C.c_float) for n in ('s_noise', 'noise_coef', 'sigma_hat', 'sigma_next', 'dt', 'half_dt',
                                          'c_in_hat', 'c_skip_hat', 'c_out_hat', 'c_in_next', 'c_skip_next', 'c_out_next',
                                          'has_second', 'pad0', 'pad1', 'pad2')]


class RowChain(C.Structure):
    _fields_ = [('x', C.c_void_p), ('ldx', C.c_int32), ('gate', C.c_void_p), ('rows_per_sample', C.c_int32),
                ('norm1', C.c_int32), ('norm1_g', C.c_void_p), ('residual', C.c_void_p), ('ldr', C.c_int32),
                ('out', C.c_void_p), ('ldo', C.c_int32), ('norm2', C.c_int32), ('norm2_g', C.c_void_p),
                ('film', C.c_void_p), ('film_ld', C.c_int32), ('out_norm', C.c_void_p), ('ld_norm', C.c_int32),
                ('M', C.c_int64), ('C', C.c_int32)]


_P, _I, _L, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float

# name -> argtypes: mirrors include/b200_imagen.h one to one (tests/test_abi.py checks every symbol)
SIGNATURES = {
    'b200_abi_version': [],
    'b200_check_device': [_I],
    'b200_sizeof': [_I],
    'b200_conv_gemm_npad': [_I],
    'b200_conv_gemm_splitk': [_I, _I, _I, _I, _I],
    'b200_conv_gemm': [C.POINTER(Src), _I, C.POINTER(Seg), _I, _I, _I, _I, _P, _I, C.POINTER(Epilogue), _I, _P, _P],
    'b200_attention': [_P, _P, _L, _L, _I, _I, _P, _P, _L, _L, _I, _I, _I, _I, _F, _P],
    'b200_linear_xattn_context': [_P, _P, _L, _I, _I, _I, _I, _I, _P, _P],
    'b200_linear_cross_attention': [_P, _P, _L, _I, _I, _P, _I, _I, _I, _P],
    'b200_rmsnorm_film_silu': [C.POINTER(Src), _I, _F, _P, _P, _I, _I, _P, _I, _L, _P],
    'b200_layernorm': [_P, _I, _P, _P, _F, _P, _I, _P, _I, _L, _I, _P],
    'b200_gca_gate': [_P, _I, _I, _I, _I, _P, _F, _P, _P, _I, _P, _P, _P, _I, _P, _P],
    'b200_row_chain': [C.POINTER(RowChain), _P],
    'b200_gca_nchunk': [_I],
    'b200_gca_chunks': [_I, _I],
    'b200_gate_residual': [_P, _I, _P, _P, _I, _P, _I, _L, _I, _I, _P],
    'b200_im2col_init': [_P, _I, _P, _I, _I, _I, _I, _I, _P, _I, _P],
    'b200_im2col_init3': [_P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P, _I, _P],
    'b200_im2col_init4': [_P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P, _I, _P],
    'b200_pixel_unshuffle': [_P, _I, _I, _I, _I, _I, _P, _P],
    'b200_nchw_to_rows': [_P, _I, _I, _I, _I, _P, _I, _P],
    'b200_make_time_cond': [_P, _P, _P, _I, _I, _P, _P],
    'b200_update_time_rows': [_P, _I, _P, _I, _I, _P],
    'b200_linear_f32': [_P, _I, _P, _P, _I, _I, _P, _I, _P, _I, _L, _I, _I, _P],
    'b200_layernorm_f32': [_P, _I, _P, _P, _F, _P, _I, _L, _I, _P],
    'b200_sinu_pos_emb': [_P, _P, _I, _I, _P, _P],
    'b200_attn_f32': [_P, _I, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    'b200_headnorm_store': [_P, _I, _I, _I, _I, _P, _P, _I, _L, _L, _L, _L, _P],
    'b200_ddpm_step': [_P, _P, _P, _P, _P, _I, _I, _L, _F, _I, _I, _I, _I, _F, _P],
    'b200_edm_phase': [_I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _F, _I, _I, _I, _F, _P],
    'b200_ddpm_step_sc': [_P, _P, _P, _P, _P, _I, _I, _L, _F, _I, _I, _I, _I, _F, _P, _P],
    'b200_edm_phase_sc': [_I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _F, _I, _I, _I, _F, _P, _P],
    'b200_inpaint_mix': [_P, _P, _P, _P, _F, _F, _I, _I, _L, _P],
    'b200_renoise': [_P, _P, _F, _F, _F, _L, _P],
    'b200_finalize_images': [_P, _P, _L, _I, _P],
}

_lib = None


class B200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                        f'(or imagen_pytorch_b200/csrc/build.sh). There is no CPU / torch fallback.')
    lib = C.CDLL(LIB_PATH)
    lib.b200_last_error.restype = C.c_char_p
    lib.b200_last_error.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    if lib.b200_abi_version() != ABI_VERSION:
        raise B200Error('libb200imagen.so ABI version mismatch')
    _lib = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        raise B200Error(f'{what} failed ({rc}): {load().b200_last_error().decode()}')


def call(name, *args):
    lib = load()
    check(getattr(lib, name)(*args), name)


def require_device(index=0):
    lib = load()
    check(lib.b200_check_device(index), 'b200_check_device')


def npad(n):
    return load().b200_conv_gemm_npad(int(n))
