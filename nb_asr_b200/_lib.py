"""ctypes binding of libnbasr.so (include/nbasr.h). Fails loudly when the library is missing."""
import ctypes as C
import os

from . import _build

F32, BF16, F16 = 0, 1, 2
PAD_L, PAD_R = 8, 4
MAX_ADD = 3

_vp, _i32, _i64, _f32, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint64


class Epilogue(C.Structure):
    _fields_ = [('bias', _vp), ('relu20', _i32), ('drop_p', _f32), ('drop_seed', _u64), ('drop_step', _vp),
                ('n_add', _i32), ('add', _vp * MAX_ADD), ('add_dtype', _i32), ('out', _vp), ('out_dtype', _i32),
                ('ld_out', _i64), ('mask_out', _vp), ('out2', _vp), ('out2_dtype', _i32), ('mask2', _vp),
                ('scale2', _f32), ('mask_rows', _i64), ('mask_w', _i32), ('mask2_w', _i32), ('accumulate', _i32),
                ('acc_scale', _f32), ('bias_scale', _f32), ('relu_hi', _f32)]


class Gemm(C.Structure):
    _fields_ = [('dtype', _i32), ('a', _vp), ('a_bs', _i64), ('a_rs', _i64), ('nb', _i32), ('nr', _i32),
                ('K', _i32), ('N', _i32), ('w', _vp), ('ldw', _i64), ('o_r0', _i64), ('o_bs', _i64),
                ('o_rs', _i64), ('epi', Epilogue)]


class Wgrad(C.Structure):
    _fields_ = [('dtype', _i32), ('dy', _vp), ('dy_bs', _i64), ('dy_rs', _i64), ('x', _vp), ('x_bs', _i64),
                ('x_rs', _i64), ('nb', _i32), ('nr', _i32), ('M', _i32), ('N', _i32), ('dw', _vp), ('ldw', _i64), ('dbias', _vp)]


class PackJob(C.Structure):
    _fields_ = [('kind', _i32), ('out_dtype', _i32), ('src', _vp), ('dst', _vp), ('n_out', _i64), ('a', _i32 * 8), ('s', _i64 * 3)]


class GConv(C.Structure):
    _fields_ = [('dtype', _i32), ('x', _vp), ('B', _i32), ('T', _i32), ('Tp', _i32), ('C', _i32), ('cpg', _i32),
                ('ktaps', _i32), ('off0', _i32), ('dstep', _i32), ('w', _vp), ('w_packed', _i32), ('epi', Epilogue)]


class GateLayer(C.Structure):
    _fields_ = [('mask', _vp), ('mask_rows', _i64), ('w', _i32), ('C', _i32), ('Tp', _i32), ('T', _i32), ('s', _i32),
                ('reserved', _i32)]


_SIGS = {
    'nbasr_gemm_tn': [C.POINTER(Gemm), _vp],
    'nbasr_gemm_wgrad': [C.POINTER(Wgrad), _vp],
    'nbasr_gconv_fwd': [C.POINTER(GConv), _vp],
    'nbasr_pack_gconv_dgrad': [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp],
    'nbasr_pack_gconv_mma': [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp],
    'nbasr_gconv_mma_pack_elems': [C.c_int, C.c_int, C.c_int],
    'nbasr_gconv_wgrad': [C.c_int, _vp, _vp] + [C.c_int] * 8 + [_vp, _vp, _vp],
    'nbasr_gconv_wgrad_x': [C.c_int, _vp, _vp, C.c_int, _f32] + [C.c_int] * 8 + [_vp, _vp, _vp],
    'nbasr_eltwise': [C.c_int, _vp, _i64, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Epilogue), _vp],
    'nbasr_colsum': [C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp],
    'nbasr_layernorm_fwd': [C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _f32, _vp, _vp, _f32, _vp, _vp],
    'nbasr_layernorm_bwd': [C.c_int, _vp, _vp, C.c_int, _f32, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp,
                            _f32, _i64, C.c_int, _vp, _vp, _vp],
    'nbasr_transpose_in': [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32, _vp],
    'nbasr_transpose_out': [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp],
    'nbasr_param_stats': [_vp, _vp, _vp, _vp, C.c_int, _i64, _vp, _vp, _vp],
    'nbasr_grad_snr': [_vp, _i64, C.c_int, _vp, _vp, C.c_int, _i64, _vp, _vp, _vp],
    'nbasr_row_gram': [_vp, C.c_int, _i64, _i64, _vp, _vp, _vp, _vp],
    'nbasr_gate_gram': [_vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp],
    'nbasr_gate_gram_work_elems': [C.c_int],
    'nbasr_pack_weight': [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _i64, _i64, _i64, _vp],
    'nbasr_convert': [_vp, _vp, C.c_int, _i64, _vp],
    'nbasr_lstm_fwd': [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp],
    'nbasr_lstm_bwd': [_vp, _i64, _i64, _i64, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp],
    'nbasr_head_fwd': [C.c_int, _vp, _i64, _i64, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp],
    'nbasr_head_bwd': [C.c_int, _vp, _i64, _i64, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _i64, _i64,
                       _vp, _vp, _vp],
    'nbasr_head_bwd_dh': [C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _i64, _i64, _vp, _vp],
    'nbasr_ctc': [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp],
    'nbasr_ctc_align': [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    'nbasr_ctc_align_work_bytes': [C.c_int] * 3,
    'nbasr_greedy_per': [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp,
                         _vp, _vp],
    'nbasr_beam_per': [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp,
                       _vp, _vp, _vp, _vp],
    'nbasr_edit_align': [_vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp],
    'nbasr_edit_align_work_bytes': [C.c_int] * 3,
    'nbasr_optim_step': [_vp, _vp, _vp, _vp, _i64, _vp, _vp, C.c_int, _i64, _f32, _f32, _f32, _f32, _f32, _vp, _vp],
    'nbasr_logmel': [_vp, _vp, C.c_int, _i64, _vp, _vp, _vp, _vp, _f32, _vp, C.c_int, _vp, _i64, _vp],
    'nbasr_logmel_work_floats': [C.c_int, _i64],
    'nbasr_pack_batch': [_vp, C.c_int, _vp, _i64, _vp],
    'nbasr_fill_u32': [_vp, C.c_uint32, _i64, _vp],
    'nbasr_version': [],
    'nbasr_sm_count': [],
}
EXPORTS = sorted(_SIGS) + ['nbasr_last_error']

_lib = None


class NbasrError(RuntimeError):
    pass


def lib_path():
    return _build.LIB


def load():
    """Load (building first if the sources are newer and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path) or (os.environ.get('NBASR_REBUILD') and _build.needs_build()):
        try:
            _build.build()
        except Exception as e:  # no nvcc / compile error: there is NO fallback path
            raise NbasrError(f'libnbasr.so is missing and could not be built ({e}); '
                             'run `python -c "import __graft_entry__ as g; g.build()"`') from e
    lib = C.CDLL(path)
    for name, args in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.nbasr_gconv_mma_pack_elems.restype = C.c_int64
    lib.nbasr_logmel_work_floats.restype = C.c_int64
    lib.nbasr_gate_gram_work_elems.restype = C.c_int64
    lib.nbasr_ctc_align_work_bytes.restype = C.c_int64
    lib.nbasr_edit_align_work_bytes.restype = C.c_int64
    lib.nbasr_last_error.restype = C.c_char_p
    lib.nbasr_last_error.argtypes = []
    _lib = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        raise NbasrError(f'{what}: {load().nbasr_last_error().decode()}')
