"""ctypes binding of ``libcgpcm_b200.so`` (the C-ABI declared in ``include/cgpcm_b200.h``).

There is no CPU fallback: if the shared library is missing or does not load, importing the binding
raises, and every entry point needs a CUDA device.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libcgpcm_b200.so')
SRC = os.path.join(_HERE, 'csrc', 'cgpcm.cu')

NVCC_FLAGS = ['-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo',
              '--extended-lambda', '-shared', '-Xcompiler', '-fPIC']

GRAD_S2, GRAD_S2F, GRAD_ALPHA, GRAD_GAMMA, GRAD_OMEGA, GRAD_MU_U, GRAD_VAR_U = [1 << i for i in range(7)]
GRAD_ALL = 0x7f
MODE_FROZEN, MODE_FULL = 0, 1

EXPORTS = ['cgpcm_create', 'cgpcm_destroy', 'cgpcm_last_error', 'cgpcm_device_count', 'cgpcm_comm_unique_id', 'cgpcm_comm_init',
           'cgpcm_set_data', 'cgpcm_set_option', 'cgpcm_psi', 'cgpcm_precompute', 'cgpcm_frozen_mats', 'cgpcm_elbo_grad', 'cgpcm_elbo_smf', 'cgpcm_elbo_smf_batch', 'cgpcm_predict_f', 'cgpcm_predict_f_batch', 'cgpcm_predict_f_cov', 'cgpcm_predict_logpdf', 'cgpcm_kernel_samples', 'cgpcm_filter_samples', 'cgpcm_akm_sample', 'cgpcm_fpi', 'cgpcm_fpi_qz', 'cgpcm_elbo_qz',
           'cgpcm_last_timing', 'cgpcm_bvn_cdf', 'cgpcm_dgemm', 'cgpcm_dgemm_tri', 'cgpcm_dgemm_sym', 'cgpcm_cholinv', 'cgpcm_math_test', 'cgpcm_math_test_fast', 'cgpcm_math_test_tab',
           'cgpcm_smf_c1_test', 'cgpcm_smf_algebra_test', 'cgpcm_smf_posterior_test', 'cgpcm_predict_quad_test',
           'cgpcm_predict_pair_test', 'cgpcm_ahx_gen_test', 'cgpcm_ahx_dot_test', 'cgpcm_axx_sum_test',
           'cgpcm_window_chol_test', 'cgpcm_sym_accum_test', 'cgpcm_potrf_test', 'cgpcm_trtri_test']


def _sources():
    d = os.path.join(_HERE, 'csrc')
    out = [os.path.join(d, f) for f in sorted(os.listdir(d))]
    out.append(os.path.join(os.path.dirname(_HERE), 'include', 'cgpcm_b200.h'))
    return out


def build(force=False, verbose=False):
    """Compile the library for sm_100a with nvcc (cross-compiles without a GPU)."""
    if not force and os.path.exists(LIB_PATH):
        newest = max(os.path.getmtime(p) for p in _sources())
        if os.path.getmtime(LIB_PATH) >= newest:
            return LIB_PATH
    os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
    nvcc = os.environ.get('NVCC', 'nvcc')
    if not any(os.access(os.path.join(p, nvcc), os.X_OK) for p in os.environ.get('PATH', '').split(os.pathsep)):
        if os.path.exists('/usr/local/cuda/bin/nvcc'):
            nvcc = '/usr/local/cuda/bin/nvcc'
    cmd = [nvcc] + NVCC_FLAGS + ['-o', LIB_PATH, SRC, '-ldl']
    if verbose:
        print(' '.join(cmd))
    subprocess.check_call(cmd)
    return LIB_PATH


_lib = None


def lib():
    """The loaded shared library (raises if it is absent: the product has no other compute path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError('cgpcm_b200: %s is missing; build it with `python -c "import __graft_entry__ as g; '
                          'g.build()"` (there is no CPU fallback)' % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, dp, i32, i64, u32, dbl = (ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                  ctypes.c_uint32, ctypes.c_double)
    L.cgpcm_create.argtypes = [ctypes.POINTER(vp), i32, i32, i32, i32, i32, vp]
    L.cgpcm_destroy.argtypes = [vp]
    L.cgpcm_last_error.argtypes = [vp]
    L.cgpcm_last_error.restype = ctypes.c_char_p
    L.cgpcm_device_count.argtypes = [ctypes.POINTER(i32)]
    L.cgpcm_comm_unique_id.argtypes = [vp]
    L.cgpcm_comm_init.argtypes = [vp, vp, i32, i32]
    L.cgpcm_set_data.argtypes = [vp, dp, dp, i64, dp, dp]
    L.cgpcm_set_option.argtypes = [vp, ctypes.c_char_p, dbl]
    L.cgpcm_psi.argtypes = [vp, dp, dp, dp, dp, dp, dp, dp]
    L.cgpcm_precompute.argtypes = [vp, dp, dbl]
    L.cgpcm_frozen_mats.argtypes = [vp, dp, dp, dp, dp]
    L.cgpcm_elbo_grad.argtypes = [vp, dp, ctypes.c_int32, u32, dbl, dp, dp, dp]
    L.cgpcm_elbo_smf.argtypes = [vp, dp, ctypes.c_int32, dbl, dp, dp, dp, dp]
    L.cgpcm_elbo_smf_batch.argtypes = [vp, dp, dbl, dp, ctypes.c_int32, dp, dp, dp]
    L.cgpcm_predict_f.argtypes = [vp, dp, dbl, dp, i64, dp, ctypes.c_int32, ctypes.c_int32, dp, dp]
    L.cgpcm_predict_f_batch.argtypes = [vp, dp, dbl, dp, i64, dp, ctypes.c_int32, ctypes.c_int32, dp, dp, dp, dp]
    L.cgpcm_predict_f_cov.argtypes = [vp, dp, dbl, dp, i64, dp, ctypes.c_int32, ctypes.c_int32, dp, dp, dp, dp, dp]
    L.cgpcm_predict_logpdf.argtypes = [vp, dp, dbl, dp, dp, i64, dp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                       dp, dp, dp]
    L.cgpcm_kernel_samples.argtypes = [vp, dp, dbl, dp, i64, dp, ctypes.c_int32, dp]
    L.cgpcm_filter_samples.argtypes = [vp, dp, dbl, dp, i64, dp, ctypes.c_int32, dp, dp]
    L.cgpcm_akm_sample.argtypes = [vp, dp, dbl, dp, i64, dp, dp, dp, dp]
    L.cgpcm_fpi.argtypes = [vp, dp, ctypes.c_int32, ctypes.c_int32, dbl, dp, dp, dp, dp]
    L.cgpcm_fpi_qz.argtypes = [vp, dp, dp, dp, ctypes.c_int32, ctypes.c_int32, dbl, dp, dp, dp, dp]
    L.cgpcm_elbo_qz.argtypes = [vp, dp, dp, dp, dbl, dp, dp]
    L.cgpcm_last_timing.argtypes = [vp, dp]
    L.cgpcm_bvn_cdf.argtypes = [dp, dp, dp, dp, ctypes.c_size_t, vp]
    L.cgpcm_dgemm.argtypes = [i32, i32, i32, i32, i32, i32, dbl, dp, i64, dp, i64, dbl, dp, i64, i32, i64, i32, vp]
    L.cgpcm_dgemm_sym.argtypes = [i32, i32, i32, dp, i64, dp, i64, dp, i64, dp, vp]
    L.cgpcm_dgemm_tri.argtypes = [i32, i32, dp, i64, dp, i64, dp, i64, vp]
    L.cgpcm_cholinv.argtypes = [dp, dp, dp, i32, i64, ctypes.POINTER(i32)]
    L.cgpcm_math_test.argtypes = [dp, i64, dp, dp, ctypes.POINTER(i32)]
    L.cgpcm_math_test_fast.argtypes = [dp, i64, dp, dp]
    L.cgpcm_math_test_tab.argtypes = [dp, i64, dp, dp, dp]
    L.cgpcm_smf_c1_test.argtypes = [dp, i64, i32, i32, dp, i32, i64, dp, vp]
    L.cgpcm_smf_algebra_test.argtypes = [dp, dp, dp, dp, dp, dp, i32, i32, i32, i64, i32, dbl, dbl, dbl, i32, i32, dp,
                                         vp, vp]
    L.cgpcm_smf_posterior_test.argtypes = [dp, dp, dp, dp, dp, dp, dp, dp, i32, i32, i32, i32, i64, i32, dbl, dbl, dbl,
                                           dbl, dp, dp, dp, vp, vp]
    L.cgpcm_predict_quad_test.argtypes = [dp, i64, i32, dp, i64, dp, i64, dp, i32, i32, i32, i32, dp, dp, dp, vp]
    L.cgpcm_predict_pair_test.argtypes = [dp, i32, dp, i32, dp, i32, dp, i32, i32, dp, i64, i32, dp, vp]
    L.cgpcm_ahx_gen_test.argtypes = [dp, dp, i32, i32, dp, i32, i32, dp, i32, i32, i32, dp, i32, i32, dbl, i32, i64, dp,
                                     dp, vp]
    L.cgpcm_ahx_dot_test.argtypes = [dp, dp, i32, i32, dp, i32, i32, dp, i32, i32, i32, dp, i32, i32, dbl, i32, i64, dp,
                                     dp, dp, dp, vp]
    L.cgpcm_axx_sum_test.argtypes = [dp, i32, i32, dp, i32, dp, i32, i32, dbl, i32, i32, i64, dp, vp]
    L.cgpcm_window_chol_test.argtypes = [dp, i64, dbl, i32, dp, i32, dp, ctypes.POINTER(i32), vp]
    L.cgpcm_sym_accum_test.argtypes = [i32, dp, dp, dp, i32, i64, dp, vp]
    L.cgpcm_potrf_test.argtypes = [dp, i32, i64, i32, ctypes.POINTER(i32), vp]
    L.cgpcm_trtri_test.argtypes = [dp, dp, i32, i64, vp]
    for name in EXPORTS:
        if name != 'cgpcm_last_error':
            getattr(L, name).restype = ctypes.c_int
    _lib = L
    return L


def ptr(a):
    """Address of a contiguous float64 numpy array or torch tensor (host or CUDA), or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if a.dtype != np.float64 or not a.flags['C_CONTIGUOUS']:
            raise ValueError('expected a C-contiguous float64 array')
        return a.ctypes.data
    # torch tensor
    import torch
    if isinstance(a, torch.Tensor):
        if a.dtype != torch.float64 or not a.is_contiguous():
            raise ValueError('expected a contiguous float64 tensor')
        return a.data_ptr()
    raise TypeError('unsupported buffer type %r' % type(a))


class CgpcmError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, 'cgpcm_b200 error %d: %s' % (code, msg))
        self.code = code


_CODES = {-1: 'bad argument', -2: 'CUDA / NCCL error', -3: 'matrix not positive definite', -4: 'non-finite input'}


def check(rc, handle=None):
    if rc == 0:
        return
    msg = _CODES.get(rc, 'unknown error')
    if handle:
        detail = lib().cgpcm_last_error(handle)
        if detail:
            msg = '%s: %s' % (msg, detail.decode())
    if rc in (-1, -4):
        raise ValueError('cgpcm_b200 error %d: %s' % (rc, msg))
    raise CgpcmError(rc, msg)
