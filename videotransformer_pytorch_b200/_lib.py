"""ctypes binding of libvt_b200.so (include/vt_b200.h) + the tensor-level kernel API used by ops.py.

There is deliberately NO fallback: if the shared library is missing or a kernel rejects its arguments a
RuntimeError is raised.  `K` is the process-wide kernel table; tests may swap it for the CPU emulation in
tests/emu_kernels.py to exercise the host-side logic without a GPU (the product never does).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libvt_b200.so')

EPI = {'bf16': 0, 'f32': 1, 'gelu': 2, 'dgelu': 3}

c_i32, c_i64, c_f32, c_vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p


class GemmParams(C.Structure):
    _fields_ = [('a', c_vp), ('b', c_vp), ('lda', c_i64), ('ldb', c_i64),
                ('M', c_i32), ('N', c_i32), ('K', c_i32),
                ('a_mn_major', c_i32), ('b_mn_major', c_i32), ('epilogue', c_i32),
                ('bias', c_vp), ('out', c_vp), ('out2', c_vp), ('aux', c_vp),
                ('ldo', c_i64), ('ldo2', c_i64), ('ldaux', c_i64),
                ('out_row', c_vp), ('aux_row', c_vp), ('row_scale', c_vp),
                ('workspace', c_vp), ('workspace_bytes', c_i64),
                ('force_splits', c_i32), ('force_bn', c_i32), ('force_cluster', c_i32), ('debug', c_vp),
                ('map_period', c_i32), ('map_skip', c_i32), ('map_tcount', c_i32), ('force_tail', c_i32),
                ('map_stride_t', c_i64), ('map_stride_p', c_i64), ('map_stride_b', c_i64), ('map_base', c_i64),
                ('map_special_base', c_i64), ('map_special_stride', c_i64), ('bias2', c_vp), ('out_zeroed', c_i32)]


class LnFwdParams(C.Structure):
    _fields_ = [('x', c_vp), ('ldx', c_i64), ('in_row', c_vp), ('gamma', c_vp), ('beta', c_vp),
                ('y', c_vp), ('mean', c_vp), ('rstd', c_vp), ('rows', c_i32), ('D', c_i32),
                ('eps', c_f32), ('y_fp32', c_i32)]


class LnBwdParams(C.Structure):
    _fields_ = [('dy', c_vp), ('dy_fp32', c_i32), ('x', c_vp), ('ldx', c_i64), ('in_row', c_vp),
                ('mean', c_vp), ('rstd', c_vp), ('gamma', c_vp),
                ('dres', c_vp), ('dx', c_vp), ('lddx', c_i64), ('dx_aux', c_vp), ('out_row', c_vp),
                ('partials', c_vp), ('rows', c_i32), ('D', c_i32)]


class ReduceParams(C.Structure):
    _fields_ = [('inp', c_vp), ('out', c_vp), ('stride', c_i64), ('S', c_i32), ('n', c_i64),
                ('accumulate', c_i32), ('scale', c_f32)]


class ColsumParams(C.Structure):
    _fields_ = [('inp', c_vp), ('ld', c_i64), ('M', c_i32), ('N', c_i32), ('out', c_vp), ('workspace', c_vp), ('counters', c_vp)]


class CastParams(C.Structure):
    _fields_ = [('src', c_vp), ('dst', c_vp), ('n', c_i64)]


class GatherCastParams(C.Structure):
    _fields_ = [('src', c_vp), ('lds', c_i64), ('in_row', c_vp), ('row_scale', c_vp), ('dst', c_vp),
                ('rows', c_i32), ('D', c_i32)]


class GeluParams(C.Structure):
    _fields_ = [('z', c_vp), ('dh', c_vp), ('out', c_vp), ('n', c_i64)]


class ClsRowsParams(C.Structure):
    _fields_ = [('src', c_vp), ('src_stride', c_i64), ('extra', c_vp), ('extra_bs', c_i64), ('T', c_i32), ('scale', c_f32),
                ('dst', c_vp), ('dst_stride', c_i64), ('B', c_i32), ('D', c_i32)]


class GatherCastColsumParams(C.Structure):
    _fields_ = [('src', c_vp), ('lds', c_i64), ('in_row', c_vp), ('row_scale', c_vp), ('dst', c_vp),
                ('rows', c_i32), ('D', c_i32), ('colsum', c_vp), ('workspace', c_vp), ('workspace_rows', c_i32),
                ('unscaled_sums', c_i32)]


class GeluBwdColsumParams(C.Structure):
    _fields_ = [('z', c_vp), ('dh', c_vp), ('out', c_vp), ('M', c_i32), ('N', c_i32), ('colsum', c_vp),
                ('workspace', c_vp), ('workspace_rows', c_i32)]


class AttnFwdParams(C.Structure):
    _fields_ = [('qkv', c_vp), ('ctx', c_vp), ('lse', c_vp), ('probs', c_vp),
                ('Bp', c_i32), ('N', c_i32), ('H', c_i32), ('hd', c_i32), ('scale', c_f32), ('impl', c_i32)]


class AttnBwdParams(C.Structure):
    _fields_ = [('qkv', c_vp), ('ctx', c_vp), ('dctx', c_vp), ('lse', c_vp), ('dqkv', c_vp),
                ('Bp', c_i32), ('N', c_i32), ('H', c_i32), ('hd', c_i32), ('scale', c_f32), ('impl', c_i32)]


class Im2colParams(C.Structure):
    _fields_ = [('x', c_vp), ('cols', c_vp), ('B', c_i32), ('T', c_i32), ('C', c_i32), ('H', c_i32),
                ('W', c_i32), ('tube', c_i32), ('ph', c_i32), ('pw', c_i32)]


class Im2colU8Params(C.Structure):
    _fields_ = [('x', c_vp), ('scale', c_vp), ('shift', c_vp), ('cols', c_vp), ('B', c_i32), ('T', c_i32), ('C', c_i32),
                ('H', c_i32), ('W', c_i32), ('tube', c_i32), ('ph', c_i32), ('pw', c_i32)]


class HogParams(C.Structure):
    _fields_ = [('frames', c_vp), ('lut', c_vp), ('feat', c_vp), ('bins', c_vp),
                ('F', c_i32), ('H', c_i32), ('W', c_i32)]


class PoolFwdParams(C.Structure):
    _fields_ = [('inp', c_vp), ('in_bs', c_i64), ('in_rs', c_i64), ('w', c_vp), ('gamma', c_vp), ('beta', c_vp),
                ('pooled', c_vp), ('out', c_vp), ('mean', c_vp), ('rstd', c_vp),
                ('B', c_i32), ('H', c_i32), ('hd', c_i32), ('T', c_i32), ('Hin', c_i32), ('Win', c_i32),
                ('st', c_i32), ('sh', c_i32), ('sw', c_i32), ('To', c_i32), ('Ho', c_i32), ('Wo', c_i32), ('eps', c_f32)]


class PoolBwdParams(C.Structure):
    _fields_ = [('dout', c_vp), ('dout_fp32', c_i32), ('pooled', c_vp), ('mean', c_vp), ('rstd', c_vp), ('gamma', c_vp),
                ('inp', c_vp), ('in_bs', c_i64), ('in_rs', c_i64), ('w', c_vp),
                ('din', c_vp), ('din_bs', c_i64), ('din_rs', c_i64),
                ('dw', c_vp), ('dgamma', c_vp), ('dbeta', c_vp), ('scratch', c_vp), ('scratch_floats', c_i64),
                ('B', c_i32), ('H', c_i32), ('hd', c_i32), ('T', c_i32), ('Hin', c_i32), ('Win', c_i32),
                ('st', c_i32), ('sh', c_i32), ('sw', c_i32), ('To', c_i32), ('Ho', c_i32), ('Wo', c_i32)]


_XA_STRIDES = [(t + s, c_i64) for t in ('q', 'k', 'v', 'o') for s in ('_bs', '_hs', '_rs')]


class XattnFwdParams(C.Structure):
    _fields_ = [('q', c_vp), ('k', c_vp), ('v', c_vp), ('o', c_vp), ('lse', c_vp)] + _XA_STRIDES + \
               [('B', c_i32), ('H', c_i32), ('Nq', c_i32), ('Nk', c_i32), ('hd', c_i32), ('scale', c_f32), ('impl', c_i32)]


class XattnBwdParams(C.Structure):
    _fields_ = [('q', c_vp), ('k', c_vp), ('v', c_vp), ('o', c_vp), ('dout', c_vp), ('lse', c_vp),
                ('delta', c_vp), ('dq', c_vp), ('dk', c_vp), ('dv', c_vp)] + _XA_STRIDES + \
               [('dq_bs', c_i64), ('dq_hs', c_i64), ('dq_rs', c_i64),
                ('B', c_i32), ('H', c_i32), ('Nq', c_i32), ('Nk', c_i32), ('hd', c_i32), ('scale', c_f32), ('impl', c_i32)]


_MP_DIMS = [(n, c_i32) for n in ('B', 'D', 'T', 'H', 'W', 'kt', 'kh', 'kw', 'st', 'sh', 'sw', 'To', 'Ho', 'Wo')]


class MaxpoolFwdParams(C.Structure):
    _fields_ = [('x', c_vp), ('y', c_vp), ('idx', c_vp)] + _MP_DIMS


class MaxpoolBwdParams(C.Structure):
    _fields_ = [('dy', c_vp), ('idx', c_vp), ('dx', c_vp)] + _MP_DIMS


class Im2col3dParams(C.Structure):
    _fields_ = [('x', c_vp), ('cols', c_vp)] + [(n, c_i32) for n in (
        'B', 'T', 'C', 'H', 'W', 'kt', 'kh', 'kw', 'st', 'sh', 'sw', 'pt', 'ph', 'pw', 'To', 'Ho', 'Wo', 'Kpad')]


class MvitTokensFwdParams(C.Structure):
    _fields_ = [('t', c_vp), ('wmask', c_vp), ('mask_token', c_vp), ('cls_token', c_vp), ('pos_s', c_vp),
                ('pos_t', c_vp), ('pos_cls', c_vp), ('x', c_vp), ('B', c_i32), ('T', c_i32), ('HW', c_i32), ('C', c_i32)]


class MvitTokensBwdParams(C.Structure):
    _fields_ = [('dx', c_vp), ('wmask', c_vp), ('dt', c_vp), ('B', c_i32), ('T', c_i32), ('HW', c_i32), ('C', c_i32)]


_MSE_DIMS = [(n, c_i32) for n in ('B', 't', 'dt', 'h', 'w', 'dc')]


class MseFwdParams(C.Structure):
    _fields_ = [('pred', c_vp), ('target', c_vp), ('mask', c_vp), ('num', c_vp), ('partials', c_vp)] + _MSE_DIMS + \
               [('target64', c_vp), ('num64', c_vp)]


class MseBwdParams(C.Structure):
    _fields_ = [('pred', c_vp), ('target', c_vp), ('mask', c_vp), ('coef', c_vp), ('dpred', c_vp)] + _MSE_DIMS + \
               [('target64', c_vp)]


class OptParams(C.Structure):
    _fields_ = [('chunks', c_vp), ('n_chunks', c_i32), ('n_tensors', c_i32),
                ('pptr', c_vp), ('gptr', c_vp), ('s1ptr', c_vp), ('s2ptr', c_vp),
                ('norm2', c_vp), ('lr', c_vp), ('wd', c_vp),
                ('clip', c_f32), ('momentum', c_f32), ('beta1', c_f32), ('beta2', c_f32), ('eps', c_f32), ('bc1', c_f32),
                ('bc2', c_f32), ('nesterov', c_i32), ('first_step', c_i32)]


class LinearSmallParams(C.Structure):
    _fields_ = [('x', c_vp), ('w', c_vp), ('b', c_vp), ('y', c_vp), ('M', c_i32), ('N', c_i32), ('K', c_i32)]


class LinearSmallBwdParams(C.Structure):
    _fields_ = [('dy', c_vp), ('x', c_vp), ('w', c_vp), ('dw', c_vp), ('db', c_vp), ('dx', c_vp),
                ('M', c_i32), ('N', c_i32), ('K', c_i32)]


class SoftmaxCeParams(C.Structure):
    _fields_ = [('logits', c_vp), ('labels', c_vp), ('soft_targets', c_vp), ('loss', c_vp), ('row_loss', c_vp),
                ('dlogits', c_vp), ('M', c_i32), ('N', c_i32)]


class ScaleParams(C.Structure):
    _fields_ = [('inp', c_vp), ('scalar', c_vp), ('out', c_vp), ('n', c_i64)]


class AttnProbsParams(C.Structure):
    _fields_ = [('qkv', c_vp), ('probs', c_vp), ('Bp', c_i32), ('N', c_i32), ('H', c_i32), ('hd', c_i32), ('scale', c_f32)]


class Im2colU8MixParams(C.Structure):
    _fields_ = [('x', c_vp), ('scale', c_vp), ('shift', c_vp), ('plan', c_vp), ('cols', c_vp), ('B', c_i32), ('T', c_i32),
                ('C', c_i32), ('H', c_i32), ('W', c_i32), ('tube', c_i32), ('ph', c_i32), ('pw', c_i32)]


class PosInterpParams(C.Structure):
    _fields_ = [('inp', c_vp), ('out', c_vp), ('D', c_i32), ('src_side', c_i32), ('out_rows', c_i32), ('out_cols', c_i32),
                ('scale_r', c_f32), ('scale_c', c_f32)]


EXPORTS = ['vt_version', 'vt_last_error', 'vt_sm_count', 'vt_set_reserved_sms', 'vt_launch_count', 'vt_gemm', 'vt_layernorm_fwd', 'vt_ln_bwd_blocks',
           'vt_layernorm_bwd', 'vt_reduce_rows', 'vt_colsum_chunks', 'vt_colsum_bf16', 'vt_cast_f32_bf16',
           'vt_cls_rows', 'vt_gather_cast_colsum_blocks', 'vt_gather_cast_colsum_bf16', 'vt_gelu_bwd_colsum_blocks', 'vt_gelu_bwd_colsum_bf16',
           'vt_gather_cast_bf16', 'vt_gelu_fwd_bf16', 'vt_gelu_bwd_bf16', 'vt_attn_fwd', 'vt_attn_bwd', 'vt_debug_buffer', 'vt_im2col_bf16', 'vt_im2col_u8_bf16', 'vt_col2im_f32', 'vt_hog',
           'vt_pool_fwd', 'vt_pool_bwd_scratch', 'vt_pool_bwd', 'vt_xattn_fwd', 'vt_xattn_bwd', 'vt_maxpool_fwd',
           'vt_maxpool_bwd', 'vt_im2col3d_bf16', 'vt_mvit_tokens_fwd', 'vt_mvit_tokens_bwd', 'vt_mse_blocks',
           'vt_mse_fwd', 'vt_mse_bwd', 'vt_opt_norm2', 'vt_opt_sgd', 'vt_opt_adamw',
           'vt_linear_small_fwd', 'vt_linear_small_bwd', 'vt_softmax_ce', 'vt_scale_by_scalar', 'vt_attn_probs',
           'vt_im2col_u8_mix_bf16', 'vt_pos_interp_fwd', 'vt_pos_interp_bwd']

_dll = None


def load_library() -> C.CDLL:
    """Load libvt_b200.so or fail loudly (no fallback path exists)."""
    global _dll
    if _dll is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} not found: build the sm_100a kernels first '
                f'(python -m videotransformer_pytorch_b200.build, or __graft_entry__.build()). '
                f'There is no CPU / library fallback for the hot path.')
        _dll = C.CDLL(LIB_PATH)
        for name in EXPORTS:
            getattr(_dll, name).restype = C.c_int
        if _dll.vt_version() != 1:
            raise RuntimeError('libvt_b200.so ABI version mismatch')
    return _dll


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(rc: int, what: str):
    if rc != 0:
        buf = C.create_string_buffer(512)
        load_library().vt_last_error(buf, 512)
        raise RuntimeError(f'{what} failed (code {rc}): {buf.value.decode(errors="replace")}')


def _req(t: torch.Tensor, dtype, name: str):
    if not t.is_cuda:
        raise RuntimeError(f'{name}: expected a CUDA tensor (the hot path has no CPU fallback)')
    if t.dtype != dtype:
        raise RuntimeError(f'{name}: expected dtype {dtype}, got {t.dtype}')
    return t


def _rows2d(t: torch.Tensor, name: str):
    if t.dim() != 2 or t.stride(1) != 1:
        raise RuntimeError(f'{name}: expected a 2-D row-contiguous tensor, got shape {tuple(t.shape)} stride {t.stride()}')
    return t


class CudaKernels:
    """Tensor-level wrappers; every method enqueues on torch's current CUDA stream."""

    name = 'cuda'

    def __init__(self):
        self._ws = {}
        self._counters = {}

    # -- scratch ------------------------------------------------------------------------------
    def workspace(self, device, nbytes: int) -> torch.Tensor:
        key = (device.index, torch.cuda.current_stream(device).cuda_stream)
        ws = self._ws.get(key)
        if ws is None or ws.numel() * 4 < nbytes:
            ws = torch.empty(max(nbytes, 64 << 20) // 4, dtype=torch.float32, device=device)
            self._ws[key] = ws
        return ws

    # -- GEMM ---------------------------------------------------------------------------------
    def gemm(self, a, b, M, N, Kdim, *, a_mn=False, b_mn=False, epi='bf16', bias=None, bias2=None, out=None, out2=None,
             aux=None, out_row=None, aux_row=None, row_scale=None, out_rows=None, split_ok=False,
             force_splits=0, force_bn=0, force_cluster=0, debug=None, row_map=None, force_tail=0, tag=None, out_zeroed=False):
        """row_map: affine description of out_row / aux_row (ops.affine_row_maps) for the fp32 residual epilogue — lets the
        kernel move 32 x 32 boxes by TMA through a tensor map of the token stream instead of per-thread rows.  tag: role label of the launch
        ('qkv', 'proj', ...) for profilers that wrap this method (bench.py); ignored here."""
        lib = load_library()
        _rows2d(_req(a, torch.bfloat16, 'gemm.a'), 'gemm.a')
        _rows2d(_req(b, torch.bfloat16, 'gemm.b'), 'gemm.b')
        exp_a = (Kdim, M) if a_mn else (M, Kdim)
        exp_b = (Kdim, N) if b_mn else (N, Kdim)
        if tuple(a.shape) != exp_a or tuple(b.shape) != exp_b:
            raise RuntimeError(f'gemm: operand shapes {tuple(a.shape)} {tuple(b.shape)} != expected {exp_a} {exp_b}')
        odt = torch.float32 if epi == 'f32' else torch.bfloat16
        if out is None:
            out = torch.empty((out_rows if out_rows is not None else M, N), dtype=odt, device=a.device)
        _rows2d(_req(out, odt, 'gemm.out'), 'gemm.out')
        if epi == 'gelu' and out2 is None:
            out2 = torch.empty_like(out)
        p = GemmParams()
        p.a, p.b = a.data_ptr(), b.data_ptr()
        p.lda, p.ldb = a.stride(0), b.stride(0)
        p.M, p.N, p.K = M, N, Kdim
        p.a_mn_major, p.b_mn_major = int(a_mn), int(b_mn)
        p.epilogue = EPI[epi]
        p.bias = _ptr(None if bias is None else _req(bias, torch.float32, 'gemm.bias'))
        if bias2 is not None:                  # fp32 epilogue with aux only: added after the row scale
            p.bias2 = _req(bias2, torch.float32, 'gemm.bias2').data_ptr()
        p.out, p.ldo = out.data_ptr(), out.stride(0)
        if out2 is not None:
            p.out2, p.ldo2 = out2.data_ptr(), out2.stride(0)
        if aux is not None:
            _rows2d(_req(aux, torch.float32 if epi == 'f32' else torch.bfloat16, 'gemm.aux'), 'gemm.aux')
            p.aux, p.ldaux = aux.data_ptr(), aux.stride(0)
        for nm, t in (('out_row', out_row), ('aux_row', aux_row)):
            if t is not None:
                _req(t, torch.int32, 'gemm.' + nm)
                if t.numel() != M:
                    raise RuntimeError(f'gemm.{nm}: expected {M} entries')
                setattr(p, nm, t.data_ptr())
        if row_scale is not None:
            _req(row_scale, torch.float32, 'gemm.row_scale')
            if row_scale.numel() != M:
                raise RuntimeError(f'gemm.row_scale: expected {M} entries, got {row_scale.numel()}')
            p.row_scale = row_scale.data_ptr()
        ws = None
        if split_ok and epi == 'f32':
            ws = self.workspace(a.device, 16 * M * N * 4)
            p.workspace, p.workspace_bytes = ws.data_ptr(), ws.numel() * 4
        p.force_splits, p.force_bn, p.force_cluster = force_splits, force_bn, force_cluster
        p.force_tail = force_tail
        p.out_zeroed = int(bool(out_zeroed) and out is not None)
        p.debug = _ptr(debug)
        p.map_special_base = -1
        if row_map is not None:
            if epi != 'f32' or aux is None:
                raise RuntimeError('gemm.row_map: only for the fp32 residual epilogue (epi="f32" with aux)')
            p.map_period, p.map_skip, p.map_tcount = row_map['period'], row_map['skip'], row_map['tcount']
            p.map_stride_t, p.map_stride_p, p.map_stride_b = row_map['stride_t'], row_map['stride_p'], row_map['stride_b']
            p.map_base = row_map['base']
            p.map_special_base, p.map_special_stride = row_map.get('special_base', -1), row_map.get('special_stride', 0)
        _check(lib.vt_gemm(C.byref(p), _stream()), 'vt_gemm')
        return (out, out2) if epi == 'gelu' else out

    # -- LayerNorm ----------------------------------------------------------------------------
    def ln_fwd(self, x2d, gamma, beta, eps, in_row=None, rows=None, out_fp32=False):
        lib = load_library()
        _rows2d(_req(x2d, torch.float32, 'ln_fwd.x'), 'ln_fwd.x')
        rows = x2d.shape[0] if rows is None else rows
        D = x2d.shape[1]
        y = torch.empty((rows, D), dtype=torch.float32 if out_fp32 else torch.bfloat16, device=x2d.device)
        mean = torch.empty(rows, dtype=torch.float32, device=x2d.device)
        rstd = torch.empty_like(mean)
        p = LnFwdParams()
        p.x, p.ldx = x2d.data_ptr(), x2d.stride(0)
        p.in_row = _ptr(None if in_row is None else _req(in_row, torch.int32, 'ln_fwd.in_row'))
        p.gamma, p.beta = _req(gamma, torch.float32, 'gamma').data_ptr(), _req(beta, torch.float32, 'beta').data_ptr()
        p.y, p.mean, p.rstd = y.data_ptr(), mean.data_ptr(), rstd.data_ptr()
        p.rows, p.D, p.eps, p.y_fp32 = rows, D, eps, int(out_fp32)
        _check(lib.vt_layernorm_fwd(C.byref(p), _stream()), 'vt_layernorm_fwd')
        return y, mean, rstd

    def ln_bwd(self, dy, x2d, mean, rstd, gamma, in_row=None, out_row=None, dres=None, dx=None, n_aux=0):
        """-> (dx [x2d.shape] or given, dx_aux [n_aux, D] or None, dgamma, dbeta)"""
        lib = load_library()
        rows, D = dy.shape
        dev = dy.device
        if dx is None:
            dx = torch.empty((x2d.shape[0], D), dtype=torch.float32, device=dev)
        dx_aux = torch.empty((n_aux, D), dtype=torch.float32, device=dev) if n_aux else None
        blocks = lib.vt_ln_bwd_blocks(rows)
        partials = torch.empty((blocks, 2, D), dtype=torch.float32, device=dev)
        p = LnBwdParams()
        p.dy, p.dy_fp32 = dy.data_ptr(), int(dy.dtype == torch.float32)
        p.x, p.ldx = x2d.data_ptr(), x2d.stride(0)
        p.in_row = _ptr(in_row)
        p.mean, p.rstd, p.gamma = mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr()
        p.dres = _ptr(dres)
        p.dx, p.lddx = dx.data_ptr(), dx.stride(0)
        p.dx_aux = _ptr(dx_aux)
        p.out_row = _ptr(out_row)
        p.partials = partials.data_ptr()
        p.rows, p.D = rows, D
        _check(lib.vt_layernorm_bwd(C.byref(p), _stream()), 'vt_layernorm_bwd')
        gb = torch.empty((2, D), dtype=torch.float32, device=dev)
        r = ReduceParams()
        r.inp, r.out, r.stride, r.S, r.n, r.accumulate, r.scale = partials.data_ptr(), gb.data_ptr(), 2 * D, blocks, 2 * D, 0, 1.0
        _check(lib.vt_reduce_rows(C.byref(r), _stream()), 'vt_reduce_rows')
        return dx, dx_aux, gb[0], gb[1]

    # -- reductions / casts -------------------------------------------------------------------
    def colsum(self, x):
        lib = load_library()
        _rows2d(_req(x, torch.bfloat16, 'colsum.x'), 'colsum.x')
        M, N = x.shape
        out = torch.empty(N, dtype=torch.float32, device=x.device)
        ws = torch.empty((lib.vt_colsum_chunks(M), N), dtype=torch.float32, device=x.device)
        key = (x.device.index, torch.cuda.current_stream(x.device).cuda_stream)
        cnt = self._counters.get(key)
        if cnt is None:
            cnt = self._counters[key] = torch.zeros(1024, dtype=torch.int32, device=x.device)
        p = ColsumParams()
        p.inp, p.ld, p.M, p.N, p.out, p.workspace = x.data_ptr(), x.stride(0), M, N, out.data_ptr(), ws.data_ptr()
        p.counters = cnt.data_ptr() if N <= 64 * 1024 else None
        _check(lib.vt_colsum_bf16(C.byref(p), _stream()), 'vt_colsum_bf16')
        return out

    def cast_bf16(self, x):
        lib = load_library()
        x = _req(x, torch.float32, 'cast.x').contiguous()
        out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
        p = CastParams()
        p.src, p.dst, p.n = x.data_ptr(), out.data_ptr(), x.numel()
        _check(lib.vt_cast_f32_bf16(C.byref(p), _stream()), 'vt_cast_f32_bf16')
        return out

    def gather_cast(self, src2d, in_row=None, row_scale=None, rows=None):
        lib = load_library()
        _rows2d(_req(src2d, torch.float32, 'gather_cast.src'), 'gather_cast.src')
        rows = src2d.shape[0] if rows is None else rows
        D = src2d.shape[1]
        out = torch.empty((rows, D), dtype=torch.bfloat16, device=src2d.device)
        p = GatherCastParams()
        p.src, p.lds = src2d.data_ptr(), src2d.stride(0)
        p.in_row, p.row_scale = _ptr(in_row), _ptr(row_scale)
        p.dst, p.rows, p.D = out.data_ptr(), rows, D
        _check(lib.vt_gather_cast_bf16(C.byref(p), _stream()), 'vt_gather_cast_bf16')
        return out

    def cls_rows(self, dst, src, extra=None, scale=1.0):
        """dst[b, :] = src[b, :] + scale * extra[b].sum(0);  dst / src: fp32 [B, D] row views (unit inner stride), extra: fp32
        contiguous [B, T, D] or None."""
        lib = load_library()
        for t, n in ((dst, 'dst'), (src, 'src')):
            _req(t, torch.float32, 'cls_rows.' + n)
            if t.dim() != 2 or t.stride(1) != 1 or t.shape != dst.shape:
                raise RuntimeError(f'cls_rows.{n}: expected a [B, D] row view with unit inner stride')
        p = ClsRowsParams()
        p.src, p.src_stride, p.dst, p.dst_stride = src.data_ptr(), src.stride(0), dst.data_ptr(), dst.stride(0)
        p.B, p.D, p.scale = dst.shape[0], dst.shape[1], float(scale)
        if extra is not None:
            _req(extra, torch.float32, 'cls_rows.extra')
            if extra.dim() != 3 or not extra.is_contiguous() or extra.shape[0] != p.B or extra.shape[2] != p.D:
                raise RuntimeError('cls_rows.extra: expected a contiguous [B, T, D] tensor')
            p.extra, p.extra_bs, p.T = extra.data_ptr(), extra.stride(0), extra.shape[1]
        _check(lib.vt_cls_rows(C.byref(p), _stream()), 'vt_cls_rows')
        return dst

    def gather_cast_colsum(self, src2d, in_row=None, row_scale=None, rows=None, unscaled_sums=False):
        """gather_cast + colsum of its output in one pass -> (bf16 [rows, D], fp32 [D]); with unscaled_sums a third result:
        the column sums of the same rows before row_scale.  D <= 1024, else separate kernels."""
        lib = load_library()
        _rows2d(_req(src2d, torch.float32, 'gather_cast.src'), 'gather_cast.src')
        rows = src2d.shape[0] if rows is None else rows
        D = src2d.shape[1]
        if D > 1024 or D % 8:
            out = self.gather_cast(src2d, in_row=in_row, row_scale=row_scale, rows=rows)
            if unscaled_sums:
                return out, self.colsum(out), self.colsum(self.gather_cast(src2d, in_row=in_row, rows=rows))
            return out, self.colsum(out)
        dev = src2d.device
        out = torch.empty((rows, D), dtype=torch.bfloat16, device=dev)
        nsum = 2 if unscaled_sums else 1
        cs = torch.empty((nsum, D), dtype=torch.float32, device=dev)
        nb = lib.vt_gather_cast_colsum_blocks(rows)
        ws = torch.empty((nb, nsum * D), dtype=torch.float32, device=dev)
        p = GatherCastColsumParams()
        p.src, p.lds = src2d.data_ptr(), src2d.stride(0)
        p.in_row, p.row_scale = _ptr(in_row), _ptr(row_scale)
        p.dst, p.rows, p.D = out.data_ptr(), rows, D
        p.colsum, p.workspace, p.workspace_rows, p.unscaled_sums = cs.data_ptr(), ws.data_ptr(), nb, int(unscaled_sums)
        _check(lib.vt_gather_cast_colsum_bf16(C.byref(p), _stream()), 'vt_gather_cast_colsum_bf16')
        return (out, cs[0], cs[1]) if unscaled_sums else (out, cs[0])

    def dgelu_colsum(self, dh, z):
        """dz = dh * gelu'(z) and the column sums of dz in one pass -> (bf16 [M, N], fp32 [N])."""
        lib = load_library()
        for t, n in ((dh, 'dh'), (z, 'z')):
            _req(t, torch.bfloat16, 'dgelu.' + n)
            if not t.is_contiguous() or t.dim() != 2:
                raise RuntimeError(f'dgelu_colsum: {n} must be a contiguous matrix')
        M, N = z.shape
        if N % 256 or N > 8192:
            out = self.dgelu(dh, z)
            return out, self.colsum(out)
        dev = z.device
        out = torch.empty_like(z)
        cs = torch.empty(N, dtype=torch.float32, device=dev)
        nb = lib.vt_gelu_bwd_colsum_blocks(M)
        ws = torch.empty((nb, N), dtype=torch.float32, device=dev)
        p = GeluBwdColsumParams()
        p.z, p.dh, p.out, p.M, p.N = z.data_ptr(), dh.data_ptr(), out.data_ptr(), M, N
        p.colsum, p.workspace, p.workspace_rows = cs.data_ptr(), ws.data_ptr(), nb
        _check(lib.vt_gelu_bwd_colsum_bf16(C.byref(p), _stream()), 'vt_gelu_bwd_colsum_bf16')
        return out, cs

    def gelu(self, z):
        lib = load_library()
        z = _req(z, torch.bfloat16, 'gelu.z')
        if not z.is_contiguous():
            raise RuntimeError('gelu: z must be contiguous')
        out = torch.empty_like(z)
        p = GeluParams()
        p.z, p.dh, p.out, p.n = z.data_ptr(), None, out.data_ptr(), z.numel()
        _check(lib.vt_gelu_fwd_bf16(C.byref(p), _stream()), 'vt_gelu_fwd_bf16')
        return out

    def dgelu(self, dh, z):
        lib = load_library()
        for t, n in ((dh, 'dh'), (z, 'z')):
            _req(t, torch.bfloat16, 'dgelu.' + n)
            if not t.is_contiguous():
                raise RuntimeError(f'dgelu: {n} must be contiguous')
        out = torch.empty_like(z)
        p = GeluParams()
        p.z, p.dh, p.out, p.n = z.data_ptr(), dh.data_ptr(), out.data_ptr(), z.numel()
        _check(lib.vt_gelu_bwd_bf16(C.byref(p), _stream()), 'vt_gelu_bwd_bf16')
        return out

    # -- attention ----------------------------------------------------------------------------
    def attn_fwd(self, qkv, Bp, N, H, hd, scale, want_probs=False, impl=0):
        lib = load_library()
        _req(qkv, torch.bfloat16, 'attn.qkv')
        if not qkv.is_contiguous() or qkv.numel() != Bp * N * 3 * H * hd:
            raise RuntimeError('attn_fwd: qkv must be contiguous [Bp, N, 3, H, hd]')
        ctx = torch.empty((Bp * N, H * hd), dtype=torch.bfloat16, device=qkv.device)
        lse = torch.empty((Bp, H, N), dtype=torch.float32, device=qkv.device)
        probs = torch.empty((Bp, H, N, N), dtype=torch.float32, device=qkv.device) if want_probs else None
        p = AttnFwdParams()
        p.qkv, p.ctx, p.lse, p.probs = qkv.data_ptr(), ctx.data_ptr(), lse.data_ptr(), _ptr(probs)
        p.Bp, p.N, p.H, p.hd, p.scale, p.impl = Bp, N, H, hd, scale, impl
        _check(lib.vt_attn_fwd(C.byref(p), _stream()), 'vt_attn_fwd')
        return ctx, lse, probs

    def attn_bwd(self, qkv, ctx, dctx, lse, Bp, N, H, hd, scale, impl=0):
        lib = load_library()
        for t, n in ((qkv, 'qkv'), (ctx, 'ctx'), (dctx, 'dctx')):
            _req(t, torch.bfloat16, 'attn_bwd.' + n)
            if not t.is_contiguous():
                raise RuntimeError(f'attn_bwd: {n} must be contiguous')
        dqkv = torch.empty_like(qkv)
        p = AttnBwdParams()
        p.qkv, p.ctx, p.dctx, p.lse, p.dqkv = qkv.data_ptr(), ctx.data_ptr(), dctx.data_ptr(), lse.data_ptr(), dqkv.data_ptr()
        p.Bp, p.N, p.H, p.hd, p.scale, p.impl = Bp, N, H, hd, scale, impl
        _check(lib.vt_attn_bwd(C.byref(p), _stream()), 'vt_attn_bwd')
        return dqkv

    def attn_probs(self, qkv, Bp, N, H, hd, scale):
        """softmax(q k^T * scale) of a packed projection [Bp, N, 3, H, hd] -> fp32 [Bp, H, N, N] (any N; head dim 64)"""
        lib = load_library()
        _req(qkv, torch.bfloat16, 'attn_probs.qkv')
        if not qkv.is_contiguous() or qkv.numel() != Bp * N * 3 * H * hd:
            raise RuntimeError('attn_probs: qkv must be contiguous [Bp, N, 3, H, hd]')
        probs = torch.empty((Bp, H, N, N), dtype=torch.float32, device=qkv.device)
        p = AttnProbsParams()
        p.qkv, p.probs = qkv.data_ptr(), probs.data_ptr()
        p.Bp, p.N, p.H, p.hd, p.scale = Bp, N, H, hd, scale
        _check(lib.vt_attn_probs(C.byref(p), _stream()), 'vt_attn_probs')
        return probs

    # -- classification head + loss -----------------------------------------------------------
    def linear_small_fwd(self, x, w, b):
        lib = load_library()
        for t, n in ((x, 'x'), (w, 'w')):
            _rows2d(_req(t, torch.float32, 'linear_small.' + n), 'linear_small.' + n)
            if not t.is_contiguous():
                raise RuntimeError(f'linear_small: {n} must be contiguous')
        M, Kd = x.shape
        N = w.shape[0]
        if w.shape[1] != Kd:
            raise RuntimeError('linear_small: shape mismatch')
        y = torch.empty((M, N), dtype=torch.float32, device=x.device)
        p = LinearSmallParams()
        p.x, p.w, p.b, p.y = x.data_ptr(), w.data_ptr(), _ptr(None if b is None else _req(b, torch.float32, 'linear_small.b')), y.data_ptr()
        p.M, p.N, p.K = M, N, Kd
        _check(lib.vt_linear_small_fwd(C.byref(p), _stream()), 'vt_linear_small_fwd')
        return y

    def linear_small_bwd(self, dy, x, w, need_dx=True, need_dw=True):
        """-> (dx | None, dw | None, db | None)"""
        lib = load_library()
        for t, n in ((dy, 'dy'), (x, 'x'), (w, 'w')):
            _req(t, torch.float32, 'linear_small_bwd.' + n)
            if not t.is_contiguous():
                raise RuntimeError(f'linear_small_bwd: {n} must be contiguous')
        M, Kd = x.shape
        N = w.shape[0]
        dev = x.device
        dx = torch.empty((M, Kd), dtype=torch.float32, device=dev) if need_dx else None
        dw = torch.empty((N, Kd), dtype=torch.float32, device=dev) if need_dw else None
        db = torch.empty(N, dtype=torch.float32, device=dev) if need_dw else None
        p = LinearSmallBwdParams()
        p.dy, p.x, p.w = dy.data_ptr(), x.data_ptr(), w.data_ptr()
        p.dw, p.db, p.dx = _ptr(dw), _ptr(db), _ptr(dx)
        p.M, p.N, p.K = M, N, Kd
        _check(lib.vt_linear_small_bwd(C.byref(p), _stream()), 'vt_linear_small_bwd')
        return dx, dw, db

    def softmax_ce(self, logits, labels=None, soft_targets=None):
        """mean cross-entropy over rows -> (loss fp32 [1], dlogits fp32 [M,N], row_loss fp32 [M])"""
        lib = load_library()
        logits = _req(logits, torch.float32, 'softmax_ce.logits')
        if logits.dim() != 2 or not logits.is_contiguous():
            raise RuntimeError('softmax_ce: logits must be contiguous [M, N]')
        M, N = logits.shape
        dev = logits.device
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        row = torch.empty(M, dtype=torch.float32, device=dev)
        dz = torch.empty_like(logits)
        p = SoftmaxCeParams()
        p.logits, p.loss, p.row_loss, p.dlogits = logits.data_ptr(), loss.data_ptr(), row.data_ptr(), dz.data_ptr()
        if (labels is None) == (soft_targets is None):
            raise RuntimeError('softmax_ce: give labels or soft_targets')
        if labels is not None:
            labels = _req(labels, torch.int64, 'softmax_ce.labels').contiguous()
            if labels.numel() != M:
                raise RuntimeError('softmax_ce: one label per row expected')
            p.labels = labels.data_ptr()
        else:
            soft_targets = _req(soft_targets, torch.float32, 'softmax_ce.soft_targets').contiguous()
            if tuple(soft_targets.shape) != (M, N):
                raise RuntimeError('softmax_ce: soft_targets must be [M, N]')
            p.soft_targets = soft_targets.data_ptr()
        p.M, p.N = M, N
        _check(lib.vt_softmax_ce(C.byref(p), _stream()), 'vt_softmax_ce')
        return loss, dz, row

    def scale_by_scalar(self, t, scalar):
        lib = load_library()
        t = _req(t, torch.float32, 'scale.t')
        if not t.is_contiguous():
            raise RuntimeError('scale_by_scalar: tensor must be contiguous')
        scalar = _req(scalar, torch.float32, 'scale.scalar')
        out = torch.empty_like(t)
        p = ScaleParams()
        p.inp, p.scalar, p.out, p.n = t.data_ptr(), scalar.data_ptr(), out.data_ptr(), t.numel()
        _check(lib.vt_scale_by_scalar(C.byref(p), _stream()), 'vt_scale_by_scalar')
        return out

    # -- patch embedding operand -------------------------------------------------------------
    def im2col(self, x, tube, ph, pw):
        lib = load_library()
        x = _req(x, torch.float32, 'im2col.x').contiguous()
        B, T, Cc, H, W = x.shape
        rows = B * (T // tube) * (H // ph) * (W // pw)
        cols = torch.empty((rows, Cc * tube * ph * pw), dtype=torch.bfloat16, device=x.device)
        p = Im2colParams()
        p.x, p.cols = x.data_ptr(), cols.data_ptr()
        p.B, p.T, p.C, p.H, p.W, p.tube, p.ph, p.pw = B, T, Cc, H, W, tube, ph, pw
        _check(lib.vt_im2col_bf16(C.byref(p), _stream()), 'vt_im2col_bf16')
        return cols

    def im2col_u8(self, x, scale, shift, tube, ph, pw):
        """x u8 [B,T,H,W,C] -> normalised bf16 patch rows [B*(T/tube)*(H/ph)*(W/pw), C*tube*ph*pw]"""
        lib = load_library()
        x = _req(x, torch.uint8, 'im2col_u8.x').contiguous()
        B, T, H, W, Cc = x.shape
        rows = B * (T // tube) * (H // ph) * (W // pw)
        cols = torch.empty((rows, Cc * tube * ph * pw), dtype=torch.bfloat16, device=x.device)
        p = Im2colU8Params()
        p.x, p.cols = x.data_ptr(), cols.data_ptr()
        p.scale, p.shift = _req(scale, torch.float32, 'im2col_u8.scale').data_ptr(), _req(shift, torch.float32, 'im2col_u8.shift').data_ptr()
        p.B, p.T, p.C, p.H, p.W, p.tube, p.ph, p.pw = B, T, Cc, H, W, tube, ph, pw
        _check(lib.vt_im2col_u8_bf16(C.byref(p), _stream()), 'vt_im2col_u8_bf16')
        return cols

    def im2col_u8_mix(self, x, scale, shift, plan, tube, ph, pw):
        """im2col_u8 with Mixup / CutMix against the flipped batch; plan: fp32 [6] device tensor {mode, lam, yl, yh, xl, xh}"""
        lib = load_library()
        x = _req(x, torch.uint8, 'im2col_u8_mix.x').contiguous()
        B, T, H, W, Cc = x.shape
        rows = B * (T // tube) * (H // ph) * (W // pw)
        cols = torch.empty((rows, Cc * tube * ph * pw), dtype=torch.bfloat16, device=x.device)
        p = Im2colU8MixParams()
        p.x, p.cols = x.data_ptr(), cols.data_ptr()
        p.scale, p.shift = _req(scale, torch.float32, 'im2col_u8_mix.scale').data_ptr(), _req(shift, torch.float32, 'im2col_u8_mix.shift').data_ptr()
        if plan.numel() < 6:
            raise RuntimeError('im2col_u8_mix: plan must hold 6 floats {mode, lam, yl, yh, xl, xh}')
        p.plan = _req(plan, torch.float32, 'im2col_u8_mix.plan').data_ptr()
        p.B, p.T, p.C, p.H, p.W, p.tube, p.ph, p.pw = B, T, Cc, H, W, tube, ph, pw
        _check(lib.vt_im2col_u8_mix_bf16(C.byref(p), _stream()), 'vt_im2col_u8_mix_bf16')
        return cols

    def col2im(self, cols, shape, tube, ph, pw):
        lib = load_library()
        cols = _req(cols, torch.float32, 'col2im.cols').contiguous()
        B, T, Cc, H, W = shape
        dx = torch.empty(shape, dtype=torch.float32, device=cols.device)
        p = Im2colParams()
        p.x, p.cols = cols.data_ptr(), dx.data_ptr()   # same POD layout: (src, dst, dims)
        p.B, p.T, p.C, p.H, p.W, p.tube, p.ph, p.pw = B, T, Cc, H, W, tube, ph, pw
        _check(lib.vt_col2im_f32(C.byref(p), _stream()), 'vt_col2im_f32')
        return dx

    # -- position-table resampling -------------------------------------------------------------
    def _pos_interp(self, fn, src, rows_out, side, rows, cols, scale_r, scale_c):
        lib = load_library()
        src = _req(src, torch.float32, fn + '.in')
        if src.dim() != 2 or not src.is_contiguous():
            raise RuntimeError(f'{fn}: expected a contiguous [rows, D] table')
        out = torch.empty((rows_out, src.shape[1]), dtype=torch.float32, device=src.device)
        p = PosInterpParams()
        p.inp, p.out = src.data_ptr(), out.data_ptr()
        p.D, p.src_side, p.out_rows, p.out_cols = src.shape[1], side, rows, cols
        p.scale_r, p.scale_c = scale_r, scale_c
        _check(getattr(lib, fn)(C.byref(p), _stream()), fn)
        return out

    def pos_interp_fwd(self, table, side, rows, cols, scale_r, scale_c):
        """fp32 [1 + side^2, D] -> bicubically resampled [1 + rows*cols, D] (cls row copied); scale_* = 1 / scale factor"""
        if table.shape[0] != 1 + side * side:
            raise RuntimeError(f'pos_interp_fwd: table has {table.shape[0]} rows, expected 1 + {side}^2')
        return self._pos_interp('vt_pos_interp_fwd', table, 1 + rows * cols, side, rows, cols, scale_r, scale_c)

    def pos_interp_bwd(self, dout, side, rows, cols, scale_r, scale_c):
        """adjoint of pos_interp_fwd: fp32 [1 + rows*cols, D] -> [1 + side^2, D]"""
        if dout.shape[0] != 1 + rows * cols:
            raise RuntimeError(f'pos_interp_bwd: gradient has {dout.shape[0]} rows, expected 1 + {rows}*{cols}')
        return self._pos_interp('vt_pos_interp_bwd', dout, 1 + side * side, side, rows, cols, scale_r, scale_c)

    # -- HOG ------------------------------------------------------------------------------------
    def hog(self, frames, lut, want_bins=False):
        lib = load_library()
        frames = _req(frames, torch.uint8, 'hog.frames').contiguous()
        F, H, W, c3 = frames.shape
        if c3 != 3:
            raise RuntimeError('hog: frames must be [F, H, W, 3] uint8')
        feat = torch.empty((F, H // 16, W // 16, 108), dtype=torch.float32, device=frames.device)
        bins = torch.empty((F, 3, H, W), dtype=torch.uint8, device=frames.device) if want_bins else None
        p = HogParams()
        p.frames, p.lut, p.feat, p.bins = frames.data_ptr(), _req(lut, torch.uint8, 'hog.lut').data_ptr(), feat.data_ptr(), _ptr(bins)
        p.F, p.H, p.W = F, H, W
        _check(lib.vt_hog(C.byref(p), _stream()), 'vt_hog')
        return feat, bins


    # -- MViT / MaskFeat (include/vt_b200.h, second half) -----------------------------------------
    @staticmethod
    def pool_out_thw(thw, stride):
        return tuple((n + 2 - 3) // s + 1 for n, s in zip(thw, stride))

    @staticmethod
    def _tok_view(t, name, B, H, hd):
        """[B, N, H*hd] bf16 view with unit last stride (a q/k/v slice of the fused projection output)."""
        _req(t, torch.bfloat16, name)
        if t.dim() != 3 or t.shape[0] != B or t.shape[2] != H * hd or t.stride(2) != 1:
            raise RuntimeError(f'{name}: expected a [B, N, H*hd] view with unit last stride, got {tuple(t.shape)} {t.stride()}')
        return t

    def pool_fwd(self, src, H, hd, thw, stride, w, gamma, beta, eps):
        """src: [B, 1+T*Hin*Win, H*hd] bf16 view -> (out bf16 [B,H,1+Lo,hd], pooled fp32, mean, rstd, out_thw)"""
        lib = load_library()
        B = src.shape[0]
        self._tok_view(src, 'pool_fwd.src', B, H, hd)
        T, Hin, Win = thw
        if src.shape[1] != 1 + T * Hin * Win:
            raise RuntimeError('pool_fwd: token count does not match thw')
        To, Ho, Wo = self.pool_out_thw(thw, stride)
        Lo1 = 1 + To * Ho * Wo
        dev = src.device
        pooled = torch.empty((B, H, Lo1, hd), dtype=torch.float32, device=dev)
        out = torch.empty((B, H, Lo1, hd), dtype=torch.bfloat16, device=dev)
        mean = torch.empty(B * H * Lo1, dtype=torch.float32, device=dev)
        rstd = torch.empty_like(mean)
        p = PoolFwdParams()
        p.inp, p.in_bs, p.in_rs = src.data_ptr(), src.stride(0), src.stride(1)
        p.w = _req(w, torch.float32, 'pool_fwd.w').contiguous().data_ptr()
        p.gamma, p.beta = _req(gamma, torch.float32, 'gamma').data_ptr(), _req(beta, torch.float32, 'beta').data_ptr()
        p.pooled, p.out, p.mean, p.rstd = pooled.data_ptr(), out.data_ptr(), mean.data_ptr(), rstd.data_ptr()
        p.B, p.H, p.hd, p.T, p.Hin, p.Win = B, H, hd, T, Hin, Win
        p.st, p.sh, p.sw = stride
        p.To, p.Ho, p.Wo, p.eps = To, Ho, Wo, eps
        _check(lib.vt_pool_fwd(C.byref(p), _stream()), 'vt_pool_fwd')
        return out, pooled, mean, rstd, (To, Ho, Wo)

    def pool_bwd(self, dout, pooled, mean, rstd, gamma, src, w, din, H, hd, thw, stride):
        """Writes din (a [B, N, H*hd] bf16 view like src) in place -> (dw [hd,27], dgamma, dbeta)"""
        lib = load_library()
        B = src.shape[0]
        self._tok_view(src, 'pool_bwd.src', B, H, hd)
        self._tok_view(din, 'pool_bwd.din', B, H, hd)
        if dout.dtype not in (torch.float32, torch.bfloat16) or not dout.is_contiguous() or dout.shape != pooled.shape:
            raise RuntimeError('pool_bwd: dout must be contiguous [B,H,1+Lo,hd] in fp32 or bf16')
        T, Hin, Win = thw
        To, Ho, Wo = self.pool_out_thw(thw, stride)
        rows_out = B * H * (1 + To * Ho * Wo)
        dev = src.device
        need = lib.vt_pool_bwd_scratch(rows_out, hd)
        if need <= 0:
            raise RuntimeError('pool_bwd: problem too large')
        scratch = torch.empty(need, dtype=torch.float32, device=dev)
        dw = torch.empty((hd, 27), dtype=torch.float32, device=dev)
        gb = torch.empty((2, hd), dtype=torch.float32, device=dev)      # adjacent: the library sums both with one launch
        dgamma, dbeta = gb[0], gb[1]
        p = PoolBwdParams()
        p.dout, p.dout_fp32 = dout.data_ptr(), int(dout.dtype == torch.float32)
        p.pooled, p.mean, p.rstd, p.gamma = pooled.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr()
        p.inp, p.in_bs, p.in_rs = src.data_ptr(), src.stride(0), src.stride(1)
        p.w = _req(w, torch.float32, 'pool_bwd.w').contiguous().data_ptr()
        p.din, p.din_bs, p.din_rs = din.data_ptr(), din.stride(0), din.stride(1)
        p.dw, p.dgamma, p.dbeta = dw.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr()
        p.scratch, p.scratch_floats = scratch.data_ptr(), need
        p.B, p.H, p.hd, p.T, p.Hin, p.Win = B, H, hd, T, Hin, Win
        p.st, p.sh, p.sw = stride
        p.To, p.Ho, p.Wo = To, Ho, Wo
        _check(lib.vt_pool_bwd(C.byref(p), _stream()), 'vt_pool_bwd')
        return dw, dgamma, dbeta

    @staticmethod
    def _bhnd(t, name):
        """[B, H, N, hd] bf16 view, unit last stride -> (ptr, bs, hs, rs)"""
        _req(t, torch.bfloat16, name)
        if t.dim() != 4 or t.stride(3) != 1:
            raise RuntimeError(f'{name}: expected a [B,H,N,hd] view with unit last stride')
        return t.data_ptr(), t.stride(0), t.stride(1), t.stride(2)

    def xattn_fwd(self, q, k, v, scale, impl=0):
        """q [B,H,Nq,hd], k/v [B,H,Nk,hd] bf16 views -> (o bf16 [B, Nq, H*hd], lse fp32 [B,H,Nq])"""
        lib = load_library()
        B, H, Nq, hd = q.shape
        Nk = k.shape[2]
        o = torch.empty((B, Nq, H * hd), dtype=torch.bfloat16, device=q.device)
        lse = torch.empty((B, H, Nq), dtype=torch.float32, device=q.device)
        p = XattnFwdParams()
        p.q, p.q_bs, p.q_hs, p.q_rs = self._bhnd(q, 'xattn.q')
        p.k, p.k_bs, p.k_hs, p.k_rs = self._bhnd(k, 'xattn.k')
        p.v, p.v_bs, p.v_hs, p.v_rs = self._bhnd(v, 'xattn.v')
        p.o, p.o_bs, p.o_hs, p.o_rs = o.data_ptr(), Nq * H * hd, hd, H * hd
        p.lse = lse.data_ptr()
        p.B, p.H, p.Nq, p.Nk, p.hd, p.scale, p.impl = B, H, Nq, Nk, hd, scale, impl
        _check(lib.vt_xattn_fwd(C.byref(p), _stream()), 'vt_xattn_fwd')
        return o, lse

    def xattn_bwd(self, q, k, v, o, dout, lse, scale, dq, impl=0):
        """o, dout: bf16 [B, Nq, H*hd] contiguous; dq: bf16 [B,H,Nq,hd] view written in place -> (dk, dv) fp32 [B,H,Nk,hd]"""
        lib = load_library()
        B, H, Nq, hd = q.shape
        Nk = k.shape[2]
        for t, n in ((o, 'o'), (dout, 'dout')):
            _req(t, torch.bfloat16, 'xattn_bwd.' + n)
            if not t.is_contiguous() or t.numel() != B * Nq * H * hd:
                raise RuntimeError(f'xattn_bwd: {n} must be contiguous [B, Nq, H*hd]')
        dev = q.device
        delta = torch.empty((B, H, Nq), dtype=torch.float32, device=dev)
        dk = torch.empty((B, H, Nk, hd), dtype=torch.float32, device=dev)
        dv = torch.empty_like(dk)
        p = XattnBwdParams()
        p.q, p.q_bs, p.q_hs, p.q_rs = self._bhnd(q, 'xattn.q')
        p.k, p.k_bs, p.k_hs, p.k_rs = self._bhnd(k, 'xattn.k')
        p.v, p.v_bs, p.v_hs, p.v_rs = self._bhnd(v, 'xattn.v')
        p.dq, p.dq_bs, p.dq_hs, p.dq_rs = self._bhnd(dq, 'xattn.dq')
        p.o, p.dout = o.data_ptr(), dout.data_ptr()
        p.o_bs, p.o_hs, p.o_rs = Nq * H * hd, hd, H * hd
        p.lse, p.delta, p.dk, p.dv = lse.data_ptr(), delta.data_ptr(), dk.data_ptr(), dv.data_ptr()
        p.B, p.H, p.Nq, p.Nk, p.hd, p.scale, p.impl = B, H, Nq, Nk, hd, scale, impl
        _check(lib.vt_xattn_bwd(C.byref(p), _stream()), 'vt_xattn_bwd')
        return dk, dv

    @staticmethod
    def maxpool_out_thw(thw, kernel, stride):
        return tuple((n + 2 * (k // 2) - k) // s + 1 for n, k, s in zip(thw, kernel, stride))

    def _mp_dims(self, p, B, D, thw, kernel, stride):
        p.B, p.D = B, D
        p.T, p.H, p.W = thw
        p.kt, p.kh, p.kw = kernel
        p.st, p.sh, p.sw = stride
        p.To, p.Ho, p.Wo = self.maxpool_out_thw(thw, kernel, stride)

    def maxpool_fwd(self, x, thw, kernel, stride):
        """x fp32 [B, 1+T*H*W, D] -> (y fp32 [B, 1+Lo, D], idx u8, out_thw)"""
        lib = load_library()
        x = _req(x, torch.float32, 'maxpool.x')
        if not x.is_contiguous() or x.shape[1] != 1 + thw[0] * thw[1] * thw[2]:
            raise RuntimeError('maxpool_fwd: x must be contiguous [B, 1+T*H*W, D]')
        B, _, D = x.shape
        out_thw = self.maxpool_out_thw(thw, kernel, stride)
        Lo1 = 1 + out_thw[0] * out_thw[1] * out_thw[2]
        y = torch.empty((B, Lo1, D), dtype=torch.float32, device=x.device)
        idx = torch.empty((B, Lo1, D), dtype=torch.uint8, device=x.device)
        p = MaxpoolFwdParams()
        p.x, p.y, p.idx = x.data_ptr(), y.data_ptr(), idx.data_ptr()
        self._mp_dims(p, B, D, thw, kernel, stride)
        _check(lib.vt_maxpool_fwd(C.byref(p), _stream()), 'vt_maxpool_fwd')
        return y, idx, out_thw

    def maxpool_bwd(self, dy, idx, thw, kernel, stride):
        lib = load_library()
        dy = _req(dy, torch.float32, 'maxpool_bwd.dy')
        if not dy.is_contiguous() or dy.shape != idx.shape:
            raise RuntimeError('maxpool_bwd: dy must be contiguous and match idx')
        B, _, D = dy.shape
        dx = torch.empty((B, 1 + thw[0] * thw[1] * thw[2], D), dtype=torch.float32, device=dy.device)
        p = MaxpoolBwdParams()
        p.dy, p.idx, p.dx = dy.data_ptr(), idx.data_ptr(), dx.data_ptr()
        self._mp_dims(p, B, D, thw, kernel, stride)
        _check(lib.vt_maxpool_bwd(C.byref(p), _stream()), 'vt_maxpool_bwd')
        return dx

    def im2col3d(self, x, kernel, stride, padding, kpad):
        """x fp32 [B,T,C,H,W] -> (cols bf16 [B*To*Ho*Wo, kpad], (To,Ho,Wo))"""
        lib = load_library()
        x = _req(x, torch.float32, 'im2col3d.x').contiguous()
        B, T, Cc, H, W = x.shape
        out = tuple((n + 2 * pd - k) // s + 1 for n, pd, k, s in zip((T, H, W), padding, kernel, stride))
        cols = torch.empty((B * out[0] * out[1] * out[2], kpad), dtype=torch.bfloat16, device=x.device)
        p = Im2col3dParams()
        p.x, p.cols = x.data_ptr(), cols.data_ptr()
        p.B, p.T, p.C, p.H, p.W = B, T, Cc, H, W
        p.kt, p.kh, p.kw = kernel
        p.st, p.sh, p.sw = stride
        p.pt, p.ph, p.pw = padding
        p.To, p.Ho, p.Wo = out
        p.Kpad = kpad
        _check(lib.vt_im2col3d_bf16(C.byref(p), _stream()), 'vt_im2col3d_bf16')
        return cols, out

    def mvit_tokens_fwd(self, t, wmask, mask_token, cls_token, pos_s, pos_t, pos_cls, B, T, HW):
        lib = load_library()
        t = _req(t, torch.float32, 'tokens.t')
        Cc = t.shape[1]
        if not t.is_contiguous() or t.shape[0] != B * T * HW:
            raise RuntimeError('mvit_tokens_fwd: t must be contiguous [B*T*HW, C]')
        x = torch.empty((B, 1 + T * HW, Cc), dtype=torch.float32, device=t.device)
        p = MvitTokensFwdParams()
        p.t, p.wmask = t.data_ptr(), _ptr(None if wmask is None else _req(wmask, torch.float32, 'tokens.wmask').contiguous())
        for n, v in (('mask_token', mask_token), ('cls_token', cls_token), ('pos_s', pos_s), ('pos_t', pos_t), ('pos_cls', pos_cls)):
            setattr(p, n, _req(v, torch.float32, 'tokens.' + n).contiguous().data_ptr())
        p.x, p.B, p.T, p.HW, p.C = x.data_ptr(), B, T, HW, Cc
        _check(lib.vt_mvit_tokens_fwd(C.byref(p), _stream()), 'vt_mvit_tokens_fwd')
        return x

    def mvit_tokens_bwd(self, dx, wmask, B, T, HW):
        lib = load_library()
        dx = _req(dx, torch.float32, 'tokens_bwd.dx')
        if not dx.is_contiguous():
            raise RuntimeError('mvit_tokens_bwd: dx must be contiguous')
        Cc = dx.shape[-1]
        dt = torch.empty((B * T * HW, Cc), dtype=torch.bfloat16, device=dx.device)
        p = MvitTokensBwdParams()
        p.dx, p.wmask, p.dt = dx.data_ptr(), _ptr(wmask), dt.data_ptr()
        p.B, p.T, p.HW, p.C = B, T, HW, Cc
        _check(lib.vt_mvit_tokens_bwd(C.byref(p), _stream()), 'vt_mvit_tokens_bwd')
        return dt

    def mse_fwd(self, pred, target, mask, dims):
        """dims = (B, t, dt, h, w, dc) -> fp32 [4]; element 0 = sum_cells mask * mean_dc (pred-target)^2.
        fp64 targets (the reference's numpy arrays): differences and sums in fp64 -> fp64 [4]."""
        lib = load_library()
        f64 = target.dtype == torch.float64
        for tns, n in ((pred, 'pred'), (mask, 'mask')):
            _req(tns, torch.float32, 'mse.' + n)
        _req(target, torch.float64 if f64 else torch.float32, 'mse.target')
        for tns, n in ((pred, 'pred'), (target, 'target'), (mask, 'mask')):
            if not tns.is_contiguous():
                raise RuntimeError(f'mse_fwd: {n} must be contiguous')
        B, t, dt, h, w, dc = dims
        cells = B * t * dt * h * w
        if pred.numel() != B * (1 + t * h * w) * dt * dc or target.numel() != cells * dc or mask.numel() != cells:
            raise RuntimeError('mse_fwd: shape mismatch')
        num = torch.zeros(4, dtype=target.dtype, device=pred.device) if f64 else torch.empty(4, dtype=torch.float32, device=pred.device)
        partials = torch.empty(lib.vt_mse_blocks(cells) * 4, dtype=target.dtype, device=pred.device)
        p = MseFwdParams()
        p.pred, p.mask, p.partials = pred.data_ptr(), mask.data_ptr(), partials.data_ptr()
        if f64:
            p.target64, p.num64 = target.data_ptr(), num.data_ptr()
        else:
            p.target, p.num = target.data_ptr(), num.data_ptr()
        p.B, p.t, p.dt, p.h, p.w, p.dc = dims
        _check(lib.vt_mse_fwd(C.byref(p), _stream()), 'vt_mse_fwd')
        return num

    def mse_bwd(self, pred, target, mask, coef, dims):
        lib = load_library()
        B, t, dt, h, w, dc = dims
        dpred = torch.empty((B * (1 + t * h * w), dt * dc), dtype=torch.bfloat16, device=pred.device)
        p = MseBwdParams()
        p.pred, p.mask = pred.data_ptr(), mask.data_ptr()
        if target.dtype == torch.float64:
            p.target64 = target.data_ptr()
        else:
            p.target = _req(target, torch.float32, 'mse.target').data_ptr()
        p.coef, p.dpred = _req(coef, torch.float32, 'mse.coef').data_ptr(), dpred.data_ptr()
        p.B, p.t, p.dt, p.h, p.w, p.dc = dims
        _check(lib.vt_mse_bwd(C.byref(p), _stream()), 'vt_mse_bwd')
        return dpred


    # -- fused clip + optimizer (multi-tensor) ---------------------------------------------------
    def _opt_params(self, tbl, clip=0.0, **hp):
        p = OptParams()
        p.chunks, p.n_chunks, p.n_tensors = tbl['chunks'].data_ptr(), tbl['n_chunks'], tbl['n_tensors']
        p.pptr, p.gptr = tbl['pptr'].data_ptr(), tbl['gptr'].data_ptr()
        p.s1ptr, p.s2ptr = tbl['s1ptr'].data_ptr(), _ptr(tbl.get('s2ptr'))
        p.norm2, p.lr, p.wd = tbl['norm2'].data_ptr(), tbl['lr'].data_ptr(), tbl['wd'].data_ptr()
        p.clip = float(clip or 0.0)
        for k, v in hp.items():
            setattr(p, k, v)
        return p

    def opt_norm2(self, tbl):
        """tbl['norm2'][i] = sum(grad_i ** 2) for every tensor of the table (optim.TensorTable)"""
        _check(load_library().vt_opt_norm2(C.byref(self._opt_params(tbl)), _stream()), 'vt_opt_norm2')
        return tbl['norm2']

    def opt_sgd(self, tbl, clip, momentum, nesterov, first_step):
        p = self._opt_params(tbl, clip, momentum=momentum, nesterov=int(nesterov), first_step=int(first_step))
        _check(load_library().vt_opt_sgd(C.byref(p), _stream()), 'vt_opt_sgd')

    def opt_adamw(self, tbl, clip, beta1, beta2, eps, bc1, bc2):
        p = self._opt_params(tbl, clip, beta1=beta1, beta2=beta2, eps=eps, bc1=bc1, bc2=bc2)
        _check(load_library().vt_opt_adamw(C.byref(p), _stream()), 'vt_opt_adamw')


def set_reserved_sms(n: int) -> None:
    """Keep n SMs free of persistent GEMM CTAs (for overlapped NCCL kernels); see vt_set_reserved_sms."""
    _check(load_library().vt_set_reserved_sms(int(n)), 'vt_set_reserved_sms')


def launch_count() -> int:
    """Kernels launched by libvt_b200.so in this process so far."""
    return int(load_library().vt_launch_count())


K = CudaKernels()
