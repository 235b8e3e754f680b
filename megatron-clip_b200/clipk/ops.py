"""Host side of the fused contrastive loss: two torch.autograd.Functions over the clipk C ABI.

Data flow on rank r of W (b local rows, N = W*b), replacing open_CLIP/src/open_clip/loss.py:20-64, 104-140:

  forward   operand pass over the local rows (normalise / cast, statistics)      \
            T_all = all-gather of the text operand rows                           |  _FusedStep: ONE enqueue,
            row AND column statistics of S = s * I_loc @ T_all^T  [b x N]         |  clipk_step_forward; between
            from ONE sweep over the tiles (two exact sweeps when unsafe)          |  2..8 ranks every exchange is a
            all-gather of the [3, N] column statistics                            |  pull from peer-mapped memory
            lse_row[b], lse_col[N], loss, s * dloss/ds                            /  (PeerContext)
  backward  G = alpha*(P_row-Id) + beta*(P_col-Id) tile by tile; dI_loc = c G @ T_all;   clipk_step_backward: the tiles of
            dT_partial[N, d] = c G^T @ I_loc; dT_loc = sum over ranks of their parts     dT go straight to their owners

The general route (_GeneralRoute: fp32 / fp16 arithmetic, widths that are not multiples of 64, more than 8 ranks, no
symmetric memory) runs the same mathematics through the individual entries (clipk_fwd_both, clipk_finalize, clipk_bwd,
...) with NCCL all_gather_into_tensor / reduce_scatter_tensor between them.  fused_clip_loss picks the route.

The [b x N] logits are never written to HBM and I_all is never gathered.  All four (local_loss,
gather_with_grad) modes of the reference are coefficient choices of this one pipeline (SURVEY.md App. A).

The kernels are reached through `_backend()`: the CUDA library, or - in CPU unit tests of the collective
orchestration only - an object installed with `set_backend_for_testing`.  There is no CPU fallback in the
product: without libclipk.so or without a compute-capability-10.x device the call raises.
"""
from __future__ import annotations

import ctypes
import os
import warnings

import torch
import torch.distributed as dist

from . import _lib

_TEST_BACKEND = None
_FEATURE_DTYPES = (torch.bfloat16, torch.float16, torch.float32)
_K_BLOCK = 64           # K extent of one TMA box / MMA stage (BK in csrc/gemm_core.cuh)


def _round_up(x, m):
    return (x + m - 1) // m * m


def set_backend_for_testing(backend):
    """Install an object with the methods of CudaBackend, peer_context included (tests only; None restores CUDA)."""
    global _TEST_BACKEND
    _TEST_BACKEND = backend


def _ptr(t):
    return None if t is None else t.data_ptr()


class Operand:
    """A feature matrix in the layout the kernels consume (see include/clipk.h, CLIPK_BF16 / F16 / F16X2)."""
    __slots__ = ("data", "dtype", "ld", "inv_scale", "rows", "d", "scale_io", "amax")

    def __init__(self, data, dtype, ld, inv_scale, rows, d, scale_io=None):
        self.data, self.dtype, self.ld, self.inv_scale, self.rows, self.d = data, dtype, ld, inv_scale, rows, d
        self.scale_io = scale_io     # keeps the device scalar behind inv_scale alive
        self.amax = None             # device float: max |x|, when the forward sweep computed it on its way

    def inv_ptr(self):
        return None if self.inv_scale is None else self.inv_scale.data_ptr()


class DenseOperand:
    """A matrix as clipk_gemm16 consumes it: one bf16 plane, or the [hi, lo] fp16 planes of an fp32 matrix."""
    __slots__ = ("planes", "ld", "k", "f16", "rows", "keep")

    def __init__(self, planes, ld, k, f16, rows, keep=None):
        self.planes, self.ld, self.k, self.f16, self.rows, self.keep = planes, ld, k, f16, rows, keep


class CudaBackend:
    """Calls libclipk.so on the current CUDA stream."""

    def __init__(self):
        self.lib = _lib.load()

    @staticmethod
    def _stream():
        return torch.cuda.current_stream().cuda_stream

    def _to_f16(self, x: torch.Tensor, planes: int, amax=None) -> Operand:
        rows, d = x.shape
        dpad = (d + 63) // 64 * 64
        out = torch.empty(rows, planes * dpad, dtype=torch.float16, device=x.device)
        scale_io = torch.empty(2, dtype=torch.float32, device=x.device)
        src_dt = _lib.BF16 if x.dtype == torch.bfloat16 else _lib.F32
        if amax is not None:
            _lib.check(self.lib.clipk_to_f16_amax(x.data_ptr(), src_dt, rows, d, x.stride(0), out.data_ptr(), planes,
                                                  planes * dpad, scale_io.data_ptr(), amax.data_ptr(), self._stream()),
                       "clipk_to_f16_amax")
        else:
            _lib.check(self.lib.clipk_to_f16(x.data_ptr(), src_dt, rows, d, x.stride(0), out.data_ptr(), planes,
                                             planes * dpad, scale_io.data_ptr(), self._stream()), "clipk_to_f16")
        return Operand(out, _lib.F16 if planes == 1 else _lib.F16X2, planes * dpad, scale_io[1:2], rows, d, scale_io)

    def prepare(self, x: torch.Tensor) -> Operand:
        """Operand of the logits GEMM: bf16 as is; fp32 as two scaled fp16 planes (CLIPK_F16X2)."""
        if x.dtype == torch.bfloat16:
            x = x.contiguous()
            return Operand(x, _lib.BF16, x.stride(0), None, x.shape[0], x.shape[1])
        if x.dtype != torch.float32:
            raise TypeError(f"clipk: unsupported feature dtype {x.dtype} (bf16 and fp32 only)")
        return self._to_f16(x.contiguous(), 2)

    def prepare_grad(self, op: Operand) -> Operand:
        """Operand of the gradient GEMMs (fp16 x fp16): exact one-plane fp16 copy of bf16 features; the two-plane
        fp16 form of fp32 features is reused as is."""
        if op.dtype == _lib.BF16:
            return self._to_f16(op.data, 1, amax=op.amax)
        return op

    def fwd_stats(self, X: Operand, Y: Operand, scale, diag_offset, want_pos, out=None):
        """(max, sum, dot) per row of s * X @ Y^T, written into out[0..2] ([3, rows] fp32), plus the positive logit."""
        dev = X.data.device
        rows, cols, d = X.rows, Y.rows, X.d
        if out is None:
            out = torch.empty(3, rows, dtype=torch.float32, device=dev)
        pos = torch.zeros(rows, dtype=torch.float32, device=dev) if want_pos else None
        nbytes = self.lib.clipk_fwd_workspace_bytes(rows, cols, d, X.dtype)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(self.lib.clipk_fwd_stats(X.data.data_ptr(), Y.data.data_ptr(), rows, cols, d, X.ld, Y.ld, X.dtype,
                                            X.inv_ptr(), Y.inv_ptr(), scale.data_ptr(), diag_offset,
                                            out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), _ptr(pos),
                                            ws.data_ptr(), nbytes, self._stream()), "clipk_fwd_stats")
        return out, pos

    def fwd_both(self, X: Operand, Y: Operand, scale, diag_offset, col_out=None, exact=False):
        """(max, sum, dot) of every row AND every column of s * X @ Y^T in one call (one sweep over the tiles when the
        logits are provably bounded, see clipk_fwd_both): row_stats [3, rows], pos [rows], col_stats [3, cols]."""
        dev = X.data.device
        rows, cols, d = X.rows, Y.rows, X.d
        row_stats = torch.empty(3, rows, dtype=torch.float32, device=dev)
        if col_out is None:
            col_out = torch.empty(3, cols, dtype=torch.float32, device=dev)
        pos = torch.zeros(rows, dtype=torch.float32, device=dev)
        # the single-sweep path leaves max |x| of both operands here (the backward's fp16 scale needs it)
        want_amax = X.dtype == _lib.BF16
        amax = torch.empty(2, dtype=torch.float32, device=dev) if want_amax else None
        nbytes = self.lib.clipk_fwd_both_workspace_bytes(rows, cols, d, X.dtype)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(self.lib.clipk_fwd_both(X.data.data_ptr(), Y.data.data_ptr(), rows, cols, d, X.ld, Y.ld, X.dtype,
                                           X.inv_ptr(), Y.inv_ptr(), scale.data_ptr(), diag_offset,
                                           row_stats.data_ptr(), pos.data_ptr(), col_out.data_ptr(), _ptr(amax),
                                           1 if exact else 0, ws.data_ptr(), nbytes, self._stream()), "clipk_fwd_both")
        if want_amax:
            X.amax, Y.amax = amax[0:1], amax[1:2]
        return row_stats, pos, col_out

    def finalize(self, row_stats, pos, col_parts, diag_offset):
        """row_stats [3, rows]; col_parts [nparts, 3, cols] fp32 (max, sum, dot).
        Returns lse_row, lse_col, sums[4] = (CE row sum, CE col sum, dscale row sum, dscale col sum)."""
        dev = row_stats.device
        rows = row_stats.shape[1]
        nparts, _, cols = col_parts.shape
        lse_row = torch.empty(rows, dtype=torch.float32, device=dev)
        lse_col = torch.empty(cols, dtype=torch.float32, device=dev)
        sums = torch.empty(4, dtype=torch.float32, device=dev)
        cbase = col_parts.data_ptr()
        _lib.check(self.lib.clipk_finalize(row_stats[0].data_ptr(), row_stats[1].data_ptr(), row_stats[2].data_ptr(),
                                           pos.data_ptr(), rows, cbase, cbase + cols * 4, cbase + 2 * cols * 4, nparts,
                                           3 * cols, cols, diag_offset, lse_row.data_ptr(), lse_col.data_ptr(),
                                           sums.data_ptr(), self._stream()), "clipk_finalize")
        return lse_row, lse_col, sums

    def bwd(self, X: Operand, Y: Operand, Xg: Operand, Yg: Operand, scale, diag_offset, lse_row, lse_col, alpha,
            beta, gscale, want_dx, want_dy, split=False):
        """split: dX from alpha (P_row - Id) only, dY from beta (P_col - Id) only, one recompute (clipk_bwd)"""
        dev = X.data.device
        rows, cols, d = X.rows, Y.rows, X.d
        dX = torch.empty(rows, d, dtype=torch.float32, device=dev) if want_dx else None
        dY = torch.empty(cols, d, dtype=torch.float32, device=dev) if want_dy else None
        nbytes = self.lib.clipk_bwd_workspace_bytes(rows, cols, d, Xg.dtype)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(self.lib.clipk_bwd(X.data.data_ptr(), Y.data.data_ptr(), rows, cols, d, X.ld, Y.ld, X.dtype,
                                      X.inv_ptr(), Y.inv_ptr(), Xg.data.data_ptr(), Yg.data.data_ptr(), Xg.ld, Yg.ld,
                                      Xg.dtype, Xg.inv_ptr(), Yg.inv_ptr(), scale.data_ptr(), diag_offset,
                                      lse_row.data_ptr(), lse_col.data_ptr(), float(alpha), float(beta), 1 if split else 0,
                                      gscale.data_ptr(), _ptr(dX), _ptr(dY), ws.data_ptr(), nbytes, self._stream()),
                   "clipk_bwd")
        return dX, dY

    # ---- the whole step in two enqueues (clipk_step_forward / clipk_step_backward)
    def peer_context(self, b, d, rank, world, group):
        """PeerContext of the fused step on 2..8 ranks, or None: the general route takes the call (see _peer_context).
        On the current device, the one the library enqueues the step on."""
        return _peer_context(b, d, rank, world, group, torch.device("cuda", torch.cuda.current_device()))

    def _c_step(self, st: "StepDesc"):
        c = st.cstruct
        if c is None:
            c = st.cstruct = _lib.Step()
            c.rows, c.cols, c.d = st.rows, st.cols, st.d
            c.src_dtype = _lib.BF16 if st.image.dtype == torch.bfloat16 else _lib.F32
            c.normalize, c.eps = int(st.normalize), float(st.eps)
            c.image, c.text = st.image.data_ptr(), st.text.data_ptr()
            c.ld_image, c.ld_text = st.image.stride(0), st.text.stride(0)
            c.logit_scale = st.scale.data_ptr()
            c.loss_div, c.grad_coef, c.grad_split = float(st.loss_div), float(st.grad_coef), int(bool(st.grad_split))
            c.x_op, c.y_all = st.x_op.data_ptr(), st.y_all.data_ptr()
            c.inv_x, c.inv_y = _ptr(st.inv_x), _ptr(st.inv_y)
            c.stats, c.lse_row, c.lse_col, c.scal = (st.stats.data_ptr(), st.lse_row.data_ptr(), st.lse_col.data_ptr(),
                                                     st.scal.data_ptr())
            c.g16 = _ptr(st.g16)
            c.workspace, c.workspace_bytes = st.ws.data_ptr(), st.ws.numel()
        c.stream = self._stream()
        return c

    def step_workspace_bytes(self, rows, cols, d, world):
        c = _lib.Step()
        c.rows, c.cols, c.d = rows, cols, d
        peer = _lib.Peer()
        peer.world = world
        if world > 1:
            c.peer = ctypes.pointer(peer)
        return int(self.lib.clipk_step_workspace_bytes(ctypes.byref(c)))

    def step_forward(self, st: "StepDesc"):
        c = self._c_step(st)
        if st.peer is not None:
            st.cpeer = st.peer.begin_forward()
            c.peer = ctypes.pointer(st.cpeer)
        _lib.check(self.lib.clipk_step_forward(ctypes.byref(c)), "clipk_step_forward")

    def step_backward(self, st: "StepDesc"):
        c = self._c_step(st)
        c.grad_out = st.grad_out.data_ptr()
        c.d_image, c.d_text, c.d_scale = _ptr(st.d_image), _ptr(st.d_text), _ptr(st.d_scale)
        c.out_dtype = _lib.BF16 if st.out_dtype == torch.bfloat16 else _lib.F32
        if st.peer is not None:
            st.cpeer = st.peer.begin_backward()
            c.peer = ctypes.pointer(st.cpeer)
        _lib.check(self.lib.clipk_step_backward(ctypes.byref(c)), "clipk_step_backward")

    # ---- SigLipLoss (clipk_siglip_forward / clipk_siglip_backward, used by clipk/siglip.py)
    def _c_siglip(self, X, Y, scale, bias, diag_offset, state):
        c = _lib.Siglip()
        c.rows, c.d = X.shape
        c.cols = Y.shape[0]
        c.x, c.ldx, c.y, c.ldy = X.data_ptr(), X.stride(0), Y.data_ptr(), Y.stride(0)
        c.logit_scale, c.logit_bias = scale.data_ptr(), _ptr(bias)
        c.diag_offset, c.state = diag_offset, state.data_ptr()
        c.stream = self._stream()
        ws = torch.empty(self.lib.clipk_siglip_workspace_bytes(ctypes.byref(c)), dtype=torch.uint8, device=X.device)
        c.workspace, c.workspace_bytes = ws.data_ptr(), ws.numel()
        return c, ws

    def siglip_forward(self, X, Y, scale, bias, diag_offset):
        """X [b, d], Y [N, d] bf16 (d % 64 == 0, unit inner stride); scale / bias: [1] fp32 device scalars (bias may be
        None).  Returns (loss as a 0-dim view, state): the state carries what the backward needs."""
        state = torch.zeros(_lib.SIGLIP_STATE_WORDS, dtype=torch.float32, device=X.device)
        c, ws = self._c_siglip(X, Y, scale, bias, diag_offset, state)
        _lib.check(self.lib.clipk_siglip_forward(ctypes.byref(c)), "clipk_siglip_forward")
        return state[0], state

    def siglip_backward(self, X, Y, scale, bias, diag_offset, state, grad_out, want_dx, want_dy, want_ds, want_dt):
        """fp32 (d_x [b, d], d_y [N, d], d_scale [1], d_bias [1]); None where not wanted.  d_y is this rank's partial of
        the gathered text gradient."""
        dev = X.device
        dX = torch.empty(X.shape, dtype=torch.float32, device=dev) if want_dx else None
        dY = torch.empty(Y.shape, dtype=torch.float32, device=dev) if want_dy else None
        ds = torch.empty(1, dtype=torch.float32, device=dev) if want_ds else None
        dt = torch.empty(1, dtype=torch.float32, device=dev) if want_dt else None
        c, ws = self._c_siglip(X, Y, scale, bias, diag_offset, state)
        c.grad_out = grad_out.data_ptr()
        c.d_x, c.d_y, c.d_scale, c.d_bias = _ptr(dX), _ptr(dY), _ptr(ds), _ptr(dt)
        _lib.check(self.lib.clipk_siglip_backward(ctypes.byref(c)), "clipk_siglip_backward")
        return dX, dY, ds, dt

    def normalize_fwd(self, x: torch.Tensor, eps: float):
        """y = x / max(|x|, eps) row-wise (same dtype), and the fp32 factors 1 / max(|x|, eps)."""
        if x.dtype not in (torch.bfloat16, torch.float32):
            raise TypeError(f"clipk: unsupported feature dtype {x.dtype} (bf16 and fp32 only)")
        x = x.contiguous()
        rows, d = x.shape
        y = torch.empty_like(x)
        inv = torch.empty(rows, dtype=torch.float32, device=x.device)
        dt = _lib.BF16 if x.dtype == torch.bfloat16 else _lib.F32
        _lib.check(self.lib.clipk_normalize_fwd(x.data_ptr(), dt, rows, d, x.stride(0), y.data_ptr(), y.stride(0),
                                                inv.data_ptr(), float(eps), self._stream()), "clipk_normalize_fwd")
        return y, inv

    def normalize_bwd(self, g: torch.Tensor, y: torch.Tensor, inv: torch.Tensor, eps: float):
        g = g.contiguous()
        rows, d = y.shape
        dx = torch.empty_like(y)
        dt = _lib.BF16 if y.dtype == torch.bfloat16 else _lib.F32
        _lib.check(self.lib.clipk_normalize_bwd(g.data_ptr(), g.stride(0), y.data_ptr(), y.stride(0), inv.data_ptr(), dt,
                                                rows, d, dx.data_ptr(), dx.stride(0), float(eps), self._stream()),
                   "clipk_normalize_bwd")
        return dx

    # ---- evaluation side: dense logits panels and target ranks (clipk/metrics.py)
    def dense_operand(self, x: torch.Tensor) -> "DenseOperand":
        """Operand of clipk_gemm16: bf16 as is (K zero-padded to whole 64-element blocks); fp32 / fp16 as two scaled
        fp16 planes [hi | lo] (clipk_to_f16), contracted pair by pair like the loss's fp32 path."""
        if x.dim() != 2 or x.shape[0] == 0 or x.shape[1] == 0:
            raise ValueError("clipk: expected a non-empty [rows, dim] matrix")
        if x.dtype == torch.bfloat16:
            k = _round_up(x.shape[1], _K_BLOCK)
            x = torch.nn.functional.pad(x, (0, k - x.shape[1])) if k != x.shape[1] else x.contiguous()
            return DenseOperand([x], x.stride(0), k, 0, x.shape[0])
        if x.dtype not in (torch.float32, torch.float16):
            raise TypeError(f"clipk: unsupported feature dtype {x.dtype} (bf16, fp16 and fp32 only)")
        op = self._to_f16(x.float().contiguous(), 2)
        k = op.ld // 2
        return DenseOperand([op.data[:, :k], op.data[:, k:]], op.ld, k, 1, x.shape[0], keep=op)

    def logits_panel(self, Q: "DenseOperand", K: "DenseOperand", r0: int, nrows: int, out: torch.Tensor):
        """out[:nrows, :] = Q[r0:r0+nrows] @ K^T (fp32; up to the operands' positive power-of-two scales).  out is
        [>= nrows, round_up(K.rows, 4)] fp32, contiguous."""
        if Q.f16 != K.f16 or Q.k != K.k:
            raise TypeError("clipk: both operands of a logits panel must have the same dtype and width")
        n4 = out.shape[1]
        pairs = [(0, 0)] if Q.f16 == 0 else [(1, 0), (0, 1), (0, 0)]      # small products first: lo.hi, hi.lo, hi.hi
        for i, (pq, pk) in enumerate(pairs):
            a = Q.planes[pq][r0:r0 + nrows]
            _lib.check(self.lib.clipk_gemm16(a.data_ptr(), K.planes[pk].data_ptr(), out.data_ptr(), nrows, n4, Q.k, Q.ld,
                                             K.ld, out.stride(0), 0, 0, Q.f16, 1 if i else 0, self._stream()),
                       "clipk_gemm16")

    def rank_count(self, S: torch.Tensor, nrows: int, cols: int, target, diag_offset: int, row0: int, greater, ties):
        _lib.check(self.lib.clipk_rank_count(S.data_ptr(), nrows, cols, S.stride(0), _ptr(target), diag_offset, row0,
                                             greater.data_ptr(), ties.data_ptr(), self._stream()), "clipk_rank_count")

    # ---- distillation term on logits panels (clipk/distill.py)
    def gemm(self, A: torch.Tensor, B: torch.Tensor, out: torch.Tensor, a_mn: bool, b_mn: bool, f16: bool,
             accumulate: bool):
        """out[M, N] (fp32) (+)= A * B^T on the tensor cores.  A is [M, K] (a_mn False) or stored [K, M] (True); B is
        [N, K] or stored [K, N]; 16-bit operands of one format (fp16 when f16).  Rows may be strided views."""
        M, N = out.shape
        K = A.shape[0] if a_mn else A.shape[1]
        _lib.check(self.lib.clipk_gemm16(A.data_ptr(), B.data_ptr(), out.data_ptr(), M, N, K, A.stride(0), B.stride(0),
                                         out.stride(0), 1 if a_mn else 0, 1 if b_mn else 0, 1 if f16 else 0,
                                         1 if accumulate else 0, self._stream()), "clipk_gemm16")

    def distill_cross(self, S, T, nrows, cols, s_mul, t_mul, t_lse_row, t_lse_col, row0, row_cross, col_part):
        _lib.check(self.lib.clipk_distill_cross(S.data_ptr(), T.data_ptr(), nrows, cols, S.stride(0), s_mul.data_ptr(),
                                                t_mul.data_ptr(), t_lse_row.data_ptr(), t_lse_col.data_ptr(), row0,
                                                row_cross.data_ptr(), col_part.data_ptr(), self._stream()),
                   "clipk_distill_cross")

    def distill_grad(self, S, T, nrows, cols, s_mul, t_mul, s_lse_row, t_lse_row, s_lse_col, t_lse_col, row0, G):
        _lib.check(self.lib.clipk_distill_grad(S.data_ptr(), T.data_ptr(), nrows, cols, S.stride(0), s_mul.data_ptr(),
                                               t_mul.data_ptr(), s_lse_row.data_ptr(), t_lse_row.data_ptr(),
                                               s_lse_col.data_ptr(), t_lse_col.data_ptr(), row0, G.data_ptr(),
                                               G.stride(0), self._stream()), "clipk_distill_grad")

    def grad_operand(self, x: torch.Tensor):
        """(fp16 copy [rows, round_up(d, 64)], inv_scale device scalar) of a bf16 matrix: exact, for the gradient GEMMs."""
        op = self._to_f16(x.contiguous(), 1)
        return op.data, op.inv_scale

    def cast(self, src: torch.Tensor, dtype: torch.dtype):
        if dtype == torch.float32:
            return src
        out = torch.empty(src.shape, dtype=dtype, device=src.device)
        _lib.check(self.lib.clipk_cast(src.data_ptr(), out.data_ptr(), src.numel(), _lib.BF16, self._stream()),
                   "clipk_cast")
        return out


_CUDA_BACKEND = None


def _backend():
    global _CUDA_BACKEND
    if _TEST_BACKEND is not None:
        return _TEST_BACKEND
    if _CUDA_BACKEND is None:
        _CUDA_BACKEND = CudaBackend()
    return _CUDA_BACKEND


def gpu_launches() -> int:
    """Number of clipk kernels launched so far in this process."""
    return 0 if _CUDA_BACKEND is None else int(_CUDA_BACKEND.lib.clipk_launch_count())


# ----------------------------------------------------------------------------------------------------- the fused step
class StepDesc:
    """Everything one loss evaluation holds between its forward and its backward (mirrors struct clipk_step)."""
    __slots__ = ("rows", "cols", "d", "world", "rank", "normalize", "eps", "image", "text", "scale", "loss_div",
                 "grad_coef", "grad_split", "x_op", "y_all", "inv_x", "inv_y", "stats", "lse_row", "lse_col", "scal", "g16", "ws",
                 "peer",
                 "grad_out", "d_image", "d_text", "d_scale", "out_dtype", "cstruct", "cpeer", "group")

    def __init__(self):
        for k in self.__slots__:
            setattr(self, k, None)


def _align(n, a=256):
    return (n + a - 1) // a * a


class PeerContext:
    """Peer-mapped (symmetric) memory of one (local batch, width, group) between the ranks of one NVLink domain.  All of
    it is double-buffered by call parity (a buffer is rewritten two calls after it was read, see peer_allgather_kernel):

      text_src  [2][b, d] bf16     this rank's text operand rows, pulled by every peer (gather_features, loss.py:20-64)
      stats_src [2][8] fp32        its operand statistics, pulled with them
      col_src   [2][3, N] fp32     column statistics of this rank's block, pulled by every peer
      slots     [2][W][b, d] fp32  slot w is written over NVLink by the gradient GEMM of rank w (the reduce-scatter of
                                   the text gradient, i.e. the backward of loss.py:50-51)
      flags     [3][8] uint32      one epoch word per peer and purpose (gather, statistics, gradient)
    """

    def __init__(self, b, d, rank, world, group, dev):
        import torch.distributed._symmetric_memory as symm     # not importable on builds without CUDA support
        pg = group if group is not None else dist.group.WORLD
        N = world * b
        sizes = [("text", 2 * _align(b * d * 2)), ("stats", 2 * 256), ("col", 2 * _align(3 * N * 4)),
                 ("slots", 2 * world * b * d * 4), ("flags", 256)]
        self.off, total = {}, 0
        for name, nbytes in sizes:
            self.off[name] = total
            total += _align(nbytes)
        self.buf = symm.empty(total, dtype=torch.uint8, device=dev)
        self.buf[self.off["flags"]:self.off["flags"] + 256].zero_()
        h = symm.rendezvous(self.buf, pg)
        if h.rank != rank or h.world_size != world:
            raise RuntimeError("rank / world_size of the loss do not match the process group")
        self.rank, self.world, self.b, self.d, self.N = rank, world, b, d, N
        self.bases = [int(p) for p in h.buffer_ptrs]
        self._handle = h
        self.n_fwd = self.n_bwd = 0
        # time-outs of the peer waits land here (pinned host memory, written by the kernels, read before every call)
        self.err = torch.zeros(4, dtype=torch.int32).pin_memory()
        torch.cuda.synchronize(dev)
        dist.barrier(group=pg)          # every rank's flags are zero before anyone signals

    def _check(self):
        code = int(self.err[0])
        if code:
            raise RuntimeError(f"clipk: a wait on a peer rank timed out (code {code}): a rank died or skipped a "
                               "collective call of the loss")

    def _fill(self, half_f, half_b):
        b, d, N, W = self.b, self.d, self.N, self.world
        p = _lib.Peer()
        p.world, p.rank = W, self.rank
        o = self.off
        for r in range(W):
            base = self.bases[r]
            p.text_src[r] = base + o["text"] + half_f * _align(b * d * 2)
            p.stats_src[r] = base + o["stats"] + half_f * 256
            p.col_src[r] = base + o["col"] + half_f * _align(3 * N * 4)
            p.grad_slot[r] = base + o["slots"] + (half_b * W + self.rank) * b * d * 4
            p.flags_gather[r] = base + o["flags"]
            p.flags_stats[r] = base + o["flags"] + 32
            p.flags_grad[r] = base + o["flags"] + 64
        p.my_slots = self.bases[self.rank] + o["slots"] + half_b * W * b * d * 4
        p.err = self.err.data_ptr()
        return p

    def begin_forward(self):
        self._check()
        self.n_fwd += 1
        p = self._fill(self.n_fwd & 1, 0)
        p.epoch_gather = p.epoch_stats = self.n_fwd & 0xffffffff
        return p

    def begin_backward(self):
        self._check()
        self.n_bwd += 1
        p = self._fill(0, self.n_bwd & 1)
        p.epoch_grad = self.n_bwd & 0xffffffff
        return p


_PEER_CONTEXTS = {}
_PEER_DISABLED = [False]
_MAX_PEER_CONTEXTS = 4      # shapes (train batch, eval batch, ...) that get symmetric buffers; more fall back to NCCL


def _peer_context(b, d, rank, world, group, dev):
    """PeerContext for this shape, or None when the collectives go through NCCL instead (CLIPK_PEER=0, no symmetric
    memory on this system, more than 8 ranks, a local batch that is not a multiple of 128)."""
    if _PEER_DISABLED[0] or os.environ.get("CLIPK_PEER", "1") == "0":
        return None
    if dev.type != "cuda" or world < 2 or world > _lib.MAX_PEERS or b % 128 != 0:
        return None
    key = (b, d, rank, world, id(group), dev.index)
    ctx = _PEER_CONTEXTS.get(key)
    if ctx is None:
        if len(_PEER_CONTEXTS) >= _MAX_PEER_CONTEXTS:
            return None
        err = None
        try:
            import torch.distributed._symmetric_memory  # noqa: F401
            ok_local = 1
        except Exception as e:          # no symmetric memory in this build
            ok_local, err = 0, e
        # all ranks take the same path: agree BEFORE the collective allocation, so that a rank that cannot even import
        # the module sends everyone to NCCL instead of leaving the others inside the rendezvous
        ok = torch.tensor([ok_local], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if int(ok.item()) == 1:
            try:
                ctx = PeerContext(b, d, rank, world, group, dev)
            except Exception as e:
                ctx, err = None, e
            ok = torch.tensor([0 if ctx is None else 1], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if int(ok.item()) == 0:
            warnings.warn(f"clipk: peer-memory collectives unavailable ({err!r}); using NCCL")
            _PEER_DISABLED[0] = True
            return None
        _PEER_CONTEXTS[key] = ctx
    return ctx


_WORKSPACES = {}
_LAST_STEP_STATS = [None]


def last_forward_was_single_sweep():
    """True / False for the most recent fused-step forward of this process (None before the first one): whether the
    kernels took the single sweep or the exact two-sweep form (decided on the device, see fwd_bound in gemm_core.cuh).
    Synchronises; for tests and bench.py only."""
    st = _LAST_STEP_STATS[0]
    if st is None:
        return None
    return bool(st.view(-1, _lib.STAT_WORDS)[:, 5].max().item() > 0.5)


def _step_workspace(be, rows, cols, d, world, dev):
    """Scratch of the fused step, shared by all calls of one shape on one stream (consumed inside each enqueue)."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else 0, rows, cols, d, world)
    ws = _WORKSPACES.get(key)
    if ws is None:
        if len(_WORKSPACES) >= 8:
            _WORKSPACES.clear()
        ws = _WORKSPACES[key] = torch.empty(be.step_workspace_bytes(rows, cols, d, world), dtype=torch.uint8, device=dev)
        ws[:256].zero_()        # the operand pass's ticket: zero at creation, returned to zero by every forward
    return ws


# ----------------------------------------------------------------------------------------------------- collectives
def _all_gather_rows(x: torch.Tensor, world_size: int, group=None) -> torch.Tensor:
    """[n, ...] per rank -> [world*n, ...], rank-major, into one contiguous buffer (no list + cat copy)."""
    out = torch.empty((world_size * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x.contiguous(), group=group)
    return out


def _reduce_scatter_rows(x: torch.Tensor, world_size: int, group=None) -> torch.Tensor:
    """[world*n, ...] per rank -> SUM over ranks of chunk `rank`, [n, ...]."""
    n = x.shape[0] // world_size
    out = torch.empty((n,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.reduce_scatter_tensor(out, x.contiguous(), op=dist.ReduceOp.SUM, group=group)
    return out


class _GatherRowsWithGrad(torch.autograd.Function):
    """all-gather whose backward is a reduce-scatter SUM (what torch.distributed.nn.all_gather does on NCCL)."""

    @staticmethod
    def forward(ctx, x, world_size, group):
        ctx.world_size, ctx.group = world_size, group
        return _all_gather_rows(x, world_size, group)

    @staticmethod
    def backward(ctx, g):
        return _reduce_scatter_rows(g, ctx.world_size, ctx.group), None, None


# ----------------------------------------------------------------------------------------------------- autograd
def _autocast_bf16(dev):
    return dev.type == "cuda" and torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16


def _row_layout_ok(x):
    """rows 16-byte aligned with unit inner stride: what prep_kernel reads in place"""
    es = x.element_size()
    return x.stride(1) == 1 and (x.stride(0) * es) % 16 == 0 and x.stride(0) >= x.shape[1] and x.data_ptr() % 16 == 0


def _kernel_features(x):
    """Contiguous features as the individual entries take them.  fp16 features (open_clip --precision fp16 / amp) become
    fp32: every fp16 value is an fp32 value, so they take the split-precision fp32 path unchanged.  The kernels stream K
    in 64-element blocks from 16-byte aligned rows, so other widths are zero-padded to the next multiple of 64: zero
    columns change no logit, and _caller_grad drops their gradient columns."""
    if x.dtype == torch.float16:
        x = x.float()
    d = _round_up(x.shape[1], _K_BLOCK)
    return x.contiguous() if d == x.shape[1] else torch.nn.functional.pad(x, (0, d - x.shape[1]))


def _caller_grad(be, g, d_in, in_dtype):
    """The fp32 gradient of a _kernel_features operand in the caller's width and dtype: the padding's columns dropped,
    cast by the kernels (clipk_cast writes bf16 or fp32), fp16 rounded from fp32 at the end."""
    if g.shape[1] != d_in:
        g = g[:, :d_in].contiguous()
    g = be.cast(g, torch.bfloat16 if in_dtype == torch.bfloat16 else torch.float32)
    return g if g.dtype == in_dtype else g.to(in_dtype)


def _mode_coefficients(b, world, local_loss, gather_with_grad):
    """(loss_div, grad_coef, grad_split) of a (local_loss, gather_with_grad) mode, SURVEY App. A: the loss divides by 2b
    on one rank and in the local modes, else by 2N; c = 1/(2b) there and for global+gather_with_grad, else 1/(2N).
    Split, loss.py:53-56 with local_loss: the gathered tensors carry no gradient, so dI sees only the image->text softmax
    and dT only the text->image one."""
    N = world * b
    local = world == 1 or local_loss
    loss_div = 2.0 * b if local else 2.0 * N
    grad_coef = 1.0 / (2.0 * b) if (local or gather_with_grad) else 1.0 / (2.0 * N)
    return loss_div, grad_coef, world > 1 and bool(local_loss) and not gather_with_grad


class _FusedStep(torch.autograd.Function):
    """The fused step: clipk_step_forward / clipk_step_backward, one enqueue per pass, on bf16 operands of a width that
    is a multiple of 64.  On 2..8 ranks every exchange is a pull from the peer-mapped memory of `peer` (PeerContext).
    With `normalize` the operand pass L2-normalises the features and the gradient pass applies the Jacobian."""

    @staticmethod
    def forward(ctx, image_features, text_features, logit_scale, local_loss, gather_with_grad, rank, world_size, group,
                peer, normalize, eps):
        be = _backend()
        b, d = image_features.shape
        W = int(world_size)
        N = W * b
        dev = image_features.device
        in_dtype = image_features.dtype
        want_feat = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        img, txt = image_features.detach(), text_features.detach()
        if not _row_layout_ok(img):
            img = img.contiguous()
        if not _row_layout_ok(txt):
            txt = txt.contiguous()
        st = StepDesc()
        st.rows, st.cols, st.d, st.world, st.rank, st.group = b, N, d, W, rank, group
        st.normalize, st.eps = bool(normalize), float(eps)
        st.image, st.text = img, txt
        st.scale = logit_scale.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        st.loss_div, st.grad_coef, st.grad_split = _mode_coefficients(b, W, local_loss, gather_with_grad)
        produced = st.normalize or in_dtype != torch.bfloat16
        # one fp32 allocation for everything the backward reads: lse_row | lse_col | scalars | statistics | inv norms
        n_f = b + N + 16 + _lib.STAT_WORDS * W + (2 * b if st.normalize else 0)
        fbuf = torch.empty(n_f, dtype=torch.float32, device=dev)
        st.lse_row, st.lse_col = fbuf[:b], fbuf[b:b + N]
        st.scal = fbuf[b + N:b + N + 16]
        o = b + N + 16
        st.stats = fbuf[o:o + _lib.STAT_WORDS * W]
        o += _lib.STAT_WORDS * W
        if st.normalize:
            st.inv_x, st.inv_y = fbuf[o:o + b], fbuf[o + b:o + 2 * b]
            o += 2 * b
        if want_feat and W > 1:
            # fp16 copies of the operands for the gradient GEMMs: made in the forward, under the wait for the
            # peers' column statistics
            st.g16 = torch.empty((b + N) * d * 2 + 256, dtype=torch.uint8, device=dev)
        st.x_op = torch.empty(b, d, dtype=torch.bfloat16, device=dev) if produced else img
        st.y_all = torch.empty(N, d, dtype=torch.bfloat16, device=dev) if (produced or W > 1) else txt
        st.ws = _step_workspace(be, b, N, d, W, dev)
        st.peer = peer
        be.step_forward(st)
        _LAST_STEP_STATS[0] = st.stats       # tests / bench: word 5 of a rank's row tells which forward ran
        pair = st.scal[4:6]
        if W > 1 and not local_loss:
            # the global (local_loss=False) loss is the same N x N problem on every rank: sum of the ranks' parts
            dist.all_reduce(pair, op=dist.ReduceOp.SUM, group=group)
        ctx.step = st
        ctx.in_dtype = in_dtype
        ctx.scale_dtype, ctx.scale_shape = logit_scale.dtype, logit_scale.shape
        # the inputs themselves are saved so that autograd notices an in-place change before the backward reads them
        ctx.save_for_backward(image_features, text_features)
        # a 0-dim view into this evaluation's own state tensor (nothing else reads that word again): no copy kernel
        return st.scal[4]

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        _ = ctx.saved_tensors            # raises if the features were modified in place since the forward
        st = ctx.step
        dev = st.scale.device
        want_feat = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        want_scale = ctx.needs_input_grad[2]
        st.grad_out = grad_out.detach().to(torch.float32).reshape(1).contiguous()
        st.out_dtype = torch.bfloat16 if ctx.in_dtype == torch.bfloat16 else torch.float32
        if want_feat:
            st.d_image = torch.empty(st.rows, st.d, dtype=st.out_dtype, device=dev)
            st.d_text = torch.empty(st.rows, st.d, dtype=st.out_dtype, device=dev)
        st.d_scale = torch.empty(1, dtype=torch.float32, device=dev) if want_scale else None
        if want_feat or want_scale or st.peer is not None:      # with peers every rank takes part in the barrier
            _backend().step_backward(st)
        d_scale = st.d_scale.reshape(ctx.scale_shape).to(ctx.scale_dtype) if want_scale else None
        ctx.step = None
        return st.d_image, st.d_text, d_scale, None, None, None, None, None, None, None, None


class _GeneralRoute(torch.autograd.Function):
    """Every call the fused step does not take: the individual kernel entries (clipk_fwd_both, clipk_finalize,
    clipk_bwd, ...) with NCCL all_gather_into_tensor / reduce_scatter_tensor between them."""

    @staticmethod
    def forward(ctx, image_features, text_features, logit_scale, local_loss, gather_with_grad, rank, world_size, group):
        be = _backend()
        b, d_in = image_features.shape
        W = int(world_size)
        N = W * b
        dev = image_features.device
        in_dtype = image_features.dtype
        scale = logit_scale.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        feats_i, feats_t = image_features.detach(), text_features.detach()
        # under torch.autocast the reference's matmuls run in the autocast dtype (SURVEY App. B)
        if in_dtype == torch.float32 and _autocast_bf16(dev):
            feats_i, feats_t = feats_i.to(torch.bfloat16), feats_t.to(torch.bfloat16)
        feats_i, feats_t = _kernel_features(feats_i), _kernel_features(feats_t)

        t_all = _all_gather_rows(feats_t, W, group) if W > 1 else feats_t
        X = be.prepare(feats_i)
        Y = be.prepare(t_all)
        off = rank * b if W > 1 else 0

        parts = torch.empty(1, 3, N, dtype=torch.float32, device=dev)        # (max, sum, dot) of every column
        row_stats, pos, _ = be.fwd_both(X, Y, scale, off, col_out=parts[0])
        if W > 1:
            parts = _all_gather_rows(parts, W, group)                        # [W, 3, N]
        lse_row, lse_col, sums = be.finalize(row_stats, pos, parts, off)

        # sums[0:2] -> loss, sums[2:4] -> s * dloss/ds; the global (local_loss=False) loss is the same N x N problem
        # on every rank, so both are all-reduced there.  dlogit_scale is never reduced by the loss in local mode
        # (DDP averages it later), exactly like the reference.
        loss_div, grad_coef, grad_split = _mode_coefficients(b, W, local_loss, gather_with_grad)
        pair = sums.view(2, 2).sum(dim=1)
        if W > 1 and not local_loss:
            dist.all_reduce(pair, op=dist.ReduceOp.SUM, group=group)
        pair = pair / loss_div

        ctx.save_for_backward(image_features, text_features, scale, lse_row, lse_col, pair)
        ctx.operands = (X, Y)
        ctx.cfg = (W, off, grad_coef, grad_split, group, in_dtype, d_in, logit_scale.dtype, logit_scale.shape)
        return pair[0].clone()

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        be = _backend()
        go = grad_out.detach().to(torch.float32).reshape(1)
        _, _, scale, lse_row, lse_col, pair = ctx.saved_tensors
        X, Y = ctx.operands
        W, off, grad_coef, grad_split, group, in_dtype, d_in, scale_dtype, scale_shape = ctx.cfg
        d_image = d_text = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            Xg, Yg = be.prepare_grad(X), be.prepare_grad(Y)
            gscale = (go * grad_coef).contiguous()
            if grad_split:
                # the two softmax parts in two planes of the panel of one recompute (one-plane operands), else (fp32
                # arithmetic: the planes are taken by [hi | lo]) two passes
                if Xg.dtype == _lib.F16 or _TEST_BACKEND is not None:
                    dX, dY = be.bwd(X, Y, Xg, Yg, scale, off, lse_row, lse_col, 1.0, 1.0, gscale, True, True, split=True)
                else:
                    dX, _ = be.bwd(X, Y, Xg, Yg, scale, off, lse_row, lse_col, 1.0, 0.0, gscale, True, False)
                    _, dY = be.bwd(X, Y, Xg, Yg, scale, off, lse_row, lse_col, 0.0, 1.0, gscale, False, True)
                dT = _reduce_scatter_rows(dY, W, group)
            else:
                dX, dY = be.bwd(X, Y, Xg, Yg, scale, off, lse_row, lse_col, 1.0, 1.0, gscale, True, True)
                dT = _reduce_scatter_rows(dY, W, group) if W > 1 else dY
            d_image, d_text = _caller_grad(be, dX, d_in, in_dtype), _caller_grad(be, dT, d_in, in_dtype)

        d_scale = None
        if ctx.needs_input_grad[2]:
            # pair[1] = s * dloss/ds, already normalised (and all-reduced in global mode) by the forward
            d_scale = (pair[1] * go[0] / scale[0]).reshape(scale_shape).to(scale_dtype)
        return d_image, d_text, d_scale, None, None, None, None, None


class _Normalize(torch.autograd.Function):
    """F.normalize(x, dim=-1) (open_clip/model.py:216,231) with its Jacobian, on the clipk kernels."""

    @staticmethod
    def forward(ctx, x, eps):
        y, inv = _backend().normalize_fwd(x.detach(), eps)
        ctx.save_for_backward(y, inv)
        ctx.eps = eps
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        y, inv = ctx.saved_tensors
        return _backend().normalize_bwd(g.to(y.dtype), y, inv, ctx.eps), None


def fused_clip_loss(image_features, text_features, logit_scale, local_loss=False, gather_with_grad=False, rank=0,
                    world_size=1, group=None, normalize=False, eps=1e-12):
    """loss = ClipLoss(local_loss, gather_with_grad, rank, world_size).forward(I, T, s)   (loss.py:123-140), of the
    L2-normalised features when `normalize`.  Picks the route once, before anything is launched: the fused step for bf16
    operands (bf16 features, or fp32 under bf16 autocast) with d % 64 == 0 on one GPU, or on several ranks when the
    backend has a peer context for them (see _peer_context); the general route for everything else."""
    if image_features.dim() != 2 or image_features.shape != text_features.shape:
        raise ValueError("image_features and text_features must both be [batch, dim]")
    if image_features.dtype != text_features.dtype:
        raise TypeError("image_features and text_features must have the same dtype")
    dtype, dev = image_features.dtype, image_features.device
    if dtype not in _FEATURE_DTYPES:
        raise TypeError(f"clipk: unsupported feature dtype {dtype} (bf16, fp16 and fp32 only)")
    if not isinstance(logit_scale, torch.Tensor):
        logit_scale = torch.tensor(float(logit_scale), dtype=torch.float32, device=dev)
    b, d = image_features.shape
    if b == 0:
        # empty batch: the reference's cross-entropy means over zero rows, i.e. NaN with empty gradients
        # (loss.py:135-138); nothing to launch
        return (image_features.sum() + text_features.sum()).float() * logit_scale.float() * float("nan")
    W = int(world_size)
    mode = (local_loss, gather_with_grad, rank, W, group)
    bf16_operands = dtype == torch.bfloat16 or (dtype == torch.float32 and _autocast_bf16(dev))
    if bf16_operands and d % _K_BLOCK == 0 and (dev.type == "cuda" or _TEST_BACKEND is not None):
        peer = _backend().peer_context(b, d, rank, W, group) if W > 1 else None
        if W == 1 or peer is not None:
            return _FusedStep.apply(image_features, text_features, logit_scale, *mode, peer, normalize, eps)
    if normalize:
        image_features, text_features = _Normalize.apply(image_features, eps), _Normalize.apply(text_features, eps)
    return _GeneralRoute.apply(image_features, text_features, logit_scale, *mode)


def fused_normalize_clip_loss(raw_image_features, raw_text_features, logit_scale, local_loss=False,
                              gather_with_grad=False, rank=0, world_size=1, group=None, eps=1e-12):
    """ClipLoss of the L2-normalised embeddings, taking the RAW tower outputs: what `model.py:216,231` followed by
    `loss.py:123-140` computes, with gradients with respect to the raw embeddings.  Opt-in - the drop-in ClipLoss does
    not normalise, exactly like the reference's (SURVEY.md section 0, point 2).

    On the fused step the normalisation lives in the load path: the pass that produces the operands (prep_kernel)
    normalises, rounds to bf16 and takes the statistics in one sweep over the rows, and the pass that casts the gradients
    (finish_grad_kernel) applies the Jacobian - no standalone normalise / cast / norm kernels.  The general route
    composes the row-wise kernels of clipk_normalize_fwd / _bwd with the loss."""
    return fused_clip_loss(raw_image_features, raw_text_features, logit_scale, local_loss, gather_with_grad, rank,
                           world_size, group, normalize=True, eps=eps)
