"""Tensor-level wrappers over the C ABI (include/ibm_b200.h).

PyTorch is used here only for device memory and streams: every function takes CUDA tensors,
passes raw device pointers + sizes + the current stream to libibm_b200.so, and returns.  No
function falls back to a torch implementation.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import ACT, BF16, F32, call

_ws_cache = {}


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.IbmError("inferbiomechanics_b200 kernels need CUDA tensors (no CPU fallback)")


def workspace(device) -> torch.Tensor:
    dev = torch.device(device)
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    if key not in _ws_cache:
        _ws_cache[key] = torch.zeros(_lib.load().ibm_workspace_bytes(), dtype=torch.uint8, device=dev)
    return _ws_cache[key]


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def pack_channel_major(srcs, T, emb, out_bf16):
    """srcs: contiguous fp32 CUDA tensors (B, C_i, T); emb fp32 [>=T, E] or None; out bf16 [B*T, ld]."""
    n = len(srcs)
    B = srcs[0].shape[0]
    ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in srcs])
    chans = (ctypes.c_int32 * n)(*[t.shape[1] for t in srcs])
    call("ibm_pack_channel_major", ptrs, chans, n, B, T, _p(emb), 0 if emb is None else emb.shape[1], _p(out_bf16), out_bf16.stride(0),
         stream_ptr())


def expand_rows_bf16(src_bf16, C, T, emb, out_bf16, v_out=None, v_col0=0):
    """src bf16 [B*T, ld_src] frame-major rows (pre-packed on the host) -> out bf16 [B*T, ld] with the temporal embedding appended."""
    n_rows = out_bf16.shape[0]
    call("ibm_expand_rows_bf16", _p(src_bf16), src_bf16.stride(0), C, n_rows, T, _p(emb), 0 if emb is None else emb.shape[1],
         _p(out_bf16), out_bf16.stride(0), _p(v_out), v_col0, stream_ptr())


# ---- GEMM ---------------------------------------------------------------------------------------
def gemm(A: torch.Tensor, B: torch.Tensor, out: torch.Tensor, M: int, N: int, K: int, *, lda=None, ldb=None, ldd=None,
         a_mn=False, b_mn=False, bias: Optional[torch.Tensor] = None, act="none", aux: Optional[torch.Tensor] = None,
         ldaux: int = 0, aux_mode: int = 0, accumulate=False, split_k: int = 0, taps: int = 1,
         colsum: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None, mask_mode: int = 0) -> torch.Tensor:
    """out[M,N] (+)= epilogue(A[M,K] · B[N,K]^T); see ibm_gemm_bf16.  Leading dims default to the
    tensors' row strides.  colsum (fp32 [N]): += column sums of the bf16 output (a bias gradient).
    mask (uint8 [M, N/8]) with mask_mode 1: sign bits of the output are written; mask_mode 2: outputs whose bit is clear
    are zeroed (ReLU derivative without re-reading the activation)."""
    _require_cuda(A, B, out)
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16
    lda = A.stride(0) if lda is None else lda
    ldb = B.stride(0) if ldb is None else ldb
    ldd = out.stride(0) if ldd is None else ldd
    if aux is not None and ldaux == 0:
        ldaux = aux.stride(0)
    od = F32 if out.dtype == torch.float32 else BF16
    call("ibm_gemm_bf16", _p(A), lda, int(a_mn), _p(B), ldb, int(b_mn), M, N, K, _p(bias), ACT[act], _p(aux), ldaux,
         aux_mode, _p(out), ldd, od, int(accumulate), split_k, taps, _p(colsum), _p(mask),
         0 if mask is None else mask.stride(0), mask_mode if mask is not None else 0, stream_ptr())
    return out


def set_walk_order(mode: int) -> None:
    """0: kernels walk rows / tiles in ascending order; 1: big launches (>= 48 MB streamed) alternate ascending /
    descending so a consumer starts on what its producer wrote last (still in L2); 2: every launch alternates (tests)."""
    call("ibm_set_walk_order", int(mode))


def colsum(X: torch.Tensor, M: int, N: int, out: torch.Tensor, ld=None) -> None:
    call("ibm_colsum_bf16", _p(X), X.stride(0) if ld is None else ld, M, N, _p(out), stream_ptr())


def act_fwd(x, y, act):
    call("ibm_act_fwd", _p(x), _p(y), x.numel(), ACT[act], stream_ptr())


def act_bwd(dy, x, dx, act):
    call("ibm_act_bwd", _p(dy), _p(x), _p(dx), x.numel(), ACT[act], stream_ptr())


def cast_f32_bf16(src, dst):
    call("ibm_cast_f32_bf16", _p(src), _p(dst), src.numel(), stream_ptr())


def cast_bf16_f32(src, dst):
    call("ibm_cast_bf16_f32", _p(src), _p(dst), src.numel(), stream_ptr())


def cast_pad(src: torch.Tensor, dst: torch.Tensor, rows: int, cols: int, ld_src=None, ld_dst=None):
    call("ibm_cast_pad_f32_bf16", _p(src), src.stride(0) if ld_src is None else ld_src, _p(dst),
         dst.stride(0) if ld_dst is None else ld_dst, rows, cols, stream_ptr())


def conv_weight_to_gemm(w: torch.Tensor, dst: torch.Tensor, cin_pad: int):
    cout, cin, kt = w.shape
    call("ibm_conv_weight_to_gemm", _p(w), cout, cin, kt, cin_pad, _p(dst), stream_ptr())


def conv_wgrad_from_gemm(g: torch.Tensor, dw: torch.Tensor, cin_pad: int, accumulate: bool):
    cout, cin, kt = dw.shape
    call("ibm_conv_wgrad_from_gemm", _p(g), cout, cin, kt, cin_pad, _p(dw), int(accumulate), stream_ptr())


def replicate_pad_rows(X, n_win, T, pad, cols):
    call("ibm_replicate_pad_rows", _p(X), X.stride(0), n_win, T, pad, cols, stream_ptr())


def fold_pad_rows(G, n_win, T, pad, cols):
    call("ibm_fold_pad_rows", _p(G), G.stride(0), n_win, T, pad, cols, stream_ptr())


def dropout(x, y, p, seed, offset, step_dev=None, step_mul=0):
    """Philox offset = offset (+ step_mul * step_dev[0], read on the device at execution time, when a counter is given)."""
    if step_dev is None:
        call("ibm_dropout_bf16", _p(x), _p(y), x.numel(), p, seed, offset, stream_ptr())
    else:
        call("ibm_dropout_bf16_dev", _p(x), _p(y), x.numel(), p, seed, offset, _p(step_dev), step_mul, stream_ptr())


def counter_add(counter_dev, inc=1):
    call("ibm_counter_add", _p(counter_dev), inc, stream_ptr())


def conv_weight_to_dgrad(w: torch.Tensor, dst: torch.Tensor, cout_pad: int):
    cout, cin, kt = w.shape
    call("ibm_conv_weight_to_dgrad", _p(w), cout, cin, kt, cout_pad, _p(dst), stream_ptr())


# ---- BatchNorm1d -----------------------------------------------------------------------------------
def batchnorm_workspace(C: int, device) -> torch.Tensor:
    return torch.zeros(_lib.load().ibm_batchnorm_workspace_floats(C), dtype=torch.float32, device=device)


def batchnorm_fwd(x, y, M, C, gamma, beta, running_mean, running_var, save_mean, save_rstd, training, momentum, eps, ws):
    call("ibm_batchnorm_fwd", _p(x), x.stride(0), _p(y), y.stride(0), M, C, _p(gamma), _p(beta), _p(running_mean), _p(running_var),
         _p(save_mean), _p(save_rstd), int(training), momentum, eps, _p(ws), stream_ptr())


def batchnorm_bwd(dy, x, dx, M, C, gamma, mean, rstd_or_var, training, eps, dgamma, dbeta, ws, act_out=None, act=None,
                  dx_colsum=None):
    call("ibm_batchnorm_bwd", _p(dy), dy.stride(0), _p(x), x.stride(0), _p(dx), 0 if dx is None else dx.stride(0), M, C, _p(gamma),
         _p(mean), _p(rstd_or_var), int(training), eps, _p(act_out), 0 if act_out is None else act_out.stride(0), ACT[act],
         _p(dgamma), _p(dbeta), _p(dx_colsum), _p(ws), stream_ptr())


# ---- LayerNorm ----------------------------------------------------------------------------------
def layernorm_fwd(s, y, gamma, beta, M, d, eps=1e-5, mean=None, rstd=None, ld=None):
    call("ibm_layernorm_fwd", _p(s), _p(y), s.stride(0) if ld is None else ld, _p(gamma), _p(beta), M, d, eps, _p(mean),
         _p(rstd), stream_ptr())


def layernorm_bwd(dy, s, gamma, mean, rstd, M, d, ds, dgamma, dbeta, dcolsum=None, ld=None):
    call("ibm_layernorm_bwd", _p(dy), _p(s), s.stride(0) if ld is None else ld, _p(gamma), _p(mean), _p(rstd), M, d,
         _p(ds), _p(dgamma), _p(dbeta), _p(dcolsum), stream_ptr())


# ---- attention ----------------------------------------------------------------------------------
def attention_fwd_fused(qkv, kv_off, o, n_win, T, H, hd, scale):
    es = qkv.element_size()
    base = qkv.data_ptr()
    call("ibm_attention_fwd", base, qkv.stride(0), base + kv_off * es, qkv.stride(0), base + 2 * kv_off * es,
         qkv.stride(0), _p(o), o.stride(0), n_win, T, H, hd, hd, scale, stream_ptr())


def attention_fwd(q, k, v, o, n_win, T, H, hd_qk, hd_v, scale):
    call("ibm_attention_fwd", _p(q), q.stride(0), _p(k), k.stride(0), _p(v), v.stride(0), _p(o), o.stride(0), n_win, T, H,
         hd_qk, hd_v, scale, stream_ptr())


def attention_bwd(qkv, kv_off, d_o, dqkv, n_win, T, H, hd, scale, dbias=None):
    """dbias (fp32 [3*kv_off]): the column sums of dqkv are added to it (in_proj_bias gradient)."""
    call("ibm_attention_bwd", _p(qkv), qkv.stride(0), kv_off, _p(d_o), d_o.stride(0), _p(dqkv), n_win, T, H, hd, scale,
         _p(dbias), stream_ptr())


def attention_bwd_long(q, k, v, o, d_o, dq, dk, dv, n_win, T, H, hd_qk, hd_v, scale, dbq=None, dbk=None, dbv=None):
    """Backward for whole windows of up to 256 frames (ibm_attention_bwd_long): q/k/v/o/d_o/dq/dk/dv are bf16 row-major
    views (one row per (window, frame), head h at columns h*hd); dv None when the values are an input."""
    call("ibm_attention_bwd_long", _p(q), q.stride(0), _p(k), k.stride(0), _p(v), v.stride(0), _p(o), o.stride(0), _p(d_o),
         d_o.stride(0), _p(dq), dq.stride(0), _p(dk), dk.stride(0), _p(dv), 0 if dv is None else dv.stride(0), n_win, T, H,
         hd_qk, hd_v, scale, _p(dbq), _p(dbk), _p(dbv), stream_ptr())


# ---- regression loss ------------------------------------------------------------------------------
def _ptr_array(ts: Sequence[torch.Tensor]):
    arr = (ctypes.c_void_p * 4)(*[t.data_ptr() for t in ts])
    return arr


def _stride_array(ts: Sequence[torch.Tensor]):
    vals = []
    for t in ts:
        assert t.dim() == 3 and t.stride(2) == 1, "loss tensors must be (B,F,C) with unit channel stride"
        vals += [t.stride(0), t.stride(1)]
    return (ctypes.c_int64 * 8)(*vals)


def regression_loss_fwd(outs: Sequence[torch.Tensor], labs: Sequence[torch.Tensor], weights30: Sequence[float],
                        threshold: float = 10.0, result: Optional[torch.Tensor] = None) -> torch.Tensor:
    """outs/labs in quantity order (cop, force, torque, wrench), fp32 (B,F,C).  Returns fp32[40]."""
    _require_cuda(*outs, *labs)
    B, F = outs[0].shape[0], outs[0].shape[1]
    if result is None:
        result = torch.empty(40, dtype=torch.float32, device=outs[0].device)
    w = (ctypes.c_float * 30)(*weights30)
    call("ibm_regression_loss_fwd", _ptr_array(outs), _stride_array(outs), _ptr_array(labs), _stride_array(labs), B, F, w,
         threshold, _p(result), _p(workspace(outs[0].device)), stream_ptr())
    return result


def regression_loss_bwd(outs, labs, weights30, grads: Sequence[torch.Tensor], upstream: Optional[torch.Tensor] = None,
                        threshold: float = 10.0) -> None:
    B, F = outs[0].shape[0], outs[0].shape[1]
    w = (ctypes.c_float * 30)(*weights30)
    gd = F32 if grads[0].dtype == torch.float32 else BF16
    call("ibm_regression_loss_bwd", _ptr_array(outs), _stride_array(outs), _ptr_array(labs), _stride_array(labs), B, F, w,
         threshold, _p(upstream), _ptr_array(grads), _stride_array(grads), gd, stream_ptr())


# ---- the evaluator's static helpers, general contract (csrc/loss_helpers.cu) -----------------------------
def sqdiff_mean_vector(o: torch.Tensor, l: torch.Tensor) -> torch.Tensor:
    _require_cuda(o, l)
    B, F, C = o.shape
    out = torch.empty(C, dtype=torch.float32, device=o.device)
    call("ibm_sqdiff_mean_vector", _p(o), o.stride(0), o.stride(1), _p(l), l.stride(0), l.stride(1), B, F, C, _p(out),
         _p(workspace(o.device)), stream_ptr())
    return out


def sqdiff_mean_vector_bwd(o, l, upstream, grad_out=None, grad_lab=None) -> None:
    B, F, C = o.shape
    call("ibm_sqdiff_mean_vector_bwd", _p(o), o.stride(0), o.stride(1), _p(l), l.stride(0), l.stride(1), B, F, C, _p(upstream),
         _p(grad_out), _p(grad_lab), stream_ptr())


def mask_by_threes(x: torch.Tensor, threshold: float) -> torch.Tensor:
    _require_cuda(x)
    B, F, C = x.shape
    out = torch.empty(B, F, C, dtype=torch.float32, device=x.device)
    call("ibm_mask_by_threes", _p(x), x.stride(0), x.stride(1), B, F, C, float(threshold), _p(out), stream_ptr())
    return out


def mean_norm_error(o: torch.Tensor, l: torch.Tensor, vec_size: int, fold_halves: bool = False) -> torch.Tensor:
    _require_cuda(o, l)
    B, F, C = o.shape
    out = torch.empty(1, dtype=torch.float32, device=o.device)
    call("ibm_mean_norm_error", _p(o), o.stride(0), o.stride(1), _p(l), l.stride(0), l.stride(1), B, F, C, int(vec_size),
         1 if fold_halves else 0, _p(out), _p(workspace(o.device)), stream_ptr())
    return out[0]


# ---- DDPM -----------------------------------------------------------------------------------------
def q_sample(x0, eps, t, sqrt_abar, sqrt_1m_abar, xt_f32=None, xt_bf16=None, bf16_ld=0, seed=0, offset=0, eps_out=None):
    B = x0.shape[0]
    per_win = x0.numel() // B
    call("ibm_q_sample", _p(x0), _p(eps), _p(t), _p(sqrt_abar), _p(sqrt_1m_abar), B, per_win, _p(xt_f32), _p(xt_bf16), bf16_ld,
         seed, offset, _p(eps_out), stream_ptr())


def _check_known(known, known_mask, M):
    """Validates the inpainting inputs of ``posterior_step`` / ``guided_step``; True when both are given."""
    if known is None and known_mask is None:
        return False
    if known is None or known_mask is None:
        raise ValueError("known and known_mask go together: give both or neither")
    for name, t, dt, shape in (("known", known, torch.float32, (M, 30)), ("known_mask", known_mask, torch.int32, (M,))):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != dt or not t.is_contiguous() or tuple(t.shape) != shape:
            raise ValueError(f"{name} must be a contiguous {dt} CUDA tensor of shape {shape}")
    return True


def posterior_step(x0_hat, x0_ld, x_t, z, t_dev, coef_x0, coef_xt, sigma, M, x_prev=None, xprev_bf16=None, bf16_ld=0,
                   seed=0, offset=0, t_next=None, t_succ=None, known=None, known_mask=None):
    """t_succ (device int32 [T]): the step of a respaced (DDIM) sequence, t_next receives t_succ[t]; None ⇒ the DDPM
    posterior step, t_next receives t-1.  ``known`` (fp32 [M, 30]) with ``known_mask`` (int32 [M], bit c = channel c is known):
    the known entries replace the prediction before the update (``ibm_ddpm_inpaint_step``, inpainting)."""
    if _check_known(known, known_mask, M):
        call("ibm_ddpm_inpaint_step", _p(x0_hat), x0_ld, _p(x_t), _p(z), _p(t_dev), _p(coef_x0), _p(coef_xt), _p(sigma), M,
             _p(x_prev), _p(xprev_bf16), bf16_ld, seed, offset, _p(t_next), _p(t_succ), 1.0, 0, _p(known), _p(known_mask),
             stream_ptr())
    elif t_succ is None:
        call("ibm_ddpm_posterior_step", _p(x0_hat), x0_ld, _p(x_t), _p(z), _p(t_dev), _p(coef_x0), _p(coef_xt), _p(sigma), M,
             _p(x_prev), _p(xprev_bf16), bf16_ld, seed, offset, _p(t_next), stream_ptr())
    else:
        call("ibm_ddpm_respaced_step", _p(x0_hat), x0_ld, _p(x_t), _p(z), _p(t_dev), _p(coef_x0), _p(coef_xt), _p(sigma), M,
             _p(x_prev), _p(xprev_bf16), bf16_ld, seed, offset, _p(t_next), _p(t_succ), stream_ptr())


def guided_step(x0_hat, x0_ld, x_t, z, t_dev, coef_x0, coef_xt, sigma, M, guidance_scale, x_prev=None, xprev_bf16=None,
                bf16_ld=0, seed=0, offset=0, t_next=None, t_succ=None, known=None, known_mask=None):
    """``posterior_step`` on a classifier-free guided prediction: x0_hat holds 2M rows, conditional then unconditional,
    combined in fp32 as u + guidance_scale (c - u); xprev_bf16 receives the bf16 rows at m and at M + m.  ``known`` /
    ``known_mask`` as in ``posterior_step``, applied to the guided prediction."""
    if _check_known(known, known_mask, M):
        call("ibm_ddpm_inpaint_step", _p(x0_hat), x0_ld, _p(x_t), _p(z), _p(t_dev), _p(coef_x0), _p(coef_xt), _p(sigma), M,
             _p(x_prev), _p(xprev_bf16), bf16_ld, seed, offset, _p(t_next), _p(t_succ), float(guidance_scale), 1, _p(known),
             _p(known_mask), stream_ptr())
    else:
        call("ibm_ddpm_guided_step", _p(x0_hat), x0_ld, _p(x_t), _p(z), _p(t_dev), _p(coef_x0), _p(coef_xt), _p(sigma), M,
             _p(x_prev), _p(xprev_bf16), bf16_ld, seed, offset, _p(t_next), _p(t_succ), float(guidance_scale), stream_ptr())


def multistep_step(x0_hat, x0_ld, x_t, t_dev, coef_x0, coef_xt, coef_prev, t_succ, M, x0_prev, x_prev=None, xprev_bf16=None,
                   bf16_ld=0, t_next=None, guidance_scale=None, known=None, known_mask=None):
    """One DPM-Solver++(2M) step (``ibm_ddpm_multistep_step``) on the tables of ``diffusion.dpm_schedule``: x_p =
    coef_x0[t] x0_hat + coef_prev[t] x0_prev + coef_xt[t] x_t, no noise; t_next receives t_succ[t].  ``x0_prev`` (fp32 [M, 30])
    holds the previous step's prediction, is read only where coef_prev[t] != 0 and receives this step's in place.
    ``guidance_scale`` None: x0_hat holds M rows; a scale: 2M rows combined as in ``guided_step``.  ``known`` /
    ``known_mask`` as in ``posterior_step``, applied after the guided combination."""
    if not isinstance(x0_prev, torch.Tensor) or not x0_prev.is_cuda or x0_prev.dtype != torch.float32 or \
            not x0_prev.is_contiguous() or tuple(x0_prev.shape) != (M, 30):
        raise ValueError(f"x0_prev must be a contiguous fp32 CUDA tensor of shape {(M, 30)}")
    _check_known(known, known_mask, M)
    guided = guidance_scale is not None
    call("ibm_ddpm_multistep_step", _p(x0_hat), x0_ld, _p(x_t), _p(t_dev), _p(coef_x0), _p(coef_xt), _p(coef_prev), _p(t_succ), M,
         _p(x0_prev), _p(x_prev), _p(xprev_bf16), bf16_ld, _p(t_next), float(guidance_scale) if guided else 1.0, int(guided),
         _p(known), _p(known_mask), stream_ptr())


def cond_dropout(xc, B, F, col0, ncols, p, seed, offset, keep_out=None):
    """Zeroes columns col0 .. col0+ncols-1 of the F rows of each dropped window of xc (bf16 [B*F, ld]); window b is dropped
    iff word 0 of Philox draw b at (seed, offset) is below uint32(p * 2^32), every window at p = 1.  keep_out (uint8 [B]):
    1 = kept.  p must lie in (0, 1]: p = 0 drops nothing, and callers launch nothing."""
    if not 0.0 < p <= 1.0:
        raise ValueError(f"condition dropout probability must lie in (0, 1], got {p}")
    if keep_out is not None and (keep_out.dtype != torch.uint8 or keep_out.numel() < B):
        raise ValueError(f"keep_out must be uint8 with at least {B} elements")
    call("ibm_cond_dropout", _p(xc), xc.stride(0), B, F, col0, ncols, p, seed, offset, _p(keep_out), stream_ptr())


# ---- ensemble scoring -------------------------------------------------------------------------------
ENSEMBLE_MAX_DRAWS = 64          # ibm_ensemble_score holds the K draws of an element in registers
ENSEMBLE_QUANTITIES = ("crps", "var", "sqerr", "pair", "count")     # rows of the fp64 [5, 30] accumulator


class EnsembleWorkspace:
    """Device buffers of ``ensemble_score``: the per-block partials (1024 x 150 fp64) and the last-block counter."""

    def __init__(self, device):
        self.partials = torch.zeros(1024 * 150, dtype=torch.float64, device=device)
        self.counter = torch.zeros(1, dtype=torch.int32, device=device)


def ensemble_score(draws: torch.Tensor, labels: torch.Tensor, acc: torch.Tensor, mean_out: torch.Tensor, ws: EnsembleWorkspace,
                   threshold: float = 10.0) -> torch.Tensor:
    """Scores K draws per window (``ibm_ensemble_score``): draws fp32 (K, B, F, 30) draw-major, as ``GaussianDiffusion.sample(...,
    num_samples=K)`` returns them; labels fp32 (B, Fo, 30) with Fo in {1, F}.  Writes the ensemble mean to ``mean_out`` (B, Fo, 30)
    and adds the batch's per-channel sums of CRPS, s^2, (m - y)^2, mean pairwise distance and the count to ``acc`` (fp64 [5, 30],
    rows in ENSEMBLE_QUANTITIES order).  CoP channels count contact rows only (label force norm > ``threshold``, the fused loss
    kernel's test).  Every check runs before the launch: a refused call launches nothing.  Returns ``mean_out``."""
    for name, t, dt in (("draws", draws, torch.float32), ("labels", labels, torch.float32), ("mean_out", mean_out, torch.float32),
                        ("acc", acc, torch.float64)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != dt or not t.is_contiguous():
            raise ValueError(f"ensemble_score: {name} must be a contiguous {dt} CUDA tensor")
    if draws.dim() != 4 or draws.shape[-1] != 30:
        raise ValueError(f"ensemble_score: draws must be (K, B, F, 30), got {tuple(draws.shape)}")
    K, B, F = draws.shape[:3]
    if not 2 <= K <= ENSEMBLE_MAX_DRAWS:
        raise ValueError(f"ensemble_score: K must lie in [2, {ENSEMBLE_MAX_DRAWS}], got {K}")
    if labels.dim() != 3 or labels.shape[0] != B or labels.shape[2] != 30 or labels.shape[1] not in (1, F):
        raise ValueError(f"ensemble_score: labels must be (B={B}, 1 or F={F}, 30), got {tuple(labels.shape)}")
    if tuple(mean_out.shape) != tuple(labels.shape):
        raise ValueError(f"ensemble_score: mean_out must have the labels' shape {tuple(labels.shape)}, got {tuple(mean_out.shape)}")
    if tuple(acc.shape) != (len(ENSEMBLE_QUANTITIES), 30):
        raise ValueError(f"ensemble_score: acc must be fp64 (5, 30), got {tuple(acc.shape)}")
    if B == 0 or F == 0:
        raise ValueError("ensemble_score: empty batch")
    call("ibm_ensemble_score", _p(draws), K, B, F, _p(labels), labels.shape[1], float(threshold), _p(mean_out), _p(acc),
         _p(ws.partials), _p(ws.counter), stream_ptr())
    return mean_out


def timestep_embed(t, out_bf16, dim, scalar=False):
    B = out_bf16.shape[0]
    call("ibm_timestep_embed", _p(t), int(scalar), B, dim, _p(out_bf16), stream_ptr())


def add_time_pos(h, temb, pos, M, F, d, t_row=None):
    """t_row (device int32[1]): temb is a per-timestep table and row t_row[0] is added to every window."""
    call("ibm_add_time_pos", _p(h), h.stride(0), _p(temb), temb.stride(0), _p(pos), M, F, d, _p(t_row), stream_ptr())


def add_time_pos_bwd(dh, dtemb, dpos, M, F, d, dbias=None):
    """dbias (fp32 [d]): += the column sums of dh over all rows (bias gradient of the Linear that produced h), same pass."""
    call("ibm_add_time_pos_bwd", _p(dh), dh.stride(0), _p(dtemb), dtemb.stride(0), _p(dpos), M, F, d, _p(dbias), stream_ptr())


# ---- window batcher ---------------------------------------------------------------------------------
def window_valid_mask(missing, trial_base, cand_trial, cand_start, window_size, stride, valid):
    call("ibm_window_valid_mask", _p(missing), _p(trial_base), _p(cand_trial), _p(cand_start), cand_trial.numel(),
         window_size, stride, _p(valid), stream_ptr())


def pack_windows(frames, C, win_row0, F, stride, out_f32=None, out_bf16=None, frame_stride=0, win_extra=0, col0=0):
    call("ibm_pack_windows", _p(frames), frames.stride(0), C, _p(win_row0), win_row0.numel(), F, stride, _p(out_f32),
         _p(out_bf16), frame_stride, win_extra, col0, stream_ptr())


def pack_inputs(srcs, n_rows, F, out_f32=None, out_bf16=None, frame_stride=0, win_extra=0, col0=0):
    """srcs: list of contiguous fp32 CUDA tensors [n_rows, w_k] (any leading shape that flattens to n_rows)."""
    n = len(srcs)
    ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in srcs])
    widths = (ctypes.c_int32 * n)(*[t.shape[-1] for t in srcs])
    call("ibm_pack_inputs", ptrs, widths, n, n_rows, F, _p(out_f32), _p(out_bf16), frame_stride, win_extra, col0, stream_ptr())


def pack_labels(raw, nb, win_row0, contact_idx, mass, F, stride, last_only, out_rows):
    call("ibm_pack_labels", _p(raw), raw.stride(0), nb, _p(win_row0), _p(contact_idx), _p(mass), win_row0.numel(), F, stride,
         int(last_only), _p(out_rows), out_rows.stride(0), stream_ptr())


# ---- optimizer ----------------------------------------------------------------------------------------
LR_SCHEDULES = {"constant": 0, "cosine": 1}


class GradClipWorkspace:
    """Device buffers of ``grad_clip_coef``: ``out`` = {pre-clip total norm, clip coefficient} (fp32[2]), the per-block
    partials and the last-block counter, and ``record`` = {sum of totals, steps, clipped steps} (fp64[3]) for reports."""

    def __init__(self, device):
        self.out = torch.zeros(2, dtype=torch.float32, device=device)
        self.partials = torch.zeros(1024, dtype=torch.float64, device=device)
        self.counter = torch.zeros(1, dtype=torch.int32, device=device)
        self.record = torch.zeros(3, dtype=torch.float64, device=device)


def grad_clip_coef(grad, max_norm, grad_scale=1.0, ws: Optional[GradClipWorkspace] = None, record=True) -> torch.Tensor:
    """torch.nn.utils.clip_grad_norm_'s total norm and clip coefficient of ``grad_scale * grad`` (a flat fp32 arena) into
    ``ws.out`` = {total, min(1, max_norm / (total + 1e-6))}, on the device, without a host synchronisation; with ``record``
    also accumulates ``ws.record``.  Returns ``ws.out``."""
    _require_cuda(grad)
    if grad.dtype != torch.float32 or not grad.is_contiguous():
        raise ValueError(f"gradient arena must be contiguous fp32, got {grad.dtype}")
    ws = ws or GradClipWorkspace(grad.device)
    call("ibm_grad_clip_coef", _p(grad), grad.numel(), grad_scale, max_norm, _p(ws.out), _p(ws.partials), _p(ws.counter),
         _p(ws.record) if record else None, stream_ptr())
    return ws.out


def optimizer_step(kind: str, param, grad, state0, state1, param_bf16, lr, grad_scale, step, step_dev=None, ema=None,
                   ema_decay=0.0, clip=None, schedule=None, warmup_steps=0, total_steps=0, lr_min=0.0):
    """``step_dev`` (device int64[1]) replaces the by-value 1-based step count (graph-replayed steps).  ``ema`` (fp32, the
    parameters' layout): also updates this exponential moving average of the parameters in the same pass, decay
    min(``ema_decay``, (1 + n) / (10 + n)) at step n.

    ``clip`` (device fp32[2] from ``grad_clip_coef``) multiplies the averaged gradient by its clip coefficient; ``schedule``
    ('constant' or 'cosine') scales ``lr`` at step n by the warm-up / cosine factor of ibm_b200.h, from ``warmup_steps``,
    ``total_steps`` and ``lr_min``.  Either one selects the scheduled kernel; with neither the call is the plain step."""
    if ema is not None:
        if ema.numel() != param.numel() or ema.dtype != torch.float32:
            raise ValueError(f"EMA arena must be fp32 with {param.numel()} elements, got {ema.dtype} x {ema.numel()}")
    if clip is not None or schedule is not None:
        if schedule is None:
            schedule = "constant"
        if schedule not in LR_SCHEDULES:
            raise ValueError(f"unknown learning-rate schedule {schedule!r}; expected one of {sorted(LR_SCHEDULES)}")
        if clip is not None and (clip.dtype != torch.float32 or clip.numel() < 2):
            raise ValueError("clip must be the fp32[2] {total, coefficient} of grad_clip_coef")
        call("ibm_optimizer_step_sched", _lib.OPT_KIND[kind], _p(param), _p(grad), _p(state0), _p(state1), _p(param_bf16),
             _p(ema), param.numel(), lr, grad_scale, ema_decay if ema is not None else 0.0, step, _p(step_dev), _p(clip),
             LR_SCHEDULES[schedule], int(warmup_steps), int(total_steps), lr_min, stream_ptr())
        return
    if ema is not None:
        call("ibm_optimizer_step_ema", _lib.OPT_KIND[kind], _p(param), _p(grad), _p(state0), _p(state1), _p(param_bf16), _p(ema),
             param.numel(), lr, grad_scale, ema_decay, step, _p(step_dev), stream_ptr())
        return
    if step_dev is not None:
        call("ibm_optimizer_step_dev", _lib.OPT_KIND[kind], _p(param), _p(grad), _p(state0), _p(state1), _p(param_bf16), param.numel(),
             lr, grad_scale, _p(step_dev), stream_ptr())
        return
    call("ibm_optimizer_step", _lib.OPT_KIND[kind], _p(param), _p(grad), _p(state0), _p(state1), _p(param_bf16), param.numel(),
         lr, grad_scale, step, stream_ptr())
