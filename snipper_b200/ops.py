"""torch custom ops over the C ABI (libmsda_b200.so).

PyTorch is plumbing here: it owns device memory and the current stream; all arithmetic happens
in the hand-written kernels.  Ops (namespace ``snipper_b200``):

  msda_forward / msda_backward          per-call op, the reference's extension functions
                                        (models/ops/src/vision.cpp:13-16)
  snippet_forward / snippet_backward    fused per-layer Snipper attention on separate offsets / logits
                                        (models/ops/modules/ms_deform_attn.py:126-225)
  snippet_attn / snippet_attn_backward  the same layer on the packed [offsets | logits] projection, with in-kernel
                                        biases, padding mask and encoder reference points; what the module runs
  masked_zero_                          in-place masked zero-fill of value (ms_deform_attn.py:116-117)
  layer_tail                            bias + residual + LayerNorm (+ pos) after a block, inference only
  layer_tail_amp                        the same on a bf16 GEMM output, also writing the next GEMMs' bf16 inputs
                                        (libmsda_b200_amp.so, for bf16 autocast)
  layer_tail_train / _backward          bias + dropout (by a given keep-mask) + residual + LayerNorm (+ pos) and its
                                        backward, for training (libmsda_b200_train.so)
  layer_tail_amp_train / _backward      the same on a bf16 GEMM output, also writing the next GEMMs' bf16 inputs, for
                                        training under bf16 autocast (libmsda_b200_amp_train.so)

The five forwards (msda_forward, snippet_forward, snippet_attn, layer_tail_train, layer_tail_amp_train) carry
``register_autograd`` formulas, so they compose with autograd / DDP as plain nodes (no host sync, no unused parameters).
"""
from typing import Optional, Tuple

import numpy as np
import torch
from torch import Tensor

from . import capi

_DTYPES = {torch.float32: capi.MSDA_DTYPE_F32, torch.float64: capi.MSDA_DTYPE_F64,
           torch.bfloat16: capi.MSDA_DTYPE_BF16}

# process-wide switch for the deterministic (atomics-free) grad_value path
_deterministic = False


# planar neighbour-frame slots (csrc/msda_planar.cu): OPT-IN (SNIPPER_B200_PLANAR=1 in the environment or
# set_planar_slots(True)).  Measured on B200 (profiles/r02_run8_*): full-line L1 wavefronts and 30 % fewer instructions
# leave the encoder gather where it was (166 vs 164 us) -- both layouts run at the L1 global-load datapath's rate --
# while the slots take 4/3 of the memory, so the cell-major slots stay the default.
_planar = __import__("os").environ.get("SNIPPER_B200_PLANAR", "0") == "1"


def set_planar_slots(flag: bool) -> None:
    global _planar
    _planar = bool(flag)


def set_deterministic(flag: bool) -> None:
    """Select the bit-reproducible two-pass backward (north_star: 'deterministic two-pass mode')."""
    global _deterministic
    _deterministic = bool(flag)


def is_deterministic() -> bool:
    return _deterministic


class LaunchStats:
    """Counts kernel launches issued through the C ABI and, when ``timing`` is on, brackets each
    launch with CUDA events on the launching stream (bench.py's roofline measurement)."""

    def __init__(self):
        self.launches = 0
        self.timing = False
        self.events = []  # (tag, dims, start_event, end_event)

    def reset(self):
        self.launches = 0
        self.events = []

    def kernel_ms(self):
        """tag -> list of per-launch durations in ms (call after a device synchronize)."""
        out = {}
        for tag, dims, s, e in self.events:
            out.setdefault((tag, dims), []).append(s.elapsed_time(e))
        return out


STATS = LaunchStats()


def _launch(entry, tag, dims, device, *args, n_kernels=1, what=None, batch=None, im2col_step=None, amp=False,
            train=False):
    """Call the C entry point ``entry`` (of libmsda_b200_amp.so when ``amp``, of libmsda_b200_train.so when ``train``,
    of libmsda_b200_amp_train.so when both) with ``args`` and ``device``'s current stream (every launching entry point
    takes the stream last), count its ``n_kernels`` kernels in STATS under ``tag`` / ``dims`` and raise on a failed
    status."""
    lib = (capi.amp_train_lib() if amp and train else capi.amp_lib() if amp else capi.train_lib() if train
           else capi.lib())
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device)
        if STATS.timing:
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record(stream)
        status = getattr(lib, entry)(*args, stream.cuda_stream)
        STATS.launches += n_kernels
        if STATS.timing:
            end.record(stream)
            STATS.events.append((tag, dims, start, end))
    last_error = (lib.msda_amp_train_last_cuda_error if amp and train else lib.msda_amp_last_cuda_error if amp
                  else lib.msda_train_last_cuda_error if train else None)
    capi.check(status, what or entry, batch, im2col_step, last_error)


def _workspace(nbytes, device):
    """-> (tensor to keep alive, 256-byte aligned pointer to ``nbytes`` bytes of it)"""
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
    return ws, (ws.data_ptr() + 255) // 256 * 256


def _require_cuda(t: Tensor, name: str) -> None:
    if not t.is_cuda:
        # reference models/ops/src/ms_deform_attn.h:38,60
        raise RuntimeError("Not implemented on the CPU" if name == "value" else "%s must be a CUDA tensor" % name)


def _require_contiguous(t: Tensor, name: str) -> None:
    if not t.is_contiguous():
        # reference models/ops/src/cuda/ms_deform_attn_cuda.cu:28-32
        raise RuntimeError("%s tensor has to be contiguous" % name)


def _value_batch_stride(value: Tensor) -> int:
    """value (N,S,M,D): the inner three dims must be dense; the batch stride is free."""
    N, S, M, D = value.shape
    if N * S * M * D == 0:
        return 0
    if value.stride(3) != 1 or value.stride(2) != D or (S > 1 and value.stride(1) != M * D):
        raise RuntimeError("value tensor has to be contiguous")
    return value.stride(0) if N > 1 else S * M * D


def _check_percall(value, spatial_shapes, level_start_index, sampling_loc, attn_weight):
    for t, name in ((value, "value"), (spatial_shapes, "spatial_shapes"),
                    (level_start_index, "level_start_index"), (sampling_loc, "sampling_loc"),
                    (attn_weight, "attn_weight")):
        _require_cuda(t, name)
    for t, name in ((spatial_shapes, "spatial_shapes"), (level_start_index, "level_start_index"),
                    (sampling_loc, "sampling_loc"), (attn_weight, "attn_weight")):
        _require_contiguous(t, name)
    if value.dim() != 4 or sampling_loc.dim() != 6 or attn_weight.dim() != 5:
        raise RuntimeError("expected value (N,S,M,D), sampling_loc (N,Lq,M,L,P,2), attn_weight (N,Lq,M,L,P)")
    if value.dtype not in _DTYPES:
        raise RuntimeError("ms_deform_attn: unsupported dtype %s (float32 / float64 / bfloat16)" % value.dtype)
    if value.dtype == torch.bfloat16:
        # bf16 mode: value / output / grad_output are bf16; locations and weights are computed in fp32
        if sampling_loc.dtype != torch.float32 or attn_weight.dtype != torch.float32:
            raise RuntimeError("bfloat16 value needs float32 sampling_loc and attn_weight")
        if value.shape[3] % 16 != 0 or value.shape[3] > 128:
            raise RuntimeError("bfloat16 ms_deform_attn needs head channels D % 16 == 0 and D <= 128")
    elif sampling_loc.dtype != value.dtype or attn_weight.dtype != value.dtype:
        raise RuntimeError("value, sampling_loc and attn_weight must share one dtype")
    if spatial_shapes.dtype != torch.int64 or level_start_index.dtype != torch.int64:
        raise RuntimeError("spatial_shapes and level_start_index must be int64")
    N, S, M, D = value.shape
    Nl, Lq, Ml, L, P, two = sampling_loc.shape
    if (Nl, Ml, two) != (N, M, 2) or tuple(attn_weight.shape) != (N, Lq, M, L, P):
        raise RuntimeError("sampling_loc / attn_weight shapes do not match value")
    if tuple(spatial_shapes.shape) != (L, 2) or level_start_index.numel() != L:
        raise RuntimeError("spatial_shapes must be (L,2) and level_start_index (L,)")
    return N, S, M, D, L, Lq, P


@torch.library.custom_op("snipper_b200::msda_forward", mutates_args=())
def msda_forward(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor,
                 sampling_loc: Tensor, attn_weight: Tensor, im2col_step: int) -> Tensor:
    N, S, M, D, L, Lq, P = _check_percall(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)
    vbs = _value_batch_stride(value)
    out = torch.empty((N, Lq, M * D), dtype=value.dtype, device=value.device)
    _launch("msda_forward", "msda_forward", (N, S, M, D, L, Lq, P), value.device,
            value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
            sampling_loc.data_ptr(), attn_weight.data_ptr(), out.data_ptr(),
            N, S, M, D, L, Lq, P, vbs, int(im2col_step), _DTYPES[value.dtype],
            what="ms_deform_attn_forward", batch=N, im2col_step=im2col_step)
    return out


@msda_forward.register_fake
def _(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step):
    N, S, M, D = value.shape
    return value.new_empty((N, sampling_loc.shape[1], M * D))


@torch.library.custom_op("snipper_b200::msda_backward", mutates_args=())
def msda_backward(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor,
                  sampling_loc: Tensor, attn_weight: Tensor, grad_output: Tensor,
                  im2col_step: int, deterministic: bool) -> Tuple[Tensor, Tensor, Tensor]:
    N, S, M, D, L, Lq, P = _check_percall(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)
    _require_cuda(grad_output, "grad_output")
    _require_contiguous(grad_output, "grad_output")
    if grad_output.dtype != value.dtype or grad_output.numel() != N * Lq * M * D:
        raise RuntimeError("grad_output must be (N,Lq,M*D) in value's dtype")
    vbs = _value_batch_stride(value)
    bf16 = value.dtype == torch.bfloat16
    if bf16 and deterministic:
        raise RuntimeError("the deterministic backward is float32 only")
    # bf16 mode accumulates grad_value in fp32 (include/msda_b200.h) and rounds once at the end
    grad_value = torch.empty((N, S, M, D), dtype=torch.float32 if bf16 else value.dtype, device=value.device)
    grad_loc = torch.empty_like(sampling_loc)
    grad_attn = torch.empty_like(attn_weight)
    flags = capi.MSDA_FLAG_DETERMINISTIC if deterministic else 0
    dt = _DTYPES[value.dtype]
    ws, ws_ptr, ws_bytes = None, 0, 0
    if deterministic:
        ws_bytes = capi.lib().msda_backward_workspace_bytes(N, S, M, D, L, Lq, P, dt, flags)
        ws, ws_ptr = _workspace(ws_bytes, value.device)
    # deterministic: no-scatter kernel, memset, count, 3 scan kernels, fill, reduce, long-list reduce
    _launch("msda_backward", "msda_backward_deterministic" if deterministic else "msda_backward",
            (N, S, M, D, L, Lq, P), value.device,
            value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
            sampling_loc.data_ptr(), attn_weight.data_ptr(), grad_output.data_ptr(),
            grad_value.data_ptr(), grad_loc.data_ptr(), grad_attn.data_ptr(),
            N, S, M, D, L, Lq, P, vbs, int(im2col_step), dt, flags, ws_ptr, ws_bytes,
            n_kernels=9 if deterministic else 2, what="ms_deform_attn_backward", batch=N, im2col_step=im2col_step)
    if bf16:
        grad_value = grad_value.to(torch.bfloat16)
    return grad_value, grad_loc, grad_attn


@msda_backward.register_fake
def _(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output, im2col_step, deterministic):
    return (value.new_empty(value.shape), torch.empty_like(sampling_loc), torch.empty_like(attn_weight))


def _msda_setup_context(ctx, inputs, output):
    value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step = inputs
    ctx.im2col_step = im2col_step
    ctx.save_for_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)


def _msda_backward_formula(ctx, grad_output):
    value, spatial_shapes, level_start_index, sampling_loc, attn_weight = ctx.saved_tensors
    gv, gl, ga = torch.ops.snipper_b200.msda_backward(
        value, spatial_shapes, level_start_index, sampling_loc, attn_weight,
        grad_output.contiguous(), ctx.im2col_step, _deterministic)
    return gv, None, None, gl, ga, None


msda_forward.register_autograd(_msda_backward_formula, setup_context=_msda_setup_context)


# ------------------------------------------------------------------------------------------
# in-place masked zero-fill (value production, SURVEY.md section 8f rank 2)
# ------------------------------------------------------------------------------------------
@torch.library.custom_op("snipper_b200::masked_zero_", mutates_args=("data",))
def masked_zero_(data: Tensor, mask: Tensor) -> None:
    """data[i] = 0 where mask[i]; both contiguous, same shape; data float32 / bfloat16, mask bool."""
    _require_cuda(data, "data")
    _require_cuda(mask, "mask")
    if data.shape != mask.shape or not data.is_contiguous() or not mask.is_contiguous():
        raise RuntimeError("masked_zero_: data and mask must be contiguous tensors of one shape")
    if mask.dtype != torch.bool or data.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError("masked_zero_: data must be float32 / bfloat16 and mask bool")
    _launch("msda_masked_zero", "masked_zero", (data.numel(),), data.device,
            data.data_ptr(), mask.data_ptr(), data.numel(), _DTYPES[data.dtype])


def masked_zero_supported(data: Tensor, mask: Tensor) -> bool:
    return (data.is_cuda and mask.is_cuda and data.dtype in (torch.float32, torch.bfloat16) and
            mask.dtype == torch.bool and data.shape == mask.shape and data.is_contiguous() and
            mask.is_contiguous() and mask.data_ptr() % 16 == 0)


# ------------------------------------------------------------------------------------------
# fused snippet op
# ------------------------------------------------------------------------------------------
def snippet_supported(n_heads: int, d_head: int, n_levels: int, n_points: int, dtype,
                      spatial_size: int = 0, batch_frames: int = 0) -> bool:
    """Shapes the fused kernels cover -- every constraint the C ABI enforces for the packed call
    (include/msda_b200.h msda_snippet_forward; msda_snippet.cu snippet_ok), so that a caller can fall back
    to the per-call loop instead of getting MSDA_ERR_INVALID_ARGUMENT."""
    esize = 2 if dtype == torch.bfloat16 else 4
    return (dtype in (torch.float32, torch.bfloat16) and d_head % 16 == 0 and d_head <= 128 and
            n_levels * n_points <= 32 and n_levels <= 64 and
            (n_heads * n_levels * n_points) % 2 == 0 and                     # float2 loads of a packed projection row
            spatial_size * n_heads * d_head * esize < (1 << 28) and          # cell byte offsets are 28-bit
            batch_frames <= 65535)                                           # gridDim.z


def _check_fused(value, spatial_shapes, level_start_index, reference_points, n_frame, *, offsets=None, logits=None,
                 proj=None, biases=(None, None), valid_ratios=None, presummed=False, T2=None, planar_dims=None):
    """Validate one fused call -> (N, T2, T1, S, M, D, L, Lq, P).

    The queries' sampling offsets and logits come as separate ``offsets`` (N,T1,Lq,M,L,P,2) and ``logits``
    (N,T1,Lq,M,L,P), or as the packed projection ``proj`` (N,T1,Lq,3*M*L*P) with optional ``biases``.  ``value`` is
    (N,T2,S,M,D), or the (N,slots,S,M,D) pre-summed slots when ``presummed`` (``T2`` then gives the source frames);
    ``planar_dims`` = (S, M, D) marks it as a planar carry (N, slots, planar_slot_elems) -- see snippet_attn."""
    ref = reference_points
    rows = (("proj", proj),) if proj is not None else (("offsets", offsets), ("logits", logits))
    for name, t in (("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
                    *rows, ("reference_points", ref)):
        if t is not None:
            _require_cuda(t, name)
    if planar_dims is not None:
        if (value.dim() != 3 or value.dtype != torch.float32 or not value.is_contiguous() or
                value.shape[2] != planar_slot_elems(*planar_dims, value.dtype) or value.data_ptr() % 128 != 0):
            raise RuntimeError("planar carry must be a contiguous float32 (N, slots, planar_slot_elems) tensor, 128-byte aligned")
        vshape = (value.shape[0], value.shape[1], *planar_dims)
    else:
        vshape = tuple(value.shape)
    if len(vshape) != 5 or (ref is not None and ref.dim() != 5):
        raise RuntimeError("expected value (N,T2,S,M,D) and reference_points (N,T1,Lq,L,2)")
    if (ref is None) == (valid_ratios is None):
        raise RuntimeError("pass either reference_points or (encoder self-attention) valid_ratios")
    N, F, S, M, D = vshape
    if proj is not None:
        L = spatial_shapes.shape[0]
        if proj.dim() != 4 or proj.shape[0] != N or proj.shape[3] % (3 * M * L) != 0:
            raise RuntimeError("proj must be (N,T1,Lq,3*M*L*P): [offsets (M,L,P,2) | logits (M,L,P)] per query")
        _, T1, Lq, W = proj.shape
        P = W // (3 * M * L)
    else:
        if offsets.dim() != 7 or logits.dim() != 6:
            raise RuntimeError("expected offsets (N,T1,Lq,M,L,P,2) and logits (N,T1,Lq,M,L,P)")
        No, T1, Lq, Mo, L, P, two = offsets.shape
        if (No, Mo, two) != (N, M, 2) or tuple(logits.shape) != (N, T1, Lq, M, L, P):
            raise RuntimeError("offsets / logits shapes do not match value")
    if tuple(spatial_shapes.shape) != (L, 2) or level_start_index.numel() != L:
        raise RuntimeError("spatial_shapes must be (L,2) and level_start_index (L,)")
    if ref is not None and (tuple(ref.shape) != (N, T1, Lq, L, 2) or ref.dtype != torch.float32):
        raise RuntimeError("reference_points must be float32 (N,T1,Lq,L,2)")
    if valid_ratios is not None:
        if (not valid_ratios.is_cuda or valid_ratios.dtype != torch.float32 or tuple(valid_ratios.shape) != (N, L, 2)
                or not valid_ratios.is_contiguous() or Lq != S):
            raise RuntimeError("valid_ratios must be contiguous float32 (N,L,2) and the queries the S pixels of the pyramid")
    if not snippet_supported(M, D, L, P, value.dtype, S, N * T1):
        raise RuntimeError("fused snippet attention needs float32 / bfloat16 value, D % 16 == 0, D <= 128, L*P <= 32")
    if any(t.dtype != torch.float32 for _, t in rows):
        raise RuntimeError("offsets and logits (or proj) must be float32")
    for b, n in zip(biases, (2 * M * L * P, M * L * P)):
        if b is not None and (not b.is_cuda or b.dtype != torch.float32 or b.numel() != n or not b.is_contiguous()):
            raise RuntimeError("biases must be contiguous float32 CUDA tensors of 2*M*L*P / M*L*P elements")
    if presummed:
        if F != num_slots(T1, n_frame) or not value.is_contiguous():
            raise RuntimeError("presummed value must be a contiguous (N, slots, S, M, D) tensor (or a planar carry)")
    else:
        T2 = F
    if not (0 < n_frame <= T2):
        raise RuntimeError("n_frame must be in (0, T2]")
    for name, t in (*rows, ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index)):
        _require_contiguous(t, name)
    return N, T2, T1, S, M, D, L, Lq, P


def _value_strides5(value):
    N, T2, S, M, D = value.shape
    if value.stride(4) != 1 or value.stride(3) != D or (S > 1 and value.stride(2) != M * D):
        raise RuntimeError("value tensor has to be contiguous in its (S,M,D) dims")
    st = value.stride(1) if T2 > 1 else S * M * D
    sn = value.stride(0) if N > 1 else st * T2
    return sn, st


def _ref_strides(ref):
    """(N,T1,Lq,L,2): inner (Lq,L,2) dense; batch / frame strides free (0 = broadcast)."""
    N, T1, Lq, L, _ = ref.shape
    if ref.numel() and (ref.stride(4) != 1 or ref.stride(3) != 2 or (Lq > 1 and ref.stride(2) != 2 * L)):
        ref = ref.contiguous()
    return ref, (ref.stride(0) if N > 1 else 0), (ref.stride(1) if T1 > 1 else 0)


def _ptr(t):
    return None if t is None else t.data_ptr()


# The two builders below are the only callers of the fused entry points: they put the named pieces of a call into the
# ABI's positional order (include/msda_b200.h).  ``value_strides`` are (batch, frame) element strides of value or the
# slots, 0 = dense; ``offsets`` / ``logits`` are (pointer, row stride in floats), 0 = dense rows; either
# ``reference_points`` or the encoder's ``valid_ratios`` is given; ``mask`` is (tensor or None, row stride, col stride)
# as mask_layout returns it.
def _issue_snippet_forward(tag, dims, n_frame, value, spatial_shapes, level_start_index, out, *, offsets, logits,
                           value_strides=(0, 0), reference_points=None, valid_ratios=None, biases=(None, None),
                           mask=(None, 0, 0), flags=0):
    N, T2, T1, S, M, D, L, Lq, P = dims
    ref, rsn, rst = _ref_strides(reference_points) if reference_points is not None else (None, 0, 0)
    _launch("msda_snippet_forward", tag, dims, value.device,
            value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(), offsets[0], logits[0], _ptr(ref),
            out.data_ptr(), N, T2, T1, int(n_frame), S, M, D, L, Lq, P, *value_strides, rsn, rst, offsets[1], logits[1],
            _ptr(biases[0]), _ptr(biases[1]), _ptr(valid_ratios), _ptr(mask[0]), mask[1], mask[2],
            _DTYPES[value.dtype], flags)


def _issue_snippet_backward(tag, n_kernels, dims, n_frame, value, spatial_shapes, level_start_index, grad_output,
                            grad_value, *, offsets, logits, grad_offsets, grad_logits, value_strides=(0, 0),
                            reference_points=None, valid_ratios=None, biases=(None, None), mask=(None, 0, 0), flags=0,
                            workspace=(None, 0)):
    """``grad_offsets`` / ``grad_logits`` are pointers with the row strides of ``offsets`` / ``logits``; ``workspace``
    is (pointer, bytes)."""
    N, T2, T1, S, M, D, L, Lq, P = dims
    ref, rsn, rst = _ref_strides(reference_points) if reference_points is not None else (None, 0, 0)
    _launch("msda_snippet_backward", tag, dims, value.device,
            value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(), offsets[0], logits[0], _ptr(ref),
            grad_output.data_ptr(), grad_value.data_ptr(), grad_offsets, grad_logits,
            N, T2, T1, int(n_frame), S, M, D, L, Lq, P, *value_strides, rsn, rst, offsets[1], logits[1],
            _ptr(biases[0]), _ptr(biases[1]), _ptr(valid_ratios), _ptr(mask[0]), mask[1], mask[2],
            _DTYPES[value.dtype], flags, *workspace, n_kernels=n_kernels)


def _grad_ref(grad_offsets, spatial_shapes):
    """grad_offsets (N,T1,Lq,M,L,P,2) -> the gradient of reference_points (N,T1,Lq,L,2):
    loc = ref + off/(W,H)  =>  dL/dref = sum_{m,p} dL/dloc = sum_{m,p} dL/doff * (W,H)"""
    wh = torch.stack([spatial_shapes[:, 1], spatial_shapes[:, 0]], -1).to(grad_offsets.dtype)
    return (grad_offsets * wh[None, None, None, None, :, None, :]).sum(dim=(3, 5))


@torch.library.custom_op("snipper_b200::snippet_forward", mutates_args=())
def snippet_forward(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor,
                    offsets: Tensor, logits: Tensor, reference_points: Tensor, n_frame: int) -> Tensor:
    """Fused layer attention on separate offsets / logits tensors, neighbour frames gathered directly."""
    dims = _check_fused(value, spatial_shapes, level_start_index, reference_points, n_frame, offsets=offsets,
                        logits=logits)
    N, T2, T1, S, M, D, L, Lq, P = dims
    out = torch.empty((N, T1, Lq, M * D), dtype=value.dtype, device=value.device)
    _issue_snippet_forward("snippet_forward", dims, n_frame, value, spatial_shapes, level_start_index, out,
                           offsets=(offsets.data_ptr(), 0), logits=(logits.data_ptr(), 0),
                           value_strides=_value_strides5(value), reference_points=reference_points)
    return out


@snippet_forward.register_fake
def _(value, spatial_shapes, level_start_index, offsets, logits, reference_points, n_frame):
    N, T2, S, M, D = value.shape
    return value.new_empty((N, offsets.shape[1], offsets.shape[2], M * D))


@torch.library.custom_op("snipper_b200::snippet_backward", mutates_args=())
def snippet_backward(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor,
                     offsets: Tensor, logits: Tensor, reference_points: Tensor, grad_output: Tensor,
                     n_frame: int) -> Tuple[Tensor, Tensor, Tensor]:
    dims = _check_fused(value, spatial_shapes, level_start_index, reference_points, n_frame, offsets=offsets,
                        logits=logits)
    N, T2, T1, S, M, D, L, Lq, P = dims
    _require_cuda(grad_output, "grad_output")
    _require_contiguous(grad_output, "grad_output")
    grad_value = torch.empty((N, T2, S, M, D), dtype=torch.float32, device=value.device)  # fp32 accumulation
    grad_offsets = torch.empty_like(offsets)
    grad_logits = torch.empty_like(logits)
    _issue_snippet_backward("snippet_backward", 2, dims, n_frame, value, spatial_shapes, level_start_index, grad_output,
                            grad_value, offsets=(offsets.data_ptr(), 0), logits=(logits.data_ptr(), 0),
                            grad_offsets=grad_offsets.data_ptr(), grad_logits=grad_logits.data_ptr(),
                            value_strides=_value_strides5(value), reference_points=reference_points)
    if value.dtype != torch.float32:
        grad_value = grad_value.to(value.dtype)
    return grad_value, grad_offsets, grad_logits


@snippet_backward.register_fake
def _(value, spatial_shapes, level_start_index, offsets, logits, reference_points, grad_output, n_frame):
    return (value.new_empty(value.shape), torch.empty_like(offsets), torch.empty_like(logits))


def _snippet_setup_context(ctx, inputs, output):
    value, spatial_shapes, level_start_index, offsets, logits, reference_points, n_frame = inputs
    ctx.n_frame = n_frame
    ctx.save_for_backward(value, spatial_shapes, level_start_index, offsets, logits, reference_points)


def _snippet_backward_formula(ctx, grad_output):
    value, spatial_shapes, level_start_index, offsets, logits, ref = ctx.saved_tensors
    gv, goff, glog = torch.ops.snipper_b200.snippet_backward(
        value, spatial_shapes, level_start_index, offsets, logits, ref, grad_output.contiguous(), ctx.n_frame)
    gref = _grad_ref(goff, spatial_shapes) if ctx.needs_input_grad[5] else None
    return gv, None, None, goff, glog, gref, None


snippet_forward.register_autograd(_snippet_backward_formula, setup_context=_snippet_setup_context)


# ------------------------------------------------------------------------------------------
# fused layer attention on the packed projection: offsets and logits are column blocks of ONE GEMM
# output, the two Linear biases are added in-kernel, the padding mask is applied inside the kernels
# (no pass over the value tensor) and, for encoder-sized query sets, the neighbour frames are summed
# BEFORE the gather (msda_frame_sum: the op is linear in value) so every sample is gathered once
# ------------------------------------------------------------------------------------------
def mask_layout(mask: Optional[Tensor], N: int, T2: int, S: int, C: int):
    """Padding mask over value (N,T2,S,C) -> (tensor to keep alive, row stride, col stride) for the C ABI
    (include/msda_b200.h, Conventions).  Accepts the reference's materialised (N,T2,S,C) bool tensor
    (models/model.py:156-157), a channel-expanded view (stride 0 in C) or a per-pixel (N,T2,S[,1]) mask."""
    if mask is None:
        return None, 0, 0
    if mask.dtype != torch.bool:
        raise RuntimeError("input_padding_mask must be a bool tensor")
    if mask.dim() == 3:
        mask = mask.unsqueeze(-1)
    if mask.dim() != 4 or tuple(mask.shape[:3]) != (N, T2, S) or mask.shape[3] not in (1, C):
        raise RuntimeError("input_padding_mask must be (N,T2,S,C), (N,T2,S,1) or (N,T2,S)")
    if mask.shape[3] == 1:
        mask = mask.expand(N, T2, S, C)
    sn, st, ss, sc = mask.stride()
    rows_ok = (S == 1 or ss > 0) and (T2 == 1 or st == S * ss) and (N == 1 or sn == T2 * S * ss)
    if not (rows_ok and sc in (0, 1) and (sc == 0 or (ss % 4 == 0 and mask.data_ptr() % 4 == 0))):
        mask = mask.contiguous()
        ss, sc = C, 1
    return mask, (ss if S > 1 else max(ss, 1)), sc


def prefers_presum(T2: int, T1: int, n_frame: int, S: int, L: int, Lq: int, P: int) -> bool:
    """True when summing the neighbour frames first (one streaming pass) beats gathering each of them."""
    return bool(capi.lib().msda_snippet_prefers_presum(T2, T1, int(n_frame), S, L, Lq, P))


def num_slots(T1: int, n_frame: int) -> int:
    return (T1 if T1 < n_frame else n_frame) + (1 if T1 > n_frame else 0)


def planar_slot_elems(S: int, M: int, D: int, dtype) -> int:
    """fp32 elements of one (n, slot) of the library's planar slot layout (csrc/msda_planar.cu), 0 when the layout
    does not apply (it is built for float32 heads of 48 channels)."""
    if dtype != torch.float32:
        return 0
    return capi.lib().msda_planar_slot_bytes(S, M, D, capi.MSDA_DTYPE_F32) // 4


def _frame_sum(value, mask, T1, n_frame, planar):
    """(N,T2,S,M,D) -> masked neighbour-frame sums, one slot per query frame: (N,slots,S,M,D) in value's dtype, or the
    same sums in the planar fp32 layout (N, slots, planar_slot_elems) laid out for the gather."""
    N, T2, S, M, D = value.shape
    sn, st = _value_strides5(value)
    slots = num_slots(T1, n_frame)
    if planar:
        vsum = torch.empty((N, slots, planar_slot_elems(S, M, D, value.dtype)), dtype=torch.float32, device=value.device)
        entry, tag, row = "msda_frame_sum_planar", "frame_sum_planar", (S, M, D)
    else:
        vsum = torch.empty((N, slots, S, M, D), dtype=value.dtype, device=value.device)
        entry, tag, row = "msda_frame_sum", "frame_sum", (S, M * D)
    _launch(entry, tag, (N, T2, T1, S, M * D), value.device, value.data_ptr(), _ptr(mask[0]), vsum.data_ptr(),
            N, T2, T1, int(n_frame), *row, sn, st, mask[1], mask[2], _DTYPES[value.dtype])
    return vsum


def _frame_unsum(grad_slots, mask, dims, n_frame, dtype, planar):
    """The adjoint of _frame_sum: fp32 slot gradients -> grad_value (N,T2,S,M,D) in ``dtype``, masked alike."""
    N, T2, T1, S, M, D = dims[:6]
    grad_value = torch.empty((N, T2, S, M, D), dtype=dtype, device=grad_slots.device)
    if planar:
        entry, tag, row = "msda_frame_unsum_planar", "frame_unsum_planar", (S, M, D)
    else:
        entry, tag, row = "msda_frame_unsum", "frame_unsum", (S, M * D)
    _launch(entry, tag, (N, T2, T1, S, M * D), grad_slots.device, grad_slots.data_ptr(), _ptr(mask[0]),
            grad_value.data_ptr(), N, T2, T1, int(n_frame), *row, mask[1], mask[2], _DTYPES[dtype])
    return grad_value


def use_planar(S: int, M: int, D: int, dtype) -> bool:
    """Planar slots when opted in (set_planar_slots), the layout applies (fp32, D = 48) and the deterministic mode
    (which walks cell-major slots) is off."""
    if not _planar:
        return False
    return planar_slot_elems(S, M, D, dtype) > 0 and not (_deterministic and torch.is_grad_enabled())


def _proj_columns(proj, mlp):
    """[offsets (M,L,P,2) | logits (M,L,P)] column blocks of a packed projection row -> two (pointer, row stride)"""
    return (proj.data_ptr(), 3 * mlp), (proj.data_ptr() + 4 * 2 * mlp, 3 * mlp)


@torch.library.custom_op("snipper_b200::snippet_attn", mutates_args=())
def snippet_attn(value: Tensor, value_mask: Optional[Tensor], spatial_shapes: Tensor, level_start_index: Tensor,
                 proj: Tensor, offsets_bias: Optional[Tensor], logits_bias: Optional[Tensor],
                 reference_points: Optional[Tensor], valid_ratios: Optional[Tensor], n_frame: int,
                 presum: bool, planar: bool = False) -> Tuple[Tensor, Tensor]:
    """The whole per-frame loop of the reference module (ms_deform_attn.py:116-117,126-225) for one layer.

    value (N,T2,S,M,D) is the raw ``value_proj`` output; ``value_mask`` the padding mask over it (any layout
    ``mask_layout`` accepts) or None; proj (N,T1,Lq,3*M*L*P) = [offsets | logits] without biases;
    ``reference_points`` (N,T1,Lq,L,2), or None with ``valid_ratios`` (N,L,2) for the encoder's self-attention,
    whose reference points the kernel then derives from the query index (deformable_transformer.py:219-232).
    Returns (out (N,T1,Lq,M*D), carry): carry is the presummed value when ``presum`` -- the only form of value the
    backward needs: (N,slots,S,M,D), or the library's planar slots (N,slots,planar_slot_elems) when ``planar`` (only
    with ``presum``; ``use_planar`` says where the layout applies) -- and an empty tensor otherwise."""
    dims = _check_fused(value, spatial_shapes, level_start_index, reference_points, n_frame, proj=proj,
                        biases=(offsets_bias, logits_bias), valid_ratios=valid_ratios)
    N, T2, T1, S, M, D, L, Lq, P = dims
    mask = mask_layout(value_mask, N, T2, S, M * D)
    out = torch.empty((N, T1, Lq, M * D), dtype=value.dtype, device=value.device)
    if planar and not (presum and planar_slot_elems(S, M, D, value.dtype) > 0):
        raise RuntimeError("planar slots need presum=True, float32 value and 48 channels per head")
    if presum:
        # the mask was applied by the frame sums; the kernel gets its strides without the pointer
        carry = _frame_sum(value, mask, T1, n_frame, planar)
        src, strides, kmask = carry, (0, 0), (None,) + mask[1:]
        flags = capi.MSDA_FLAG_PRESUMMED | (capi.MSDA_FLAG_PLANAR if planar else 0)
        tag = "snippet_forward_planar" if planar else "snippet_forward_presummed"
    else:
        carry = value.new_empty((0,))
        src, strides, kmask, flags, tag = value, _value_strides5(value), mask, 0, "snippet_forward"
    offsets, logits = _proj_columns(proj, M * L * P)
    _issue_snippet_forward(tag, dims, n_frame, src, spatial_shapes, level_start_index, out, offsets=offsets,
                           logits=logits, value_strides=strides, reference_points=reference_points,
                           valid_ratios=valid_ratios, biases=(offsets_bias, logits_bias), mask=kmask, flags=flags)
    return out, carry


@snippet_attn.register_fake
def _(value, value_mask, spatial_shapes, level_start_index, proj, offsets_bias, logits_bias, reference_points,
      valid_ratios, n_frame, presum, planar=False):
    N, T2, S, M, D = value.shape
    out = value.new_empty((N, proj.shape[1], proj.shape[2], M * D))
    if planar:
        return out, value.new_empty((N, num_slots(proj.shape[1], n_frame), planar_slot_elems(S, M, D, value.dtype)))
    if presum:
        return out, value.new_empty((N, num_slots(proj.shape[1], n_frame), S, M, D))
    return out, value.new_empty((0,))


@torch.library.custom_op("snipper_b200::snippet_attn_backward", mutates_args=())
def snippet_attn_backward(value_or_vsum: Tensor, value_mask: Optional[Tensor], spatial_shapes: Tensor,
                          level_start_index: Tensor, proj: Tensor, offsets_bias: Optional[Tensor],
                          logits_bias: Optional[Tensor], reference_points: Optional[Tensor],
                          valid_ratios: Optional[Tensor], grad_output: Tensor,
                          n_frame: int, presum: bool, n_src_frames: int, deterministic: bool,
                          value_dims: Optional[list[int]] = None) -> Tuple[Tensor, Tensor]:
    """Returns (grad_value (N,T2,S,M,D) in value's dtype, grad_proj with proj's layout [grad_offsets | grad_logits]).
    ``value_or_vsum`` is what the forward carried: the presummed value when ``presum`` (planar when
    ``value_dims`` = [S, M, D] is given: the 3-d carry does not say), else value itself."""
    planar = value_dims is not None
    if planar and not presum:
        raise RuntimeError("planar slots exist on the pre-summed path only")
    dims = _check_fused(value_or_vsum, spatial_shapes, level_start_index, reference_points, n_frame, proj=proj,
                        biases=(offsets_bias, logits_bias), valid_ratios=valid_ratios, presummed=presum,
                        T2=n_src_frames, planar_dims=tuple(value_dims) if planar else None)
    N, T2, T1, S, M, D, L, Lq, P = dims
    _require_cuda(grad_output, "grad_output")
    _require_contiguous(grad_output, "grad_output")
    if grad_output.dtype != value_or_vsum.dtype or grad_output.numel() != N * T1 * Lq * M * D:
        raise RuntimeError("grad_output must be (N,T1,Lq,M*D) in value's dtype")
    dev, dt = value_or_vsum.device, value_or_vsum.dtype
    mask = mask_layout(value_mask, N, T2, S, M * D)
    grad_proj = torch.empty_like(proj)
    if deterministic and not (presum and dt == torch.float32 and not planar):
        raise RuntimeError("the deterministic fused backward runs on the pre-summed (cell-major) float32 path")
    ws, workspace = None, (None, 0)
    if planar:
        grad_src = torch.empty_like(value_or_vsum)                                  # planar fp32 slots, zero-filled by the call
        flags, tag, n_kernels = capi.MSDA_FLAG_PRESUMMED | capi.MSDA_FLAG_PLANAR, "snippet_backward_planar", 2
    elif presum:
        grad_src = torch.empty((N, value_or_vsum.shape[1], S, M, D), dtype=torch.float32, device=dev)  # fp32 accumulation
        flags, tag, n_kernels = capi.MSDA_FLAG_PRESUMMED, "snippet_backward_presummed", 2
        if deterministic:
            # bit-reproducible: no-scatter kernel + two-pass ordered grad_value over the slots (include/msda_b200.h)
            flags |= capi.MSDA_FLAG_DETERMINISTIC
            ws_bytes = capi.lib().msda_snippet_backward_workspace_bytes(N, T1, int(n_frame), S, M, D, L, Lq, P,
                                                                        _DTYPES[dt], flags)
            ws, ws_ptr = _workspace(ws_bytes, dev)
            workspace = (ws_ptr, ws_bytes)
            tag, n_kernels = "snippet_backward_deterministic", 10
    else:
        grad_src = torch.empty((N, T2, S, M, D), dtype=torch.float32, device=dev)  # fp32 accumulation
        flags, tag, n_kernels = 0, "snippet_backward", 2
    offsets, logits = _proj_columns(proj, M * L * P)
    grad_offsets, grad_logits = _proj_columns(grad_proj, M * L * P)
    _issue_snippet_backward(tag, n_kernels, dims, n_frame, value_or_vsum, spatial_shapes, level_start_index,
                            grad_output, grad_src, offsets=offsets, logits=logits, grad_offsets=grad_offsets[0],
                            grad_logits=grad_logits[0], value_strides=(0, 0) if presum else _value_strides5(value_or_vsum),
                            reference_points=reference_points, valid_ratios=valid_ratios,
                            biases=(offsets_bias, logits_bias), mask=(None, 0, 0) if presum else mask, flags=flags,
                            workspace=workspace)
    if presum:
        return _frame_unsum(grad_src, mask, dims, n_frame, dt, planar), grad_proj
    return (grad_src if dt == torch.float32 else grad_src.to(dt)), grad_proj


@snippet_attn_backward.register_fake
def _(value_or_vsum, value_mask, spatial_shapes, level_start_index, proj, offsets_bias, logits_bias,
      reference_points, valid_ratios, grad_output, n_frame, presum, n_src_frames, deterministic, value_dims=None):
    if value_dims is not None:
        S, M, D = value_dims
        return value_or_vsum.new_empty((value_or_vsum.shape[0], n_src_frames, S, M, D)), torch.empty_like(proj)
    N, _, S, M, D = value_or_vsum.shape
    return value_or_vsum.new_empty((N, n_src_frames, S, M, D)), torch.empty_like(proj)


def _attn_setup_context(ctx, inputs, output):
    (value, value_mask, spatial_shapes, level_start_index, proj, ob, lb, reference_points, valid_ratios, n_frame,
     presum, planar) = inputs
    out, carry = output
    ctx.n_frame, ctx.presum, ctx.T2 = n_frame, bool(presum), value.shape[1]
    ctx.value_dims = list(value.shape[2:]) if planar else None    # the 3-d planar carry does not say
    # the presummed value replaces value itself: the backward reads nothing else of it
    ctx.save_for_backward(carry if presum else value, spatial_shapes, level_start_index, proj, reference_points,
                          valid_ratios, ob, lb, value_mask)
    ctx.set_materialize_grads(False)


def _attn_backward_formula(ctx, grad_output, grad_carry):
    value, spatial_shapes, level_start_index, proj, ref, vr, ob, lb, value_mask = ctx.saved_tensors
    if grad_output is None:
        return (None,) * 12
    if _deterministic and ctx.value_dims is not None:
        raise RuntimeError("set_deterministic(True) must be in effect during the forward as well: this graph carried planar "
                           "slots, which the deterministic two-pass backward does not walk")
    gv, gproj = torch.ops.snipper_b200.snippet_attn_backward(
        value, value_mask, spatial_shapes, level_start_index, proj, ob, lb, ref, vr, grad_output.contiguous(),
        ctx.n_frame, ctx.presum, ctx.T2, _deterministic, ctx.value_dims)
    M = gv.shape[3]
    L = spatial_shapes.shape[0]
    mlp = proj.shape[-1] // 3
    P = mlp // (M * L)
    gob = glb = gref = None
    if ctx.needs_input_grad[5] or ctx.needs_input_grad[6]:
        col = gproj.sum(dim=(0, 1, 2))                       # bias gradients = column sums of the projection gradient
        gob = col[:2 * mlp] if ctx.needs_input_grad[5] else None
        glb = col[2 * mlp:] if ctx.needs_input_grad[6] else None
    if ref is not None and ctx.needs_input_grad[7]:
        gref = _grad_ref(gproj[..., :2 * mlp].view(proj.shape[0], proj.shape[1], proj.shape[2], M, L, P, 2),
                         spatial_shapes)
    return gv, None, None, None, gproj, gob, glb, gref, None, None, None, None


snippet_attn.register_autograd(_attn_backward_formula, setup_context=_attn_setup_context)


def snippet_attention(value: Tensor, value_mask: Optional[Tensor], spatial_shapes: Tensor, level_start_index: Tensor,
                      proj: Tensor, offsets_bias: Optional[Tensor], logits_bias: Optional[Tensor],
                      reference_points: Optional[Tensor], n_frame: int, presum: Optional[bool] = None,
                      valid_ratios: Optional[Tensor] = None) -> Tensor:
    """Fused layer attention; picks the neighbour-frame strategy (``presum=None``) from the shapes.
    ``reference_points=None, valid_ratios=(N,L,2)``: encoder self-attention with in-kernel reference points."""
    N, T2, S, M, D = value.shape
    _, T1, Lq, W = proj.shape
    L = spatial_shapes.shape[0]
    if presum is None:
        presum = prefers_presum(T2, T1, n_frame, S, L, Lq, W // (3 * M * L)) or (_deterministic and torch.is_grad_enabled())
    # decided HERE, not inside the op: a custom op body runs with grad mode off
    planar = bool(presum) and use_planar(S, M, D, value.dtype)
    out, _ = torch.ops.snipper_b200.snippet_attn(value, value_mask, spatial_shapes, level_start_index, proj,
                                                 offsets_bias, logits_bias, reference_points, valid_ratios, n_frame,
                                                 bool(presum), planar)
    return out


# ------------------------------------------------------------------------------------------
# layer tail (SURVEY.md section 8f rank 3): bias + residual + LayerNorm (+ pos) in one pass
# ------------------------------------------------------------------------------------------
def layer_tail_supported(y: Tensor, residual: Tensor) -> bool:
    """fp32 CUDA rows of 128*k <= 1024 channels, inference (no autograd formula exists for this op)."""
    C = y.shape[-1]
    return (y.is_cuda and y.dtype == torch.float32 and residual.dtype == torch.float32 and C % 128 == 0 and C <= 1024
            and y.shape == residual.shape and not (torch.is_grad_enabled() and (y.requires_grad or residual.requires_grad)))


@torch.library.custom_op("snipper_b200::layer_tail", mutates_args=())
def layer_tail(y: Tensor, bias: Optional[Tensor], residual: Tensor, gamma: Tensor, beta: Tensor,
               pos: Optional[Tensor], eps: float) -> Tuple[Tensor, Tensor]:
    """(LayerNorm(residual + y + bias), that + pos) -- the second tensor is empty when ``pos`` is None.
    Reference: deformable_transformer.py:204-205 / :194-198 / :294-295 and with_pos_embed :188-190."""
    _require_cuda(y, "y")
    C = y.shape[-1]
    if y.dtype != torch.float32 or C % 128 != 0 or C > 1024 or residual.shape != y.shape:
        raise RuntimeError("layer_tail: float32 rows of 128*k <= 1024 channels, residual shaped like y")
    y, residual = y.contiguous(), residual.contiguous()
    for t, n in ((bias, C), (gamma, C), (beta, C)):
        if t is not None and (t.numel() != n or t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("layer_tail: bias / gamma / beta must be contiguous float32 vectors of C elements")
    rows = y.numel() // C
    out = torch.empty_like(y)
    if pos is not None:
        if pos.shape != y.shape or pos.dtype != torch.float32:
            raise RuntimeError("layer_tail: pos must be shaped like y")
        pos = pos.contiguous()
        out_pos = torch.empty_like(y)
    else:
        out_pos = y.new_empty((0,))
    _launch("msda_layer_tail", "layer_tail", (rows, C, int(pos is not None)), y.device,
            y.data_ptr(), _ptr(bias), residual.data_ptr(), gamma.data_ptr(), beta.data_ptr(), _ptr(pos),
            out.data_ptr(), out_pos.data_ptr() if pos is not None else None, rows, C, float(eps), capi.MSDA_DTYPE_F32)
    return out, out_pos


@layer_tail.register_fake
def _(y, bias, residual, gamma, beta, pos, eps):
    return torch.empty_like(y), (torch.empty_like(y) if pos is not None else y.new_empty((0,)))


# ------------------------------------------------------------------------------------------
# layer tail under bf16 autocast (libmsda_b200_amp.so): the block's Linear returned bf16, the residual stream stays
# fp32, and the next GEMMs want bf16 copies of the result -- written by the same pass
# ------------------------------------------------------------------------------------------
def layer_tail_amp_supported(residual: Tensor, pos: Optional[Tensor] = None) -> bool:
    """fp32 or bf16 CUDA residual rows of 128*k <= 1024 channels, ``pos`` absent or fp32 shaped like them, inference
    (no autograd formula exists for this op).  The GEMM output the op adds is bf16 rows of the same shape."""
    C = residual.shape[-1]
    return (residual.is_cuda and residual.dtype in (torch.float32, torch.bfloat16) and C % 128 == 0 and C <= 1024 and
            (pos is None or (pos.dtype == torch.float32 and pos.shape == residual.shape)) and
            not (torch.is_grad_enabled() and (residual.requires_grad or (pos is not None and pos.requires_grad))))


@torch.library.custom_op("snipper_b200::layer_tail_amp", mutates_args=())
def layer_tail_amp(y: Tensor, bias: Optional[Tensor], residual: Tensor, gamma: Tensor, beta: Tensor,
                   pos: Optional[Tensor], eps: float, emit_bf16: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """(out, out_bf16, out_pos_bf16) with out = LayerNorm(residual + (y + bias)) in fp32 -- the bits ``layer_tail``
    gives for y.float(), residual.float() -- out_bf16 = out rounded to bf16 (empty unless ``emit_bf16``) and
    out_pos_bf16 = (out + pos) rounded to bf16 (empty when ``pos`` is None).  y is bf16, residual fp32 or bf16,
    bias / gamma / beta / pos fp32."""
    _require_cuda(y, "y")
    C = y.shape[-1]
    if (y.dtype != torch.bfloat16 or residual.dtype not in (torch.float32, torch.bfloat16) or C % 128 != 0 or
            C > 1024 or residual.shape != y.shape):
        raise RuntimeError("layer_tail_amp: bfloat16 rows of 128*k <= 1024 channels, residual float32 / bfloat16 "
                           "shaped like y")
    y, residual = y.contiguous(), residual.contiguous()
    for t, n in ((bias, C), (gamma, C), (beta, C)):
        if t is not None and (t.numel() != n or t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("layer_tail_amp: bias / gamma / beta must be contiguous float32 vectors of C elements")
    rows = y.numel() // C
    out = torch.empty(y.shape, dtype=torch.float32, device=y.device)
    out_bf16 = torch.empty_like(y) if emit_bf16 else y.new_empty((0,))
    if pos is not None:
        if pos.shape != y.shape or pos.dtype != torch.float32:
            raise RuntimeError("layer_tail_amp: pos must be float32 shaped like y")
        pos = pos.contiguous()
        out_pos = torch.empty_like(y)
    else:
        out_pos = y.new_empty((0,))
    _launch("msda_amp_layer_tail", "layer_tail_amp", (rows, C, residual.element_size(), int(emit_bf16), int(pos is not None)),
            y.device,
            y.data_ptr(), _ptr(bias), residual.data_ptr(), _DTYPES[residual.dtype], gamma.data_ptr(), beta.data_ptr(),
            _ptr(pos), out.data_ptr(), out_bf16.data_ptr() if emit_bf16 else None,
            out_pos.data_ptr() if pos is not None else None, rows, C, float(eps), amp=True)
    return out, out_bf16, out_pos


@layer_tail_amp.register_fake
def _(y, bias, residual, gamma, beta, pos, eps, emit_bf16):
    return (torch.empty(y.shape, dtype=torch.float32, device=y.device),
            torch.empty_like(y) if emit_bf16 else y.new_empty((0,)),
            torch.empty_like(y) if pos is not None else y.new_empty((0,)))


# ------------------------------------------------------------------------------------------
# layer tail for training (libmsda_b200_train.so): the dropout in front of the norm applies a keep-mask the caller drew
# (snipper_b200/layers.py draws it with torch's generator), and the op has a backward of its own
# ------------------------------------------------------------------------------------------
def layer_tail_train_supported(residual: Tensor, pos: Optional[Tensor] = None) -> bool:
    """fp32 CUDA residual rows of 128*k <= 1024 channels, ``pos`` absent or fp32 shaped like them.  Autograd may record
    (the op has a gradient formula); the GEMM output the op adds is fp32 rows of the same shape."""
    C = residual.shape[-1]
    return (residual.is_cuda and residual.dtype == torch.float32 and C % 128 == 0 and C <= 1024 and
            (pos is None or (pos.dtype == torch.float32 and pos.shape == residual.shape)))


def keep_scale(p: float) -> float:
    """1 / (1 - p) rounded to float, as torch's dropout scales the kept elements."""
    return float(np.float32(1.0) / np.float32(1.0 - p))


def _dense16(t: Tensor) -> Tensor:
    """``t`` with dense rows at a 16-byte aligned address (the C ABI's layout), copied only when it is not."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _check_train_mask(keep_mask, y, p):
    if not (0.0 <= p < 1.0):
        raise RuntimeError("layer_tail_train: dropout probability must be in [0, 1)")
    if keep_mask is None:
        return None
    if keep_mask.shape != y.shape or keep_mask.dtype not in (torch.uint8, torch.bool) or not keep_mask.is_cuda:
        raise RuntimeError("layer_tail_train: keep_mask must be a uint8 / bool CUDA tensor shaped like y")
    return _dense16(keep_mask.view(torch.uint8) if keep_mask.dtype == torch.bool else keep_mask)


@torch.library.custom_op("snipper_b200::layer_tail_train", mutates_args=())
def layer_tail_train(y: Tensor, bias: Optional[Tensor], residual: Tensor, keep_mask: Optional[Tensor], p: float,
                     gamma: Tensor, beta: Tensor, pos: Optional[Tensor], eps: float
                     ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """(out, out_pos, h, mean_rstd): h = residual + d with d = ((y + bias) * keep_scale(p)) * keep_mask, or y + bias
    without a mask; out = LayerNorm(h) * gamma + beta; out_pos = out + pos (empty when ``pos`` is None); mean_rstd the
    (mean, rstd) of every row, shaped (..., 2).  h and mean_rstd are what the backward reads.  Without a mask ``out``
    has the bits of ``layer_tail``; with one, the bits ``layer_tail`` gives for the pre-dropped input and no bias."""
    _require_cuda(y, "y")
    C = y.shape[-1]
    if (y.dtype != torch.float32 or residual.dtype != torch.float32 or C % 128 != 0 or C > 1024 or
            residual.shape != y.shape):
        raise RuntimeError("layer_tail_train: float32 rows of 128*k <= 1024 channels, residual shaped like y")
    keep_mask = _check_train_mask(keep_mask, y, p)
    y, residual = _dense16(y), _dense16(residual)
    for t in (bias, gamma, beta):
        if t is not None and (t.numel() != C or t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("layer_tail_train: bias / gamma / beta must be contiguous float32 vectors of C elements")
    # locals: an aligned copy must stay alive until the kernel that reads it has run
    bias = _dense16(bias) if bias is not None else None
    gamma, beta = _dense16(gamma), _dense16(beta)
    rows = y.numel() // C
    out, h = torch.empty_like(y), torch.empty_like(y)
    mean_rstd = y.new_empty((*y.shape[:-1], 2))
    if pos is not None:
        if pos.shape != y.shape or pos.dtype != torch.float32:
            raise RuntimeError("layer_tail_train: pos must be float32 shaped like y")
        pos = _dense16(pos)
        out_pos = torch.empty_like(y)
    else:
        out_pos = y.new_empty((0,))
    _launch("msda_train_layer_tail_forward", "layer_tail_train", (rows, C, int(keep_mask is not None), int(pos is not None)),
            y.device, y.data_ptr(), _ptr(bias), residual.data_ptr(), _ptr(keep_mask),
            keep_scale(p) if keep_mask is not None else 1.0, gamma.data_ptr(), beta.data_ptr(),
            _ptr(pos), out.data_ptr(), out_pos.data_ptr() if pos is not None else None, h.data_ptr(),
            mean_rstd.data_ptr(), rows, C, float(eps), train=True)
    return out, out_pos, h, mean_rstd


@layer_tail_train.register_fake
def _(y, bias, residual, keep_mask, p, gamma, beta, pos, eps):
    return (torch.empty_like(y), torch.empty_like(y) if pos is not None else y.new_empty((0,)), torch.empty_like(y),
            y.new_empty((*y.shape[:-1], 2)))


@torch.library.custom_op("snipper_b200::layer_tail_train_backward", mutates_args=())
def layer_tail_train_backward(grad_out: Tensor, grad_out_pos: Optional[Tensor], h: Tensor, mean_rstd: Tensor,
                              keep_mask: Optional[Tensor], p: float, gamma: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """(grad_residual, grad_y, param_grads): param_grads is (3, C) = (grad_gamma, grad_beta, grad_bias), reduced in a
    fixed order without atomics, so two calls on the same inputs give the same bits.  grad_y is also the gradient of
    y + bias; with no mask it equals grad_residual."""
    _require_cuda(h, "h")
    C = h.shape[-1]
    if (h.dtype != torch.float32 or C % 128 != 0 or C > 1024 or grad_out.shape != h.shape or
            grad_out.dtype != torch.float32 or mean_rstd.shape != (*h.shape[:-1], 2) or
            (grad_out_pos is not None and (grad_out_pos.shape != h.shape or grad_out_pos.dtype != torch.float32))):
        raise RuntimeError("layer_tail_train_backward: float32 rows of 128*k <= 1024 channels, gradients shaped like h, "
                           "mean_rstd (..., 2)")
    if gamma.numel() != C or gamma.dtype != torch.float32:
        raise RuntimeError("layer_tail_train_backward: gamma must be a float32 vector of C elements")
    keep_mask = _check_train_mask(keep_mask, h, p)
    rows = h.numel() // C
    grad_out, h, mean_rstd, gamma = _dense16(grad_out), _dense16(h), _dense16(mean_rstd), _dense16(gamma)
    if grad_out_pos is not None:
        grad_out_pos = _dense16(grad_out_pos)
    grad_residual, grad_y = torch.empty_like(h), torch.empty_like(h)
    # the parameter gradients get a tensor of their own: autograd may keep them as .grad, the partials go with the call
    param_grads = torch.zeros((3, C), dtype=torch.float32, device=h.device) if rows == 0 else \
        torch.empty((3, C), dtype=torch.float32, device=h.device)
    ws_bytes = capi.train_lib().msda_train_layer_tail_workspace_bytes(rows, C)
    ws = torch.empty(max(ws_bytes // 4, 1), dtype=torch.float32, device=h.device)
    _launch("msda_train_layer_tail_backward", "layer_tail_train_backward",
            (rows, C, int(keep_mask is not None), int(grad_out_pos is not None)), h.device,
            grad_out.data_ptr(), _ptr(grad_out_pos), h.data_ptr(), mean_rstd.data_ptr(), _ptr(keep_mask),
            keep_scale(p) if keep_mask is not None else 1.0, gamma.data_ptr(), grad_residual.data_ptr(),
            grad_y.data_ptr(), param_grads.data_ptr(), ws.data_ptr(), rows, C, n_kernels=2, train=True)
    return grad_residual, grad_y, param_grads


@layer_tail_train_backward.register_fake
def _(grad_out, grad_out_pos, h, mean_rstd, keep_mask, p, gamma):
    return torch.empty_like(h), torch.empty_like(h), h.new_empty((3, h.shape[-1]))


def _tail_train_setup_context(ctx, inputs, output):
    y, bias, residual, keep_mask, p, gamma, beta, pos, eps = inputs
    out, out_pos, h, mean_rstd = output
    ctx.p, ctx.has_bias, ctx.has_pos = p, bias is not None, pos is not None
    # what stock saves for the same block: dropout its mask, layer_norm its input and (mean, rstd)
    ctx.save_for_backward(h, mean_rstd, keep_mask, gamma)
    ctx.set_materialize_grads(False)


def _tail_train_backward_formula(ctx, grad_out, grad_out_pos, grad_h, grad_mean_rstd):
    h, mean_rstd, keep_mask, gamma = ctx.saved_tensors
    if not ctx.has_pos:
        grad_out_pos = None
    if grad_out is None and grad_out_pos is None:
        return (None,) * 9
    if grad_out is None:
        grad_out = torch.zeros_like(h)
    grad_residual, grad_y, pg = torch.ops.snipper_b200.layer_tail_train_backward(
        grad_out, grad_out_pos, h, mean_rstd, keep_mask, ctx.p, gamma)
    return (grad_y, pg[2] if ctx.has_bias else None, grad_residual, None, None, pg[0], pg[1], grad_out_pos, None)


layer_tail_train.register_autograd(_tail_train_backward_formula, setup_context=_tail_train_setup_context)


# ------------------------------------------------------------------------------------------
# layer tail for training under bf16 autocast (libmsda_b200_amp_train.so): layer_tail_train's dropout, saved h and
# (mean, rstd) and ordered parameter-gradient sum, with layer_tail_amp's bf16 GEMM output in and bf16 copies out
# ------------------------------------------------------------------------------------------
def layer_tail_amp_train_supported(residual: Tensor, pos: Optional[Tensor] = None) -> bool:
    """fp32 or bf16 CUDA residual rows of 128*k <= 1024 channels, ``pos`` absent or fp32 shaped like them.  Autograd
    may record (the op has a gradient formula); the GEMM output the op adds is bf16 rows of the same shape."""
    C = residual.shape[-1]
    return (residual.is_cuda and residual.dtype in (torch.float32, torch.bfloat16) and C % 128 == 0 and C <= 1024 and
            (pos is None or (pos.dtype == torch.float32 and pos.shape == residual.shape)))


@torch.library.custom_op("snipper_b200::layer_tail_amp_train", mutates_args=())
def layer_tail_amp_train(y: Tensor, bias: Optional[Tensor], residual: Tensor, keep_mask: Optional[Tensor], p: float,
                         gamma: Tensor, beta: Tensor, pos: Optional[Tensor], eps: float, emit_bf16: bool
                         ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """(out, out_bf16, out_pos_bf16, h, mean_rstd): ``layer_tail_train`` on y.float(), residual.float() -- out, h and
    mean_rstd have its bits -- with out_bf16 = out rounded to bf16 (empty unless ``emit_bf16``) and out_pos_bf16 =
    (out + pos) rounded to bf16 (empty when ``pos`` is None).  y is bf16, residual fp32 or bf16, bias / gamma / beta /
    pos fp32."""
    _require_cuda(y, "y")
    C = y.shape[-1]
    if (y.dtype != torch.bfloat16 or residual.dtype not in (torch.float32, torch.bfloat16) or C % 128 != 0 or
            C > 1024 or residual.shape != y.shape):
        raise RuntimeError("layer_tail_amp_train: bfloat16 rows of 128*k <= 1024 channels, residual float32 / "
                           "bfloat16 shaped like y")
    keep_mask = _check_train_mask(keep_mask, y, p)
    y, residual = _dense16(y), _dense16(residual)
    for t in (bias, gamma, beta):
        if t is not None and (t.numel() != C or t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("layer_tail_amp_train: bias / gamma / beta must be contiguous float32 vectors of C "
                               "elements")
    # locals: an aligned copy must stay alive until the kernel that reads it has been enqueued
    bias = _dense16(bias) if bias is not None else None
    gamma, beta = _dense16(gamma), _dense16(beta)
    rows = y.numel() // C
    out = torch.empty(y.shape, dtype=torch.float32, device=y.device)
    h = torch.empty_like(out)
    mean_rstd = out.new_empty((*y.shape[:-1], 2))
    out_bf16 = torch.empty_like(y) if emit_bf16 else y.new_empty((0,))
    if pos is not None:
        if pos.shape != y.shape or pos.dtype != torch.float32:
            raise RuntimeError("layer_tail_amp_train: pos must be float32 shaped like y")
        pos = _dense16(pos)
        out_pos = torch.empty_like(y)
    else:
        out_pos = y.new_empty((0,))
    _launch("msda_amp_train_layer_tail_forward", "layer_tail_amp_train",
            (rows, C, residual.element_size(), int(keep_mask is not None), int(emit_bf16), int(pos is not None)),
            y.device, y.data_ptr(), _ptr(bias), residual.data_ptr(), _DTYPES[residual.dtype], _ptr(keep_mask),
            keep_scale(p) if keep_mask is not None else 1.0, gamma.data_ptr(), beta.data_ptr(), _ptr(pos),
            out.data_ptr(), out_bf16.data_ptr() if emit_bf16 else None,
            out_pos.data_ptr() if pos is not None else None, h.data_ptr(), mean_rstd.data_ptr(), rows, C, float(eps),
            amp=True, train=True)
    return out, out_bf16, out_pos, h, mean_rstd


@layer_tail_amp_train.register_fake
def _(y, bias, residual, keep_mask, p, gamma, beta, pos, eps, emit_bf16):
    out = torch.empty(y.shape, dtype=torch.float32, device=y.device)
    return (out, torch.empty_like(y) if emit_bf16 else y.new_empty((0,)),
            torch.empty_like(y) if pos is not None else y.new_empty((0,)), torch.empty_like(out),
            out.new_empty((*y.shape[:-1], 2)))


@torch.library.custom_op("snipper_b200::layer_tail_amp_train_backward", mutates_args=())
def layer_tail_amp_train_backward(grad_out: Tensor, grad_out_bf16: Optional[Tensor], grad_out_pos_bf16: Optional[Tensor],
                                  h: Tensor, mean_rstd: Tensor, keep_mask: Optional[Tensor], p: float, gamma: Tensor,
                                  residual_bf16: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """(grad_residual, grad_y, param_grads) of ``layer_tail_amp_train`` for the incoming gradients grad_out (fp32) and
    the optional bf16 grad_out_bf16 / grad_out_pos_bf16 of its bf16 copies, added as (grad_out + grad_out_bf16) +
    grad_out_pos_bf16 in fp32.  grad_residual is bf16 when ``residual_bf16`` (else fp32) and grad_y bf16, each rounded
    once from fp32; param_grads is (3, C) fp32 = (grad_gamma, grad_beta, grad_bias), with grad_bias summed from the fp32
    grad_y, reduced in a fixed order without atomics."""
    _require_cuda(h, "h")
    C = h.shape[-1]
    if (h.dtype != torch.float32 or C % 128 != 0 or C > 1024 or grad_out.shape != h.shape or
            grad_out.dtype != torch.float32 or mean_rstd.shape != (*h.shape[:-1], 2) or
            any(g is not None and (g.shape != h.shape or g.dtype != torch.bfloat16)
                for g in (grad_out_bf16, grad_out_pos_bf16))):
        raise RuntimeError("layer_tail_amp_train_backward: float32 rows of 128*k <= 1024 channels, grad_out float32 "
                           "and the optional bf16 gradients shaped like h, mean_rstd (..., 2)")
    if gamma.numel() != C or gamma.dtype != torch.float32:
        raise RuntimeError("layer_tail_amp_train_backward: gamma must be a float32 vector of C elements")
    keep_mask = _check_train_mask(keep_mask, h, p)
    rows = h.numel() // C
    grad_out, h, mean_rstd, gamma = _dense16(grad_out), _dense16(h), _dense16(mean_rstd), _dense16(gamma)
    grad_out_bf16 = _dense16(grad_out_bf16) if grad_out_bf16 is not None else None
    grad_out_pos_bf16 = _dense16(grad_out_pos_bf16) if grad_out_pos_bf16 is not None else None
    rdt = torch.bfloat16 if residual_bf16 else torch.float32
    grad_residual = torch.empty(h.shape, dtype=rdt, device=h.device)
    grad_y = torch.empty(h.shape, dtype=torch.bfloat16, device=h.device)
    param_grads = torch.zeros((3, C), dtype=torch.float32, device=h.device) if rows == 0 else \
        torch.empty((3, C), dtype=torch.float32, device=h.device)
    ws_bytes = capi.amp_train_lib().msda_amp_train_layer_tail_workspace_bytes(rows, C)
    ws = torch.empty(max(ws_bytes // 4, 1), dtype=torch.float32, device=h.device)
    _launch("msda_amp_train_layer_tail_backward", "layer_tail_amp_train_backward",
            (rows, C, grad_residual.element_size(), int(keep_mask is not None), int(grad_out_bf16 is not None),
             int(grad_out_pos_bf16 is not None)), h.device,
            grad_out.data_ptr(), _ptr(grad_out_bf16), _ptr(grad_out_pos_bf16), h.data_ptr(), mean_rstd.data_ptr(),
            _ptr(keep_mask), keep_scale(p) if keep_mask is not None else 1.0, gamma.data_ptr(),
            grad_residual.data_ptr(), _DTYPES[rdt], grad_y.data_ptr(), param_grads.data_ptr(), ws.data_ptr(), rows, C,
            n_kernels=2, amp=True, train=True)
    return grad_residual, grad_y, param_grads


@layer_tail_amp_train_backward.register_fake
def _(grad_out, grad_out_bf16, grad_out_pos_bf16, h, mean_rstd, keep_mask, p, gamma, residual_bf16):
    return (torch.empty(h.shape, dtype=torch.bfloat16 if residual_bf16 else torch.float32, device=h.device),
            torch.empty(h.shape, dtype=torch.bfloat16, device=h.device), h.new_empty((3, h.shape[-1])))


def _tail_amp_train_setup_context(ctx, inputs, output):
    y, bias, residual, keep_mask, p, gamma, beta, pos, eps, emit_bf16 = inputs
    out, out_bf16, out_pos, h, mean_rstd = output
    ctx.p, ctx.has_bias, ctx.has_pos, ctx.emit_bf16 = p, bias is not None, pos is not None, emit_bf16
    ctx.residual_bf16 = residual.dtype == torch.bfloat16
    # what stock autocast saves for the same block: dropout its mask, layer_norm its fp32 input and (mean, rstd)
    ctx.save_for_backward(h, mean_rstd, keep_mask, gamma)
    ctx.set_materialize_grads(False)


def _tail_amp_train_backward_formula(ctx, grad_out, grad_out_bf16, grad_out_pos, grad_h, grad_mean_rstd):
    h, mean_rstd, keep_mask, gamma = ctx.saved_tensors
    if not ctx.emit_bf16:
        grad_out_bf16 = None
    if not ctx.has_pos:
        grad_out_pos = None
    if grad_out is None and grad_out_bf16 is None and grad_out_pos is None:
        return (None,) * 10
    if grad_out is None:
        grad_out = torch.zeros_like(h)
    grad_residual, grad_y, pg = torch.ops.snipper_b200.layer_tail_amp_train_backward(
        grad_out, grad_out_bf16, grad_out_pos, h, mean_rstd, keep_mask, ctx.p, gamma, ctx.residual_bf16)
    # out_pos_bf16 = bf16(out + pos): pos gets the gradient of that copy, in pos's dtype
    grad_pos = grad_out_pos.float() if (grad_out_pos is not None and ctx.needs_input_grad[7]) else None
    return (grad_y, pg[2] if ctx.has_bias else None, grad_residual, None, None, pg[0], pg[1], grad_pos, None, None)


layer_tail_amp_train.register_autograd(_tail_amp_train_backward_formula, setup_context=_tail_amp_train_setup_context)
