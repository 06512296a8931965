"""Opt-in fused LAYER TAILS for the callers of ``MSDeformAttn`` (SURVEY.md section 8f rank 3).

The reference's encoder / decoder layers (models/deformable_transformer.py:170-210, :244-300) end every
attention block and every FFN block with ``x = x + dropout(Linear(..)); x = norm(x)`` and begin the next
attention block with ``with_pos_embed(x, pos)``.  ``enable_fused_layer_tails(model)`` rebinds the ``forward``
of those layer objects (module tree, parameters and state-dict keys untouched -- a reference checkpoint still
loads) to a version that

  * takes ``MSDeformAttn``'s output before ``output_proj``'s bias and folds bias + residual + LayerNorm into
    ONE kernel pass (``msda_layer_tail``), likewise for the FFN's second Linear;
  * lets the last tail of a layer also emit ``x + pos``, the next layer's query, so the separate
    ``with_pos_embed`` pass disappears;
  * runs ``relu(linear1(x))`` as one cuBLASLt call with a bias+ReLU epilogue (stock library, no extra pass);
  * makes the ENCODER hand its layers an ``EncoderGrid`` instead of the materialised reference-point tensor
    (get_reference_points, :219-232), so the fused kernels compute the reference points from the query index
    (SURVEY.md section 8f rank 2).

``_eligible`` alone decides, per call, which of five forwards runs:

  * the layer's ORIGINAL forward (stock);
  * the fp32 tails (``layer_tail``), when autocast is off for CUDA and the residual stream is fp32 on CUDA with
    C = 128*k <= 1024 channels (what the kernel covers);
  * the bf16 autocast tails (``layer_tail_amp``, libmsda_b200_amp.so), when the layer was switched with
    ``enable_fused_layer_tails(model, autocast=True)``, autocast is on for CUDA with dtype bfloat16, the residual
    stream is fp32 or bf16 on CUDA with C = 128*k <= 1024, and ``pos`` / ``query_pos`` is absent or fp32.  The GEMM
    in front of each tail returns bf16 there; the tail reads it, writes the fp32 residual stream (what autocast's
    fp32 LayerNorm gives) and, in the same pass, the bf16 copies the next GEMMs take -- ``linear1``'s input, and the
    next encoder layer's ``value_proj`` input and query (the decoder's cross-attention query) -- with exactly the
    bits autocast's own cast would give them.  The FFN's first GEMM then runs in bf16 with its bias + ReLU
    epilogue.  The result is not bit-identical to the stock autocast network (the output_proj / linear2 bias is
    added in fp32 rather than in a bf16 GEMM epilogue, and the LayerNorm sums in another order), which is why it
    is opt-in per model.  Autocast to float16 keeps the stock layers.
  * the training tails (``layer_tail_train``, libmsda_b200_train.so), when the layer was switched with
    ``enable_fused_layer_tails(model, training=True)`` and neither inference forward applies -- see below;
  * the bf16 autocast training tails (``layer_tail_amp_train``, libmsda_b200_amp_train.so), when the layer was switched
    with ``enable_fused_layer_tails(model, amp_training=True)`` and neither inference forward applies -- see below.

Both inference forwards further need all of these:

  * nothing would need a gradient: grad mode is off, or no parameter of the layer and no tensor argument of its
    forward (src / tgt, pos / query_pos, reference points, the decoder's src, masks) requires grad -- the tail
    ops have no autograd formula;
  * every dropout of the layer is inactive (p = 0 or eval mode);
  * the FFN activation is ReLU (``layer.activation is F.relu`` where the layer has one, as the reference's do);
  * every norm is an ``nn.LayerNorm`` with both weight and bias, and ``linear1`` has a bias.

In every other situation the layer's ORIGINAL forward runs, so training, fp16 autocast and any layer variant keep
exactly the stock behaviour -- unless the layer opted in to the training tails.  Those run while autograd records and
while dropouts are active, when autocast is off for CUDA, the residual stream is fp32 on CUDA with C = 128*k <= 1024,
``pos`` / ``query_pos`` is absent or fp32, the activation is ReLU, the norms are affine, ``linear1`` has a bias and
every tail dropout (the one in front of each norm: encoder ``dropout1``, ``dropout3``; decoder ``dropout2``,
``dropout1``, ``dropout4``) has p < 1 (or is in eval mode).  Each tail draws its dropout keep-mask with
``draw_keep_mask`` -- torch's generator, so ``torch.manual_seed`` repeats a step -- and the kernels only read it.  No
mask is drawn in eval mode or at p = 0.  The FFN's inner dropout and the decoder's ``nn.MultiheadAttention`` stay
stock, and the FFN's first GEMM is ``relu(linear(x, w, b))`` (``_addmm_activation`` has no derivative).  The stock
layers draw their masks from the same generator in another order and another dtype, so a step is not bit-identical
to the stock one; it computes the same function of its masks (tests/test_layer_tails_train_gpu.py).

The bf16 autocast training tails follow the same rules under ``torch.autocast("cuda", dtype=torch.bfloat16)``, with
the amp tails' I/O: the residual stream is fp32 or bf16, the GEMM in front of each tail returns bf16, and each tail
also writes, with exactly autocast's rounding, the bf16 copies the next GEMMs take (``linear1``'s input, the next
encoder layer's ``value_proj`` input and query, the decoder's cross-attention query).  ``linear1`` runs as
``relu(linear(x16, w, b))``, autocast casting w and b.  The gradient of the GEMM output is bf16, rounded once from
fp32; the output_proj / linear2 bias gradient is summed from the fp32 values before that rounding, where stock autocast
sums the bf16 GEMM-output gradient (tests/test_layer_tails_amp_train_gpu.py).  The new keyword is needed because
``autocast=True, training=True`` keeps the stock layers in autocast training.  fp16 autocast keeps the stock layers.
Works on the reference's own layer classes (after ``install_module()``) and on the bench harness' layers: both
expose the reference's attribute names (self_attn / cross_attn, norm1..3, linear1/2, dropout1..4).
"""
import types

import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from .modules import EncoderGrid, MSDeformAttn

_PLUS_POS = "_snipper_b200_plus_pos"   # attribute on a layer's output tensor: (pos tensor, output + pos)
_AS_BF16 = "_snipper_b200_as_bf16"     # attribute on an amp layer's output tensor: the output rounded to bf16


def _dropout_off(layer):
    return not any(isinstance(m, nn.Dropout) and m.p > 0 and m.training for m in layer.children())


def _affine_layer_norm(norm):
    return isinstance(norm, nn.LayerNorm) and norm.weight is not None and norm.bias is not None


def _eligible(layer, x, pos, *inputs):
    """Which forward computes what ``layer``'s own forward would (the module docstring lists the conditions):
    None (the layer's own), "fp32", "amp", "train" or "amp_train".  ``x`` is the residual stream, ``pos`` the positional
    embedding (``pos`` / ``query_pos``), ``inputs`` every other argument of the layer's forward."""
    path = _inference_path(layer, x, pos, *inputs)
    return path if path is not None else _train_path(layer, x, pos)


def _inference_path(layer, x, pos, *inputs):
    """None, "fp32" or "amp": the inference forwards' conditions."""
    if torch.is_autocast_enabled("cuda"):
        if not (getattr(layer, "_amp_tails", False) and torch.get_autocast_dtype("cuda") == torch.bfloat16 and
                ops.layer_tail_amp_supported(x, pos)):
            return None
        path = "amp"
    elif ops.layer_tail_supported(x, x):
        path = "fp32"
    else:
        return None
    if not _dropout_off(layer):
        return None
    if torch.is_grad_enabled() and (any(p.requires_grad for p in layer.parameters()) or
                                    any(torch.is_tensor(t) and t.requires_grad for t in (pos,) + inputs)):
        return None
    return path if _fusable_structure(layer) else None


def _fusable_structure(layer):
    """ReLU FFN, affine norms, a bias on linear1."""
    norms = [getattr(layer, n) for n in ("norm1", "norm2", "norm3") if hasattr(layer, n)]
    return (getattr(layer, "activation", F.relu) is F.relu and all(_affine_layer_norm(n) for n in norms) and
            layer.linear1.bias is not None)


# the dropout in front of each norm, in the order the layer's tails run
_TAIL_DROPOUTS = {"encoder": ("dropout1", "dropout3"), "decoder": ("dropout2", "dropout1", "dropout4")}


def _train_path(layer, x, pos):
    """None, "train" or "amp_train": the training forwards' conditions."""
    if torch.is_autocast_enabled("cuda"):
        if not (getattr(layer, "_amp_train_tails", False) and torch.get_autocast_dtype("cuda") == torch.bfloat16 and
                ops.layer_tail_amp_train_supported(x, pos)):
            return None
        path = "amp_train"
    elif getattr(layer, "_train_tails", False) and ops.layer_tail_train_supported(x, pos):
        path = "train"
    else:
        return None
    drops = [getattr(layer, n, None) for n in _TAIL_DROPOUTS["decoder" if hasattr(layer, "cross_attn") else "encoder"]]
    if not all(isinstance(d, nn.Dropout) and _dropout_p(d) < 1 for d in drops):
        return None
    return path if _fusable_structure(layer) else None


def _dropout_p(dropout):
    return dropout.p if dropout.training else 0.0


def draw_keep_mask(shape, p, device):
    """The keep-mask of a training tail's dropout: one byte per element, 1 with probability 1 - p, drawn by torch's
    generator (``torch.manual_seed`` repeats it; CUDA RNG state stays torch's).  Every training tail draws through
    this function, so a test can substitute a recorder for it."""
    return torch.empty(shape, dtype=torch.uint8, device=device).bernoulli_(1 - p)


def _train_tail(y, bias, residual, dropout, norm, pos=None, amp=False, emit_bf16=False):
    """_tail with ``dropout`` before the residual add, differentiable: -> (norm(residual + dropout(y + bias)) in fp32,
    that in bf16 or None, that + pos or None).  ``amp``: y is a bf16 GEMM output; out + pos is then returned in bf16
    and ``emit_bf16`` asks for the bf16 copy of out."""
    p = _dropout_p(dropout)
    mask = draw_keep_mask(y.shape, p, y.device) if p > 0 else None
    if amp:
        out, out16, out_pos, _, _ = torch.ops.snipper_b200.layer_tail_amp_train(
            y, bias, residual, mask, float(p), norm.weight, norm.bias, pos, norm.eps, emit_bf16)
        return out, (out16 if emit_bf16 else None), (out_pos if pos is not None else None)
    out, out_pos, _, _ = torch.ops.snipper_b200.layer_tail_train(y, bias, residual, mask, float(p), norm.weight,
                                                                 norm.bias, pos, norm.eps)
    return out, None, (out_pos if pos is not None else None)


def _tail(y, bias, residual, norm, pos=None, amp=False, emit_bf16=False):
    """-> (out fp32, out in bf16 or None, out + pos or None).  ``amp``: y is a bf16 GEMM output; out + pos is then
    returned in bf16 and ``emit_bf16`` asks for the bf16 copy of out."""
    if amp:
        out, out16, out_pos = torch.ops.snipper_b200.layer_tail_amp(y, bias, residual, norm.weight, norm.bias, pos,
                                                                    norm.eps, emit_bf16)
        return out, (out16 if emit_bf16 else None), (out_pos if pos is not None else None)
    out, out_pos = torch.ops.snipper_b200.layer_tail(y, bias, residual, norm.weight, norm.bias, pos, norm.eps)
    return out, None, (out_pos if pos is not None else None)


def _ffn_hidden(layer, x):
    """relu(linear1(x)) with the bias + ReLU applied in the GEMM epilogue.  A bf16 ``x`` (an amp tail's copy) makes
    it a bf16 GEMM: ``_addmm_activation`` is not on autocast's cast list, so the weight and bias are rounded here as
    autocast would round them."""
    c = x.shape[-1]
    w, b = layer.linear1.weight, layer.linear1.bias
    if x.dtype != w.dtype:
        w, b = w.to(x.dtype), b.to(x.dtype)
    return torch._addmm_activation(b, x.reshape(-1, c), w.t())


def _with_pos(x, pos, amp):
    """x + pos, taken from the previous layer's tail when it already produced it for this very ``pos`` (in bf16 on
    the ``amp`` path, where the query only feeds a bf16 GEMM; else in fp32)."""
    if pos is None:
        return x
    cached = getattr(x, _PLUS_POS, None)
    if cached is not None and cached[0] is pos and (cached[1].dtype == torch.bfloat16) == amp:
        return cached[1]
    return x + pos


def _encoder_forward(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask=None):
    """reference deformable_transformer.py:200-210 (forward) and :192-198 (forward_ffn)"""
    path = _eligible(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask)
    if path is None:
        return self._stock_forward(src, pos, reference_points, spatial_shapes, level_start_index, padding_mask)
    if path in ("train", "amp_train"):
        return _encoder_train_forward(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask,
                                      amp=path == "amp_train")
    amp = path == "amp"
    attn = self.self_attn
    value_in = getattr(src, _AS_BF16, src) if amp else src                   # the previous amp tail's bf16 copy
    core, _ = attn._attend(_with_pos(src, pos, amp), reference_points, value_in, spatial_shapes, level_start_index,
                           padding_mask)
    y = F.linear(core, attn.output_proj.weight)                              # bias joins the tail
    x, x16, _ = _tail(y, attn.output_proj.bias, src, self.norm1, amp=amp, emit_bf16=amp)   # :204-205
    ff = F.linear(_ffn_hidden(self, x16 if amp else x), self.linear2.weight).view_as(x)  # :194
    emit = pos if (self._emit_next_query and pos is not None) else None
    out, out16, out_pos = _tail(ff, self.linear2.bias, x, self.norm2, emit,  # :195-197 (+ the next layer's :202)
                                amp=amp, emit_bf16=amp and self._emit_next_query)
    if out_pos is not None:
        setattr(out, _PLUS_POS, (pos, out_pos))
    if out16 is not None:
        setattr(out, _AS_BF16, out16)
    return out


def _decoder_forward(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                     src_padding_mask=None):
    """reference deformable_transformer.py:279-300 (forward) and :268-274 (forward_ffn)"""
    path = _eligible(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                     src_padding_mask)
    if path is None:
        return self._stock_forward(tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                                   src_padding_mask)
    if path in ("train", "amp_train"):
        return _decoder_train_forward(self, tgt, query_pos, reference_points, src, src_spatial_shapes,
                                      level_start_index, src_padding_mask, amp=path == "amp_train")
    amp = path == "amp"
    bs, t, lq, c = tgt.shape
    x = tgt.reshape(bs, t * lq, c)
    qp = None if query_pos is None else query_pos.reshape(bs, t * lq, c)
    qk = (x if qp is None else x + qp).transpose(0, 1)
    sa = self.self_attn(qk, qk, x.transpose(0, 1))[0].transpose(0, 1)        # :285 (nn.MultiheadAttention, stock)
    x, _, xq = _tail(sa, None, x, self.norm2, qp, amp=amp)                   # :286-287 (+ with_pos_embed of :292)
    q = (x if xq is None else xq).view(bs, t, lq, c)
    x = x.view(bs, t, lq, c)
    attn = self.cross_attn
    core, vis = attn._attend(q, reference_points, src, src_spatial_shapes, level_start_index, src_padding_mask)
    y = F.linear(core, attn.output_proj.weight)
    x, x16, _ = _tail(y, attn.output_proj.bias, x, self.norm1, amp=amp, emit_bf16=amp)   # :294-295
    ff = F.linear(_ffn_hidden(self, x16 if amp else x), self.linear2.weight).view_as(x)  # :270
    out, _, _ = _tail(ff, self.linear2.bias, x, self.norm3, amp=amp)         # :271-273
    return out, vis


def _encoder_train_forward(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask,
                           amp=False):
    """_encoder_forward with dropout and autograd: the tails apply dropout1 / dropout3.  ``amp``: under bf16 autocast,
    the tails hand their bf16 copies to linear1 and to the next layer, as on the amp inference path."""
    attn = self.self_attn
    value_in = getattr(src, _AS_BF16, src) if amp else src                   # the previous amp tail's bf16 copy
    core, _ = attn._attend(_with_pos(src, pos, amp), reference_points, value_in, spatial_shapes, level_start_index,
                           padding_mask)
    y = F.linear(core, attn.output_proj.weight)
    x, x16, _ = _train_tail(y, attn.output_proj.bias, src, self.dropout1, self.norm1, amp=amp,
                            emit_bf16=amp)                                                    # :204-205
    hidden = F.relu(F.linear(x16 if amp else x, self.linear1.weight, self.linear1.bias))
    ff = F.linear(self.dropout2(hidden), self.linear2.weight)                                 # :194
    emit = pos if (self._emit_next_query and pos is not None) else None
    out, out16, out_pos = _train_tail(ff, self.linear2.bias, x, self.dropout3, self.norm2, emit, amp=amp,
                                      emit_bf16=amp and self._emit_next_query)              # :195-197 (+ :202)
    if out_pos is not None:
        setattr(out, _PLUS_POS, (pos, out_pos))
    if out16 is not None:
        setattr(out, _AS_BF16, out16)
    return out


def _decoder_train_forward(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                           src_padding_mask, amp=False):
    """_decoder_forward with dropout and autograd: the tails apply dropout2 / dropout1 / dropout4.  ``amp``: under bf16
    autocast, the cross-attention query and linear1's input are the tails' bf16 copies."""
    bs, t, lq, c = tgt.shape
    x = tgt.reshape(bs, t * lq, c)
    qp = None if query_pos is None else query_pos.reshape(bs, t * lq, c)
    qk = (x if qp is None else x + qp).transpose(0, 1)
    sa = self.self_attn(qk, qk, x.transpose(0, 1))[0].transpose(0, 1)        # :285 (nn.MultiheadAttention, stock)
    x, _, xq = _train_tail(sa, None, x, self.dropout2, self.norm2, qp, amp=amp)  # :286-287 (+ with_pos_embed of :292)
    q = (x if xq is None else xq).view(bs, t, lq, c)
    x = x.view(bs, t, lq, c)
    attn = self.cross_attn
    core, vis = attn._attend(q, reference_points, src, src_spatial_shapes, level_start_index, src_padding_mask)
    y = F.linear(core, attn.output_proj.weight)
    x, x16, _ = _train_tail(y, attn.output_proj.bias, x, self.dropout1, self.norm1, amp=amp,
                            emit_bf16=amp)                                                    # :294-295
    hidden = F.relu(F.linear(x16 if amp else x, self.linear1.weight, self.linear1.bias))
    ff = F.linear(self.dropout3(hidden), self.linear2.weight)                                 # :270
    out, _, _ = _train_tail(ff, self.linear2.bias, x, self.dropout4, self.norm3, amp=amp)    # :271-273
    return out, vis


def _reference_encoder_forward(self, src, spatial_shapes, level_start_index, valid_ratios, pos=None, padding_mask=None,
                               n_frame=1):
    """reference DeformableTransformerEncoder.forward (deformable_transformer.py:234-241) without building the
    (N,T,S,L,2) reference-point tensor: the layers receive its closed form (``EncoderGrid``)."""
    if not (torch.is_tensor(spatial_shapes) and
            _eligible(self.layers[0], src, pos, valid_ratios, spatial_shapes, level_start_index, padding_mask)):
        return self._stock_forward(src, spatial_shapes, level_start_index, valid_ratios, pos, padding_mask, n_frame)
    grid = EncoderGrid(valid_ratios, _sizes_of(self, spatial_shapes), n_frame)
    output = src
    for layer in self.layers:
        output = layer(output, pos, grid, spatial_shapes, level_start_index, padding_mask)
    return output


def _sizes_of(encoder, spatial_shapes):
    """Python (H, W) pairs of a device shape tensor, read back ONCE per distinct tensor contents holder (the reference
    itself iterates the device tensor in get_reference_points, i.e. synchronises every forward)."""
    key = (spatial_shapes.data_ptr(), spatial_shapes._version, tuple(spatial_shapes.shape))
    cache = encoder.__dict__.setdefault("_snipper_b200_sizes", {})
    if key not in cache:
        cache.clear()
        cache[key] = [tuple(int(v) for v in row) for row in spatial_shapes.tolist()]
    return cache[key]


def _is_encoder_layer(m):
    return (isinstance(getattr(m, "self_attn", None), MSDeformAttn) and not hasattr(m, "cross_attn") and
            all(hasattr(m, a) for a in ("norm1", "norm2", "linear1", "linear2")))


def _is_decoder_layer(m):
    return (isinstance(getattr(m, "cross_attn", None), MSDeformAttn) and
            isinstance(getattr(m, "self_attn", None), nn.MultiheadAttention) and
            all(hasattr(m, a) for a in ("norm1", "norm2", "norm3", "linear1", "linear2")))


def enable_fused_layer_tails(model, autocast=False, training=False, amp_training=False):
    """Rebind ``forward`` of every deformable encoder / decoder layer under ``model`` (idempotent).
    ``autocast=True`` also lets the layers run their tails under bf16 autocast, ``training=True`` lets them run the
    training tails while autograd records and dropouts are active, ``amp_training=True`` the training tails under bf16
    autocast (the module docstring says what each changes); calling again with other values updates every switched
    layer.  Returns the number of layers newly switched.
    ``disable_fused_layer_tails`` undoes it."""
    n = 0
    for parent in model.modules():
        layers = getattr(parent, "layers", None)
        if not isinstance(layers, nn.ModuleList):
            continue
        for i, layer in enumerate(layers):
            enc, dec = _is_encoder_layer(layer), _is_decoder_layer(layer)
            if not (enc or dec):
                continue
            layer._amp_tails = bool(autocast)
            layer._train_tails = bool(training)
            layer._amp_train_tails = bool(amp_training)
            if hasattr(layer, "_stock_forward"):
                continue
            layer._stock_forward = layer.forward
            layer._emit_next_query = enc and i + 1 < len(layers) and _is_encoder_layer(layers[i + 1])
            layer.forward = types.MethodType(_encoder_forward if enc else _decoder_forward, layer)
            n += 1
        # the encoder itself: in-kernel reference points
        if len(layers) and all(_is_encoder_layer(l) for l in layers) and not hasattr(parent, "_stock_forward"):
            if hasattr(parent, "analytic_reference_points"):          # the bench harness' encoder has a switch
                parent.analytic_reference_points = True
                parent.analytic_reference_points_with_grad = bool(training or amp_training)
            elif hasattr(parent, "get_reference_points"):             # the reference's DeformableTransformerEncoder
                parent._stock_forward = parent.forward
                parent.forward = types.MethodType(_reference_encoder_forward, parent)
    return n


def disable_fused_layer_tails(model):
    n = 0
    for m in model.modules():
        if getattr(m, "analytic_reference_points", False) is True:
            m.analytic_reference_points = False
            m.analytic_reference_points_with_grad = False
        if hasattr(m, "_stock_forward") and "forward" in m.__dict__:
            del m.__dict__["forward"]
            del m.__dict__["_stock_forward"]
            n += _is_encoder_layer(m) or _is_decoder_layer(m)
        for a in ("_amp_tails", "_train_tails", "_amp_train_tails", "_emit_next_query"):
            m.__dict__.pop(a, None)
    return n
