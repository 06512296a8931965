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

``_eligible`` alone decides, per call, whether the fused forward runs.  It runs only when all of these hold:

  * the residual stream is fp32 on CUDA with C = 128*k <= 1024 channels (what the kernel covers);
  * autocast is off for CUDA (under autocast the GEMMs return bf16 / fp16, which the fp32 kernel does not take);
  * nothing would need a gradient: grad mode is off, or no parameter of the layer and no tensor argument of its
    forward (src / tgt, pos / query_pos, reference points, the decoder's src, masks) requires grad -- the tail
    op has no autograd formula;
  * every dropout of the layer is inactive (p = 0 or eval mode);
  * the FFN activation is ReLU (``layer.activation is F.relu`` where the layer has one, as the reference's do);
  * every norm is an ``nn.LayerNorm`` with both weight and bias, and ``linear1`` has a bias.

In every other situation the layer's ORIGINAL forward runs, so training, autocast and any layer variant keep
exactly the stock behaviour.
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


def _dropout_off(layer):
    return not any(isinstance(m, nn.Dropout) and m.p > 0 and m.training for m in layer.children())


def _affine_layer_norm(norm):
    return isinstance(norm, nn.LayerNorm) and norm.weight is not None and norm.bias is not None


def _eligible(layer, x, *inputs):
    """Whether the fused forward computes what ``layer``'s own forward would (the module docstring lists the
    conditions).  ``x`` is the residual stream, ``inputs`` every other argument of the layer's forward."""
    if torch.is_autocast_enabled("cuda") or not ops.layer_tail_supported(x, x) or not _dropout_off(layer):
        return False
    if torch.is_grad_enabled() and (any(p.requires_grad for p in layer.parameters()) or
                                    any(torch.is_tensor(t) and t.requires_grad for t in inputs)):
        return False
    norms = [getattr(layer, n) for n in ("norm1", "norm2", "norm3") if hasattr(layer, n)]
    return (getattr(layer, "activation", F.relu) is F.relu and all(_affine_layer_norm(n) for n in norms) and
            layer.linear1.bias is not None)


def _tail(y, bias, residual, norm, pos=None):
    out, out_pos = torch.ops.snipper_b200.layer_tail(y, bias, residual, norm.weight, norm.bias, pos, norm.eps)
    return out, (out_pos if pos is not None else None)


def _ffn_hidden(layer, x):
    """relu(linear1(x)) with the bias + ReLU applied in the GEMM epilogue."""
    c = x.shape[-1]
    return torch._addmm_activation(layer.linear1.bias, x.reshape(-1, c), layer.linear1.weight.t())


def _with_pos(x, pos):
    """x + pos, taken from the previous layer's tail when it already produced it for this very ``pos``."""
    if pos is None:
        return x
    cached = getattr(x, _PLUS_POS, None)
    if cached is not None and cached[0] is pos:
        return cached[1]
    return x + pos


def _encoder_forward(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask=None):
    """reference deformable_transformer.py:200-210 (forward) and :192-198 (forward_ffn)"""
    if not _eligible(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask):
        return self._stock_forward(src, pos, reference_points, spatial_shapes, level_start_index, padding_mask)
    attn = self.self_attn
    core, _ = attn._attend(_with_pos(src, pos), reference_points, src, spatial_shapes, level_start_index, padding_mask)
    y = F.linear(core, attn.output_proj.weight)                              # bias joins the tail
    x, _ = _tail(y, attn.output_proj.bias, src, self.norm1)                  # :204-205
    ff = F.linear(_ffn_hidden(self, x), self.linear2.weight).view_as(x)      # :194
    emit = pos if (self._emit_next_query and pos is not None) else None
    out, out_pos = _tail(ff, self.linear2.bias, x, self.norm2, emit)         # :195-197 (+ the next layer's :202)
    if out_pos is not None:
        setattr(out, _PLUS_POS, (pos, out_pos))
    return out


def _decoder_forward(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                     src_padding_mask=None):
    """reference deformable_transformer.py:279-300 (forward) and :268-274 (forward_ffn)"""
    if not _eligible(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                     src_padding_mask):
        return self._stock_forward(tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                                   src_padding_mask)
    bs, t, lq, c = tgt.shape
    x = tgt.reshape(bs, t * lq, c)
    qp = None if query_pos is None else query_pos.reshape(bs, t * lq, c)
    qk = (x if qp is None else x + qp).transpose(0, 1)
    sa = self.self_attn(qk, qk, x.transpose(0, 1))[0].transpose(0, 1)        # :285 (nn.MultiheadAttention, stock)
    x, xq = _tail(sa, None, x, self.norm2, qp)                               # :286-287 (+ with_pos_embed of :292)
    q = (x if xq is None else xq).view(bs, t, lq, c)
    x = x.view(bs, t, lq, c)
    attn = self.cross_attn
    core, vis = attn._attend(q, reference_points, src, src_spatial_shapes, level_start_index, src_padding_mask)
    y = F.linear(core, attn.output_proj.weight)
    x, _ = _tail(y, attn.output_proj.bias, x, self.norm1)                    # :294-295
    ff = F.linear(_ffn_hidden(self, x), self.linear2.weight).view_as(x)      # :270
    out, _ = _tail(ff, self.linear2.bias, x, self.norm3)                     # :271-273
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


def enable_fused_layer_tails(model):
    """Rebind ``forward`` of every deformable encoder / decoder layer under ``model`` (idempotent).
    Returns the number of layers switched.  ``disable_fused_layer_tails`` undoes it."""
    n = 0
    for parent in model.modules():
        layers = getattr(parent, "layers", None)
        if not isinstance(layers, nn.ModuleList):
            continue
        for i, layer in enumerate(layers):
            enc, dec = _is_encoder_layer(layer), _is_decoder_layer(layer)
            if not (enc or dec) or hasattr(layer, "_stock_forward"):
                continue
            layer._stock_forward = layer.forward
            layer._emit_next_query = enc and i + 1 < len(layers) and _is_encoder_layer(layers[i + 1])
            layer.forward = types.MethodType(_encoder_forward if enc else _decoder_forward, layer)
            n += 1
        # the encoder itself: in-kernel reference points
        if len(layers) and all(_is_encoder_layer(l) for l in layers) and not hasattr(parent, "_stock_forward"):
            if hasattr(parent, "analytic_reference_points"):          # the bench harness' encoder has a switch
                parent.analytic_reference_points = True
            elif hasattr(parent, "get_reference_points"):             # the reference's DeformableTransformerEncoder
                parent._stock_forward = parent.forward
                parent.forward = types.MethodType(_reference_encoder_forward, parent)
    return n


def disable_fused_layer_tails(model):
    n = 0
    for m in model.modules():
        if getattr(m, "analytic_reference_points", False) is True:
            m.analytic_reference_points = False
        if hasattr(m, "_stock_forward") and "forward" in m.__dict__:
            del m.__dict__["forward"]
            del m.__dict__["_stock_forward"]
            n += _is_encoder_layer(m) or _is_decoder_layer(m)
    return n
