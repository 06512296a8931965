"""``MSDeformAttn`` -- drop-in for the reference's Snipper-modified attention module
(models/ops/modules/ms_deform_attn.py:37-243).

Same constructor signature (including the reference's ``use_pytroch_deform`` spelling), same
``forward`` contract, same parameter names / state-dict keys
(``sampling_offsets.{i}``, ``attention_weights.{i}``, ``value_proj``, ``output_proj``; the frame
slots alias ONE Linear each, :68-71), same initialisation (:78-97), so checkpoints load and
``models/deformable_transformer.py`` constructs and calls it unchanged (:178, :251-252, :202, :292).

What differs is the execution:

* fused path (default): offsets and logits are computed ONCE for all query frames, by ONE GEMM
  over the stacked weights (the reference recomputes the same two GEMMs for every (t1,t2) pair
  -- 20 GEMMs per layer at T=4, only 2 distinct), then ONE kernel launch per layer (``snipper_b200::snippet_attn``) does the
  offset normalisation, the softmax over levels x points x neighbour frames and the gather from
  all neighbour frames.  No ``.contiguous()`` copies, no stack+sum, no host sync (the
  reference's shape assert at :112 synchronises the stream every call).
* per-call path (``fused=False``, or when the frame slots do not alias / shapes are outside the
  fused kernels' range): the reference's loop, one ``MSDeformAttnFunction`` call per (t1,t2).

``use_pytroch_deform`` is accepted and ignored: there is no PyTorch/CPU implementation in this
package -- the CUDA kernels always run.
"""
import math

import torch
import torch.nn.functional as F
from torch import nn

from .. import ops
from ..functions import MSDeformAttnFunction


def neighbour_frames(t1, n_frame, n_src_frames):
    """Source frames a query frame attends to (reference :137-140 observed, :189/:201 future)."""
    if t1 < n_frame:
        return [t for t in (t1 - 1, t1, t1 + 1) if 0 <= t < n_frame]
    return list(range(n_src_frames))


class EncoderGrid:
    """Stand-in for the ENCODER's ``reference_points`` tensor (reference get_reference_points,
    models/deformable_transformer.py:219-232): the reference point of query q on level l is a closed-form function of
    q and the per-level valid ratios, so the fused kernels compute it from the query index instead of reading a
    (N,T,S,L,2) tensor that the reference materialises per forward and every layer re-reads.  Opt-in: pass an instance
    as ``reference_points`` (snipper_b200.enable_fused_layer_tails does it for the encoder).  ``valid_ratios`` is
    the (N,L,2) tensor of DeformableTransformer.get_valid_ratio; ``tensor()`` builds the reference's tensor (used by
    the per-call fallback path and by tests)."""

    def __init__(self, valid_ratios, spatial_sizes, n_frame):
        self.valid_ratios = valid_ratios.float().contiguous()
        self.spatial_sizes = [(int(h), int(w)) for h, w in spatial_sizes]
        self.n_frame = n_frame

    def tensor(self):
        vr, dev = self.valid_ratios, self.valid_ratios.device
        pts = []
        for l, (H, W) in enumerate(self.spatial_sizes):
            ys, xs = torch.meshgrid(torch.linspace(0.5, H - 0.5, H, dtype=torch.float32, device=dev),
                                    torch.linspace(0.5, W - 0.5, W, dtype=torch.float32, device=dev), indexing="ij")
            ys = ys.reshape(-1)[None] / (vr[:, None, l, 1] * H)
            xs = xs.reshape(-1)[None] / (vr[:, None, l, 0] * W)
            pts.append(torch.stack((xs, ys), -1))
        ref = torch.cat(pts, 1)[:, :, None] * vr[:, None]
        return ref.unsqueeze(1).expand(-1, self.n_frame, -1, -1, -1)


class _LazyList(list):
    """A list whose elements are produced on first access (len, indexing, iteration)."""

    def __init__(self, owner, which):
        super().__init__()
        self._owner, self._which, self._ready = owner, which, False

    def _fill(self):
        if not self._ready:
            self._ready = True
            super().extend(self._owner.materialise()[self._which])

    def __len__(self):
        self._fill()
        return super().__len__()

    def __getitem__(self, i):
        self._fill()
        return super().__getitem__(i)

    def __iter__(self):
        self._fill()
        return super().__iter__()

    def __repr__(self):
        self._fill()
        return super().__repr__()


class LazyVis:
    """The decoder's ``attention_vis`` payload (reference :228-233: per query frame, sampling locations
    (N,Lq,M,L,P,k,2) and attention weights (N,Lq,M,L,P,k)).  Only the reference's visualiser reads them, so
    the fused path hands out two lists that compute their tensors when first touched instead of running
    ~20 small launches in every decoder layer of every forward.  The inputs are kept by reference: read the
    lists before the buffers are reused (e.g. before the next CUDA-graph replay)."""

    def __init__(self, module, proj, off_bias, logit_bias, ref, spatial_shapes, T2):
        self.args = (module, proj, off_bias, logit_bias, ref, spatial_shapes, T2)
        self.out = None

    def lists(self):
        return _LazyList(self, 0), _LazyList(self, 1)

    def materialise(self):
        if self.out is None:
            module, proj, off_bias, logit_bias, ref, spatial_shapes, T2 = self.args
            N, T1, Lq, _ = proj.shape
            M, L, P = module.n_heads, module.n_levels, module.n_points
            n_off = 2 * M * L * P
            offsets = (proj[..., :n_off] + off_bias).view(N, T1, Lq, M, L, P, 2)
            logits = (proj[..., n_off:] + logit_bias).view(N, T1, Lq, M, L, P)
            self.out = module._vis_fused(offsets, logits, ref, spatial_shapes, T2)
            self.args = None
        return self.out


class MSDeformAttn(nn.Module):
    def __init__(self, d_model=256, n_levels=4, n_heads=8, n_points=4, n_frame=4,
                 mode="encoder", use_pytroch_deform=False, attention_vis=False):
        super().__init__()
        if d_model % n_heads != 0:
            raise ValueError("d_model must be divisible by n_heads, but got {} and {}".format(d_model, n_heads))
        assert mode in ("encoder", "decoder")
        self.im2col_step = 64
        self.d_model = d_model
        self.n_levels = n_levels
        self.n_heads = n_heads
        self.n_points = n_points
        self.n_frame = n_frame
        self.use_pytroch_deform = use_pytroch_deform  # kept for signature parity; ignored
        self.mode = mode
        self.attention_vis = attention_vis
        self.fused = True
        self._proj_cache = None

        offsets = nn.Linear(d_model, n_heads * n_levels * n_points * 2)
        self.sampling_offsets = nn.ModuleList([offsets for _ in range(n_frame)])
        weights = nn.Linear(d_model, n_heads * n_levels * n_points)
        self.attention_weights = nn.ModuleList([weights for _ in range(n_frame)])
        self.value_proj = nn.Linear(d_model, d_model)
        self.output_proj = nn.Linear(d_model, d_model)
        self._reset_parameters()

    def _reset_parameters(self):
        # head h looks along angle 2*pi*h/M, scaled so the larger component is 1; point p sits
        # (p+1) pixels out; attention starts uniform (reference :78-97)
        M, L, P = self.n_heads, self.n_levels, self.n_points
        theta = torch.arange(M, dtype=torch.float32) * (2.0 * math.pi / M)
        direction = torch.stack([theta.cos(), theta.sin()], -1)
        direction = direction / direction.abs().max(-1, keepdim=True)[0]
        steps = torch.arange(1, P + 1, dtype=torch.float32).view(1, 1, P, 1)
        bias = (direction.view(M, 1, 1, 2) * steps).expand(M, L, P, 2).reshape(-1)
        with torch.no_grad():
            for lin in self.sampling_offsets:
                lin.weight.zero_()
                lin.bias.copy_(bias)
            for lin in self.attention_weights:
                lin.weight.zero_()
                lin.bias.zero_()
            nn.init.xavier_uniform_(self.value_proj.weight)
            self.value_proj.bias.zero_()
            nn.init.xavier_uniform_(self.output_proj.weight)
            self.output_proj.bias.zero_()

    # -------------------------------------------------------------------------------------
    def _slots_aliased(self):
        so, aw = self.sampling_offsets, self.attention_weights
        return all(m is so[0] for m in so) and all(m is aw[0] for m in aw)

    def _can_fuse(self, value, spatial_size=0, batch_frames=0):
        """Every condition the fused C entry points check (so anything else degrades to the per-call loop
        instead of raising): aliased frame slots, supported head size / sample count, 28-bit cell offsets,
        gridDim.z, and a float32 deterministic mode."""
        if ops.is_deterministic() and torch.is_grad_enabled() and value.dtype != torch.float32:
            return False  # the deterministic grad_value path is float32 only
        return (self.fused and self._slots_aliased() and value.is_cuda and
                ops.snippet_supported(self.n_heads, self.d_model // self.n_heads, self.n_levels,
                                      self.n_points, value.dtype, spatial_size, batch_frames))

    def _stacked_projection(self):
        """[sampling_offsets | attention_weights] weights as ONE (3*M*L*P, C) matrix and the two biases in
        fp32.  Rebuilt only when a parameter changed (inference: once); under autograd it is a plain cat
        so the gradient reaches both Linear layers."""
        so, aw = self.sampling_offsets[0], self.attention_weights[0]
        if torch.is_grad_enabled() and (so.weight.requires_grad or aw.weight.requires_grad):
            return torch.cat((so.weight, aw.weight), 0), so.bias.float(), aw.bias.float()
        key = (so.weight.data_ptr(), so.weight._version, aw.weight.data_ptr(), aw.weight._version,
               so.bias.data_ptr(), so.bias._version, aw.bias.data_ptr(), aw.bias._version, so.weight.dtype)
        if self._proj_cache is None or self._proj_cache[0] != key:
            with torch.no_grad():
                self._proj_cache = (key, torch.cat((so.weight, aw.weight), 0).contiguous(),
                                    so.bias.detach().float().contiguous(), aw.bias.detach().float().contiguous())
        return self._proj_cache[1:]

    def forward(self, query, reference_points, input_flatten, input_spatial_shapes,
                input_level_start_index, input_padding_mask=None):
        """query (N,T1,Lq,C); reference_points (N,T1,Lq,L,2) in [0,1]; input_flatten (N,T2,S,C);
        input_spatial_shapes (L,2) int64; input_level_start_index (L,) int64;
        input_padding_mask (N,T2,S,C) bool, True = padding -- also accepted: a channel-expanded view or a
        per-pixel (N,T2,S[,1]) mask, which the kernels then read as one byte per pixel.
        Returns (N,T1,Lq,C), plus ``(sampling_locations per t1, attention_weights per t1)`` when
        ``attention_vis``."""
        out, vis = self._attend(query, reference_points, input_flatten, input_spatial_shapes,
                                input_level_start_index, input_padding_mask)
        out = self.output_proj(out)
        if self.attention_vis:
            return out, vis
        return out

    def _attend(self, query, reference_points, input_flatten, input_spatial_shapes,
                input_level_start_index, input_padding_mask=None):
        """Everything of ``forward`` up to (not including) ``output_proj``: (N,T1,Lq,C) attention output and the
        visualisation payload (None unless ``attention_vis``).  The fused layer tails (snipper_b200/layers.py)
        apply ``output_proj`` themselves so that its bias folds into the residual + LayerNorm pass."""
        N, T1, Lq, _ = query.shape
        _, T2, S, _ = input_flatten.shape
        M, L, P = self.n_heads, self.n_levels, self.n_points
        if input_spatial_shapes.shape[0] != L or input_level_start_index.numel() != L:
            raise RuntimeError("input_spatial_shapes must be (n_levels, 2) and input_level_start_index (n_levels,)")

        value = self.value_proj(input_flatten)

        if self._can_fuse(value, S, N * T1):
            # ONE GEMM for both per-query projections (the reference runs the two Linear layers once per
            # (t1,t2) pair, :143-145,162-163): the weights are stacked [sampling_offsets | attention_weights],
            # the biases are added inside the kernel (no GEMM epilogue pass over the projection output), and
            # the kernel reads its offsets / logits as column blocks of the one output.  The padding mask
            # (:116-117) is applied inside the kernels as well -- value is never re-written.
            # value may be bf16 or fp16 (autocast): the kernels gather 16-bit values and keep every location / weight
            # computation in fp32, so the projection and the reference points go in as fp32.
            weight, off_bias, logit_bias = self._stacked_projection()
            proj = F.linear(query, weight)
            if proj.dtype != torch.float32:
                proj = proj.float()
            if isinstance(reference_points, EncoderGrid) and Lq == S:
                ref, valid_ratios = None, reference_points.valid_ratios      # reference points computed in-kernel
            else:
                if isinstance(reference_points, EncoderGrid):
                    reference_points = reference_points.tensor()
                ref, valid_ratios = reference_points, None
                if ref.dtype != torch.float32:
                    ref = ref.float()
            out = ops.snippet_attention(value.view(N, T2, S, M, self.d_model // M), input_padding_mask,
                                        input_spatial_shapes, input_level_start_index, proj, off_bias, logit_bias,
                                        ref, self.n_frame, valid_ratios=valid_ratios)
            vis = None
            if self.attention_vis:
                if ref is None:
                    ref = reference_points.tensor()
                vis = LazyVis(self, proj.detach(), off_bias.detach(), logit_bias.detach(), ref.detach(),
                              input_spatial_shapes, T2).lists()
        else:
            if input_padding_mask is not None:
                mask = input_padding_mask
                if mask.dim() == 3:
                    mask = mask.unsqueeze(-1)
                value = value.masked_fill(mask, 0.0)
            value = value.view(N, T2, S, M, self.d_model // M)
            if isinstance(reference_points, EncoderGrid):
                reference_points = reference_points.tensor()
            out, vis = self._forward_per_call(query, reference_points, value, input_spatial_shapes,
                                              input_level_start_index)
        return out, vis

    # -------------------------------------------------------------------------------------
    def _vis_fused(self, offsets, logits, reference_points, spatial_shapes, T2):
        """The (detached) tensors the decoder hands to the visualiser (reference :228-233)."""
        with torch.no_grad():
            N, T1, Lq, M, L, P, _ = offsets.shape
            wh = torch.stack([spatial_shapes[:, 1], spatial_shapes[:, 0]], -1).to(offsets.dtype)
            loc = reference_points[:, :, :, None, :, None, :] + offsets / wh[None, None, None, None, :, None, :]
            att = F.softmax(logits.flatten(-2), -1).view(N, T1, Lq, M, L, P)
            locs, atts = [], []
            for t1 in range(T1):
                k = len(neighbour_frames(t1, self.n_frame, T2))
                locs.append(loc[:, t1].unsqueeze(-2).expand(N, Lq, M, L, P, k, 2))
                atts.append((att[:, t1] / k).unsqueeze(-1).expand(N, Lq, M, L, P, k))
        return locs, atts

    def _forward_per_call(self, query, reference_points, value, spatial_shapes, level_start_index):
        """One op call per (query frame, neighbour frame), as the reference does (:130-225)."""
        N, T1, Lq, _ = query.shape
        T2 = value.shape[1]
        M, L, P = self.n_heads, self.n_levels, self.n_points
        wh = torch.stack([spatial_shapes[:, 1], spatial_shapes[:, 0]], -1)
        outs, vis_loc, vis_att = [], [], []
        for t1 in range(T1):
            frames = neighbour_frames(t1, self.n_frame, T2)
            q = query[:, t1]
            logits = torch.stack([self.attention_weights[t2](q).view(N, Lq, M, L, P) for t2 in frames], -1)
            att = F.softmax(logits.flatten(-3), -1).view(N, Lq, M, L, P, len(frames))
            if value.dtype in (torch.bfloat16, torch.float16):
                att = att.float()
            acc, locs = None, []
            for j, t2 in enumerate(frames):
                off = self.sampling_offsets[t2](q).view(N, Lq, M, L, P, 2)
                loc = reference_points[:, t1, :, None, :, None, :] + off / wh[None, None, None, :, None, :]
                if value.dtype in (torch.bfloat16, torch.float16):
                    loc = loc.float()
                if self.attention_vis:
                    locs.append(loc.detach())
                # value[:, t2] keeps its batch stride (no copy); loc/att slices are materialised
                o = MSDeformAttnFunction.apply(value[:, t2], spatial_shapes, level_start_index,
                                               loc.contiguous(), att[..., j].contiguous(), self.im2col_step)
                acc = o if acc is None else acc + o
            outs.append(acc)
            if self.attention_vis:
                vis_loc.append(torch.stack(locs, dim=-2))
                vis_att.append(att.detach())
        return torch.stack(outs, dim=1), (vis_loc, vis_att)
