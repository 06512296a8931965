"""Bench / test HARNESS (stock PyTorch, not the product): a restatement of the Snipper network
around the hot path, so end-to-end snippets/s can be measured on a box that has no copy of the
reference.  Everything here except the injected attention class is plain torch / torchvision
(cuDNN / cuBLAS) and is out of scope for optimisation per BASELINE.json's north_star.

Mirrors, with the SAME module tree and state-dict keys (a reference checkpoint loads strictly):
  models/model.py:45-221          SnipperDeformable (input_proj, query_embed, heads, forward)
  models/backbone.py:27-131       frozen-BN ResNet-50, layers 2-4, strides 8/16/32
  models/position_encoding.py:19-63  3-D (t,y,x) sine embedding, hidden//3 features per axis
  models/deformable_transformer.py:21-343  encoder / decoder stacks and their layers
The attention class is a constructor argument (``attn_cls``): the product passes
``snipper_b200.MSDeformAttn``; tests and the CPU baseline pass the oracle restatement.
"""
import copy
import math
from types import SimpleNamespace

import torch
import torch.nn.functional as F
from torch import nn


def default_config(**kw):
    """Flags of the reference that shape the network (main.py:20-153), README values."""
    cfg = dict(hidden_dim=384, nheads=8, num_feature_levels=3, enc_layers=6, dec_layers=6,
               dim_feedforward=1024, dropout=0.1, enc_n_points=4, dec_n_points=4, num_frames=4,
               num_future_frames=0, num_queries=60, num_kpts=15, aux_loss=True, backbone="resnet50")
    cfg.update(kw)
    return SimpleNamespace(**cfg)


def inverse_sigmoid(x, eps=1e-5):
    x = x.clamp(min=0, max=1)
    return torch.log(x.clamp(min=eps) / (1 - x).clamp(min=eps))


class FrozenBatchNorm2d(nn.Module):
    """Affine transform with fixed statistics (reference models/backbone.py:27-63)."""

    def __init__(self, n, eps=1e-5):
        super().__init__()
        self.register_buffer("weight", torch.ones(n))
        self.register_buffer("bias", torch.zeros(n))
        self.register_buffer("running_mean", torch.zeros(n))
        self.register_buffer("running_var", torch.ones(n))
        self.eps = eps

    def _load_from_state_dict(self, state_dict, prefix, *args):
        state_dict.pop(prefix + "num_batches_tracked", None)
        super()._load_from_state_dict(state_dict, prefix, *args)

    def forward(self, x):
        scale = self.weight * (self.running_var + self.eps).rsqrt()
        shift = self.bias - self.running_mean * scale
        return x * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)


class _ResNetBody(nn.Module):
    """layers 2..4 of a torchvision ResNet (keys live under ``body.`` like IntermediateLayerGetter)."""

    def __init__(self, name):
        super().__init__()
        import torchvision
        net = getattr(torchvision.models, name)(weights=None, norm_layer=FrozenBatchNorm2d)
        self.body = nn.ModuleDict({k: getattr(net, k) for k in
                                   ("conv1", "bn1", "relu", "maxpool", "layer1", "layer2", "layer3", "layer4")})
        self.strides = [8, 16, 32]
        self.num_channels = [512, 1024, 2048]

    def forward(self, x):
        b = self.body
        x = b["maxpool"](b["relu"](b["bn1"](b["conv1"](x))))
        x = b["layer1"](x)
        c3 = b["layer2"](x)
        c4 = b["layer3"](c3)
        c5 = b["layer4"](c4)
        return [c3, c4, c5]


class SineEmbedding3D(nn.Module):
    """(t, y, x) sine position embedding, normalised to 2*pi (reference position_encoding.py:19-63)."""

    def __init__(self, feats, frames, temperature=10000):
        super().__init__()
        self.feats, self.frames, self.temperature = feats, frames, temperature

    def forward(self, mask):  # mask (b*t, h, w) bool, True = padding
        n, h, w = mask.shape
        valid = ~mask.view(n // self.frames, self.frames, h, w)
        scale, eps = 2 * math.pi, 1e-6
        z = valid.cumsum(1, dtype=torch.float32)
        y = valid.cumsum(2, dtype=torch.float32)
        x = valid.cumsum(3, dtype=torch.float32)
        z = z / (z[:, -1:] + eps) * scale
        y = y / (y[:, :, -1:] + eps) * scale
        x = x / (x[:, :, :, -1:] + eps) * scale
        i = torch.arange(self.feats, dtype=torch.float32, device=mask.device)
        freq = self.temperature ** (2 * (i // 2) / self.feats)

        def enc(e):
            p = e[..., None] / freq
            return torch.stack((p[..., 0::2].sin(), p[..., 1::2].cos()), dim=5).flatten(4)

        return torch.cat((enc(z), enc(y), enc(x)), dim=4).permute(0, 1, 4, 2, 3)  # (b,t,3*feats,h,w)


class Joiner(nn.Sequential):
    def __init__(self, backbone, pos):
        super().__init__(backbone, pos)
        self.strides, self.num_channels = backbone.strides, backbone.num_channels


def _clones(m, n):
    return nn.ModuleList([copy.deepcopy(m) for _ in range(n)])


class EncoderLayer(nn.Module):
    """reference deformable_transformer.py:170-210"""

    def __init__(self, attn_cls, d, ffn, dropout, L, M, P, n_frame):
        super().__init__()
        self.self_attn = attn_cls(d, L, M, P, n_frame, "encoder", False)
        self.dropout1, self.norm1 = nn.Dropout(dropout), nn.LayerNorm(d)
        self.linear1, self.dropout2 = nn.Linear(d, ffn), nn.Dropout(dropout)
        self.linear2, self.dropout3, self.norm2 = nn.Linear(ffn, d), nn.Dropout(dropout), nn.LayerNorm(d)

    def forward(self, src, pos, ref, shapes, lsi, mask):
        src = self.norm1(src + self.dropout1(self.self_attn(src + pos, ref, src, shapes, lsi, mask)))
        ff = self.linear2(self.dropout2(F.relu(self.linear1(src))))
        return self.norm2(src + self.dropout3(ff))


class Encoder(nn.Module):
    def __init__(self, layer, n):
        super().__init__()
        self.layers, self.num_layers = _clones(layer, n), n
        self.analytic_reference_points = False   # snipper_b200.enable_fused_layer_tails: closed form, computed in-kernel
        self.analytic_reference_points_with_grad = False   # ... also while autograd records (training=True)

    @staticmethod
    def reference_points(sizes, valid_ratios, device):
        """Pixel centres of every level, in every level's normalised frame (:219-232)."""
        pts = []
        for l, (H, W) in enumerate(sizes):
            ys, xs = torch.meshgrid(torch.linspace(0.5, H - 0.5, H, dtype=torch.float32, device=device),
                                    torch.linspace(0.5, W - 0.5, W, dtype=torch.float32, device=device),
                                    indexing="ij")
            ys = ys.reshape(-1)[None] / (valid_ratios[:, None, l, 1] * H)
            xs = xs.reshape(-1)[None] / (valid_ratios[:, None, l, 0] * W)
            pts.append(torch.stack((xs, ys), -1))
        return torch.cat(pts, 1)[:, :, None] * valid_ratios[:, None]  # (b, S, L, 2)

    def forward(self, src, sizes, shapes, lsi, valid_ratios, pos, mask, n_frame):
        if self.analytic_reference_points and (self.analytic_reference_points_with_grad or not torch.is_grad_enabled()):
            from ..modules import EncoderGrid
            ref = EncoderGrid(valid_ratios, sizes, n_frame)
        else:
            ref = self.reference_points(sizes, valid_ratios, src.device).unsqueeze(1).expand(-1, n_frame, -1, -1, -1)
        for layer in self.layers:
            src = layer(src, pos, ref, shapes, lsi, mask)
        return src


class DecoderLayer(nn.Module):
    """reference deformable_transformer.py:244-300"""

    def __init__(self, attn_cls, d, ffn, dropout, L, M, P, n_frame):
        super().__init__()
        self.cross_attn = attn_cls(d, L, M, P, n_frame, "decoder", False, True)
        self.dropout1, self.norm1 = nn.Dropout(dropout), nn.LayerNorm(d)
        self.self_attn = nn.MultiheadAttention(d, M, dropout=dropout)
        self.dropout2, self.norm2 = nn.Dropout(dropout), nn.LayerNorm(d)
        self.linear1, self.dropout3 = nn.Linear(d, ffn), nn.Dropout(dropout)
        self.linear2, self.dropout4, self.norm3 = nn.Linear(ffn, d), nn.Dropout(dropout), nn.LayerNorm(d)

    def forward(self, tgt, qpos, ref, src, shapes, lsi, mask):
        b, t, lq, c = tgt.shape
        x, p = tgt.view(b, t * lq, c), qpos.view(b, t * lq, c)
        qk = (x + p).transpose(0, 1)
        x = self.norm2(x + self.dropout2(self.self_attn(qk, qk, x.transpose(0, 1))[0].transpose(0, 1)))
        x = x.view(b, t, lq, c)
        y, att = self.cross_attn(x + qpos, ref, src, shapes, lsi, mask)
        x = self.norm1(x + self.dropout1(y))
        ff = self.linear2(self.dropout3(F.relu(self.linear1(x))))
        return self.norm3(x + self.dropout4(ff)), att


class Decoder(nn.Module):
    def __init__(self, layer, n):
        super().__init__()
        self.layers, self.num_layers = _clones(layer, n), n
        self.root_embed = None
        self.class_embed = None

    def forward(self, tgt, ref, src, shapes, lsi, valid_ratios, qpos, mask):
        outs, refs, atts = [], [], []
        for i, layer in enumerate(self.layers):
            ref_in = ref[:, :, :, None, :] * valid_ratios[:, None, None, :, :]
            tgt, att = layer(tgt, qpos, ref_in, src, shapes, lsi, mask)
            if self.root_embed is not None:  # iterative refinement of the reference points (:328-332)
                delta = self.root_embed[i](tgt)[..., 0:2]
                ref = (delta + inverse_sigmoid(ref)).sigmoid().detach()
            outs.append(tgt)
            refs.append(ref)
            atts.append(att)
        return torch.stack(outs), torch.stack(refs), atts


class Transformer(nn.Module):
    """reference deformable_transformer.py:21-167"""

    def __init__(self, cfg, attn_cls):
        super().__init__()
        d, M, L = cfg.hidden_dim, cfg.nheads, cfg.num_feature_levels
        self.d_model, self.nhead = d, M
        self.n_frame, self.n_future_frame, self.num_keypoints = cfg.num_frames, cfg.num_future_frames, cfg.num_kpts
        self.encoder = Encoder(EncoderLayer(attn_cls, d, cfg.dim_feedforward, cfg.dropout, L, M,
                                            cfg.enc_n_points, cfg.num_frames), cfg.enc_layers)
        self.decoder = Decoder(DecoderLayer(attn_cls, d, cfg.dim_feedforward, cfg.dropout, L, M,
                                            cfg.dec_n_points, cfg.num_frames), cfg.dec_layers)
        self.level_embed = nn.Parameter(torch.empty(L, d))
        self.temporal_embed = nn.Parameter(torch.empty(cfg.num_frames + cfg.num_future_frames, d))
        self.reference_points = nn.Linear(d, 2)
        self._attn_cls = attn_cls
        self._shape_cache = {}
        self._reset_parameters()

    def _reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)
        for m in self.modules():
            if isinstance(m, self._attn_cls):
                m._reset_parameters()
        nn.init.xavier_uniform_(self.reference_points.weight, gain=1.0)
        nn.init.zeros_(self.reference_points.bias)
        nn.init.normal_(self.level_embed)

    @staticmethod
    def valid_ratio(mask):  # (b, c, t, h, w)
        _, _, _, H, W = mask.shape
        vh = (~mask[:, 0, 0, :, 0]).sum(1).float() / H
        vw = (~mask[:, 0, 0, 0, :]).sum(1).float() / W
        return torch.stack([vw, vh], -1)

    def forward(self, srcs, masks, poss, query_embed):
        flat_src, flat_mask, flat_pos, sizes = [], [], [], []
        for l, (s, m, p) in enumerate(zip(srcs, masks, poss)):
            b, c, t, h, w = s.shape
            sizes.append((h, w))
            flat_src.append(s.flatten(3).permute(0, 2, 3, 1))
            flat_mask.append(m.flatten(3).permute(0, 2, 3, 1))
            flat_pos.append(p.flatten(3).permute(0, 2, 3, 1) + self.level_embed[l].view(1, 1, 1, -1))
        src, mask, pos = torch.cat(flat_src, 2), torch.cat(flat_mask, 2), torch.cat(flat_pos, 2)
        key = (tuple(sizes), src.device)
        if key not in self._shape_cache:  # host->device copy once, not per forward (CUDA-graph safe)
            shapes = torch.as_tensor(sizes, dtype=torch.long, device=src.device)
            self._shape_cache[key] = (shapes, torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1])))
        shapes, lsi = self._shape_cache[key]
        valid_ratios = torch.stack([self.valid_ratio(m) for m in masks], 1)

        memory = self.encoder(src, sizes, shapes, lsi, valid_ratios, pos, mask, self.n_frame)

        b, _, _, c = memory.shape
        heatmaps, start = [], 0
        for (h, w) in sizes:  # first num_keypoints channels of every head double as heatmaps (:141-150)
            lvl = memory[:, :, start:start + h * w].reshape(b, self.n_frame, h, w, self.nhead, c // self.nhead)
            heatmaps.append(lvl[..., 0:self.num_keypoints])
            start += h * w

        t = self.n_frame + self.n_future_frame
        nq = query_embed.shape[0] // t
        qpos, qobj = torch.split(query_embed, c, dim=-1)
        qpos = qpos.reshape(t, nq, c).unsqueeze(0).expand(b, -1, -1, -1) + self.temporal_embed.view(1, t, 1, c)
        qobj = qobj.reshape(t, nq, c).unsqueeze(0).expand(b, -1, -1, -1)
        ref0 = self.reference_points(qpos).sigmoid()
        hs, refs, atts = self.decoder(qobj, ref0, memory, shapes, lsi, valid_ratios, qpos, mask)
        return hs, heatmaps, ref0, refs, atts


class MLP(nn.Module):
    def __init__(self, i, h, o, n):
        super().__init__()
        self.num_layers = n
        dims = [h] * (n - 1)
        self.layers = nn.ModuleList(nn.Linear(a, b) for a, b in zip([i] + dims, dims + [o]))

    def forward(self, x):
        for k, layer in enumerate(self.layers):
            x = F.relu(layer(x)) if k < self.num_layers - 1 else layer(x)
        return x


class SnipperNet(nn.Module):
    """reference models/model.py:45-237 (SnipperDeformable)."""

    def __init__(self, cfg, attn_cls):
        super().__init__()
        self.cfg = cfg
        d = cfg.hidden_dim
        backbone = _ResNetBody(cfg.backbone)
        for name, p in backbone.named_parameters():  # reference backbone.py:69-71
            if "layer2" not in name and "layer3" not in name and "layer4" not in name:
                p.requires_grad_(False)
        self.num_queries, self.num_frames = cfg.num_queries, cfg.num_frames
        self.num_future_frames, self.num_keypoints = cfg.num_future_frames, cfg.num_kpts
        self.num_feature_levels, self.aux_loss = cfg.num_feature_levels, cfg.aux_loss
        self.transformer = Transformer(cfg, attn_cls)
        self.backbone = Joiner(backbone, SineEmbedding3D(d // 3, cfg.num_frames))
        self.input_proj = nn.ModuleList([
            nn.Sequential(nn.Conv2d(ch, d, kernel_size=1), nn.GroupNorm(32, d)) for ch in backbone.num_channels])
        self.query_embed = nn.Embedding(cfg.num_queries * (cfg.num_frames + cfg.num_future_frames), d * 2)
        n_dec = cfg.dec_layers
        cls, root = nn.Linear(d, 2), MLP(d, d, 4, 1)
        joints = nn.ModuleList([MLP(d, d, 4, 1) for _ in range(cfg.num_kpts - 1)])
        self.class_embed = nn.ModuleList([cls] * n_dec)   # shared across decoder layers (:98-100)
        self.root_embed = nn.ModuleList([root] * n_dec)
        self.joint_embed = nn.ModuleList([joints] * n_dec)
        self.transformer.decoder.root_embed = self.root_embed
        self.transformer.decoder.class_embed = self.class_embed

    def forward(self, images):
        """images (N, 3*T, H, W) in [0,1]  ->  (dict of predictions, (ref0, refs, attention data))."""
        N, C, H, W = images.shape
        T = self.num_frames
        frames = images.reshape(N * T, 3, H, W)
        pix_mask = torch.zeros((N * T, H, W), dtype=torch.bool, device=images.device)  # no padding
        feats = self.backbone[0](frames)
        srcs, masks, poss = [], [], []
        for l, f in enumerate(feats):
            m = F.interpolate(pix_mask[None].float(), size=f.shape[-2:]).to(torch.bool)[0]
            s = self.input_proj[l](f)
            n, c, h, w = s.shape
            srcs.append(s.reshape(N, T, c, h, w).transpose(1, 2))
            masks.append(m.reshape(N, T, 1, h, w).expand(N, T, c, h, w).transpose(1, 2))
            poss.append(self.backbone[1](m).to(s.dtype).transpose(1, 2))
        hs, heatmaps, ref0, refs, atts = self.transformer(srcs, masks, poss, self.query_embed.weight)

        n_dec, bs, t, _, c = hs.shape
        classes, kpts = [], []
        for l in range(n_dec):
            classes.append(self.class_embed[l](hs[l]).transpose(1, 2))
            base = inverse_sigmoid(ref0 if l == 0 else refs[l - 1])
            root = self.root_embed[l](hs[l]).view(bs, t, self.num_queries, 1, 4)
            root = torch.cat([root[..., :2] + base[:, :, :, None, :], root[..., 2:]], -1).sigmoid()
            joints = torch.cat([self.joint_embed[l][i](hs[l]).reshape(bs, t, self.num_queries, 1, 4)
                                for i in range(self.num_keypoints - 1)], dim=3)
            kpts.append(torch.cat([root, joints], dim=3).transpose(1, 2))
        classes, kpts = torch.stack(classes), torch.stack(kpts)
        out = {"pred_logits": classes[-1], "pred_kpts2d": kpts[-1, ..., 0:3], "pred_depth": kpts[-1, ..., 3:4],
               "heatmaps": heatmaps}
        if self.aux_loss:
            out["aux_outputs"] = [{"pred_logits": classes[i], "pred_kpts2d": kpts[i, ..., 0:3],
                                   "pred_depth": kpts[i, ..., 3:4]} for i in range(n_dec - 1)]
        return out, (ref0, refs, atts)


def build_snipper(attn_cls, **cfg_overrides):
    return SnipperNet(default_config(**cfg_overrides), attn_cls)
