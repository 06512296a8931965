"""The UNMODIFIED reference network on the GPU, with the product plugged in through each drop-in surface
(SURVEY.md section 8b).  The reference's own A/B switch ``use_pytorch_deform`` (modules/ms_deform_attn.py:172-181)
is the yardstick: its grid_sample path (``=1``) is the oracle, and

  surface 1  ``install_extension_shim()``: the reference's ``MSDeformAttn`` / ``MSDeformAttnFunction`` /
             ``deformable_transformer.py`` run as they are with ``use_pytorch_deform = 0`` and reach our
             per-call kernels through the module name ``MultiScaleDeformableAttention``;
  surface 3  ``install_module()``: the reference's ``build_model`` constructs ``snipper_b200.MSDeformAttn``
             (fused kernels), same state dict.

must reproduce it: forward at the 1e-5 scale (a whole network in fp32, so a small multiple of it), gradients at
1e-4-scale, with ``sampling_offsets.weight`` perturbed off its degenerate zero init (SURVEY section 7: at
random init every sample sits on an integer pixel coordinate, where grad_sampling_loc is one-sided).
The reference comes from /root/reference or from the copy staged in baseline/_ref/ (GPU box)."""
import sys

import pytest
import torch

import ref_loader
from conftest import rel_err

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not ref_loader.available(), reason="original Snipper source tree not found (set SNIPPER_REFERENCE to it)")]
DEV = "cuda:0"
KW = dict(hidden_dim=384, nheads=8, num_feature_levels=3, enc_n_points=4, dec_n_points=4, num_frames=4,
          num_future_frames=2, enc_layers=2, dec_layers=2, num_queries=9, dim_feedforward=256, dropout=0.0)
# whole network (ResNet-50 + 4 attention layers + heads) in fp32, two formulations of every attention call; the
# gradient tolerances are those of tests/test_model_gpu.py (backbone convolutions: cuDNN algorithm choice is looser)
FWD_TOL, BWD_TOL, BWD_TOL_BACKBONE = 1e-4, 5e-3, 3e-2


@pytest.fixture(autouse=True)
def strict_fp32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _perturb(model):
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if "sampling_offsets" in n and n.endswith("weight"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            if "attention_weights" in n:
                p.copy_(torch.randn(p.shape, generator=g) * 0.2)


def _reference_model():
    torch.manual_seed(3)
    model, _ = ref_loader.build_reference_model(use_pytorch_deform=1, **KW)
    _perturb(model)
    return model.to(DEV).eval()


def _set_deform_path(model, use_pytorch):
    import models.ops.modules as ref_modules
    n = 0
    for m in model.modules():
        if isinstance(m, ref_modules.MSDeformAttn):
            m.use_pytroch_deform = bool(use_pytorch)   # (sic) the reference's attribute, ms_deform_attn.py:56
            n += 1
    return n


def _run(model, x, weights):
    """Forward + a fixed linear functional of every prediction, backward; returns (outputs, grads by name)."""
    for p in model.parameters():
        p.grad = None
    out, _ = model(x)
    tensors = [out["pred_logits"], out["pred_kpts2d"], out["pred_depth"]] + list(out["heatmaps"])
    tensors += [a[k] for a in out["aux_outputs"] for k in ("pred_logits", "pred_kpts2d", "pred_depth")]
    loss = sum((t * w).sum() for t, w in zip(tensors, weights))
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return [t.detach() for t in tensors], grads


def _weights_like(model, x):
    with torch.no_grad():
        out, _ = model(x)
    tensors = [out["pred_logits"], out["pred_kpts2d"], out["pred_depth"]] + list(out["heatmaps"])
    tensors += [a[k] for a in out["aux_outputs"] for k in ("pred_logits", "pred_kpts2d", "pred_depth")]
    g = torch.Generator().manual_seed(5)
    return [torch.randn(t.shape, generator=g).to(DEV) for t in tensors]


def _compare(got, want):
    for i, (a, b) in enumerate(zip(got[0], want[0])):
        assert rel_err(a, b) < FWD_TOL, ("output", i, rel_err(a, b))
    assert set(got[1]) == set(want[1])
    errs = sorted(((rel_err(got[1][n], want[1][n]), n) for n in want[1] if float(want[1][n].abs().max()) > 1e-8), reverse=True)
    assert len(errs) > 50
    for e, n in errs:
        assert e < (BWD_TOL_BACKBONE if n.startswith("backbone.") else BWD_TOL), errs[:5]


def test_extension_shim_runs_the_unmodified_reference():
    """Surface 1: reference model, use_pytorch_deform=0 -> MSDeformAttnFunction -> MSDA shim -> msda_forward/backward."""
    import snipper_b200
    from snipper_b200 import ops
    model = _reference_model()
    x = torch.rand(1, 3 * KW["num_frames"], 192, 256, device=DEV)
    w = _weights_like(model, x)
    want = _run(model, x, w)                                    # the reference's grid_sample path
    import models.ops.functions.ms_deform_attn_func as ref_func
    before = getattr(ref_func, "MSDA", None)
    try:
        snipper_b200.install_extension_shim()
        assert _set_deform_path(model, use_pytorch=False) == KW["enc_layers"] + KW["dec_layers"]
        ops.STATS.reset()
        got = _run(model, x, w)
        # 10 (t1,t2) pairs per encoder layer, 10 + 2*4 per decoder layer (T = 4 + 2): one forward launch and one
        # grad_value memset + one backward launch per pair
        assert ops.STATS.launches == 3 * (KW["enc_layers"] * 10 + KW["dec_layers"] * 18)
    finally:
        if before is not None:
            ref_func.MSDA = before
        _set_deform_path(model, use_pytorch=True)
    _compare(got, want)


def test_fused_module_builds_into_the_unmodified_reference():
    """Surface 3: the reference's build_model constructs the fused module; same weights, same results."""
    import snipper_b200
    import models.ops.modules as ref_modules
    model = _reference_model()
    x = torch.rand(1, 3 * KW["num_frames"], 192, 256, device=DEV)
    w = _weights_like(model, x)
    want = _run(model, x, w)
    ref_cls = ref_modules.MSDeformAttn
    try:
        snipper_b200.install_module()
        torch.manual_seed(3)
        ours, _ = ref_loader.build_reference_model(use_pytorch_deform=0, **KW)
    finally:
        for name in ("models.ops.modules", "models.ops.modules.ms_deform_attn", "models.deformable_transformer"):
            sys.modules[name].MSDeformAttn = ref_cls
    ours.load_state_dict(model.state_dict(), strict=True)
    ours = ours.to(DEV).eval()
    mods = [m for m in ours.modules() if isinstance(m, snipper_b200.MSDeformAttn)]
    assert len(mods) == KW["enc_layers"] + KW["dec_layers"]
    got = _run(ours, x, w)
    _compare(got, want)
    # the attention payload the reference's decoder hands upward (deformable_transformer.py:292,339) keeps its shapes
    with torch.no_grad():
        _, (_, _, att_ref) = model(x)
        _, (_, _, att_ours) = ours(x)
    assert len(att_ours) == len(att_ref) == KW["dec_layers"]
    for (loc_r, w_r), (loc_o, w_o) in zip(att_ref, att_ours):
        assert len(loc_o) == len(loc_r) == KW["num_frames"] + KW["num_future_frames"]
        for a, b in zip(loc_o, loc_r):
            assert a.shape == b.shape and rel_err(a, b) < FWD_TOL
        for a, b in zip(w_o, w_r):
            assert a.shape == b.shape and rel_err(a, b) < FWD_TOL


def test_fused_layer_tails_on_the_reference_layers():
    """The opt-in layer tails + in-kernel encoder reference points applied to the REFERENCE's own layer / encoder
    classes (built with the fused module): inference outputs of the whole network stay at the forward tolerance."""
    import snipper_b200
    from snipper_b200 import ops
    import models.ops.modules as ref_modules
    model = _reference_model()
    x = torch.rand(1, 3 * KW["num_frames"], 192, 256, device=DEV)
    ref_cls = ref_modules.MSDeformAttn
    try:
        snipper_b200.install_module()
        torch.manual_seed(3)
        ours, _ = ref_loader.build_reference_model(use_pytorch_deform=0, **KW)
    finally:
        for name in ("models.ops.modules", "models.ops.modules.ms_deform_attn", "models.deformable_transformer"):
            sys.modules[name].MSDeformAttn = ref_cls
    ours.load_state_dict(model.state_dict(), strict=True)
    ours = ours.to(DEV).eval()
    assert snipper_b200.enable_fused_layer_tails(ours) == KW["enc_layers"] + KW["dec_layers"]
    assert "forward" in ours.transformer.encoder.__dict__                 # the reference's encoder hands out an EncoderGrid
    with torch.no_grad():
        want, _ = model(x)
        ops.STATS.reset()
        ops.STATS.timing = True
        got, _ = ours(x)
        ops.STATS.timing = False
    assert len([e for e in ops.STATS.events if e[0] == "layer_tail"]) == 2 * KW["enc_layers"] + 3 * KW["dec_layers"]
    for k in ("pred_logits", "pred_kpts2d", "pred_depth"):
        assert rel_err(got[k], want[k]) < FWD_TOL, k
    for a, b in zip(got["heatmaps"], want["heatmaps"]):
        assert rel_err(a, b) < FWD_TOL
    assert sorted(ours.state_dict().keys()) == sorted(model.state_dict().keys())
    assert snipper_b200.disable_fused_layer_tails(ours) == KW["enc_layers"] + KW["dec_layers"]
    assert "forward" not in ours.transformer.encoder.__dict__
