"""The bench harness network (snipper_b200/harness) is a faithful restatement of the reference
model: load the REAL reference's state_dict into it and compare outputs on CPU.  Runs only in
the build container (skipped where /root/reference is absent)."""
import pytest
import torch

import ref_loader
from conftest import rel_err
from oracle import torch_ref

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason="original Snipper source tree not found (set SNIPPER_REFERENCE to it)")


@pytest.mark.parametrize("num_future", [0, 2])
def test_harness_matches_reference_model(num_future):
    from snipper_b200.harness.snipper_net import build_snipper
    torch.manual_seed(0)
    kw = dict(hidden_dim=96, num_frames=2, num_future_frames=num_future, enc_layers=1, dec_layers=2,
              num_queries=5, dim_feedforward=64, dropout=0.0)
    ref_model, args = ref_loader.build_reference_model(use_pytorch_deform=1, **kw)
    ref_model.eval()
    with torch.no_grad():  # leave the degenerate init so the attention actually depends on the queries
        for n, p in ref_model.named_parameters():
            if "sampling_offsets" in n and n.endswith("weight"):
                p.normal_(0, 0.05)
            if "attention_weights" in n:
                p.normal_(0, 0.2)
    mine = build_snipper(torch_ref.SnippetMSDeformAttnRef, **kw).eval()
    missing, unexpected = mine.load_state_dict(ref_model.state_dict(), strict=True)
    assert not missing and not unexpected
    x = torch.rand(1, 3 * 2, 96, 128)
    with torch.no_grad():
        want, (w_ref0, w_refs, w_att) = ref_model(x)
        got, (g_ref0, g_refs, g_att) = mine(x)
    for k in ("pred_logits", "pred_kpts2d", "pred_depth"):
        assert rel_err(got[k], want[k]) < 1e-5, k
    for a, b in zip(got["heatmaps"], want["heatmaps"]):
        assert rel_err(a, b) < 1e-5
    for a, b in zip(got["aux_outputs"], want["aux_outputs"]):
        for k in a:
            assert rel_err(a[k], b[k]) < 1e-5
    assert rel_err(g_refs, w_refs) < 1e-5
    assert len(g_att) == len(w_att)


def test_drop_in_surfaces_rebind_the_unmodified_reference():
    """install_module() makes the reference's own build_model construct the fused class (surface 3) with the
    reference's state-dict layout; install_extension_shim() rebinds the name the reference's
    MSDeformAttnFunction resolves at call time (surface 1, ms_deform_attn_func.py:28,38)."""
    import sys
    import snipper_b200
    kw = dict(hidden_dim=96, num_frames=2, num_future_frames=1, enc_layers=2, dec_layers=3, num_queries=5,
              dim_feedforward=64, use_pytorch_deform=0)
    ref_model, _ = ref_loader.build_reference_model(**kw)
    import models.deformable_transformer as dt
    import models.ops.modules as ref_modules
    ref_cls = ref_modules.MSDeformAttn
    assert sum(isinstance(m, ref_cls) for m in ref_model.modules()) == 2 + 3
    try:
        snipper_b200.install_module()
        assert dt.MSDeformAttn is snipper_b200.MSDeformAttn
        ours, _ = ref_loader.build_reference_model(**kw)
        mods = [m for m in ours.modules() if isinstance(m, snipper_b200.MSDeformAttn)]
        assert len(mods) == 2 + 3 and not any(isinstance(m, ref_cls) for m in ours.modules())
        assert [m.mode for m in mods] == ["encoder"] * 2 + ["decoder"] * 3
        assert [m.attention_vis for m in mods] == [False] * 2 + [True] * 3
        assert all(m.n_frame == 2 and m.d_model == 96 for m in mods)
        # DeformableTransformer._reset_parameters type-tests the class (deformable_transformer.py:62-64): ours was re-initialised
        assert all(float(m.sampling_offsets[0].weight.abs().max()) == 0.0 for m in mods)
        missing, unexpected = ours.load_state_dict(ref_model.state_dict(), strict=True)   # same keys, aliased slots included
        assert not missing and not unexpected
    finally:
        for name in ("models.ops.modules", "models.ops.modules.ms_deform_attn", "models.deformable_transformer"):
            sys.modules[name].MSDeformAttn = ref_cls
    import models.ops.functions.ms_deform_attn_func as ref_func
    before = getattr(ref_func, "MSDA", None)
    try:
        shim = snipper_b200.install_extension_shim()
        assert ref_func.MSDA is shim and hasattr(shim, "ms_deform_attn_forward") and hasattr(shim, "ms_deform_attn_backward")
    finally:
        if before is not None:
            ref_func.MSDA = before
