"""Host-side logic of the drop-in plugin that needs no GPU: registry names, constructor contracts,
state_dict layout, initialisers, the SCA pair plan, config reading."""
import os

import pytest
import torch

from bevformer_b200 import synthetic as syn
from bevformer_b200.plugin import (ATTENTION, TRANSFORMER_LAYER, TRANSFORMER_LAYER_SEQUENCE, ScaPlan,
                                   build_transformer_layer_sequence, config)
from oracle import torch_ref
from tests.util import golden, layout, reference_initialisers


def test_registry_names():
    for reg, names in ((ATTENTION, ["TemporalSelfAttention", "SpatialCrossAttention",
                                    "MSDeformableAttention3D"]),
                       (TRANSFORMER_LAYER, ["BEVFormerLayer", "MyCustomBaseTransformerLayer"]),
                       (TRANSFORMER_LAYER_SEQUENCE, ["BEVFormerEncoder"])):
        for n in names:
            assert reg.get(n) is not None, n


def test_dropin_import_paths():
    from projects.mmdet3d_plugin.bevformer.modules import (BEVFormerEncoder, BEVFormerLayer,  # noqa
                                                           MSDeformableAttention3D,
                                                           SpatialCrossAttention,
                                                           TemporalSelfAttention)
    from projects.mmdet3d_plugin.bevformer.modules.multi_scale_deformable_attn_function import (  # noqa
        MultiScaleDeformableAttnFunction_fp16, MultiScaleDeformableAttnFunction_fp32)
    from projects.mmdet3d_plugin.bevformer.modules.spatial_cross_attention import (  # noqa
        MultiScaleDeformableAttnFunction_fp32 as again)
    assert again is MultiScaleDeformableAttnFunction_fp32


@pytest.mark.parametrize("name", ["toy", "small4"])
def test_build_from_spelled_out_cfg(name):
    w = syn.WORKLOADS[name]
    enc = build_transformer_layer_sequence(syn.encoder_cfg(w))
    enc.load_state_dict(syn.make_state_dict(w), strict=True)
    assert len(enc.layers) == w.num_layers and enc.embed_dims == 256 and not enc.pre_norm
    per_layer = sum(p.numel() for p in enc.layers[0].parameters())
    if name == "small4":
        assert per_layer == 823488        # SURVEY.md Appendix C


@pytest.mark.parametrize("name", ["tiny", "small", "base"])
def test_build_from_unchanged_reference_config(name, tmp_path):
    """A config file carrying the encoder dict that the reference's shipped config evaluates to builds the
    encoder the reference builds from that config (golden encoder_layout_<name>.npz)."""
    g = golden("encoder_layout_" + name)
    path = tmp_path / os.path.basename(syn.WORKLOADS[name].config_file)
    path.write_text(f"model = dict(pts_bbox_head=dict(transformer=dict(encoder={g['cfg'].item()})))\n")
    enc = config.build_encoder(str(path))
    ours, theirs = enc.state_dict(), layout(g)
    assert list(ours.keys()) == list(theirs)
    for k in ours:
        assert tuple(ours[k].shape) == theirs[k], k
    # deterministic initialisers agree exactly (ring bias, zero logits, LN)
    ref_init = reference_initialisers(g)
    for k in ours:
        if "sampling_offsets" in k or "attention_weights" in k or ".norms." in k:
            assert torch.equal(ours[k], ref_init[k]), k
    assert sum(p.numel() for p in enc.parameters()) == int(g["nparams"]) == {"tiny": 2026368, "small": 2026368,
                                                                             "base": 4940928}[name]


def test_constructor_errors_match_reference():
    from bevformer_b200.plugin import MSDeformableAttention3D, TemporalSelfAttention
    with pytest.raises(ValueError, match="divisible"):
        TemporalSelfAttention(embed_dims=250, num_heads=8)
    with pytest.raises(ValueError, match="divisible"):
        MSDeformableAttention3D(embed_dims=250, num_heads=8)
    with pytest.raises(AssertionError):
        build_transformer_layer_sequence(dict(
            type="BEVFormerEncoder", num_layers=1, pc_range=syn.PC_RANGE,
            transformerlayers=dict(type="BEVFormerLayer", attn_cfgs=[
                dict(type="TemporalSelfAttention", embed_dims=256, num_levels=1)],
                feedforward_channels=512, operation_order=("self_attn", "norm"))))


def test_sca_plan_matches_reference_rebatch():
    """The compact pair list is the reference's per-camera nonzero lists, concatenated; the divisor
    is the per-item camera count (spatial_cross_attention.py:138-141,169-171)."""
    w = syn.WORKLOADS["toy"]
    ref3d = torch_ref.reference_points_3d(w.bev_h, w.bev_w, 8.0, 4, 2, torch.float32)
    metas = syn.make_img_metas(w, 2)
    metas[1]["lidar2img"] = [m.copy() for m in metas[1]["lidar2img"]]
    metas[1]["lidar2img"][0][0, 3] += 30.0            # batch item 1 sees something else
    ref_cam, mask = torch_ref.point_sampling(ref3d, syn.PC_RANGE, metas)
    plan = ScaPlan.build(mask, ref_cam)
    lists = [mask[i, 0].sum(-1).nonzero().squeeze(-1) for i in range(w.num_cams)]
    assert plan.num_pairs == sum(len(x) for x in lists)
    assert torch.equal(plan.pair_q.long(), torch.cat(lists))
    assert torch.equal(plan.pair_cam.long(),
                       torch.cat([torch.full((len(x),), i) for i, x in enumerate(lists)]))
    count = (mask.sum(-1) > 0).permute(1, 2, 0).sum(-1).clamp(min=1.0)
    assert torch.allclose(plan.inv_count, 1.0 / count)
    r = plan.num_pairs
    assert torch.equal(plan.row_map[:r].long(), plan.pair_cam.long())
    assert torch.equal(plan.row_map[r:].long(), plan.pair_cam.long() + w.num_cams)
    back = plan.pair_of[plan.pair_cam.long(), plan.pair_q.long()]
    assert torch.equal(back.long(), torch.arange(r))
    assert (plan.pair_of >= 0).sum().item() == r


def test_get_reference_points_matches_reference_formula():
    from bevformer_b200.plugin import BEVFormerEncoder
    a = BEVFormerEncoder.get_reference_points(6, 5, 8, 4, "3d", 2, "cpu", torch.float32)
    b = torch_ref.reference_points_3d(6, 5, 8.0, 4, 2, torch.float32)
    assert torch.equal(a, b)
    a2 = BEVFormerEncoder.get_reference_points(6, 5, dim="2d", bs=2, device="cpu", dtype=torch.float32)
    assert torch.equal(a2, torch_ref.reference_points_2d(6, 5, 2, torch.float32))


def test_no_cpu_fallback():
    w = syn.WORKLOADS["toy"]
    enc = build_transformer_layer_sequence(syn.encoder_cfg(w)).eval()
    inp = syn.make_encoder_inputs(w)
    with pytest.raises(RuntimeError, match="CUDA"):
        enc(inp.bev_query, inp.feat, inp.feat, **inp.kwargs())


def _toy_perception_transformer(cls):
    w = syn.WORKLOADS["toy"]
    return cls(num_feature_levels=len(w.levels), num_cams=w.num_cams, encoder=syn.encoder_cfg(w), decoder=None,
               embed_dims=w.embed_dims)


def test_perception_transformer_state_dict_matches_reference():
    """Same parameter names and shapes as the reference PerceptionTransformer (decoder=None; golden
    perception_layout_toy.npz)."""
    from bevformer_b200.plugin import PerceptionTransformer
    g = golden("perception_layout_toy")
    ours = _toy_perception_transformer(PerceptionTransformer)
    a = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    b = layout(g, "pt:layout")
    assert a == b
    ours.load_state_dict({k: torch.zeros(s) for k, s in b.items()})


def test_perception_transformer_has_no_cpu_path():
    from bevformer_b200.plugin import PerceptionTransformer
    w = syn.WORKLOADS["toy"]
    m = PerceptionTransformer(num_feature_levels=len(w.levels), num_cams=w.num_cams,
                              encoder=syn.encoder_cfg(w), decoder=None, embed_dims=w.embed_dims)
    inp = syn.make_perception_inputs(w, bs=1)
    with pytest.raises(RuntimeError):
        m.get_bev_features(inp.mlvl_feats, inp.bev_queries, w.bev_h, w.bev_w, bev_pos=inp.bev_pos,
                           prev_bev=inp.prev_bev, img_metas=inp.img_metas)


def test_patch_reference_installs_get_bev_features():
    """INTEGRATION.md: the reference class keeps its decoder forward and gains our get_bev_features.  The
    class patched here carries exactly the public attributes and submodules the reference's constructor sets
    (golden perception_layout_toy.npz) and methods of its own under the patched names."""
    import ast
    from bevformer_b200.plugin.transformer import PerceptionTransformer, patch_reference
    g = golden("perception_layout_toy")

    def _own(self, *a, **k):
        raise AssertionError("the class's own method ran")

    ref_cls = type("ReferenceLike", (PerceptionTransformer,),
                   {"forward": _own, "get_bev_features": _own, "_shift": _own, "_rotate_prev": _own})
    sub = type("Patched", (ref_cls,), {})          # patch a subclass: the stand-in class stays pristine
    patch_reference(sub)
    assert sub.get_bev_features is PerceptionTransformer.get_bev_features
    assert sub._shift is PerceptionTransformer._shift and sub._rotate_prev is PerceptionTransformer._rotate_prev
    assert sub.forward is ref_cls.forward
    w = syn.WORKLOADS["toy"]
    m = _toy_perception_transformer(sub)
    ref_attrs = ast.literal_eval(g["pt:attrs"].item())
    assert {k: v for k, v in vars(m).items() if k in ref_attrs} == ref_attrs
    assert list(m._modules) == [str(k) for k in g["pt:modules"]]
    inp = syn.make_perception_inputs(w, bs=1)
    with pytest.raises(RuntimeError, match="CUDA"):     # our method runs (and refuses CPU tensors)
        m.get_bev_features(inp.mlvl_feats, inp.bev_queries, w.bev_h, w.bev_w, bev_pos=inp.bev_pos,
                           prev_bev=inp.prev_bev, img_metas=inp.img_metas)
