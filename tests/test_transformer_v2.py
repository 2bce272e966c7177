"""BEVFormerV2's BEV-encoder wrapper (SURVEY.md §8f rank 4): restatement against the reference's own
class on CPU, CUDA drop-in against the restatement on GPU -- with and without the BEV augmentation
resampling branch."""
import numpy as np
import pytest
import torch

from bevformer_b200 import synthetic as syn
from oracle import torch_ref
from tests.util import fingerprint_err, golden, layout, rel_err

W = syn.WORKLOADS["toy"]


def _metas(bs, aug):
    metas = syn.make_img_metas(W, bs)
    if aug is not None:
        a = np.deg2rad(12.0)
        mat = torch.tensor([[np.cos(a), -np.sin(a), 0, 0], [np.sin(a), np.cos(a), 0, 0],
                            [0, 0, 1, 0], [0, 0, 0, 1]], dtype=torch.float32) * 1.05
        for m in metas:
            m["aug_param"] = {"GlobalRotScaleTransImage_param": (12.0, 1.05, False, False, mat, aug == "only_gt")}
    return metas


def _sd(dtype=torch.float32):
    sd = syn.make_perception_state_dict(W)
    return {k: v.to(dtype) for k, v in sd.items()
            if k.startswith("encoder.") or k in ("level_embeds", "cams_embeds")}


def _restatement(inp, metas, sd):
    return torch_ref.bev_encoder_v2(sd, W.num_layers, inp.mlvl_feats, inp.bev_queries, W.bev_h, W.bev_w,
                                    bev_pos=inp.bev_pos, img_metas=metas, tsa_points=W.tsa_points,
                                    sca_points=W.sca_points)


@pytest.mark.parametrize("aug", [None, "only_gt", "images_too"])
@pytest.mark.parametrize("bs", [1, 2])
def test_restatement_vs_reference_class_fp64(aug, bs):
    """Against the reference class's fp64 result on the same inputs (golden v2_encoder_fp64_toy.npz)."""
    if aug == "only_gt" and bs > 1:
        pytest.skip("the reference's resampling branch builds a batch-1 grid: it only runs with 1 sample per GPU")
    inp = syn.make_perception_inputs(W, bs=bs, dtype=torch.float64)
    with torch.no_grad():
        got = _restatement(inp, _metas(bs, aug), _sd(torch.float64))
    assert fingerprint_err(got, golden("v2_encoder_fp64_toy"), f"{aug}_bs{bs}:") < 1e-9


# constructor options whose state_dict layout is compared with the reference class
V2_EXTRA_KWARGS = (dict(), dict(use_cams_embeds=False))


def test_dropin_parameters_match_reference():
    from bevformer_b200.plugin import PerceptionTransformerBEVEncoder
    g = golden("perception_layout_toy")
    kw = dict(num_feature_levels=len(W.levels), num_cams=W.num_cams, encoder=syn.encoder_cfg(W), embed_dims=W.embed_dims)
    for i, extra in enumerate(V2_EXTRA_KWARGS):
        a = PerceptionTransformerBEVEncoder(**kw, **extra)
        assert {k: tuple(v.shape) for k, v in a.state_dict().items()} == layout(g, f"v2_{i}:layout")


def test_no_cpu_path():
    from bevformer_b200.plugin import PerceptionTransformerBEVEncoder
    m = PerceptionTransformerBEVEncoder(num_feature_levels=len(W.levels), num_cams=W.num_cams,
                                        encoder=syn.encoder_cfg(W), embed_dims=W.embed_dims)
    inp = syn.make_perception_inputs(W, bs=1)
    with pytest.raises(RuntimeError):
        m(inp.mlvl_feats, inp.bev_queries, W.bev_h, W.bev_w, bev_pos=inp.bev_pos, img_metas=inp.img_metas)


@pytest.mark.gpu
@pytest.mark.parametrize("aug", [None, "only_gt", "images_too"])
def test_dropin_on_gpu_vs_restatement(aug):
    from bevformer_b200.plugin import PerceptionTransformerBEVEncoder
    bs = 2
    m = PerceptionTransformerBEVEncoder(num_feature_levels=len(W.levels), num_cams=W.num_cams,
                                        encoder=syn.encoder_cfg(W), embed_dims=W.embed_dims)
    sd = _sd()
    m.load_state_dict(sd)
    m = m.cuda().eval()
    metas = _metas(bs, aug)
    cpu = syn.make_perception_inputs(W, bs=bs)
    with torch.no_grad():
        want = _restatement(cpu, metas, sd)
    dev = syn.make_perception_inputs(W, bs=bs, device="cuda")
    with torch.no_grad():
        got = m(dev.mlvl_feats, dev.bev_queries, W.bev_h, W.bev_w, bev_pos=dev.bev_pos, prev_bev=dev.prev_bev,
                img_metas=metas)
    assert got.shape == want.shape
    assert rel_err(got.cpu(), want) < 1e-3


# ------------------------------------------------------------------------------------------------
# PerceptionTransformerV2 + ResNetFusion (transformerV2.py:16-51, 177-353)
# ------------------------------------------------------------------------------------------------
def _build_v2(w):
    import copy
    from bevformer_b200.plugin import PerceptionTransformerV2
    from tests.golden.make_golden import V2_KW
    m = PerceptionTransformerV2(num_feature_levels=len(w.levels), num_cams=w.num_cams, encoder=syn.encoder_cfg(w),
                                decoder=copy.deepcopy(syn.DECODER_CFG), embed_dims=w.embed_dims,
                                rotate_center=[w.bev_h // 2, w.bev_w // 2], **V2_KW)
    m.load_state_dict(syn.make_random_state_dict(m, 0))
    return m


def test_v2_parameters_match_reference_class():
    from tests.util import golden
    w = syn.WORKLOADS["toy"]
    m = _build_v2(w)
    assert sorted(m.state_dict()) == [str(k) for k in golden("v2_toy")["keys"]]
    assert hasattr(m, "fusion") and len(m.fusion.layers) == 2 and m.fusion.layers[0].downsample is None


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_v2_forward_against_reference_golden(dtype):
    from tests.golden.make_golden import grid_length_of, v2_inputs
    from tests.util import golden, rel_err
    g = golden("v2_toy")
    w = syn.WORKLOADS["toy"]
    m = _build_v2(w).to("cuda", dtype).eval()
    inp, oq, reg = v2_inputs(w)
    feats = [f.to("cuda", dtype) for f in inp.mlvl_feats]
    with torch.no_grad():
        bev, states, ref0, refs = m(feats, inp.bev_queries.to("cuda", dtype), oq.to("cuda", dtype), w.bev_h, w.bev_w,
                                    grid_length=list(grid_length_of(w)), bev_pos=inp.bev_pos.to("cuda", dtype),
                                    reg_branches=reg.to("cuda", dtype), cls_branches=None,
                                    prev_bev=[inp.prev_bev.to("cuda", dtype), None], img_metas=inp.img_metas)
    tol = 2e-3 if dtype == torch.float32 else 8e-2     # fp32: cuDNN convolutions (TF32 off) + 9 layers; bf16 encoder-level bar
    assert rel_err(bev.float().cpu(), g["bev"]) < tol
    assert rel_err(states.float().cpu(), g["states"]) < tol
    assert rel_err(ref0.float().cpu(), g["ref0"]) < 1e-2 and rel_err(refs.float().cpu(), g["refs"]) < 3e-2
