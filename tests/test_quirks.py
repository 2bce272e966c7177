"""One test per observable item of SURVEY.md Appendix D (the reference's quirk checklist).

CPU half (no marker): the repo-resident restatement reproduces the quirk exactly as the reference's own
unmodified modules do (Oracle-R, through golden fp64 results).  GPU half (``gpu`` marker): the CUDA drop-in
reproduces it against the restatement.  Quirks 2, 3, 4, 6, 7, 8, 9 and 12 are exercised by every golden
encoder case (bs = 2, with / without prev_bev, non-zero shift, eval mode); the scenarios here isolate the
ones a golden case with a single rig and identical image shapes cannot see: 1, 5, 10, 11 (and 8b)."""
import copy

import numpy as np
import pytest
import torch

from bevformer_b200 import synthetic as syn
from oracle import torch_ref
from tests.util import fingerprint_err, golden, max_err, rel_err

W = syn.WORKLOADS["toy"]


def _yawed(l2i, deg):
    """lidar2img of a rig rotated about the ego z axis."""
    a = np.deg2rad(deg)
    rot = np.eye(4)
    rot[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    return [m @ rot for m in l2i]


def scenario(kind, dtype=torch.float32):
    """(inputs, description) for a quirk scenario on the toy workload, bs = 2."""
    inp = syn.make_encoder_inputs(W, bs=2, seed=3, dtype=dtype)
    g = torch.Generator().manual_seed(5)
    inp.feat = inp.feat + (0.5 * torch.randn(inp.feat.shape, generator=g)).to(dtype)
    metas = copy.deepcopy(inp.img_metas)
    if kind == "q1":       # sample 1 sees the scene through a rig yawed by 25 degrees: its own bev_mask differs
        metas[1]["lidar2img"] = _yawed(metas[1]["lidar2img"], 25.0)
    elif kind == "q10":    # other image shapes for sample 1 / cameras >= 1: must be ignored (img_metas[0][..][0] rules)
        h, wd = W.img_hw
        metas[0]["img_shape"] = [(h, wd, 3)] + [(h // 2, wd * 3, 3)] * (W.num_cams - 1)
        metas[1]["img_shape"] = [(h * 2, wd // 2, 3)] * W.num_cams
    inp.img_metas = metas
    return inp


def _restatement(inp, dtype=torch.float32):
    sd = syn.make_state_dict(W, dtype=dtype)
    with torch.no_grad():
        return torch_ref.encoder_forward(sd, W.num_layers, inp.bev_query, inp.feat, **inp.kwargs())


# ---------------------------------------------------------------------------------------------------
# CPU: restatement == the reference's own modules under each scenario
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["q1", "q10"])
def test_restatement_reproduces_quirk_like_reference(kind):
    """fp64, against the reference encoder's result on the same scenario (golden encoder_fp64_toy.npz)."""
    inp = scenario(kind, torch.float64)
    assert fingerprint_err(_restatement(inp, torch.float64), golden("encoder_fp64_toy"), kind + ":") < 1e-9


def test_quirk1_is_visible_in_the_scenario():
    """The scenario is not vacuous: sample 1's own mask differs from sample 0's, and using it for the
    hit lists would change the result."""
    inp = scenario("q1")
    ref3d = torch_ref.reference_points_3d(W.bev_h, W.bev_w, 8.0, 4, 2, torch.float32)
    _, mask = torch_ref.point_sampling(ref3d, syn.PC_RANGE, inp.img_metas)
    seen = mask.any(-1)                                   # (cam, bs, Nq)
    assert (seen[:, 0] != seen[:, 1]).any()
    base = scenario("none")
    assert rel_err(_restatement(inp)[1], _restatement(base)[1]) > 1e-3


def test_quirk10_image_shape_of_other_samples_is_ignored():
    assert max_err(_restatement(scenario("q10")), _restatement(scenario("none"))) == 0.0


def test_quirk5_unseen_queries_get_the_output_bias():
    """slots / count happens before output_proj: a query no camera sees leaves SCA as
    output_proj.bias + residual (spatial_cross_attention.py:169-175).  tiny config: the five queries
    around the ego origin project into no camera."""
    w = syn.WORKLOADS["tiny"]
    inp = syn.make_encoder_inputs(w, bs=1, seed=2)
    sd = syn.make_state_dict(w)
    ref3d = torch_ref.reference_points_3d(w.bev_h, w.bev_w, 8.0, 4, 1, torch.float32)
    ref_cam, mask = torch_ref.point_sampling(ref3d, syn.PC_RANGE, inp.img_metas)
    unseen = ~mask.any(-1).any(0)[0]                      # (Nq,)
    assert unseen.any()
    q = inp.bev_query.permute(1, 0, 2)
    pre = "layers.0.attentions.1."
    out = torch_ref.spatial_cross_attention(sd, pre, q, inp.feat, ref_cam, mask,
                                            [tuple(x) for x in inp.spatial_shapes.tolist()],
                                            inp.level_start_index.tolist(), torch_ref._sampler(False), 8,
                                            w.sca_points)
    want = q[0, unseen] + sd[pre + "output_proj.bias"]
    assert max_err(out[0, unseen], want) < 1e-6


# ---------------------------------------------------------------------------------------------------
# GPU: the CUDA drop-in reproduces them
# ---------------------------------------------------------------------------------------------------
def _plugin(dtype=torch.float32):
    from bevformer_b200.plugin import build_transformer_layer_sequence
    enc = build_transformer_layer_sequence(syn.encoder_cfg(W))
    enc.load_state_dict(syn.make_state_dict(W))
    return enc.to("cuda", dtype).eval()


def _to_cuda(inp):
    for k in ("bev_query", "feat", "bev_pos", "prev_bev", "shift", "spatial_shapes", "level_start_index"):
        t = getattr(inp, k)
        if t is not None:
            setattr(inp, k, t.to("cuda"))
    return inp


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["q1", "q10", "none"])
def test_plugin_reproduces_quirk(kind):
    want = _restatement(scenario(kind))
    inp = _to_cuda(scenario(kind))
    with torch.no_grad():
        got = _plugin()(inp.bev_query, inp.feat, inp.feat, **inp.kwargs())
    assert rel_err(got, want) < 1e-3, kind


@pytest.mark.gpu
def test_plugin_quirk5_unseen_queries_get_the_output_bias():
    from bevformer_b200 import ops
    from bevformer_b200.plugin import ScaPlan, build_transformer_layer_sequence
    w = syn.WORKLOADS["tiny"]
    enc = build_transformer_layer_sequence(syn.encoder_cfg(w))
    enc.load_state_dict(syn.make_state_dict(w))
    enc = enc.cuda().eval()
    inp = _to_cuda(syn.make_encoder_inputs(w, bs=1, seed=2))
    l2i = torch.as_tensor(np.asarray([m["lidar2img"] for m in inp.img_metas], dtype=np.float32)).cuda()
    z = (torch.linspace(0.5, 7.5, 4) / 8.0).tolist()
    ref_cam, mask = ops.point_sampling(l2i, syn.PC_RANGE, z, w.img_hw[0], w.img_hw[1], w.bev_h, w.bev_w)
    unseen = ~mask.bool().any(-1).any(0)[0]
    assert unseen.any()
    sca = enc.layers[0].attentions[1]
    q = inp.bev_query.permute(1, 0, 2).contiguous()
    with torch.no_grad():
        pre = sca.attend(q, inp.feat, ref_cam, mask.bool(), inp.spatial_shapes, inp.level_start_index,
                         ScaPlan.build(mask.bool(), ref_cam))
    assert max_err(pre[0, unseen], sca.output_proj.bias.expand(int(unseen.sum()), -1)) < 1e-5


@pytest.mark.gpu
def test_plugin_quirk11_fp32_function_under_autocast():
    """MultiScaleDeformableAttnFunction_fp32 computes in fp32 under autocast (…function.py:93)."""
    from bevformer_b200 import ops
    v, ss, lsi, loc, attn = syn.make_msda_inputs(1, [(6, 4), (3, 2)], 5, 8, 32, 2, seed=1)
    v, ss, lsi, loc, attn = (t.cuda() for t in (v, ss, lsi, loc, attn))
    with torch.autocast("cuda", dtype=torch.float16):
        out = ops.MultiScaleDeformableAttnFunction_fp32.apply(v.half(), ss, lsi, loc.half(), attn.half(), 64)
    assert out.dtype == torch.float32


@pytest.mark.gpu
def test_plugin_quirk8b_no_prev_bev_restacks_each_layers_query():
    """prev_bev=None: every layer's TSA stacks its own current query twice (encoder.py:214-232 with
    temporal_self_attention.py:177-180), not the layer-0 input."""
    inp = syn.make_encoder_inputs(W, bs=1, seed=4, with_prev=False)
    want = _restatement(inp)
    inp = _to_cuda(inp)
    with torch.no_grad():
        got = _plugin()(inp.bev_query, inp.feat, inp.feat, **inp.kwargs())
    assert rel_err(got, want) < 1e-3
