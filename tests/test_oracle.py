"""CPU tests that pin the oracle: Oracle-S (C) and the torch restatement against the golden vectors
made from the reference's own modules (fp32, and fp64 for the exact comparisons) and against autograd
of the grid_sample form."""
import numpy as np
import pytest
import torch

from bevformer_b200 import synthetic as syn
from oracle import msda_oracle, torch_ref
from tests.util import (fingerprint_err, fixed_projection, golden, layout, max_err, msda_case_inputs,
                        reference_initialisers, stats, stats_close)

OP_CASES = ["kat", "kat_oob", "config0", "pyramid"]


@pytest.mark.parametrize("case", OP_CASES)
def test_oracle_s_matches_golden(case):
    g = golden("msda_" + case)
    v, ss, lsi, loc, attn = msda_case_inputs(g, torch.float64)
    out = msda_oracle.msda_forward(v, ss, lsi, loc, attn)
    rq, rs = g["rows_q"], g["rows_s"]
    assert max_err(out[:, rq], g["out_rows"]) < 1e-6          # golden rows are stored as fp32
    assert stats_close(stats(out), g["out_stats"], 1e-9)
    gv, gl, ga = msda_oracle.msda_backward(v, ss, lsi, loc, attn,
                                           fixed_projection(out.shape, dtype=torch.float64))
    assert max_err(gv[:, rs], g["grad_value_rows"]) < 1e-5
    assert max_err(gl[:, rq], g["grad_loc_rows"]) < 1e-4
    assert max_err(ga[:, rq], g["grad_attn_rows"]) < 1e-5
    assert stats_close(stats(gv), g["grad_value_stats"], 1e-9)
    assert stats_close(stats(gl), g["grad_loc_stats"], 1e-9)
    assert stats_close(stats(ga), g["grad_attn_stats"], 1e-9)


def test_oracle_s_fp32_against_fp64():
    g = golden("msda_pyramid")
    v, ss, lsi, loc, attn = msda_case_inputs(g, torch.float32)
    out = msda_oracle.msda_forward(v, ss, lsi, loc, attn)
    assert out.dtype == torch.float32
    assert max_err(out[:, g["rows_q"]], g["out_rows"]) < 2e-5


@pytest.mark.parametrize("dim", [4, 30, 32, 64, 71])   # mmcv's gradcheck channel list (SURVEY §4)
def test_oracle_s_equals_grid_sample_autograd(dim):
    v, ss, lsi, loc, attn = syn.make_msda_inputs(2, [(6, 4), (3, 2)], 7, 2, dim, 2, seed=dim,
                                                 dtype=torch.float64, loc_range=(-0.2, 1.2))
    v.requires_grad_(); loc.requires_grad_(); attn.requires_grad_()
    ref = torch_ref.msda_grid_sample(v, ss, loc, attn)
    gout = torch.randn_like(ref)
    ref.backward(gout)
    out = msda_oracle.msda_forward(v, ss, lsi, loc, attn)
    gv, gl, ga = msda_oracle.msda_backward(v, ss, lsi, loc, attn, gout)
    assert max_err(out, ref) < 1e-13
    assert max_err(gv, v.grad) < 1e-13
    assert max_err(gl, loc.grad) < 1e-11
    assert max_err(ga, attn.grad) < 1e-13


def test_oracle_s_gradcheck():
    v, ss, lsi, loc, attn = syn.make_msda_inputs(1, [(5, 4), (3, 2)], 3, 2, 4, 2, seed=1,
                                                 dtype=torch.float64, loc_range=(0.05, 0.95))
    v.requires_grad_(); loc.requires_grad_(); attn.requires_grad_()
    fn = lambda a, b, c: msda_oracle.MSDAOracleFunction.apply(a, ss, lsi, b, c, 64)
    assert torch.autograd.gradcheck(fn, (v, loc, attn), eps=1e-6, atol=1e-4, rtol=1e-3,
                                    nondet_tol=0.0)


def test_oracle_s_properties():
    ss = torch.tensor([[4, 5]]); lsi = torch.tensor([0])
    value = torch.randn(1, 20, 1, 8, dtype=torch.float64)
    # integer pixel centres reproduce value exactly
    ys, xs = torch.meshgrid(torch.arange(4, dtype=torch.float64),
                            torch.arange(5, dtype=torch.float64), indexing="ij")
    loc = torch.stack([(xs + 0.5) / 5, (ys + 0.5) / 4], -1).reshape(1, 20, 1, 1, 1, 2)
    out = msda_oracle.msda_forward(value, ss, lsi, loc, torch.ones(1, 20, 1, 1, 1).double())
    assert max_err(out, value.view(1, 20, 8)) < 1e-14
    # locations at least one pixel outside contribute exactly zero (x <= -1 px or >= W px)
    far = torch.tensor([[-0.5 / 5 - 1e-9, 0.5], [1.0 + 0.5 / 5, 0.5], [0.5, -0.125 - 1e-9],
                        [0.5, 1.125], [1e9, 0.5], [0.5, -1e9]], dtype=torch.float64)
    out = msda_oracle.msda_forward(value, ss, lsi, far.view(1, 6, 1, 1, 1, 2),
                                   torch.ones(1, 6, 1, 1, 1).double())
    assert out.abs().max().item() == 0.0
    # empty query set
    out = msda_oracle.msda_forward(value, ss, lsi, loc[:, :0], torch.ones(1, 0, 1, 1, 1).double())
    assert out.shape == (1, 0, 8)


ENC_CASES = [("toy", "toy", 1, True), ("toy_bs2", "toy", 2, True), ("toy_noprev", "toy", 1, False),
             ("tiny", "tiny", 1, True), ("tiny_noprev", "tiny", 1, False)]


def _enc_inputs(workload, bs, with_prev, seed=0, dtype=torch.float32):
    w = syn.WORKLOADS[workload]
    inp = syn.make_encoder_inputs(w, bs=bs, seed=seed, with_prev=with_prev, dtype=dtype)
    if bs > 1:
        g = torch.Generator().manual_seed(99)
        inp.feat = inp.feat + (0.5 * torch.randn(inp.feat.shape, generator=g)).to(dtype)
        inp.bev_query = inp.bev_query + (0.1 * torch.randn(inp.bev_query.shape, generator=g)).to(dtype)
    return w, inp


@pytest.mark.parametrize("name,workload,bs,with_prev", ENC_CASES)
@pytest.mark.parametrize("use_c", [False, True])
def test_restatement_matches_golden(name, workload, bs, with_prev, use_c):
    g = golden("encoder_" + name)
    w, inp = _enc_inputs(workload, bs, with_prev)
    sd = syn.make_state_dict(w)
    with torch.no_grad():
        out = torch_ref.encoder_forward(sd, w.num_layers, inp.bev_query, inp.feat,
                                        use_c_oracle=use_c, **inp.kwargs())
    assert max_err(out[:, g["rows_q"]], g["out_rows"]) < 2e-4
    if "out_full" in g:
        assert max_err(out, g["out_full"]) < 2e-4
    assert stats_close(stats(out), g["out_stats"], 1e-4)


def test_restatement_backward_matches_golden():
    g = golden("encoder_toy")
    w, inp = _enc_inputs("toy", 1, True)
    sd = {k: v.clone().requires_grad_(True) for k, v in syn.make_state_dict(w).items()}
    inp.bev_query.requires_grad_(True); inp.feat.requires_grad_(True)
    out = torch_ref.encoder_forward(sd, w.num_layers, inp.bev_query, inp.feat, use_c_oracle=True,
                                    **inp.kwargs())
    (out * fixed_projection(out.shape)).sum().backward()
    assert max_err(inp.bev_query.grad[g["rows_q"]], g["grad_query_rows"]) < 5e-4
    assert max_err(inp.feat.grad[:, g["rows_s"]], g["grad_feat_rows"]) < 5e-4
    for k, p in sd.items():
        assert stats_close(stats(p.grad), g["gstat:" + k], 2e-3), k


@pytest.mark.parametrize("bs,with_prev", [(1, True), (2, True), (1, False)])
def test_restatement_vs_reference_fp64(bs, with_prev):
    """Against the reference's unmodified modules, in fp64 (no rounding slack; golden encoder_fp64_toy.npz)."""
    g = golden("encoder_fp64_toy")
    w, inp = _enc_inputs("toy", bs, with_prev, dtype=torch.float64)
    sd = syn.make_state_dict(w, dtype=torch.float64)
    with torch.no_grad():
        out = torch_ref.encoder_forward(sd, w.num_layers, inp.bev_query, inp.feat, **inp.kwargs())
    # point_sampling runs in fp32 in both (encoder.py:87-93); everything else is fp64
    assert fingerprint_err(out, g, f"bs{bs}_{'prev' if with_prev else 'noprev'}:") < 1e-9


def test_state_dict_layout_equals_reference():
    for name in ("tiny", "small", "base"):
        g = golden("encoder_layout_" + name)   # the reference encoder built from its own config
        w = syn.WORKLOADS[name]
        ref_shapes, sd = layout(g), syn.make_state_dict(w)
        assert list(sd.keys()) == list(ref_shapes) or set(sd) == set(ref_shapes)
        for k in sd:
            assert tuple(sd[k].shape) == ref_shapes[k], k
        ref_init = reference_initialisers(g)
        sd0 = syn.make_state_dict(w, trained_like=False)
        for k in sd0:   # the deterministic reference initialisers
            if "sampling_offsets" in k or "attention_weights" in k or "norms" in k:
                assert torch.equal(sd0[k], ref_init[k]), k


def test_rig_hit_counts():
    """SURVEY.md §8d: the synthetic rig gives these per-camera hit counts at base."""
    w = syn.WORKLOADS["base"]
    ref3d = torch_ref.reference_points_3d(w.bev_h, w.bev_w, 8.0, 4, 1, torch.float32)
    _, mask = torch_ref.point_sampling(ref3d, syn.PC_RANGE, syn.make_img_metas(w))
    hits = [(mask[i, 0].sum(-1) > 0).sum().item() for i in range(6)]
    assert hits == [6071, 7481, 7417, 9507, 7049, 6986]


# ---- PerceptionTransformer.get_bev_features (SURVEY.md §8f, first "next" row) -----------------------
PER_CASES = [("toy", "toy", 2, True), ("toy_noprev", "toy", 1, False), ("tiny", "tiny", 1, True)]


def _grid_length(w):
    return (0.512 * 200 / w.bev_h, 0.512 * 200 / w.bev_w)


def _per_restatement(w, inp, sd):
    return torch_ref.get_bev_features(sd, w.num_layers, inp.mlvl_feats, inp.bev_queries, w.bev_h, w.bev_w,
                                      grid_length=_grid_length(w), bev_pos=inp.bev_pos,
                                      prev_bev=inp.prev_bev, img_metas=inp.img_metas,
                                      rotate_center=(w.bev_h // 2, w.bev_w // 2),
                                      tsa_points=w.tsa_points, sca_points=w.sca_points)


@pytest.mark.parametrize("name,workload,bs,with_prev", PER_CASES)
def test_perception_restatement_matches_golden(name, workload, bs, with_prev):
    g = golden("perception_" + name)
    w = syn.WORKLOADS[workload]
    inp = syn.make_perception_inputs(w, bs=bs, with_prev=with_prev)
    sd = {k: v.clone().requires_grad_(True) for k, v in syn.make_perception_state_dict(w).items()}
    for f in inp.mlvl_feats:
        f.requires_grad_(True)
    inp.bev_queries.requires_grad_(True)
    prev0 = None if inp.prev_bev is None else inp.prev_bev.clone()
    out = _per_restatement(w, inp, sd)
    assert max_err(out[:, g["rows_q"]], g["out_rows"]) < 2e-4
    assert stats_close(stats(out), g["out_stats"], 1e-4)
    if prev0 is not None:
        assert torch.equal(prev0, inp.prev_bev)                  # the restatement does not rotate in place
    (out * fixed_projection(out.shape)).sum().backward()
    assert max_err(inp.bev_queries.grad[g["rows_q"]], g["grad_queries_rows"]) < 5e-4
    for i, f in enumerate(inp.mlvl_feats):
        assert max_err(f.grad[:, :, :8, :2], g[f"grad_feat{i}_slice"]) < 5e-4
        assert stats_close(stats(f.grad), g[f"grad_feat{i}_stats"], 2e-3)
    for k in ("level_embeds", "cams_embeds", "can_bus_mlp.0.weight", "can_bus_mlp.norm.bias"):
        assert max_err(sd[k].grad, g["gfull:" + k]) < 2e-3 * max(1.0, float(np.abs(g["gfull:" + k]).max())), k


@pytest.mark.parametrize("bs,with_prev", [(2, True), (1, False)])
def test_perception_restatement_vs_reference_fp64(bs, with_prev):
    """Against the reference's own PerceptionTransformer class in fp64 (golden perception_fp64_toy.npz)."""
    g = golden("perception_fp64_toy")
    w = syn.WORKLOADS["toy"]
    sd = syn.make_perception_state_dict(w)
    inp = syn.make_perception_inputs(w, bs=bs, with_prev=with_prev, dtype=torch.float64)
    with torch.no_grad():
        mine = _per_restatement(w, inp, {k: v.double() for k, v in sd.items()})
    assert fingerprint_err(mine, g, f"bs{bs}_{'prev' if with_prev else 'noprev'}:") < 1e-9


# ---- randomized properties of the op (SURVEY.md §8c item 4), on Oracle-S -------------------------------
from hypothesis import given, settings, strategies as st  # noqa: E402


@st.composite
def _op_shapes(draw):
    levels = draw(st.lists(st.tuples(st.integers(1, 6), st.integers(1, 7)), min_size=1, max_size=3))
    return dict(bs=draw(st.integers(1, 2)), levels=levels, nq=draw(st.integers(1, 6)),
                heads=draw(st.integers(1, 3)), dim=draw(st.sampled_from([1, 4, 7, 32])),
                pts=draw(st.integers(1, 3)), seed=draw(st.integers(0, 10_000)))


@settings(max_examples=40, deadline=None)
@given(_op_shapes())
def test_oracle_s_random_properties(sh):
    v, ss, lsi, loc, attn = syn.make_msda_inputs(sh["bs"], sh["levels"], sh["nq"], sh["heads"], sh["dim"],
                                                 sh["pts"], seed=sh["seed"], dtype=torch.float64,
                                                 loc_range=(-0.6, 1.6))
    out = msda_oracle.msda_forward(v, ss, lsi, loc, attn)
    # equals the grid_sample formulation the reference falls back to (mmcv's pure-PyTorch path)
    want = torch_ref.msda_grid_sample(v, [tuple(x) for x in ss.tolist()], loc, attn)
    assert max_err(out, want) < 1e-12
    # permuting the queries permutes the output rows
    perm = torch.randperm(sh["nq"], generator=torch.Generator().manual_seed(sh["seed"]))
    assert max_err(msda_oracle.msda_forward(v, ss, lsi, loc[:, perm], attn[:, perm]), out[:, perm]) == 0.0
    # linear in value and in the attention weights
    assert max_err(msda_oracle.msda_forward(2.5 * v, ss, lsi, loc, attn), 2.5 * out) < 1e-12
    assert max_err(msda_oracle.msda_forward(v, ss, lsi, loc, 0.5 * attn), 0.5 * out) < 1e-12
    # samples a full pixel outside the map contribute nothing: pushing every location there zeroes the output
    assert msda_oracle.msda_forward(v, ss, lsi, loc * 0 + 7.0, attn).abs().max().item() == 0.0
    # backward is the exact transpose: <grad_out, J dv> == <J^T grad_out, dv>
    g = torch.randn(out.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(1 + sh["seed"]))
    gv, _, _ = msda_oracle.msda_backward(v, ss, lsi, loc, attn, g)
    dv = torch.randn(v.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(2 + sh["seed"]))
    lhs = (g * msda_oracle.msda_forward(dv, ss, lsi, loc, attn)).sum()
    assert abs(lhs.item() - (gv * dv).sum().item()) < 1e-9 * max(1.0, abs(lhs.item()))
