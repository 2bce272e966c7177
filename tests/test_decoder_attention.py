"""CustomMSDeformableAttention (decoder cross-attention, SURVEY.md §8f rank 2): the third call site of the
sampler.  CPU: the restatement and the drop-in's module logic against the reference's own class; GPU:
the drop-in on the CUDA kernels against the restatement."""
import pytest
import torch

from oracle import torch_ref
from tests.util import fingerprint_err, golden, max_err, rel_err


def make_case(levels, nq, bs, ref_dim, seed=0, dtype=torch.float32, with_mask=False):
    g = torch.Generator().manual_seed(100 + seed)
    c = 256
    s = sum(h * w for h, w in levels)
    query = torch.randn(nq, bs, c, generator=g)
    qpos = torch.randn(nq, bs, c, generator=g) * 0.3
    value = torch.randn(s, bs, c, generator=g)
    if ref_dim == 2:
        ref = torch.rand(bs, nq, len(levels), 2, generator=g) * 1.2 - 0.1
    else:
        ref = torch.cat([torch.rand(bs, nq, len(levels), 2, generator=g),
                         torch.rand(bs, nq, len(levels), 2, generator=g) * 0.3], -1)
    mask = (torch.rand(bs, s, generator=g) < 0.1) if with_mask else None
    ss = torch.tensor(levels, dtype=torch.int64)
    lsi = torch.cat([ss.new_zeros(1), ss.prod(1).cumsum(0)[:-1]])
    return dict(query=query.to(dtype), query_pos=qpos.to(dtype), value=value.to(dtype),
                reference_points=ref.to(dtype), key_padding_mask=mask, spatial_shapes=ss,
                level_start_index=lsi)


def make_sd(levels, points, seed=0, dtype=torch.float32):
    """Trained-like parameters with the reference's key names; the same values in every run (the
    projections keep their xavier initialisation, drawn from a seeded generator)."""
    from bevformer_b200.plugin import CustomMSDeformableAttention
    with torch.random.fork_rng():
        torch.manual_seed(300 + seed)
        m = CustomMSDeformableAttention(num_levels=len(levels), num_points=points)
    g = torch.Generator().manual_seed(200 + seed)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    sd["sampling_offsets.weight"] = torch.randn(sd["sampling_offsets.weight"].shape, generator=g) * 0.02
    sd["attention_weights.weight"] = torch.randn(sd["attention_weights.weight"].shape, generator=g) * 0.1
    sd["attention_weights.bias"] = torch.randn(sd["attention_weights.bias"].shape, generator=g) * 0.1
    for k in ("value_proj.bias", "output_proj.bias"):
        sd[k] = torch.randn(sd[k].shape, generator=g) * 0.02
    return {k: v.to(dtype) for k, v in sd.items()}


CASES = [([(12, 10)], 4, 7, 2, 2, False), ([(8, 14), (4, 7)], 4, 9, 1, 2, True),
         ([(8, 14), (4, 7)], 2, 5, 2, 4, False)]


def _restatement(sd, case, points):
    out = torch_ref.custom_ms_deformable_attention(
        sd, "", case["query"].permute(1, 0, 2), case["value"].permute(1, 0, 2), case["reference_points"],
        case["spatial_shapes"], torch_ref._sampler(False), query_pos=case["query_pos"].permute(1, 0, 2),
        key_padding_mask=case["key_padding_mask"], num_points=points)
    return out.permute(1, 0, 2)


# constructor calls whose state_dict and deterministic initialisers are compared with the reference class
INIT_KWARGS = (dict(), dict(num_levels=1, num_points=8, num_heads=4), dict(batch_first=True))
INIT_KEYS = ("sampling_offsets.weight", "sampling_offsets.bias", "attention_weights.weight",
             "attention_weights.bias", "value_proj.bias")


@pytest.mark.parametrize("levels,points,nq,bs,ref_dim,with_mask", CASES)
def test_restatement_vs_reference_class_fp64(levels, points, nq, bs, ref_dim, with_mask):
    """Against the reference's own class in fp64 (golden decoder_attention_ref.npz, tests/golden/make_golden.py)."""
    g = golden("decoder_attention_ref")
    i = CASES.index((levels, points, nq, bs, ref_dim, with_mask))
    sd = make_sd(levels, points, dtype=torch.float64)
    case = make_case(levels, nq, bs, ref_dim, dtype=torch.float64, with_mask=with_mask)
    with torch.no_grad():
        got = _restatement(sd, case, points)
    assert fingerprint_err(got, g, f"case{i}:") < 1e-10


def test_dropin_parameters_and_initialisers_match_reference():
    from bevformer_b200.plugin import CustomMSDeformableAttention
    g = golden("decoder_attention_ref")
    for i, kw in enumerate(INIT_KWARGS):
        a = CustomMSDeformableAttention(**kw)
        sa = a.state_dict()
        assert list(sa) == [str(k) for k in g[f"kw{i}:keys"]]
        for k in INIT_KEYS:
            assert torch.equal(sa[k], torch.from_numpy(g[f"kw{i}:init:{k}"])), k   # deterministic initialisers
        assert a.batch_first == bool(g[f"kw{i}:batch_first"])
    with pytest.raises(ValueError):
        CustomMSDeformableAttention(embed_dims=250, num_heads=8)


@pytest.mark.parametrize("levels,points,nq,bs,ref_dim,with_mask", CASES)
def test_dropin_module_logic_on_cpu(levels, points, nq, bs, ref_dim, with_mask, monkeypatch):
    """Everything around the kernels (layouts, stacked head projection, softmax, both reference-point
    forms, mask, residual) with the sampler replaced by the test oracle: equals the restatement."""
    from bevformer_b200 import ops
    from bevformer_b200.plugin import CustomMSDeformableAttention

    class _OracleSampler:
        @staticmethod
        def apply(value, ss, lsi, loc, attn, step):
            return torch_ref.msda_grid_sample(value, [tuple(x) for x in ss.tolist()], loc, attn)

    monkeypatch.setattr(ops, "MultiScaleDeformableAttnFunction_fp32", _OracleSampler)
    m = CustomMSDeformableAttention(num_levels=len(levels), num_points=points).eval()
    sd = make_sd(levels, points)
    m.load_state_dict(sd)
    case = make_case(levels, nq, bs, ref_dim, with_mask=with_mask)
    with torch.no_grad():
        got = m(**case)
        want = _restatement(sd, case, points)
    assert got.shape == case["query"].shape
    assert max_err(got, want) < 1e-5
    with pytest.raises(ValueError):
        m(case["query"], value=case["value"], reference_points=case["reference_points"][..., :1].repeat(1, 1, 1, 3),
          spatial_shapes=case["spatial_shapes"], level_start_index=case["level_start_index"])


def test_no_cpu_path_without_the_kernels():
    from bevformer_b200.plugin import CustomMSDeformableAttention
    m = CustomMSDeformableAttention(num_levels=1).eval()
    case = make_case([(6, 5)], 3, 1, 2)
    with pytest.raises(RuntimeError):
        m(**case)


# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-3), (torch.bfloat16, 3e-2)])
@pytest.mark.parametrize("levels,points,nq,bs,ref_dim,with_mask",
                         CASES + [([(50, 50)], 4, 900, 1, 2, False)])       # last: the tiny decoder shape
def test_dropin_on_gpu_vs_restatement(levels, points, nq, bs, ref_dim, with_mask, dtype, tol):
    from bevformer_b200 import _lib
    from bevformer_b200.plugin import CustomMSDeformableAttention
    sd = make_sd(levels, points)
    case = make_case(levels, nq, bs, ref_dim, with_mask=with_mask)
    with torch.no_grad():
        want = _restatement(sd, case, points)
    m = CustomMSDeformableAttention(num_levels=len(levels), num_points=points)
    m.load_state_dict(sd)
    m = m.to("cuda", dtype).eval()
    dev = {k: (v.cuda() if v is not None else None) for k, v in case.items()}
    # reference points stay fp32: a bf16 coordinate has 8 mantissa bits (0.2 px on a 50-px map), which
    # alone moves the result by 8e-2 on the 900-query case -- an input-precision effect, not a kernel one
    for k in ("query", "query_pos", "value"):
        dev[k] = dev[k].to(dtype)
    before = _lib.launch_count()
    with torch.no_grad():
        got = m(**dev)
    assert _lib.launch_count() > before
    assert got.dtype == dtype and got.shape == want.shape
    assert rel_err(got.float().cpu(), want) < tol


@pytest.mark.gpu
def test_dropin_backward_on_gpu():
    from bevformer_b200.plugin import CustomMSDeformableAttention
    levels, points = [(8, 14), (4, 7)], 4
    sd = make_sd(levels, points)
    case = make_case(levels, 9, 2, 2)
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    cq = case["query"].clone().requires_grad_(True)
    cv = case["value"].clone().requires_grad_(True)
    want = torch_ref.custom_ms_deformable_attention(
        sdr, "", cq.permute(1, 0, 2), cv.permute(1, 0, 2), case["reference_points"], case["spatial_shapes"],
        torch_ref._sampler(True), query_pos=case["query_pos"].permute(1, 0, 2), num_points=points).permute(1, 0, 2)
    proj = torch.randn(want.shape, generator=torch.Generator().manual_seed(1))
    (want * proj).sum().backward()
    m = CustomMSDeformableAttention(num_levels=len(levels), num_points=points)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    q = case["query"].cuda().requires_grad_(True)
    v = case["value"].cuda().requires_grad_(True)
    got = m(q, value=v, query_pos=case["query_pos"].cuda(), reference_points=case["reference_points"].cuda(),
            spatial_shapes=case["spatial_shapes"].cuda(), level_start_index=case["level_start_index"].cuda())
    (got * proj.cuda()).sum().backward()
    assert rel_err(q.grad.cpu(), cq.grad) < 2e-3
    assert rel_err(v.grad.cpu(), cv.grad) < 2e-3
    for k, p in m.named_parameters():
        assert rel_err(p.grad.cpu(), sdr[k].grad) < 5e-3, k


# ------------------------------------------------------------------------------------------------
# DetectionTransformerDecoder (decoder.py:52-129): the refinement loop around the cross-attention
# ------------------------------------------------------------------------------------------------
def _build_decoder():
    import copy
    from bevformer_b200 import synthetic as syn
    from bevformer_b200.plugin import build_transformer_layer_sequence
    dec = build_transformer_layer_sequence(copy.deepcopy(syn.DECODER_CFG))
    dec.load_state_dict(syn.make_random_state_dict(dec, 0))
    return dec


def test_decoder_builds_from_config_with_reference_keys():
    """Same parameter names as the reference decoder built from the same dict (golden 'keys' comes from the
    reference's own DetectionTransformerDecoder)."""
    from tests.util import golden
    dec = _build_decoder()
    assert sorted(dec.state_dict()) == [str(k) for k in golden("decoder_toy")["keys"]]
    assert len(dec.layers) == 3 and dec.return_intermediate


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_decoder_loop_against_reference_golden(dtype):
    from bevformer_b200 import synthetic as syn
    from tests.util import fixed_projection, golden, rel_err
    g = golden("decoder_toy")
    w = syn.WORKLOADS["toy"]
    dec = _build_decoder().to("cuda", dtype).eval()
    query, query_pos, bev, ref, reg = syn.make_decoder_inputs(w)
    reg = reg.to("cuda", dtype)
    q = query.to("cuda", dtype).requires_grad_(True)
    b = bev.to("cuda", dtype).requires_grad_(True)
    states, refs = dec(query=q, key=None, value=b, query_pos=query_pos.to("cuda", dtype),
                       reference_points=ref.to("cuda", dtype), reg_branches=reg, cls_branches=None,
                       spatial_shapes=torch.tensor([[w.bev_h, w.bev_w]], device="cuda"),
                       level_start_index=torch.tensor([0], device="cuda"))
    assert states.shape == g["states"].shape and refs.shape == g["refs"].shape
    tol = 1e-3 if dtype == torch.float32 else 6e-2
    assert rel_err(states.float().cpu(), g["states"]) < tol
    # bf16: the points themselves live in bf16 (2^-9 of [0, 1]) and pass three inverse-sigmoid updates
    assert rel_err(refs.float().cpu(), g["refs"]) < (1e-4 if dtype == torch.float32 else 5e-2)
    if dtype == torch.float32:
        (states * fixed_projection(states.shape).cuda()).sum().backward()
        assert rel_err(q.grad.cpu(), g["grad_query"]) < 2e-3
        assert rel_err(b.grad.cpu()[:16], g["grad_bev_rows"]) < 2e-3
