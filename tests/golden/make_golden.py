"""Generates the golden vectors under tests/golden/ from the REFERENCE'S OWN unmodified modules
(Oracle-R, oracle/mmcv_stub.py).  Run in the dev container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference ships no tests and no golden vectors for this path (SURVEY.md §4), so these files are
what pins parity.  Inputs are never stored: every consumer regenerates them from the same seeded
generators (bevformer_b200/synthetic.py), which are deterministic on CPU.  Stored per case: a fixed
subset of rows of each result plus whole-tensor statistics, small enough to commit.
"""
from __future__ import annotations

import os
import sys
import time
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from bevformer_b200 import synthetic as syn  # noqa: E402
from oracle import mmcv_stub  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
warnings.filterwarnings("ignore")


def stats(t: torch.Tensor) -> np.ndarray:
    t = t.detach().double()
    return np.array([t.sum().item(), t.abs().sum().item(), t.square().sum().item(),
                     t.abs().max().item()], dtype=np.float64)


def row_subset(n: int, k: int, seed: int = 7) -> np.ndarray:
    g = np.random.default_rng(seed)
    return np.sort(g.choice(n, size=min(k, n), replace=False)).astype(np.int64)


def fixed_projection(shape, seed=11, dtype=torch.float32) -> torch.Tensor:
    """The test loss is (out * R).sum() with this fixed R (a LayerNorm-terminated encoder has ~zero
    gradient under out.square().mean(), SURVEY.md §8c)."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g).to(dtype)


# ------------------------------------------------------------------------------------------------
def op_case(name, bs, levels, nq, heads, dim, pts, seed, dtype=torch.float64, loc_range=(-0.1, 1.1),
            value_scale=1.0, keep_rows=256):
    ref = mmcv_stub.load_reference_modules()
    v, ss, lsi, loc, attn = syn.make_msda_inputs(bs, levels, nq, heads, dim, pts, seed=seed,
                                                 dtype=dtype, loc_range=loc_range,
                                                 value_scale=value_scale)
    v.requires_grad_(True); loc.requires_grad_(True); attn.requires_grad_(True)
    out = ref.msda_pytorch(v, ss, loc, attn)
    gout = fixed_projection(out.shape, dtype=dtype)
    (out * gout).sum().backward()
    rq = row_subset(nq, keep_rows)
    rs = row_subset(v.shape[1], keep_rows, seed=8)
    np.savez_compressed(
        os.path.join(OUT, f"msda_{name}.npz"),
        meta=np.array([bs, nq, heads, dim, pts, seed], dtype=np.int64),
        levels=np.array(levels, dtype=np.int64), loc_range=np.array(loc_range),
        value_scale=np.array(value_scale),
        rows_q=rq, rows_s=rs,
        out_rows=out.detach()[:, rq].float().numpy(), out_stats=stats(out),
        grad_value_rows=v.grad[:, rs].float().numpy(), grad_value_stats=stats(v.grad),
        grad_loc_rows=loc.grad[:, rq].float().numpy(), grad_loc_stats=stats(loc.grad),
        grad_attn_rows=attn.grad[:, rq].float().numpy(), grad_attn_stats=stats(attn.grad))
    print(f"msda_{name}: out {tuple(out.shape)} |max| {out.abs().max():.4f}")


def encoder_case(name, workload, bs=1, with_prev=True, seed=0, keep_rows=512, backward=True,
                 full_output=False):
    w = syn.WORKLOADS[workload]
    cfg = (mmcv_stub.load_reference_encoder_cfg(w.config_file) if w.config_file
           else syn.encoder_cfg(w))
    enc = mmcv_stub.build_reference_encoder(encoder_cfg=cfg).eval()   # eval(): dropout = identity
    enc.load_state_dict(syn.make_state_dict(w, seed=seed))
    inp = syn.make_encoder_inputs(w, bs=bs, seed=seed, with_prev=with_prev)
    if bs > 1:   # make the batch items differ
        g = torch.Generator().manual_seed(99)
        inp.feat = inp.feat + 0.5 * torch.randn(inp.feat.shape, generator=g)
        inp.bev_query = inp.bev_query + 0.1 * torch.randn(inp.bev_query.shape, generator=g)
    t0 = time.time()
    save = {}
    if backward:
        inp.bev_query.requires_grad_(True)
        inp.feat.requires_grad_(True)
        inp.bev_pos.requires_grad_(True)      # the learned positional encoding trains (every layer's TSA adds it)
    with torch.set_grad_enabled(backward):
        out = enc(inp.bev_query, inp.feat, inp.feat, **inp.kwargs())
    rq = row_subset(w.num_query, keep_rows)
    save.update(out_rows=out.detach()[:, rq].numpy(), out_stats=stats(out), rows_q=rq)
    if full_output:
        save["out_full"] = out.detach().numpy()
    if backward:
        proj = fixed_projection(out.shape)
        (out * proj).sum().backward()
        rs = row_subset(w.num_value, keep_rows, seed=8)
        save.update(rows_s=rs,
                    grad_query_rows=inp.bev_query.grad[rq].numpy(),
                    grad_query_stats=stats(inp.bev_query.grad),
                    grad_feat_rows=inp.feat.grad[:, rs].numpy(),
                    grad_feat_stats=stats(inp.feat.grad),
                    grad_pos_rows=inp.bev_pos.grad[rq].numpy(),
                    grad_pos_stats=stats(inp.bev_pos.grad))
        for k, p in enc.named_parameters():
            save["gstat:" + k] = stats(p.grad)
            if p.grad.numel() <= 1024:
                save["gfull:" + k] = p.grad.numpy()
            elif p.dim() == 2:
                save["grows:" + k] = p.grad[: min(4, p.shape[0])].numpy()
    np.savez_compressed(os.path.join(OUT, f"encoder_{name}.npz"),
                        meta=np.array([bs, int(with_prev), seed], dtype=np.int64), **save)
    print(f"encoder_{name}: out {tuple(out.shape)} in {time.time() - t0:.1f}s")


def grid_length_of(w):
    """BEV cell size that keeps the 102.4 m range at this BEV resolution."""
    return (0.512 * 200 / w.bev_h, 0.512 * 200 / w.bev_w)


def perception_case(name, workload, bs=2, with_prev=True, seed=0, keep_rows=512):
    """PerceptionTransformer.get_bev_features of the reference's own class (fp32, eval mode)."""
    w = syn.WORKLOADS[workload]
    PT = mmcv_stub.load_reference_transformer()
    cfg = (mmcv_stub.load_reference_encoder_cfg(w.config_file) if w.config_file
           else syn.encoder_cfg(w))
    m = PT(num_feature_levels=len(w.levels), num_cams=w.num_cams, encoder=cfg, decoder=None,
           embed_dims=w.embed_dims, rotate_center=[w.bev_h // 2, w.bev_w // 2]).eval()
    m.load_state_dict(syn.make_perception_state_dict(w, seed=seed))
    inp = syn.make_perception_inputs(w, bs=bs, seed=seed, with_prev=with_prev)
    for f in inp.mlvl_feats:
        f.requires_grad_(True)
    inp.bev_queries.requires_grad_(True)
    t0 = time.time()
    prev = None if inp.prev_bev is None else inp.prev_bev.clone()      # the reference rotates in place
    out = m.get_bev_features(inp.mlvl_feats, inp.bev_queries, w.bev_h, w.bev_w,
                             grid_length=grid_length_of(w), bev_pos=inp.bev_pos, prev_bev=prev,
                             img_metas=inp.img_metas)
    (out * fixed_projection(out.shape)).sum().backward()
    rq = row_subset(w.num_query, keep_rows)
    save = dict(out_rows=out.detach()[:, rq].numpy(), out_stats=stats(out), rows_q=rq,
                grad_queries_rows=inp.bev_queries.grad[rq].numpy(),
                grad_queries_stats=stats(inp.bev_queries.grad))
    for i, f in enumerate(inp.mlvl_feats):
        save[f"grad_feat{i}_stats"] = stats(f.grad)
        save[f"grad_feat{i}_slice"] = f.grad[:, :, :8, :2].numpy()
    for k, p in m.named_parameters():
        if k.startswith("encoder.") or p.grad is None:
            continue
        save["gstat:" + k] = stats(p.grad)
        save["gfull:" + k] = p.grad.numpy()
    np.savez_compressed(os.path.join(OUT, f"perception_{name}.npz"),
                        meta=np.array([bs, int(with_prev), seed], dtype=np.int64), **save)
    print(f"perception_{name}: out {tuple(out.shape)} in {time.time() - t0:.1f}s")


def sequence_inputs(w, frames=4, seed=0):
    """A short video for the temporal tests: per-frame pyramids, ABSOLUTE can_bus (ego position / heading
    accumulate), two scenes (the scene changes at the last frame)."""
    g = torch.Generator().manual_seed(9000 + seed)
    feats = [torch.randn(1, frames, w.num_cams, w.embed_dims, h, ww, generator=g) for h, ww in w.levels]
    bev_queries = torch.randn(w.num_query, w.embed_dims, generator=g)
    bev_pos = torch.rand(1, w.embed_dims, w.bev_h, w.bev_w, generator=g)
    metas = []
    pos, ang = np.array([10.0, -4.0, 0.0]), 30.0
    for i in range(frames):
        m = syn.make_img_metas(w, 1)[0]
        cb = np.array(syn.make_can_bus(i), dtype=np.float64)
        pos = pos + np.array([0.9 + 0.2 * i, -0.3 + 0.1 * i, 0.0])
        ang = ang + 4.0 - 1.5 * i
        cb[:3], cb[-1] = pos, ang
        m["can_bus"] = cb
        m["scene_token"] = "scene-a" if i < frames - 1 else "scene-b"
        m["prev_bev_exists"] = i > 0
        metas.append(m)
    return feats, bev_queries, bev_pos, metas


def temporal_case(name, workload, frames=4, seed=0):
    """Golden for the temporal plumbing, produced by the REFERENCE's PerceptionTransformer driven exactly as
    detectors/bevformer.py does: (a) obtain_history_bev (:158-177) over the first frames-1 frames with
    can_bus already expressed as deltas (what the dataset pipeline provides in training,
    datasets/nuscenes_dataset.py:86-103); (b) forward_test's prev_frame_info update (:236-269) over all
    frames with absolute can_bus."""
    w = syn.WORKLOADS[workload]
    PT = mmcv_stub.load_reference_transformer()
    cfg = (mmcv_stub.load_reference_encoder_cfg(w.config_file) if w.config_file else syn.encoder_cfg(w))
    m = PT(num_feature_levels=len(w.levels), num_cams=w.num_cams, encoder=cfg, decoder=None,
           embed_dims=w.embed_dims, rotate_center=[w.bev_h // 2, w.bev_w // 2]).eval()
    m.load_state_dict(syn.make_perception_state_dict(w, seed=seed))
    feats, bev_queries, bev_pos, metas = sequence_inputs(w, frames, seed)
    gl = list(grid_length_of(w))
    import copy
    with torch.no_grad():
        # (a) training-time history: deltas precomputed, first frame has no history
        tm = copy.deepcopy(metas[: frames - 1])
        for i in range(len(tm) - 1, 0, -1):
            tm[i]["can_bus"][:3] -= tm[i - 1]["can_bus"][:3]
            tm[i]["can_bus"][-1] -= tm[i - 1]["can_bus"][-1]
        tm[0]["can_bus"][:3] = 0
        tm[0]["can_bus"][-1] = 0
        prev = None
        for i in range(frames - 1):
            if not tm[i]["prev_bev_exists"]:
                prev = None
            prev = m.get_bev_features([f[:, i] for f in feats], bev_queries, w.bev_h, w.bev_w, grid_length=gl,
                                      bev_pos=bev_pos, prev_bev=prev, img_metas=[tm[i]])
        history = prev
        # (b) test-time stream, absolute can_bus, the reference's in-place delta logic
        info = {"prev_bev": None, "scene_token": None, "prev_pos": 0, "prev_angle": 0}
        stream = []
        sm = copy.deepcopy(metas)
        for i in range(frames):
            if sm[i]["scene_token"] != info["scene_token"]:
                info["prev_bev"] = None
            info["scene_token"] = sm[i]["scene_token"]
            tmp_pos = copy.deepcopy(sm[i]["can_bus"][:3])
            tmp_angle = copy.deepcopy(sm[i]["can_bus"][-1])
            if info["prev_bev"] is not None:
                sm[i]["can_bus"][:3] -= info["prev_pos"]
                sm[i]["can_bus"][-1] -= info["prev_angle"]
            else:
                sm[i]["can_bus"][-1] = 0
                sm[i]["can_bus"][:3] = 0
            bev = m.get_bev_features([f[:, i] for f in feats], bev_queries, w.bev_h, w.bev_w, grid_length=gl,
                                     bev_pos=bev_pos, prev_bev=info["prev_bev"], img_metas=[sm[i]])
            info["prev_pos"], info["prev_angle"], info["prev_bev"] = tmp_pos, tmp_angle, bev
            stream.append(bev)
    np.savez_compressed(os.path.join(OUT, f"temporal_{name}.npz"), meta=np.array([frames, seed], dtype=np.int64),
                        history=history.numpy(), history_stats=stats(history),
                        **{f"stream{i}": b.numpy() for i, b in enumerate(stream)})
    print(f"temporal_{name}: {frames} frames, history {tuple(history.shape)}")


def decoder_case(name, workload, seed=0):
    """The reference's own DetectionTransformerDecoder (decoder.py:52-129) + CustomMSDeformableAttention,
    built from the decoder dict the configs use (3 layers here), eval mode, with regression branches."""
    import copy
    w = syn.WORKLOADS[workload]
    D = mmcv_stub.load_reference_decoder()
    cfg = copy.deepcopy(syn.DECODER_CFG)
    cfg.pop("type")
    dec = D(**cfg).eval()
    dec.load_state_dict(syn.make_random_state_dict(dec, seed))
    query, query_pos, bev, ref, reg = syn.make_decoder_inputs(w, seed=seed)
    query.requires_grad_(True); bev.requires_grad_(True)
    states, refs = dec(query=query, key=None, value=bev, query_pos=query_pos, reference_points=ref,
                       reg_branches=reg, cls_branches=None,
                       spatial_shapes=torch.tensor([[w.bev_h, w.bev_w]]), level_start_index=torch.tensor([0]))
    (states * fixed_projection(states.shape)).sum().backward()
    np.savez_compressed(os.path.join(OUT, f"decoder_{name}.npz"), states=states.detach().numpy(),
                        refs=refs.detach().numpy(), grad_query=query.grad.numpy(),
                        grad_bev_stats=stats(bev.grad), grad_bev_rows=bev.grad[:16].numpy(),
                        keys=np.array(sorted(dec.state_dict())))
    print(f"decoder_{name}: states {tuple(states.shape)} refs {tuple(refs.shape)}")


V2_KW = dict(frames=(-1, 0), num_fusion=2)


def v2_inputs(w, seed=0, num_query=40):
    inp = syn.make_perception_inputs(w, bs=1, seed=seed, with_prev=True)
    g = torch.Generator().manual_seed(15000 + seed)
    oq = torch.randn(num_query, 2 * w.embed_dims, generator=g)
    reg = torch.nn.ModuleList([torch.nn.Linear(w.embed_dims, 10) for _ in range(syn.DECODER_CFG["num_layers"])])
    with torch.no_grad():
        for lin in reg:
            lin.weight.copy_(0.05 * torch.randn(lin.weight.shape, generator=g))
            lin.bias.copy_(0.05 * torch.randn(lin.bias.shape, generator=g))
    return inp, oq, reg


def v2_case(name, workload, seed=0):
    """The reference's own PerceptionTransformerV2.forward (transformerV2.py:243-353): BEV encoder, two-frame
    ResNetFusion, decoder with box refinement; eval mode (BatchNorm running statistics)."""
    import copy
    w = syn.WORKLOADS[workload]
    mmcv_stub.load_reference_decoder()
    V2 = mmcv_stub.load_reference_transformer_v2().module.PerceptionTransformerV2
    m = V2(num_feature_levels=len(w.levels), num_cams=w.num_cams, encoder=syn.encoder_cfg(w),
           decoder=copy.deepcopy(syn.DECODER_CFG), embed_dims=w.embed_dims,
           rotate_center=[w.bev_h // 2, w.bev_w // 2], **V2_KW).eval()
    m.load_state_dict(syn.make_random_state_dict(m, seed))
    inp, oq, reg = v2_inputs(w, seed)
    with torch.no_grad():
        bev, states, ref0, refs = m(inp.mlvl_feats, inp.bev_queries, oq, w.bev_h, w.bev_w,
                                    grid_length=list(grid_length_of(w)), bev_pos=inp.bev_pos, reg_branches=reg,
                                    cls_branches=None, prev_bev=[inp.prev_bev.clone(), None],
                                    img_metas=inp.img_metas)
    np.savez_compressed(os.path.join(OUT, f"v2_{name}.npz"), bev=bev.numpy(), states=states.numpy(),
                        ref0=ref0.numpy(), refs=refs.numpy(), keys=np.array(sorted(m.state_dict())))
    print(f"v2_{name}: bev {tuple(bev.shape)} states {tuple(states.shape)}")


# ------------------------------------------------------------------------------------------------
# fp64 results and module layouts of the reference's own classes, for the CPU tests that compare the
# restatement / the drop-in with them (inputs come from the tests' own seeded builders)
# ------------------------------------------------------------------------------------------------
def _prefixed(prefix, d):
    return {prefix + k: v for k, v in d.items()}


def _layout(sd):
    """A state_dict's keys, in order, with their shapes (read back with tests.util.layout)."""
    return np.array(repr({k: tuple(v.shape) for k, v in sd.items()}))


def encoder_fp64_case():
    """The reference encoder in fp64: the toy cases of tests/test_oracle.py and the quirk scenarios of
    tests/test_quirks.py."""
    from tests.test_oracle import _enc_inputs
    from tests.test_quirks import scenario
    from tests.util import fingerprint
    w = syn.WORKLOADS["toy"]
    runs = {f"bs{bs}_{'prev' if p else 'noprev'}": _enc_inputs("toy", bs, p, dtype=torch.float64)[1]
            for bs, p in ((1, True), (2, True), (1, False))}
    runs.update({k: scenario(k, torch.float64) for k in ("q1", "q10")})
    save = {}
    for name, inp in runs.items():
        enc = mmcv_stub.build_reference_encoder(encoder_cfg=syn.encoder_cfg(w)).eval().double()
        enc.load_state_dict(syn.make_state_dict(w, dtype=torch.float64))
        with torch.no_grad():
            save.update(_prefixed(name + ":", fingerprint(enc(inp.bev_query, inp.feat, inp.feat, **inp.kwargs()))))
    np.savez_compressed(os.path.join(OUT, "encoder_fp64_toy.npz"), **save)
    print(f"encoder_fp64_toy: {sorted(runs)}")


def perception_fp64_case():
    """PerceptionTransformer.get_bev_features of the reference's own class in fp64 (tests/test_oracle.py)."""
    from tests.util import fingerprint
    w = syn.WORKLOADS["toy"]
    PT = mmcv_stub.load_reference_transformer()
    save = {}
    for bs, with_prev in ((2, True), (1, False)):
        m = PT(num_feature_levels=len(w.levels), num_cams=w.num_cams, encoder=syn.encoder_cfg(w), decoder=None,
               embed_dims=w.embed_dims, rotate_center=[w.bev_h // 2, w.bev_w // 2])
        m.load_state_dict(syn.make_perception_state_dict(w))
        m = m.double().eval()
        inp = syn.make_perception_inputs(w, bs=bs, with_prev=with_prev, dtype=torch.float64)
        prev = None if inp.prev_bev is None else inp.prev_bev.clone()
        with torch.no_grad():
            ref = m.get_bev_features(inp.mlvl_feats, inp.bev_queries, w.bev_h, w.bev_w,
                                     grid_length=grid_length_of(w), bev_pos=inp.bev_pos, prev_bev=prev,
                                     img_metas=inp.img_metas)
        save.update(_prefixed(f"bs{bs}_{'prev' if with_prev else 'noprev'}:", fingerprint(ref)))
    np.savez_compressed(os.path.join(OUT, "perception_fp64_toy.npz"), **save)
    print("perception_fp64_toy")


def v2_encoder_fp64_case():
    """PerceptionTransformerBEVEncoder (transformerV2.py) of the reference in fp64, with and without the BEV
    augmentation resampling (tests/test_transformer_v2.py)."""
    from tests.test_transformer_v2 import W, _metas, _sd
    from tests.util import fingerprint
    cls = mmcv_stub.load_reference_transformer_v2()
    save = {}
    for aug in (None, "only_gt", "images_too"):
        for bs in (1, 2):
            if aug == "only_gt" and bs > 1:      # the reference's resampling branch builds a batch-1 grid
                continue
            m = cls(num_feature_levels=len(W.levels), num_cams=W.num_cams, encoder=syn.encoder_cfg(W),
                    embed_dims=W.embed_dims).double().eval()
            m.load_state_dict(_sd(torch.float64))
            inp = syn.make_perception_inputs(W, bs=bs, dtype=torch.float64)
            with torch.no_grad():
                want = m(inp.mlvl_feats, inp.bev_queries, W.bev_h, W.bev_w, bev_pos=inp.bev_pos,
                         prev_bev=inp.prev_bev, img_metas=_metas(bs, aug))
            save.update(_prefixed(f"{aug}_bs{bs}:", fingerprint(want)))
    np.savez_compressed(os.path.join(OUT, "v2_encoder_fp64_toy.npz"), **save)
    print("v2_encoder_fp64_toy")


def decoder_attention_case():
    """CustomMSDeformableAttention of the reference: fp64 outputs on the cases of
    tests/test_decoder_attention.py, and its state_dict / deterministic initialisers per constructor call."""
    from tests.test_decoder_attention import CASES, INIT_KEYS, INIT_KWARGS, make_case, make_sd
    from tests.util import fingerprint
    ref_cls = mmcv_stub.load_reference_decoder_attention()
    save = {}
    for i, (levels, points, nq, bs, ref_dim, with_mask) in enumerate(CASES):
        m = ref_cls(num_levels=len(levels), num_points=points).double().eval()
        m.load_state_dict(make_sd(levels, points, dtype=torch.float64))
        case = make_case(levels, nq, bs, ref_dim, dtype=torch.float64, with_mask=with_mask)
        with torch.no_grad():
            save.update(_prefixed(f"case{i}:", fingerprint(m(**case))))
    for i, kw in enumerate(INIT_KWARGS):
        b = ref_cls(**kw)
        sb = b.state_dict()
        save[f"kw{i}:keys"] = np.array(list(sb))
        save.update({f"kw{i}:init:{k}": sb[k].numpy() for k in INIT_KEYS})
        save[f"kw{i}:batch_first"] = np.array(b.batch_first)
    np.savez_compressed(os.path.join(OUT, "decoder_attention_ref.npz"), **save)
    print("decoder_attention_ref")


def encoder_layout_case(name):
    """The encoder an unchanged reference config describes: the encoder dict the config evaluates to, and
    the state_dict layout, deterministic initialisers and parameter count of the reference encoder built
    from it."""
    w = syn.WORKLOADS[name]
    cfg = mmcv_stub.load_reference_encoder_cfg(w.config_file)
    enc = mmcv_stub.build_reference_encoder(w.config_file)
    sd = enc.state_dict()
    init = [v.reshape(-1) for k, v in sd.items() if "sampling_offsets" in k or "attention_weights" in k or "norms" in k]
    save = dict(layout=_layout(sd), init=torch.cat(init).numpy(), cfg=np.array(repr(cfg)),
                nparams=np.array(sum(p.numel() for p in enc.parameters())))
    np.savez_compressed(os.path.join(OUT, f"encoder_layout_{name}.npz"), **save)
    print(f"encoder_layout_{name}: {len(sd)} tensors")


def perception_layout_case():
    """State_dict layouts of the reference's PerceptionTransformer (decoder=None) and
    PerceptionTransformerBEVEncoder on the toy workload, and the PerceptionTransformer's public attributes
    and submodules (what a get_bev_features installed on that class reads)."""
    from tests.test_transformer_v2 import V2_EXTRA_KWARGS
    w = syn.WORKLOADS["toy"]
    kw = dict(num_feature_levels=len(w.levels), num_cams=w.num_cams, encoder=syn.encoder_cfg(w), embed_dims=w.embed_dims)
    ref = mmcv_stub.load_reference_transformer()(decoder=None, **kw)
    save = {"pt:layout": _layout(ref.state_dict()),
            "pt:attrs": np.array(repr({k: v for k, v in vars(ref).items() if not k.startswith("_")})),
            "pt:modules": np.array(list(ref._modules))}
    for i, extra in enumerate(V2_EXTRA_KWARGS):
        save[f"v2_{i}:layout"] = _layout(mmcv_stub.load_reference_transformer_v2()(**kw, **extra).state_dict())
    np.savez_compressed(os.path.join(OUT, "perception_layout_toy.npz"), **save)
    print("perception_layout_toy")


def main(which):
    if not mmcv_stub.reference_available():
        raise SystemExit("needs /root/reference (dev container only)")
    torch.manual_seed(0)
    cases = {
        # mmcv's upstream known-answer geometry (SURVEY.md §4): N=1, M=2, D=2, Lq=2, L=2, P=2
        "kat": lambda: op_case("kat", 1, [(6, 4), (3, 2)], 2, 2, 2, 2, seed=3, value_scale=0.01,
                               loc_range=(0.0, 1.0)),
        # same geometry with out-of-range locations and an odd head_dim (generic kernel)
        "kat_oob": lambda: op_case("kat_oob", 2, [(6, 4), (3, 2)], 5, 2, 30, 3, seed=4,
                                   loc_range=(-0.4, 1.4)),
        # BASELINE.json configs[0]: 1 cam, 1 level, 64x64 BEV, 4 points
        "config0": lambda: op_case("config0", 1, [(64, 64)], 4096, 8, 32, 4, seed=0),
        # a 4-level pyramid with SCA's point count
        "pyramid": lambda: op_case("pyramid", 2, [(29, 50), (15, 25), (8, 13), (4, 7)], 700, 8, 32,
                                   8, seed=5, loc_range=(-0.2, 1.2)),
        "enc_toy": lambda: encoder_case("toy", "toy", full_output=True),
        "enc_toy_bs2": lambda: encoder_case("toy_bs2", "toy", bs=2, full_output=True),
        "enc_toy_noprev": lambda: encoder_case("toy_noprev", "toy", with_prev=False,
                                               full_output=True),
        "enc_tiny": lambda: encoder_case("tiny", "tiny", keep_rows=256),
        "enc_tiny_noprev": lambda: encoder_case("tiny_noprev", "tiny", with_prev=False,
                                                backward=False),
        "enc_small": lambda: encoder_case("small", "small", keep_rows=256),
        "enc_small4": lambda: encoder_case("small4", "small4", keep_rows=256),
        "enc_base": lambda: encoder_case("base", "base", keep_rows=256),
        # PerceptionTransformer.get_bev_features: CAN-bus shift / MLP, prev_bev rotation, level + camera
        # embeddings, then the encoder
        "per_toy": lambda: perception_case("toy", "toy", bs=2),
        "per_toy_noprev": lambda: perception_case("toy_noprev", "toy", bs=1, with_prev=False),
        "per_tiny": lambda: perception_case("tiny", "tiny", bs=1, keep_rows=256),
        # temporal plumbing (SURVEY.md §8 f3): history recurrence + streaming prev_frame_info, 4 frames, 2 scenes
        "temporal_toy": lambda: temporal_case("toy", "toy"),
        # decoder loop (SURVEY.md §8 f2): 3 layers, 40 object queries into the 12x10 BEV map, box refinement
        "decoder_toy": lambda: decoder_case("toy", "toy"),
        # BEVFormerV2 transformer (SURVEY.md §8 f4): encoder + 2-frame ResNetFusion + decoder
        "v2_toy": lambda: v2_case("toy", "toy"),
        "encoder_fp64": encoder_fp64_case,
        "perception_fp64": perception_fp64_case,
        "v2_encoder_fp64": v2_encoder_fp64_case,
        "decoder_attention": decoder_attention_case,
        "layout_tiny": lambda: encoder_layout_case("tiny"),
        "layout_small": lambda: encoder_layout_case("small"),
        "layout_base": lambda: encoder_layout_case("base"),
        "layout_perception": perception_layout_case,
    }
    for k in (which or cases):
        cases[k]()


if __name__ == "__main__":
    main(sys.argv[1:])
