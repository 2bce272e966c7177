"""Shared helpers of the test-suite: golden-file access and comparison metrics."""
import ast
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def stats(t: torch.Tensor) -> np.ndarray:
    t = t.detach().double().cpu()
    return np.array([t.sum().item(), t.abs().sum().item(), t.square().sum().item(),
                     t.abs().max().item()])


def fixed_projection(shape, seed=11, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g).to(dtype)


def max_err(a, b) -> float:
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return (a - b).abs().max().item() if a.numel() else 0.0


def rel_err(a, b) -> float:
    """max |a-b| / max(1, max|b|): the form in which the 1e-3 (fp32) / 1e-2 (bf16) bars are read."""
    b_ = torch.as_tensor(b).detach().double().cpu()
    scale = max(1.0, b_.abs().max().item()) if b_.numel() else 1.0
    return max_err(a, b) / scale


def layout(g, key="layout") -> dict:
    """{state_dict key: shape}, in the state_dict's order, as tests/golden/make_golden.py stores it."""
    return ast.literal_eval(g[key].item())


def reference_initialisers(g) -> dict:
    """{key: tensor} of the deterministic initialisers (sampling offsets, attention weights, norms) stored
    flat, in state_dict order, in an encoder_layout_<name> golden file."""
    shapes = layout(g)
    keys = [k for k in shapes if "sampling_offsets" in k or "attention_weights" in k or "norms" in k]
    parts = torch.from_numpy(g["init"]).split([int(np.prod(shapes[k])) for k in keys])
    return {k: p.reshape(shapes[k]) for k, p in zip(keys, parts)}


def fingerprint(t: torch.Tensor, n: int = 128, seed: int = 7) -> dict:
    """What a golden file keeps of a result too large to store whole: a fixed seeded sample of its
    elements, its sums over the last axis and whole-tensor statistics."""
    t = t.detach().double().cpu()
    flat = t.reshape(-1)
    idx = np.sort(np.random.default_rng(seed).choice(flat.numel(), size=min(n, flat.numel()), replace=False))
    return {"shape": np.array(t.shape, dtype=np.int32), "idx": idx.astype(np.int32),
            "vals": flat[torch.from_numpy(idx)].numpy(), "sums": t.sum(-1).numpy(), "stats": stats(t)}


def fingerprint_err(t, g, prefix: str = "") -> float:
    """Largest deviation of `t` from the fingerprint stored under `prefix` in golden file `g`: sampled
    elements, max |t|, and the last-axis sums divided by that axis' length; inf if the shape differs."""
    t = torch.as_tensor(t).detach().double().cpu()
    if tuple(t.shape) != tuple(int(x) for x in g[prefix + "shape"]):
        return float("inf")
    e_vals = max_err(t.reshape(-1)[torch.from_numpy(g[prefix + "idx"]).long()], g[prefix + "vals"])
    e_sums = max_err(t.sum(-1), g[prefix + "sums"]) / max(1, t.shape[-1])
    e_max = abs(t.abs().max().item() - float(g[prefix + "stats"][3]))
    return max(e_vals, e_sums, e_max)


def stats_close(got: np.ndarray, want: np.ndarray, rtol: float) -> bool:
    """sum |x|, sum x^2 and max |x| of the whole tensor agree (sum x itself cancels too much)."""
    return bool(np.all(np.abs(got[1:] - want[1:]) <= rtol * np.maximum(np.abs(want[1:]), 1e-12)))


def msda_case_inputs(g, dtype=torch.float32, device="cpu"):
    from bevformer_b200 import synthetic as syn
    bs, nq, heads, dim, pts, seed = [int(x) for x in g["meta"]]
    levels = [tuple(int(v) for v in row) for row in g["levels"]]
    return syn.make_msda_inputs(bs, levels, nq, heads, dim, pts, seed=seed, dtype=dtype,
                                device=device, loc_range=tuple(float(x) for x in g["loc_range"]),
                                value_scale=float(g["value_scale"]))
