"""Deterministic test problems shared by tests/golden/make_golden.py (which runs the unmodified
reference on them) and the parity tests (which run the oracle / the CUDA path on the same inputs)."""
from __future__ import annotations

import hashlib
from typing import Dict

import torch

from patchmatchnet_b200 import synthetic

NET_KWARGS = synthetic.DEFAULT_NET_KWARGS
FEATURES = {1: 16, 2: 32, 3: 64}
GROUPS = {1: 4, 2: 8, 3: 8}

# small per-stage problems: batch of 2, sizes that are NOT multiples of the warp tile
STAGE_CASES = {
    "stage3_small": dict(stage=3, B=2, V=3, H=13, W=21, seed=11, with_depth=False),
    "stage2_small": dict(stage=2, B=2, V=2, H=19, W=27, seed=12, with_depth=True),
    "stage1_small": dict(stage=1, B=2, V=4, H=22, W=35, seed=13, with_depth=True),
}
# BASELINE.json configs[0]: 1 ref + 2 src, 160x128 image -> stage-1 feature map 64x80, 8 hypotheses
CONFIG1 = dict(stage=1, B=1, V=2, H=64, W=80, seed=21, with_depth=True)
# full cascade, 1 ref + 2 src, 64x80 image
NET_CASE = dict(B=1, n_views=3, H=64, W=80, seed=31)


def stage_ctor_kwargs(stage: int) -> Dict:
    i = stage - 1
    k = NET_KWARGS
    return dict(
        propagation_out_range=k["propagation_range"][i],
        patchmatch_iteration=k["patchmatch_iteration"][i],
        patchmatch_num_sample=k["patchmatch_num_sample"][i],
        patchmatch_interval_scale=k["patchmatch_interval_scale"][i],
        num_feature=FEATURES[stage],
        G=GROUPS[stage],
        propagate_neighbors=k["propagate_neighbors"][i],
        evaluate_neighbors=k["evaluate_neighbors"][i],
        stage=stage,
    )


def stage_state(weights: Dict[str, torch.Tensor], stage: int) -> Dict[str, torch.Tensor]:
    pre = f"patchmatch_{stage}."
    return {k[len(pre):]: v for k, v in weights.items() if k.startswith(pre)}


def make_stage_inputs(spec: Dict) -> Dict:
    """CPU inputs of one standalone PatchMatch call (keyword names = the forward's)."""
    stage, B, V, H, W = spec["stage"], spec["B"], spec["V"], spec["H"], spec["W"]
    g = torch.Generator().manual_seed(spec["seed"])
    C = FEATURES[stage]
    scale = {3: 8, 2: 4, 1: 2}[stage]
    ref = torch.randn(B, C, H, W, generator=g) * 0.5
    srcs = [torch.randn(B, C, H, W, generator=g) * 0.5 for _ in range(V)]
    Kc, Ec = synthetic.make_cameras(B, V + 1, H * scale, W * scale)
    ref_proj, src_projs = synthetic.stage_projections(Kc, Ec, stage)
    dmin = torch.full((B,), synthetic.DEPTH_MIN) + torch.arange(B) * 5.0
    dmax = torch.full((B,), synthetic.DEPTH_MAX) - torch.arange(B) * 7.0
    if spec["with_depth"]:
        depth = 450.0 + 450.0 * torch.rand(B, 1, H, W, generator=g)
        vw = torch.rand(B, V, H, W, generator=g)
    else:
        depth = torch.empty(0)
        vw = torch.empty(0)
    rand48 = None
    if not spec["with_depth"]:
        # what the reference's internal torch.rand returns after torch.manual_seed(seed + 1000) on CPU
        state = torch.get_rng_state()
        torch.manual_seed(spec["seed"] + 1000)
        rand48 = torch.rand(size=(B, 48, H, W))
        torch.set_rng_state(state)
    return dict(
        ref_feature=ref, src_features=srcs, ref_proj=ref_proj.contiguous(), src_projs=[m.contiguous() for m in src_projs],
        depth_min=dmin, depth_max=dmax, depth=depth, view_weights=vw, rand48=rand48,
    )


def make_net_inputs(spec: Dict) -> Dict:
    inp = synthetic.make_inputs(spec["B"], spec["n_views"], spec["H"], spec["W"], seed=spec["seed"])
    state = torch.get_rng_state()
    torch.manual_seed(spec["seed"] + 1000)
    inp["rand48"] = torch.rand(size=(spec["B"], 48, spec["H"] // 8, spec["W"] // 8))
    torch.set_rng_state(state)
    return inp


def warp_inputs():
    """Inputs of the homography-warp / sampling-grid comparison: stage2_small's features and cameras, three depth
    hypotheses per pixel (plane 0 behind the camera), and random offsets for the 16 propagation / 9 evaluation neighbours."""
    case = make_stage_inputs(STAGE_CASES["stage2_small"])
    B, _, H, W = case["ref_feature"].shape
    g = torch.Generator().manual_seed(7)
    depth = 400.0 + 600.0 * torch.rand(B, 3, H, W, generator=g)
    depth[:, 0] = -50.0
    offsets = {count: torch.randn(B, 2 * count, H * W, generator=g) for count in (16, 9)}
    return case, depth, offsets


def checksum(case: Dict) -> str:
    h = hashlib.sha256()

    def feed(x):
        if isinstance(x, torch.Tensor):
            h.update(x.detach().cpu().contiguous().numpy().tobytes())
        elif isinstance(x, (list, tuple)):
            for y in x:
                feed(y)

    for k in sorted(case):
        feed(case[k])
    return h.hexdigest()


def rel_l1(a: torch.Tensor, b: torch.Tensor) -> float:
    """north_star's metric: sum|a-b| / sum|b|."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().sum() / b.abs().sum().clamp_min(1e-30))
