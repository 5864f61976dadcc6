"""Pin the oracle bit for bit against what the UNMODIFIED reference computed on the same inputs: its stage and network
outputs (tests/golden/stage_cases.pt, net_case.pt, written by tests/golden/make_golden.py) and its warp and
sampling-grid helpers (tests/golden/warp_case.pt, written by tests/golden/make_reference_golden.py).  The reference
draws its random hypotheses from the global CPU generator; the oracle is seeded the same way."""
import os

import pytest
import torch

from oracle import pm_oracle
from patchmatchnet_b200.net import PatchmatchNet, load_reference_state
from tests import pm_cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _oracle_stage(weights, stage):
    mod = pm_oracle.PatchMatchOracle(**pm_cases.stage_ctor_kwargs(stage))
    missing, unexpected = mod.load_state_dict(pm_cases.stage_state(weights, stage), strict=True)
    assert not missing and not unexpected
    return mod.eval()


@pytest.mark.parametrize("name", list(pm_cases.STAGE_CASES))
def test_stage_bit_identical(golden_weights, golden_stage_cases, name):
    spec = pm_cases.STAGE_CASES[name]
    case = pm_cases.make_stage_inputs(spec)
    a = golden_stage_cases[name]
    assert pm_cases.checksum(case) == a["checksum"], "seeded inputs differ from the ones the fixture was made with"
    kw = {k: case[k] for k in ("ref_feature", "src_features", "ref_proj", "src_projs", "depth_min", "depth_max", "depth", "view_weights")}
    mod = _oracle_stage(golden_weights, spec["stage"])
    with torch.no_grad():
        torch.manual_seed(spec["seed"] + 1000)  # what the fixture's reference run drew from
        b = mod(**kw)
    assert len(a["depths"]) == len(b[0])
    for x, y in zip(a["depths"], b[0]):
        assert torch.equal(x, y)
    assert torch.equal(a["score"], b[1]) and torch.equal(a["view_weights"], b[2])


def test_warp_and_helpers_bit_identical():
    want = torch.load(os.path.join(GOLDEN, "warp_case.pt"), map_location="cpu")
    case, depth, offsets = pm_cases.warp_inputs()
    B, C, H, W = case["ref_feature"].shape
    b = pm_oracle.homography_warp(case["src_features"][0], case["src_projs"][0], case["ref_proj"], depth)
    assert torch.equal(want["warped"], b)
    assert float(b[:, :, 0].abs().max()) == 0.0  # behind the camera -> exactly zero
    # neighbour tables + grid
    for kind, count in (("propagation", 16), ("evaluation", 9)):
        g_or = pm_oracle.sampling_grid(pm_oracle.neighbour_table(kind, count, want["dilation"]), offsets[count], H, W)
        assert torch.equal(want["grids"][kind], g_or)


def test_full_network_bit_identical(golden_weights, golden_net_case):
    mine = PatchmatchNet(**pm_cases.NET_KWARGS, patchmatch_cls=pm_oracle.PatchMatchOracle)
    load_reference_state(mine, golden_weights)
    mine.eval()
    mine.stack_views = False  # the reference runs FeatureNet view by view
    inp = pm_cases.make_net_inputs(pm_cases.NET_CASE)
    assert pm_cases.checksum(inp) == golden_net_case["checksum"]
    seed = pm_cases.NET_CASE["seed"] + 1000
    with torch.no_grad():
        torch.manual_seed(seed)
        b = mine([i.clone() for i in inp["images"]], inp["intrinsics"].clone(), inp["extrinsics"].clone(), inp["depth_min"], inp["depth_max"])
    assert torch.equal(golden_net_case["depth"], b[0]) and torch.equal(golden_net_case["confidence"], b[1])
    assert sorted(golden_net_case["per_stage"]) == sorted(b[2])
    for s, ds in golden_net_case["per_stage"].items():
        assert len(ds) == len(b[2][s])
        for x, y in zip(ds, b[2][s]):
            assert torch.equal(x, y)
