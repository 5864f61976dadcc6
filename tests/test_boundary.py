"""The drop-in boundary (SURVEY.md 8b): constructor / forward signatures, parameter names and shapes,
error conventions -- checked without a GPU -- and that our PatchMatch takes the constructor and forward calls the
reference's UNMODIFIED models/net.py makes and loads its checkpoint."""
import inspect

import pytest
import torch

from oracle import pm_oracle
from patchmatchnet_b200 import PatchMatch, PatchmatchNet, load_reference_state
from tests import pm_cases


def test_constructor_signature_matches_reference_defaults():
    sig = inspect.signature(PatchMatch.__init__)
    want = [("propagation_out_range", 2), ("patchmatch_iteration", 2), ("patchmatch_num_sample", 16),
            ("patchmatch_interval_scale", 0.025), ("num_feature", 64), ("G", 8), ("propagate_neighbors", 16),
            ("evaluate_neighbors", 9), ("stage", 3)]  # reference models/patchmatch.py:245-256
    got = [(n, p.default) for n, p in list(sig.parameters.items())[1:]]
    assert got == want
    fwd = list(inspect.signature(PatchMatch.forward).parameters)[1:]
    assert fwd == ["ref_feature", "src_features", "ref_proj", "src_projs", "depth_min", "depth_max", "depth", "view_weights"]
    net = list(inspect.signature(PatchmatchNet.__init__).parameters)[1:7]
    assert net == ["patchmatch_interval_scale", "propagation_range", "patchmatch_iteration", "patchmatch_num_sample",
                   "propagate_neighbors", "evaluate_neighbors"]  # reference models/net.py:128-136
    assert list(inspect.signature(PatchmatchNet.forward).parameters)[1:] == ["images", "intrinsics", "extrinsics", "depth_min", "depth_max"]


@pytest.mark.parametrize("stage", [1, 2, 3])
def test_state_dict_names_and_shapes_match_checkpoint(golden_weights, stage):
    mod = PatchMatch(**pm_cases.stage_ctor_kwargs(stage))
    want = pm_cases.stage_state(golden_weights, stage)
    got = mod.state_dict()
    assert set(got) == set(want)
    for k in want:
        assert tuple(got[k].shape) == tuple(want[k].shape), k
    mod.load_state_dict(want, strict=True)
    # same key set as the oracle restatement of the reference module
    assert set(got) == set(pm_oracle.PatchMatchOracle(**pm_cases.stage_ctor_kwargs(stage)).state_dict())


def test_offset_convs_are_zero_initialised():
    mod = PatchMatch()
    for conv in (mod.propa_conv, mod.eval_conv):  # reference patchmatch.py:297-298, 310-311
        assert float(conv.weight.abs().max()) == 0.0 and float(conv.bias.abs().max()) == 0.0
    assert PatchMatch(propagate_neighbors=0).propa_conv.out_channels == 1  # max(2*0, 1), patchmatch.py:290


def test_whole_network_loads_reference_checkpoint(golden_weights):
    net = PatchmatchNet(**pm_cases.NET_KWARGS)
    load_reference_state(net, {"module." + k: v for k, v in golden_weights.items()})  # DataParallel prefix, eval.py:33-35
    assert sum(p.numel() for p in net.parameters()) == 222632  # SURVEY.md 2.1 #14


def test_error_conventions_cpu():
    case = pm_cases.make_stage_inputs(pm_cases.STAGE_CASES["stage3_small"])
    kw = {k: case[k] for k in ("ref_feature", "src_features", "ref_proj", "src_projs", "depth_min", "depth_max", "depth", "view_weights")}
    mod = PatchMatch(**pm_cases.stage_ctor_kwargs(3)).eval()
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            mod(**kw)
        bad = dict(kw, src_projs=kw["src_projs"][:-1])
        with pytest.raises(AssertionError, match="Different number of images and projection matrices"):
            mod(**bad)
        bad = dict(kw, view_weights=torch.rand(2, 7, 13, 21))
        with pytest.raises(AssertionError, match="Different number of images and view weights"):
            mod(**bad)
        with pytest.raises(NotImplementedError):
            PatchMatch(propagate_neighbors=5)(**kw)
        with pytest.raises(NotImplementedError):
            PatchMatch(evaluate_neighbors=10)(**kw)


def _recorded_kwargs(call):
    return {k: (type(v)(t.clone() for t in v) if isinstance(v, (list, tuple)) else v.clone()) for k, v in call["inputs"].items()}


def test_drops_into_unmodified_reference_net(reference_net_calls, golden_weights):
    """models/net.py binds PatchMatch by name at import (net.py:6), so rebinding that one name swaps the hot path: the
    class must accept the constructor keywords the reference network passes for each stage, load that stage's checkpoint
    entries, and take the keyword call the network makes (all recorded from the unmodified reference)."""
    rec = reference_net_calls
    assert rec["forward_parameters"] == list(inspect.signature(PatchMatch.forward).parameters)[1:]
    assert rec["state_keys"] == sorted(golden_weights)
    mods = {}
    for stage, kw in rec["ctor_kwargs"].items():
        mods[stage] = PatchMatch(**kw)
        missing, unexpected = mods[stage].load_state_dict(pm_cases.stage_state(golden_weights, stage), strict=True)
        assert not missing and not unexpected
        assert set(mods[stage].state_dict()) == {k[len(f"patchmatch_{stage}."):] for k in rec["state_keys"] if k.startswith(f"patchmatch_{stage}.")}
    assert sorted(mods) == [1, 2, 3]
    first = rec["calls"][0]
    assert first["stage"] == 3
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        # the first PatchMatch call of the reference's forward, on the CPU tensors it passed
        mods[3].eval()(**_recorded_kwargs(first))


def test_zero_copy_view_detection_needs_one_storage():
    """Back-to-back addresses are not enough (the caching allocator can place separate tensors adjacently):
    the zero-copy re-view is only taken for views of ONE storage."""
    from patchmatchnet_b200 import ops
    from patchmatchnet_b200.net import _adjacent_views

    stacked = torch.arange(3 * 2 * 4 * 5 * 6, dtype=torch.float32).view(6, 4, 5, 6)
    views = [stacked[0:2], stacked[2:4], stacked[4:6]]
    assert _adjacent_views(views)
    assert not _adjacent_views([v.clone() for v in views])
    assert not _adjacent_views([views[0], views[2], views[1]])
    net = PatchmatchNet(**pm_cases.NET_KWARGS, patchmatch_cls=pm_oracle.PatchMatchOracle).eval()
    imgs = torch.rand(3, 1, 3, 16, 24)
    with torch.no_grad():
        a = net.extract_features([imgs[0], imgs[1], imgs[2]])           # views of one buffer
        b = net.extract_features([imgs[i].clone() for i in range(3)])   # separate tensors -> torch.cat
    for fa, fb in zip(a, b):
        for k in fa:
            assert torch.equal(fa[k], fb[k])
    cl = stacked.contiguous(memory_format=torch.channels_last)
    assert ops._is_packed_nhwc([cl[0:2], cl[2:4], cl[4:6]])
    assert not ops._is_packed_nhwc([cl[0:2].clone(memory_format=torch.channels_last), cl[2:4], cl[4:6]])
    assert not ops._is_packed_nhwc(views)


def test_composed_feature_heads_equal_the_layerwise_top_down():
    """FeatureNet's eval fast path composes the linear top-down ops (reference net.py:52-66); the composed weights
    must reproduce the layer-by-layer outputs (pure tensor algebra, checked here in fp64 on the CPU)."""
    import torch
    import torch.nn.functional as F

    from patchmatchnet_b200.net import FeatureNet

    torch.manual_seed(0)
    net = FeatureNet().double().eval()
    x = torch.randn(2, 3, 32, 48, dtype=torch.float64)
    with torch.no_grad():
        want = net(x)
        half = net._trunk(net._trunk(x, 0, 1), 2, 4)
        quarter = net._trunk(half, 5, 7)
        eighth = net._trunk(quarter, 8, 10)
        h = {k: v.double() for k, v in net.composed_heads().items()}
        up = lambda t: F.interpolate(t, scale_factor=2.0, mode="bilinear", align_corners=False)
        out2 = up(F.conv2d(eighth, h["u_o"])) + F.conv2d(quarter, h["l2_o"], h["c2_o"])
        t = up(F.conv2d(eighth, h["u_t"])) + F.conv2d(quarter, h["l2_t"], h["c2_t"])
        out1 = up(t) + F.conv2d(half, h["l1"], h["c1"])
    # composed weights are rounded to fp32 once: agreement to fp32 resolution of the output scale
    for got, ref in ((out2, want[2]), (out1, want[1])):
        assert got.shape == ref.shape
        assert float((got - ref).abs().max() / ref.abs().max()) < 5e-6
