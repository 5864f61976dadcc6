"""Whole PatchMatch stages on the CPU box: the package's REAL host code (ops wrappers + PatchMatch._forward_eager, the
orchestration that otherwise only ever runs on the GPU) driving the CPU-emulated kernels through tests/emu_backend.py,
against the oracle and the reference-generated golden outputs -- the CPU twin of the GPU stage tests.  Tolerance as there:
depth rel-L1 <= 1e-4 (north_star allows 1e-3)."""
import pytest
import torch

from oracle import pm_oracle
from patchmatchnet_b200 import PatchMatch, ops
from tests import emu_backend, pm_cases
from tests.test_emulated_conv import emu_conv  # noqa: F401  (fixtures)
from tests.test_emulated_kernels import emu  # noqa: F401

NAMES = ("ref_feature", "src_features", "ref_proj", "src_projs", "depth_min", "depth_max", "depth", "view_weights")


def _aligned_like(t):
    """contiguous copy whose storage is 32-byte aligned (the feature packs are read with 256-bit loads)"""
    buf = torch.empty(t.numel() + 8, dtype=t.dtype)
    shift = (-buf.data_ptr() // t.element_size()) % 8
    out = buf[shift:shift + t.numel()].view(t.shape)
    out.copy_(t)
    return out


@pytest.fixture()
def backend(monkeypatch, emu, emu_conv):  # noqa: F811
    real_pack = ops.pack_nhwc
    facade = emu_backend.install(monkeypatch, emu, emu_conv)
    # torch's CPU allocator gives 64-byte alignment, but be explicit about the contract of the gather loads
    monkeypatch.setattr(ops, "pack_nhwc", lambda maps: _aligned_like(real_pack(maps)))
    return facade


@pytest.mark.parametrize("name", list(pm_cases.STAGE_CASES))
@pytest.mark.parametrize("fused", [True, False])
def test_native_stage_on_emulated_kernels_matches_oracle(backend, golden_weights, name, fused):
    spec = pm_cases.STAGE_CASES[name]
    stage = spec["stage"]
    case = pm_cases.make_stage_inputs(spec)
    state = pm_cases.stage_state(golden_weights, stage)
    mine = PatchMatch(**pm_cases.stage_ctor_kwargs(stage))
    mine.load_state_dict(state, strict=True)
    mine = mine.eval()
    mine.fuse_heads = fused
    orc = pm_oracle.PatchMatchOracle(**pm_cases.stage_ctor_kwargs(stage))
    orc.load_state_dict(state, strict=True)
    orc.eval()
    kw = {k: case[k] for k in NAMES}
    u = torch.rand(kw["ref_feature"].shape[0], 48, *kw["ref_feature"].shape[2:], generator=torch.Generator().manual_seed(3))
    mine.rand_source = lambda size, device: u  # one shared draw for the random initialisation
    orc.rand_source = lambda size, device: u
    with torch.no_grad():
        want = orc(**kw)
        got = mine(**kw)
    assert len(got[0]) == len(want[0])
    for a, b in zip(got[0], want[0]):
        assert a.shape == b.shape and pm_cases.rel_l1(a, b) <= 1e-4
    assert float((got[2] - want[2]).abs().max()) <= 1e-4  # view weights
    # probabilities: a hypothesis that sits on a bilinear cell boundary moves a little probability mass at single pixels
    # (the GPU stage tests bound the maximum by 2e-3 against the golden outputs; the emulated build differs from the GPU
    # in the last bits -- exact division instead of the fast reciprocal -- so bound the mean tightly and the maximum loosely)
    dp = (got[1] - want[1]).abs()
    assert float((got[1].sum(1) - 1.0).abs().max()) <= 1e-5 and float(dp.mean()) <= 2e-5 and float(dp.max()) <= 5e-3


def test_native_network_on_emulated_kernels_matches_oracle(backend, golden_weights, monkeypatch):
    """The whole cascade -- FeatureNet (native channels-last convs with folded BatchNorm, composed top-down heads, fused
    upsample-add), three PatchMatch stages, Refinement, photometric confidence -- through the package's inference fast path
    (the code that otherwise needs the GPU), every hand-written kernel emulated, against the oracle network on the CPU."""
    from patchmatchnet_b200 import net as native_net, synthetic
    from patchmatchnet_b200.net import PatchmatchNet, load_reference_state

    monkeypatch.setattr(native_net, "_fast", lambda x: True)
    monkeypatch.setattr(native_net, "_FUSED_CONV_RELU", False)  # the FLOP-bound layers stay library convs: plain conv2d + relu here
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)  # native convs in the fp32-accurate 3xTF32 mode
    kw = dict(synthetic.DEFAULT_NET_KWARGS)
    mine = PatchmatchNet(**kw)
    load_reference_state(mine, golden_weights)
    mine = mine.eval()
    orc = PatchmatchNet(**kw, patchmatch_cls=pm_oracle.PatchMatchOracle)
    load_reference_state(orc, golden_weights)
    orc = orc.eval()
    inp = synthetic.make_inputs(1, 3, 48, 64, seed=5)
    u = torch.rand(1, 48, 6, 8, generator=torch.Generator().manual_seed(9))
    for net in (mine, orc):
        net.patchmatch_3.rand_source = lambda size, device: u
    args = lambda: (list(inp["images"]), inp["intrinsics"].clone(), inp["extrinsics"], inp["depth_min"], inp["depth_max"])
    with torch.no_grad():
        monkeypatch.setattr(native_net, "_fast", lambda x: False)  # the oracle network: plain torch ops
        want_depth, want_conf, _ = orc(*args())
        monkeypatch.setattr(native_net, "_fast", lambda x: True)
        got_depth, got_conf, stages = mine(*args())
    assert got_depth.shape == want_depth.shape and pm_cases.rel_l1(got_depth, want_depth) <= 2e-4
    assert float(((got_conf - want_conf).abs() > 1e-3).float().mean()) <= 0.01  # the regressed index truncates to an integer
    assert sorted(stages) == [0, 1, 2, 3]
    n = backend.calls
    # the launches of one fused inference forward (DESIGN.md "Launches per forward"): 3 projections, 3 K-A'+head, 5 K-C,
    # 1 K-A view weights, 1 aggregate+head, 4 K-A+head, 5 K-B, the native convs, the confidence tail
    assert n.get("pmb200_relative_projection") == 3 and n.get("pmb200_offset_corr_weight") == 3 and n.get("pmb200_init_propagate") == 5
    assert n.get("pmb200_warp_corr_view_weights") == 1 and n.get("pmb200_aggregate_views_score") == 1
    assert n.get("pmb200_warp_corr_score") == 4 and n.get("pmb200_adaptive_eval") == 5 and n.get("pmb200_photometric_confidence") == 1
    assert n.get("pmb200_conv2d_nhwc", 0) >= 10, n
    # FeatureNet's conv0 -> conv1 (K-S) and Refinement (K-R) each ran as their fused exact-fp32 launches
    assert n.get("pmb200_conv_stem") == 1 and n.get("pmb200_refine_low") == 1 and n.get("pmb200_refine_full") == 1, n


def test_drop_in_executes_inside_the_unmodified_reference_net(backend, golden_weights, reference_net_calls, monkeypatch):
    """The drop-in, EXECUTED: each of the three PatchMatch modules the reference's own `models/net.py` builds, constructed
    by this package's class from the keywords the network passes, loaded with the shipped checkpoint's entries for its
    stage with every key matched, and run -- real host code, every hand-written kernel under the emulator -- on the exact
    inputs the unmodified network handed to its stage on pm_cases.NET_CASE; each stage's depths, probabilities and view
    weights are compared with what the reference's PatchMatch returned there (tests/golden/net_calls.pt).  (VERDICT r1,
    missing #6.)"""
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)  # native offset convs in the fp32-accurate mode
    rec = reference_net_calls
    inp = pm_cases.make_net_inputs(pm_cases.NET_CASE)
    assert pm_cases.checksum(inp) == rec["checksum"]
    assert [c["stage"] for c in rec["calls"]] == [3, 2, 1]
    for call in rec["calls"]:
        stage = call["stage"]
        mod = PatchMatch(**rec["ctor_kwargs"][stage])
        missing, unexpected = mod.load_state_dict(pm_cases.stage_state(golden_weights, stage), strict=True)
        assert not missing and not unexpected
        mod.eval()
        if stage == 3:
            mod.rand_source = lambda size, device: inp["rand48"]  # the draw the reference made for the fixture
        kw = {k: (type(v)(t.clone() for t in v) if isinstance(v, (list, tuple)) else v.clone()) for k, v in call["inputs"].items()}
        with torch.no_grad():
            depths, score, vw = mod(**kw)
        assert len(depths) == len(call["depths"])
        for x, y in zip(depths, call["depths"]):
            assert x.shape == y.shape and pm_cases.rel_l1(x, y) <= 2e-4
        assert score.shape == call["score"].shape and float((score - call["score"]).abs().mean()) <= 1e-3
        assert vw.shape == call["view_weights"].shape and float((vw - call["view_weights"]).abs().mean()) <= 1e-3
    n = backend.calls  # the native path ran (not a torch re-implementation): 5 fused warp+correlation launches, 5 K-B, 5 K-C
    assert n.get("pmb200_warp_corr_score") == 4 and n.get("pmb200_warp_corr_view_weights") == 1
    assert n.get("pmb200_adaptive_eval") == 5 and n.get("pmb200_init_propagate") == 5 and n.get("pmb200_conv2d_nhwc", 0) >= 5


# ------------------------------------------------------------------------------------------------
# training configuration: native forward + native backward kernels behind patchmatchnet_b200.autograd, on the CPU box
# ------------------------------------------------------------------------------------------------


def _close(got, want, tol):
    got, want = got.detach().double(), want.detach().double()
    scale = max(1e-12, float(want.abs().max()))
    err = float((got - want).abs().max())
    assert got.shape == want.shape and err <= tol * scale, f"max err {err:.3e} vs scale {scale:.3e}"


def _compare_param_grads(mine, want, rtol, atol_of_global):
    assert set(mine) == set(want)
    glob = max(float(w.abs().max()) for w in want.values() if w is not None)
    bad = []
    for k, w in want.items():
        if w is None:  # parameters the reference graph never reaches (SURVEY.md 3.4)
            assert mine[k] is None or float(mine[k].abs().max()) == 0.0, k
            continue
        assert mine[k] is not None, k
        err = float((mine[k].double() - w.double()).abs().max())
        if err > rtol * float(w.abs().max()) + atol_of_global * glob:
            bad.append((k, err, float(w.abs().max())))
    assert not bad, f"global grad scale {glob:.3e}; offenders: {bad[:8]}"


@pytest.mark.parametrize("name", list(pm_cases.STAGE_CASES))
def test_native_stage_training_gradients_on_emulated_kernels(backend, golden_weights, name):
    """train() mode, loss = sum of smooth-L1 of every iteration's depth (reference net.py:336-342): parameter and
    input-feature gradients of the native path (autograd bridges over the emulated backward kernels) against torch autograd
    on the oracle -- the CPU twin of tests/test_gpu_backward.py::test_stage_training_gradients_match_oracle."""
    import torch.nn.functional as F

    spec = pm_cases.STAGE_CASES[name]
    case = pm_cases.make_stage_inputs(spec)
    state = pm_cases.stage_state(golden_weights, spec["stage"])
    target = 500.0 + 300.0 * torch.rand(case["ref_feature"].shape[0], 1, *case["ref_feature"].shape[2:], generator=torch.Generator().manual_seed(9))

    def run(mod):
        mod.load_state_dict(state, strict=True)
        mod = mod.train()
        if case["rand48"] is not None:
            mod.rand_source = lambda size, device: case["rand48"]
        ref = case["ref_feature"].detach().clone().requires_grad_(True)
        srcs = [s.detach().clone().requires_grad_(True) for s in case["src_features"]]
        depths, score, vw = mod(ref_feature=ref, src_features=srcs, ref_proj=case["ref_proj"], src_projs=list(case["src_projs"]),
                                depth_min=case["depth_min"], depth_max=case["depth_max"], depth=case["depth"], view_weights=case["view_weights"])
        loss = sum(F.smooth_l1_loss(d, target, reduction="mean") for d in depths)
        loss.backward()
        grads = {k: (p.grad.detach() if p.grad is not None else None) for k, p in mod.named_parameters()}
        return loss.item(), [d.detach() for d in depths], ref.grad, [s.grad for s in srcs], grads

    lo, do, gro, gso, po = run(pm_oracle.PatchMatchOracle(**pm_cases.stage_ctor_kwargs(spec["stage"])))
    lm, dm, grm, gsm, pmine = run(PatchMatch(**pm_cases.stage_ctor_kwargs(spec["stage"])))
    for a, b in zip(dm, do):
        assert pm_cases.rel_l1(a, b) <= 1e-4
    assert abs(lm - lo) <= 1e-4 * abs(lo)
    _close(grm, gro, 2e-3)
    for a, b in zip(gsm, gso):
        _close(a, b, 2e-3)
    _compare_param_grads(pmine, po, rtol=5e-3, atol_of_global=1e-4)
    assert backend.calls.get("pmb200_warp_corr_backward", 0) >= 1 and backend.calls.get("pmb200_adaptive_eval_backward", 0) >= 1


def test_native_network_training_step_on_emulated_kernels(backend, golden_weights):
    """BASELINE.json configs[4] in miniature on the CPU box: full cascade in train() mode, reference loss (net.py:321-342),
    backward; every parameter gradient of the native path against torch autograd on the oracle behind the same shell."""
    from patchmatchnet_b200 import PatchmatchNet, load_reference_state, patchmatchnet_loss, synthetic

    spec = dict(B=1, n_views=3, H=48, W=64, seed=41)
    inp = synthetic.make_inputs(spec["B"], spec["n_views"], spec["H"], spec["W"], seed=spec["seed"])
    g = torch.Generator().manual_seed(5)
    rand48 = torch.rand(spec["B"], 48, spec["H"] // 8, spec["W"] // 8, generator=g)
    gts, masks = [], []
    for lvl in range(4):
        h, w = spec["H"] >> lvl, spec["W"] >> lvl
        gts.append(500.0 + 350.0 * torch.rand(spec["B"], 1, h, w, generator=g))
        masks.append(torch.rand(spec["B"], 1, h, w, generator=g) > 0.2)

    def run(cls):
        net = PatchmatchNet(**pm_cases.NET_KWARGS) if cls is None else PatchmatchNet(**pm_cases.NET_KWARGS, patchmatch_cls=cls)
        load_reference_state(net, golden_weights)
        net = net.train()
        net.patchmatch_3.rand_source = lambda size, device: rand48
        depth, conf, per_stage = net(list(inp["images"]), inp["intrinsics"].clone(), inp["extrinsics"], inp["depth_min"], inp["depth_max"])
        assert conf.numel() == 0  # train mode returns an empty confidence (net.py:286-287)
        loss = patchmatchnet_loss(per_stage, gts, masks)
        loss.backward()
        return loss.item(), {k: (p.grad.detach() if p.grad is not None else None) for k, p in net.named_parameters()}

    lo, go = run(pm_oracle.PatchMatchOracle)
    lm, gm = run(None)
    assert abs(lm - lo) <= 2e-4 * abs(lo)
    never = sorted(k for k, v in go.items() if v is None)
    assert any("patchmatch_1.propa_conv" in k for k in never) and any("patchmatch_2.evaluation.pixel_wise_net" in k for k in never)
    _compare_param_grads(gm, go, rtol=2e-2, atol_of_global=2e-3)
