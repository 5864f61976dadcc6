"""TorchScript row of the boundary (SURVEY.md 8b): the reference scripts its whole model for deployment
(train.py:50-55, eval.py:38), so the drop-in PatchMatch must script, save and load; its kernels are reachable from
TorchScript as `torch.ops.pmb200.*` (csrc/torch_binding.cpp over the C ABI).  CPU tests: registration, schemas,
compile + save + load (no kernel runs without a GPU).  GPU tests: scripted == eager, bit for bit."""
import io

import pytest
import torch

from patchmatchnet_b200 import PatchMatch, _native
from tests import pm_cases

OPS = ["relative_projection", "pack_nhwc", "warp_corr", "aggregate_views", "warp_corr_view_weights", "warp_corr_score_",
       "aggregate_views_score_", "offset_corr", "offset_corr_weight", "init_propagate", "adaptive_eval",
       "adaptive_eval_planar", "photometric_confidence"]
DEV = "cuda:0"


@pytest.fixture(scope="module", autouse=True)
def _ops_loaded():
    _native.build_torch_library()
    _native.load_torch_ops()


def test_operators_are_registered_with_schemas():
    assert torch.ops.pmb200.abi_version() == 1
    for name in OPS:
        schema = str(getattr(torch.ops.pmb200, name).default._schema)
        assert schema.startswith(f"pmb200::{name}("), schema
    # the in-place score epilogues declare what they mutate
    assert "Tensor(a!) xs" in str(torch.ops.pmb200.warp_corr_score_.default._schema)
    assert "Tensor(a!) xs" in str(torch.ops.pmb200.aggregate_views_score_.default._schema)


def test_no_cpu_backend():
    """CUDA is the only registered backend: a CPU tensor reaches no kernel."""
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.pmb200.aggregate_views(torch.zeros(1, 1, 1, 1, 1, 1), torch.zeros(1, 1, 1, 1))
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.pmb200.pack_nhwc([torch.zeros(1, 8, 4, 4)])


def _scripted_stage(weights, stage):
    mod = PatchMatch(**pm_cases.stage_ctor_kwargs(stage))
    mod.load_state_dict(pm_cases.stage_state(weights, stage), strict=True)
    mod.eval()
    return mod, torch.jit.script(mod)


@pytest.mark.parametrize("stage", [1, 2, 3])
def test_patchmatch_scripts_saves_and_loads(golden_weights, stage):
    mod, sm = _scripted_stage(golden_weights, stage)
    graph = str(sm._forward_script.graph)
    for op in ("pmb200::pack_nhwc", "pmb200::relative_projection", "pmb200::offset_corr_weight", "pmb200::init_propagate",
               "pmb200::warp_corr_score_", "pmb200::adaptive_eval"):
        assert op in graph, op
    # the folded heads travel inside the archive and equal the eager path's
    buf = io.BytesIO()
    torch.jit.save(sm, buf)
    buf.seek(0)
    back = torch.jit.load(buf)
    for name, head in (("_head_fw", mod.feature_weight_net), ("_head_pw", mod.evaluation.pixel_wise_net),
                       ("_head_sim", mod.evaluation.similarity_net)):
        assert torch.equal(getattr(back, name), head.folded_tensor())
        assert float(getattr(back, name).abs().sum()) > 0
    assert set(back.state_dict()) == set(mod.state_dict())  # still exactly the reference's keys


def test_script_heads_follow_the_weights(golden_weights):
    mod = PatchMatch(**pm_cases.stage_ctor_kwargs(2)).eval()
    before = mod._head_sim.clone()
    mod.load_state_dict(pm_cases.stage_state(golden_weights, 2), strict=True)  # post-hook refolds in eval mode
    assert not torch.equal(before, mod._head_sim)
    assert torch.equal(mod._head_sim, mod.evaluation.similarity_net.folded_tensor())
    mod.train()
    with torch.no_grad():
        mod.evaluation.similarity_net.similarity.bias.add_(1.0)
    mod.eval()  # eval() refolds: this is the call the reference makes right before torch.jit.script (train.py:52)
    assert float(mod._head_sim[-1]) == pytest.approx(float(mod.evaluation.similarity_net.similarity.bias.detach()), abs=0)


def test_scripted_module_is_inference_only(golden_weights):
    mod = PatchMatch(**pm_cases.stage_ctor_kwargs(3))
    sm = torch.jit.script(mod.train())
    case = pm_cases.make_stage_inputs(pm_cases.STAGE_CASES["stage3_small"])
    kw = [case[k] for k in ("ref_feature", "src_features", "ref_proj", "src_projs", "depth_min", "depth_max", "depth", "view_weights")]
    with pytest.raises(Exception, match="inference-only"):
        sm(*kw)


def test_unmodified_reference_net_scripts_with_the_rebind(reference_net_calls, golden_weights, tmp_path):
    """What train.py:50-55 does with models.net.PatchMatch rebound -- eval(), torch.jit.script, save; then eval.py:38's
    torch.jit.load -- for each PatchMatch the reference network builds.  The network's scripted calls type-check against
    the scripted forward: its arguments and result must be those of the reference's own PatchMatch (schema recorded)."""
    rec = reference_net_calls
    want = rec["forward_schema"]
    for stage, kw in rec["ctor_kwargs"].items():
        mod = PatchMatch(**kw)
        mod.load_state_dict(pm_cases.stage_state(golden_weights, stage), strict=True)
        sm = torch.jit.script(mod.eval())
        schema = sm.forward.schema
        assert [(a.name, str(a.type)) for a in schema.arguments[1:]] == want["arguments"]
        assert [str(r.type) for r in schema.returns] == want["returns"]
        path = str(tmp_path / f"patchmatch_{stage}.pt")
        sm.save(path)
        back = torch.jit.load(path)
        assert "pmb200::warp_corr_score_" in str(back._forward_script.graph)
        assert {f"patchmatch_{stage}.{k}" for k in back.state_dict()} == {k for k in golden_weights if k.startswith(f"patchmatch_{stage}.")}
        if stage == 3:
            call = {k: (list(v) if isinstance(v, tuple) else v) for k, v in rec["calls"][0]["inputs"].items()}
            with torch.no_grad(), pytest.raises(Exception):  # the first pmb200 op has no CPU backend
                back(**call)


# ----------------------------------------------------------------------------------------------------------------
def _stage_kwargs(case):
    return [
        case["ref_feature"].to(DEV), [s.to(DEV) for s in case["src_features"]], case["ref_proj"].to(DEV),
        [m.to(DEV) for m in case["src_projs"]], case["depth_min"].to(DEV), case["depth_max"].to(DEV),
        case["depth"].to(DEV), case["view_weights"].to(DEV),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(pm_cases.STAGE_CASES))
def test_scripted_stage_equals_eager(golden_weights, name):
    spec = pm_cases.STAGE_CASES[name]
    case = pm_cases.make_stage_inputs(spec)
    mod, sm = _scripted_stage(golden_weights, spec["stage"])
    mod.to(DEV)
    sm.to(DEV)
    args = _stage_kwargs(case)
    with torch.no_grad():
        torch.manual_seed(11)
        torch.cuda.manual_seed(11)
        d0, p0, v0 = mod(*args)
        torch.manual_seed(11)
        torch.cuda.manual_seed(11)
        d1, p1, v1 = sm(*args)
    assert len(d0) == len(d1)
    for a, b in zip(d0, d1):
        assert torch.equal(a, b)
    assert torch.equal(p0, p1) and torch.equal(v0, v1)


@pytest.mark.gpu
def test_scripted_stage_survives_save_load_and_raises_torch_errors(golden_weights, tmp_path):
    spec = pm_cases.STAGE_CASES["stage2_small"] if "stage2_small" in pm_cases.STAGE_CASES else list(pm_cases.STAGE_CASES.values())[0]
    case = pm_cases.make_stage_inputs(spec)
    mod, sm = _scripted_stage(golden_weights, spec["stage"])
    path = str(tmp_path / "stage.pt")
    sm.save(path)
    back = torch.jit.load(path).to(DEV)
    mod.to(DEV)
    args = _stage_kwargs(case)
    with torch.no_grad():
        torch.manual_seed(5)
        torch.cuda.manual_seed(5)
        d0, p0, _ = mod(*args)
        torch.manual_seed(5)
        torch.cuda.manual_seed(5)
        d1, p1, _ = back(*args)
    assert torch.equal(d0[-1], d1[-1]) and torch.equal(p0, p1)
    # error convention of the op layer: exceptions, not status codes
    with pytest.raises(RuntimeError, match="inconsistent shapes"):
        torch.ops.pmb200.warp_corr(torch.zeros(1, 4, 4, 16, device=DEV), torch.zeros(2, 1, 4, 4, 8, device=DEV),
                                   torch.zeros(2, 1, 12, device=DEV), torch.ones(1, 2, 4, 4, device=DEV), None, 4)
    with pytest.raises(NotImplementedError):
        torch.ops.pmb200.offset_corr(torch.zeros(1, 4, 4, 16, device=DEV), torch.zeros(1, 20, 4, 4, device=DEV), 4, 10, 1)


@pytest.mark.gpu
def test_ops_equal_the_ctypes_wrappers():
    from patchmatchnet_b200 import ops

    g = torch.Generator().manual_seed(3)
    B, V, C, G, H, W, D = 2, 3, 32, 8, 24, 40, 8
    ref = torch.randn(B, H, W, C, generator=g).to(DEV)
    src = torch.randn(V, B, H, W, C, generator=g).to(DEV)
    rt = torch.tensor([1, 0, 0, 0, 1, 0, 0, 0, 1, 3.0, -2.0, 0.0]).repeat(V, B, 1).to(DEV)
    depth = (1 + torch.rand(B, D, H, W, generator=g)).to(DEV)
    vw = torch.rand(B, V, H, W, generator=g).to(DEV)
    assert torch.equal(torch.ops.pmb200.warp_corr(ref, src, rt, depth, None, G), ops.warp_corr(ref, src, rt, depth, G))
    assert torch.equal(torch.ops.pmb200.warp_corr(ref, src, rt, depth, vw, G), ops.warp_corr(ref, src, rt, depth, G, vw))
    sims = ops.warp_corr(ref, src, rt, depth, G)
    assert torch.equal(torch.ops.pmb200.aggregate_views(sims, vw), ops.aggregate_views(sims, vw))
    off = (0.5 * torch.randn(B, 18, H, W, generator=g)).to(DEV)
    assert torch.equal(torch.ops.pmb200.offset_corr(ref, off, G, 9, 2), ops.offset_corr(ref, off, G, 9, 2))
    maps = [torch.randn(B, C, H, W, generator=g).to(DEV) for _ in range(3)]
    assert torch.equal(torch.ops.pmb200.pack_nhwc(maps), ops.pack_nhwc(maps))
    prob = torch.softmax(torch.randn(B, D, H, W, generator=g), 1).to(DEV)
    assert torch.equal(torch.ops.pmb200.photometric_confidence(prob, 2 * H, 2 * W), ops.photometric_confidence(prob, 2 * H, 2 * W))
