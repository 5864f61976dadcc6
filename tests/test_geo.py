"""Geometric-consistency filtering (SURVEY.md 8f row f4; reference eval.py:86-190, :220-256).

CPU: the oracle (oracle/geo_oracle.py) is pinned bit for bit against (a) cv2.remap for its restatement of the bilinear
sampler, (b) what the reference's own source text computed on a seeded scene (tests/golden/geo_source_case.npz), (c) the
committed reference-generated fixture.
GPU (-m gpu): the one-launch kernel, through the C ABI, against the oracle and the fixture.  The masks are thresholded
quantities: a pixel whose distance / relative depth difference lies within rounding of its threshold may legitimately flip
(the kernel's float64 dot products are fused multiply-adds, BLAS's are not), so the bound is a fraction of pixels:
<= 1e-4 of the pixels per mask, and the averaged depth must agree to 1e-6 relative wherever the masks agree."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import geo_oracle as go
from tests import geo_cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "geo_case.npz")
SOURCE_CASE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "geo_source_case.npz")


@pytest.fixture(scope="module")
def golden():
    z = np.load(GOLDEN)
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def source_case():
    z = np.load(SOURCE_CASE)
    return {k: z[k] for k in z.files}


def test_remap_restatement_is_bit_exact_against_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(1)
    img = rng.uniform(400, 900, size=(61, 83)).astype(np.float32)
    H, W = img.shape
    mx = rng.uniform(-5, W + 5, size=(H, W)).astype(np.float32)
    my = rng.uniform(-5, H + 5, size=(H, W)).astype(np.float32)
    mx[0, :8] = [np.nan, np.inf, -np.inf, 1e9, -1e9, 40000.3, -40000.7, 0.015625]
    my[0, :8] = [1, 2, 3, 4, 5, 6, 7, 0.984375]
    mx[1, :4] = [-1.0, -0.5, W - 1, W - 0.5]  # footprints straddling the border
    my[1, :4] = [0.25, H - 1, H - 0.5, -0.99]
    want = cv2.remap(img, mx, my, interpolation=cv2.INTER_LINEAR)
    assert np.array_equal(want, go.remap_linear(img, mx, my))


def test_oracle_is_bit_identical_to_the_reference_source(source_case):
    """eval.py:86-190, executed unmodified from the reference's source text (tests/golden/make_reference_golden.py)."""
    sc = geo_cases.make_scene(seed=3, H=72, W=100, n_src=3)
    assert np.array_equal(sc["ref_depth"], source_case["ref_depth"]), "seeded scene differs from the one the fixture was made with"
    for v, (d, k, e) in enumerate(zip(sc["src_depths"], sc["src_Ks"], sc["src_Es"])):
        rm, rd = source_case[f"view{v}.mask"], source_case[f"view{v}.depth"]
        om, od = go.check_geometric_consistency(sc["ref_depth"], sc["ref_K"], sc["ref_E"], d, k, e, 1.0, 0.01)
        assert np.array_equal(rm, om) and np.array_equal(rd, od)
        assert 0.05 < rm.mean() < 0.95, "the scene must exercise both outcomes"
        o3 = go.reproject_with_depth(sc["ref_depth"], sc["ref_K"], sc["ref_E"], d, k, e)
        r3 = [source_case[f"view{v}.reproject{i}"] for i in range(len(o3))]
        assert f"view{v}.reproject{len(o3)}" not in source_case
        assert all(np.array_equal(a, b) for a, b in zip(r3, o3))


def test_oracle_reproduces_the_reference_fixture(golden):
    sc = geo_cases.make_scene(seed=0)
    assert np.array_equal(sc["ref_depth"], golden["ref_depth"]) and np.array_equal(np.stack(sc["src_depths"]), golden["src_depths"])
    photo, msum, final, avg = go.fuse_reference_view(
        golden["ref_depth"], golden["ref_K"], golden["ref_E"], list(golden["src_depths"]), list(golden["src_Ks"]),
        list(golden["src_Es"]), golden["confidence"])
    assert np.array_equal(photo, golden["photo_mask"]) and np.array_equal(msum, golden["geo_mask_sum"])
    assert np.array_equal(final, golden["final_mask"]) and np.array_equal(avg, golden["depth_est_averaged"])
    assert avg.dtype == np.float64 and set(np.unique(msum)) == {0, 1, 2, 3, 4}


def test_camera_composition_matches_numpy_float32(golden):
    from patchmatchnet_b200 import ops

    cams = ops.compose_filter_cameras(golden["ref_K"], golden["ref_E"], list(golden["src_Ks"]), list(golden["src_Es"]))
    assert cams.shape == (4, 60) and cams.dtype == torch.float64
    t1 = np.matmul(golden["src_Es"][2], np.linalg.inv(golden["ref_E"]))
    assert np.array_equal(cams[2, 9:21].numpy().reshape(3, 4), t1[:3].astype(np.float64))
    assert np.array_equal(cams[2, :9].numpy().reshape(3, 3), np.linalg.inv(golden["ref_K"]).astype(np.float64))


def test_geometric_filter_rejects_bad_arguments_without_gpu():
    from patchmatchnet_b200 import _native, ops

    lib = _native.lib()
    assert lib.pmb200_geometric_filter(None, None, None, None, 1, 4, 4, 4, 4, 1.0, 0.01, 0.8, 3, None, None, None, None, None) == -1
    assert b"null pointer" in lib.pmb200_last_error()
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.geometric_filter(torch.zeros(4, 4), torch.zeros(4, 4), torch.zeros(1, 4, 4), torch.zeros(1, 60, dtype=torch.float64))


def _run_host(hostmath, sc):
    """The kernel's own per-pixel function (csrc/pm_geo_math.cuh) compiled for the host, pixel by pixel."""
    import ctypes

    from patchmatchnet_b200 import ops

    cams = ops.compose_filter_cameras(sc["ref_K"], sc["ref_E"], list(sc["src_Ks"]), list(sc["src_Es"])).numpy()
    ref = np.ascontiguousarray(sc["ref_depth"], dtype=np.float32)
    conf = np.ascontiguousarray(sc["confidence"], dtype=np.float32)
    src = np.ascontiguousarray(np.stack(list(sc["src_depths"])), dtype=np.float32)
    H, W = ref.shape
    V, Hs, Ws = src.shape
    msum = np.empty((H, W), np.int32)
    photo = np.empty((H, W), np.uint8)
    final = np.empty((H, W), np.uint8)
    avg = np.empty((H, W), np.float64)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    fn = hostmath.hm_geometric_filter
    fn.restype = None
    fn.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int] * 5 + [ctypes.c_double, ctypes.c_float, ctypes.c_float, ctypes.c_int] + [ctypes.c_void_p] * 4
    fn(ptr(ref), ptr(conf), ptr(src), ptr(cams), V, H, W, Hs, Ws, 1.0, 0.01, 0.8, 3, ptr(msum), ptr(photo), ptr(final), ptr(avg))
    return [photo.astype(bool), msum, final.astype(bool), avg]


def test_kernel_remap_function_is_bit_exact_against_cv2(hostmath):
    """pmgeo::remap_linear (the function the kernel inlines) against cv2.remap, including non-finite / huge coordinates."""
    import ctypes

    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(11)
    img = rng.uniform(400, 900, size=(37, 53)).astype(np.float32)
    H, W = img.shape
    mx = rng.uniform(-4, W + 4, size=(H, W)).astype(np.float32)
    my = rng.uniform(-4, H + 4, size=(H, W)).astype(np.float32)
    mx[0, :8] = [np.nan, np.inf, -np.inf, 1e9, -1e9, 40000.3, -40000.7, 0.015625]
    my[0, :8] = [1, 2, 3, 4, 5, 6, 7, 0.984375]
    mx[1, :4] = [-1.0, -0.5, W - 1, W - 0.5]
    my[1, :4] = [0.25, H - 1, H - 0.5, -0.99]
    want = cv2.remap(img, mx, my, interpolation=cv2.INTER_LINEAR)
    got = np.empty_like(want)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    fn = hostmath.hm_remap_linear
    fn.restype = None
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    fn(ptr(img), H, W, ptr(mx), ptr(my), H * W, ptr(got))
    assert np.array_equal(want, got)


def test_kernel_pixel_function_matches_the_reference_fixture(hostmath, golden):
    sc = dict(ref_depth=golden["ref_depth"], ref_K=golden["ref_K"], ref_E=golden["ref_E"], src_depths=golden["src_depths"],
              src_Ks=golden["src_Ks"], src_Es=golden["src_Es"], confidence=golden["confidence"])
    _compare(_run_host(hostmath, sc), (golden["photo_mask"], golden["geo_mask_sum"], golden["final_mask"], golden["depth_est_averaged"]))


@pytest.mark.parametrize("H,W,n_src,seed", [(72, 100, 3, 3), (33, 47, 1, 5)])
def test_kernel_pixel_function_matches_the_oracle(hostmath, H, W, n_src, seed):
    sc, want = _oracle_case(H, W, n_src, seed)
    got = _run_host(hostmath, sc)
    got[3][~np.isfinite(want[3])] = 1.0
    w3 = np.where(np.isfinite(want[3]), want[3], 1.0)
    _compare(got, (want[0], want[1], want[2], w3))


def _oracle_case(H, W, n_src, seed):
    sc = geo_cases.make_scene(seed=seed, H=H, W=W, n_src=n_src)
    if H * W < 8000:  # degenerate inputs: zero depth, NaN confidence
        sc["ref_depth"][0, :5] = 0.0
        sc["confidence"][1, :3] = np.nan
    with np.errstate(divide="ignore", invalid="ignore"):
        want = go.fuse_reference_view(sc["ref_depth"], sc["ref_K"], sc["ref_E"], sc["src_depths"], sc["src_Ks"], sc["src_Es"], sc["confidence"])
    return sc, want


def _run_gpu(sc):
    from patchmatchnet_b200 import ops

    dev = "cuda:0"
    cams = ops.compose_filter_cameras(sc["ref_K"], sc["ref_E"], list(sc["src_Ks"]), list(sc["src_Es"]))
    out = ops.geometric_filter(torch.from_numpy(sc["ref_depth"]).to(dev), torch.from_numpy(sc["confidence"]).to(dev),
                               torch.from_numpy(np.stack(list(sc["src_depths"]))).to(dev), cams)
    torch.cuda.synchronize()
    return [o.cpu().numpy() for o in out]


def _compare(got, want):
    photo, msum, final, avg = got
    wphoto, wsum, wfinal, wavg = want
    n = wsum.size
    assert np.array_equal(photo, wphoto)
    flipped = msum != wsum
    assert flipped.sum() <= max(1, int(1e-4 * n)), f"{flipped.sum()} of {n} pixels disagree on the geometric mask count"
    assert (final != wfinal).sum() <= max(1, int(1e-4 * n))
    same = ~flipped
    err = np.abs(avg[same] - wavg[same])
    assert avg.dtype == np.float64 and np.all(err <= 1e-6 * np.abs(wavg[same])), err.max()  # (0 vs 0 passes; NaN fails)


@pytest.mark.gpu
def test_gpu_filter_matches_the_reference_fixture(golden):
    sc = dict(ref_depth=golden["ref_depth"], ref_K=golden["ref_K"], ref_E=golden["ref_E"], src_depths=golden["src_depths"],
              src_Ks=golden["src_Ks"], src_Es=golden["src_Es"], confidence=golden["confidence"])
    _compare(_run_gpu(sc), (golden["photo_mask"], golden["geo_mask_sum"], golden["final_mask"], golden["depth_est_averaged"]))


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n_src,seed", [(72, 100, 3, 3), (33, 47, 1, 5), (512, 640, 4, 7)])
def test_gpu_filter_matches_the_oracle(H, W, n_src, seed):
    sc, want = _oracle_case(H, W, n_src, seed)
    got = _run_gpu(sc)
    # pixels with a zero / non-finite reference depth: masks must still agree, the averaged depth is not compared
    got[3][~np.isfinite(want[3])] = 1.0
    w3 = np.where(np.isfinite(want[3]), want[3], 1.0)
    _compare(got, (want[0], want[1], want[2], w3))


# ------------------------------------------------------------------------------------------------
# fusion half (reference eval.py:273-296): masked back-projection, colours, order-preserving compaction, PLY body
# ------------------------------------------------------------------------------------------------


def _fusion_case(H, W, n_src, seed):
    sc, (photo, msum, final, avg) = _oracle_case(H, W, n_src, seed)
    rng = np.random.default_rng(seed + 100)
    img = (rng.integers(0, 256, size=(H, W, 3)).astype(np.float32) / np.float32(255.0)).astype(np.float32)  # read_image: uint8 / 255
    if n_src < 3:  # fewer source views than geo_mask_thres: nothing would survive -- keep the photometric mask instead
        final = photo
    final = np.logical_and(final, np.isfinite(avg))
    return sc, final, np.where(np.isfinite(avg), avg, 0.0), img


def test_fusion_oracle_is_bit_identical_to_the_reference_source(source_case):
    """eval.py:273-281, the body of filter_depth's loop, executed from the reference's source text on this case."""
    sc, final, avg, img = _fusion_case(72, 100, 3, 3)
    assert np.array_equal(final, source_case["fusion.final_mask"])
    v, c = go.fuse_points(final, avg, img, sc["ref_K"], sc["ref_E"])
    assert 100 < len(v) < final.size and np.array_equal(source_case["fusion.vertices"], v) and np.array_equal(source_case["fusion.colors"], c)


def _check_body(body, want_v, want_c):
    """records against the oracle: colours exact; coordinates equal after the cast to float32 up to one float32 ulp on a
    small share of the values (the kernel's fused multiply-add chain vs BLAS's summation of the same four products)"""
    body = np.asarray(body, dtype=np.uint8).reshape(-1, 15)
    assert body.shape[0] == want_v.shape[0]
    got_v = body[:, :12].copy().view(np.float32).reshape(-1, 3)
    assert np.array_equal(body[:, 12:], want_c)
    if body.shape[0] == 0:
        return
    w32 = want_v.astype(np.float32)
    diff = got_v != w32
    assert diff.mean() <= 0.02, diff.mean()
    assert np.all(np.abs(got_v - w32) <= np.spacing(np.abs(w32)))


def test_kernel_fusion_function_matches_the_oracle(hostmath):
    for (H, W, n_src, seed) in ((72, 100, 3, 3), (33, 47, 1, 5)):
        sc, final, avg, img = _fusion_case(H, W, n_src, seed)
        want_v, want_c = go.fuse_points(final, avg, img, sc["ref_K"], sc["ref_E"])
        from patchmatchnet_b200 import ops

        cam = ops.compose_fusion_camera(sc["ref_K"], sc["ref_E"]).numpy()
        body = np.zeros((H * W, 15), dtype=np.uint8)
        mask8 = final.astype(np.uint8)
        P = ctypes.c_void_p
        hostmath.hm_fuse_points.argtypes = [P, P, P, P, ctypes.c_int, ctypes.c_int, P]
        n = hostmath.hm_fuse_points(mask8.ctypes.data, np.ascontiguousarray(avg).ctypes.data, img.ctypes.data, cam.ctypes.data, H, W, body.ctypes.data)
        assert n == int(final.sum())
        _check_body(body[:n], want_v, want_c)
        assert bytes(body[:n].tobytes())[12:15] == go.ply_vertex_body(want_v, want_c)[12:15]


def test_save_ply_layout(tmp_path):
    from patchmatchnet_b200 import data_io

    v = np.array([[1.5, -2.0, 3.25], [0.0, 1e-3, 7.0]])
    c = np.array([[255, 0, 7], [1, 2, 3]], dtype=np.uint8)
    body = torch.from_numpy(np.frombuffer(go.ply_vertex_body(v, c), dtype=np.uint8).reshape(-1, 15).copy())
    path = str(tmp_path / "fused.ply")
    data_io.save_ply(path, [body[:1], body[1:]])
    raw = open(path, "rb").read()
    head, _, rest = raw.partition(b"end_header\n")
    assert head.startswith(b"ply\nformat binary_little_endian 1.0\nelement vertex 2\nproperty float x\n") and b"property uchar blue\n" in head
    assert rest == go.ply_vertex_body(v, c) and len(rest) == 30


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n_src,seed", [(72, 100, 3, 3), (33, 47, 1, 5), (512, 640, 4, 7)])
def test_gpu_fusion_matches_the_oracle(H, W, n_src, seed):
    from patchmatchnet_b200 import ops

    dev = "cuda:0"
    sc, final, avg, img = _fusion_case(H, W, n_src, seed)
    want_v, want_c = go.fuse_points(final, avg, img, sc["ref_K"], sc["ref_E"])
    body = ops.fuse_points(torch.from_numpy(final).to(dev), torch.from_numpy(avg).to(dev), torch.from_numpy(img).to(dev),
                           ops.compose_fusion_camera(sc["ref_K"], sc["ref_E"]))
    assert body.shape == (int(final.sum()), 15)
    _check_body(body.cpu().numpy(), want_v, want_c)
    v32, c8 = ops.split_ply_body(body)
    assert v32.shape == (body.shape[0], 3) and c8.dtype == torch.uint8
    # nothing survives / everything survives
    none = ops.fuse_points(torch.zeros(H, W, dtype=torch.bool, device=dev), torch.from_numpy(avg).to(dev), torch.from_numpy(img).to(dev),
                           ops.compose_fusion_camera(sc["ref_K"], sc["ref_E"]))
    assert none.shape == (0, 15)
    every = ops.fuse_points(torch.ones(H, W, dtype=torch.bool, device=dev), torch.from_numpy(avg).to(dev), torch.from_numpy(img).to(dev),
                            ops.compose_fusion_camera(sc["ref_K"], sc["ref_E"]))
    wv, wc = go.fuse_points(np.ones((H, W), dtype=bool), avg, img, sc["ref_K"], sc["ref_E"])
    _check_body(every.cpu().numpy(), wv, wc)
