"""Depth-map files (SURVEY.md 8f row f5; reference datasets/data_io.py:128-322): PFM and COLMAP .bin.

Integer / byte work: the bar is bit-exact -- identical bytes on disk, identical arrays in memory.
  oracle (oracle/mapio_oracle.py)  vs what the unmodified reference functions wrote and read
                                   (tests/golden/maps/reference_cases.npz) and the reference-written fixture files tests/golden/maps/*;
  native (libpmb200.so through patchmatchnet_b200.data_io, the mirror of the reference's API)  vs the oracle, the
                                   fixtures and the reference; error texts as the reference raises them;
  -m gpu: file -> pinned buffer -> device and back."""
import builtins
import os
import re

import numpy as np
import pytest
import torch

from oracle import mapio_oracle as mo
from patchmatchnet_b200 import data_io as dio

MAPS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "maps")
NAMES = ("depth_hw", "conf_hw1", "color_hw3")


def _same(a, b):
    """bit-identical float arrays (NaN payloads and signed zeros included)"""
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.fixture(scope="module")
def expected():
    z = np.load(os.path.join(MAPS, "expected.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def ref_io():
    """What the unmodified reference's save_map / save_pfm wrote and read_map / read_pfm returned for `_cases()`,
    `SCALES` and `BAD_PFM` (tests/golden/make_reference_golden.py)."""
    z = np.load(os.path.join(MAPS, "reference_cases.npz"))
    return {k: z[k] for k in z.files}


SCALES = (1, 2.5, 0, 0.0, 1e-3, 123456.789)
BAD_PFM = ((b"P6\n4 4\n-1.0\n" + bytes(64), Exception, "Not a PFM file."),
           (b"Pf\n4  4\n-1.0\n" + bytes(64), Exception, "Malformed PFM header."),
           (b"Pf\n4 4\n-1.0\n" + bytes(60), ValueError, "cannot reshape array of size 15 into shape"),
           (b"Pf\n4 4\nabc\n" + bytes(64), ValueError, "could not convert string to float"))


def _cases():
    rng = np.random.default_rng(5)
    yield "hw", rng.uniform(425, 935, size=(31, 45)).astype(np.float32)
    yield "hw1", rng.uniform(0, 1, size=(8, 5, 1)).astype(np.float32)
    yield "hw3", rng.normal(size=(12, 7, 3)).astype(np.float32)
    yield "row", rng.normal(size=(1, 9)).astype(np.float32)
    yield "col", rng.normal(size=(9, 1)).astype(np.float32)
    yield "tall", rng.normal(size=(1300, 3)).astype(np.float32)  # more rows than one I/O-vector batch
    yield "noncontig", np.asfortranarray(rng.normal(size=(6, 10)).astype(np.float32))
    yield "strided", rng.normal(size=(12, 20)).astype(np.float32)[::2, ::3]


# ---------------------------------------------------------------- oracle pinning

@pytest.mark.parametrize("name", NAMES)
def test_oracle_reproduces_the_reference_written_fixtures(expected, name):
    arr = expected[f"{name}.input"]
    assert mo.encode_pfm(arr) == open(os.path.join(MAPS, f"{name}.pfm"), "rb").read()
    assert mo.encode_bin(arr) == open(os.path.join(MAPS, f"{name}.bin"), "rb").read()
    got, scale = mo.decode_pfm(open(os.path.join(MAPS, f"{name}.pfm"), "rb").read())
    assert scale == 1.0 and _same(got, expected[f"{name}.pfm"])
    assert _same(mo.decode_bin(open(os.path.join(MAPS, f"{name}.bin"), "rb").read()), expected[f"{name}.bin"])


def test_oracle_reads_the_foreign_big_endian_fixture(expected):
    got, scale = mo.decode_pfm(open(os.path.join(MAPS, "foreign_be.pfm"), "rb").read())
    assert scale == 2.5 and _same(got, expected["foreign_be.pfm"])


def test_oracle_matches_the_unmodified_reference(ref_io):
    for tag, arr in _cases():
        assert np.array_equal(ref_io[f"{tag}.input"], arr), tag
        for ext, enc in (("pfm", mo.encode_pfm), ("bin", mo.encode_bin)):
            blob = ref_io[f"{tag}.{ext}.bytes"].tobytes()
            assert enc(arr) == blob, (tag, ext)
            want = ref_io[f"{tag}.{ext}.read"]
            got = mo.decode_pfm(blob)[0] if ext == "pfm" else mo.decode_bin(blob)
            assert _same(want, got), (tag, ext)


# ---------------------------------------------------------------- native library (host code: runs on the CPU box too)

@pytest.mark.parametrize("name", NAMES)
def test_native_reads_the_reference_written_fixtures(expected, name):
    got, scale = dio.read_pfm(os.path.join(MAPS, f"{name}.pfm"))
    assert scale == 1.0 and _same(got, expected[f"{name}.pfm"])
    assert _same(dio.read_bin(os.path.join(MAPS, f"{name}.bin")), expected[f"{name}.bin"])
    assert _same(dio.read_map(os.path.join(MAPS, f"{name}.bin")), expected[f"{name}.bin"])
    assert _same(dio.read_map(os.path.join(MAPS, f"{name}.pfm")), expected[f"{name}.pfm"])


@pytest.mark.parametrize("name", NAMES)
def test_native_writes_the_reference_bytes(expected, name, tmp_path):
    arr = expected[f"{name}.input"]
    for ext in ("pfm", "bin"):
        p = str(tmp_path / f"out.{ext}")
        dio.save_map(p, arr)
        assert open(p, "rb").read() == open(os.path.join(MAPS, f"{name}.{ext}"), "rb").read()


def test_native_reads_big_endian_pfm_with_scale(expected):
    got, scale = dio.read_pfm(os.path.join(MAPS, "foreign_be.pfm"))
    assert scale == 2.5 and _same(got, expected["foreign_be.pfm"])


def test_native_matches_the_oracle_on_ragged_shapes(tmp_path):
    for tag, arr in _cases():
        for ext, enc in (("pfm", mo.encode_pfm), ("bin", mo.encode_bin)):
            p = str(tmp_path / f"{tag}.{ext}")
            dio.save_map(p, arr)
            blob = open(p, "rb").read()
            assert blob == enc(arr), (tag, ext)
            want = mo.decode_pfm(blob)[0] if ext == "pfm" else mo.decode_bin(blob)
            assert _same(dio.read_map(p), want), (tag, ext)


def test_native_matches_the_unmodified_reference_both_directions(ref_io, tmp_path):
    for tag, arr in _cases():
        for ext in ("pfm", "bin"):
            mine, theirs = str(tmp_path / f"mine_{tag}.{ext}"), str(tmp_path / f"theirs_{tag}.{ext}")
            dio.save_map(mine, arr)
            with open(theirs, "wb") as f:
                f.write(ref_io[f"{tag}.{ext}.bytes"].tobytes())
            assert open(mine, "rb").read() == open(theirs, "rb").read(), (tag, ext)
            # (the bytes are equal, so the reference reads `mine` as it read its own file)
            assert _same(dio.read_map(theirs), ref_io[f"{tag}.{ext}.read"]), (tag, ext)
    p = str(tmp_path / "scaled.pfm")
    for i, scale in enumerate(SCALES):
        dio.save_pfm(p, arr, scale)
        assert open(p, "rb").read() == ref_io[f"scaled{i}.bytes"].tobytes(), scale
        assert dio.read_pfm(p)[1] == float(ref_io[f"scaled{i}.scale"])


def test_empty_maps_round_trip(tmp_path):
    for shape in ((0, 5), (4, 0), (0, 0, 3)):
        arr = np.zeros(shape, np.float32)
        for ext, enc in (("pfm", mo.encode_pfm), ("bin", mo.encode_bin)):
            p = str(tmp_path / f"e.{ext}")
            dio.save_map(p, arr)
            assert open(p, "rb").read() == enc(arr)
            back = dio.read_pfm(p)[0] if ext == "pfm" else dio.read_bin(p)  # (read_map of a 0 x 0 map divides by zero, as in the reference)
            assert back.shape == (shape[0], shape[1], shape[2] if len(shape) == 3 else 1) and back.dtype == np.float32


def test_error_behaviour_follows_the_reference(tmp_path):
    f32 = np.zeros((4, 4), np.float32)
    with pytest.raises(Exception, match="only pfm and bin are supported"):
        dio.save_map(str(tmp_path / "x.png"), f32)
    with pytest.raises(Exception, match="only pfm and bin are supported"):
        dio.read_map(str(tmp_path / "x.exr"))
    with pytest.raises(Exception, match="Image dtype must be float32."):
        dio.save_pfm(str(tmp_path / "x.pfm"), f32.astype(np.float64))
    with pytest.raises(Exception, match="Image data type must be float32."):
        dio.save_bin(str(tmp_path / "x.bin"), f32.astype(np.float64))
    for fn in (dio.save_pfm, dio.save_bin):
        with pytest.raises(Exception, match="H x W x 3, H x W x 1 or H x W"):
            fn(str(tmp_path / "y.pfm"), np.zeros((4, 4, 2), np.float32))
    with pytest.raises(FileNotFoundError):
        dio.read_pfm(str(tmp_path / "missing.pfm"))
    bad = tmp_path / "bad.pfm"
    bad.write_bytes(b"P6\n4 4\n-1.0\n" + bytes(64))
    with pytest.raises(Exception, match="Not a PFM file."):
        dio.read_pfm(str(bad))
    bad.write_bytes(b"Pf\n4  4\n-1.0\n" + bytes(64))
    with pytest.raises(Exception, match="Malformed PFM header."):
        dio.read_pfm(str(bad))
    bad.write_bytes(b"Pf\n4 4\n-1.0\n" + bytes(60))  # one float short
    with pytest.raises(ValueError, match="cannot reshape array of size 15 into shape"):
        dio.read_pfm(str(bad))
    bad.write_bytes(b"Pf\n4 4\nabc\n" + bytes(64))
    with pytest.raises(ValueError, match="could not convert string to float"):
        dio.read_pfm(str(bad))
    badbin = tmp_path / "bad.bin"
    badbin.write_bytes(b"4&4&1&" + bytes(60))
    with pytest.raises(ValueError, match="cannot reshape array of size 15 into shape"):
        dio.read_bin(str(badbin))


def test_reference_raises_the_same_errors(ref_io, tmp_path):
    bad = tmp_path / "bad.pfm"
    for i, (blob, exc, text) in enumerate(BAD_PFM):
        kind, message = str(ref_io[f"error{i}.type"]), str(ref_io[f"error{i}.message"])
        assert issubclass(getattr(builtins, kind), exc) and re.search(text, message), (kind, message)
        bad.write_bytes(blob)
        with pytest.raises(exc, match=text):
            dio.read_pfm(str(bad))


def test_c_abi_rejects_bad_arguments(tmp_path):
    from patchmatchnet_b200 import _native

    lib = _native.lib()
    info = _native.MapInfo()
    assert lib.pmb200_map_probe(None, 1, info) == -1
    assert lib.pmb200_map_probe(b"/nonexistent/x.pfm", 7, info) == -1
    assert lib.pmb200_map_probe(b"/nonexistent/x.pfm", 1, info) == -3 and b"No such file" in lib.pmb200_last_error()
    assert lib.pmb200_map_write(str(tmp_path / "x.pfm").encode(), 1, None, 4, 4, 2, 1.0) == -1
    p = os.path.join(MAPS, "depth_hw.pfm").encode()
    small = np.zeros(8, np.float32)
    assert lib.pmb200_map_read(p, 1, small.ctypes.data, 8, info) == -1 and b"too small" in lib.pmb200_last_error()
    assert (info.width, info.height, info.channels, info.big_endian, info.scale) == (37, 23, 1, 0, 1.0)


@pytest.mark.gpu
def test_device_round_trip_through_pinned_buffers(expected, tmp_path):
    dev = torch.device("cuda:0")
    for name in NAMES:
        for ext in ("pfm", "bin"):
            t = dio.read_map_to_device(os.path.join(MAPS, f"{name}.{ext}"), dev)
            torch.cuda.synchronize()
            assert t.is_cuda and _same(t.cpu().numpy(), expected[f"{name}.{ext}"])
            out = str(tmp_path / f"{name}.{ext}")
            dio.save_map_from_device(out, t)
            assert open(out, "rb").read() == open(os.path.join(MAPS, f"{name}.{ext}"), "rb").read()
    # a [H,W] device map (what the network emits) and a non-contiguous view
    d = torch.from_numpy(expected["depth_hw.input"]).to(dev)
    dio.save_map_from_device(str(tmp_path / "d.pfm"), d)
    assert open(str(tmp_path / "d.pfm"), "rb").read() == open(os.path.join(MAPS, "depth_hw.pfm"), "rb").read()
    dio.save_map_from_device(str(tmp_path / "dt.bin"), d.t())
    assert open(str(tmp_path / "dt.bin"), "rb").read() == mo.encode_bin(np.ascontiguousarray(expected["depth_hw.input"].T))
