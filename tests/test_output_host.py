"""Output stage (src/gui.cpp) on the CPU side: the oracle restatement against the reference's golden vectors
(tests/golden/output_kat.npz, made by make_golden.py from the compiled gui.cpp) and against the compiled reference, live
or through its stored outputs (tests/golden/pin_live.npz); the product's host-only pieces (camera orbit, PNG writer);
and the no-GPU error behaviour of the device entry points."""
import struct
import zlib
from pathlib import Path

import numpy as np
import pytest

from helpers import assert_same_record, bits, reference_record
from ipt_b200 import capi

GOLD = Path(__file__).resolve().parent / "golden"


@pytest.fixture(scope="module")
def kat():
    return np.load(GOLD / "output_kat.npz")


@pytest.mark.parametrize("name", ["synthetic", "box"])
def test_oracle_output_stage_equals_reference_golden(name, kat, oracle):
    img = kat[f"{name}_image"]
    assert np.array_equal(bits(oracle.image_normalize(img)), bits(kat[f"{name}_normalize"]))
    assert np.array_equal(oracle.image_save_bytes(img), kat[f"{name}_bytes"])
    for c, g in zip(kat[f"{name}_cutoffs"], kat[f"{name}_glare"]):
        assert np.array_equal(bits(oracle.image_glare(img, float(c))), bits(g)), c
    assert kat[f"{name}_bytes"].max() == 255 and len(np.unique(kat[f"{name}_bytes"])) > 50


def test_oracle_camera_orbit_equals_reference_golden(kat, oracle):
    cams = kat["orbit_cameras"]
    for i, k in enumerate(kat["orbit_keys"]):
        got = oracle.camera_orbit(cams[i, 0], cams[i, 1], int(k))
        assert np.array_equal(bits(got), bits(cams[i + 1])), (i, k)


def output_record(chk):
    """Random images, ragged sizes: normalize(), Gui::save bytes and glare() of src/gui.cpp, and a run of camera keys, on
    either checker (the oracle or the compiled reference: same interface)."""
    rng = np.random.default_rng(17)
    out = {}
    for (h, w) in [(1, 1), (3, 5), (40, 57), (64, 64)]:
        img = (rng.random((h, w)).astype(np.float32) ** 5 * np.float32(6.0)).astype(np.float32)
        img[rng.random((h, w)) < 0.3] = 0
        img.flat[0] = 2.5  # never black
        out[f"normalize_{h}x{w}"] = bits(chk.image_normalize(img))
        out[f"bytes_{h}x{w}"] = chk.image_save_bytes(img)
        for c in [1.01, 0.4, 100.0]:
            out[f"glare_{h}x{w}_{c}"] = bits(chk.image_glare(img, c))
    pos, d = np.array([1.5, -2.0, 0.7], np.float32), np.array([-0.3, 0.9, -0.2], np.float32)
    for i, k in enumerate([0, 1, 2, 3, 1, 1, 3, 0]):
        cam = chk.camera_orbit(pos, d, k)
        out[f"orbit_{i}"] = bits(cam)
        pos, d = cam[0], cam[1]
    return out


def test_oracle_output_stage_live_against_reference(oracle, ref_or_none, pins):
    """Every function of the restatement is bit-identical to the compiled gui.cpp: live where the reference is built,
    else against its stored outputs (tests/golden/pin_live.npz)."""
    want = reference_record(pins, ref_or_none, "output", output_record)
    assert_same_record(output_record(oracle), want)


def test_product_camera_orbit_bit_exact(kat, lib):
    """ipt_camera_orbit is host arithmetic: runs without a GPU, equal to the reference's glm expressions to the bit."""
    cams = kat["orbit_cameras"]
    for i, k in enumerate(kat["orbit_keys"]):
        cam = capi.Camera()
        cam.position[:] = cams[i, 0].tolist(); cam.direction[:] = cams[i, 1].tolist()
        capi.camera_orbit(cam, int(k))
        got = np.array([list(cam.position), list(cam.direction), list(cam.right), list(cam.up)], np.float32)
        assert np.array_equal(bits(got), bits(cams[i + 1])), (i, k)
    assert lib.ipt_camera_orbit(None, 0) != 0 and lib.ipt_camera_orbit(capi.Camera(), 9) != 0
    # 24 lefts are a full turn (pi/12 each) up to rounding
    cam = capi.Camera(); cam.position[:] = [0.0, -3.0, 0.1]; cam.direction[:] = [0.0, 0.8, -0.6]
    for _ in range(24):
        capi.camera_orbit(cam, 0)
    assert np.allclose(list(cam.position), [0.0, -3.0, 0.1], atol=2e-5)


def decode_png_gray8(data: bytes):
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, idat, w = 8, b"", None
    while pos < len(data):
        (n,), typ = struct.unpack(">I", data[pos:pos + 4]), data[pos + 4:pos + 8]
        body = data[pos + 8:pos + 8 + n]
        (crc,) = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        assert zlib.crc32(typ + body) == crc, typ
        if typ == b"IHDR":
            w, h, depth, colour, comp, filt, lace = struct.unpack(">IIBBBBB", body)
            assert (depth, colour, comp, filt, lace) == (8, 0, 0, 0, 0)
        elif typ == b"IDAT":
            idat += body
        pos += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(h, w + 1)
    assert (raw[:, 0] == 0).all()
    return raw[:, 1:]


@pytest.mark.parametrize("shape", [(1, 1), (7, 300), (300, 301)])
def test_png_writer_round_trip(shape, lib, tmp_path):
    """ipt_write_png_gray8 (host only): valid signature, chunk CRCs, zlib stream (stored blocks > 64 KiB), same pixels."""
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    path = tmp_path / "x.png"
    capi.write_png_gray8(path, img)
    assert np.array_equal(decode_png_gray8(path.read_bytes()), img)
    try:
        from PIL import Image
        assert np.array_equal(np.asarray(Image.open(path)), img)
    except ImportError:
        pass
    with pytest.raises(capi.IptError):
        capi.write_png_gray8(tmp_path / "no_such_dir" / "x.png", img)


def test_output_stage_fails_loudly_without_gpu(lib, has_gpu):
    if has_gpu:
        pytest.skip("GPU present")
    img = np.ones((4, 4), np.float32)
    for fn in (lambda: capi.image_glare(img, 0.5), lambda: capi.image_normalize(img), lambda: capi.image_save_bytes(img)):
        with pytest.raises(capi.IptError) as e:
            fn()
        assert e.value.code == capi.IPT_ERR_NO_DEVICE
