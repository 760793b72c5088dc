"""CPU: pins the line front-end oracle (oracle/lines.cc).

* LSD: the restatement of cv::LineSegmentDetector is compared bit-for-bit with cv2 4.13
  `createLineSegmentDetector(1, 0.5, 0.6, 2.0, 22.5, 1.0, 0.6, 1024)` (the options of line_extractor.cc:113-122), in the
  "det" mode the CUDA path implements and in the "cv" mode (libm, sequential sums).
* the OpenCV primitives LBD uses (GaussianBlur 5x5 sigma 1, Sobel 3x3 -> CV_16S, LineIterator count) against cv2;
* LBD itself is vendored reference source (binary_descriptor_custom.cpp) restated line by line: structural checks.
* detmath (deterministic sin/cos/atan2) against libm, and the two textual copies are identical.
"""
import math
from pathlib import Path

import numpy as np
import pytest

import oracle_api
import synth

cv2 = pytest.importorskip("cv2")
ROOT = Path(__file__).resolve().parent.parent


def _images():
    out = [("texture640", synth.make_texture(1)), ("texture752", synth.make_texture(2, h=480, w=752)),
           ("lines640", synth.make_line_image(1)), ("lines752", synth.make_line_image(2, 480, 752)),
           ("noise", np.random.default_rng(5).integers(0, 256, (480, 640), dtype=np.uint8)),
           ("flat", np.full((480, 640), 77, np.uint8))]
    # the reference's test/data/equirectangular_image_00{1,2}.jpg at 640x480, central 240 rows (tools/gen_golden.py)
    for i in (1, 2):
        f = f"equirectangular_image_00{i}_band.png"
        out.append((f, cv2.imread(str(ROOT / "tests" / "golden" / f), cv2.IMREAD_GRAYSCALE)))
    return out


def _cv_lsd(img):
    lsd = cv2.createLineSegmentDetector(1, 0.5, 0.6, 2.0, 22.5, 1.0, 0.6, 1024)
    r = lsd.detect(img)[0]
    return np.zeros((0, 4), np.float32) if r is None else r.reshape(-1, 4)


def test_scaled_image_matches_cv2(orc):
    for name, img in _images():
        g = cv2.GaussianBlur(img, (11, 11), 1.2)
        s = cv2.resize(g, None, fx=0.5, fy=0.5, interpolation=cv2.INTER_LINEAR_EXACT)
        assert np.array_equal(orc.lsd_scaled(img), s), name


@pytest.mark.parametrize("mode", [oracle_api.LSD_DET, oracle_api.LSD_CV])
def test_lsd_segments_bit_exact_vs_cv2(orc, mode):
    total = 0
    for name, img in _images():
        ref = _cv_lsd(img)
        got = orc.lsd_detect(img, mode)
        assert got.shape == ref.shape, f"{name}: {len(got)} vs {len(ref)} segments"
        assert np.array_equal(got, ref), name
        total += len(ref)
    assert total > 2000


def test_lbd_gradients_match_cv2(orc):
    for name, img in _images()[:5]:
        g = cv2.GaussianBlur(img, (5, 5), 1)
        dx = cv2.Sobel(g, cv2.CV_16S, 1, 0, ksize=3)
        dy = cv2.Sobel(g, cv2.CV_16S, 0, 1, ksize=3)
        ox, oy = orc.lbd_gradients(img)
        assert np.array_equal(ox, dx) and np.array_equal(oy, dy), name


def test_keyline_fields_and_line_iterator_count(orc):
    img = synth.make_line_image(3)
    kls = orc.lsd_keylines(img, 60.0)
    assert len(kls) > 50
    assert np.array_equal(kls["class_id"], np.arange(len(kls)))
    assert (kls["octave"] == 0).all() and (kls["line_length"] > 60).all()
    for k in kls[:40]:
        # cv::LineIterator count == number of pixels cv2.line sets (8-connected, thickness 1)
        canvas = np.zeros(img.shape, np.uint8)
        p0 = (int(np.rint(k["start_x"])), int(np.rint(k["start_y"])))
        p1 = (int(np.rint(k["end_x"])), int(np.rint(k["end_y"])))
        cv2.line(canvas, p0, p1, 255, 1, cv2.LINE_8)
        assert int(np.count_nonzero(canvas)) == int(k["num_pixels"])
        assert abs(k["angle"] - math.atan2(k["end_y"] - k["start_y"], k["end_x"] - k["start_x"])) < 1e-6
        assert k["response"] == np.float32(k["line_length"]) / np.float32(640)


def test_line_extract_structure(orc):
    img = synth.make_line_image(4)
    kl, lbd, fn = orc.line_extract(img)
    assert 60 < len(kl) < 1024 and lbd.shape == (len(kl), 32) and fn.shape == (len(kl), 3)
    assert (kl["line_length"] >= 60).all()
    # line function: both end points lie on it, normalised normal
    sp = np.stack([kl["start_x"], kl["start_y"], np.ones(len(kl))], 1).astype(np.float64)
    ep = np.stack([kl["end_x"], kl["end_y"], np.ones(len(kl))], 1).astype(np.float64)
    assert np.abs((sp * fn).sum(1)).max() < 1e-9 and np.abs((ep * fn).sum(1)).max() < 1e-9
    assert np.allclose(np.hypot(fn[:, 0], fn[:, 1]), 1.0, atol=1e-12)
    # float descriptor: unit norm, binary = 8 comparisons per band pair
    d8, df = orc.lbd_compute(img, kl)
    assert np.array_equal(d8, lbd)
    assert np.allclose((df.astype(np.float64) ** 2).sum(1), 1.0, atol=1e-5)
    comb = [(0, 1), (0, 2), (0, 3), (0, 4), (0, 5), (0, 6), (1, 2), (1, 3), (1, 4), (1, 5), (1, 6), (2, 3), (2, 4), (2, 5),
            (2, 6), (2, 7), (2, 8), (3, 4), (3, 5), (3, 6), (3, 7), (3, 8), (4, 5), (4, 6), (4, 7), (4, 8), (5, 6), (5, 7),
            (5, 8), (6, 7), (6, 8), (7, 8)]
    for c, (i, j) in enumerate(comb):
        bits = (df[:, 8 * i:8 * i + 8] > df[:, 8 * j:8 * j + 8]).astype(np.uint8)
        assert np.array_equal((bits << np.arange(8, dtype=np.uint8)).sum(1).astype(np.uint8), d8[:, c])
    # the descriptor of a line is (nearly) independent of libm vs detmath
    d8m, _ = orc.lbd_compute(img, kl, libm=1)
    assert (np.unpackbits(d8 ^ d8m, axis=1).sum(1) <= 2).all()
    # a flat image has no line and the extractor returns nothing
    kl0, lbd0, fn0 = orc.line_extract(np.full((480, 640), 9, np.uint8))
    assert len(kl0) == 0


def test_detmath_copies_identical_and_accurate(orc):
    a = (ROOT / "oracle" / "detmath.h").read_text()
    b = (ROOT / "structure-plp-slam_b200" / "csrc" / "detmath.h").read_text()
    assert a == b
    import ctypes as C
    import subprocess
    import tempfile
    src = '#include "%s"\nextern "C" { double t_sin(double x){return det_sin(x);} double t_cos(double x){return det_cos(x);}' \
          ' double t_atan2(double y,double x){return det_atan2(y,x);} }\n' % (ROOT / "oracle" / "detmath.h")
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "t.cc").write_text(src)
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", str(Path(d) / "t.cc"), "-o",
                        str(Path(d) / "t.so")], check=True)
        lib = C.CDLL(str(Path(d) / "t.so"))
        for f in (lib.t_sin, lib.t_cos):
            f.restype, f.argtypes = C.c_double, [C.c_double]
        lib.t_atan2.restype, lib.t_atan2.argtypes = C.c_double, [C.c_double, C.c_double]
        rng = np.random.default_rng(0)
        for x in rng.uniform(-4 * math.pi, 4 * math.pi, 20000):
            assert abs(lib.t_sin(x) - math.sin(x)) < 2.3e-16 and abs(lib.t_cos(x) - math.cos(x)) < 2.3e-16
            xf = float(np.float32(x))
            assert np.float32(lib.t_cos(xf)) == np.float32(math.cos(xf))
        for y, x in rng.uniform(-700, 700, (20000, 2)):
            assert abs(lib.t_atan2(y, x) - math.atan2(y, x)) < 9e-16
        assert lib.t_atan2(0.0, -1.0) == math.pi and lib.t_atan2(1.0, 0.0) == math.pi / 2
