"""Oracle 8-bit image primitives vs the in-container cv2 (the live golden; OpenCV is
a system dependency of the reference, SURVEY.md §8c / Appendix B) and vs literal
formulas for the app/deepseg.cc helpers."""
import os

import cv2
import numpy as np
import pytest

from oracle import pyoracle as po
from tests.conftest import ROOT

RNG = np.random.default_rng(42)

# every hot-path geometry of SURVEY.md §8 + ragged ones
RESIZES = [
    (480, 480, 256, 256, 3), (720, 720, 257, 257, 3), (1280, 720, 256, 144, 3), (640, 480, 192, 144, 3),
    (480, 480, 257, 257, 3), (640, 480, 128, 96, 3),
    (256, 256, 480, 480, 1), (256, 144, 1280, 720, 1), (192, 144, 640, 480, 1), (257, 257, 720, 720, 1),
    (33, 33, 480, 480, 1), (1280, 720, 640, 480, 3), (512, 512, 256, 256, 3), (100, 37, 313, 211, 3),
    (640, 480, 640, 480, 3), (7, 5, 3, 2, 1), (2, 2, 9, 9, 3), (1, 1, 4, 4, 1),
]


@pytest.mark.parametrize("sw,sh,dw,dh,cn", RESIZES)
def test_resize_linear_bit_exact(sw, sh, dw, dh, cn):
    src = RNG.integers(0, 256, (sh, sw, cn) if cn > 1 else (sh, sw), dtype=np.uint8)
    assert np.array_equal(po.resize_linear_u8(src, dw, dh), cv2.resize(src, (dw, dh)))


@pytest.mark.slow
def test_resize_linear_4k():
    src = RNG.integers(0, 256, (540, 960, 3), dtype=np.uint8)
    assert np.array_equal(po.resize_linear_u8(src, 3840, 2160), cv2.resize(src, (3840, 2160)))


@pytest.mark.parametrize("w,h", [(480, 480), (1280, 720), (7, 5), (5, 5), (640, 480), (3, 9)])
def test_box_blur_bit_exact(w, h):
    src = RNG.integers(0, 256, (h, w), dtype=np.uint8)
    assert np.array_equal(po.box_blur5(src), cv2.blur(src, (5, 5)))
    sat = np.full((h, w), 255, np.uint8)
    assert np.array_equal(po.box_blur5(sat), cv2.blur(sat, (5, 5)))


def test_box_blur_rounding_identity():
    """cvRound(S/25.0) == (S + 12) // 25 for every reachable window sum (used by the CUDA kernel)."""
    s = np.arange(0, 25 * 255 + 1)
    assert np.array_equal(np.rint(s * (1.0 / 25)).astype(int), (s + 12) // 25)


def test_rgb2yuv_bit_exact():
    src = RNG.integers(0, 256, (480, 640, 3), dtype=np.uint8)
    assert np.array_equal(po.rgb2yuv(src), cv2.cvtColor(src, cv2.COLOR_RGB2YUV))
    # all 2^24 colours
    g = np.arange(256, dtype=np.uint8)
    cube = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(4096, 4096, 3)
    assert np.array_equal(po.rgb2yuv(cube), cv2.cvtColor(cube, cv2.COLOR_RGB2YUV))


def test_yuyv_pack_literal():  # app/deepseg.cc:87-106
    src = RNG.integers(0, 256, (6, 8, 3), dtype=np.uint8)
    yuv = cv2.cvtColor(src, cv2.COLOR_RGB2YUV).reshape(-1, 3).astype(int)
    exp = np.empty((48, 2), np.uint8)
    for i in range(0, 48, 2):
        exp[i] = (yuv[i, 0], (yuv[i, 2] + yuv[i + 1, 2]) // 2)
        exp[i + 1] = (yuv[i + 1, 0], (yuv[i, 1] + yuv[i + 1, 1]) // 2)
    assert np.array_equal(po.convert_rgb_to_yuyv(src).reshape(-1, 2), exp)


def test_alpha_blend_literal_and_division_identity():  # app/deepseg.cc:108-134
    a = RNG.integers(0, 256, (16, 16, 3), dtype=np.uint8)
    b = RNG.integers(0, 256, (16, 16, 3), dtype=np.uint8)
    m = RNG.integers(0, 256, (16, 16), dtype=np.uint8)
    exp = ((a.astype(int) * m[..., None] + b.astype(int) * (255 - m[..., None].astype(int))) // 255).astype(np.uint8)
    assert np.array_equal(po.alpha_blend(a, b, m), exp)
    # x/255 == (x + 1 + (x >> 8)) >> 8 on [0, 255*255] — the CUDA kernel's division-free form
    x = np.arange(0, 255 * 255 + 1)
    assert np.array_equal(x // 255, (x + 1 + (x >> 8)) >> 8)
    # extremes: mask 255 -> background, mask 0 -> frame
    assert np.array_equal(po.alpha_blend(a, b, np.full((16, 16), 255, np.uint8)), a)
    assert np.array_equal(po.alpha_blend(a, b, np.zeros((16, 16), np.uint8)), b)


def _cv_convert(s, alpha, beta):
    g_in = cv2.GMat()
    comp = cv2.GComputation(g_in, cv2.gapi.convertTo(g_in, cv2.CV_32F, alpha, beta))
    return comp.apply(cv2.gin(s))


@pytest.mark.parametrize("alpha,beta", [(float(np.float32(1 / 255.0)), 0.0), (float(np.float32(1 / 127.5)), -1.0)])
def test_convert_to_bit_exact(alpha, beta):  # lib/libbackscrub.cc:302 via Mat::convertTo
    s = RNG.integers(0, 256, (257, 257, 3), dtype=np.uint8)
    try:
        ref = _cv_convert(s, alpha, beta)
    except Exception:
        pytest.skip("cv2.gapi.convertTo unavailable")
    got = po.convert_u8_f32(s, alpha, beta)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("w,h", [(256, 256), (257, 257), (256, 144), (160, 96)])
def test_bilateral_vs_cv2(w, h):
    """cv::bilateralFilter(5,100,100).  OpenCV's own code paths (IPP / AVX2+FMA / SSE
    baseline) already disagree with one another on a few pixels per image by 1 LSB
    (float summation order), so the pin is: max |diff| <= 1 and <= 1e-4 of the values."""
    img = cv2.imread(os.path.join(ROOT, "backgrounds", "screenshot.jpg"))
    srcs = [cv2.resize(img[:, :640], (w, h)), RNG.integers(0, 256, (h, w, 3), dtype=np.uint8)]
    for src in srcs:
        got = po.bilateral_d5(src).astype(int)
        for ipp in (True, False):
            cv2.ipp.setUseIPP(ipp)
            ref = cv2.bilateralFilter(src, 5, 100.0, 100.0).astype(int)
            d = np.abs(got - ref)
            assert d.max() <= 1
            assert (d != 0).mean() <= 1e-4
        cv2.ipp.setUseIPP(True)


def test_bilateral_constant_and_border():
    c = np.full((9, 11, 3), 77, np.uint8)
    assert np.array_equal(po.bilateral_d5(c), c)
    z = np.zeros((8, 8, 3), np.uint8)
    assert np.array_equal(po.bilateral_d5(z), z)


def test_yuyv_to_bgr_bit_exact():
    """cv::cvtColor(COLOR_YUV2BGR_YUYV) — the camera ingest conversion (app/deepseg.cc:553,725)."""
    src = RNG.integers(0, 256, (48, 64, 2), dtype=np.uint8)
    assert np.array_equal(po.yuyv_to_bgr(src), cv2.cvtColor(src, cv2.COLOR_YUV2BGR_YUYV))
    # every (Y, U, V) combination on a coarse-but-complete grid of the extremes + all Y
    y = np.arange(256, dtype=np.uint8)
    for u in (0, 1, 16, 127, 128, 129, 240, 255):
        for v in (0, 1, 16, 127, 128, 129, 240, 255):
            row = np.empty((1, 256, 2), np.uint8)
            row[0, :, 0] = y
            row[0, 0::2, 1] = u
            row[0, 1::2, 1] = v
            assert np.array_equal(po.yuyv_to_bgr(row), cv2.cvtColor(row, cv2.COLOR_YUV2BGR_YUYV))


@pytest.mark.parametrize("k", [1, 3, 5, 7, 9, 11, 25, 51, 101])
def test_gaussian_blur_bit_exact(k):  # app/deepseg.cc:657-658 `-p bgblur:k`
    """cv::GaussianBlur(8UC3, k x k, sigma 0): OpenCV's bit-exact 8.8 fixed-point path, IPP on and off,
    including kernels wider than the image (multiple border reflections)."""
    for shape in [(48, 64, 3), (30, 17, 3), (120, 200, 3)]:
        src = RNG.integers(0, 256, shape, dtype=np.uint8)
        got = po.gaussian_blur(src, k)
        for ipp in (True, False):
            cv2.ipp.setUseIPP(ipp)
            assert np.array_equal(got, cv2.GaussianBlur(src, (k, k), 0)), (k, shape, ipp)
        cv2.ipp.setUseIPP(True)


def test_gaussian_taps_all_strengths():
    """taps for every odd k: the error-diffused 8.8 quantisation of cv2.getGaussianKernel(k, 0), summing to 256;
    even / out-of-range strengths are rejected (app/deepseg.cc:423-426)."""
    for k in range(1, 256, 2):
        kd = cv2.getGaussianKernel(k, 0).ravel()
        ref = np.zeros(k, np.int64)
        err, acc = 0.0, 0
        for i in range(k // 2):
            adj = kd[i] * 256.0 + err
            v = int(np.rint(adj))
            err = adj - v
            ref[i] = ref[k - 1 - i] = v
            acc += v
        ref[k // 2] = 256 - 2 * acc
        q = po.gaussian_kernel_q8(k)
        assert np.array_equal(q, ref) and q.sum() == 256, k
    for bad in (0, 2, 24, 257, -3):
        with pytest.raises(ValueError):
            po.gaussian_kernel_q8(bad)


def test_flip_bit_exact():  # app/deepseg.cc:667-673
    src = RNG.integers(0, 256, (21, 34, 3), dtype=np.uint8)
    for code, (fh, fv) in {1: (1, 0), 0: (0, 1), -1: (1, 1)}.items():
        assert np.array_equal(po.flip(src, fh, fv), cv2.flip(src, code))


def test_composite_ex_matches_cv2_composition():
    """or_composite_ex (the main-loop body with its options) vs the same steps composed from cv2 calls."""
    from tests import synth
    from tests.conftest import model_path
    W, H = 640, 480
    bg_raw = synth.background()
    fr = synth.frame(W, H, t=2)
    for bg_src, k, fh, fv, osz in [(bg_raw, 25, True, False, (320, 240)), (None, 9, False, True, (854, 480)), (bg_raw, 0, True, True, None)]:
        o = po.MaskGen(model_path("meet_lite"), W, H)
        out, yuyv, mask = o.composite_ex(fr, bg_src, bgblur=k, flip_h=fh, flip_v=fv, out_size=osz)
        bg = cv2.resize(bg_src, (W, H)) if bg_src is not None else fr.copy()
        if k:
            bg = cv2.GaussianBlur(bg, (k, k), 0)
        ref = po.alpha_blend(bg, fr, mask)
        if fh or fv:
            ref = cv2.flip(ref, -1 if (fh and fv) else (1 if fh else 0))
        if osz:
            ref = cv2.resize(ref, osz)
        assert np.array_equal(out, ref)
        assert np.array_equal(yuyv, po.convert_rgb_to_yuyv(ref))
