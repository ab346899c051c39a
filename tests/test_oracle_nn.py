"""Oracle fp32 ops vs the reference's own single-op known-answer tests.

Vectors transcribed (as data) from the vendored TFLite tests the survey lists
(§4, §8c): kernels/conv_test.cc, depthwise_conv_test.cc, pooling_test.cc,
resize_bilinear_test.cc, activations_test.cc, transpose_conv_test.cc,
fully_connected_test.cc — tolerance ArrayFloatNear 1e-5 (kernels/test_util.h:56-57).
Also pins or_tconv_bias against the stored outputs of the reference's own
lib/transpose_conv_bias.cc (tests/golden/tconv_ref_golden.npz).
"""
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from tests.conftest import ROOT

TOL = 1e-5
TCONV_REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "tconv_ref_golden.npz")


def near(a, b, tol=TOL):
    np.testing.assert_allclose(np.asarray(a, np.float32).ravel(), np.asarray(b, np.float32).ravel(), rtol=0, atol=tol)


# ---- conv_test.cc ---------------------------------------------------------
def test_conv_simple_float32():  # conv_test.cc:165 (stride 2x2, VALID, two batches)
    flt = np.array([1, 2, 3, 4, -1, 1, -1, 1, -1, -1, 1, 1], np.float32).reshape(3, 2, 2, 1)
    bias = [1, 2, 3]
    b0 = np.array([1, 1, 1, 1, 2, 2, 2, 2], np.float32).reshape(2, 4, 1)
    b1 = np.array([1, 2, 3, 4, 1, 2, 3, 4], np.float32).reshape(2, 4, 1)
    near(po.conv2d(b0, flt, bias, stride=(2, 2), padding=po.PAD_VALID), [18, 2, 5, 18, 2, 5])
    near(po.conv2d(b1, flt, bias, stride=(2, 2), padding=po.PAD_VALID), [17, 4, 3, 37, 4, 3])


def test_conv_padding_same():  # conv_test.cc:389 PaddingTest
    flt = np.array([1, 2, 3, 4, -1, 1, -1, 1, -1, -1, 1, 1], np.float32).reshape(3, 2, 2, 1)
    x = np.array([1, 1, 1, 1, 2, 2, 3, 2], np.float32).reshape(2, 4, 1)
    exp = [18, 2, 5, 22, 3, 6, 21, 1, 6, 8, -1, 4, 7, 2, -1, 9, 3, -2, 8, 1, -2, 3, 0, 1]
    near(po.conv2d(x, flt, [1, 2, 3], stride=(1, 1), padding=po.PAD_SAME), exp)


def test_conv_pointwise():  # conv_test.cc:423 PointwiseFloat32
    flt = np.array([1, 2], np.float32).reshape(1, 1, 1, 2)
    b1 = np.array([0.5, 0.5, 1, 1, 1.5, 1.5, 2, 2] * 2, np.float32).reshape(2, 4, 2)
    near(po.conv2d(b1, flt, [0], stride=(1, 1), padding=po.PAD_VALID), [1.5, 3., 4.5, 6.] * 2)


def test_conv_hand_calculated():  # conv_test.cc:508 HandCalculatedFloat32
    x = np.arange(1, 13, dtype=np.float32).reshape(3, 4, 1)
    flt = np.array([1, 4, 7, 2, 5, 8, 3, 6, 9], np.float32).reshape(1, 3, 3, 1)
    near(po.conv2d(x, flt, [0], padding=po.PAD_SAME),
         [105, 150, 183, 95, 235, 312, 357, 178, 187, 234, 261, 121])
    # conv_test.cc:653 HandCalculatedValidFloat32
    near(po.conv2d(x, flt, [0], padding=po.PAD_VALID), [312, 357])


def test_conv_dilation():  # conv_test.cc:805 SimpleTestFloatWithDilation
    x = np.zeros((9, 9, 1), np.float32)
    x[3:6, 3:6] = 1
    flt = np.arange(1, 10, dtype=np.float32).reshape(1, 3, 3, 1)
    near(po.conv2d(x, flt, [0], dil=(3, 3), padding=po.PAD_VALID), [5] * 9)


# ---- depthwise_conv_test.cc -----------------------------------------------
def test_depthwise_activation_relu():  # depthwise_conv_test.cc:162 (depth multiplier 2)
    x = np.array([1, 2, 7, 8, 3, 4, 9, 10, 5, 6, 11, 12], np.float32).reshape(3, 2, 2)
    flt = np.array([1, 2, 3, 4, -9, 10, -11, 12, 5, 6, 7, 8, 13, -14, 15, -16], np.float32).reshape(1, 2, 2, 4)
    out = po.depthwise_conv2d(x, flt, [1, 2, 3, 4], padding=po.PAD_VALID, mult=2, act=po.ACT["RELU"])
    near(out, [71, 0, 99, 0, 91, 0, 127, 0])


def test_depthwise_dilated_same():  # depthwise_conv_test.cc:430-466 SimpleDilatedTestPaddingSame
    x = np.ones((3, 3, 1), np.float32)
    flt = np.array([1, 2, 3, 4], np.float32).reshape(1, 2, 2, 1)
    near(po.depthwise_conv2d(x, flt, [0], dil=(2, 2), padding=po.PAD_SAME), [4, 7, 3, 6, 10, 4, 2, 3, 1])


def test_depthwise_dilated_valid():  # depthwise_conv_test.cc:370-418
    x = np.zeros((9, 9, 1), np.float32)
    x[3:6, 3:6] = 1
    flt = np.arange(1, 10, dtype=np.float32).reshape(1, 3, 3, 1)
    near(po.depthwise_conv2d(x, flt, [0], dil=(3, 3), padding=po.PAD_VALID), [5] * 9)


# ---- pooling_test.cc --------------------------------------------------------
def test_average_pool():  # pooling_test.cc:140
    x = np.array([0, 6, 2, 4, 3, 2, 10, 7], np.float32).reshape(2, 4, 1)
    near(po.average_pool(x, 2, 2, stride=(2, 2)), [2.75, 5.75])


def test_average_pool_relu():  # pooling_test.cc:153
    x = np.array([0, -6, 2, 4, 3, 2, -10, 7], np.float32).reshape(2, 4, 1)
    near(po.average_pool(x, 2, 2, stride=(2, 2), act=po.ACT["RELU"]), [0.0, 0.75])


def test_average_pool_global_matches_mean():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((16, 16, 8)).astype(np.float32)
    out = po.average_pool(x, 16, 16, stride=(16, 16))
    near(out, x.astype(np.float64).mean(axis=(0, 1)), 1e-6)


# ---- resize_bilinear_test.cc ------------------------------------------------
def test_resize_horizontal_vertical():  # :84, :123
    near(po.resize_bilinear(np.array([3, 6], np.float32).reshape(1, 2, 1), 1, 3), [3, 5, 6])
    near(po.resize_bilinear(np.array([3, 9], np.float32).reshape(2, 1, 1), 3, 1), [3, 7, 9])


def test_resize_two_dimensional():  # :156
    x = np.array([3, 6, 9, 12], np.float32).reshape(2, 2, 1)
    near(po.resize_bilinear(x, 3, 3), [3, 5, 6, 7, 9, 10, 9, 11, 12])


def test_resize_half_pixel():  # :236-257
    x = np.array([1, 2, 3, 4], np.float32).reshape(2, 2, 1)
    near(po.resize_bilinear(x, 3, 3, half_pixel=True), [1, 1.5, 2, 2, 2.5, 3, 3, 3.5, 4])


def test_resize_three_dimensional():  # :259
    x = np.array([3, 4, 6, 10, 9, 10, 12, 16], np.float32).reshape(2, 2, 2)
    near(po.resize_bilinear(x, 3, 3), [3, 4, 5, 8, 6, 10, 7, 8, 9, 12, 10, 14, 9, 10, 11, 14, 12, 16])


def test_resize_2x_half_pixel_closed_form():
    """SURVEY Appendix A: exact 2x half-pixel = 1/4,3/4 taps with clamped indices."""
    rng = np.random.default_rng(0)
    x = rng.standard_normal((5, 7, 3)).astype(np.float32)
    out = po.resize_bilinear(x, 10, 14, half_pixel=True)
    def up(a, axis):
        n = a.shape[axis]
        idx = np.arange(n)
        prev = np.take(a, np.clip(idx - 1, 0, n - 1), axis=axis)
        nxt = np.take(a, np.clip(idx + 1, 0, n - 1), axis=axis)
        even = 0.25 * prev + 0.75 * a
        odd = 0.75 * a + 0.25 * nxt
        return np.stack([even, odd], axis=axis + 1).reshape([s * (2 if i == axis else 1) for i, s in enumerate(a.shape)])
    near(out, up(up(x.astype(np.float64), 0), 1), 1e-6)


def test_resize_align_corners_broadcast_and_identity():
    """DeepLab's [1,1,C]->33x33 broadcast and 33->33 identity (align_corners)."""
    v = np.arange(5, dtype=np.float32).reshape(1, 1, 5)
    out = po.resize_bilinear(v, 4, 3, align_corners=True)
    assert np.array_equal(out, np.broadcast_to(v, (4, 3, 5)))
    x = np.random.default_rng(1).standard_normal((6, 6, 2)).astype(np.float32)
    assert np.array_equal(po.resize_bilinear(x, 6, 6, align_corners=True), x)


# ---- activations_test.cc ----------------------------------------------------
def test_logistic_kat():  # activations_test.cc:1037-1049
    x = np.array([0, -6, 2, 4, 3, -2, 10, 1], np.float32)
    near(po.logistic(x), [0.5, 0.002473, 0.880797, 0.982014, 0.952574, 0.119203, 0.999955, 0.731059], 1e-5)


def test_logistic_cutoffs():  # reference/logistic.h:30-57
    x = np.array([17.0, 16.7, -9.5, -20.0, -100.0], np.float32)
    out = po.logistic(x)
    assert out[0] == 1.0 and out[1] == 1.0
    near(out[2:4], np.exp(x[2:4].astype(np.float64)), 1e-9)
    assert out[4] == 0.0


def test_hard_swish_closed_form():  # activations_test.cc:381-499 (closed form on U(-10,10))
    x = np.random.default_rng(7).uniform(-10, 10, 4096).astype(np.float32)
    ref = x.astype(np.float64) * np.clip(x.astype(np.float64) + 3, 0, 6) / 6
    near(po.hard_swish(x), ref, 1e-5)


def test_relu6():  # activations_test.cc:345
    x = np.array([0, -6, 2, 4, 3, -2, 10, 1], np.float32)
    near(po.relu(x, po.ACT["RELU6"]), [0, 0, 2, 4, 3, 0, 6, 1])
    near(po.relu(x, po.ACT["RELU"]), [0, 0, 2, 4, 3, 0, 10, 1])


def test_expf_accuracy():
    x = np.concatenate([np.linspace(-87, 88, 20001), np.linspace(-1, 1, 2001)]).astype(np.float32)
    got = po.expf_array(x).astype(np.float64)
    ref = np.exp(x.astype(np.float64))
    rel = np.abs(got - ref) / ref
    assert rel.max() < 2.5e-7, rel.max()       # ~2 ulp of binary32
    assert po.expf(0.0) == 1.0
    assert po.expf(100.0) == np.inf and po.expf(-100.0) == 0.0


def test_half_to_float_exhaustive():
    L = po.lib()
    h = np.arange(65536, dtype=np.uint16)
    ref = h.view(np.float16).astype(np.float32)
    got = np.array([L.or_half_to_float(int(v)) for v in h], np.float32)
    m = ~np.isnan(ref)
    assert np.array_equal(got[m].view(np.uint32), ref[m].view(np.uint32))
    assert np.isnan(got[~m]).all()


# ---- fully_connected_test.cc ------------------------------------------------
def test_fully_connected_simple():  # fully_connected_test.cc SimpleTest (float)
    w = np.array([list(range(1, 11))] * 3, np.float32)
    x = np.array([[1, 2, 3, 4, 5, 6, 7, 8, -9, -10], [1, 2, 3, 4, 5, 6, 7, -8, 9, -10]], np.float32)
    near(po.fully_connected(x, w, [1, 2, 3]), [24, 25, 26, 58, 59, 60])


# ---- add / mul --------------------------------------------------------------
def test_add_mul():
    a = np.array([-2.0, 0.2, 0.7, 0.8], np.float32)
    b = np.array([0.1, 0.2, 0.3, 0.5], np.float32)
    near(po.add(a, b), [-1.9, 0.4, 1.0, 1.3])                      # add_test.cc FloatAddOpModel
    near(po.mul(a.reshape(4, 1), b.reshape(4, 1)), [-0.2, 0.04, 0.21, 0.4])  # mul_test.cc
    x = np.arange(12, dtype=np.float32).reshape(2, 2, 3)
    s = np.array([1, 10, 100], np.float32)
    near(po.mul(x, s), x * s)


# ---- transpose conv (custom op) ---------------------------------------------
def test_tconv_simple_kat():  # transpose_conv_test.cc:145 (k3 s1 SAME, bias 0)
    x = np.arange(1, 17, dtype=np.float32).reshape(4, 4, 1)
    w = np.arange(1, 10, dtype=np.float32).reshape(1, 3, 3, 1)
    exp = [29, 62, 83, 75, 99, 192, 237, 198, 207, 372, 417, 330, 263, 446, 485, 365]
    near(po.tconv_bias(x, w, [0], stride=(1, 1)), exp)


def test_tconv_two_filters_kat():  # transpose_conv_test.cc:172
    x = np.arange(1, 33, dtype=np.float32).reshape(4, 4, 2)
    w = np.arange(1, 19, dtype=np.float32).reshape(1, 3, 3, 2)
    exp = [184, 412, 568, 528, 678, 1347, 1689, 1434, 1494, 2715, 3057, 2442, 1968, 3352, 3652, 2760]
    near(po.tconv_bias(x, w, [0], stride=(1, 1)), exp)


def test_tconv_survey_known_answer():  # SURVEY.md §8c (probe of the compiled reference op)
    x = np.array([1, 2, 3, 4], np.float32).reshape(2, 2, 1)
    w = np.array([1, 10, 100, 1000], np.float32).reshape(1, 2, 2, 1)
    exp = [1.5, 10.5, 2.5, 20.5, 100.5, 1000.5, 200.5, 2000.5, 3.5, 30.5, 4.5, 40.5, 300.5, 3000.5, 400.5, 4000.5]
    near(po.tconv_bias(x, w, [0.5]), exp)


@pytest.mark.parametrize("shape", [(8, 8, 16, 1), (5, 7, 16, 2), (3, 3, 4, 3)])
def test_tconv_matches_compiled_reference(shape):
    """or_tconv_bias vs the reference's own lib/transpose_conv_bias.cc (k2 s2 SAME, the
    MLKit/Meet configuration), whose outputs on these seeded inputs are stored in
    tests/golden/tconv_ref_golden.npz (tests/golden/make_golden.py).  The reference accumulates
    `+= a*b` (compiler-dependent contraction) and the oracle uses fmaf, so the bound is a few
    ulp, not bit equality."""
    ih, iw, ic, oc = shape
    z = np.load(TCONV_REF_GOLDEN)
    key = "case_%dx%dx%dx%d" % shape
    x, w, b, ref = z[key + "_x"], z[key + "_w"], z[key + "_b"], z[key + "_y"]
    got = po.tconv_bias(x, w, b)
    # lib/transpose_conv_bias.cc:157-184: SAME trims (k - (in-1)%stride - 1) -> 2*in for even, 2*in-1 for odd sizes
    assert ref.shape == got.shape == (2 * ih - ih % 2, 2 * iw - iw % 2, oc)
    np.testing.assert_allclose(got, ref, rtol=3e-6, atol=3e-6)


def test_ref_tconv_known_answer():
    """The stored output of the compiled reference op on the survey's known-answer input."""
    exp = [1.5, 10.5, 2.5, 20.5, 100.5, 1000.5, 200.5, 2000.5, 3.5, 30.5, 4.5, 40.5, 300.5, 3000.5, 400.5, 4000.5]
    near(np.load(TCONV_REF_GOLDEN)["kat_y"], exp)


def test_same_padding_rules():  # kernels/padding.h:23-82; SURVEY Appendix A closed forms
    assert po.conv_out_size(256, 3, 2, 1, po.PAD_SAME) == (128, 0)   # even, k3 s2: (0 before, 1 after)
    assert po.conv_out_size(257, 3, 2, 1, po.PAD_SAME) == (129, 1)   # odd: (1, 1)
    assert po.conv_out_size(32, 5, 2, 1, po.PAD_SAME) == (16, 1)     # k5 s2 even: (1, 2)
    assert po.conv_out_size(33, 3, 1, 4, po.PAD_SAME) == (33, 4)     # dilation 4
    assert po.conv_out_size(9, 3, 1, 3, po.PAD_VALID) == (3, 0)
