"""Generate the committed golden fixtures (needs cv2 4.13, and a checkout of the original
backscrub tree: oracle/_ref built from it for tconv_ref_golden.npz, its path in
BACKSCRUB_REFERENCE for reference_header_symbols.txt):

  image_ops_golden.npz   cv2 outputs for small seeded inputs (resize/blur/RGB2YUV/
                         bilateral/convertTo) — pins the oracle's image primitives on
                         boxes whose cv2 build may differ.
  tconv_ref_golden.npz   outputs of the REFERENCE's lib/transpose_conv_bias.cc
                         (oracle/_ref) for seeded inputs, including the cases and the
                         known answer of tests/test_oracle_nn.py.
  model_torch_golden.npz torch-fp64 evaluation of each .tflite on one synthetic input:
                         decision bitmap + output statistics.
  pipeline_golden.npz    oracle regression outputs (mask bits, composite checksums).
  reference_header_symbols.txt
                         mangled names of the C++-linkage functions that tests/cpp/dropin_test.cc
                         needs when compiled against the REFERENCE's own lib/libbackscrub.h and
                         app/background.h (include order of its CMakeLists.txt:72).

    python tests/golden/make_golden.py
"""
import os
import subprocess
import sys
import tempfile

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402
from tests import synth, torch_graph  # noqa: E402
from tests.conftest import MODELS, model_path  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
TCONV_CASES = [(8, 8, 16, 1), (5, 7, 16, 2), (3, 3, 4, 3)]


def image_ops():
    rng = np.random.default_rng(2024)
    d = {}
    for i, (sw, sh, dw, dh, cn) in enumerate([(48, 36, 25, 19, 3), (25, 19, 64, 48, 1), (64, 64, 32, 32, 3), (31, 17, 77, 40, 3)]):
        src = rng.integers(0, 256, (sh, sw, cn) if cn > 1 else (sh, sw), dtype=np.uint8)
        d[f"resize{i}_src"] = src
        d[f"resize{i}_dst"] = cv2.resize(src, (dw, dh))
    src = rng.integers(0, 256, (23, 31), dtype=np.uint8)
    d["blur_src"], d["blur_dst"] = src, cv2.blur(src, (5, 5))
    src = rng.integers(0, 256, (16, 24, 3), dtype=np.uint8)
    d["yuv_src"], d["yuv_dst"] = src, cv2.cvtColor(src, cv2.COLOR_RGB2YUV)
    src = cv2.resize(cv2.imread(os.path.join(ROOT, "backgrounds", "screenshot.jpg"))[:, :640], (64, 48))
    cv2.ipp.setUseIPP(False)
    d["bilateral_src"], d["bilateral_dst"] = src, cv2.bilateralFilter(src, 5, 100.0, 100.0)
    cv2.ipp.setUseIPP(True)
    g_in = cv2.GMat()
    for name, (a, b) in {"unit": (float(np.float32(1 / 255.0)), 0.0), "deeplab": (float(np.float32(1 / 127.5)), -1.0)}.items():
        comp = cv2.GComputation(g_in, cv2.gapi.convertTo(g_in, cv2.CV_32F, a, b))
        d[f"convert_{name}"] = comp.apply(cv2.gin(np.arange(256, dtype=np.uint8).reshape(16, 16)))
    # `-p bgblur:k` (app/deepseg.cc:657-658) and cv::flip (:667-673)
    for k, (w, h) in {25: (56, 40), 7: (30, 20), 51: (40, 24)}.items():
        src = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        d[f"gauss{k}_src"], d[f"gauss{k}_dst"] = src, cv2.GaussianBlur(src, (k, k), 0)
    d["gauss_taps25"] = np.rint(cv2.getGaussianKernel(25, 0).ravel() * 256)   # informative only (no error diffusion)
    src = rng.integers(0, 256, (9, 14, 3), dtype=np.uint8)
    d["flip_src"] = src
    for code in (1, 0, -1):
        d[f"flip_{code}"] = cv2.flip(src, code)
    np.savez_compressed(os.path.join(OUT, "image_ops_golden.npz"), **d)


def tconv_ref():
    if po.ref_tconv_lib() is None:
        print("oracle/_ref missing; skipping tconv_ref_golden")
        return
    d = {}
    for i, (ih, iw, ic, oc) in enumerate([(8, 8, 16, 1), (6, 10, 16, 2), (5, 7, 8, 3)]):
        rng = np.random.default_rng(100 + i)
        x = rng.standard_normal((ih, iw, ic)).astype(np.float32)
        w = rng.standard_normal((oc, 2, 2, ic)).astype(np.float32)
        b = rng.standard_normal(oc).astype(np.float32)
        d[f"x{i}"], d[f"w{i}"], d[f"b{i}"], d[f"y{i}"] = x, w, b, po.ref_tconv_bias(x, w, b)
    # the cases of tests/test_oracle_nn.py, which compare the oracle with these stored outputs
    for ih, iw, ic, oc in TCONV_CASES:
        rng = np.random.default_rng(ih * 100 + oc)
        x = rng.standard_normal((ih, iw, ic)).astype(np.float32)
        w = rng.standard_normal((oc, 2, 2, ic)).astype(np.float32)
        b = rng.standard_normal(oc).astype(np.float32)
        key = "case_%dx%dx%dx%d" % (ih, iw, ic, oc)
        d[key + "_x"], d[key + "_w"], d[key + "_b"], d[key + "_y"] = x, w, b, po.ref_tconv_bias(x, w, b)
    x = np.array([1, 2, 3, 4], np.float32).reshape(2, 2, 1)
    w = np.array([1, 10, 100, 1000], np.float32).reshape(1, 2, 2, 1)
    d["kat_y"] = po.ref_tconv_bias(x, w, [0.5])
    np.savez_compressed(os.path.join(OUT, "tconv_ref_golden.npz"), **d)


def model_torch():
    d = {}
    for key in MODELS:
        g = po.MaskGen(model_path(key), 640, 480)
        g.process(synth.frame(640, 480, t=3))
        x = g.input_f32
        out = torch_graph.run(model_path(key), x)
        if key == "deeplab":
            dec = out.argmax(-1) == 15
            margin = np.sort(out, -1)[..., -1] - np.sort(out, -1)[..., -2]
        elif key.startswith("meet"):
            dec = out[..., 0] < out[..., 1]
            margin = np.abs(out[..., 0] - out[..., 1])
        else:
            dec = out[..., 0] > 0.65
            margin = np.abs(out[..., 0] - 0.65)
        d[f"{key}_decision"] = np.packbits(dec)
        d[f"{key}_margin_small"] = np.packbits(margin < 1e-3)   # pixels whose decision is numerically fragile
        d[f"{key}_out_f16"] = out.astype(np.float16) if out.size < 300000 else out[::4, ::4].astype(np.float16)
    np.savez_compressed(os.path.join(OUT, "model_torch_golden.npz"), **d)


def pipeline():
    d = {"n_frames": 4}
    for key in ("mlkit", "meet_full"):
        g = po.MaskGen(model_path(key), 640, 480)
        for t in range(4):
            out, yuyv, mask = g.composite(synth.frame(640, 480, t=t), synth.background())
        d[f"{key}_maskbits"] = np.packbits(mask < 128)
        d[f"{key}_outsum"] = out.astype(np.int64).sum()
        d[f"{key}_yuyvsum"] = yuyv.astype(np.int64).sum()
    np.savez_compressed(os.path.join(OUT, "pipeline_golden.npz"), **d)


def model_cv2dnn():
    """Whole-model output of the MLKit graph computed by OpenCV's own dnn module (cv2.dnn.readNetFromTFLite): a
    third-party implementation of the same .tflite file.  Stored as float16-rounded probabilities plus the decision
    bitmap (the comparison tolerance is 1e-3 on the rounded values, exact on the decisions away from the threshold)."""
    g = po.MaskGen(model_path("mlkit"), 640, 480)
    g.process(synth.frame(640, 480, t=3))
    x = g.input_f32
    net = cv2.dnn.readNetFromTFLite(model_path("mlkit"))
    net.setInput(np.ascontiguousarray(x.transpose(2, 0, 1)[None]))
    out = net.forward()[0, 0]
    np.savez_compressed(os.path.join(OUT, "model_cv2dnn_golden.npz"), mlkit_prob_f16=out.astype(np.float16),
                        mlkit_decision=np.packbits(out > 0.65), mlkit_margin_ok=np.packbits(np.abs(out - 0.65) > 1e-3))


def reference_header_symbols():
    ref = os.environ.get("BACKSCRUB_REFERENCE")
    if not ref:
        print("BACKSCRUB_REFERENCE not set; skipping reference_header_symbols")
        return
    cpp = os.path.join(ROOT, "tests", "cpp")
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "dropin_test_ref.o")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-c", "-I" + os.path.join(cpp, "stub"), "-I" + ref, "-I" + os.path.join(ref, "app"),
                               "-I" + os.path.join(ROOT, "include"), "-o", obj, os.path.join(cpp, "dropin_test.cc")])
        undef = [ln.split()[-1] for ln in subprocess.run(["nm", "-u", obj], capture_output=True, text=True, check=True).stdout.splitlines()]
    names = subprocess.run(["c++filt"], input="\n".join(undef), capture_output=True, text=True, check=True).stdout.splitlines()
    keep = sorted(m for m, d in zip(undef, names) if d.startswith(("bs_", "load_background(", "grab_background(", "grab_thumbnail(")))
    with open(os.path.join(OUT, "reference_header_symbols.txt"), "w") as f:
        f.write("\n".join(keep) + "\n")


if __name__ == "__main__":
    image_ops(); tconv_ref(); model_torch(); pipeline(); model_cv2dnn(); reference_header_symbols()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
