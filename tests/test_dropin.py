"""The reference-facing C++ layer (SURVEY.md §8b): include/lib/libbackscrub.h + include/background.h, defined by
backscrub_b200/shim/*.cc over the C ABI, exercised by tests/cpp/dropin_test.cc — a translation unit with the
reference's own include lines and call shapes (app/deepseg.cc:24-25,203,246,269,351,596,649).  The image has no
OpenCV C++ headers, so a minimal cv::Mat / cv::VideoCapture / cv::imread stand-in (tests/cpp/stub) is used.

* `-m "not gpu"`: builds against this repo's headers and checks that it defines every symbol the program needs when
  compiled against the reference's own headers (include order of the reference's CMakeLists.txt:72; the list is
  stored under tests/golden); links the product library; on the GPU-less box the program must fail loudly
  (no CPU path); the same program linked with the kernel-logic emulator build runs the whole flow and is compared
  with the oracle.
* `-m gpu`: the whole flow on the real library."""
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from tests.conftest import ROOT, model_path

CPP = os.path.join(ROOT, "tests", "cpp")


def _build(target):
    lib = os.path.join(ROOT, "backscrub_b200", "libbackscrub_b200.so")
    if not os.path.exists(lib):
        import __graft_entry__
        __graft_entry__.build()
    if target == "dropin_test_emu":
        from tests.emu.emu_lib import emu
        emu()
    subprocess.check_call(["make", "-C", CPP, "-s", target])
    return os.path.join(CPP, target)


def _write_still(path, img):
    with open(path, "wb") as f:
        f.write(b"RAWI" + struct.pack("<ii", img.shape[1], img.shape[0]) + img.tobytes())


def _write_video(path, frames, fps, seekable):
    with open(path, "wb") as f:
        f.write(b"RAWV" + struct.pack("<iiiii", frames.shape[2], frames.shape[1], frames.shape[0], fps, int(seekable)) + frames.tobytes())


def _run_flow(exe, tmp_path, key, W, H, n, background, timeout=900):
    from tests import synth
    frames = np.stack([synth.frame(W, H, t=t) for t in range(max(n, 1))])[:n]
    fin = tmp_path / "frames.bgr"
    frames.tofile(fin)
    prefix = str(tmp_path / "out")
    r = subprocess.run([exe, model_path(key), str(W), str(H), str(fin), str(n), str(background), prefix],
                       capture_output=True, text=True, timeout=timeout)
    return r, frames, prefix


def _check_flow(r, frames, prefix, key, W, H, n, bg_first):
    from oracle import pyoracle as po
    assert r.returncode == 0, r.stdout + r.stderr
    assert "load_background: ok" in r.stdout and "load_background(missing): nullptr" in r.stdout
    assert "grab_background(nullptr) = -1" in r.stdout
    # onprep, oninfer, onmask in order, once per processed frame (n frames + the oversize one; the short frame is rejected)
    assert "callbacks: " + "PIM" * (n + 1) in r.stdout
    assert "short frame -> 0" in r.stdout
    assert f"oversize frame -> 1 mask {W}x{H}" in r.stdout
    masks = np.fromfile(prefix + ".masks", np.uint8).reshape(n, H, W)
    o = po.MaskGen(model_path(key), W, H)
    for t in range(n):
        assert np.array_equal(masks[t], o.process(frames[t])), f"mask {t} differs from the oracle"
    bg = np.fromfile(prefix + ".bg", np.uint8).reshape(H, W, 3)
    assert np.array_equal(bg, po.resize_linear_u8(bg_first, W, H)), "grab_background differs from cv::resize (oracle)"


def test_links_against_the_reference_headers(tmp_path):
    """The reference's OWN lib/libbackscrub.h and app/background.h first on the include path (as inside the reference
    tree): the C++-linkage symbols they declare are the ones the shims define, so the program links.  The symbols that
    tests/cpp/dropin_test.cc needs when compiled that way are stored in tests/golden/reference_header_symbols.txt
    (tests/golden/make_golden.py); every one must be defined by the program built from this repo's headers and shims."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_header_symbols.txt")) as f:
        needed = f.read().split()
    demangled = subprocess.run(["c++filt"], input="\n".join(needed), capture_output=True, text=True, check=True).stdout
    for s in ["bs_maskgen_new(std::", "bs_maskgen_process(void*, cv::Mat&, cv::Mat&)", "bs_maskgen_delete(void*)", "bs_tensorflow_version()",
              "load_background(std::", "grab_background(std::shared_ptr<background_t>, int, int, cv::Mat&)",
              "grab_thumbnail(std::shared_ptr<background_t>, cv::Mat&)"]:
        assert s in demangled, s
    exe = _build("dropin_test")
    defined = set(subprocess.run(["nm", "--defined-only", exe], capture_output=True, text=True, check=True).stdout.split())
    for s in needed:
        assert s in defined, s


def test_fails_loudly_without_gpu(tmp_path):
    import backscrub_b200 as bs
    if bs.device_count() > 0:
        pytest.skip("a GPU is present")
    from tests import synth
    exe = _build("dropin_test")
    still = tmp_path / "bg.rawi"
    _write_still(still, synth.background()[:90, :160])
    r, _, _ = _run_flow(exe, tmp_path, "meet_lite", 320, 240, 0, still, timeout=120)
    assert r.returncode == 3 and "returned nullptr" in r.stdout and "no CUDA device" in r.stderr
    assert "load_background: ok" in r.stdout          # decoding / provider set-up needs no GPU


def test_flow_on_the_emulator_still_background(tmp_path):
    from tests import synth
    exe = _build("dropin_test_emu")
    W, H, n = 320, 240, 2
    img = np.ascontiguousarray(synth.background()[:180, :320])
    still = tmp_path / "bg.rawi"
    _write_still(still, img)
    r, frames, prefix = _run_flow(exe, tmp_path, "meet_lite", W, H, n, still)
    _check_flow(r, frames, prefix, "meet_lite", W, H, n, img)
    assert "grab_background frame=1" in r.stdout                      # still image: frame number 1, always
    assert re.search(r"frames:( 1){12}", r.stdout)


def test_flow_on_the_emulator_looping_video(tmp_path):
    from tests import synth
    exe = _build("dropin_test_emu")
    W, H, n = 320, 240, 1
    base = np.ascontiguousarray(synth.background()[:90, :160])
    vid = np.stack([np.roll(base, 8 * i, axis=1) for i in range(6)])
    path = tmp_path / "bg.rawv"
    _write_video(path, vid, fps=40, seekable=True)
    r, frames, prefix = _run_flow(exe, tmp_path, "meet_lite", W, H, n, path)
    assert r.returncode == 0, r.stdout + r.stderr
    nums = [int(x) for x in re.search(r"frames:((?: -?\d+)+)", r.stdout).group(1).split()]
    assert all(0 <= x <= 6 for x in nums)
    # real-time pacing: 40 fps sampled every >= 50 ms => the counter moves by about 2 per sample, never stalls, and
    # wraps to 0 at the end of the 6-frame loop (app/background.cc:93-96)
    wraps = sum(1 for a, b in zip(nums, nums[1:]) if b < a)
    assert wraps >= 1 and len(set(nums)) >= 3, nums
    # debug = 2 => the reader publishes 160-pixel-wide thumbnails
    assert "grab_thumbnail rc=0 size=160x90" in r.stdout


def test_video_that_cannot_rewind_stops_at_its_last_frame(tmp_path):
    from tests import synth
    exe = _build("dropin_test_emu")
    base = np.ascontiguousarray(synth.background()[:90, :160])
    vid = np.stack([np.roll(base, 8 * i, axis=1) for i in range(4)])
    path = tmp_path / "bg.rawv"
    _write_video(path, vid, fps=200, seekable=False)
    r, _, _ = _run_flow(exe, tmp_path, "meet_lite", 320, 240, 1, path)
    assert r.returncode == 0, r.stdout + r.stderr
    nums = [int(x) for x in re.search(r"frames:((?: -?\d+)+)", r.stdout).group(1).split()]
    # the probe consumed two frames and could not rewind: counting starts at 2 (app/background.cc:146-149), two more
    # frames arrive, then the reader stops and callers keep getting the last frame
    assert nums[-1] == 4 and nums == sorted(nums), nums
    assert "not resettable" in r.stderr


@pytest.mark.gpu
def test_flow_on_the_gpu(tmp_path):
    from tests import synth
    exe = _build("dropin_test")
    W, H, n = 640, 480, 3
    img = np.ascontiguousarray(synth.background())
    still = tmp_path / "bg.rawi"
    _write_still(still, img)
    r, frames, prefix = _run_flow(exe, tmp_path, "mlkit", W, H, n, still)
    _check_flow(r, frames, prefix, "mlkit", W, H, n, img)
    assert "grab_background frame=1" in r.stdout
