"""The C++ facade's setDecodeScale: tests/cpp/scaled_main.cpp decodes what compress() wrote at 1/2, 1/4 and 1/8 on a
colour (422) and a gray (400) runner, compiled with g++ against the cv::Mat shim as tests/test_gpu_facade_cpp.py builds
demo_main.cpp; the pixels must equal the reduced-size CPU checker's."""
import os
import subprocess

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp):
    exe = os.path.join(tmp, "scaled")
    libdir = os.path.join(ROOT, "nvjpeg_imagecompressor_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-DB2J_USE_CV_SHIM", "-o", exe, os.path.join(ROOT, "tests/cpp/scaled_main.cpp"),
                           os.path.join(ROOT, "facade/ImageCompressor.cpp"), "-L" + libdir, "-lb2jpeg", "-Wl,-rpath," + libdir])
    return exe


def test_scaled_facade_compiles_without_gpu(tmp_path):
    from nvjpeg_imagecompressor_b200 import _native as N
    N.build()
    assert os.path.exists(_build(str(tmp_path)))


@pytest.mark.gpu
def test_cpp_scaled_decode(tmp_path, oracle):
    from nvjpeg_imagecompressor_b200 import _native as N
    N.lib()
    exe = _build(str(tmp_path))
    W, H = 641, 359
    bgr = oracle.synth(W, H, 1, 8)
    gray = np.ascontiguousarray(oracle.synth(W, H, 2, 8)[..., 1])
    bgr.tofile(tmp_path / "in.bgr")
    gray.tofile(tmp_path / "in.gray")
    r = subprocess.run([exe, str(W), str(H), str(tmp_path / "in.bgr"), str(tmp_path / "in.gray"), str(tmp_path)],
                       capture_output=True, text=True, env=dict(os.environ, B2J_QUIET="1"))
    assert r.returncode == 0, r.stdout + r.stderr
    for name in ("bgr", "gray"):
        jpg = np.fromfile(tmp_path / f"{name}.jpeg", np.uint8)
        for d in O.SCALES:
            want = O.decode_scaled(jpg, d, gray=name == "gray")
            got = np.fromfile(tmp_path / f"{name}.d{d}.raw", np.uint8).reshape(want.shape)
            assert np.array_equal(got, want), (name, d)
