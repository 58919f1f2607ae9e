"""The C++ facade with sampling 400 (gray): tests/cpp/gray_main.cpp runs the reference demo's call order on CV_8UC1
images, compiled with g++ against the cv::Mat shim as tests/test_gpu_facade_cpp.py builds demo_main.cpp."""
import os
import subprocess

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp):
    exe = os.path.join(tmp, "gray")
    libdir = os.path.join(ROOT, "nvjpeg_imagecompressor_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-DB2J_USE_CV_SHIM", "-o", exe, os.path.join(ROOT, "tests/cpp/gray_main.cpp"),
                           os.path.join(ROOT, "facade/ImageCompressor.cpp"), "-L" + libdir, "-lb2jpeg", "-Wl,-rpath," + libdir])
    return exe


def test_gray_facade_compiles_without_gpu(tmp_path):
    from nvjpeg_imagecompressor_b200 import _native as N
    N.build()
    assert os.path.exists(_build(str(tmp_path)))


@pytest.mark.gpu
def test_cpp_gray_demo_sequence(tmp_path, oracle):
    from nvjpeg_imagecompressor_b200 import _native as N
    N.lib()
    exe = _build(str(tmp_path))
    W, H = 641, 359
    a = np.ascontiguousarray(oracle.synth(W, H, 1, 8)[..., 1])
    b = np.ascontiguousarray(oracle.synth(W, H, 2, 8)[..., 1])
    a.tofile(tmp_path / "a.gray")
    b.tofile(tmp_path / "b.gray")
    r = subprocess.run([exe, str(W), str(H), str(tmp_path / "a.gray"), str(tmp_path / "b.gray"), str(tmp_path)],
                       capture_output=True, text=True, env=dict(os.environ, B2J_MULTI_DEVICES="0,0"))
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("[INFO] Successful.") == 4
    for name, img in (("1", a), ("2", b)):
        jpg = np.fromfile(tmp_path / f"{name}.jpeg", np.uint8)
        want = O.encode_gray(img, 95, 1)
        assert np.array_equal(jpg, want)
        dec = np.fromfile(tmp_path / f"{name}.dec.gray", np.uint8).reshape(H, W)
        assert np.array_equal(dec, O.decode_gray(want))
