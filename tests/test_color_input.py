"""Colour input without a device: the conversion rule against cv2.cvtColor, and the C-ABI, ctypes and C++ shim surface of
orbx_set_input_format."""
import ctypes as C
import os
import re
import subprocess

import cv2
import numpy as np
import pytest

from orb_slam2_ros2_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the weights of R, G, B in cv::cvtColor's 8-bit RGB -> gray (15 fractional bits), as the level-0 pyramid kernel applies them
W_R, W_G, W_B = 9798, 19235, 3735
CODES = {api.FORMAT_RGB8: (cv2.COLOR_RGB2GRAY, (0, 1, 2)), api.FORMAT_BGR8: (cv2.COLOR_BGR2GRAY, (2, 1, 0)),
         api.FORMAT_RGBA8: (cv2.COLOR_RGBA2GRAY, (0, 1, 2)), api.FORMAT_BGRA8: (cv2.COLOR_BGRA2GRAY, (2, 1, 0))}


def rule(img: np.ndarray, fmt: int) -> np.ndarray:
    r, g, b = (img[..., i].astype(np.uint32) for i in CODES[fmt][1])
    return ((W_R * r + W_G * g + W_B * b + 16384) >> 15).astype(np.uint8)


def _all_triples(bpp: int) -> np.ndarray:
    """every (c0, c1, c2) byte triple once, as one 4096 x 4096 image (cv2's vector path); alpha = the low byte of c0 + c2"""
    v = np.arange(1 << 24, dtype=np.uint32)
    ch = [(v >> 16) & 255, (v >> 8) & 255, v & 255]
    if bpp == 4:
        ch.append((ch[0] + ch[2]) & 255)
    return np.stack(ch, -1).astype(np.uint8).reshape(4096, 4096, bpp)


@pytest.mark.parametrize("fmt", list(CODES), ids=["rgb8", "bgr8", "rgba8", "bgra8"])
def test_rule_equals_cvtcolor_on_every_triple(fmt):
    cv2.setNumThreads(1)
    img = _all_triples(api.FORMAT_BPP[fmt])
    assert np.array_equal(rule(img, fmt), cv2.cvtColor(img, CODES[fmt][0]))
    # odd widths take cv2's scalar tails
    rng = np.random.default_rng(fmt)
    for w in range(1, 70):
        small = rng.integers(0, 256, (3, w, api.FORMAT_BPP[fmt]), dtype=np.uint8)
        assert np.array_equal(rule(small, fmt), cv2.cvtColor(small, CODES[fmt][0])), w


def test_older_rules_differ():
    """the 14-bit (4899 / 9617 / 1868) rule is not the one cv2 applies: the weights must come from the 15-bit table"""
    img = _all_triples(3)
    r, g, b = (img[..., i].astype(np.uint32) for i in range(3))
    old = ((4899 * r + 9617 * g + 1868 * b + 8192) >> 14).astype(np.uint8)
    assert (old != cv2.cvtColor(img, cv2.COLOR_RGB2GRAY)).sum() > 10000


def test_header_declares_the_formats():
    txt = open(os.path.join(ROOT, "include", "orbx.h")).read()
    consts = dict((k, int(v)) for k, v in re.findall(r"#define ORBX_FORMAT_([A-Z0-9]+) (\d+)", txt))
    assert consts == {"GRAY8": api.FORMAT_GRAY8, "RGB8": api.FORMAT_RGB8, "BGR8": api.FORMAT_BGR8, "RGBA8": api.FORMAT_RGBA8, "BGRA8": api.FORMAT_BGRA8}
    assert consts["GRAY8"] == 0  # the default, today's behaviour
    assert re.search(r"int orbx_set_input_format\(orbx_ctx \*ctx, int format\);", txt)
    assert api.FORMAT_BPP == {0: 1, 1: 3, 2: 3, 3: 4, 4: 4}


def test_ctypes_mirror():
    L = api.load_library()
    assert "orbx_set_input_format" in api.EXPORTS
    assert L.orbx_set_input_format.argtypes == [C.c_void_p, C.c_int]
    assert L.orbx_set_input_format(None, api.FORMAT_BGR8) == api.ORBX_ERR_INVALID_ARG
    assert "set_input_format" in vars(api.Context)
    assert api.Camera().rgb is False and api.Camera(rgb=True).rgb is True


def test_image_format_and_shapes():
    assert api.image_format(np.zeros((4, 5), np.uint8)) == api.FORMAT_GRAY8
    assert api.image_format(np.zeros((4, 5, 3), np.uint8)) == api.FORMAT_BGR8
    assert api.image_format(np.zeros((4, 5, 3), np.uint8), rgb=True) == api.FORMAT_RGB8
    assert api.image_format(np.zeros((4, 5, 4), np.uint8)) == api.FORMAT_BGRA8
    assert api.image_format(np.zeros((4, 5, 4), np.uint8), rgb=True) == api.FORMAT_RGBA8
    for bad in ((4, 5, 2), (4, 5, 1, 3), (4,)):
        with pytest.raises(ValueError):
            api.image_format(np.zeros(bad, np.uint8))
    img = np.arange(4 * 10 * 3, dtype=np.uint8).reshape(4, 10, 3)
    assert api._as_image(img, 4, 10, 3) is img
    sub = img[:, ::2]  # pixels not packed: copied
    assert api._as_image(sub, 4, 5, 3).strides == (15, 3, 1)
    rows = np.zeros((4, 40), np.uint8)[:, :30].reshape(4, 10, 3)  # padded rows keep their stride
    assert api._as_image(rows, 4, 10, 3).strides == (40, 3, 1)
    with pytest.raises(ValueError):
        api._as_image(img, 4, 10, 1)


def test_shim_color_driver_compiles_and_refuses_other_types(tmp_path):
    """the shim takes CV_8UC3 / CV_8UC4 against the repository's cv:: stand-in and refuses other types before any device
    work; tests/cpp/shim_color_main.cpp drives it"""
    api.load_library()
    out = str(tmp_path / "shim_color_main")
    libdir = os.path.join(ROOT, "orb_slam2_ros2_b200")
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle", "stub"),
           os.path.join(ROOT, "tests", "cpp", "shim_color_main.cpp"), "-o", out, "-L", libdir, "-lorbx", f"-Wl,-rpath,{libdir}", "-pthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([out, "types"], capture_output=True, text=True)
    assert r.returncode == 0 and "types ok=2" in r.stdout
