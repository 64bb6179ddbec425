"""C-ABI surface checks that need no GPU: the library loads, exports every symbol include/orbx.h declares, and fails
loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import hashlib
import os
import re

import numpy as np
import pytest

from orb_slam2_ros2_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "orbx.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(orbx_[a-z_0-9]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    L = api.load_library()
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), f"liborbx.so does not export {s}"
    assert sorted(api.EXPORTS) == syms


def test_status_strings():
    L = api.load_library()
    assert L.orbx_status_string(0) == b"ok"
    assert b"ImageSizeError" in L.orbx_status_string(api.ORBX_ERR_IMAGE_SIZE)
    assert b"FileNotOpenError" in L.orbx_status_string(api.ORBX_ERR_FILE_NOT_OPEN)


def test_keypoint_layout_matches_cv_keypoint():
    assert api.KP_DTYPE.itemsize == 28
    assert [api.KP_DTYPE.fields[n][1] for n in ("x", "y", "size", "angle", "response", "octave", "class_id")] == [0, 4, 8, 12, 16, 20, 24]


def test_template_loader(template_path, oracle):
    pat = api.load_brief_template(template_path)
    assert pat.shape == (256, 4) and np.array_equal(pat, oracle.default_pattern())
    with pytest.raises(api.FileNotOpenError):
        api.load_brief_template("/nonexistent/brief_template.txt")


# SHA-256 of the reference's config/brief_template.txt as load_brief_template parses it (256 x 4 float32); the reference
# sources are not part of this repository.  The table is OpenCV's bit_pattern_31_.
REF_TEMPLATE_SHA256 = "90daff40faf42ee5c044e5f7f0578a0a73787af9dbd4a68f83d967c7aa41310e"


def test_builtin_pattern_equals_reference_template(oracle):
    pat = oracle.default_pattern()
    assert pat.dtype == np.float32 and pat.shape == (256, 4)
    assert hashlib.sha256(pat.tobytes()).hexdigest() == REF_TEMPLATE_SHA256
    assert pat[0].tolist() == [8, -3, 9, 5] and pat[-1].tolist() == [-1, -6, 0, -11]


def test_invalid_config_rejected():
    L = api.load_library()
    cfg = api.OrbxConfig()
    L.orbx_default_config(C.byref(cfg))
    assert (cfg.width, cfg.height, cfg.n_features, cfg.n_levels) == (1241, 376, 2000, 8)
    h = C.c_void_p()
    cfg.scale_factor = 1.0
    assert L.orbx_create(C.byref(cfg), C.byref(h)) == api.ORBX_ERR_INVALID_ARG
    assert L.orbx_create(None, C.byref(h)) == api.ORBX_ERR_INVALID_ARG


def test_no_cpu_fallback_without_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(api.OrbxCudaError):
        api.Context(1241, 376)


def test_header_is_valid_c99_and_links_against_the_library(tmp_path):
    """include/orbx.h is a plain C header (the boundary a cgo / JNI / ctypes binding would consume): compile a C99 client
    with -pedantic and link it against liborbx.so; running it without a GPU must fail loudly with ORBX_ERR_NO_DEVICE."""
    import subprocess

    api.load_library()
    src = tmp_path / "client.c"
    src.write_text(
        '#include <stdio.h>\n#include "orbx.h"\n'
        "int main(void) {\n"
        "  orbx_config cfg; orbx_ctx *ctx = 0; orbx_default_config(&cfg);\n"
        "  cfg.width = 320; cfg.height = 240; cfg.max_batch = 1;\n"
        "  int rc = orbx_create(&cfg, &ctx);\n"
        '  printf("%d %s %d\\n", rc, orbx_status_string(rc), (int)sizeof(orbx_area_query));\n'
        "  if (ctx) orbx_destroy(ctx);\n"
        "  return 0;\n}\n")
    exe = tmp_path / "client"
    libdir = os.path.join(ROOT, "orb_slam2_ros2_b200")
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                        "-L", libdir, "-lorbx", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()
    import torch

    assert int(out[-1]) == 24
    if not torch.cuda.is_available():
        assert int(out[0]) == api.ORBX_ERR_NO_DEVICE
    else:
        assert int(out[0]) == 0
