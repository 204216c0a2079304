"""Host-side checks of the denoiser's interface and of its NumPy restatement (tests/denoise_ref.py); no GPU."""
import os
import re

import ctypes as C
import numpy as np

import denoise_ref as R
from learn_path_tracing_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_denoise_params_struct_matches_the_header():
    src = open(os.path.join(ROOT, "include", "pt_api.h")).read()
    m = re.search(r"typedef struct PtDenoiseParams \{(.*?)\} PtDenoiseParams; /\* (\d+) bytes \*/", src, re.S)
    assert m, "PtDenoiseParams not found in pt_api.h"
    assert C.sizeof(_lib.PtDenoiseParams) == int(m.group(2)) == 32
    fields = re.findall(r"\b(int32_t|float)\s+([^;]+);", m.group(1))
    names = [n.strip() for _, decl in fields for n in decl.split(",")]
    assert names == [f for f, _ in _lib.PtDenoiseParams._fields_]
    for sym in ("pt_render_features", "pt_denoise"):
        assert re.search(r"\bint %s\(" % sym, src) and sym in _lib.API_SYMBOLS


def _synthetic(W, H, spp, seed=0):
    rng = np.random.default_rng(seed)
    n = W * H
    s = np.zeros((n, 4), np.float32)
    s[:, :3] = rng.uniform(0.0, 2.0, (n, 3)) * spp
    q = np.zeros_like(s)
    q[:, :3] = s[:, :3] ** 2 / spp + rng.uniform(0.0, 1.0, (n, 3)) * spp
    f = np.zeros((2, n, 4), np.float32)
    nrm = rng.normal(size=(n, 3))
    f[0, :, :3] = nrm * spp
    f[0, :, 3] = rng.uniform(1, 3, n) * spp
    f[1, :, :3] = rng.uniform(0.05, 1.0, (n, 3)) * spp
    f[1, :, 3] = spp
    return s, q, f


def test_reference_zero_iterations_is_the_mean():
    W, H, N = 7, 5, 8
    s, q, f = _synthetic(W, H, N)
    assert np.array_equal(R.denoise(s, q, f, W, H, N, iterations=0), s[:, :3].astype(np.float64) / N)


def test_reference_keeps_a_constant_image():
    W, H, N = 9, 6, 4
    _, _, f = _synthetic(W, H, N, 1)
    s = np.zeros((W * H, 4), np.float32)
    s[:, :3] = (0.25, 0.5, 0.75)
    s[:, :3] *= N
    q = np.zeros_like(s)
    q[:, :3] = s[:, :3] ** 2 / N
    out = R.denoise(s, q, f, W, H, N, iterations=4)
    assert np.allclose(out, s[:, :3] / N, rtol=1e-12, atol=0)


def test_reference_guides_of_sky_and_one_pixel_axes():
    f = np.zeros((2, 3, 4), np.float32)       # a 1 x 3 image: no hit anywhere
    z, gx, gy, n, has = R.guides(f, 1, 3)
    assert not has.any() and (n == 0).all() and (gx == 0).all() and (gy == 0).all() and (z == 0).all()
