"""Cross-check against the outputs of the REFERENCE'S OWN CUDA kernels.

The reference's kernels are kornia-rs' CUDA source strings, NVRTC-compiled with its options (compute_100, --fmad=false)
and launched with its launch geometry (baseline/extract_ref_kernels.py, baseline/ref_gpu.py).  For every case below
tests/golden/ref_kernels.json keeps a SHA-256 digest of the output those kernels produce on the case's inputs, and our
kernels must produce the SAME BITS (in f32, +0.0 and -0.0 count as equal) — parity anchored on outputs of the reference
itself, next to the oracle-based parity of test_gpu_parity.py.  tests/golden/make_ref_kernel_digests.py records the
digests; how they were obtained is stated in the JSON file.
"""
import functools
import hashlib
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.json")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def cu(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def digest(t: torch.Tensor) -> str:
    """dtype, shape and SHA-256 of the output's bytes, with -0.0 written as +0.0 in f32 outputs."""
    a = t.cpu().numpy()
    if a.dtype == np.float32:
        a = np.where(a == 0, np.float32(0), a)
    return f"{a.dtype}{list(a.shape)}:" + hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@functools.cache
def reference_digests() -> dict:
    with open(GOLDEN) as f:
        return json.load(f)["digests"]


def same_bits(key: str, got: torch.Tensor, what: str = ""):
    want = reference_digests().get(key)
    assert want is not None, f"{key}: no reference output recorded in {GOLDEN}"
    assert digest(got) == want, f"{what or key}: output differs from the reference kernel's ({digest(got)} != {want})"


@pytest.mark.parametrize("sw,sh,dw,dh", [(384, 216, 128, 72), (640, 360, 320, 180), (640, 360, 213, 120), (129, 97, 64, 48), (64, 48, 129, 97)])
def test_resize_bilinear_matches_reference_kernel(kb, oracle, dev, sw, sh, dw, dh):
    n = 2
    src = cu(oracle.pattern_f32(n * sw * sh * 3).reshape(n, sh, sw, 3), dev)
    got = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), 3, torch.float32, dev, batch=n)
    kb.imgproc.resize(kb.Image(src), got, kb.InterpolationMode.Bilinear)
    same_bits(f"resize {sw}x{sh}->{dw}x{dh}", got.data)


H_CASES = [((129, 97), [1.03, 0.05, -3.0, -0.02, 0.97, 4.0, 2.0 / (97 * 129), 1.5 / (129 * 97), 1.0]),
           ((320, 240), [0.9, 0.15, 10.0, -0.1, 1.1, -6.0, 0.0, 0.0, 1.0]),
           ((640, 360), [1.02, 0.03, -7.0, -0.03, 1.01, 4.0, 1.2e-5, 7.0e-6, 1.0]),
           ((256, 192), [0.8, 0.45, -20.0, -0.5, 0.85, 60.0, 1.0e-4, -6.0e-5, 1.0])]


@pytest.mark.parametrize("size,h", H_CASES)
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
def test_warp_perspective_matches_reference_kernel(kb, oracle, dev, size, h, interp):
    sw, sh = size
    src = cu(oracle.pattern_f32(sw * sh * 3).reshape(1, sh, sw, 3), dev)
    got = kb.Image.from_size_val(kb.ImageSize(sw, sh), 3.0, 3, torch.float32, dev)
    kb.imgproc.warp_perspective(kb.Image(src[0]), got, h, kb.InterpolationMode.Bilinear if interp == "bilinear" else kb.InterpolationMode.Nearest)
    same_bits(f"warp_perspective {interp} {size}", got.data, f"warp_perspective {interp} {size} ({kb._lib.last_kernel()})")


@pytest.mark.parametrize("size,angle", [((128, 96), 30.0), ((256, 192), -17.5), ((97, 61), 45.0), ((640, 360), 3.0)])
@pytest.mark.parametrize("interp", ["bilinear", "nearest"])
def test_warp_affine_matches_reference_kernel(kb, oracle, dev, size, angle, interp):
    sw, sh = size
    src = cu(oracle.pattern_f32(sw * sh * 3).reshape(1, sh, sw, 3), dev)
    m = kb.imgproc.get_rotation_matrix2d((sw / 2.0, sh / 2.0), angle, 1.0)
    got = kb.Image.from_size_val(kb.ImageSize(sw, sh), 3.0, 3, torch.float32, dev)
    kb.imgproc.warp_affine(kb.Image(src[0]), got, m, kb.InterpolationMode.Bilinear if interp == "bilinear" else kb.InterpolationMode.Nearest)
    same_bits(f"warp_affine {interp} {size} {angle}", got.data, f"warp_affine {interp} {size} {angle} ({kb._lib.last_kernel()})")


@pytest.mark.parametrize("w,h,c", [(97, 61, 3), (700, 37, 3), (1100, 40, 1), (520, 33, 4)])
@pytest.mark.parametrize("k", [3, 5, 7])
def test_gaussian_blur_matches_reference_kernels(kb, oracle, dev, w, h, c, k):
    src = cu(oracle.pattern_f32(w * h * c).reshape(1, h, w, c), dev)
    got = kb.Image.zeros_cuda(kb.ImageSize(w, h), c, torch.float32, dev)
    kb.imgproc.gaussian_blur(kb.Image(src[0]), got, (k, k), (1.5, 1.5))
    same_bits(f"gaussian k={k} {w}x{h}x{c}", got.data, f"gaussian k={k} {w}x{h}x{c} ({kb._lib.last_kernel()})")


@pytest.mark.parametrize("w,h,c", [(97, 61, 3), (700, 37, 3), (1100, 40, 1)])
@pytest.mark.parametrize("ksize", [3, 5])
def test_sobel_matches_reference_kernels(kb, oracle, dev, w, h, c, ksize):
    src = cu(oracle.pattern_f32(w * h * c).reshape(1, h, w, c), dev)
    got = kb.Image.zeros_cuda(kb.ImageSize(w, h), c, torch.float32, dev)
    kb.imgproc.sobel(kb.Image(src[0]), got, ksize)
    same_bits(f"sobel k={ksize} {w}x{h}x{c}", got.data)


def test_gray_and_nv12_match_reference_kernels(kb, oracle, dev):
    w, h = 320, 180
    f = cu(oracle.pattern_f32(w * h * 3).reshape(1, h, w, 3), dev)
    got = kb.Image.zeros_cuda(kb.ImageSize(w, h), 1, torch.float32, dev)
    kb.imgproc.gray_from_rgb(kb.Image(f[0]), got)   # LEAF_SCALAR = the CUDA kernel's expression
    same_bits("gray f32", got.data)
    u = cu(oracle.pattern_u8(w * h * 3).reshape(1, h, w, 3), dev)
    got8 = kb.Image.zeros_cuda(kb.ImageSize(w, h), 1, torch.uint8, dev)
    kb.imgproc.gray_from_rgb(kb.Image(u[0]), got8)
    same_bits("gray u8", got8.data)
    n = 2
    raw = cu(oracle.pattern_u8(n * w * h * 3 // 2, 0xC0FFEE).reshape(n, w * h * 3 // 2), dev)
    gotrgb = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev, batch=n)
    kb.imgproc.rgb_from_nv12(raw, gotrgb)
    same_bits("nv12", gotrgb.data)


def raw_bytes(n, k):
    i = np.arange(n, dtype=np.int64)
    return (((i * 7 + 13) % 251) + 31 * k).astype(np.uint8)


@pytest.mark.parametrize("mode,dw,dh", [("Stretch", 192, 108), ("Letterbox", 64, 64), ("Letterbox", 100, 60), ("Stretch", 77, 41)])
@pytest.mark.parametrize("f16", [False, True])
def test_preprocess_nv12_matches_reference_kernel(kb, oracle, dev, mode, dw, dh, f16):
    """The camera preprocess has no CPU implementation: the reference's CUDA kernel IS the spec."""
    w, h, n = 192, 108, 3
    frames = [cu(raw_bytes(w * h * 3 // 2, k), dev) for k in range(n)]
    pre = (kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).mode(kb.ResizeMode[mode]).normalize(kb.Normalize.imagenet()).build_cuda())
    got = torch.zeros((n, 3, dh, dw), dtype=torch.float16 if f16 else torch.float32, device=dev)
    (pre.run_raw_batch_f16 if f16 else pre.run_raw_batch)(frames, w, h, got)
    same_bits(f"preprocess {mode} {dw}x{dh} {'f16' if f16 else 'f32'}", got)


# ── bicubic / Lanczos: the reference's own kernels are the byte-exact spec (interpolation/bicubic.rs:1-8) ──────
@pytest.mark.parametrize("sw,sh,dw,dh", [(129, 97, 64, 48), (64, 48, 129, 97), (320, 180, 213, 120), (40, 30, 40, 77)])
def test_resize_bicubic_and_lanczos_match_reference_kernels(kb, oracle, dev, sw, sh, dw, dh):
    n = 2
    src = cu(oracle.pattern_f32(n * sw * sh * 3).reshape(n, sh, sw, 3), dev)
    got = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), 3, torch.float32, dev, batch=n)
    kb.imgproc.resize(kb.Image(src), got, kb.InterpolationMode.Bicubic)
    same_bits(f"bicubic {sw}x{sh}->{dw}x{dh}", got.data)
    kb.imgproc.resize(kb.Image(src), got, kb.InterpolationMode.Lanczos)
    same_bits(f"lanczos {sw}x{sh}->{dw}x{dh}", got.data)


@pytest.mark.parametrize("interp", ["bicubic", "lanczos"])
@pytest.mark.parametrize("size,h", H_CASES)
def test_warp_perspective_hq_matches_reference_kernel(kb, oracle, dev, size, h, interp):
    sw, sh = size
    src = cu(oracle.pattern_f32(sw * sh * 3).reshape(1, sh, sw, 3), dev)
    got = kb.Image.from_size_val(kb.ImageSize(sw, sh), 3.0, 3, torch.float32, dev)
    kb.imgproc.warp_perspective(kb.Image(src[0]), got, h, kb.InterpolationMode.Bicubic if interp == "bicubic" else kb.InterpolationMode.Lanczos)
    same_bits(f"warp_perspective {interp} {size}", got.data)


@pytest.mark.parametrize("interp", ["bicubic", "lanczos"])
@pytest.mark.parametrize("size,angle", [((128, 96), 30.0), ((97, 61), 90.0), ((256, 192), -17.5)])
def test_warp_affine_hq_matches_reference_kernel(kb, oracle, dev, size, angle, interp):
    sw, sh = size
    src = cu(oracle.pattern_f32(sw * sh * 3).reshape(1, sh, sw, 3), dev)
    m = kb.imgproc.get_rotation_matrix2d((sw / 2.0, sh / 2.0), angle, 1.0)
    got = kb.Image.from_size_val(kb.ImageSize(sw, sh), 3.0, 3, torch.float32, dev)
    kb.imgproc.warp_affine(kb.Image(src[0]), got, m, kb.InterpolationMode.Bicubic if interp == "bicubic" else kb.InterpolationMode.Lanczos)
    same_bits(f"warp_affine {interp} {size} {angle}", got.data)


@pytest.mark.parametrize("mode,dw,dh", [("Letterbox", 64, 64), ("Stretch", 77, 41), ("Stretch", 300, 200)])
@pytest.mark.parametrize("fmt", ["Nv12", "Rgb8"])
def test_preprocess_lanczos_matches_reference_kernel(kb, oracle, dev, mode, dw, dh, fmt):
    """sample_lanczos (preprocess.rs:565-590) uses the CUDA math library's sinf: the reference's kernel is the bit spec;
    the C++ oracle (host sinf) is checked within the 1e-4 tolerance in test_gpu_variants.py."""
    w, h, n = 192, 108, 2
    nbytes = w * h * 3 // 2 if fmt == "Nv12" else w * h * 3
    frames = [cu(raw_bytes(nbytes, k), dev) for k in range(n)]
    pre = (kb.Preprocessor.builder().source_format(kb.SourceFormat[fmt]).mode(kb.ResizeMode[mode]).sampling(kb.InterpolationMode.Lanczos)
           .normalize(kb.Normalize.imagenet()).build_cuda())
    got = torch.zeros((n, 3, dh, dw), dtype=torch.float32, device=dev)
    pre.run_raw_batch(frames, w, h, got)
    same_bits(f"preprocess lanczos {fmt} {mode} {dw}x{dh}", got)
