"""GPU parity tests proper: the CUDA path, called through the C-ABI (via the package), against the CPU oracle
on the same seeded inputs.  Bars (BASELINE.json north_star): bit-exact for integer / byte paths; ≤ 1e-4 abs
for f32 paths — and because every kernel keeps the reference's expression trees under -fmad=false, the f32
paths are asserted BIT-EXACT too (TOL is what the contract requires; equality is what we deliver).

Sizes are small enough for the oracle to finish in seconds; odd / prime sizes hit every vector-width tail.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-4  # north_star: f32 interpolation / filter paths within 1e-4 abs


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


def cu(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def assert_f32_equal(got, want, what=""):
    got = np.asarray(got)
    want = np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    d = np.abs(got.astype(np.float64) - want.astype(np.float64))
    assert np.nanmax(d) <= TOL, f"{what}: max abs diff {np.nanmax(d)} > {TOL}"
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), \
        f"{what}: within tolerance (max {np.nanmax(d):.3g}) but not bit-identical ({int((got.view(np.uint32) != want.view(np.uint32)).sum())} elements)"


# ── colour ───────────────────────────────────────────────────────────────────
@pytest.mark.parametrize("npx", [1, 3, 7, 8, 64, 1001, 258 * 195, 4096 * 3 + 5])
@pytest.mark.parametrize("leaf", [0, 1])
def test_gray_from_rgb_f32(kb, oracle, dev, npx, leaf):
    src = oracle.pattern_f32(npx * 3).reshape(1, npx, 3)
    dst = kb.Image.zeros_cuda(kb.ImageSize(npx, 1), 1, torch.float32, dev)
    kb.imgproc.gray_from_rgb(kb.Image(cu(src, dev)), dst, leaf=leaf)
    assert_f32_equal(dst.numpy(), oracle.gray_from_rgb_f32(src, leaf), f"gray f32 leaf={leaf} n={npx}")


def test_gray_from_rgb_f32_unaligned_view(kb, oracle, dev):
    # a buffer whose base is only 4-byte aligned must take the scalar path and still be exact
    npx = 1000
    src = oracle.pattern_f32(npx * 3 + 1)
    t = cu(src, dev)[1:].reshape(1, npx, 3)
    dst = kb.Image.zeros_cuda(kb.ImageSize(npx, 1), 1, torch.float32, dev)
    kb.imgproc.gray_from_rgb(kb.Image(t), dst)
    assert_f32_equal(dst.numpy(), oracle.gray_from_rgb_f32(src[1:].reshape(1, npx, 3), 0))


@pytest.mark.parametrize("npx", [1, 5, 15, 16, 17, 4099, 640 * 480])
def test_gray_from_rgb_u8(kb, oracle, dev, npx):
    src = oracle.pattern_u8(npx * 3).reshape(1, npx, 3)
    dst = kb.Image.zeros_cuda(kb.ImageSize(npx, 1), 1, torch.uint8, dev)
    kb.imgproc.gray_from_rgb(kb.Image(cu(src, dev)), dst)
    np.testing.assert_array_equal(dst.numpy(), oracle.gray_from_rgb_u8(src))


@pytest.mark.parametrize("w,h,n", [(4, 4, 1), (64, 6, 1), (70, 4, 2), (128, 96, 3), (1920, 8, 1), (18, 2, 1)])
def test_rgb_from_nv12(kb, oracle, dev, w, h, n):
    frame = w * h * 3 // 2
    raw = oracle.pattern_u8(frame * n, 0xC0FFEE).reshape(n, frame)
    dst = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev, batch=n)
    kb.imgproc.rgb_from_nv12(cu(raw, dev), dst)
    want = np.stack([oracle.rgb_from_nv12(raw[i], w, h) for i in range(n)])
    np.testing.assert_array_equal(dst.numpy(), want)


def test_rgb_from_nv12_cv2_fixture(kb, dev):
    import os
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "nv12_cv2.npz"))
    for k in "abcd":
        w, h = (int(v) for v in z[f"{k}_wh"])
        dst = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev)
        kb.imgproc.rgb_from_nv12(cu(z[f"{k}_raw"], dev), dst)
        np.testing.assert_array_equal(dst.numpy(), z[f"{k}_rgb"])


@pytest.mark.parametrize("w,h,n", [(2, 1, 1), (64, 5, 1), (130, 7, 2), (16, 16, 4)])
def test_rgb_from_yuyv(kb, oracle, dev, w, h, n):
    frame = w * h * 2
    raw = oracle.pattern_u8(frame * n, 0xBEEF).reshape(n, frame)
    dst = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev, batch=n)
    kb.imgproc.rgb_from_yuyv(cu(raw, dev), dst)
    want = np.stack([oracle.rgb_from_yuyv(raw[i], w, h) for i in range(n)])
    np.testing.assert_array_equal(dst.numpy(), want)


# ── resize ───────────────────────────────────────────────────────────────────
RESIZE_CASES = [(3, 4, 2, 3), (129, 97, 64, 48), (64, 48, 129, 97), (258, 195, 128, 128), (37, 23, 37, 23), (31, 17, 7, 5),
                (5, 7, 31, 17), (640, 360, 213, 120)]


@pytest.mark.parametrize("sw,sh,dw,dh", RESIZE_CASES)
@pytest.mark.parametrize("mode", ["Bilinear", "Nearest"])
@pytest.mark.parametrize("c", [1, 3])
def test_resize_f32(kb, oracle, dev, sw, sh, dw, dh, mode, c):
    src = oracle.pattern_f32(sw * sh * c).reshape(sh, sw, c)
    dst = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), c, torch.float32, dev)
    kb.imgproc.resize(kb.Image(cu(src, dev)), dst, kb.InterpolationMode[mode])
    want = oracle.resize_f32(src, dw, dh, oracle.BILINEAR if mode == "Bilinear" else oracle.NEAREST)
    assert_f32_equal(dst.numpy(), want, f"resize {mode} c={c} {sw}x{sh}->{dw}x{dh}")


def test_resize_f32_batched(kb, oracle, dev):
    n, sw, sh, dw, dh = 3, 97, 61, 40, 30
    src = oracle.pattern_f32(n * sw * sh * 3).reshape(n, sh, sw, 3)
    dst = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), 3, torch.float32, dev, batch=n)
    kb.imgproc.resize(kb.Image(cu(src, dev)), dst, kb.InterpolationMode.Bilinear)
    want = np.stack([oracle.resize_f32(src[i], dw, dh) for i in range(n)])
    assert_f32_equal(dst.numpy(), want)


def test_resize_smoke_ch3_reference_vector(kb, dev):
    # resize/mod.rs:447-489 through the GPU path
    img = np.arange(36, dtype=np.float32).reshape(4, 3, 3)
    dst = kb.Image.zeros_cuda(kb.ImageSize(2, 3), 3, torch.float32, dev)
    kb.imgproc.resize(kb.Image(cu(img, dev)), dst, kb.InterpolationMode.Bilinear)
    want = np.array([2.25, 3.25, 4.25, 6.75, 7.75, 8.75, 14.25, 15.25, 16.25, 18.75, 19.75, 20.75, 26.25, 27.25, 28.25,
                     30.75, 31.75, 32.75], np.float32)
    assert np.abs(dst.numpy().reshape(-1) - want).max() < 1e-4


def test_resize_bilinear_normalize(kb, oracle, dev):
    sw, sh, dw, dh = 129, 97, 64, 48
    src = oracle.pattern_f32(sw * sh * 3).reshape(sh, sw, 3)
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    dst = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), 3, torch.float32, dev)
    kb.imgproc.resize_bilinear_normalize(kb.Image(cu(src, dev)), dst, mean, std)
    base = oracle.resize_f32(src, dw, dh)
    inv = np.float32(1.0) / np.array(std, np.float32)
    want = (base - np.array(mean, np.float32)) * inv  # (ch - mean) * inv_std   cuda/resize.rs:229-233
    assert_f32_equal(dst.numpy(), want.astype(np.float32))
    with pytest.raises(kb.ImageError, match="std must be non-zero"):
        kb.imgproc.resize_bilinear_normalize(kb.Image(cu(src, dev)), dst, mean, [0.0, 1.0, 1.0])


FUSED_CASES = [(60, 40, 37, 23), (74, 10, 37, 5), (384, 216, 128, 72), (128, 72, 384, 216), (100, 75, 33, 41), (40, 24, 20, 12),
               (67, 33, 66, 32), (3840, 24, 1280, 8),
               # 16-byte-aligned rows: the TMA row-span staged kernel (several x-tiles, ragged last tile, up/down, 1:1-ish)
               (256, 64, 100, 30), (512, 40, 171, 13), (1024, 30, 1000, 29), (1600, 21, 300, 9), (640, 18, 1279, 35),
               (1920, 27, 1281, 19), (48, 9, 50, 10), (16, 16, 3, 3),
               # integer downscales: odd ratios have a vertical weight of exactly 0 (single-row staging), even ones 0.5
               (160, 45, 32, 9), (320, 35, 64, 5), (256, 64, 64, 16), (96, 63, 80, 21), (768, 36, 256, 9), (1280, 30, 1280, 10),
               # exact 2x (box average) on 16-byte-aligned rows: the staged box mode, full / ragged / multi-tile widths
               (256, 64, 128, 32), (96, 20, 48, 10), (3840, 16, 1920, 8), (1312, 12, 656, 6), (544, 10, 272, 5)]


@pytest.mark.parametrize("sw,sh,dw,dh", FUSED_CASES)
@pytest.mark.parametrize("leaf", [0, 1, 2])
def test_fused_resize_normalize_chw(kb, oracle, dev, sw, sh, dw, dh, leaf):
    src = oracle.pattern_u8(sw * sh * 3).reshape(sh, sw, 3)
    scale, bias = oracle.normalize_params_from_mean_std([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])
    out = kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(cu(src, dev), dw, dh, scale, bias, leaf=leaf)
    want = oracle.resize_normalize_u8_to_f32_chw(src, dw, dh, scale, bias, leaf)
    assert_f32_equal(out.cpu().numpy()[0], want, f"fused {sw}x{sh}->{dw}x{dh} leaf={leaf}")


ROW_CASES = [(384, 216, 128, 72), (160, 45, 32, 9), (256, 64, 64, 16), (96, 63, 80, 21), (1280, 30, 1280, 10), (60, 40, 37, 23), (64, 32, 32, 16)]


@pytest.mark.parametrize("sw,sh,dw,dh", ROW_CASES)
def test_fused_resize_row_compacted_source(kb, oracle, dev, sw, sh, dw, dh):
    """kb200_resize_normalize_chw_u8_f32_rows over only the rows the geometry taps == the full-image result == oracle."""
    n = 3
    src = np.stack([oracle.pattern_u8(sw * sh * 3, 0xBEEF + i).reshape(sh, sw, 3) for i in range(n)])
    scale, bias = oracle.normalize_params_from_mean_std([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])
    P, F, K = kb.imgproc.resize_row_plan(sh, dh)
    assert sh % P == 0 and F + K <= P
    keep = np.array([y for y in range(sh) if F <= y % P < F + K])
    compact = np.ascontiguousarray(src[:, keep])
    assert compact.shape[1] == sh // P * K
    for leaf in (0, 1, 2):
        want = np.stack([oracle.resize_normalize_u8_to_f32_chw(src[i], dw, dh, scale, bias, leaf) for i in range(n)])
        got = kb.imgproc.resize_normalize_rows(cu(compact, dev), sw, sh, dw, dh, scale, bias, (P, F, K), leaf=leaf)
        assert_f32_equal(got.cpu().numpy(), want, f"rows {sw}x{sh}->{dw}x{dh} map={(P, F, K)} leaf={leaf}")
    # the dense map is always accepted; a map that drops tapped rows is rejected
    full = kb.imgproc.resize_normalize_rows(cu(src, dev), sw, sh, dw, dh, scale, bias, (1, 0, 1))
    assert_f32_equal(full.cpu().numpy(), np.stack([oracle.resize_normalize_u8_to_f32_chw(src[i], dw, dh, scale, bias) for i in range(n)]))
    if (P, F, K) == (1, 0, 1) and sh % 2 == 0:
        with pytest.raises(kb.ImageError, match="row map"):
            kb.imgproc.resize_normalize_rows(cu(src[:, ::2].copy(), dev), sw, sh, dw, dh, scale, bias, (2, 0, 1))


@pytest.mark.parametrize("sw,sh,dw,dh", [(384, 216, 128, 72), (256, 64, 64, 16), (100, 75, 33, 41), (40, 24, 20, 12), (512, 40, 171, 13)])
@pytest.mark.parametrize("pinned", [True, False])
def test_fused_resize_host_pipeline(kb, oracle, dev, sw, sh, dw, dh, pinned):
    """Host images in, host tensor out (the reference operator's own signature) through the staging ring: small
    staging buffers force several chunks per stream, a ragged last chunk and ring wrap-around."""
    n = 11
    src = np.stack([oracle.pattern_u8(sw * sh * 3, 0xC0FFEE + i).reshape(sh, sw, 3) for i in range(n)])
    scale, bias = oracle.normalize_params_from_mean_std([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])
    want = np.stack([oracle.resize_normalize_u8_to_f32_chw(src[i], dw, dh, scale, bias) for i in range(n)])
    P, F, K = kb.imgproc.resize_row_plan(sh, dh)
    frame_up = sw * 3 * (sh // P * K)
    pipe = kb.imgproc.HostPipeline(dev, src_chunk_bytes=2 * sw * sh * 3 + 7, dst_chunk_bytes=3 * dw * dh * 12, depth=2)
    hs = torch.from_numpy(src)
    hd = torch.zeros((n, 3, dh, dw), dtype=torch.float32)
    if pinned:
        hs, hd = hs.pin_memory(), hd.pin_memory()
    with torch.cuda.device(dev):
        for _ in range(2):  # second call reuses the ring while nothing is in flight
            hd.zero_()
            out = kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(hs, dw, dh, scale, bias, out=hd, pipeline=pipe)
            torch.cuda.current_stream().synchronize()
            assert out is hd
            assert_f32_equal(hd.numpy(), want, f"host pipeline {sw}x{sh}->{dw}x{dh}")
    up, down = pipe.last_transfer()
    assert up == n * frame_up and down == n * dw * dh * 12
    # staging smaller than one frame is an argument error, not a crash
    tiny = kb.imgproc.HostPipeline(dev, src_chunk_bytes=256, dst_chunk_bytes=256, depth=1)
    with torch.cuda.device(dev), pytest.raises(kb.ImageError, match="smaller than one frame"):
        kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(hs, dw, dh, scale, bias, out=hd, pipeline=tiny)
    pipe.close(); tiny.close()


def test_fused_resize_batched_unit_scale(kb, oracle, dev):
    n, sw, sh, dw, dh = 4, 96, 54, 32, 18
    src = np.stack([oracle.pattern_u8(sw * sh * 3, 0x12345678 + i).reshape(sh, sw, 3) for i in range(n)])
    scale, bias = [1 / 255.0] * 3, [0.0] * 3
    out = kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(cu(src, dev), dw, dh, scale, bias)
    want = np.stack([oracle.resize_normalize_u8_to_f32_chw(src[i], dw, dh, scale, bias) for i in range(n)])
    assert_f32_equal(out.cpu().numpy(), want)
    p = kb.imgproc.NormalizeParams.from_mean_std([0.5, 0.4, 0.3], [0.25, 0.2, 0.3])
    s2, b2 = oracle.normalize_params_from_mean_std([0.5, 0.4, 0.3], [0.25, 0.2, 0.3])
    assert p.scale == s2.tolist() and p.bias == b2.tolist()


@pytest.mark.parametrize("sw,sh,dw,dh,c", [(13, 9, 7, 5, 3), (64, 48, 129, 97, 1), (129, 97, 64, 48, 4), (1920, 16, 640, 5, 3)])
def test_resize_bilinear_u8_q14(kb, oracle, dev, sw, sh, dw, dh, c):
    src = oracle.pattern_u8(sw * sh * c).reshape(sh, sw, c)
    dst = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), c, torch.uint8, dev)
    kb.imgproc.resize_fast_u8(kb.Image(cu(src, dev)), dst)
    np.testing.assert_array_equal(dst.numpy(), oracle.resize_bilinear_u8(src, dw, dh))


U8_FAST = [  # (sw, sh, dw, dh, c, mode)  mode: 1 = Bilinear, 0 = Nearest
    (64, 48, 32, 24, 3, 1), (2, 2, 1, 1, 3, 1), (130, 6, 65, 3, 3, 1), (3840, 8, 1920, 4, 3, 1), (72, 10, 36, 5, 3, 1), (1928, 6, 964, 3, 3, 1),   # pyrdown arm (byte and word kernels)
    (2, 2, 4, 4, 3, 1), (3, 4, 6, 8, 3, 1), (17, 9, 34, 18, 3, 1), (33, 6, 66, 12, 3, 1), (640, 5, 1280, 10, 3, 1),   # pyrup arm
    (64, 48, 32, 24, 1, 1), (64, 48, 32, 24, 4, 1), (13, 9, 7, 5, 3, 1), (96, 63, 32, 21, 3, 1), (3840, 9, 1280, 3, 3, 1), (36, 9, 12, 3, 3, 1), (30, 9, 10, 3, 3, 1),                                     # 2x but not RGB / generic → Q14 arm
    (7, 5, 3, 2, 3, 0), (5, 5, 9, 7, 1, 0), (64, 48, 1, 1, 4, 0), (1, 1, 8, 8, 2, 0), (23, 37, 11, 17, 5, 0), (1920, 9, 640, 3, 3, 0), (96, 63, 32, 21, 3, 0), (30, 9, 10, 3, 3, 0),
]


@pytest.mark.parametrize("sw,sh,dw,dh,c,mode", U8_FAST)
def test_resize_fast_u8_cascade(kb, oracle, dev, sw, sh, dw, dh, c, mode):
    """resize_fast_u8_aa path selection (exact-2x pyramid arms, nearest, Q14) — bit-exact, batched."""
    n = 3
    src = np.stack([oracle.pattern_u8(sw * sh * c, 0xABCD + i).reshape(sh, sw, c) for i in range(n)])
    want = np.stack([oracle.resize_fast_u8(src[i], dw, dh, mode) for i in range(n)])
    s_img = kb.Image(cu(src, dev))
    d_img = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), c, torch.uint8, dev, batch=n)
    kb.imgproc.resize_fast_u8(s_img, d_img, kb.InterpolationMode.Bilinear if mode else kb.InterpolationMode.Nearest)
    np.testing.assert_array_equal(d_img.numpy(), want)


def test_resize_fast_u8_errors(kb, dev):
    d = kb.Image.zeros_cuda(kb.ImageSize(3, 3), 2, torch.uint8, dev)
    with pytest.raises(kb.ImageError, match="Unsupported channel count 2"):
        kb.imgproc.resize_fast_u8(kb.Image.zeros_cuda(kb.ImageSize(4, 4), 2, torch.uint8, dev), d)
    d3 = kb.Image.zeros_cuda(kb.ImageSize(3, 3), 3, torch.uint8, dev)
    with pytest.raises(kb.ImageError, match="Invalid image size"):
        kb.imgproc.resize_fast_u8(kb.Image.zeros_cuda(kb.ImageSize(1, 4), 3, torch.uint8, dev), d3)
    with pytest.raises(kb.ImageError):
        kb.imgproc.resize_fast_u8(kb.Image.zeros_cuda(kb.ImageSize(4, 4), 3, torch.uint8, dev), d3, kb.InterpolationMode.Bicubic)


AFFINES_U8 = [
    [1, 0, 0, 0, 1, 0], [-1, 0, 63, 0, 1, 0], [1, 0, 5.5, 0, 1, -3.25], [0.7, 0.0, 3.0, 0.0, 1.3, -2.0], [1.0, 0.2, -4.0, -0.1, 0.95, 6.0],
    [0.8660254, 0.5, -10.0, -0.5, 0.8660254, 20.0], [0.0, 1.0, 0.0, -1.0, 0.0, 47.0], [1e-9, 1.0, 3.0, 1.0, 0.0, 0.0], [2.5, 0, -30, 0, 2.5, -20],
]
PERSP_U8 = [
    [1.02, 0.03, -5.0, -0.03, 1.01, 2.0, 0.00005, 0.00003, 1.0], [0.9, 0.15, 10.0, -0.1, 1.1, -6.0, 0.0, 0.0, 1.0],
    [1.03, 0.05, -3.0, -0.02, 0.97, 4.0, 2.0 / (97 * 129), 1.5 / (129 * 97), 1.0], [-1.0, 0.0, 63.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0],
    [1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.02, 0.0, -0.5], [0.7, 0.0, 3.0, 0.0, 1.3, -2.0, 0.0, 0.001, 1.0], [1, 0, 0, 0, 1, 0, 0, 0, 1],
]


@pytest.mark.parametrize("mi", range(len(AFFINES_U8)))
@pytest.mark.parametrize("c", [1, 3, 4])
def test_warp_affine_u8(kb, oracle, dev, mi, c):
    """warp_affine_u8 (Q16 span walk + Q10 blend) — bit-exact, batched, source and destination sizes differ."""
    m = AFFINES_U8[mi]
    n, sw, sh, dw, dh = 2, 64, 48, 70, 41
    src = np.stack([oracle.pattern_u8(sw * sh * c, 0x51 + i).reshape(sh, sw, c) for i in range(n)])
    want = np.stack([oracle.warp_affine_u8(src[i], dw, dh, m) for i in range(n)])
    d = kb.Image(torch.full((n, dh, dw, c), 0xCD, dtype=torch.uint8, device=dev))
    kb.imgproc.warp_affine_u8(kb.Image(cu(src, dev)), d, m)
    np.testing.assert_array_equal(d.numpy(), want)


@pytest.mark.parametrize("mi", range(len(PERSP_U8)))
@pytest.mark.parametrize("c", [1, 3, 4])
def test_warp_perspective_u8(kb, oracle, dev, mi, c):
    m = PERSP_U8[mi]
    n, sw, sh, dw, dh = 2, 64, 48, 64, 48
    src = np.stack([oracle.pattern_u8(sw * sh * c, 0x61 + i).reshape(sh, sw, c) for i in range(n)])
    want = np.stack([oracle.warp_perspective_u8(src[i], dw, dh, m) for i in range(n)])
    d = kb.Image(torch.full((n, dh, dw, c), 0xCD, dtype=torch.uint8, device=dev))
    kb.imgproc.warp_perspective_u8(kb.Image(cu(src, dev)), d, m)
    np.testing.assert_array_equal(d.numpy(), want)


def test_warp_u8_large_and_errors(kb, oracle, dev):
    src = oracle.pattern_u8(640 * 360 * 3, 9).reshape(360, 640, 3)
    H = [1.02, 0.03, -40.0 / 6, -0.03, 1.01, 25.0 / 6, 2.0e-6 * 6, 1.2e-6 * 6, 1.0]
    d = kb.Image.zeros_cuda(kb.ImageSize(640, 360), 3, torch.uint8, dev)
    kb.imgproc.warp_perspective_u8(kb.Image(cu(src, dev)), d, H)
    np.testing.assert_array_equal(d.numpy(), oracle.warp_perspective_u8(src, 640, 360, H))
    M = kb.imgproc.get_rotation_matrix2d((320.0, 180.0), 30.0, 1.0)
    kb.imgproc.warp_affine_u8(kb.Image(cu(src, dev)), d, M)
    np.testing.assert_array_equal(d.numpy(), oracle.warp_affine_u8(src, 640, 360, M))
    with pytest.raises(kb.ImageError, match="singular|determinant"):
        kb.imgproc.warp_perspective_u8(kb.Image(cu(src, dev)), d, [1, 2, 3, 2, 4, 6, 0, 0, 1])
    with pytest.raises(kb.ImageError, match="Unsupported channel count"):
        kb.imgproc.warp_affine_u8(kb.Image.zeros_cuda(kb.ImageSize(8, 8), 2, torch.uint8, dev), kb.Image.zeros_cuda(kb.ImageSize(8, 8), 2, torch.uint8, dev), [1, 0, 0, 0, 1, 0])


U8_BLURS = [  # (rows, cols, c, kx, ky, sx, sy)
    (37, 83, 1, 5, 5, 1.0, 1.0), (37, 83, 1, 7, 7, 2.0, 2.0), (17, 45, 3, 3, 3, 1.0, 1.0), (23, 31, 3, 5, 3, 1.5, 2.0), (23, 31, 4, 9, 9, 0.0, 0.0),
    (9, 11, 3, 3, 3, 2.0, 2.0), (70, 65, 3, 0, 0, 0.8, 0.0), (33, 64, 3, 31, 31, 4.0, 4.0), (5, 1, 1, 3, 3, 1.0, 1.0), (1, 5, 1, 3, 3, 1.0, 1.0),
    (100, 130, 3, 5, 5, 1.5, 1.5), (2, 2, 4, 7, 7, 1.0, 1.0),
]


@pytest.mark.parametrize("rows,cols,c,kx,ky,sx,sy", U8_BLURS)
def test_gaussian_blur_u8(kb, oracle, dev, rows, cols, c, kx, ky, sx, sy):
    n = 2
    src = np.stack([oracle.pattern_u8(rows * cols * c, 0x71 + i).reshape(rows, cols, c) for i in range(n)])
    want = np.stack([oracle.gaussian_blur_u8(src[i], (kx, ky), (sx, sy)) for i in range(n)])
    d = kb.Image(torch.full((n, rows, cols, c), 0xCD, dtype=torch.uint8, device=dev))
    kb.imgproc.gaussian_blur_u8(kb.Image(cu(src, dev)), d, (kx, ky), (sx, sy))
    np.testing.assert_array_equal(d.numpy(), want)


@pytest.mark.parametrize("kx,ky", [(3, 3), (5, 5), (7, 3), (1, 9), (15, 15)])
def test_box_blur_u8(kb, oracle, dev, kx, ky):
    src = oracle.pattern_u8(41 * 67 * 3, 0x81).reshape(41, 67, 3)
    d = kb.Image.zeros_cuda(kb.ImageSize(67, 41), 3, torch.uint8, dev)
    kb.imgproc.box_blur_u8(kb.Image(cu(src, dev)), d, (kx, ky))
    np.testing.assert_array_equal(d.numpy(), oracle.box_blur_u8(src, (kx, ky)))


def test_blur_u8_errors_and_4k(kb, oracle, dev):
    s3 = kb.Image.zeros_cuda(kb.ImageSize(8, 8), 3, torch.uint8, dev)
    with pytest.raises(kb.ImageError, match="Invalid sigma"):
        kb.imgproc.box_blur_u8(s3, kb.Image.zeros_cuda(kb.ImageSize(8, 8), 3, torch.uint8, dev), (4, 3))
    with pytest.raises(kb.ImageError, match="Invalid sigma"):
        kb.imgproc.gaussian_blur_u8(s3, kb.Image.zeros_cuda(kb.ImageSize(8, 8), 3, torch.uint8, dev), (4, 4), (1.0, 1.0))
    with pytest.raises(kb.ImageError, match="Invalid image size"):
        kb.imgproc.gaussian_blur_u8(s3, kb.Image.zeros_cuda(kb.ImageSize(9, 8), 3, torch.uint8, dev), (3, 3), (1.0, 1.0))
    src = oracle.pattern_u8(1920 * 270 * 3, 3).reshape(270, 1920, 3)
    d = kb.Image.zeros_cuda(kb.ImageSize(1920, 270), 3, torch.uint8, dev)
    kb.imgproc.gaussian_blur_u8(kb.Image(cu(src, dev)), d, (5, 5), (1.5, 1.5))
    np.testing.assert_array_equal(d.numpy(), oracle.gaussian_blur_u8(src, (5, 5), (1.5, 1.5)))


def _remap_maps(dw, dh, sw, sh, kind, rng):
    y, x = np.meshgrid(np.arange(dh, dtype=np.float32), np.arange(dw, dtype=np.float32), indexing="ij")
    if kind == "identity":
        return x * np.float32(sw / dw), y * np.float32(sh / dh)
    if kind == "swirl":   # smooth distortion that leaves the image on all sides, with NaN / inf holes
        cx, cy = np.float32(sw / 2), np.float32(sh / 2)
        r2 = ((x - dw / 2) ** 2 + (y - dh / 2) ** 2).astype(np.float32) / np.float32(dw * dw)
        mx = (cx + (x - dw / 2) * (1 + 1.5 * r2) * np.float32(sw / dw)).astype(np.float32)
        my = (cy + (y - dh / 2) * (1 + 1.5 * r2) * np.float32(sh / dh)).astype(np.float32)
        mx[0, 0] = np.nan; my[1, 1] = np.inf; mx[2, 2] = -np.inf; mx[3, 3] = sw - 0.25; my[3, 3] = sh - 0.25; mx[4, 4] = sw; my[5, 5] = -0.0
        return mx, my
    mx = rng.uniform(-3, sw + 3, (dh, dw)).astype(np.float32); my = rng.uniform(-3, sh + 3, (dh, dw)).astype(np.float32)
    return mx, my


@pytest.mark.parametrize("kind", ["identity", "swirl", "random"])
@pytest.mark.parametrize("mode", [0, 1])
def test_remap_f32(kb, oracle, dev, kind, mode):
    n, sw, sh, dw, dh = 2, 64, 48, 57, 39
    rng = np.random.default_rng(11)
    src = np.stack([oracle.pattern_f32(sw * sh * 3, 0x91 + i).reshape(sh, sw, 3) for i in range(n)])
    mx, my = _remap_maps(dw, dh, sw, sh, kind, rng)
    want = np.stack([oracle.remap(src[i], mx, my, mode) for i in range(n)])
    d = kb.Image(torch.full((n, dh, dw, 3), float("nan"), dtype=torch.float32, device=dev))
    kb.imgproc.remap(kb.Image(cu(src, dev)), d, kb.Image(cu(mx[..., None], dev)), kb.Image(cu(my[..., None], dev)),
                     kb.InterpolationMode.Bilinear if mode else kb.InterpolationMode.Nearest)
    assert_f32_equal(d.numpy(), want, f"remap f32 {kind} mode={mode}")


@pytest.mark.parametrize("kind", ["identity", "swirl", "random"])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("c", [1, 3, 4])
def test_remap_u8(kb, oracle, dev, kind, mode, c):
    n, sw, sh, dw, dh = 2, 64, 48, 57, 39
    rng = np.random.default_rng(12)
    src = np.stack([oracle.pattern_u8(sw * sh * c, 0xA1 + i).reshape(sh, sw, c) for i in range(n)])
    mx, my = _remap_maps(dw, dh, sw, sh, kind, rng)
    want = np.stack([oracle.remap(src[i], mx, my, mode) for i in range(n)])
    d = kb.Image(torch.full((n, dh, dw, c), 0xCD, dtype=torch.uint8, device=dev))
    kb.imgproc.remap_u8(kb.Image(cu(src, dev)), d, kb.Image(cu(mx[..., None], dev)), kb.Image(cu(my[..., None], dev)),
                        kb.InterpolationMode.Bilinear if mode else kb.InterpolationMode.Nearest)
    np.testing.assert_array_equal(d.numpy(), want)


def test_remap_errors(kb, dev):
    s = kb.Image.zeros_cuda(kb.ImageSize(8, 8), 3, torch.float32, dev)
    d = kb.Image.zeros_cuda(kb.ImageSize(6, 5), 3, torch.float32, dev)
    m65 = kb.Image.zeros_cuda(kb.ImageSize(6, 5), 1, torch.float32, dev)
    m66 = kb.Image.zeros_cuda(kb.ImageSize(6, 6), 1, torch.float32, dev)
    with pytest.raises(kb.ImageError, match="Invalid image size"):
        kb.imgproc.remap(s, d, m65, m66, kb.InterpolationMode.Bilinear)
    with pytest.raises(kb.ImageError, match="Invalid image size"):
        kb.imgproc.remap(s, d, m66, m66, kb.InterpolationMode.Bilinear)
    with pytest.raises(kb.ImageError, match="Unsupported interpolation"):
        kb.imgproc.remap(s, d, m65, m65, kb.InterpolationMode.Bicubic)
    host_map = kb.Image(torch.zeros((5, 6, 1), dtype=torch.float32))
    with pytest.raises(kb.ImageError, match="device-resident"):
        kb.imgproc.remap(s, d, host_map, m65, kb.InterpolationMode.Bilinear)


# ── warps ────────────────────────────────────────────────────────────────────
AFFINES = [
    ("identity", [1, 0, 0, 0, 1, 0]),
    ("hflip", [-1, 0, 63, 0, 1, 0]),
    ("shift", [1, 0, 5.5, 0, 1, -3.25]),
    ("scale", [0.7, 0.0, 3.0, 0.0, 1.3, -2.0]),
    ("shear", [1.0, 0.2, -4.0, -0.1, 0.95, 6.0]),
]


@pytest.mark.parametrize("name,m", AFFINES)
@pytest.mark.parametrize("mode", ["Bilinear", "Nearest"])
def test_warp_affine(kb, oracle, dev, name, m, mode):
    sw, sh, dw, dh = 64, 48, 71, 53
    src = oracle.pattern_f32(sw * sh * 3).reshape(sh, sw, 3)
    dst = kb.Image.from_size_val(kb.ImageSize(dw, dh), -1.0, 3, torch.float32, dev)
    kb.imgproc.warp_affine(kb.Image(cu(src, dev)), dst, m, kb.InterpolationMode[mode])
    want = oracle.warp_affine_f32(src, m, dw, dh, oracle.BILINEAR if mode == "Bilinear" else oracle.NEAREST)
    assert_f32_equal(dst.numpy(), want, f"warp_affine {name} {mode}")


@pytest.mark.parametrize("angle", [30.0, 45.0, 90.0, 180.0, 270.0, -17.5])
def test_warp_affine_rotations(kb, oracle, dev, angle):
    # right-angle rotations exercise the degenerate-axis validity rule (cuda/warp_affine.rs:103-112)
    sw, sh = 97, 61
    src = oracle.pattern_f32(sw * sh * 3).reshape(sh, sw, 3)
    m = kb.imgproc.get_rotation_matrix2d((sw / 2.0, sh / 2.0), angle, 1.0)
    assert m == oracle.get_rotation_matrix2d((sw / 2.0, sh / 2.0), angle, 1.0).tolist()
    for mode, om in (("Bilinear", oracle.BILINEAR), ("Nearest", oracle.NEAREST)):
        dst = kb.Image.zeros_cuda(kb.ImageSize(sw, sh), 3, torch.float32, dev)
        kb.imgproc.warp_affine(kb.Image(cu(src, dev)), dst, m, kb.InterpolationMode[mode])
        assert_f32_equal(dst.numpy(), oracle.warp_affine_f32(src, m, sw, sh, om), f"rot {angle} {mode}")


HOMOGRAPHIES = [
    # cuda/warp_perspective.rs:784-808 — the reference's own GPU-parity matrices and sizes
    ((129, 97), [1.03, 0.05, -3.0, -0.02, 0.97, 4.0, 2.0 / (97 * 129), 1.5 / (129 * 97), 1.0]),
    ((320, 240), [0.9, 0.15, 10.0, -0.1, 1.1, -6.0, 0.0, 0.0, 1.0]),
    ((64, 48), [1, 0, 0, 0, 1, 0, 0, 0, 1]),
    ((64, 48), [-1, 0, 63, 0, 1, 0, 0, 0, 1]),
    ((120, 160), [1.02, 0.03, -5.0, -0.03, 1.01, 2.0, 0.00005, 0.00003, 1.0]),  # warp/perspective.rs:652
]


@pytest.mark.parametrize("size,h", HOMOGRAPHIES)
@pytest.mark.parametrize("mode", ["Bilinear", "Nearest"])
def test_warp_perspective(kb, oracle, dev, size, h, mode):
    sw, sh = size
    src = oracle.pattern_f32(sw * sh * 3).reshape(sh, sw, 3)
    dst = kb.Image.from_size_val(kb.ImageSize(sw, sh), 7.0, 3, torch.float32, dev)  # GPU rule: OOB written 0
    kb.imgproc.warp_perspective(kb.Image(cu(src, dev)), dst, h, kb.InterpolationMode[mode])
    want = oracle.warp_perspective_f32(src, h, sw, sh, oracle.BILINEAR if mode == "Bilinear" else oracle.NEAREST)
    assert_f32_equal(dst.numpy(), want, f"warp_perspective {mode} {size}")


def test_warp_perspective_batched_and_resize_equivalence(kb, oracle, dev):
    # warp/perspective.rs:537-589: the half-pixel 2x downscale homography equals resize bit-for-bit
    n = 3
    src = oracle.pattern_f32(n * 16 * 16 * 3).reshape(n, 16, 16, 3)
    m = [0.5, 0, -0.25, 0, 0.5, -0.25, 0, 0, 1]
    a = kb.Image.zeros_cuda(kb.ImageSize(8, 8), 3, torch.float32, dev, batch=n)
    b = kb.Image.zeros_cuda(kb.ImageSize(8, 8), 3, torch.float32, dev, batch=n)
    kb.imgproc.warp_perspective(kb.Image(cu(src, dev)), a, m, kb.InterpolationMode.Bilinear)
    kb.imgproc.resize(kb.Image(cu(src, dev)), b, kb.InterpolationMode.Bilinear)
    np.testing.assert_array_equal(a.numpy(), b.numpy())
    assert_f32_equal(a.numpy(), np.stack([oracle.resize_f32(src[i], 8, 8) for i in range(n)]))


def test_warp_errors(kb, oracle, dev):
    src = kb.Image(cu(oracle.pattern_f32(8 * 8 * 3).reshape(8, 8, 3), dev))
    dst = kb.Image.zeros_cuda(kb.ImageSize(8, 8), 3, torch.float32, dev)
    with pytest.raises(kb.ImageError, match="singular"):
        kb.imgproc.warp_perspective(src, dst, [1, 2, 3, 2, 4, 6, 3, 6, 9], kb.InterpolationMode.Bilinear)
    for mode in (kb.InterpolationMode.Bicubic, kb.InterpolationMode.Lanczos):   # warp/affine.rs:528-550: all modes are supported
        kb.imgproc.warp_affine(src, dst, [1, 0, 0, 0, 1, 0], mode)
    gray = kb.Image.zeros_cuda(kb.ImageSize(8, 8), 1, torch.float32, dev)
    with pytest.raises(kb.ImageError, match="3-channel f32 images only"):
        kb.imgproc.warp_affine(gray, gray, [1, 0, 0, 0, 1, 0], kb.InterpolationMode.Bilinear)
    host = kb.Image(torch.zeros(8, 8, 3))
    with pytest.raises(kb.ImageError) as e:
        kb.imgproc.warp_affine(host, dst, [1, 0, 0, 0, 1, 0], kb.InterpolationMode.Bilinear)
    assert e.value.kind == "MixedResidency"
    with pytest.raises(kb.ImageError) as e:
        kb.imgproc.warp_affine(host, host, [1, 0, 0, 0, 1, 0], kb.InterpolationMode.Bilinear)
    assert e.value.kind == "UnsupportedDevice"  # no CPU fallback


# ── filters ──────────────────────────────────────────────────────────────────
@pytest.mark.parametrize("w,h,c", [(5, 5, 1), (97, 61, 3), (64, 32, 3), (130, 67, 1), (33, 200, 4), (300, 40, 2)])
@pytest.mark.parametrize("k,sigma", [((3, 3), (0.5, 0.5)), ((5, 5), (1.5, 1.5)), ((7, 3), (2.0, 0.8)), ((0, 0), (1.5, 0.0)),
                                     ((9, 9), (0.0, 0.0))])
def test_gaussian_blur(kb, oracle, dev, w, h, c, k, sigma):
    src = oracle.pattern_f32(w * h * c).reshape(h, w, c)
    dst = kb.Image.zeros_cuda(kb.ImageSize(w, h), c, torch.float32, dev)
    kb.imgproc.gaussian_blur(kb.Image(cu(src, dev)), dst, k, sigma)
    assert_f32_equal(dst.numpy(), oracle.gaussian_blur(src, k, sigma), f"gaussian {w}x{h}x{c} k={k}")


def test_gaussian_blur_reference_vectors(kb, dev):
    # filter/ops.rs:2184-2206 exact output through the GPU path
    img = np.arange(25, dtype=np.float32).reshape(5, 5, 1)
    dst = kb.Image.zeros_cuda(kb.ImageSize(5, 5), 1, torch.float32, dev)
    kb.imgproc.gaussian_blur(kb.Image(cu(img, dev)), dst, (3, 3), (0.5, 0.5))
    want = np.array([0.57097936, 1.4260278, 2.3195207, 3.213014, 3.5739717, 4.5739717, 5.999999, 7.0, 7.999999, 7.9349294,
                     9.041435, 10.999999, 12.0, 12.999998, 12.402394, 13.5089, 15.999998, 17.0, 17.999996, 16.86986,
                     15.58594, 18.230816, 19.124311, 20.017801, 18.588936], np.float32)
    np.testing.assert_array_equal(dst.numpy().reshape(-1), want)


@pytest.mark.parametrize("w,h,c", [(11, 7, 3), (97, 61, 3), (128, 64, 1), (70, 33, 2)])
@pytest.mark.parametrize("ksize", [3, 5])
def test_sobel(kb, oracle, dev, w, h, c, ksize):
    src = oracle.pattern_f32(w * h * c).reshape(h, w, c)
    dst = kb.Image.zeros_cuda(kb.ImageSize(w, h), c, torch.float32, dev)
    kb.imgproc.sobel(kb.Image(cu(src, dev)), dst, ksize)
    assert_f32_equal(dst.numpy(), oracle.sobel(src, ksize), f"sobel {w}x{h}x{c} k={ksize}")


def test_separable_filter_generic_and_batched(kb, oracle, dev):
    n, w, h, c = 2, 75, 49, 3
    src = oracle.pattern_f32(n * w * h * c).reshape(n, h, w, c)
    kx = [0.1, -0.3, 0.5, 0.25, 0.0, 0.7, -0.2, 0.05, 0.3, 0.11, -0.09]  # 11 taps: runtime-loop instance
    ky = [0.2, 0.6, 0.2, -0.1]  # even length
    dst = kb.Image.zeros_cuda(kb.ImageSize(w, h), c, torch.float32, dev, batch=n)
    kb.imgproc.separable_filter(kb.Image(cu(src, dev)), dst, kx, ky)
    want = np.stack([oracle.separable_filter(src[i], kx, ky) for i in range(n)])
    assert_f32_equal(dst.numpy(), want)
    with pytest.raises(kb.ImageError) as e:
        kb.imgproc.separable_filter(kb.Image(cu(src, dev)), dst, [], ky)
    assert e.value.kind == "InvalidKernelLength"
    with pytest.raises(kb.ImageError) as e:
        kb.imgproc.gaussian_blur(kb.Image(cu(src, dev)), dst, (2, 3), (1.0, 1.0))
    assert e.value.kind == "InvalidSigmaValue"
    with pytest.raises(kb.ImageError) as e:
        kb.imgproc.sobel(kb.Image(cu(src, dev)), dst, 7)
    assert e.value.kind == "InvalidKernelLength"


# ── normalize / statistics ───────────────────────────────────────────────────
@pytest.mark.parametrize("npx,c", [(4, 3), (1001, 3), (97 * 61, 3), (500, 1), (333, 4)])
def test_normalize_mean_std(kb, oracle, dev, npx, c):
    src = oracle.pattern_f32(npx * c).reshape(1, npx, c)
    mean = [0.485, 0.456, 0.406, 0.5][:c]
    std = [0.229, 0.224, 0.225, 0.25][:c]
    dst = kb.Image.zeros_cuda(kb.ImageSize(npx, 1), c, torch.float32, dev)
    kb.imgproc.normalize_mean_std(kb.Image(cu(src, dev)), dst, mean, std)
    assert_f32_equal(dst.numpy(), oracle.normalize_mean_std(src, mean, std))


def test_normalize_min_max_and_find(kb, oracle, dev):
    src = (oracle.pattern_f32(97 * 61 * 3) * np.float32(3.5) - np.float32(1.25)).reshape(61, 97, 3)
    im = kb.Image(cu(src, dev))
    assert kb.imgproc.find_min_max(im) == oracle.find_min_max(src)
    dst = kb.Image.zeros_cuda(kb.ImageSize(97, 61), 3, torch.float32, dev)
    kb.imgproc.normalize_min_max(im, dst, -1.0, 2.0)
    assert_f32_equal(dst.numpy(), oracle.normalize_min_max(src, -1.0, 2.0))


@pytest.mark.parametrize("npx", [2, 8, 1000, 1003])
@pytest.mark.parametrize("leaf", [0, 1])
def test_normalize_rgb_u8(kb, oracle, dev, npx, leaf):
    src = oracle.pattern_u8(npx * 3, 0xDEADBEEF)
    scale = [1 / (0.229 * 255), 1 / (0.224 * 255), 1 / (0.225 * 255)]
    off = [-0.485 / 0.229, -0.456 / 0.224, -0.406 / 0.225]
    dst = torch.zeros(npx * 3, dtype=torch.float32, device=dev)
    kb.imgproc.normalize_rgb_u8(cu(src, dev), dst, npx, scale, off, leaf=leaf)
    assert_f32_equal(dst.cpu().numpy(), oracle.normalize_rgb_u8(src, scale, off, leaf).reshape(-1))


@pytest.mark.parametrize("w,h", [(2, 2), (97, 61), (1920, 1080), (3, 1)])
def test_std_mean(kb, oracle, dev, w, h):
    if (w, h) == (2, 2):
        src = np.array([0, 1, 2, 253, 254, 255, 128, 129, 130, 64, 65, 66], np.uint8).reshape(2, 2, 3)  # core.rs:27-40
    else:
        src = oracle.pattern_u8(w * h * 3).reshape(h, w, 3)
    im = kb.Image(cu(src, dev))
    std, mean = kb.imgproc.std_mean(im)
    ostd, omean, osums = oracle.std_mean(src)
    assert kb.imgproc.std_mean_sums(im).tolist() == [int(v) for v in osums]
    assert std == ostd.tolist() and mean == omean.tolist()  # exact f64 equality
    if (w, h) == (2, 2):
        assert std == [93.5183805462862] * 3 and mean == [111.25, 112.25, 113.25]


# ── camera preprocess ────────────────────────────────────────────────────────
def raw_bytes(n, k=0):
    return ((np.arange(n, dtype=np.int64) * 7 + 13) % 251 + 31 * k).astype(np.uint8)  # preprocess.rs:1765-1767, :1868


FMTS = {"Nv12": (3, lambda w, h: w * h * 3 // 2), "Yuyv": (4, lambda w, h: w * h * 2), "Gray8": (2, lambda w, h: w * h),
        "Rgb8": (0, lambda w, h: w * h * 3), "Bgr8": (1, lambda w, h: w * h * 3), "Rgba8": (0, lambda w, h: w * h * 4),
        "Bgra8": (1, lambda w, h: w * h * 4)}


@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("mode", ["Letterbox", "Stretch"])
@pytest.mark.parametrize("sampling", ["Bilinear", "Nearest"])
@pytest.mark.parametrize("geom", [(8, 6, 7, 5), (64, 48, 40, 40), (64, 48, 64, 48), (30, 20, 61, 47), (128, 72, 40, 24),
                                  (96, 54, 32, 32), (32, 24, 64, 48), (192, 108, 64, 36)])
def test_preprocess_formats(kb, oracle, dev, fmt, mode, sampling, geom):
    w, h, dw, dh = geom
    code, blen = FMTS[fmt]
    raw = raw_bytes(blen(w, h))
    pre = (kb.Preprocessor.builder().source_format(kb.SourceFormat[fmt]).mode(kb.ResizeMode[mode])
           .sampling(kb.InterpolationMode[sampling]).normalize(kb.Normalize.imagenet()).pad_value(114).build_cuda())
    dst = torch.zeros((1, 3, dh, dw), dtype=torch.float32, device=dev)
    pre.run_raw(cu(raw, dev), w, h, dst)
    inv = tuple(float(np.float32(1.0) / np.float32(s)) for s in kb.IMAGENET_STD)
    cfg = oracle.PreprocessCfg(mode=oracle.LETTERBOX if mode == "Letterbox" else oracle.STRETCH, fmt=code,
                               bpp=4 if fmt.endswith("a8") else None, mean=kb.IMAGENET_MEAN, inv_std=inv, pad_value=114.0,
                               sampling=oracle.BILINEAR if sampling == "Bilinear" else oracle.NEAREST)
    want = oracle.preprocess_frame(raw, cfg, w, h, dw, dh)
    assert_f32_equal(dst.cpu().numpy()[0], want, f"preprocess {fmt} {mode} {sampling} {geom}")


def test_preprocess_batch_matches_single_and_errors(kb, oracle, dev):
    # preprocess.rs:1855-1896
    w, h = 8, 6
    pre = kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).build_cuda()
    raws = [cu(raw_bytes(w * h * 3 // 2, k), dev) for k in range(3)]
    batch = torch.zeros((3, 3, 5, 7), dtype=torch.float32, device=dev)
    pre.run_raw_batch(raws, w, h, batch)
    for i, r in enumerate(raws):
        one = torch.zeros((1, 3, 5, 7), dtype=torch.float32, device=dev)
        pre.run_raw(r, w, h, one)
        assert torch.equal(batch[i], one[0])
        want = oracle.preprocess_frame(r.cpu().numpy(), oracle.PreprocessCfg(fmt=oracle.FMT_NV12), w, h, 7, 5)
        assert_f32_equal(batch[i].cpu().numpy(), want)
    bad = torch.zeros((2, 3, 5, 7), dtype=torch.float32, device=dev)
    with pytest.raises(kb.PreprocessError) as e:
        pre.run_raw_batch(raws, w, h, bad)
    assert e.value.kind == "BatchMismatch" and e.value.fields == {"dst_n": 2, "frames": 3}
    # preprocess.rs:1902-1938
    dst = torch.zeros((1, 3, 4, 4), dtype=torch.float32, device=dev)
    with pytest.raises(kb.PreprocessError) as e:
        pre.run_raw(cu(raw_bytes(60), dev), 8, 6, dst)
    assert e.value.kind == "InvalidRawSource" and e.value.fields["need"] == 72
    with pytest.raises(kb.PreprocessError) as e:
        pre.run_raw(cu(raw_bytes(80), dev), 8, 5, dst)
    assert e.value.kind == "InvalidRawSource"
    surf = kb.PitchedSurface(cu(raw_bytes(8 * 6 * 4), dev), 8, 6, 32, 4)
    with pytest.raises(kb.PreprocessError) as e:
        pre.run_surface(surf, dst)
    assert e.value.kind == "FormatNeedsRawBuffer"


def test_preprocess_strided_ring_buffer(kb, oracle, dev):
    w, h, n = 32, 16, 5
    frame = w * h * 3 // 2
    stride = frame + 64  # padded slots
    ring = np.zeros(stride * n, np.uint8)
    for k in range(n):
        ring[k * stride:k * stride + frame] = raw_bytes(frame, k)
    pre = kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).mode(kb.ResizeMode.Stretch).build_cuda()
    dst = torch.zeros((n, 3, 12, 20), dtype=torch.float32, device=dev)
    pre.run_raw_strided(cu(ring, dev), stride, n, w, h, dst)
    cfg = oracle.PreprocessCfg(mode=oracle.STRETCH, fmt=oracle.FMT_NV12)
    want = np.stack([oracle.preprocess_frame(ring[k * stride:k * stride + frame], cfg, w, h, 20, 12) for k in range(n)])
    assert_f32_equal(dst.cpu().numpy(), want)


def test_preprocess_f16_and_pitched(kb, oracle, dev):
    # f16 == RNE(f32) (preprocess.rs:1646-1675) ; pitched == tight (preprocess.rs:1593-1640)
    w, h, pitch = 23, 17, 23 * 4 + 13
    tight = oracle.pattern_u8(w * h * 4, 99).reshape(h, w, 4)
    pitched = np.full(pitch * h, 0xAA, np.uint8)
    for y in range(h):
        pitched[y * pitch:y * pitch + w * 4] = tight[y].reshape(-1)
    for mode in (kb.ResizeMode.Letterbox, kb.ResizeMode.Stretch):
        pre = kb.Preprocessor.builder().mode(mode).normalize(kb.Normalize.imagenet()).build_cuda()
        d_img = torch.zeros((1, 3, 6, 8), dtype=torch.float32, device=dev)
        pre.run(kb.Image(cu(tight, dev)), d_img)
        d_surf = torch.zeros((1, 3, 6, 8), dtype=torch.float32, device=dev)
        pre.run_surface(kb.PitchedSurface(cu(pitched, dev), w, h, pitch, 4), d_surf)
        assert torch.equal(d_img, d_surf)
        d16 = torch.zeros((1, 3, 6, 8), dtype=torch.float16, device=dev)
        pre.run_f16(kb.Image(cu(tight, dev)), d16)
        np.testing.assert_array_equal(d16.cpu().numpy().view(np.uint16), d_img.cpu().numpy().astype(np.float16).view(np.uint16))
        inv = tuple(float(np.float32(1.0) / np.float32(s)) for s in kb.IMAGENET_STD)
        cfg = oracle.PreprocessCfg(mode=oracle.LETTERBOX if mode is kb.ResizeMode.Letterbox else oracle.STRETCH, bpp=4,
                                   mean=kb.IMAGENET_MEAN, inv_std=inv)
        assert_f32_equal(d_img.cpu().numpy()[0], oracle.preprocess_frame(tight, cfg, w, h, 8, 6))
        want16 = oracle.preprocess_frame(tight, cfg, w, h, 8, 6, f16=True)
        np.testing.assert_array_equal(d16.cpu().numpy()[0].view(np.uint16), want16.view(np.uint16))


def test_preprocess_typed_run_rejections(kb, dev):
    # preprocess.rs:1741-1761, :1511-1554
    src = kb.Image(torch.zeros((4, 4, 3), dtype=torch.uint8, device=dev))
    dst = torch.zeros((1, 3, 4, 4), dtype=torch.float32, device=dev)
    pre = kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).build_cuda()
    with pytest.raises(kb.PreprocessError) as e:
        pre.run(src, dst)
    assert e.value.kind == "FormatNeedsRawBuffer"
    pre = kb.Preprocessor.builder().source_format(kb.SourceFormat.Rgba8).build_cuda()
    with pytest.raises(kb.PreprocessError) as e:
        pre.run(src, dst)
    assert e.value.kind == "FormatNeedsRawBuffer"
    pre = kb.Preprocessor.builder().build_cuda()
    with pytest.raises(kb.PreprocessError) as e:
        pre.run(kb.Image(torch.zeros((2, 2, 1), dtype=torch.uint8, device=dev)), dst)
    assert e.value.kind == "UnsupportedChannels"
    with pytest.raises(kb.PreprocessError) as e:
        pre.run(src, torch.zeros((1, 1, 4, 4), dtype=torch.float32, device=dev))
    assert e.value.kind == "BadOutputShape"
    with pytest.raises(kb.PreprocessError) as e:
        kb.Preprocessor.builder().normalize(kb.Normalize.MeanStd([0.5] * 3, [0.0, 0.2, 0.2])).build_cuda()
    assert e.value.kind == "InvalidNormalize"
    with pytest.raises(kb.PreprocessError) as e:
        kb.Preprocessor.builder().sampling(kb.InterpolationMode.Bicubic).build_cuda()
    assert e.value.kind == "UnsupportedSampling"


# ── config 1 and full-size properties ────────────────────────────────────────
def test_config1_dog_gray_resize(kb, dev):
    import os
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "dog_cfg1.npz"))
    f = z["rgb"].astype(np.float32) * np.float32(1.0 / 255.0)
    gray = kb.Image.zeros_cuda(kb.ImageSize(258, 195), 1, torch.float32, dev)
    kb.imgproc.gray_from_rgb(kb.Image(cu(f, dev)), gray)
    assert_f32_equal(gray.numpy(), z["gray"], "cfg1 gray")
    small = kb.Image.zeros_cuda(kb.ImageSize(128, 128), 1, torch.float32, dev)
    kb.imgproc.resize(gray, small, kb.InterpolationMode.Bilinear)
    assert_f32_equal(small.numpy(), z["resized"], "cfg1 resize")


def test_full_size_properties_config2(kb, oracle, dev):
    """BASELINE config 2 at FULL size (3840x2160 → 1280x720, a few frames), checked through properties that do
    not need the oracle at full size: (1) exact equality with the oracle on sampled rows, (2) linearity in
    (scale, bias), (3) batch element i == single-frame call."""
    n, sw, sh, dw, dh = 2, 3840, 2160, 1280, 720
    src = np.stack([oracle.pattern_u8(sw * sh * 3, 0x12345678 + i).reshape(sh, sw, 3) for i in range(n)])
    t = cu(src, dev)
    scale, bias = oracle.normalize_params_from_mean_std(kb.IMAGENET_MEAN, kb.IMAGENET_STD)
    out = kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(t, dw, dh, scale, bias)
    # (1) the oracle on a 24-row source band reproduces dst rows exactly (scale 3: dst row y uses src rows 3y+1, 3y+2)
    for y0 in (0, 357, 712):
        band = src[0, 3 * y0:3 * y0 + 24]
        want = oracle.resize_normalize_u8_to_f32_chw(band, dw, 8, scale, bias)
        assert_f32_equal(out[0, :, y0:y0 + 8].cpu().numpy(), want, f"cfg2 band {y0}")
    # (3)
    one = kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(t[1], dw, dh, scale, bias)
    assert torch.equal(one[0], out[1])
    # (2) unit-scale output u: ImageNet output must equal fma(u*255-ish…) only approximately; check affine relation
    unit = kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(t[:1], dw, dh, [1.0] * 3, [0.0] * 3)
    for c in range(3):
        approx = unit[0, c] * float(scale[c]) + float(bias[c])
        assert (approx - out[0, c]).abs().max().item() < 1e-5


def test_full_size_properties_nv12_1080p(kb, oracle, dev):
    """Config 3a at full size: 1080p NV12 → [N,3,1080,1920] stretch (scale 1) must equal decode-then-normalise."""
    w, h, n = 1920, 1080, 2
    frame = w * h * 3 // 2
    raws = [raw_bytes(frame, k) for k in range(n)]
    pre = (kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).mode(kb.ResizeMode.Stretch)
           .normalize(kb.Normalize.imagenet()).build_cuda())
    dst = torch.zeros((n, 3, h, w), dtype=torch.float32, device=dev)
    pre.run_raw_batch([cu(r, dev) for r in raws], w, h, dst)
    inv = np.array([np.float32(1.0) / np.float32(s) for s in kb.IMAGENET_STD], np.float32)
    mean = np.array(kb.IMAGENET_MEAN, np.float32)
    for k in range(n):
        rgb = oracle.rgb_from_nv12(raws[k], w, h).astype(np.float32)
        want = ((rgb / np.float32(255.0) - mean) * inv).transpose(2, 0, 1)
        assert_f32_equal(dst[k].cpu().numpy(), want.astype(np.float32), f"3a frame {k}")
    # and the standalone decoder agrees with the decode fused in the taps
    rgb_dev = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev)
    kb.imgproc.rgb_from_nv12(cu(raws[0], dev), rgb_dev)
    np.testing.assert_array_equal(rgb_dev.numpy(), oracle.rgb_from_nv12(raws[0], w, h))


def test_interop_dlpack_and_cai(kb, dev):
    t = torch.arange(2 * 3 * 3, dtype=torch.float32, device=dev).reshape(2, 3, 3)
    im = kb.Image(t)
    cai = im.__cuda_array_interface__
    assert cai["shape"] == (2, 3, 3) and cai["typestr"] == "<f4" and cai["data"] == (t.data_ptr(), False)
    assert cai["strides"] is None and cai["version"] == 3 and isinstance(cai["stream"], int) and cai["stream"] != 0
    back = torch.from_dlpack(im)
    assert back.data_ptr() == t.data_ptr()
    im2 = kb.Image.from_dlpack(t)
    assert im2.data.data_ptr() == t.data_ptr()
    im3 = kb.Image.from_cuda_array_interface(im)
    assert im3.data.data_ptr() == t.data_ptr()
    assert kb.Image(torch.zeros(2, 2, 3, dtype=torch.uint8, device=dev)).__cuda_array_interface__["typestr"] == "|u1"
    with pytest.raises(AttributeError):
        kb.Image(torch.zeros(2, 2, 3)).__cuda_array_interface__


@pytest.mark.parametrize("w,h,n", [(64, 48, 2), (8, 2, 1), (1928, 6, 1), (72, 10, 3), (4, 2, 1), (132, 4, 2)])
@pytest.mark.parametrize("f16", [False, True])
def test_preprocess_nv12_identity_fast_path(kb, oracle, dev, w, h, n, f16):
    """Scale 1 / no pad takes the streaming NV12 kernel: every decoded value 0..255 must normalise to the same bits
    as the reference's `px / 255.0f` division, in f32 and (RNE) f16, through both frame-addressing modes."""
    frame = w * h * 3 // 2
    raws = [oracle.pattern_u8(frame, 0xABCD + k) for k in range(n)]
    raws[0][:min(frame, 512)] = np.arange(min(frame, 512)) % 256  # every Y value appears
    for mode in (kb.ResizeMode.Stretch, kb.ResizeMode.Letterbox):
        pre = (kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).mode(mode).normalize(kb.Normalize.imagenet()).build_cuda())
        dst = torch.zeros((n, 3, h, w), dtype=torch.float16 if f16 else torch.float32, device=dev)
        frames = [cu(r, dev) for r in raws]
        (pre.run_raw_batch_f16 if f16 else pre.run_raw_batch)(frames, w, h, dst)
        inv = tuple(float(np.float32(1.0) / np.float32(s)) for s in kb.IMAGENET_STD)
        cfg = oracle.PreprocessCfg(mode=oracle.STRETCH, fmt=oracle.FMT_NV12, mean=kb.IMAGENET_MEAN, inv_std=inv)
        want = np.stack([oracle.preprocess_frame(r, cfg, w, h, w, h, f16=f16) for r in raws])
        got = dst.cpu().numpy()
        if f16:
            np.testing.assert_array_equal(got.view(np.uint16), want.view(np.uint16))
        else:
            assert_f32_equal(got, want)
        # strided addressing of the same frames
        ring = torch.cat(frames)
        dst2 = torch.zeros_like(dst)
        pre.run_raw_strided(ring, frame, n, w, h, dst2, f16=f16)
        assert torch.equal(dst, dst2)


def test_div255_identity_exhaustive(kb, dev):
    """The 3-instruction `p/255` (Markstein correction with c = RN(1/255)) equals the IEEE division for EVERY
    float in [0, 256) — checked exhaustively on the device (1.13e9 inputs)."""
    from kornia_rs_b200 import _lib

    out = torch.zeros(1, dtype=torch.int64, device=dev)
    _lib.set_device(0)
    assert _lib.lib().kb200_selftest_div255(torch.cuda.current_stream(dev).cuda_stream, out.data_ptr()) == 0
    torch.cuda.synchronize()
    print("div255 mismatches:", int(out.item()))
    assert int(out.item()) == 0


def test_entry_points_are_cuda_graph_capturable(kb, oracle, dev):
    """The launchers only enqueue on the caller's stream and never allocate or synchronise, so — once warm — a sequence of
    them can be captured into a CUDA graph and replayed (the convention of the reference launchers, resize/cuda.rs:103-109;
    kornia-py captures its preprocess pipeline this way, cuda_ext/mod.rs:1726-1790)."""
    sw, sh, dw, dh = 384, 216, 128, 72
    src8 = np.stack([oracle.pattern_u8(sw * sh * 3, 0x3000 + i).reshape(sh, sw, 3) for i in range(2)])
    scale, bias = oracle.normalize_params_from_mean_std([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])
    t8 = cu(src8, dev)
    fused = torch.empty((2, 3, dh, dw), dtype=torch.float32, device=dev)
    f32 = kb.Image(cu(oracle.pattern_f32(256 * 96 * 3).reshape(96, 256, 3), dev))
    blur = kb.Image.zeros_cuda(kb.ImageSize(256, 96), 3, torch.float32, dev)
    edge = kb.Image.zeros_cuda(kb.ImageSize(256, 96), 3, torch.float32, dev)
    warped = kb.Image.zeros_cuda(kb.ImageSize(256, 96), 3, torch.float32, dev)
    H = [1.02, 0.03, -4.0, -0.03, 1.01, 2.5, 2.0e-5, 1.2e-5, 1.0]
    u8w = kb.Image.zeros_cuda(kb.ImageSize(sw, sh), 3, torch.uint8, dev, batch=2)

    def pipeline():
        kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(t8, dw, dh, scale, bias, out=fused)
        kb.imgproc.gaussian_blur(f32, blur, (5, 5), (1.5, 1.5))
        kb.imgproc.sobel(blur, edge, 3)
        kb.imgproc.warp_perspective(f32, warped, H, kb.InterpolationMode.Bilinear)
        kb.imgproc.warp_perspective_u8(kb.Image(t8), u8w, [1.0, 0.02, -3.0, -0.01, 1.0, 2.0, 1e-5, 0.0, 1.0])

    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        pipeline()                       # warm: function attributes, occupancy queries, tensor-map encoder lookup
        side.synchronize()
        want = [t.clone() for t in (fused, blur.data, edge.data, warped.data, u8w.data)]
        for t in (fused, blur.data, edge.data, warped.data, u8w.data):
            t.zero_()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            pipeline()
        for _ in range(2):
            g.replay()
        side.synchronize()
    for got, ref in zip((fused, blur.data, edge.data, warped.data, u8w.data), want):
        assert torch.equal(got, ref)


@pytest.mark.parametrize("w,h", [(8, 6), (34, 18), (1920, 22), (130, 4)])
def test_video_encode(kb, oracle, dev, w, h):
    """yuyv_from_rgb / nv12_from_rgb (Q8 BT.601 limited) — bit-exact, batched; and decode(encode(x)) runs end to end."""
    n = 3
    src = np.stack([oracle.pattern_u8(w * h * 3, 0x5150 + i).reshape(h, w, 3) for i in range(n)])
    img = kb.Image(cu(src, dev))
    yuyv = torch.full((n, w * h * 2), 0xCD, dtype=torch.uint8, device=dev)
    kb.imgproc.yuyv_from_rgb(img, yuyv)
    np.testing.assert_array_equal(yuyv.cpu().numpy(), np.stack([oracle.yuyv_from_rgb(src[i]) for i in range(n)]))
    nv12 = torch.full((n, w * h * 3 // 2), 0xCD, dtype=torch.uint8, device=dev)
    kb.imgproc.nv12_from_rgb(img, nv12)
    np.testing.assert_array_equal(nv12.cpu().numpy(), np.stack([oracle.nv12_from_rgb(src[i]) for i in range(n)]))
    back = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev, batch=n)
    kb.imgproc.rgb_from_nv12(nv12, back)
    np.testing.assert_array_equal(back.numpy(), np.stack([oracle.rgb_from_nv12(oracle.nv12_from_rgb(src[i]), w, h) for i in range(n)]))
    with pytest.raises(kb.ImageError, match="Invalid image size"):
        kb.imgproc.nv12_from_rgb(img, torch.zeros(7, dtype=torch.uint8, device=dev))


def test_bench_dump_outputs_is_the_timed_result(kb, oracle, tmp_path):
    """bench.py --dump-outputs: the same seeded sample of the headline output for any --steps, at most 64 MB, and the
    sampled elements of frame 0 equal the oracle's fused resize of frame 0's source."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for steps in (1, 2):
        out = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", str(steps), "--warmup", "1", "--no-ops", "--no-cpu",
                            "--no-e2e", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
        lines = [l for l in r.stdout.splitlines() if l.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps, r.stdout
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
        dumps.append((np.load(out / "resize_normalize_chw.npy"), np.load(out / "resize_normalize_chw_index.npy")))
    (vals, idx), (vals2, idx2) = dumps
    assert vals.dtype == np.float32 and idx.dtype == np.float64 and vals.shape == idx.shape and vals.size > 4_000_000
    assert np.array_equal(idx, idx2) and np.array_equal(vals.view(np.uint32), vals2.view(np.uint32))
    sw, sh, dw, dh = 3840, 2160, 1280, 720
    p = kb.imgproc.NormalizeParams.from_mean_std(kb.IMAGENET_MEAN, kb.IMAGENET_STD)
    want = oracle.resize_normalize_u8_to_f32_chw(oracle.pattern_u8(sw * sh * 3, 0x12345678).reshape(sh, sw, 3), dw, dh, p.scale, p.bias).reshape(-1)
    frame0 = idx < want.size
    assert frame0.sum() > 10_000
    assert_f32_equal(vals[frame0], want[idx[frame0].astype(np.int64)], "bench dump, frame 0")

