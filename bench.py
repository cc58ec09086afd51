#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on BASELINE.json's config, one JSON line on stdout (rank 0).

Workload (N=1): configs[1] — "bilinear resize 3840x2160 -> 1280x720 RGB u8 -> f32, batch=64, 1xB200": the
fused u8 HWC -> f32 CHW half-pixel bilinear resize + normalise (resize/fused.rs:147), one launch per step over
the whole batch.  A "step" = one pass of that hot path over one batch of 64 synthetic frames (LCG pattern,
seed 0x12345678+n per frame, SURVEY §8(d) cfg 2).  metric = Mpix/s of DESTINATION pixels.

  value     whole-job throughput, inputs resident in HBM, CUDA-event timed on the launch stream, K steps
            bracketed by barrier + synchronize, max over ranks.  Each step streams a 1.59 GB source batch (the
            kernel addresses the 0.53 GB of rows with a non-zero weight) and writes 0.71 GB — far beyond the 126 MB L2.
  e2e       same metric through the public API with HOST (pinned) images and a host output tensor
            (kb200_resize_normalize_chw_u8_f32_host): per step the upload of the tapped source rows, the kernel and
            the download of the [64,3,720,1280] f32 result, chunked over a 3-stream ring so copies overlap compute.
  roofline  HBM-bound: algorithmic bytes per launch (4/9 of the source + the destination, SURVEY §8(d)) / mean
            launch time, against MEASURED_PEAKS.json's copy bandwidth.
  cpu_baseline  the oracle (C++ restatement of the reference CPU path — the Rust reference cannot be built
            here) timed on this box's host cores on a bounded sample.
  ops       the other hot-path kernels (configs 3, 4, 5 + extras) with their own roofline fractions.

N>1 (torchrun, one rank per GPU): every rank processes its own 64-frame batch (weak scaling), no data-path
collective; ONE NCCL broadcast of the normalisation parameters at plan creation.

`--impl reference`: the reference arm — the reference's CPU implementation of the same path (oracle port, all
host threads) on the same config/metric, bounded sample per step.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SW, SH, DW, DH, BATCH = 3840, 2160, 1280, 720, 64
IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
METRIC, UNIT = "Mpix/s (dst pixels) fused bilinear resize 4K->720p RGB u8->f32 CHW", "Mpix/s"
WORKLOAD = "configs[1]: fused bilinear resize+normalize 3840x2160->1280x720 RGB u8 HWC -> f32 CHW, batch=64 per GPU"


# stdout carries exactly ONE JSON line.  Native libraries write banners to fd 1 (NCCL prints its version there when
# NCCL_DEBUG is set in the environment), so fd 1 is pointed at stderr for the whole run and the line goes out through
# a saved duplicate of the original stdout.
_JSON_FD = None


def claim_stdout() -> None:
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(line) + "\n").encode())


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class LcgPattern:
    """cuda/color/mod.rs:303-316 pattern_u8 with a per-frame seed, vectorised: the k-th LCG state is
    A_k*seed + C_k (mod 2^32) with A_k = a^k, C_k = c*(1 + a + … + a^(k-1)); int64 cumprod/cumsum wrap mod 2^64,
    whose low 32 bits are exact mod 2^32.  A and C do not depend on the seed: computed once, reused per frame."""

    def __init__(self, n: int, device):
        import torch

        self.n = n
        self.prefix = torch.tensor([0, 255, 255, 0, 0, 0, 255, 255, 255, 1, 254, 128, 128, 128, 64], dtype=torch.uint8, device=device)[:n]
        m = max(n - 15, 0)
        a = torch.full((m,), 1664525, dtype=torch.int64, device=device)
        self.A = torch.cumprod(a, 0) & 0xFFFFFFFF                                      # a^1 … a^m
        aprev = torch.cat([torch.ones(1, dtype=torch.int64, device=device), self.A[:-1]]) if m else self.A
        self.C = (1013904223 * (torch.cumsum(aprev, 0) & 0xFFFFFFFF)) & 0xFFFFFFFF
        del a, aprev

    def frame(self, seed: int, out):
        """Writes the pattern for `seed` into the flat uint8 tensor `out` (3 kernel launches)."""
        out[:len(self.prefix)] = self.prefix
        if self.n > 15:
            out[15:] = (((self.A * (seed & 0xFFFFFFFF) + self.C) & 0xFFFFFFFF) >> 24).to(out.dtype)


def lcg_pattern_u8(n: int, seed: int, device):
    import torch

    out = torch.empty(n, dtype=torch.uint8, device=device)
    LcgPattern(n, device).frame(seed, out)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed regions run."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                clk, cmax, power = float(parts[0]), float(parts[1]), float(parts[2])
            except ValueError:
                continue
            mx.append(cmax)
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk); pw.append(power)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than a sampling period: use everything we saw
            for ts, line in self.rows:
                parts = [p.strip() for p in line.split(",")]
                try:
                    sm.append(float(parts[0]))
                except Exception:
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ─────────────────────────────────────────────────────────────────────────────
def host_threads() -> int:
    """Threads this process may actually use (cgroup / affinity aware; os.cpu_count() reports the whole host)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


_FULL_AFFINITY = None


def remember_affinity() -> None:
    global _FULL_AFFINITY
    try:
        _FULL_AFFINITY = os.sched_getaffinity(0)
    except Exception:
        _FULL_AFFINITY = None


def restore_affinity() -> None:
    """The GPU arm binds each rank to its GPU's NUMA node; the CPU legs model the reference's rayon pool on ALL host
    cores, so they run under the affinity the process started with."""
    if _FULL_AFFINITY:
        try:
            os.sched_setaffinity(0, _FULL_AFFINITY)
        except Exception:
            pass


CPU_ROTATION = 8   # distinct 4K sources in rotation (199 MB): the host L3 cannot hold them (BASELINE.md protocol)


class CpuArm:
    """The reference's CPU implementation of config 2 — the oracle port of resize_normalize_to_tensor_u8_to_f32_bilinear
    (AVX2+FMA leaf, OpenMP 8-row tasks like rayon) — with ONE procedure shared by `--impl reference` and the
    `cpu_baseline` leg: 8 rotating sources, thread count chosen once from >= 0.5 s trials per candidate."""

    def __init__(self):
        from oracle import oracle as o

        self.o = o
        self.srcs = [o.pattern_u8(SW * SH * 3, 0x12345678 + i).reshape(SH, SW, 3) for i in range(CPU_ROTATION)]
        self.scale, self.bias = o.normalize_params_from_mean_std(IMAGENET_MEAN, IMAGENET_STD)
        self.i = 0
        self.threads = self._pick_threads()

    def frame(self) -> None:
        self.o.resize_normalize_u8_to_f32_chw(self.srcs[self.i % CPU_ROTATION], DW, DH, self.scale, self.bias, self.o.LEAF_X86)
        self.i += 1

    def _rate(self, seconds: float) -> float:
        n, t0 = 0, time.perf_counter()
        while True:
            self.frame()
            n += 1
            dt = time.perf_counter() - t0
            if dt >= seconds:
                return n / dt

    def _pick_threads(self) -> int:
        avail = host_threads()
        cands = sorted({t for t in (avail, avail // 2, 64, 32, 16, 8) if 1 <= t <= avail}, reverse=True)
        best, best_r = cands[-1], 0.0
        for t in cands:
            self.o.set_threads(t)
            self._rate(0.15)            # warm the pool
            r = self._rate(0.5)
            if r > best_r:
                best, best_r = t, r
        self.o.set_threads(best)
        return best

    def describe(self, frames: int, seconds: float) -> str:
        return (f"{frames} frames of config 2 ({CPU_ROTATION} distinct 4K sources in rotation) in {seconds:.1f} s; oracle C++ port of the reference CPU "
                f"path (AVX2+FMA leaf, OpenMP {self.threads} threads, 8-row tasks like rayon)")


def run_reference_arm(args) -> None:
    """The reference's own CPU implementation of the path (the oracle's C++ port of the Rust crate), all host
    threads, same config/metric.  One step = a bounded sample (4 frames) of the batch; --steps steps are timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm()
    frames = 4  # bounded sample: 4 of the 64 frames per step

    def step():
        for _ in range(frames):
            arm.frame()

    for _ in range(max(1, min(args.warmup, 3))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = frames * DW * DH * args.steps / 1e6 / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": headline_config(args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": arm.threads, "kind": "port",
                         "sample": f"{frames} of {BATCH} frames per step; " + arm.describe(frames * args.steps, dt)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def cpu_baseline_sample(budget_s: float = 12.0) -> dict:
    arm = CpuArm()
    n, t0 = 0, time.perf_counter()
    while True:
        arm.frame()
        n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s:
            break
    return {"value": n * DW * DH / 1e6 / dt, "unit": UNIT, "cores": arm.threads, "kind": "port", "sample": arm.describe(n, dt)}


def headline_config(n_gpus: int) -> dict:
    """Identical in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "global_batch": BATCH * n_gpus, "parallelism": f"dp{n_gpus} (batch shards, no data-path collective)",
            "l2": "inputs larger than L2: each step walks a 1.59 GB source batch (0.53 GB of tapped rows read) + 0.71 GB destination",
            "leaf": "x86 AVX2+FMA leaf of the reference (bit-identical)"}


def time_launches(fn, iters: int, warmup: int, stream) -> float:
    """Mean ms per call of `fn` (CUDA events on `stream`, sync on both sides)."""
    import torch

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


H_CFG5 = [1.02, 0.03, -40.0, -0.03, 1.01, 25.0, 2.0e-6, 1.2e-6, 1.0]   # SURVEY §8(d) cfg 5


def load_ref_gpu(dev):
    """The GPU baseline (the reference's own kernels, baseline/ref_gpu.py) — None when baseline/_ref was not built."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import ref_gpu

        if not ref_gpu.available():
            return None
        return ref_gpu.RefGpu(dev.index or 0)
    except Exception as ex:  # the table must survive a missing driver binding
        log(f"[bench] reference GPU kernels unavailable: {ex!r}")
        return None


def op_table(kb, dev, peak_gbs: float, quick: bool, n_gpus: int, rank: int) -> dict:
    """Every hot-path op at N GPUs: each rank runs the op on ITS shard (weak scaling: cfg 3 = 256 frames per GPU,
    cfg 4 = 16 images per GPU, cfg 5 = 64 images per GPU — at N = 8 exactly BASELINE's 128 / 512-image configs), inputs
    from SURVEY §8(d)'s generators, CUDA events on the launch stream, MAX over ranks; Mpix/s is the whole job's.
    `ref_gpu_ms` / `vs_ref_gpu`: the reference's own CUDA kernels (NVRTC compute_100, fmad=false, 32x8 / 256-thread
    launches, one launch per image) timed on rank 0 on the SAME buffers."""
    import numpy as np
    import torch

    import ctypes as C

    def preprocess_affine(mode, sw, sh, dw, dh):        # Affine::new through the product's host helper
        a = (C.c_float * 4)()
        kb._lib.lib().kb200_preprocess_affine(0 if mode == kb.ResizeMode.Letterbox else 1, sw, sh, dw, dh, a)
        return tuple(a)

    def tapped_pixels(sw, sh, dw, dh, fused):
        """Distinct source pixels addressed by >= 1 tap (SURVEY §8(d)'s algorithmic-bytes rule), from the samplers' own
        f32 coordinate expressions (resize/mod.rs:161-179; resize/fused.rs:196-201); separable, so nx * ny."""
        def axis(s_len, d_len):
            i = np.arange(d_len, dtype=np.float32)
            a = np.float32(s_len) / np.float32(d_len)
            if fused:
                f = np.maximum((i + np.float32(0.5)) * a - np.float32(0.5), np.float32(0))
            else:
                f = np.minimum(np.maximum(a * i + (np.float32(0.5) * a - np.float32(0.5)), np.float32(0)), np.float32(s_len - 1))
            i0 = np.minimum(f.astype(np.int64), s_len - 1)
            i1 = np.minimum(i0 + 1, s_len - 1)
            return len(np.union1d(i0, i1))
        return axis(sw, dw) * axis(sh, dh)

    st = torch.cuda.current_stream(dev)
    out = {}
    ref = load_ref_gpu(dev) if rank == 0 else None
    it, wu = (5, 3) if quick else (20, 5)
    rit, rwu = (2, 1) if quick else (4, 2)

    def rec(name, fn, units_mpix, alg_bytes, batch, note="", ref_fn=None):
        kb.dist.barrier(dev)
        try:
            ms_local = time_launches(fn, it, wu, st)
        except Exception as ex:   # one failing row must not take the table down (all ranks still meet at the collectives)
            log(f"[bench] op {name} failed: {ex!r}")
            ms_local = float("nan")
        ms = kb.dist.max_over_ranks(ms_local if ms_local == ms_local else 1e30, dev)
        if not (ms < 1e29):
            out[name] = {"error": "failed on at least one rank (see stderr)"}
            kb.dist.barrier(dev)
            return
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        row = {"ms": round(ms, 4), "mpix_s": round(n_gpus * units_mpix / (ms * 1e-3), 1), "alg_gb_per_gpu": round(alg_bytes / 1e9, 4),
               "gbs_per_gpu": round(gbs, 1), "frac": round(gbs / peak_gbs, 3), "batch_per_gpu": batch, "kernel": kb._lib.last_kernel()}
        if note:
            row["note"] = note
        if ref is not None and ref_fn is not None:
            try:
                rms = time_launches(ref_fn, rit, rwu, st)
                row["ref_gpu_ms"] = round(rms, 4)
                row["vs_ref_gpu"] = round(rms / time_launches(fn, rit, rwu, st), 2)   # same-rank, same-moment ratio
            except Exception as ex:
                row["ref_gpu_error"] = repr(ex)
        kb.dist.barrier(dev)
        out[name] = row

    first = rank   # this rank's units start at global index rank * share

    # ── config 3: NV12 1080p frames, bytes ((i*7+13) % 251) + 31k (preprocess.rs:1765-1767) ────────────────────────
    w, h, n = 1920, 1080, 64 if quick else 256
    frame = w * h * 3 // 2
    base = ((torch.arange(frame, device=dev, dtype=torch.int64) * 7 + 13) % 251)
    raw = torch.empty((n, frame), dtype=torch.uint8, device=dev)
    for k in range(n):
        raw[k] = ((base + 31 * (first * n + k)) & 0xFF).to(torch.uint8)
    del base
    frames = [raw[i] for i in range(n)]
    inv_std = [float(np.float32(1.0) / np.float32(v)) for v in IMAGENET_STD]
    for tag, mode, (dw, dh), src_bytes in (("cfg3a_nv12_1080p_to_chw1080p", kb.ResizeMode.Stretch, (w, h), frame),
                                           ("cfg3b_nv12_1080p_letterbox640", kb.ResizeMode.Letterbox, (640, 640), 1958400)):
        pre = kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).mode(mode).normalize(kb.Normalize.imagenet()).build_cuda()
        dst = torch.empty((n, 3, dh, dw), dtype=torch.float32, device=dev)
        aff = preprocess_affine(mode, w, h, dw, dh)
        rec(tag, lambda: pre.run_raw_batch(frames, w, h, dst), n * dw * dh / 1e6, n * (src_bytes + 3 * dw * dh * 4), n,
            "one launch per batch; 3b source bytes = distinct tapped bytes, counted by tests/test_abi_and_host.py::test_cfg3b_algorithmic_bytes",
            ref_fn=(lambda: ref.preprocess(frames, w, h, dst, aff, IMAGENET_MEAN, inv_std, 114.0)) if ref else None)
        del dst
    rgb = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev, batch=n)
    rec("rgb_from_nv12_1080p", lambda: kb.imgproc.rgb_from_nv12(raw, rgb), n * w * h / 1e6, n * (frame + w * h * 3), n,
        ref_fn=(lambda: ref.rgb_from_nv12(raw, rgb.data, w, h)) if ref else None)
    del raw, frames, rgb

    # ── 4K f32 sources: pattern_f32 = pattern_u8 / 255, seed 0x12345678 + image index (cuda/color/mod.rs:303-321) ──
    w, h = 3840, 2160
    n5 = 8 if quick else 64          # config 5 share
    n4 = 4 if quick else 16          # config 4 share
    gen = LcgPattern(w * h * 3, dev)
    src5 = torch.empty((n5, h, w, 3), dtype=torch.float32, device=dev)
    tmp = torch.empty(w * h * 3, dtype=torch.uint8, device=dev)
    for i in range(n5):
        gen.frame(0x12345678 + first * n5 + i, tmp)
        src5[i] = (tmp.to(torch.float32) / 255.0).view(h, w, 3)
    u8src = torch.empty((n4, h, w, 3), dtype=torch.uint8, device=dev)
    for i in range(n4):
        gen.frame(0x0BADF00D + first * n4 + i, u8src[i].view(-1))
    del gen, tmp
    S5 = kb.Image(src5)
    S4 = kb.Image(src5[:n4])
    px = w * h
    full = px * 3 * 4 * 2          # src + dst bytes of one 4K f32 image

    # config 5: warp_perspective
    d5 = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.float32, dev, batch=n5)
    hinv = kb.imgproc.invert_homography(H_CFG5)
    rec("cfg5_warp_perspective_4k_f32", lambda: kb.imgproc.warp_perspective(S5, d5, H_CFG5, kb.InterpolationMode.Bilinear), n5 * px / 1e6, n5 * full, n5,
        "alg bytes = full src + dst (>= 97 % of the source is addressed)",
        ref_fn=(lambda: ref.warp("perspective", "bilinear", src5, d5.data, hinv)) if ref else None)
    del d5
    a = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.float32, dev, batch=n4)
    b = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.float32, dev, batch=n4)
    M = kb.imgproc.get_rotation_matrix2d((w / 2, h / 2), 30.0, 1.0)
    minv = kb.imgproc.invert_affine_transform(M)
    rec("warp_affine_rot30_4k_f32", lambda: kb.imgproc.warp_affine(S4, b, M, kb.InterpolationMode.Bilinear), n4 * px / 1e6, n4 * full, n4,
        ref_fn=(lambda: ref.warp("affine", "bilinear", src5[:n4], b.data, minv)) if ref else None)
    # config 4: gaussian 5x5 sigma 1.5, then sobel 3 on its output
    scratch = torch.empty((h, w, 3), dtype=torch.float32, device=dev) if ref else None
    taps = kb.imgproc.gaussian_kernel_1d(5, 1.5) if ref else None
    rec("cfg4_gaussian5x5_4k_f32", lambda: kb.imgproc.gaussian_blur(S4, a, (5, 5), (1.5, 1.5)), n4 * px / 1e6, n4 * full, n4,
        ref_fn=(lambda: ref.separable_filter(src5[:n4], b.data, scratch, taps, taps)) if ref else None)
    gx = torch.empty((1, h, w, 3), dtype=torch.float32, device=dev) if ref else None
    gy = torch.empty((1, h, w, 3), dtype=torch.float32, device=dev) if ref else None
    rec("cfg4_sobel3_4k_f32", lambda: kb.imgproc.sobel(a, b, 3), n4 * px / 1e6, n4 * full, n4,
        ref_fn=(lambda: ref.sobel(a.data, b.data, scratch, gx, gy, 3)) if ref else None)
    del scratch, gx, gy
    # a1: f32 HWC bilinear resize at three ratios (3:1 exact, 2:1 exact = the reference's published config, 2.4:1)
    for dw, dh in ((1280, 720), (1920, 1080), (1600, 900)):
        small = kb.Image.zeros_cuda(kb.ImageSize(dw, dh), 3, torch.float32, dev, batch=n4)
        tapped = tapped_pixels(w, h, dw, dh, False)
        rec(f"resize_f32_4k_to_{dw}x{dh}", lambda: kb.imgproc.resize(S4, small, kb.InterpolationMode.Bilinear), n4 * dw * dh / 1e6,
            n4 * (tapped * 12 + dw * dh * 12), n4, f"distinct tapped source pixels: {tapped}",
            ref_fn=(lambda: ref.resize_bilinear(src5[:n4], small.data)) if ref else None)
        del small
    gray = kb.Image.zeros_cuda(kb.ImageSize(w, h), 1, torch.float32, dev, batch=n4)
    rec("gray_from_rgb_f32_4k", lambda: kb.imgproc.gray_from_rgb(S4, gray), n4 * px / 1e6, n4 * px * 16, n4,
        ref_fn=(lambda: ref.gray_f32(src5[:n4], gray.data)) if ref else None)
    rec("normalize_mean_std_4k_f32", lambda: kb.imgproc.normalize_mean_std(S4, a, IMAGENET_MEAN, IMAGENET_STD), n4 * px / 1e6, n4 * px * 24, n4)
    del gray

    # a2 beyond the headline geometry: every mode of the fused u8 -> f32 CHW resize (the headline runs FR_POINT)
    sc, bi = kb.imgproc.NormalizeParams.from_mean_std(IMAGENET_MEAN, IMAGENET_STD).scale, kb.imgproc.NormalizeParams.from_mean_std(IMAGENET_MEAN, IMAGENET_STD).bias
    for tag, sw_, (dw, dh) in (("fused_resize_u8_4k_to_1080p_box2x", w, (1920, 1080)), ("fused_resize_u8_4k_to_1600x900_general", w, (1600, 900)),
                               ("fused_resize_u8_3838w_to_720p_gather_fallback", 3838, (1280, 720))):
        s8 = u8src if sw_ == w else u8src.view(n4, -1)[:, :h * sw_ * 3].contiguous().view(n4, h, sw_, 3)
        dstc = torch.empty((n4, 3, dh, dw), dtype=torch.float32, device=dev)
        tapped = tapped_pixels(sw_, h, dw, dh, True)
        rec(tag, lambda: kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(s8, dw, dh, sc, bi, out=dstc), n4 * dw * dh / 1e6,
            n4 * (tapped * 3 + dw * dh * 12), n4, f"distinct tapped source pixels: {tapped}")
        del dstc
    rec("std_mean_4k_u8", lambda: kb.imgproc.std_mean_sums(kb.Image(u8src)), n4 * px / 1e6, n4 * px * 3, n4)

    # ── SURVEY §8(f) rows: u8 twins, remap ───────────────────────────────────────────────────────────────────────
    s8 = kb.Image(u8src)
    d8 = kb.Image.zeros_cuda(kb.ImageSize(w, h), 3, torch.uint8, dev, batch=n4)
    tot = n4 * px
    half = kb.Image.zeros_cuda(kb.ImageSize(w // 2, h // 2), 3, torch.uint8, dev, batch=n4)
    rec("next_resize_fast_u8_pyrdown_4k_to_1080p", lambda: kb.imgproc.resize_fast_u8(s8, half, kb.InterpolationMode.Bilinear), tot / 4 / 1e6, tot * 3 + tot * 3 // 4, n4)
    third = kb.Image.zeros_cuda(kb.ImageSize(w // 3, h // 3), 3, torch.uint8, dev, batch=n4)
    rec("next_resize_fast_u8_4k_to_720p", lambda: kb.imgproc.resize_fast_u8(s8, third, kb.InterpolationMode.Bilinear), tot / 9 / 1e6, tot * 3 * 4 // 9 + tot * 3 // 9, n4,
        "u8 twin of config 2 (4/9 of the source + destination)")
    del third, half
    rec("next_warp_perspective_u8_4k", lambda: kb.imgproc.warp_perspective_u8(s8, d8, H_CFG5), tot / 1e6, tot * 6, n4)
    rec("next_warp_affine_u8_rot30_4k", lambda: kb.imgproc.warp_affine_u8(s8, d8, M), tot / 1e6, tot * 6, n4)
    rec("next_gaussian_blur_u8_5x5_4k", lambda: kb.imgproc.gaussian_blur_u8(s8, d8, (5, 5), (1.5, 1.5)), tot / 1e6, tot * 6, n4)
    yy, xx = torch.meshgrid(torch.arange(h, device=dev, dtype=torch.float32), torch.arange(w, device=dev, dtype=torch.float32), indexing="ij")
    r2 = ((xx - w / 2) ** 2 + (yy - h / 2) ** 2) / float(w * w)
    mx = kb.Image((w / 2 + (xx - w / 2) * (1 + 0.05 * r2)).unsqueeze(-1).contiguous())
    my = kb.Image((h / 2 + (yy - h / 2) * (1 + 0.05 * r2)).unsqueeze(-1).contiguous())
    del yy, xx, r2
    rec("next_remap_u8_4k", lambda: kb.imgproc.remap_u8(s8, d8, mx, my, kb.InterpolationMode.Bilinear), tot / 1e6, tot * 6 + px * 8, n4, "radial-distortion map shared by the batch")
    rec("next_remap_f32_4k", lambda: kb.imgproc.remap(S4, a, mx, my, kb.InterpolationMode.Bilinear), tot / 1e6, tot * 24 + px * 8, n4,
        ref_fn=(lambda: ref.remap(src5[:n4], a.data, mx.data, my.data)) if ref else None)
    return out


DUMP_DRAWS = 1 << 22   # draws of the output sample: ~4.15 M distinct elements, ~50 MB of .npy


def dump_outputs(out_dir: str, dst) -> None:
    """--dump-outputs: a fixed sample of the headline output `dst` ([BATCH, 3, DH, DW] f32).  The element indices come
    from a seeded generator, so two runs (or two builds) write the same elements and compare value for value:
    resize_normalize_chw.npy holds the values (f32), resize_normalize_chw_index.npy their flat indices into `dst`
    (f64, exact for any index below 2^53)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    idx = np.unique(np.random.default_rng(0).integers(0, dst.numel(), DUMP_DRAWS))
    vals = dst.reshape(-1)[torch.from_numpy(idx).to(dst.device)].cpu().numpy()
    np.save(os.path.join(out_dir, "resize_normalize_chw.npy"), vals.astype(np.float32))
    np.save(os.path.join(out_dir, "resize_normalize_chw_index.npy"), idx.astype(np.float64))


def e2e_config3(kb, dev, st, n: int, steps: int, n_gpus: int) -> dict:
    import torch

    w, h = 1920, 1080
    frame = w * h * 3 // 2
    base = ((torch.arange(frame, dtype=torch.int64) * 7 + 13) % 251)
    host = torch.empty((n, frame), dtype=torch.uint8, pin_memory=True)
    for k in range(n):
        host[k] = ((base + 31 * (kb.dist.rank() * n + k)) & 0xFF).to(torch.uint8)
    pre = kb.Preprocessor.builder().source_format(kb.SourceFormat.Nv12).mode(kb.ResizeMode.Stretch).normalize(kb.Normalize.imagenet()).build_cuda()
    chunk = 8
    out = {}
    for tag, f16 in (("f32", False), ("f16", True)):
        esz = 2 if f16 else 4
        pipe = kb.imgproc.HostPipeline(dev, src_chunk_bytes=chunk * (frame + 16), dst_chunk_bytes=chunk * 3 * w * h * esz, depth=3)
        dst = torch.empty((n, 3, h, w), dtype=torch.float16 if f16 else torch.float32, pin_memory=True)
        fn = lambda: pre.run_raw_host(host, w, h, (w, h), out=dst, f16=f16, pipeline=pipe)
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        kb.dist.barrier(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(steps):
            fn()
        e1.record(st)
        torch.cuda.synchronize()
        kb.dist.barrier(dev)
        ms = kb.dist.max_over_ranks(e0.elapsed_time(e1), dev) / steps
        h2d, d2h = pipe.last_transfer()
        # spot check against the device-buffer path
        dev_dst = torch.empty((2, 3, h, w), dtype=dst.dtype, device=dev)
        (pre.run_raw_batch_f16 if f16 else pre.run_raw_batch)([host[i].to(dev) for i in range(2)], w, h, dev_dst)
        same = bool(torch.equal(dev_dst.cpu(), dst[:2]))
        pipe.close()
        out[tag] = {"value": n_gpus * n * w * h / 1e6 / (ms * 1e-3), "unit": "Mpix/s", "ms_per_step": ms, "frames_per_gpu": n, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "h2d_gbs_per_rank": round(h2d / ms / 1e6, 1), "d2h_gbs_per_rank": round(d2h / ms / 1e6, 1),
                    "matches_device_result": same}
        del dst, dev_dst
    out["how"] = ("Preprocessor.run_raw_host (kb200_preprocess_host): NV12 1080p frames from pinned host memory -> [N,3,1080,1920] host tensor; "
                  f"chunks of {chunk} frames over a 3-stream ring, one fused launch per chunk")
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-ops", action="store_true", help="skip the per-op table")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline sample")
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="tuning sweeps only: skip the host-buffer (e2e) leg; the line then has e2e = null")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed, seeded sample of the output of the last timed step (rank 0) to DIR as .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    claim_stdout()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch

    import kornia_rs_b200 as kb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback on the product path)")
    remember_affinity()
    dev = kb.dist.init_from_env()      # binds this rank to its GPU's NUMA node before any pinned allocation
    rank, ws = kb.dist.rank(), kb.dist.world_size()
    if ws != args.gpus and ws > 1:
        log(f"[bench] WORLD_SIZE={ws} differs from --gpus={args.gpus}; using WORLD_SIZE")
    n_gpus = ws
    st = torch.cuda.current_stream(dev)
    peak_gbs, peak_src = measured_peak_gbs()

    # plan creation: ONE broadcast of the parameter block (normalisation scale/bias) from rank 0
    p = kb.imgproc.NormalizeParams.from_mean_std(IMAGENET_MEAN, IMAGENET_STD)
    params = kb.dist.broadcast_params({"scale": p.scale, "bias": p.bias}, device=dev)
    scale, bias = params["scale"], params["bias"]

    # this rank's shard of the image stream: its own 64-frame batch (weak scaling)
    shard = kb.dist.shard_range(BATCH * n_gpus, rank, n_gpus)
    src = torch.empty((BATCH, SH, SW, 3), dtype=torch.uint8, device=dev)
    gen = LcgPattern(SW * SH * 3, dev)
    for i in range(BATCH):
        gen.frame(0x12345678 + shard.start + i, src[i].view(-1))
    del gen
    dst = torch.empty((BATCH, 3, DH, DW), dtype=torch.float32, device=dev)
    fn = lambda: kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(src, DW, DH, scale, bias, out=dst)

    sampler = ClockSampler(dev.index or 0) if rank == 0 else None
    for _ in range(args.warmup):
        fn()
    kb.dist.barrier(dev)
    torch.cuda.synchronize()
    t_wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(args.steps):
        fn()
    e1.record(st)
    torch.cuda.synchronize()
    kb.dist.barrier(dev)
    ms_total = kb.dist.max_over_ranks(e0.elapsed_time(e1), dev)
    ms_step = ms_total / args.steps
    dst_mpix_step = BATCH * DW * DH / 1e6 * n_gpus
    value = dst_mpix_step / (ms_step * 1e-3)

    # roofline of the dominant (only) kernel: algorithmic bytes per launch / mean launch duration on this rank
    alg_bytes = BATCH * (SW * SH * 3 * 4 // 9 + DW * DH * 3 * 4)  # 22,118,400 B/frame (SURVEY §8(d) cfg 2)
    ms_launch = e0.elapsed_time(e1) / args.steps
    achieved = alg_bytes / (ms_launch * 1e-3) / 1e9
    # dram bytes of this kernel from the committed ncu --set full capture — only if the capture was taken from the
    # kernel source that is running now (hash recorded with it); a stale capture reports null, never a stale number
    traffic, traffic_src = None, "no ncu capture recorded for the current kernel source"
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            import hashlib

            tj = json.load(open(tpath))
            cur = hashlib.sha256(open(os.path.join(ROOT, "kornia-rs_b200", "csrc", "resize_fused.cu"), "rb").read()).hexdigest()[:16]
            if tj.get("fused_resize_cfg2_source_sha16") == cur:
                traffic = tj.get("fused_resize_cfg2_bytes_per_launch")
                traffic_src = tj.get("fused_resize_cfg2_capture", "profiles/traffic.json")
        except Exception:
            traffic = None

    e2e = None
    t_wall1 = time.time()
    if not args.no_e2e:
        # e2e: the operator called with HOST (pinned) images and a host output tensor — kb200_resize_normalize_chw_u8_f32_host:
        # per step, upload -> kernel -> download of the whole batch inside the timed region, chunked over a 3-stream ring.
        chunk, nstreams = 8, 3
        host_src = torch.empty((BATCH, SH, SW, 3), dtype=torch.uint8, pin_memory=True)
        host_src.copy_(src)
        host_dst = torch.empty((BATCH, 3, DH, DW), dtype=torch.float32, pin_memory=True)
        pipe = kb.imgproc.HostPipeline(dev, src_chunk_bytes=chunk * SW * SH * 3, dst_chunk_bytes=chunk * 3 * DW * DH * 4, depth=nstreams)

        def e2e_step():
            kb.imgproc.resize_normalize_to_tensor_u8_to_f32_bilinear(host_src, DW, DH, scale, bias, out=host_dst, pipeline=pipe)

        e2e_steps = max(2, min(args.steps, 10))
        for _ in range(2):
            e2e_step()
        torch.cuda.synchronize()
        kb.dist.barrier(dev)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(st)
        for _ in range(e2e_steps):
            e2e_step()
        s1.record(st)
        torch.cuda.synchronize()
        kb.dist.barrier(dev)
        e2e_ms = kb.dist.max_over_ranks(s0.elapsed_time(s1), dev) / e2e_steps
        e2e_value = dst_mpix_step / (e2e_ms * 1e-3)
        t_wall1 = time.time()
        # spot-check: the e2e result equals the device-resident result
        same = bool(torch.equal(host_dst.to(dev), dst))
        h2d_step, d2h_step = pipe.last_transfer()
        row_map = kb.imgproc.resize_row_plan(SH, DH)
        pipe.close()
        del host_src, host_dst
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": d2h_step,
               "ms_per_step": e2e_ms, "steps": e2e_steps, "matches_device_result": same,
               "h2d_gbs_per_rank": round(h2d_step / (e2e_ms * 1e-3) / 1e9, 1), "d2h_gbs_per_rank": round(d2h_step / (e2e_ms * 1e-3) / 1e9, 1),
               "numa": kb.dist.numa_binding(),
               "host_src_bytes_per_step": BATCH * SW * SH * 3, "row_map": list(row_map),
               "how": f"kb200_resize_normalize_chw_u8_f32_host on pinned host buffers: chunks of <= {chunk} frames over a {nstreams}-stream ring "
                      f"(strided upload of the tapped source rows only — period/first/keep = {row_map} — kernel, download)"}
        # config 3 end to end: raw NV12 camera frames in HOST memory -> normalised CHW tensor in HOST memory through
        # Preprocessor.run_raw_host (kb200_preprocess_host): f32, and the reference's f16 output (preprocess.rs:1086) which
        # halves the download — the larger half of the link traffic
        e2e["config3"] = e2e_config3(kb, dev, st, 16 if args.quick else 64, max(2, min(args.steps, 6)), n_gpus)
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs and rank == 0:   # dst still holds the last timed step's result: the e2e leg writes host buffers
        dump_outputs(args.dump_outputs, dst)
    del src, dst

    ops = None
    if not args.no_ops:   # every rank takes part (each op is timed on every shard, max over ranks)
        try:
            ops = op_table(kb, dev, peak_gbs, args.quick, n_gpus, rank)
        except Exception as ex:  # the headline must survive an op failing
            import traceback

            log(traceback.format_exc())
            ops = {"error": repr(ex)}
    cpu = None
    if rank == 0 and not args.no_cpu and n_gpus == 1:
        restore_affinity()
        try:
            cpu = cpu_baseline_sample(4.0 if args.quick else 12.0)
        except Exception as ex:
            cpu = {"error": repr(ex)}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": headline_config(n_gpus),
            "e2e": e2e,
            "gpu_launches": args.steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "frac_of_traffic": (traffic / (ms_launch * 1e-3) / 1e9 / peak_gbs) if traffic else None,
                         "note": "algorithmic bytes count all four taps per pixel (SURVEY 8(d)); at 3:1 three have weight exactly 0 and are "
                                 "not fetched, so the bytes moved (traffic) are below the algorithmic bytes and frac can exceed 1; "
                                 "frac_of_traffic = bytes actually moved / time / peak",
                         "peak_source": peak_src, "kernel": "fused_rows_kernel (resize_fused.cu)",
                         "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": ms_launch},
            "clocks": clocks,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if ops is not None:
            line["ops"] = ops
        emit(line)
    if kb.dist.is_initialized():
        import torch.distributed as td

        td.destroy_process_group()


if __name__ == "__main__":
    main()
