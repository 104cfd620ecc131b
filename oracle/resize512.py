"""CPU ORACLE for the denoiser's 512x512 input (TEST INFRASTRUCTURE, NOT PRODUCT CODE).

The reference loader builds the conditioning image as ``cv2.resize(rgb_u8, (512, 512), INTER_LINEAR) / 255``
(datasets/doc_dataset/doc_benchmark.py:68-81 in the reference).  This restates OpenCV's fixed-point bilinear resize of uint8
images in numpy, so that the GPU kernel (dvd_b200/csrc/prep.cu) can be checked without the library:

  * coefficients per output column dx (rows dy alike, with H):
      scale = 1.0 / (512.0 / W)                         (double)
      f = float((dx + 0.5) * scale - 0.5); s = floor(f); f -= s      (float)
      columns only: s < 0 -> s = 0, f = 0;  s >= W-1 -> s = W-1, f = 0   (rows keep f; only their indices are clamped)
      c0 = rint((1 - f) * 2048), c1 = rint(f * 2048)    (round half to even)
  * horizontal pass, int32: h = P[r, s] * a0 + P[r, min(s+1, W-1)] * a1
  * vertical pass in OpenCV's SIMD form (VResizeLinearVec_32s8u):
      R = clamp((((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2, 0, 255)
  * y512[c, dy, dx] = float32(R[dy, dx, c]) / float32(255)   (an IEEE division, not a multiply by 1/255)
"""
from __future__ import annotations

import numpy as np

SIZE = 512


def _coeffs(n: int, clamp_frac: bool):
    """(i0, i1, c0, c1) integer arrays of length SIZE for a source axis of length n"""
    scale = 1.0 / (SIZE / float(n))
    f = ((np.arange(SIZE, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f)
    f = (f - s).astype(np.float32)
    s = s.astype(np.int64)
    if clamp_frac:
        lo, hi = s < 0, s >= n - 1
        f[lo | hi] = 0.0
        s = np.where(lo, 0, np.where(hi, n - 1, s))
    c0 = np.rint((np.float32(1.0) - f) * np.float32(2048.0)).astype(np.int32)
    c1 = np.rint(f * np.float32(2048.0)).astype(np.int32)
    return np.clip(s, 0, n - 1), np.clip(s + 1, 0, n - 1), c0, c1


def resize512_u8(photo_hwc: np.ndarray) -> np.ndarray:
    """uint8 HxWx3 -> uint8 512x512x3, equal to cv2.resize(photo, (512, 512), interpolation=cv2.INTER_LINEAR)"""
    p = np.asarray(photo_hwc)
    if p.dtype != np.uint8 or p.ndim != 3 or p.shape[0] < 1 or p.shape[1] < 1:
        raise ValueError(f"expected a uint8 HxWxC photo, got {p.dtype} {p.shape}")
    H, W = p.shape[:2]
    x0, x1, a0, a1 = _coeffs(W, True)
    y0, y1, b0, b1 = _coeffs(H, False)
    rows = np.unique(np.concatenate([y0, y1]))                 # only the source rows some output row reads
    src = p[rows].astype(np.int32)
    h = src[:, x0] * a0[None, :, None] + src[:, x1] * a1[None, :, None]          # [rows, 512, C]
    pos = np.searchsorted(rows, np.arange(H))
    h0, h1 = h[pos[y0]], h[pos[y1]]
    r = (((b0[:, None, None] * (h0 >> 4)) >> 16) + ((b1[:, None, None] * (h1 >> 4)) >> 16) + 2) >> 2
    return np.clip(r, 0, 255).astype(np.uint8)


def y512_from_photo(photo_hwc: np.ndarray) -> np.ndarray:
    """uint8 HxWx3 -> float32 [3, 512, 512] = resize512_u8(photo) / 255, channel-major"""
    r = resize512_u8(photo_hwc).transpose(2, 0, 1)
    return np.ascontiguousarray(r.astype(np.float32) / np.float32(255.0))
