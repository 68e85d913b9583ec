"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the NV12 input contract (FM_FLAG_NV12): an NV12 frame behaves as if
it had been converted by cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12).

An NV12 frame is (H + H/2) x W bytes: the H luma rows, then H/2 rows of interleaved U, V bytes (U first).  Pixel
(x, y) takes U, V from UV row y >> 1, bytes 2 (x >> 1) and 2 (x >> 1) + 1, and cv2 converts in BT.601 fixed point:
  y' = max(Y - 16, 0) * 1220542;  u = U - 128;  v = V - 128
  R = sat((y' + 1673527 v + 2^19) >> 20)
  G = sat((y' - 852492 v - 409993 u + 2^19) >> 20)
  B = sat((y' + 2116026 u + 2^19) >> 20)
(csrc/fm_device.cuh, fm_nv12_bgr).  Checked against cv2 by tests/test_nv12_oracle.py.
"""
from __future__ import annotations

import numpy as np

CY, CVR, CVG, CUG, CUB = 1220542, 1673527, -852492, -409993, 2116026


def bgr_from_nv12(nv: np.ndarray) -> np.ndarray:
    """[H * 3 // 2, W] uint8 NV12 -> [H, W, 3] uint8 BGR."""
    H, W = nv.shape[0] * 2 // 3, nv.shape[1]
    assert nv.shape == (H * 3 // 2, W) and W % 2 == 0 and H % 2 == 0
    Y = nv[:H].astype(np.int32)
    UV = nv[H:].reshape(H // 2, W // 2, 2).astype(np.int32)
    u = np.repeat(np.repeat(UV[..., 0] - 128, 2, 0), 2, 1)
    v = np.repeat(np.repeat(UV[..., 1] - 128, 2, 0), 2, 1)
    y = np.maximum(Y - 16, 0) * CY                     # every term fits an int32
    r = (y + CVR * v + (1 << 19)) >> 20
    g = (y + CVG * v + CUG * u + (1 << 19)) >> 20
    b = (y + CUB * u + (1 << 19)) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def nv12_from_bgr(bgr: np.ndarray) -> np.ndarray:
    """[..., H, W, 3] BGR -> [..., H * 3 // 2, W] NV12 through cv2's I420 (COLOR_BGR2YUV_I420), chroma interleaved:
    the synthetic decoder output of the GPU tests."""
    import cv2
    lead = bgr.shape[:-3]
    H, W = bgr.shape[-3:-1]
    flat = bgr.reshape((-1, H, W, 3))
    out = np.empty((flat.shape[0], H * 3 // 2, W), np.uint8)
    for i, f in enumerate(flat):
        yuv = cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)
        q = (H // 2) * (W // 2)                     # the U plane, then the V plane (not whole rows of W when H/2 is odd)
        U, V = yuv[H:].reshape(-1)[:q].reshape(H // 2, W // 2), yuv[H:].reshape(-1)[q:].reshape(H // 2, W // 2)
        out[i, :H] = yuv[:H]
        out[i, H:] = np.stack([U, V], -1).reshape(H // 2, W)
    return out.reshape(lead + (H * 3 // 2, W))


def exhaustive_planes():
    """One NV12 frame (W = 512, H = 64 * 512) holding every (Y, U, V) triple once: 256 x 256 chroma blocks per 512-row
    band cover all (U, V) pairs, and the 4 luma bytes of the blocks of band k are 4k .. 4k + 3."""
    W = Hb = 512
    u, v = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    uv = np.stack([u, v], -1).reshape(Hb // 2, W)
    Y = np.empty((64 * Hb, W), np.uint8)
    for k in range(64):
        q = np.array([[4 * k, 4 * k + 1], [4 * k + 2, 4 * k + 3]], np.uint8)
        Y[k * Hb:(k + 1) * Hb] = np.tile(q, (Hb // 2, W // 2))
    return np.concatenate([Y, np.tile(uv, (64, 1))], 0)
