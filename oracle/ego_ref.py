"""Numpy restatement of the ego-motion ops (test infrastructure; pinned to the reference's own code by
tests/test_ego_cpu.py through tests/golden/ego.npz).

  rotate           torchvision.transforms.functional.rotate(img[C, H, W], angle, center) with its defaults
                   (nearest, expand=False, zero fill), as PerceptionTransformer.get_bev_features calls it, plus the
                   cells whose fp64 source coordinate lies within `tol` px of a rounding / zero-fill boundary
  align_points     ViDARHeadV1._get_reference_gt_points for one sample, in input order (x, y, z, slot), with
                   (NaN, NaN, NaN, -1) for points of frames without a slot, and the sensor origins
"""
import math

import numpy as np


def inverse_affine(center, angle, width, height):
    """torchvision's rotate -> _get_inverse_affine_matrix(center_f, -angle, [0, 0], 1.0, [0, 0]) in double."""
    center_f = [1.0 * (c - s * 0.5) for c, s in zip(center, [width, height])]
    rot = math.radians(-angle)
    sx = sy = 0.0
    cx, cy = center_f
    a = math.cos(rot - sy) / math.cos(sy)
    b = -math.cos(rot - sy) * math.tan(sx) / math.cos(sy) - math.sin(rot)
    c = math.sin(rot - sy) / math.cos(sy)
    d = -math.sin(rot - sy) * math.tan(sx) / math.cos(sy) + math.cos(rot)
    m = [d, -b, 0.0, -c, a, 0.0]
    m[2] += m[0] * (-cx) + m[1] * (-cy)
    m[5] += m[3] * (-cx) + m[4] * (-cy)
    m[2] += cx
    m[5] += cy
    return m


def rescaled_theta(angle, center, height, width):
    """_gen_affine_grid's `theta.transpose(1, 2) / [0.5 w, 0.5 h]` in fp32 -> [3, 2]."""
    theta = np.asarray(inverse_affine(center, angle, width, height), np.float32).reshape(2, 3)
    return theta.T / np.asarray([0.5 * width, 0.5 * height], np.float32)


def source_coords(angle, center, height, width):
    """fp64 unnormalised source coordinates (x, y) [H, W] of every output cell for the fp32 θ."""
    r = rescaled_theta(angle, center, height, width).astype(np.float64)
    bx = np.arange(width, dtype=np.float64) - width * 0.5 + 0.5
    by = np.arange(height, dtype=np.float64) - height * 0.5 + 0.5
    bx, by = np.meshgrid(bx, by)
    gx = bx * r[0, 0] + by * r[1, 0] + r[2, 0]
    gy = bx * r[0, 1] + by * r[1, 1] + r[2, 1]
    return ((gx + 1) * width - 1) / 2, ((gy + 1) * height - 1) / 2


def _gather(img, ix, iy):
    C, H, W = img.shape
    ok = (ix >= 0) & (ix <= W - 1) & (iy >= 0) & (iy <= H - 1)
    xi = np.where(ok, ix, 0).astype(np.int64)
    yi = np.where(ok, iy, 0).astype(np.int64)
    return np.where(ok[None], img[:, yi, xi], 0).astype(img.dtype)


def rotate(img, angle, center, tol=1e-3):
    """img [C, H, W] -> (rotated [C, H, W], near [H, W] bool: cells within `tol` px of a boundary, candidates
    [4, C, H, W]: the outputs for the source coordinate moved by +-tol in x and y)."""
    C, H, W = img.shape
    r = rescaled_theta(angle, center, H, W)
    bx = (np.arange(W, dtype=np.float32) - np.float32(W * 0.5) + np.float32(0.5))
    by = (np.arange(H, dtype=np.float32) - np.float32(H * 0.5) + np.float32(0.5))
    bx, by = np.meshgrid(bx, by)
    gx = (bx * r[0, 0] + by * r[1, 0]) + r[2, 0]
    gy = (bx * r[0, 1] + by * r[1, 1]) + r[2, 1]
    ix = np.rint(((gx + np.float32(1)) * np.float32(W) - np.float32(1)) / np.float32(2))
    iy = np.rint(((gy + np.float32(1)) * np.float32(H) - np.float32(1)) / np.float32(2))
    out = _gather(img, ix, iy)
    x64, y64 = source_coords(angle, center, H, W)
    dx = np.abs(x64 - np.floor(x64) - 0.5)
    dy = np.abs(y64 - np.floor(y64) - 0.5)
    near = (dx < tol) | (dy < tol)
    cands = np.stack([_gather(img, np.rint(x64 + sx), np.rint(y64 + sy)) for sx in (-tol, tol) for sy in (-tol, tol)])
    return out, near, cands


def align_points(points, slot_of_frame, mats):
    """points [M, 4] (x, y, z, frame), slot_of_frame {frame: slot}, mats [S, 4, 4] fp32 (p' = p @ M)
    -> (out [M, 4] float32, origins [S, 3])."""
    points = np.asarray(points, np.float32)
    mats = np.asarray(mats, np.float32)
    out = np.full((points.shape[0], 4), np.nan, np.float32)
    out[:, 3] = -1
    for f, s in slot_of_frame.items():
        sel = points[:, 3] == f
        h = np.concatenate([points[sel, :3], np.ones((int(sel.sum()), 1), np.float32)], 1)
        out[sel, :3] = (h @ mats[s])[:, :3]
        out[sel, 3] = s
    origins = np.stack([(np.array([0, 0, 0, 1], np.float32) @ m)[:3] for m in mats])
    return out, origins
