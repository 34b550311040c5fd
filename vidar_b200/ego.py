"""Ego motion: the reference's per-frame pose alignment, from the `img_metas` of
projects/mmdet3d_plugin/datasets/nuscenes_vidar_dataset_v1.py:40-200 (row-vector convention, p' = p @ M).

  rotate_prev_bev                    the previous BEV rotated by the yaw change (`can_bus[-1]`, degrees) about
                                     `rotate_center`: PerceptionTransformer.get_bev_features
                                     (bevformer/modules/transformer.py:136-149) -- CUDA, csrc/ego.cu
  bev_shift                          its shift of the previous-BEV reference points (transformer.py:120-134)
  history_ref_to_previous_transform  ViDAR._get_history_ref_to_previous_transform (detectors/vidar.py:173-191)
  align_bev_coordinates              ViDAR._align_bev_coordnates (vidar.py:193-237): the future decoder's query grid
                                     in the target frame and its position in the previous frames (torch, one matmul)
  align_gt_points                    ViDARHeadV1._get_reference_gt_points (dense_heads/vidar_head_v1.py:94-148):
                                     GT of frame src in the coordinates of frame tgt, and the sensor origins --
                                     CUDA, csrc/ego.cu, no per-frame masks and no host sync

The rotation is forward only: in the reference the previous BEV never carries a gradient
(`backwarded_prev_frame_num` is 0 in every config, bevformer.py:44,219).
"""
import math

import numpy as np
import torch

from . import _lib, bev_geometry


def rotation_theta(angle, center, bev_h, bev_w):
    """The [3, 2] fp32 matrix torchvision's rotate(img[C, bev_h, bev_w], angle, center=center) samples with:
    `_get_inverse_affine_matrix(center_f, -angle, ...)` in double (host metadata), rounded to fp32, transposed and
    divided by [w/2, h/2] in fp32 (`_gen_affine_grid`)."""
    cx, cy = (1.0 * (c - s * 0.5) for c, s in zip(center, (bev_w, bev_h)))
    rot = math.radians(-float(angle))
    a, b, c, d = math.cos(rot), -math.sin(rot), math.sin(rot), math.cos(rot)      # zero shear, unit scale
    m = [d, -b, 0.0, -c, a, 0.0]
    m[2] += m[0] * (-cx) + m[1] * (-cy)
    m[5] += m[3] * (-cx) + m[4] * (-cy)
    m[2] += cx
    m[5] += cy
    theta = np.asarray(m, np.float32).reshape(2, 3)
    return np.ascontiguousarray(theta.T / np.asarray([0.5 * bev_w, 0.5 * bev_h], np.float32))


def rotate_prev_bev(prev_bev, angles_deg, center, bev_h, bev_w):
    """prev_bev [bs, bev_h * bev_w, C] (CUDA, channel-last), angles_deg: bs host angles (degrees, counter-clockwise
    like torchvision) -> the rotated BEV, same shape, fp32.  Nearest sampling, zero fill, exactly torchvision's
    rotate per sample (one kernel launch for the batch, no host sync)."""
    _lib.require_cuda(prev_bev=prev_bev)
    if prev_bev.requires_grad and torch.is_grad_enabled():
        raise RuntimeError("rotate_prev_bev is forward only: prev_bev requires grad (run it under torch.no_grad() "
                           "or detach the previous BEV)")
    bs, Q, ch = prev_bev.shape
    if Q != bev_h * bev_w:
        raise ValueError(f"rotate_prev_bev: prev_bev has {Q} cells, bev_h * bev_w = {bev_h * bev_w}")
    angles = np.asarray(angles_deg, np.float64).reshape(-1)
    if angles.shape[0] != bs:
        raise ValueError(f"rotate_prev_bev: {angles.shape[0]} angles for a batch of {bs}")
    src = _lib.aligned(prev_bev.float().contiguous())
    out = torch.empty_like(src)
    theta = np.ascontiguousarray(np.stack([rotation_theta(a, center, bev_h, bev_w) for a in angles]), np.float32)
    with torch.cuda.device(src.device):
        _lib.check(_lib.lib().vidar_bev_rotate_forward(_lib.ptr(src), theta.ctypes.data, _lib.ptr(out), bs, bev_h,
                                                       bev_w, ch, _lib.stream_ptr(src.device)))
    return out


def bev_shift(img_metas, grid_length, bev_h, bev_w, use_shift=True):
    """transformer.py:120-134: the ego translation `can_bus[:3]` (global) rotated into the LiDAR frame by
    inv(lidar2global_rotation), in BEV units -> float64 [bs, 2] (x, y) host array."""
    delta_global = np.array([each["can_bus"][:3] for each in img_metas])
    lidar2global_rotation = np.array([each["lidar2global_rotation"] for each in img_metas])
    delta_lidar = np.array([np.linalg.inv(lidar2global_rotation[i]) @ delta_global[i] for i in range(len(img_metas))])
    shift_y = delta_lidar[:, 1] / grid_length[0] / bev_h * use_shift
    shift_x = delta_lidar[:, 0] / grid_length[1] / bev_w * use_shift
    return np.stack([shift_x, shift_y], 1)


def history_ref_to_previous_transform(tensor, num_frames, img_metas_list):
    """vidar.py:173-191 -> [bs, num_frames, 4, 4] (dtype / device of `tensor`)."""
    return tensor.new_tensor(np.array([[m[i]["ref_lidar_to_cur_lidar"] for i in range(num_frames)]
                                       for m in img_metas_list]))


def align_bev_coordinates(frame_idx, ref_to_history, img_metas, bev_h, bev_w, pc_range):
    """vidar.py:193-237 -> (tgt_grids [bs, Q, 2] in [0, 1], aligned grids [bs, Q, num_frames, 2] in [0, 1],
    ref2future [bs, 4, 4])."""
    bs, num_frame = ref_to_history.shape[:2]
    future2ref = ref_to_history.new_tensor(np.array([m["future2ref_lidar_transform"][frame_idx] for m in img_metas]))
    ref2future = ref_to_history.new_tensor(np.array([m["ref2future_lidar_transform"][frame_idx] for m in img_metas]))
    future2ref = future2ref.unsqueeze(1).repeat(1, num_frame, 1, 1).contiguous()
    future_to_history = torch.matmul(future2ref, ref_to_history)
    bev_grids = bev_geometry.get_bev_grids(bev_h, bev_w, bs * num_frame, device=ref_to_history.device,
                                           dtype=ref_to_history.dtype)
    bev_grids = bev_grids.view(bs, num_frame, -1, 2)
    bev_coords = bev_geometry.bev_grids_to_coordinates(bev_grids, pc_range)
    aligned = torch.cat([bev_coords, torch.ones_like(bev_coords[..., :2])], -1)
    aligned = torch.matmul(aligned, future_to_history)[..., :2]
    aligned, _ = bev_geometry.bev_coords_to_grids(aligned, bev_h, bev_w, pc_range)
    aligned = ((aligned + 1) / 2.).permute(0, 2, 1, 3).contiguous()
    return bev_grids[:, -1].contiguous(), aligned, ref2future


def src_to_tgt_matrices(src_frames, tgt_frames, img_metas):
    """[bs, S, 4, 4] fp32: `total_cur2ref_lidar_transform[src] @ total_ref2cur_lidar_transform[tgt]`, an fp32
    matmul of fp32 matrices like vidar_head_v1.py:112-116."""
    out = []
    for s, t in zip(src_frames, tgt_frames):
        a = torch.from_numpy(np.array([m["total_cur2ref_lidar_transform"][s] for m in img_metas], np.float32))
        b = torch.from_numpy(np.array([m["total_ref2cur_lidar_transform"][t] for m in img_metas], np.float32))
        out.append(torch.matmul(a, b))
    return torch.stack(out, 1).numpy()


def align_gt_points(gt_points, src_frames, tgt_frames, img_metas):
    """GT points of frame src_frames[s] moved into frame tgt_frames[s], for every slot s.

    gt_points: list over the batch of CUDA [M_b, >= 4] tensors (x, y, z, ..., frame).  -> (list of [M_b, 4] views
    (x, y, z, slot) in input order, with (NaN, NaN, NaN, -1) for points of frames that have no slot; origins
    [bs, S, 3]).  `ViDARRayHead._process_gt_points` turns these into the reference's rays (stable order by slot,
    the rest padding), so both are drop-in inputs of `ViDARRayHead.loss` / `evaluate` (`batched_origin_points=`)."""
    src = [int(s) for s in np.asarray(src_frames).reshape(-1)]
    tgt = [int(t) for t in np.asarray(tgt_frames).reshape(-1)]
    if len(src) != len(tgt) or not src:
        raise ValueError(f"align_gt_points: {len(src)} source and {len(tgt)} target frames")
    if len(set(src)) != len(src):
        raise ValueError(f"align_gt_points: source frames must be distinct, got {src}")
    bs = len(gt_points)
    if bs == 0 or len(img_metas) != bs:
        raise ValueError(f"align_gt_points: {bs} point lists and {len(img_metas)} img_metas")
    for b, p in enumerate(gt_points):
        _lib.require_cuda(**{f"gt_points[{b}]": p.contiguous()})
    dev = gt_points[0].device
    S = len(src)
    # a negative source frame selects no point (the reference's `p[:, -1] == src`); its matrix is the reference's
    # Python index into the metas all the same
    slot_of_frame = np.full(max(max(src) + 1, 1), -1, np.int32)
    for s, f in enumerate(src):
        if f >= 0:
            slot_of_frame[f] = s
    mats = np.ascontiguousarray(src_to_tgt_matrices(src, tgt, img_metas), np.float32)
    offsets = np.zeros(bs + 1, np.int64)
    offsets[1:] = np.cumsum([int(p.shape[0]) for p in gt_points])
    packed = torch.cat([torch.cat([p[:, :3], p[:, -1:]], 1).float() for p in gt_points], 0).contiguous()
    out = torch.empty_like(packed)
    origins = torch.empty((bs, S, 3), dtype=torch.float32, device=dev)
    N = int(offsets[-1])
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vidar_ego_align_points(
            _lib.ptr(packed) if N else None, offsets.ctypes.data, slot_of_frame.ctypes.data, len(slot_of_frame),
            mats.ctypes.data, _lib.ptr(out) if N else None, _lib.ptr(origins), bs, S, _lib.stream_ptr(dev)))
    return [out[offsets[b]:offsets[b + 1]] for b in range(bs)], origins


def full_prev_bev_exists(img_metas):
    """vidar.py:302-314 (the reference loops over a batch of one): every frame but the first continues its
    predecessor's scene."""
    return all(bool(m[k]["prev_bev_exists"]) for m in img_metas for k in range(1, len(m)))

