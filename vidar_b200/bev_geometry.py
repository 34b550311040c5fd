"""Geometry helpers on either side of the hot-path ops (host mirrors of reference functions).

  get_reference_points  BEVFormerEncoder.get_reference_points  (modules/encoder.py:53-92)
  point_sampling        BEVFormerEncoder.point_sampling        (modules/encoder.py:94-156) -- CUDA
                        kernel csrc/sca_glue.cu instead of a 61 MB repeat + batched matmul + masks
  coords_to_voxel_grids / get_bev_grids / get_bev_grids_3d / bev_grids_to_coordinates / bev_coords_to_grids
                        bevformer/utils/e2e_predictor_utils.py:8-45, 48-83
Index/grid generation is plain torch on the target device (no arithmetic worth a kernel).
"""
import copy

import numpy as np
import torch

from . import _lib


def get_reference_points(H, W, Z=8, num_points_in_pillar=4, dim="3d", bs=1, device="cuda", dtype=torch.float):
    if dim == "3d":
        zs = torch.linspace(0.5, Z - 0.5, num_points_in_pillar, dtype=dtype, device=device) / Z
        xs = torch.linspace(0.5, W - 0.5, W, dtype=dtype, device=device) / W
        ys = torch.linspace(0.5, H - 0.5, H, dtype=dtype, device=device) / H
        D = num_points_in_pillar
        ref = torch.stack((xs.view(1, 1, W).expand(D, H, W), ys.view(1, H, 1).expand(D, H, W),
                           zs.view(D, 1, 1).expand(D, H, W)), -1)               # [D,H,W,3]
        return ref.reshape(D, H * W, 3)[None].repeat(bs, 1, 1, 1)               # [bs,D,HW,3]
    if dim == "2d":
        ys = torch.linspace(0.5, H - 0.5, H, dtype=dtype, device=device) / H
        xs = torch.linspace(0.5, W - 0.5, W, dtype=dtype, device=device) / W
        ref_y, ref_x = torch.meshgrid(ys, xs, indexing="ij")
        ref = torch.stack((ref_x.reshape(-1), ref_y.reshape(-1)), -1)
        return ref[None].repeat(bs, 1, 1).unsqueeze(2)                          # [bs,HW,1,2]
    raise ValueError(f"dim must be '3d' or '2d', got {dim}")


def point_sampling(reference_points, pc_range, img_metas):
    """reference_points [bs, D, Q, 3] in [0,1]; img_metas: list (len bs) of dicts with 'lidar2img'
    (num_cam 4x4) and 'img_shape' -> (reference_points_cam [cams,bs,Q,D,2], bev_mask [cams,bs,Q,D] bool)."""
    _lib.require_cuda(reference_points=reference_points.contiguous())
    ref = reference_points.float().contiguous()
    lidar2img = np.asarray([m["lidar2img"] for m in img_metas])
    l2i = ref.new_tensor(lidar2img).float().contiguous()                        # [bs, cams, 4, 4]
    bs, D, Q, _ = ref.shape
    cams = l2i.shape[1]
    img_h, img_w = img_metas[0]["img_shape"][0][0], img_metas[0]["img_shape"][0][1]
    ref_cam = torch.empty((cams, bs, Q, D, 2), dtype=torch.float32, device=ref.device)
    mask = torch.empty((cams, bs, Q, D), dtype=torch.uint8, device=ref.device)
    import ctypes as C
    rng = (C.c_float * 6)(*[float(v) for v in pc_range])
    with torch.cuda.device(ref.device):
        _lib.check(_lib.lib().vidar_point_sampling(
            _lib.ptr(ref), _lib.ptr(l2i), C.cast(rng, C.c_void_p), _lib.ptr(ref_cam), _lib.ptr(mask),
            bs, D, Q, cams, float(img_h), float(img_w), _lib.stream_ptr(ref.device)))
    return ref_cam, mask.bool()


def coords_to_voxel_grids(ref_coords, bev_h, bev_w, pillar_num, pc_range):
    g = copy.deepcopy(ref_coords)
    g[..., 0] = ((g[..., 0] - pc_range[0]) / (pc_range[3] - pc_range[0])) * bev_w
    g[..., 1] = ((g[..., 1] - pc_range[1]) / (pc_range[4] - pc_range[1])) * bev_h
    g[..., 2] = ((g[..., 2] - pc_range[2]) / (pc_range[5] - pc_range[2])) * pillar_num
    return g


def get_bev_grids(H, W, bs=1, device="cuda", dtype=torch.float, offset=0.5):
    ys = torch.linspace(offset, H - (1 - offset), H, dtype=dtype, device=device)
    xs = torch.linspace(offset, W - (1 - offset), W, dtype=dtype, device=device)
    ref_y, ref_x = torch.meshgrid(ys, xs, indexing="ij")
    ref = torch.stack((ref_x.reshape(-1)[None] / W, ref_y.reshape(-1)[None] / H), -1)
    return ref.repeat(bs, 1, 1)


def bev_grids_to_coordinates(ref_grids, pc_range):
    """e2e_predictor_utils.py:8-14: [0, 1] grids -> metric x, y."""
    c = copy.deepcopy(ref_grids)
    c[..., 0:1] = c[..., 0:1] * (pc_range[3] - pc_range[0]) + pc_range[0]
    c[..., 1:2] = c[..., 1:2] * (pc_range[4] - pc_range[1]) + pc_range[1]
    return c


def bev_coords_to_grids(ref_coords, bev_h, bev_w, pc_range):
    """e2e_predictor_utils.py:16-33: metric x, y -> ([-1, 1] grids, mask of the cells off the border)."""
    g = copy.deepcopy(ref_coords)
    g[..., 0] = (g[..., 0] - pc_range[0]) / (pc_range[3] - pc_range[0])
    g[..., 1] = (g[..., 1] - pc_range[1]) / (pc_range[4] - pc_range[1])
    g = g * 2 - 1.
    x_min, x_max = 0.5 / bev_w * 2 - 1, (bev_w - 0.5) / bev_w * 2 - 1
    y_min, y_max = 0.5 / bev_h * 2 - 1, (bev_h - 0.5) / bev_h * 2 - 1
    valid = (g[..., 0:1] > x_min) & (g[..., 0:1] < x_max) & (g[..., 1:2] > y_min) & (g[..., 1:2] < y_max)
    return g, valid


def get_bev_grids_3d(H, W, Z, bs=1, device="cuda", dtype=torch.float):
    return get_reference_points(H, W, Z, Z, "3d", bs, device, dtype)


def flatten_fpn(mlvl_feats, cams_embeds=None, level_embeds=None):
    """PerceptionTransformer.get_bev_features' feature flattening (modules/transformer.py:159-179):
    list of [bs, cams, C, h, w] -> (feat_flatten [cams, sum(hw), bs, C], spatial_shapes [L,2] int64,
    level_start_index [L] int64), camera / level embeddings added when given."""
    flat, shapes = [], []
    for lvl, feat in enumerate(mlvl_feats):
        bs, cams, c, h, w = feat.shape
        f = feat.flatten(3).permute(1, 0, 3, 2)
        if cams_embeds is not None:
            f = f + cams_embeds[:, None, None, :].to(f.dtype)
        if level_embeds is not None:
            f = f + level_embeds[None, None, lvl:lvl + 1, :].to(f.dtype)
        shapes.append((h, w))
        flat.append(f)
    flat = torch.cat(flat, 2).permute(0, 2, 1, 3)
    shapes = torch.as_tensor(shapes, dtype=torch.long, device=flat.device)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    return flat, shapes, lsi


def value_from_fpn(mlvl_feats, cams_embeds, level_embeds, value_proj, num_heads):
    """Producer side of the MSDA value layout (SURVEY.md 8f-4): the `value` tensor
    MSDeformableAttention3D samples, `value_proj(feat_flatten)` viewed [bs*cams, sum(hw), H, C]
    (spatial_cross_attention.py:158-160,333-336), straight from the FPN maps.  The camera and level
    embeddings are folded into a per-(camera, level) bias,
        value = feat^T W^T + (W (cam_e + lvl_e) + b),
    and each level is one batched GEMM that reads the NCHW map transposed, so `feat_flatten`
    (190 MB at 6 x 30825 x 256) and its three elementwise passes are never materialised.
    Returns (value [bs*cams, sum(hw), num_heads, C/num_heads], spatial_shapes, level_start_index);
    rows are ordered (bs, cams) like SpatialCrossAttention's `value.permute(2,0,1,3).reshape(bs*cams, ...)`."""
    W, b = value_proj.weight, value_proj.bias
    outs, shapes = [], []
    for lvl, feat in enumerate(mlvl_feats):
        bs, cams, c, h, w = feat.shape
        e = level_embeds[lvl].to(feat.dtype).expand(cams, -1)
        if cams_embeds is not None:
            e = e + cams_embeds.to(feat.dtype)
        bias = torch.nn.functional.linear(e, W, b)                                 # [cams, C_out]
        a = feat.reshape(bs * cams, c, h * w).transpose(1, 2)                      # [bs*cams, hw, c] view of NCHW
        v = torch.baddbmm(bias.repeat(bs, 1)[:, None, :], a, W.t().expand(bs * cams, -1, -1))
        outs.append(v)
        shapes.append((h, w))
    value = torch.cat(outs, 1)
    shapes = torch.as_tensor(shapes, dtype=torch.long, device=value.device)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    return value.view(value.shape[0], value.shape[1], num_heads, -1), shapes, lsi
