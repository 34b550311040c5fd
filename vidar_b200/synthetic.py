"""Seeded synthetic workloads of the hot path (SURVEY.md 8d): the BASELINE.json configurations as
tensors.  Used by bench.py, __graft_entry__.smoke(), tools/ and the tests -- there is no dataset
and no checkpoint in this tier, so the workload generators are part of the package.

  sca_like_inputs    configs[1]: MSDA operands at the SpatialCrossAttention shape
  dvr_inputs_lidar   configs[2]: sigma volume + LiDAR-like rays
  camera_rig         cfg4: a nuScenes-like 6-camera rig (lidar2img matrices) for point_sampling
  ego_queue          a vehicle on a curved path through a static world: the reference's `img_metas` of one
                     training / test queue and the LiDAR returns of every frame
"""
import math

import numpy as np
import torch

SCA_LEVELS = ((116, 200), (58, 100), (29, 50), (15, 25))   # 928x1600 input, strides 8..64
IMG_HW = (928, 1600)


def level_tensors(levels, device="cpu"):
    shapes = torch.tensor(levels, dtype=torch.int64, device=device)
    hw = shapes[:, 0] * shapes[:, 1]
    lsi = torch.cat([hw.new_zeros(1), hw.cumsum(0)[:-1]])
    return shapes, lsi


def sca_like_inputs(device, cams=6, Q=40000, seed=0, levels=SCA_LEVELS, heads=8, head_dim=32, points=8,
                    rows=None):
    """Every camera sees a fan of Q pillars of its own frustum: perspective projection of a
    sqrt(Q) x sqrt(Q) polar BEV patch with 4 Z-anchors (-4,-2,0,2 m, camera at 1.5 m), f = 1266 px
    on a 1600x928 image, plus N(0, 4 px) learned-offset noise per (head, level, point)
    (SURVEY.md 8d cfg2).  Bottom anchors of near pillars fall outside the image, as in the real rig.
    `rows`: keep only the first `rows` queries of every camera (the "rebatched" mode, 10240)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    L, P, H = len(levels), points, heads
    K = sum(h * w for h, w in levels)
    n = int(math.isqrt(Q))
    assert n * n == Q
    iy, ix = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
    depth = 2.0 + 49.0 * (iy.reshape(-1).float() + 0.5) / n               # 2 .. 51 m
    ang = ((ix.reshape(-1).float() + 0.5) / n - 0.5) * math.radians(60.0)
    u = 0.5 + torch.tan(ang) * 1266.0 / 1600.0
    zs = torch.tensor([-4.0, -2.0, 0.0, 2.0])
    v = (491.0 + 1266.0 * (1.5 - zs)[None, :] / depth[:, None]) / 928.0    # [Q, 4]
    ref = torch.stack([u[:, None].expand(-1, 4), v], -1)                   # [Q, 4(z), 2]
    ref = ref[None].expand(cams, -1, -1, -1).clone()
    ref += 0.01 * torch.randn(cams, 1, 1, 2, generator=g)                  # per-camera jitter
    if rows is not None:
        # rebatched mode: a camera keeps an evenly strided subset of its pillars
        keep = torch.linspace(0, Q - 1, rows).round().long()
        ref, Q = ref[:, keep].contiguous(), rows
    ref = ref.to(device)
    wh = torch.tensor([[w, h] for h, w in levels], dtype=torch.float32, device=device)
    dg = torch.Generator(device=device).manual_seed(seed + 1)
    off = 4.0 * torch.randn(cams, Q, H, L, P, 2, device=device, generator=dg) / wh.view(1, 1, 1, L, 1, 2)
    # point p = j*4 + z uses Z-anchor z (spatial_cross_attention.py:356-371)
    loc = off.view(cams, Q, H, L, P // 4, 4, 2) + ref.view(cams, Q, 1, 1, 1, 4, 2)
    loc = loc.view(cams, Q, H, L, P, 2).contiguous()
    attn = torch.softmax(torch.randn(cams, Q, H, L * P, device=device, generator=dg), -1)
    attn = attn.view(cams, Q, H, L, P).contiguous()
    value = torch.randn(cams, K, H, head_dim, device=device, generator=dg)
    grad_out = torch.randn(cams, Q, H * head_dim, device=device, generator=dg)
    shapes, lsi = level_tensors(levels, device)
    return dict(value=value, shapes=shapes, lsi=lsi, loc=loc, attn=attn, grad_out=grad_out)


def dvr_inputs_lidar(M=30000, T=3, grid=(16, 200, 200), seed=0, N=1, pad=0):
    """BASELINE.json configs[2]: sigma [N,T,16,200,200] = softplus(N(0,1)), origin ~ grid centre,
    32-beam LiDAR-like endpoints, range U(2,70) m at 0.512 m/voxel (SURVEY.md 8d cfg3)."""
    rng = np.random.default_rng(seed)
    Z, Y, X = grid
    sigma = np.log1p(np.exp(rng.standard_normal((N, T, Z, Y, X)))).astype(np.float32)
    origin = (np.array([X / 2, Y / 2, Z * 5.0 / 8.0]) + rng.normal(0, 0.5, (N, T, 3))).astype(np.float32)
    beams = np.deg2rad(np.linspace(-30, 10, 32))
    elev = beams[rng.integers(0, 32, (N, M))]
    azim = rng.uniform(-np.pi, np.pi, (N, M))
    rng_m = rng.uniform(2, 70, (N, M)) / 0.512
    tindex = (np.arange(M) * T // M).astype(np.float32)[None].repeat(N, 0)
    d = np.stack([np.cos(elev) * np.cos(azim), np.cos(elev) * np.sin(azim),
                  np.sin(elev) * (Z / 8.0) / (X / 102.4)], -1)  # z voxels are 0.5 m, x/y 0.512 m
    o_per_ray = np.take_along_axis(origin, tindex.astype(np.int64)[..., None].repeat(3, -1), 1)
    points = (o_per_ray + d * rng_m[..., None]).astype(np.float32)
    if pad:
        points[:, -pad:] = np.nan
        tindex[:, -pad:] = -1
    return sigma, origin, points, tindex


def camera_rig(cams=6, img_hw=(900, 1600), f=1266.0, pp=(816.0, 491.0), cam_height=1.5, seed=0):
    """lidar2img [cams,4,4] (float32) of a nuScenes-like rig (SURVEY.md 8d cfg4): yaw
    {0, +-55, +-110, 180} deg, focal 1266 px, principal point (816, 491), cameras 1.5 m above the
    LiDAR origin plane and ~1 m out from the centre, so each BEV pillar projects into 1-2 cameras."""
    yaws = np.deg2rad([0.0, 55.0, -55.0, 110.0, -110.0, 180.0])[:cams]
    rng = np.random.default_rng(seed)
    K = np.array([[f, 0, pp[0], 0], [0, f, pp[1], 0], [0, 0, 1, 0], [0, 0, 0, 1]], np.float64)
    # camera axes in the LiDAR frame: z forward, x right, y down
    mats = []
    for yaw in yaws:
        yaw = yaw + rng.normal(0, 0.01)
        fwd = np.array([np.cos(yaw), np.sin(yaw), 0.0])
        right = np.array([np.sin(yaw), -np.cos(yaw), 0.0])
        down = np.array([0.0, 0.0, -1.0])
        R = np.stack([right, down, fwd], 0)                 # rows: camera axes
        pos = fwd * 1.0 + np.array([0, 0, cam_height])
        E = np.eye(4)
        E[:3, :3] = R
        E[:3, 3] = -R @ pos
        mats.append(K @ E)
    return torch.from_numpy(np.stack(mats, 0).astype(np.float32))


def _yaw_matrix(yaw):
    c, s = math.cos(yaw), math.sin(yaw)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def _yaw_quaternion(yaw):
    return np.array([math.cos(yaw / 2), 0.0, 0.0, math.sin(yaw / 2)])          # (w, x, y, z)


def _transform_matrix(translation, rotation, inverse=False):
    """nuscenes.utils.geometry_utils.transform_matrix with a rotation matrix in place of the quaternion."""
    m = np.eye(4)
    if inverse:
        m[:3, :3] = rotation.T
        m[:3, 3] = -rotation.T @ np.asarray(translation)
    else:
        m[:3, :3] = rotation
        m[:3, 3] = translation
    return m


def ego_queue(bs=1, T=4, future=4, speed=8.0, yaw_rate=0.15, seed=0, dt=0.5, points_per_frame=2000, cams=6,
              img_hw=IMG_HW, world_points=None, max_range=60.0):
    """A vehicle drives a curved path (`speed` m/s, `yaw_rate` rad/s, one frame every `dt` s) through a static
    synthetic world.  Queue frame i = 0 .. T - 1 + future: T - 1 history frames, the current frame T - 1 and
    `future` future frames, like `previous_queue[:-1] + future_queue` of
    projects/mmdet3d_plugin/datasets/nuscenes_vidar_dataset_v1.py.  Every sample starts from its own pose and
    speed.

    -> dict(img_metas, gt_points): img_metas[b][t] for the T input frames with the keys and meanings of
    `union2one` (nuscenes_vidar_dataset_v1.py:40-200) and `get_data_info` (nuscenes_dataset.py:153-225):
    `can_bus` (18: deltas of position and yaw against the previous frame, the first frame zeroed),
    `lidar2global_rotation`, `prev_bev_exists`, `ref_lidar_to_cur_lidar`, `lidar2img`, `img_shape`, the poses;
    the current frame additionally `future_can_bus`, `future2ref_lidar_transform`, `ref2future_lidar_transform`,
    `total_cur2ref_lidar_transform` and `total_ref2cur_lidar_transform` (row-vector convention, p' = p @ M).
    gt_points[b]: float32 [M, 4] = the LiDAR returns of the static world from each frame's pose, in that frame's
    LiDAR coordinates, last column = queue index.  Here the poses are synthetic in place of nuScenes records."""
    rng = np.random.default_rng(seed)
    world_points = max(40000, 4 * points_per_frame) if world_points is None else world_points
    n_frames = T + future
    lidar2img = camera_rig(cams, seed=seed).numpy().astype(np.float64)
    l2e_t, l2e_yaw = np.array([0.94, 0.0, 1.84]), math.pi / 2          # LiDAR mounted like nuScenes': yawed 90 deg
    l2e_r = _yaw_matrix(l2e_yaw)
    metas_all, pts_all = [], []
    for b in range(bs):
        yaw0 = rng.uniform(-math.pi, math.pi)
        v = speed * rng.uniform(0.8, 1.2)
        w = yaw_rate * rng.uniform(0.8, 1.2) * (1 if b % 2 == 0 else -1)
        pos = np.array([rng.uniform(300, 1800), rng.uniform(300, 1800), 0.0])
        poses = []                                                          # ego2global (translation, yaw)
        for _ in range(n_frames):
            poses.append((pos.copy(), yaw0))
            pos = pos + v * dt * np.array([math.cos(yaw0 + w * dt / 2), math.sin(yaw0 + w * dt / 2), 0.0])
            yaw0 = yaw0 + w * dt
        centre = np.mean([p for p, _ in poses], 0)
        world = np.concatenate([centre[None, :2] + rng.uniform(-max_range - 40, max_range + 40, (world_points, 2)),
                                rng.uniform(-1.6, 2.5, (world_points, 1))], 1)
        raw = []                                                            # get_data_info: per-frame metas
        for t, yaw in poses:
            patch_angle = math.degrees(yaw) % 360.0
            can_bus = np.zeros(18)
            can_bus[:3] = t
            can_bus[3:7] = _yaw_quaternion(yaw)
            can_bus[12] = w
            can_bus[13] = v
            can_bus[-2] = patch_angle / 180 * np.pi
            can_bus[-1] = patch_angle
            raw.append(dict(ego2global_translation=t, ego2global_rotation=_yaw_quaternion(yaw),
                            lidar2ego_translation=l2e_t, lidar2ego_rotation=_yaw_quaternion(l2e_yaw),
                            lidar2global_rotation=_yaw_matrix(yaw) @ l2e_r, scene_token=f"synthetic-{seed}-{b}",
                            can_bus=can_bus, lidar2img=lidar2img, img_shape=[(img_hw[0], img_hw[1], 3)] * cams,
                            _e2g=(t, _yaw_matrix(yaw))))
        # union2one 1: every frame <-> the reference (current) frame, and the points of every frame
        ref_t, ref_r = raw[T - 1]["_e2g"]
        ref_e2g, ref_g2e = _transform_matrix(ref_t, ref_r), _transform_matrix(ref_t, ref_r, inverse=True)
        ref_l2e, ref_e2l = _transform_matrix(l2e_t, l2e_r), _transform_matrix(l2e_t, l2e_r, inverse=True)
        cur2ref, ref2cur, pts = [], [], []
        for i, m in enumerate(raw):
            t, r = m["_e2g"]
            e2g, g2e = _transform_matrix(t, r), _transform_matrix(t, r, inverse=True)
            l2e, e2l = _transform_matrix(l2e_t, l2e_r), _transform_matrix(l2e_t, l2e_r, inverse=True)
            cur2ref.append(l2e.T @ e2g.T @ ref_g2e.T @ ref_e2l.T)
            ref2cur.append(ref_l2e.T @ ref_e2g.T @ g2e.T @ e2l.T)
            # LiDAR returns: the world in this frame's LiDAR coordinates, within range
            g2l = e2l @ g2e
            local = world @ g2l[:3, :3].T + g2l[:3, 3]
            keep = np.flatnonzero((np.abs(local[:, 0]) < max_range) & (np.abs(local[:, 1]) < max_range)
                                  & (np.hypot(local[:, 0], local[:, 1]) > 2.0))
            keep = rng.choice(keep, min(points_per_frame, keep.size), replace=False)
            pts.append(np.concatenate([local[keep], np.full((keep.size, 1), i)], 1))
        # union2one 2: can_bus deltas of the previous frames, future can_bus and transforms
        metas, prev_pos, prev_angle = [], None, None
        for i in range(T):
            m = {k: v_ for k, v_ in raw[i].items() if k != "_e2g"}
            m["can_bus"] = raw[i]["can_bus"].copy()
            if i == 0:
                m["prev_bev_exists"] = False
                prev_pos, prev_angle = m["can_bus"][:3].copy(), m["can_bus"][-1]
                m["can_bus"][:3], m["can_bus"][-1] = 0, 0
            else:
                m["prev_bev_exists"] = True
                tmp_pos, tmp_angle = m["can_bus"][:3].copy(), m["can_bus"][-1]
                m["can_bus"][:3], m["can_bus"][-1] = tmp_pos - prev_pos, tmp_angle - prev_angle
                prev_pos, prev_angle = tmp_pos, tmp_angle
            m["ref_lidar_to_cur_lidar"] = ref2cur[i]
            metas.append(m)
        future_can_bus, future2ref, ref2future, ref_can_bus = [], [], [], None
        for i in range(future + 1):
            future2ref.append(cur2ref[i + T - 1])
            ref2future.append(ref2cur[i + T - 1])
            c = raw[i + T - 1]["can_bus"].copy()
            if i == 0:
                ref_can_bus = c.copy()
                c[:3], c[-1] = 0, 0
            else:
                p = np.array([0, 0, 0, 1]).reshape(1, 4) @ future2ref[-1] @ ref2future[-2]
                angle = c[-1] - ref_can_bus[-1]
                ref_can_bus = c.copy()
                c[:3], c[-1] = p[:, :3], angle
            future_can_bus.append(c)
        cur = metas[T - 1]
        cur["future_can_bus"] = np.array(future_can_bus)
        cur["future2ref_lidar_transform"] = np.array(future2ref)
        cur["ref2future_lidar_transform"] = np.array(ref2future)
        cur["total_cur2ref_lidar_transform"] = np.array(cur2ref)
        cur["total_ref2cur_lidar_transform"] = np.array(ref2cur)
        metas_all.append(metas)
        pts_all.append(np.concatenate(pts, 0).astype(np.float32))
    return dict(img_metas=metas_all, gt_points=pts_all)
