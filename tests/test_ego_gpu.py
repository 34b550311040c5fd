"""Ego motion on the device (vidar_b200/ego.py, csrc/ego.cu): the previous-BEV rotation against torchvision's rotate
on the same device and against the reference's golden, the GT alignment against the oracle and the golden without a
host sync, identity poses through the img_metas path, a moving ego through forward_train / forward_test (1 and 2
GPUs)."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ego_ref

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ego.npz")
SMALL = dict(encoder_layers=3, decoder_layers=2, future_frames=2, bev_hw=(50, 50), ray_grid_num=64, test_future_frames=3,
             rotate_center=(25, 25))
EGO_SAMPLE = dict(frames=4, img_hw=(96, 160), rays_per_frame=600, future_frames=3)


def _tv_rotate(x, angle, center):
    from torchvision.transforms.functional import rotate
    return rotate(x, float(angle), center=list(center))


def _candidates(img_hwc, angle, center, tol=1e-3):
    """The outputs of the source coordinate moved by +-tol px in x and y (oracle's fp64 coordinate), on the device."""
    H, W, _ = img_hwc.shape
    x64, y64 = ego_ref.source_coords(angle, center, H, W)
    out = []
    for sx in (-tol, tol):
        for sy in (-tol, tol):
            ix, iy = np.rint(x64 + sx), np.rint(y64 + sy)
            ok = (ix >= 0) & (ix <= W - 1) & (iy >= 0) & (iy <= H - 1)
            flat = torch.from_numpy(np.where(ok, iy * W + ix, 0).astype(np.int64)).to(img_hwc.device).view(-1)
            c = img_hwc.view(H * W, -1)[flat] * torch.from_numpy(ok.reshape(-1, 1)).to(img_hwc.device)
            out.append(c)
    x64d, y64d = np.abs(x64 - np.floor(x64) - 0.5), np.abs(y64 - np.floor(y64) - 0.5)
    near = torch.from_numpy(((x64d < tol) | (y64d < tol)).reshape(-1)).to(img_hwc.device)
    return torch.stack(out), near


@pytest.mark.parametrize("bs,C,H,W", [(1, 256, 200, 200), (2, 8, 200, 200), (4, 8, 100, 150), (2, 6, 100, 150)])
def test_rotation_equals_torchvision_on_device(cuda, bs, C, H, W):
    from vidar_b200 import ego
    g = torch.Generator(device="cpu").manual_seed(bs * 1000 + C)
    prev = torch.randn(bs, H * W, C, generator=g).to(cuda)
    center = (100, 100)
    rng = np.random.default_rng(bs + C)
    for angles in (rng.uniform(-180, 180, bs), np.resize([0.0, 90.0, -90.0, 180.0], bs)):
        with torch.no_grad():
            out = ego.rotate_prev_bev(prev, angles, center, H, W)
            again = ego.rotate_prev_bev(prev, angles, center, H, W)
        assert torch.equal(out, again), "two calls differ"
        near_total = 0
        for b in range(bs):
            img = prev[b].view(H, W, C)
            want = _tv_rotate(img.permute(2, 0, 1), angles[b], center).permute(1, 2, 0).reshape(H * W, C)
            got = out[b]
            cands, near = _candidates(img, angles[b], center)
            if float(angles[b]) in (0.0, 90.0, -90.0, 180.0):
                assert torch.equal(got, want), f"angle {angles[b]}: not exact"
                continue
            assert torch.equal(got[~near], want[~near]), f"angle {angles[b]}: cells off the boundaries differ"
            assert (cands == got[None]).all(-1).any(0)[near].all(), f"angle {angles[b]}: a boundary cell is no candidate"
            near_total += int(near.sum())
        assert near_total < 0.01 * bs * H * W


def test_rotation_equals_reference_golden(cuda):
    from vidar_b200 import ego
    z = np.load(GOLDEN)
    H = W = 200
    idx = torch.arange(1, H * W + 1, dtype=torch.float32, device=cuda)[None, :, None].repeat(2, 1, 8)
    for k in range(4):
        angles = z[f"rot{k}.angles"]
        with torch.no_grad():
            out = ego.rotate_prev_bev(idx, angles, [100, 100], H, W)
        assert torch.equal(out, out[..., :1].expand_as(out))
        for b in range(2):
            want = z[f"rot{k}.src_index"][b].astype(np.float32)
            _, near, cands = ego_ref.rotate(np.arange(1, H * W + 1, dtype=np.float32).reshape(1, H, W), float(angles[b]),
                                            [100, 100])
            got = out[b, :, 0].cpu().numpy()
            near = near.reshape(-1)
            np.testing.assert_array_equal(got[~near], want[~near])
            assert (cands[:, 0].reshape(4, -1) == got[None]).any(0)[near].all()


def test_rotation_is_forward_only(cuda):
    from vidar_b200 import ego
    prev = torch.randn(1, 16, 8, device=cuda, requires_grad=True)
    with pytest.raises(RuntimeError, match="forward only"):
        ego.rotate_prev_bev(prev, [10.0], [2, 2], 4, 4)
    with torch.no_grad():
        ego.rotate_prev_bev(prev, [10.0], [2, 2], 4, 4)


def _gt_case(z, case, cuda, empty_sample=False):
    keys = ("total_cur2ref_lidar_transform", "total_ref2cur_lidar_transform")
    metas = [{k: z[f"gt.{k}"][b] for k in keys} for b in range(2)]
    pts = [torch.from_numpy(z[f"gt.points{b}"]).to(cuda) for b in range(2)]
    if empty_sample:
        pts[1] = pts[1][:0]
    return metas, pts, z[f"gt.{case}.src"], z[f"gt.{case}.tgt"]


@pytest.mark.parametrize("case", ["loss0", "loss2", "loss4", "test"])
def test_alignment_equals_oracle_and_golden_without_host_sync(cuda, case):
    from vidar_b200 import ego
    z = np.load(GOLDEN)
    metas, pts, src, tgt = _gt_case(z, case, cuda)
    ego.align_gt_points(pts, src, tgt, metas)                   # load the library
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out, origins = ego.align_gt_points(pts, src, tgt, metas)
        again, _ = ego.align_gt_points(pts, src, tgt, metas)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    mats = ego.src_to_tgt_matrices(src, tgt, metas)
    slots = {int(f): s for s, f in enumerate(src)}
    for b in range(2):
        got = out[b].cpu().numpy()
        assert got.shape == (pts[b].shape[0], 4) and torch.equal(out[b].view(torch.int32), again[b].view(torch.int32))
        want, want_o = ego_ref.align_points(pts[b].cpu().numpy(), slots, mats[b])
        np.testing.assert_array_equal(got[:, 3], want[:, 3])
        keep = want[:, 3] >= 0
        assert np.isnan(got[~keep, :3]).all()
        scale = np.abs(want[keep, :3]).max()
        np.testing.assert_allclose(got[keep, :3], want[keep, :3], rtol=0, atol=1e-6 * scale)
        np.testing.assert_allclose(origins[b].cpu().numpy(), want_o, rtol=0, atol=1e-6)
        order = np.argsort(np.where(keep, got[:, 3], len(src)), kind="stable")
        g = got[order][: int(keep.sum())]
        ref = z[f"gt.{case}.out{b}"]
        np.testing.assert_array_equal(g[:, 3], ref[:, 3])
        np.testing.assert_allclose(g[:, :3], ref[:, :3], rtol=0, atol=1e-6 * np.abs(ref[:, :3]).max())


def test_alignment_with_an_empty_sample(cuda):
    from vidar_b200 import ego
    z = np.load(GOLDEN)
    metas, pts, src, tgt = _gt_case(z, "loss1", cuda, empty_sample=True)
    out, origins = ego.align_gt_points(pts, src, tgt, metas)
    assert out[1].shape == (0, 4) and out[0].shape[0] == pts[0].shape[0]
    mats = ego.src_to_tgt_matrices(src, tgt, metas)
    np.testing.assert_allclose(origins[1].cpu().numpy(), mats[1][:, 3, :3], rtol=0, atol=1e-6)


def _identity_metas(bs, T, future, lidar2img, img_hw):
    eye = np.eye(4)
    metas = []
    for _ in range(bs):
        frames = [dict(can_bus=np.zeros(18), lidar2global_rotation=np.eye(3), prev_bev_exists=t > 0,
                       ref_lidar_to_cur_lidar=eye, lidar2img=lidar2img, img_shape=[(img_hw[0], img_hw[1], 3)])
                  for t in range(T)]
        n = T + future
        frames[-1].update(future_can_bus=np.zeros((future + 1, 18)), future2ref_lidar_transform=np.stack([eye] * (future + 1)),
                          ref2future_lidar_transform=np.stack([eye] * (future + 1)),
                          total_cur2ref_lidar_transform=np.stack([eye] * n), total_ref2cur_lidar_transform=np.stack([eye] * n))
        metas.append(frames)
    return metas


def test_identity_poses_equal_the_no_metas_path(cuda):
    from vidar_b200 import bev_geometry, ego, pretrain
    model, _ = pretrain.build(cuda, None, seed=1, **SMALL)
    T = 4
    sample = pretrain.synthetic_sample(cuda, frames=T, img_hw=(96, 160), rays_per_frame=300, future_frames=3, bev_hw=(50, 50))
    metas = _identity_metas(1, T, 3, sample["lidar2img"][0], (96, 160))
    preds = []
    head = model.forward_head

    def capture(x):
        preds.append(head(x))
        return preds[-1]
    model.forward_head = capture
    model.forward_test(sample["img"], sample["lidar2img"], sample["gt_points"])
    gt = [torch.cat([p[:, :3], p[:, 3:] + (T - 1)], 1) for p in sample["gt_points"]]
    model.forward_test(sample["img"], sample["lidar2img"], gt, img_metas=metas)
    a, b = preds
    assert (a - b).abs().max().item() <= 1e-4 * a.abs().max().item()
    # the decoder's aligned grids differ from the plain reference points by fp32 rounding only
    r2h = ego.history_ref_to_previous_transform(torch.zeros(1, 1, device=cuda), 1, [[metas[0][-1]]])
    tgt, aligned, _ = ego.align_bev_coordinates(1, r2h, [metas[0][-1]], 50, 50, pretrain.PC_RANGE)
    ref = bev_geometry.get_reference_points(50, 50, dim="2d", bs=1, device=cuda)
    assert torch.equal(tgt.unsqueeze(2), ref)
    assert (aligned - ref).abs().max().item() <= 1e-6


def test_static_world_aligns_and_origins_are_the_poses(cuda):
    from vidar_b200 import chamfer, ego, synthetic
    T, future = 4, 4
    q = synthetic.ego_queue(bs=2, T=T, future=future, seed=9, points_per_frame=1500, world_points=4000)
    metas = [m[T - 1] for m in q["img_metas"]]
    pts = [torch.from_numpy(p).to(cuda) for p in q["gt_points"]]
    frames = np.arange(T + future)
    out, origins = ego.align_gt_points(pts, frames, np.full_like(frames, T - 1), metas)
    for b in range(2):
        c2r, r2c = metas[b]["total_cur2ref_lidar_transform"], metas[b]["total_ref2cur_lidar_transform"]
        for k in frames:
            want = (np.array([0, 0, 0, 1.0]) @ c2r[k] @ r2c[T - 1])[:3]
            np.testing.assert_allclose(origins[b, k].cpu().numpy(), want, rtol=0, atol=1e-4)
        ref = out[b][out[b][:, 3] == T - 1, :3]
        for k in frames:
            moved = out[b][out[b][:, 3] == k, :3]
            d = chamfer.knn_points(moved[None].contiguous(), ref[None].contiguous()).dists[0, :, 0].sqrt()
            assert (d < 1e-4).float().mean().item() > 0.3, (b, k, d.median().item())


def test_forward_train_and_test_with_a_moving_ego(cuda):
    from vidar_b200 import pretrain
    model, _ = pretrain.build(cuda, None, seed=1, **SMALL)
    sample = pretrain.synthetic_ego_sample(cuda, bs=2, **EGO_SAMPLE)
    with pytest.raises(ValueError, match="either can_bus or img_metas"):
        model.forward_train(sample["img"], sample["lidar2img"], sample["gt_points"], can_bus=torch.zeros(2, 18, device=cuda),
                            img_metas=sample["img_metas"])
    losses = model.forward_train(sample["img"], sample["lidar2img"], sample["gt_points"], img_metas=sample["img_metas"])
    assert set(losses) == {f"frame.{i}.{k}" for i in range(5) for k in ("regularization.loss", "loss.dense_voxel")}
    assert all(torch.isfinite(v) for v in losses.values()), losses
    sum(losses.values()).backward()
    missing = [n for n, p in model.named_parameters() if p.requires_grad and p.grad is None]
    assert not missing, missing
    assert all(torch.isfinite(p.grad).all() for p in model.parameters() if p.grad is not None)
    (ret,) = model.forward_test(sample["img"], sample["lidar2img"], sample["gt_points"], img_metas=sample["img_metas"])
    assert model.training
    assert list(ret) == [f"frame.{i}" for i in range(1 + SMALL["test_future_frames"])]
    for v in ret.values():
        assert v["count"] == 2
        assert all(np.isfinite(v[k]) for k in ("chamfer_distance", "l1_error", "absrel_error")), v


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from vidar_b200 import pretrain
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = []
    for group in (None, dist.group.WORLD):
        model, _ = pretrain.build(dev, group, seed=1, **SMALL)
        sample = pretrain.synthetic_ego_sample(dev, **EGO_SAMPLE)
        res.append(model.forward_test(sample["img"], sample["lidar2img"], sample["gt_points"],
                                      img_metas=sample["img_metas"])[0])
    gathered = [None] * world
    dist.all_gather_object(gathered, res[1])
    if rank == 0:
        torch.save((res[0], gathered), out)
    dist.barrier()
    dist.destroy_process_group()


def test_camera_sharded_forward_test_with_ego_motion(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = str(tmp_path / "ret.pt")
    mp.spawn(_worker, args=(2, 29640 + os.getpid() % 100, out), nprocs=2, join=True)
    single, sharded = torch.load(out, weights_only=False)
    for key in single:
        for k in ("chamfer_distance", "l1_error", "absrel_error"):
            a, b = sharded[0][key][k], sharded[1][key][k]
            assert np.float64(a).tobytes() == np.float64(b).tobytes(), f"{key}.{k}: ranks differ"
            np.testing.assert_allclose(float(a), float(single[key][k]), rtol=2e-2, err_msg=f"{key}.{k}")
        assert sharded[0][key]["count"] == single[key]["count"]
