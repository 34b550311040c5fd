"""Point-cloud forecasting metrics on the device (vidar_b200/evaluation.py, csrc/eval.cu): the drop-ins against the
reference's goldens, evaluate_rays against the oracle per (sample, frame), no host sync, determinism, the head's
evaluate against the reference-shaped loop and SyntheticViDAR.forward_test (1 and 2 GPUs)."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import eval_ref
from tests.eval_cases import PC_RANGE, cases

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "eval.npz")
SMALL = dict(encoder_layers=3, decoder_layers=2, future_frames=2, bev_hw=(40, 40), ray_grid_num=64, test_future_frames=3)
SAMPLE = dict(frames=2, img_hw=(96, 160), rays_per_frame=800, future_frames=3, bev_hw=(40, 40))


@pytest.mark.parametrize("name", sorted(cases()))
def test_dropins_equal_reference_goldens(cuda, name):
    from vidar_b200 import evaluation
    z = np.load(GOLDEN)
    pred, gt, o = (torch.from_numpy(z[f"{name}.{k}"]).to(cuda) for k in ("pred", "gt", "origin"))
    cd = evaluation.compute_chamfer_distance_inner(pred, gt, PC_RANGE)
    want = float(z[f"{name}.chamfer"])
    if want == 0.0:
        assert cd == 0.0 and isinstance(cd, float)
    else:
        assert torch.is_tensor(cd) and cd.is_cuda
        np.testing.assert_allclose(cd.item(), want, rtol=1e-5)
    if bool(z[f"{name}.raises"]):
        with pytest.raises(RuntimeError, match="identical"):
            evaluation.compute_ray_errors(pred, gt, o, cuda)
        return
    l1, absrel = evaluation.compute_ray_errors(pred, gt, o, cuda)
    np.testing.assert_allclose(l1, z[f"{name}.l1"], rtol=1e-5, equal_nan=True)
    np.testing.assert_allclose(absrel, z[f"{name}.absrel"], rtol=1e-5, equal_nan=True)


def _random_batch(seed, bs=2, F=7, M=900, pad=120):
    """Padded decode outputs: LiDAR-like rays of random frames (some frames empty), NaN / -1 padding, some rays with
    gt_dist 0, predictions around the GT depth, a few beyond the eval box and pc_range."""
    rng = np.random.default_rng(seed)
    origin = rng.normal(0, 0.5, (bs, F, 3)).astype(np.float32)
    tindex = rng.integers(0, F, (bs, M)).astype(np.float32)
    tindex[0][tindex[0] == 3] = 5            # frame 3 of sample 0 has no ray
    az, el = rng.uniform(-np.pi, np.pi, (bs, M)), np.deg2rad(rng.uniform(-25, 10, (bs, M)))
    u = np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], -1)
    r = rng.uniform(1.0, 90.0, (bs, M))
    o_ray = np.take_along_axis(origin, tindex.astype(np.int64)[..., None].repeat(3, -1), 1)
    points = (o_ray + u * r[..., None]).astype(np.float32)
    gt_dist = (r * rng.uniform(0.95, 1.05, (bs, M))).astype(np.float32)
    gt_dist[rng.random((bs, M)) < 0.05] = 0.0
    pred_dist = (gt_dist * rng.uniform(0.5, 1.5, (bs, M))).astype(np.float32)
    points[:, -pad:] = np.nan
    tindex[:, -pad:] = -1
    return origin, points, tindex, gt_dist, pred_dist


def _to(cuda, *arrays):
    return [torch.from_numpy(a).to(cuda) for a in arrays]


@pytest.mark.parametrize("within", [False, True])
def test_evaluate_rays_equals_oracle_per_segment(cuda, within):
    from vidar_b200 import evaluation
    o, p, t, g, d = _random_batch(1)
    got = evaluation.evaluate_rays(*_to(cuda, o, p, t, g, d), PC_RANGE, o.shape[1], eval_within_grid=within).cpu().numpy()
    want = eval_ref.evaluate_rays(o, p, t, g, d, PC_RANGE, eval_within_grid=within)
    np.testing.assert_array_equal(got[..., 3], want[..., 3])
    assert got[0, 3, 3] == 0 and np.isnan(got[0, 3, 1]) and got[0, 3, 0] == 0.0        # the empty frame
    np.testing.assert_allclose(got[..., :3], want[..., :3], rtol=1e-5, atol=1e-7, equal_nan=True)


def test_evaluate_rays_makes_no_host_sync_and_is_deterministic(cuda):
    from vidar_b200 import evaluation
    args = _to(cuda, *_random_batch(2))
    evaluation.evaluate_rays(*args, PC_RANGE, 7)          # load the library, allocate
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a = evaluation.evaluate_rays(*args, PC_RANGE, 7)
        b = evaluation.evaluate_rays(*args, PC_RANGE, 7)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.equal(a.view(torch.int64), b.view(torch.int64)), "two calls differ"


def _pred_dict(cuda, seed=0, frames=4, bs=2, bev=(40, 40), heights=16):
    g = torch.Generator(device="cpu").manual_seed(seed)
    preds = torch.randn(frames, 2, bs, bev[0] * bev[1], heights, generator=g)
    return dict(next_bev_preds=preds.to(cuda), valid_frames=list(range(frames)))


def test_head_evaluate_equals_reference_loop(cuda):
    """ViDARRayHead.evaluate == get_point_cloud_prediction followed by the oracle per (sample, frame), summed like
    vidar.py:450-497."""
    from vidar_b200 import pretrain, synthetic  # noqa: F401
    from vidar_b200.head import ViDARRayHead
    head = ViDARRayHead(ray_grid_num=64, ray_grid_step=1.0, loss_weight=[[1.0]] * 4)
    pd = _pred_dict(cuda)
    samples = [pretrain.synthetic_sample(cuda, frames=1, img_hw=(8, 8), rays_per_frame=300, future_frames=3, seed=s,
                                         bev_hw=(40, 40))["gt_points"][0] for s in (0, 1)]
    ret = head.evaluate(pd, samples, 0, 40, 40, pretrain.PC_RANGE)
    dec = head.get_point_cloud_prediction(pd, samples, 0, 40, 40, pretrain.PC_RANGE)
    assert list(ret) == [f"frame.{i}" for i in range(4)]
    for f in range(4):
        cd = l1 = ar = 0.0
        for b in range(2):
            pred, gt = dec["pred_pcds"][b][f].cpu().numpy(), dec["gt_pcds"][b][f].cpu().numpy()
            o = dec["origin"][b, f].cpu().numpy()
            cd += float(eval_ref.compute_chamfer_distance_inner(pred, gt, pretrain.PC_RANGE))
            r1, r2 = eval_ref.compute_ray_errors(pred, gt, o)
            l1, ar = l1 + float(r1), ar + float(r2)
        e = ret[f"frame.{f}"]
        assert e["count"] == 2
        np.testing.assert_allclose([e["chamfer_distance"], e["l1_error"], e["absrel_error"]], [cd, l1, ar], rtol=1e-5)


def test_forward_test_small(cuda):
    from vidar_b200 import pretrain
    model, _ = pretrain.build(cuda, None, seed=1, **SMALL)
    sample = pretrain.synthetic_sample(cuda, **SAMPLE)
    (ret,) = model.forward_test(sample["img"], sample["lidar2img"], sample["gt_points"])
    assert model.training, "forward_test restores the training mode"
    assert list(ret) == [f"frame.{i}" for i in range(1 + SMALL["test_future_frames"])]
    for v in ret.values():
        assert v["count"] == 1
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
        sample = pretrain.synthetic_sample(dev, **SAMPLE)
        res.append(model.forward_test(sample["img"], sample["lidar2img"], sample["gt_points"])[0])
    gathered = [None] * world
    dist.all_gather_object(gathered, res[1])
    if rank == 0:
        torch.save((res[0], gathered), out)
    dist.barrier()
    dist.destroy_process_group()


def test_camera_sharded_forward_test(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = str(tmp_path / "ret.pt")
    mp.spawn(_worker, args=(2, 29540 + os.getpid() % 100, out), nprocs=2, join=True)
    single, sharded = torch.load(out, weights_only=False)
    for key in single:
        for k in ("chamfer_distance", "l1_error", "absrel_error"):
            a, b = sharded[0][key][k], sharded[1][key][k]
            assert np.float64(a).tobytes() == np.float64(b).tobytes(), f"{key}.{k}: ranks differ"
            np.testing.assert_allclose(float(a), float(single[key][k]), rtol=2e-2, err_msg=f"{key}.{k}")
        assert sharded[0][key]["count"] == single[key]["count"]
