"""Ego motion on one GPU -> one JSON line (and --out FILE).

  * previous-BEV rotation, 200 x 200 x 256 fp32 at bs 1 and 4: `ego.rotate_prev_bev` (one kernel) against the
    reference's statements (transformer.py:136-149: per sample a permute to [C, H, W], torchvision's rotate, a permute
    back, then a stack), each call timed alone with CUDA events after a 256 MB write that evicts the L2; achieved
    GB/s against the 2 * bs * H * W * C * 4 bytes the kernel must move;
  * GT alignment of one ViDARHeadV1 loss (5 calls, 1 + 3 frames, 30 k rays per frame): `ego.align_gt_points`
    against the reference's mask-and-matmul statements (vidar_head_v1.py:94-148), host clock ending in a device
    synchronise;
  * full-size forward_train (+ backward) and forward_test with and without img_metas (T = 4 frames of 6 x 3 x 928 x
    1600, 200 x 200 BEV, 30 k rays per frame), mean of --steps calls after --warmup, host clock + synchronise;
  * the GPU's name and power limit, read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_eval import gpu_info  # noqa: E402


def reference_rotate(prev_bev, angles, center, bev_h, bev_w):
    from torchvision.transforms.functional import rotate
    out = []
    for i in range(prev_bev.shape[0]):
        t = prev_bev[i].reshape(bev_h, bev_w, -1).permute(2, 0, 1)
        t = rotate(t, float(angles[i]), center=center)
        out.append(t.permute(1, 2, 0).reshape(bev_h * bev_w, -1))
    return torch.stack(out, 0)


def reference_align(gt_points, src_list, tgt_list, img_metas):
    """vidar_head_v1.py:94-148's statements."""
    bs = len(gt_points)
    aligned, origins = [], []
    for frame_idx, (s, t) in enumerate(zip(src_list, tgt_list)):
        pts = [p[p[:, -1] == s] for p in gt_points]
        s2r = gt_points[0].new_tensor(np.array([m["total_cur2ref_lidar_transform"][s] for m in img_metas]))
        r2t = gt_points[0].new_tensor(np.array([m["total_ref2cur_lidar_transform"][t] for m in img_metas]))
        s2t = torch.matmul(s2r, r2t)
        per = []
        for b, p in enumerate(pts):
            q = torch.cat([p[:, :3], p.new_ones(p.shape[0], 1)], 1)
            q = torch.matmul(q, s2t[b])
            q[..., -1] = frame_idx
            per.append(q)
        aligned.append(per)
        o = torch.cat([torch.zeros(bs, 1, 3, device=s2t.device), torch.ones(bs, 1, 1, device=s2t.device)], -1)
        origins.append(torch.matmul(o, s2t)[..., :3])
    return [torch.cat([aligned[f][b] for f in range(len(src_list))], 0) for b in range(bs)], torch.cat(origins, 1)


def time_events(fn, n, flush):
    ts = []
    for _ in range(n):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def time_host(fn, n):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rays", type=int, default=30000)
    ap.add_argument("--skip-model", action="store_true", help="kernels only")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from vidar_b200 import ego, pretrain, synthetic
    dev = torch.device("cuda:0")
    info = gpu_info()
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)        # 256 MB > 126 MB L2
    res = dict(tool="bench_ego", **info)
    H = W = 200
    C = 256
    rot = {}
    for bs in (1, 4):
        x = torch.randn(bs, H * W, C, device=dev)
        angles = np.random.default_rng(bs).uniform(-5, 5, bs)
        with torch.no_grad():
            mine = ego.rotate_prev_bev(x, angles, [100, 100], H, W)
            ref = reference_rotate(x, angles, [100, 100], H, W)
            med, best = time_events(lambda: ego.rotate_prev_bev(x, angles, [100, 100], H, W), 50, flush)
            rmed, _ = time_events(lambda: reference_rotate(x, angles, [100, 100], H, W), 50, flush)
        nbytes = 2 * bs * H * W * C * 4
        rot[f"bs{bs}"] = dict(kernel_ms=med, kernel_best_ms=best, achieved_GBps=nbytes / (med * 1e-3) / 1e9,
                              bytes=nbytes, reference_ms=rmed, speedup=rmed / med,
                              cells_differing_from_reference=int((mine != ref).any(-1).sum()))
    res["rotation"] = rot
    # GT alignment for one V1 loss: 5 pred indices, 1 + 3 frames each
    T, F = 4, 3
    q = synthetic.ego_queue(bs=1, T=T, future=F + 1, seed=0, points_per_frame=a.rays)
    metas = [m[T - 1] for m in q["img_metas"]]
    pts = [torch.from_numpy(p).to(dev) for p in q["gt_points"]]
    valid = np.arange(1 + F)
    hq = ph = T - 1
    calls = [(valid + hq - ph + i, valid + hq) for i in range(5)]
    md = 0.0
    for s, t in calls:
        (o,), og = ego.align_gt_points(pts, s, t, metas)
        (r,), rg = reference_align(pts, s, t, metas)
        o = o[torch.argsort(torch.where(o[:, 3] < 0, 99.0, o[:, 3]), stable=True)][: r.shape[0]]
        md = max(md, float((o - r).abs().max()), float((og - rg).abs().max()))
    res["gt_alignment"] = dict(
        points=int(pts[0].shape[0]), calls=5, rays_per_frame=a.rays,
        ms=time_host(lambda: [ego.align_gt_points(pts, s, t, metas) for s, t in calls], 20),
        reference_ms=time_host(lambda: [reference_align(pts, s, t, metas) for s, t in calls], 20), max_abs_diff=md)
    res["gt_alignment"]["speedup"] = res["gt_alignment"]["reference_ms"] / res["gt_alignment"]["ms"]
    if not a.skip_model:
        model, _ = pretrain.build(dev, None, seed=0)
        plain = pretrain.synthetic_sample(dev, frames=T, rays_per_frame=a.rays, future_frames=6)
        moving = pretrain.synthetic_ego_sample(dev, frames=T, rays_per_frame=a.rays, future_frames=6)

        def train(sample, metas):
            model.zero_grad(set_to_none=True)
            losses = model.forward_train(sample["img"], sample["lidar2img"], sample["gt_points"], img_metas=metas)
            sum(losses.values()).backward()

        def test(sample, metas):
            model.forward_test(sample["img"], sample["lidar2img"], sample["gt_points"], img_metas=metas)

        steps = {}
        for name, fn in (("forward_train_backward", train), ("forward_test", test)):
            for tag, sample, metas in (("no_metas", plain, None), ("img_metas", moving, moving["img_metas"])):
                for _ in range(a.warmup):
                    fn(sample, metas)
                steps[f"{name}.{tag}_ms"] = time_host(lambda: fn(sample, metas), a.steps)
        steps.update(frames=T, img_hw=list(synthetic.IMG_HW), bev=[H, W], rays_per_frame=a.rays, steps=a.steps,
                     warmup=a.warmup, peak_mem_gib=round(torch.cuda.max_memory_allocated() / 2**30, 3))
        res["model"] = steps
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
