"""Point-cloud forecasting evaluation on one GPU -> one JSON line.

  * forward_test at full size: T = 4 frames of 6 x 3 x 928 x 1600, 200 x 200 BEV, 6 future roll-outs, 30 k rays per
    frame; stage times from CUDA events (mean of --steps timed calls after --warmup), peak memory;
  * the metric stage alone on the same decode output: `evaluation.evaluate_rays` (device, CUDA events) against the
    reference-shaped flow -- per-(sample, frame) boolean masks (`get_rendered_pcds`), `.cpu()` copies, the numpy clamp of
    oracle/eval_ref.py and this package's ChamferDistance on the GPU where the reference runs chamferdist -- timed with a
    host clock that ends in a device synchronise, and the largest difference between the two results;
  * the GPU's name and power limit, read in the same run.
Writes nothing into the tree; --out FILE additionally writes the JSON line there."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # nvidia-smi missing: still report what torch knows
        return dict(gpu=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def reference_flow(head, origin, points, tindex, gt_dist, pred_dist, pc_range):
    """forward_test's metric loop (vidar.py:450-497) with this package's GPU ChamferDistance and the oracle's numpy
    clamp -> [bs, F, 4] like evaluate_rays."""
    from oracle import eval_ref
    from vidar_b200 import chamfer
    from vidar_b200.head import get_inside_mask
    cd_op = chamfer.ChamferDistance()
    dev = points.device

    def nn(sph_g, sph_p):
        _, (_, idx) = cd_op(torch.from_numpy(sph_p[None]).to(dev), torch.from_numpy(sph_g[None]).to(dev), reverse=True,
                            reduction="mean")
        return idx[0].cpu().numpy()

    pred_pcds = head.get_rendered_pcds(origin, points, tindex, gt_dist, pred_dist, pc_range)
    gt_pcds = head.get_rendered_pcds(origin, points, tindex, gt_dist, gt_dist, pc_range)
    bs, F = origin.shape[:2]
    out = np.zeros((bs, F, 4))
    for f in range(F):
        for b in range(bs):
            pred, gt = pred_pcds[b][f], gt_pcds[b][f]
            pm, gm = get_inside_mask(pred, pc_range), get_inside_mask(gt, pc_range)
            cd = 0.0
            if pm.sum() > 0 and gm.sum() > 0:
                cd = chamfer.compute_chamfer_distance(pred[pm], gt[gm]).item()
            r = eval_ref.ray_errors_detail(pred.cpu().numpy(), gt.cpu().numpy(), origin[b, f].cpu().numpy(), nn=nn)
            out[b, f] = (cd, r["l1"], r["absrel"], r["count"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--metric-steps", type=int, default=20)
    ap.add_argument("--rays", type=int, default=30000)
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--test-future-frames", type=int, default=6)
    ap.add_argument("--img-hw", type=int, nargs=2, default=(928, 1600))
    ap.add_argument("--bev", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py needs a CUDA device")
    from vidar_b200 import evaluation, pretrain
    dev = torch.device("cuda:0")
    info = gpu_info()
    bev = (a.bev, a.bev)
    model, _ = pretrain.build(dev, None, seed=0, bev_hw=bev, test_future_frames=a.test_future_frames)
    sample = pretrain.synthetic_sample(dev, frames=a.frames, img_hw=tuple(a.img_hw), rays_per_frame=a.rays,
                                       future_frames=a.test_future_frames, bev_hw=bev)
    args = (sample["img"], sample["lidar2img"], sample["gt_points"])
    for _ in range(a.warmup):
        model.forward_test(*args)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    stages, totals = {}, []
    for _ in range(a.steps):
        model.timings = []
        model._mark("start")
        (ret,) = model.forward_test(*args)
        torch.cuda.synchronize()
        ev = model.timings
        model.timings = None
        for i in range(len(ev) - 1):
            stages.setdefault(ev[i + 1][0], []).append(ev[i][1].elapsed_time(ev[i + 1][1]))
        totals.append(ev[0][1].elapsed_time(ev[-1][1]))
    peak = torch.cuda.max_memory_allocated() / 2 ** 30

    # the metric stage alone, on the decode output of the same model
    model.eval()
    with torch.no_grad():
        img_metas = [dict(lidar2img=np.asarray(sample["lidar2img"][0]), img_shape=[(a.img_hw[0], a.img_hw[1], 3)])]
        can_bus = torch.zeros(1, 18, device=dev)
        prev = None
        for t in range(a.frames):
            feats, shapes, lsi = model.extract_feat(sample["img"][:, t])
            prev = model.encode(feats, shapes, lsi, img_metas, can_bus, prev)
        feats_l = [prev.unsqueeze(0).repeat(len(model.bev_pred_head), 1, 1, 1)]
        q = prev.unsqueeze(1)
        for _ in range(a.test_future_frames):
            pf, last = model.decode_future(q, can_bus)
            feats_l.append(pf)
            q = last.unsqueeze(1)
        preds = model.forward_head(torch.stack(feats_l, 0))
        pd = dict(next_bev_preds=preds[:, :, model.history_frames], valid_frames=list(range(1 + a.test_future_frames)))
        dec = model.ray_head._decode_rays(pd, sample["gt_points"], 0, bev[0], bev[1], pretrain.PC_RANGE, None)
        origin = dec[0]
        F = origin.shape[1]
        for _ in range(3):
            m_dev = evaluation.evaluate_rays(*dec, pretrain.PC_RANGE, F)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.metric_steps):
            m_dev = evaluation.evaluate_rays(*dec, pretrain.PC_RANGE, F)
        e1.record()
        torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1) / a.metric_steps
        m_dev = m_dev.cpu().numpy()
        reference_flow(model.ray_head, *dec, pretrain.PC_RANGE)        # warm-up (allocations, NN kernel)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m_ref = reference_flow(model.ray_head, *dec, pretrain.PC_RANGE)
        torch.cuda.synchronize()
        ref_ms = (time.perf_counter() - t0) * 1e3
    model.train()
    rel = np.abs(m_dev[..., :3] - m_ref[..., :3]) / np.maximum(np.abs(m_ref[..., :3]), 1e-12)
    rays = int(m_dev[..., 3].sum())
    res = dict(
        tool="bench_eval", **info,
        forward_test=dict(frames=a.frames, test_future_frames=a.test_future_frames, img_hw=list(a.img_hw), bev=list(bev),
                          rays_per_frame=a.rays, steps=a.steps, warmup=a.warmup, total_ms=float(np.mean(totals)),
                          stage_ms={k: float(np.mean(v)) for k, v in stages.items()}, peak_mem_gib=round(peak, 3),
                          frames_out=len(ret)),
        metric_stage=dict(segments=int(m_dev.shape[0] * m_dev.shape[1]), gt_rays=rays, evaluate_rays_ms=dev_ms,
                          reference_flow_ms=ref_ms, speedup=ref_ms / dev_ms,
                          max_rel_diff=float(np.nanmax(rel)), counts_equal=bool((m_dev[..., 3] == m_ref[..., 3]).all())),
    )
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
