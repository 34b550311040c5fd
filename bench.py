#!/usr/bin/env python
"""bench.py -- the hot path on synthetic data, one JSON line.

A "step" is one pass of ViDAR's two hot paths over one synthetic sample
(BASELINE.json configs[1] + configs[2], SURVEY.md 8d):
  (i)  MSDA forward + backward at the SpatialCrossAttention shape: 6 cameras, 4-level FPN of a
       928x1600 input (30825 keys/cam), 200x200 = 40000 BEV queries per camera, 8 heads x 32
       channels, 8 sampling points per level (4 Z-anchors x 2);
  (ii) LatentRendering module forward + backward on a [1,200,200,256] BEV embedding
       (pred_height 16, 256 waypoints of step 0.5, sigmoid; projections fused around the ray-marching core);
  (iii) ViDAR-head ray sampler + cross-entropy forward + backward: sigma [3,16,200,200], 30000
       LiDAR-like rays over 3 frames, 512 waypoints + the GT sample per ray;
  (iv) voxel ray-caster forward + loss backward (`dvr.render`, L2) on the same volume and rays, and the
       dvxlr autograd layer (`DifferentiableVoxelRendering`) forward + backward on them.
metric = rays/sec = 30000 rays / step time (whole job); ms_per_step is the same thing as time.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
For N>1 launch under torchrun (one rank per GPU); the (camera, query) rows and the rays are
sharded over ranks (strong scaling: total work fixed); per step one all-reduce of the BEV grid
(the local scatter-add of SpatialCrossAttention's rows, 41 MB) and one of each grad_sigma.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

LEVELS = ((116, 200), (58, 100), (29, 50), (15, 25))
NUM_CAMS, BEV_Q, HEADS, HEAD_DIM, POINTS = 6, 40000, 8, 32, 8
RAYS, FRAMES, GRID = 30000, 3, (16, 200, 200)
WAYPOINTS, LR_GRID_NUM, EMBED = 512, 256, 256
METRIC = "rays/sec (fwd+bwd step: 6-cam 200x200-BEV MSDA + latent rendering + 30k-ray head CE + voxel render + dvxlr layer)"
WORKLOAD = ("configs[1]+[2]: MSDA fwd+bwd B=6 K=30825 Q=40000 H=8 C=32 L=4 P=8; LatentRendering fwd+bwd "
            "embed[1,200,200,256] pred_height=16 grid_num=256; ray sampler+CE fwd+bwd sigma[3,16,200,200] "
            "30000 rays x 513 samples; dvr.render(l2) sigma[1,3,16,200,200] 30000 rays; DifferentiableVoxelRendering "
            "(dvxlr autograd layer) fwd+bwd on the same rays")
LR_CFG = dict(type="LatentRendering", embed_dims=EMBED, num_pred_fcs=0, pred_height=GRID[0],
              grid_num=LR_GRID_NUM, grid_step=0.5, reduction=16, act="sigmoid")


def set_workload(bev=200, rays=30000, frames=3):
    """configs[4] sweep (tools/sweep_multi.py): resize the step -- BEV bev x bev queries / cells / volume,
    `rays` LiDAR rays over `frames` frames.  The headline line always uses the defaults."""
    global BEV_Q, RAYS, FRAMES, GRID
    BEV_Q, RAYS, FRAMES, GRID = bev * bev, rays, frames, (16, bev, bev)


# ------------------------------------------------------------------------------------------
# synthetic inputs
# ------------------------------------------------------------------------------------------
def sca_like_inputs(device, cams=NUM_CAMS, Q=None, seed=0):
    from vidar_b200 import synthetic
    Q = BEV_Q if Q is None else Q
    return synthetic.sca_like_inputs(device, cams=cams, Q=Q, seed=seed, levels=LEVELS, heads=HEADS,
                                     head_dim=HEAD_DIM, points=POINTS)


def ray_inputs():
    from vidar_b200 import synthetic
    return synthetic.dvr_inputs_lidar(M=RAYS, T=FRAMES, grid=GRID, seed=0)


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def msda_algorithmic_bytes(rows, cams_touched):
    """SURVEY.md 8(d): fwd = value + 4096 B/query; bwd = 3 x value + 7168 B/query (fp32,
    H=8, L*P=32, C=32).  `rows` = (camera, query) rows, value counted once per camera."""
    value = sum(h * w for h, w in LEVELS) * HEADS * HEAD_DIM * 4
    fwd = cams_touched * value + rows * 4096
    bwd = cams_touched * 3 * value + rows * 7168
    return fwd, bwd


def msda_algorithmic_bytes_q(rows, cams_touched, queries):
    """as msda_algorithmic_bytes; `queries` is unused (per-row bytes do not depend on the BEV size)."""
    return msda_algorithmic_bytes(rows, cams_touched)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms; started before warm-up so it is
    already streaming when the timed region begins; only samples that arrived between mark_begin()
    and mark_end() are reported."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.12)
        self.proc.terminate()
        inside = [r for t, r in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or t) + 0.06]
        scope = "timed region"
        if not inside:          # region shorter than the sampling period: nearest samples
            inside = [r for _, r in self.rows[-3:]]
            scope = "nearest samples (timed region shorter than 50 ms sampling)"

        def num(x):
            try:
                return float(x)
            except ValueError:
                return None
        sm = [num(r[0]) for r in inside if r and num(r[0]) is not None]
        mx = [num(r[1]) for r in inside if len(r) > 1 and num(r[1]) is not None]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in inside if len(r) >= 7
                          for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "scope": scope}


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
_CAM_GROUPS = {}


def _camera_groups(world, rank):
    from vidar_b200 import sca
    if world not in _CAM_GROUPS:
        _CAM_GROUPS[world] = sca.camera_groups(world, NUM_CAMS, rank)
    return _CAM_GROUPS[world]


def bench_config(world):
    """The `config` object of the JSON line -- identical for the GPU arm and the reference arm."""
    return {"workload": WORKLOAD,
            "l2_policy": "inputs larger than L2 (1.4 GB of MSDA operands per step)",
            "sharding": ("cameras sharded over ranks as (camera, interleaved 64-row sub-slice) units "
                         "(vidar_b200.sca.unit_plan); per step: reduce-scatter of the partial BEV slot grids "
                         "(41 MB) + ONE all-gather of the BEV grid, backward = all-gather of the row gradients; "
                         "rays split over ranks, one all-reduce of both ray stages' grad_sigma (2 x 7.7 MB); "
                         "LatentRendering: BEV rows/cells split over ranks, row-sharded in/out (all-gather of the 2.56 MB maps only)") if world > 1 else "single GPU"}


def run_ours(args, light=False):
    import torch.distributed as dist

    from vidar_b200 import _lib, ray_head, render, sca, sharding
    from vidar_b200.registry import build_attention
    import vidar_b200.modules  # noqa: F401  (registers LatentRendering)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun)"
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    grp = None
    if world > 1:
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=dev)
        grp = dist.group.WORLD

    # ---- device-resident inputs (this rank's shard): the product's own unit plan decides who owns what
    full = sca_like_inputs(dev)
    plan = sca.unit_plan(world, rank, NUM_CAMS)
    cam_groups = _camera_groups(world, rank) if world > 1 else {}
    groups = []
    for cam0, ncl, S, lo, hi in plan:
        sl = slice(cam0, cam0 + ncl)
        groups.append(dict(plan=(cam0, ncl, S, lo, hi), value=full["value"][sl].contiguous(),
                           loc=full["loc"][sl].contiguous(), attn=full["attn"][sl].contiguous()))
    nblk = -(-BEV_Q // sca.SLICE_ROWS)
    rows = 0                      # (camera, query) rows this rank samples
    for cam0, ncl, S, lo, hi in plan:
        per_cam = sum(min(sca.SLICE_ROWS, BEV_Q - blk * sca.SLICE_ROWS) for blk in range(nblk) if lo <= blk % S < hi)
        rows += ncl * per_cam
    my_cams = sca.plan_cameras(plan)
    shapes, lsi = full["shapes"], full["lsi"]
    # the gradient of the BEV grid (one per pillar, as in the model) and 1 / #cameras (every camera sees every
    # pillar in the dense cfg2 shape): SpatialCrossAttention's normalisation (spatial_cross_attention.py:168-171)
    gg = torch.Generator(device=dev).manual_seed(11)
    grad_bev = torch.randn(BEV_Q, HEADS * HEAD_DIM, device=dev, generator=gg)
    inv_count = torch.full((1, BEV_Q), 1.0 / NUM_CAMS, device=dev)
    sigma_np, origin_np, points_np, tindex_np = ray_inputs()
    r0, r1 = rank * RAYS // world, (rank + 1) * RAYS // world
    sigma = torch.from_numpy(sigma_np).to(dev)
    origin = torch.from_numpy(origin_np).to(dev)
    points = torch.from_numpy(points_np[:, r0:r1].copy()).to(dev)
    tindex = torch.from_numpy(tindex_np[:, r0:r1].copy()).to(dev)
    del full
    # head ray sampler: same rays, per-frame volumes = sigma[0]; LatentRendering: replicated per rank
    ce_points = points[0].contiguous()
    ce_frame = tindex[0].to(torch.int32).contiguous()
    ce_origin = origin[0].contiguous()
    torch.manual_seed(0)
    latent = build_attention(LR_CFG).to(dev)
    if world > 1:
        latent.process_group = grp      # shard the BEV cells of the latent-rendering core
    lg = torch.Generator(device=dev).manual_seed(7)
    embed = torch.randn(1, GRID[1], GRID[2], EMBED, device=dev, generator=lg)
    grad_embed = torch.randn(1, GRID[1], GRID[2], EMBED, device=dev, generator=lg)

    lr0, lr1 = sharding.shard_range(GRID[1] * GRID[2], rank, world)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    names = ["msda_fwd", "msda_bwd", "latent_render", "ray_ce", "render"]
    ray_grads = torch.empty((3,) + tuple(sigma.shape[1:]), device=dev) if world > 1 else None
    marks = []

    def msda_stage(gs, group, world_):
        """SpatialCrossAttention's sampling stage through the product API: rows of this rank's (camera,
        sub-slice) units reduced straight into the BEV slots (vidar_b200.sca.MSDARowsFunction), then the
        exchange on the BEV grid.  -> (bev [Q, 256] replicated, leaves)"""
        leaves, flat = [], []
        for g_ in gs:
            t = [g_["value"].detach().requires_grad_(True), g_["loc"].detach().requires_grad_(True),
                 g_["attn"].detach().requires_grad_(True)]
            leaves.append(t)
            flat += t
        slots = sca.MSDARowsFunction.apply([g_["plan"] for g_ in gs], 1, BEV_Q, shapes, lsi, None, None, inv_count, *flat)
        bev = slots[0]
        if world_ > 1:
            bev = sharding.all_gather_rows(sharding.reduce_scatter_rows(bev, group), BEV_Q, group)
        return bev, leaves

    def step(record):
        e = [ev() for _ in range(6)] if record else None
        if record:
            e[0].record()
        bev, leaves = msda_stage(groups, grp, world)
        if record:
            e[1].record()
        bev.backward(grad_bev)
        for g_, t in zip(groups, leaves):   # a camera split over ranks: sum its partial grad_value
            cam0, ncl = g_["plan"][0], g_["plan"][1]
            for c in range(cam0, cam0 + ncl):
                if c in cam_groups:
                    dist.all_reduce(t[0].grad[c - cam0], group=cam_groups[c])
        if record:
            e[2].record()
        latent.zero_grad(set_to_none=True)
        if world > 1:
            # row-sharded in / out (the module's consumers in the encoder -- LayerNorm, FFN -- are row-wise): only the
            # 2.56 MB occupancy / feature / prob maps cross NVLink, never the 41 MB grid
            emb = embed.view(-1, EMBED)[lr0:lr1].detach().requires_grad_(True)
            lat = latent.forward_rows(emb, 1, GRID[1], GRID[2])
            lat.backward(grad_embed.view(-1, EMBED)[lr0:lr1])
        else:
            emb = embed.detach().requires_grad_(True)
            lat = latent(emb)
            lat.backward(grad_embed)
        if record:
            e[3].record()
        sg = sigma[0].detach().requires_grad_(True)
        ce, valid = ray_head.ray_ce(sg, ce_origin, ce_points, ce_frame, WAYPOINTS, 1.0)
        ce.sum().backward()
        if record:
            e[4].record()
        pred, gt, grad_sigma = render.dvr.render(sigma, origin, points, tindex, "l2")
        # the dvxlr autograd layer (e2e_predictor_utils.py:91-115): forward + backward of sum(pred)
        sgd = sigma.detach().requires_grad_(True)
        dpred, _ = render.DifferentiableVoxelRendering(sgd, origin, points, tindex)
        dpred.sum().backward()
        ce_grad, dv_grad = sg.grad, sgd.grad
        if world > 1:
            # the three ray stages' partial sigma gradients (7.7 MB each) travel in ONE all-reduce
            ray_grads[0].copy_(ce_grad)
            ray_grads[1].copy_(grad_sigma[0])
            ray_grads[2].copy_(dv_grad[0])
            dist.all_reduce(ray_grads)
            ce_grad, grad_sigma, dv_grad = ray_grads[0], ray_grads[1][None], ray_grads[2][None]
        if record:
            e[5].record()
            marks.append(e)
        forward = dict(latent_out=lat.detach(), ray_ce_loss=ce.detach(), ray_ce_valid=valid, render_gt=gt,
                       dvxlr_pred=dpred.detach())
        return bev.detach(), leaves, pred, grad_sigma, emb.grad, ce_grad, dv_grad, forward

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step(False)
    sync()
    # ---- the step as ONE CUDA graph (kernels, memsets and the NCCL collectives): at N > 1 the ~40 launches
    #      and ~10 collectives of a 2 ms step are otherwise bound by the host's launch rate, not by the GPUs
    graph, mode = None, "eager"
    if args.graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                step(False)
            torch.cuda.current_stream(dev).wait_stream(side)
            sync()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                last = step(False)
            mode = "cuda graph replay (one graph per step)"
            graph.replay()                       # first replay outside the timed region
            sync()
        except Exception as ex:                  # capture is an optimisation: fall back to eager launches
            graph, mode = None, f"eager (graph capture failed: {type(ex).__name__}: {str(ex)[:120]})"
            torch.cuda.synchronize()
    ok = torch.tensor([1 if graph is not None else 0], device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) == 0 and graph is not None:   # every rank must take the same path
        graph, mode = None, "eager (graph capture failed on another rank)"
    sampler.mark_begin()
    n0 = _lib.launch_count()
    t0, t1 = ev(), ev()
    t0.record()
    for _ in range(args.steps):
        if graph is not None:
            graph.replay()
        else:
            last = step(True)
    t1.record()
    sync()
    sampler.mark_end()
    launches = _lib.launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None
    total_ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_step = total_ms / args.steps
    if getattr(args, "dump_outputs", None):
        # `last` holds the last timed step: the captured graph's output buffers after its final replay, or the
        # tensors of the last eager step
        dump_outputs(args.dump_outputs, step_outputs(last))
    if graph is not None:
        # per-stage breakdown (and the roofline's kernel time): the same step launched eagerly with events between
        # the stages -- identical kernels, outside the headline's timed region
        n1 = _lib.launch_count()
        for _ in range(args.steps):
            last = step(True)
        sync()
        launches = _lib.launch_count() - n1     # launches of K steps (a replayed graph does not pass through the C entry points)
    # median over the steps: the first eagerly launched step after a graph capture pays one-off allocations
    parts = {n: float(np.median([m[i].elapsed_time(m[i + 1]) for m in marks])) for i, n in enumerate(names)}

    if light:                                          # sweep: timing only
        if clocks is None and rank == 0:
            clocks = {}
        return {"ms_per_step": ms_step, "rays_per_s": RAYS / (ms_step * 1e-3), "breakdown_ms": parts, "launch_mode": mode,
                "rows_this_rank": rows}
    if os.environ.get("VIDAR_BENCH_PROFILE") == "1":   # under ncu: kernels only
        # one more step inside a cudaProfilerStart/Stop range: `ncu --profile-from-start off`
        # captures exactly this step's kernels (tools/profile_round.sh)
        torch.cuda.profiler.start()
        step(False)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        if rank == 0:
            _emit(json.dumps({"profile_only": True, "ms_per_step": ms_step, "breakdown_ms": parts}))
        return

    # ---- sharded == single GPU: every rank recomputes nothing; rank-summed results are compared with an
    #      unsharded recompute of the same step on rank 0 (outside the timed region)
    sharded_check = None
    if world > 1:
        sharded_check = check_sharded(dev, rank, world, grp, last, groups, msda_stage, grad_bev, latent, embed, grad_embed,
                                      sigma, origin, (points_np, tindex_np), shapes, lsi, cam_groups)

    # ---- end-to-end through the plugin API with HOST buffers (pinned), copies timed
    e2e = None
    host_in = []                 # one piece per camera so that uploads, compute and downloads pipeline
    for g_ in groups:
        cam0, ncl, S, lo, hi = g_["plan"]
        for cl in range(ncl):
            host_in.append(dict(plan=(cam0 + cl, 1, S, lo, hi),
                                **{k: g_[k][cl:cl + 1].cpu().pin_memory() for k in ("value", "loc", "attn")}))
    h_gbev = grad_bev.cpu().pin_memory()
    h_sigma, h_origin = sigma.cpu().pin_memory(), origin.cpu().pin_memory()
    h_points, h_tindex = points.cpu().pin_memory(), tindex.cpu().pin_memory()
    h_embed, h_gembed = embed.cpu().pin_memory(), grad_embed.cpu().pin_memory()
    h2d = sum(h[k].numel() * 4 for h in host_in for k in ("value", "loc", "attn")) + 4 * (
        h_gbev.numel() + h_sigma.numel() + h_origin.numel() + h_points.numel() + h_tindex.numel()
        + h_embed.numel() + h_gembed.numel())
    # Copies and compute are pipelined on three streams (H2D / compute / D2H): while camera c
    # computes, camera c+1 is uploading and camera c-1 is downloading (PCIe is full duplex).
    # A step still ends with every result in pinned host memory.
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    s_cmp = torch.cuda.current_stream(dev)

    def upload(host_tensors):
        with torch.cuda.stream(s_in):
            t = [h.to(dev, non_blocking=True) for h in host_tensors]
            ev_ = torch.cuda.Event()
            ev_.record(s_in)
        return t, ev_

    def download(dev_tensors, key):
        nonlocal host_out
        if key not in host_out:
            host_out[key] = [torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in dev_tensors]
        done = torch.cuda.Event()
        done.record(s_cmp)
        with torch.cuda.stream(s_out):
            s_out.wait_event(done)
            for hb, t in zip(host_out[key], dev_tensors):
                hb.copy_(t, non_blocking=True)
                t.record_stream(s_out)

    host_out = {}

    def e2e_step():
        ups = [upload([h[k] for k in ("value", "loc", "attn")]) for h in host_in]
        up_g = upload([h_gbev])
        up_r = upload([h_sigma, h_origin, h_points, h_tindex])
        up_l = upload([h_embed, h_gembed])
        parts_, leaves_ = [], []
        for h, (t, e_) in zip(host_in, ups):
            s_cmp.wait_event(e_)
            for x in t:
                x.record_stream(s_cmp)
            v, loc, aw = t
            v.requires_grad_(True), loc.requires_grad_(True), aw.requires_grad_(True)
            parts_.append(sca.MSDARowsFunction.apply([h["plan"]], 1, BEV_Q, shapes, lsi, None, None, inv_count, v, loc, aw)[0])
            leaves_.append((h["plan"][0], v, loc, aw))
        bev = parts_[0] if len(parts_) == 1 else torch.stack(parts_).sum(0)
        if world > 1:
            bev = sharding.all_gather_rows(sharding.reduce_scatter_rows(bev, grp), BEV_Q, grp)
        download([bev.detach()], "bev")
        (gb,), e_ = up_g
        s_cmp.wait_event(e_)
        gb.record_stream(s_cmp)
        bev.backward(gb)
        for i, (c, v, loc, aw) in enumerate(leaves_):
            if c in cam_groups:
                dist.all_reduce(v.grad, group=cam_groups[c])
            download([v.grad, loc.grad, aw.grad], ("msda", i))
        (sg, og, pt, ti), e_ = up_r
        s_cmp.wait_event(e_)
        for x in (sg, og, pt, ti):
            x.record_stream(s_cmp)
        (emb, gemb), e_ = up_l
        s_cmp.wait_event(e_)
        emb.record_stream(s_cmp), gemb.record_stream(s_cmp)
        emb.requires_grad_(True)
        lo = latent(emb)
        lo.backward(gemb)
        download([lo.detach(), emb.grad], "latent")
        sg2 = sg[0].detach().requires_grad_(True)
        ce, valid = ray_head.ray_ce(sg2, og[0].contiguous(), pt[0].contiguous(), ti[0].to(torch.int32), WAYPOINTS, 1.0)
        ce.sum().backward()
        download([ce.detach(), sg2.grad] + list(render.dvr.render(sg, og, pt, ti, "l2")), "rays")
        s_cmp.wait_stream(s_out)        # the step's results are on the host before it ends

    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        e2e_step()
    sync()
    a, b = ev(), ev()
    a.record()
    for _ in range(e2e_steps):
        e2e_step()
    b.record()
    sync()
    e2e_ms = a.elapsed_time(b) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    d2h = sum(t.numel() * 4 for ts in host_out.values() for t in ts)
    e2e = {"value": RAYS / (e2e_ms * 1e-3), "unit": "rays/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "api": "vidar_b200.sca.MSDARowsFunction (rows -> BEV slots) + BEV-grid exchange + backward, LatentRendering "
                  "module, ray_head.ray_ce, dvr.render; pinned host tensors in, pinned host tensors out; "
                  "H2D / compute / D2H on three streams"}

    if rank != 0:
        _finish(world)
        return

    # ---- roofline of the dominant kernel (msda_backward_kernel), this rank's launches
    peak, peak_src = peaks()
    fwd_b, bwd_b = msda_algorithmic_bytes(rows, len(my_cams))
    dom = "msda_bwd" if parts["msda_bwd"] >= parts["msda_fwd"] else "msda_fwd"
    dom_bytes = bwd_b if dom == "msda_bwd" else fwd_b
    n_launch = len(groups)
    achieved = dom_bytes / (parts[dom] * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp) and world == 1:
        with open(tp) as fh:
            traffic = json.load(fh).get(dom)
    roofline = {"bound": "hbm", "kernel": "msda_backward_kernel<8>" if dom == "msda_bwd" else "msda_forward_kernel<8>",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom_bytes / n_launch,
                "avg_launch_ms": parts[dom] / n_launch,
                "note": "duration = CUDA events around the op in the timed region (incl. grad_value "
                        "zero-fill for bwd); gather traffic is served by L2, see DESIGN.md"}
    cpu = cpu_baseline(sample_only=True) if world == 1 else {"note": "timed at N=1 only (rank 0), see the N=1 line"}
    line = {
        "metric": METRIC, "value": RAYS / (ms_step * 1e-3), "unit": "rays/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (seeded: perspective pillar fan per camera, LiDAR-like rays)",
        "config": bench_config(world),
        "breakdown_ms": parts, "launch_mode": mode, "sharded_check": sharded_check, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu,
        "msda_query_samples_per_s": NUM_CAMS * BEV_Q * HEADS * len(LEVELS) * POINTS / ((parts["msda_fwd"] + parts["msda_bwd"]) * 1e-3),
    }
    _emit(json.dumps(line))
    _finish(world)


DUMP_SAMPLE = 1 << 20        # elements kept of a larger output: the 14 outputs of a step stay under 64 MB


def step_outputs(last):
    """{name: tensor} of what one step hands its caller: the forward results and the input gradients of every stage."""
    bev, leaves, pred, grad_sigma, gemb, ce_grad, dv_grad, forward = last
    out = {"msda_bev": bev}
    for i, name in enumerate(("value", "sampling_loc", "attention_weights")):
        out[f"msda_grad_{name}"] = torch.cat([t[i].grad.reshape(-1) for t in leaves])
    out.update(latent_out=forward["latent_out"], latent_grad_embed=gemb, ray_ce_loss=forward["ray_ce_loss"],
               ray_ce_valid=forward["ray_ce_valid"], ray_ce_grad_sigma=ce_grad, render_pred=pred,
               render_gt=forward["render_gt"], render_grad_sigma=grad_sigma, dvxlr_pred=forward["dvxlr_pred"],
               dvxlr_grad_sigma=dv_grad)
    return out


def dump_outputs(out_dir, arrays):
    """Write every tensor as out_dir/<name>.npy in float32.  An output of more than DUMP_SAMPLE elements is
    flattened and reduced to DUMP_SAMPLE of its elements, at ascending flat indices drawn from a fixed seed: the
    same elements on every run, so two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
    assert total <= 64 << 20, f"--dump-outputs wrote {total} bytes"


def check_sharded(dev, rank, world, grp, last, groups, msda_stage, grad_bev, latent, embed, grad_embed, sigma, origin,
                  rays_np, shapes, lsi, cam_groups):
    """Sharded == single GPU, checked on the lease the scaling run gets (SCALE_rNN.json carries the result).
    The last timed step's results -- BEV grid, grad_value / grad_loc / grad_attn (summed over ranks into full
    tensors), both ray stages' grad_sigma, LatentRendering's input gradient -- against an UNSHARDED recompute of
    the same step on every rank (plan for world 1, all rays, no process group).  -> {name: max|a-b| / max|b|}"""
    import torch.distributed as dist

    from vidar_b200 import ray_head, render, sca
    bev, leaves, pred, grad_sigma, gemb, ce_grad, dv_grad, _ = last
    full = sca_like_inputs(dev)
    ref_groups = [dict(plan=sca.unit_plan(1, 0, NUM_CAMS)[0], value=full["value"], loc=full["loc"], attn=full["attn"])]
    rbev, rleaves = msda_stage(ref_groups, None, 1)
    rbev.backward(grad_bev)
    rv, rl, ra = (t.grad for t in rleaves[0])

    def rel(a, b):
        return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    out = {"bev_grid": rel(bev, rbev.detach())}
    gv = torch.zeros_like(rv)
    gl, ga = torch.zeros_like(rl), torch.zeros_like(ra)
    for g_, t in zip(groups, leaves):
        cam0, ncl = g_["plan"][0], g_["plan"][1]
        for cl in range(ncl):
            c = cam0 + cl
            # a shared camera's grad_value was already summed inside its group: count it once
            owner = c not in cam_groups or dist.get_rank(cam_groups[c]) == 0
            if owner:
                gv[c] += t[0].grad[cl]
            gl[c] += t[1].grad[cl]
            ga[c] += t[2].grad[cl]
    for t in (gv, gl, ga):
        dist.all_reduce(t, group=grp)
    out["grad_value"], out["grad_sampling_loc"], out["grad_attn_weight"] = rel(gv, rv), rel(gl, rl), rel(ga, ra)
    del full, ref_groups, rleaves, gv, gl, ga
    # rays: all of them on this rank
    points_np, tindex_np = rays_np
    pts, ti = torch.from_numpy(points_np).to(dev), torch.from_numpy(tindex_np).to(dev)
    sg = sigma[0].detach().requires_grad_(True)
    ce, _ = ray_head.ray_ce(sg, origin[0].contiguous(), pts[0].contiguous(), ti[0].to(torch.int32).contiguous(), WAYPOINTS, 1.0)
    ce.sum().backward()
    _, _, rgs = render.dvr.render(sigma, origin, pts, ti, "l2")
    out["ray_ce_grad_sigma"], out["render_grad_sigma"] = rel(ce_grad, sg.grad), rel(grad_sigma, rgs)
    sgd = sigma.detach().requires_grad_(True)
    dp, _ = render.DifferentiableVoxelRendering(sgd, origin, pts, ti)
    dp.sum().backward()
    out["dvxlr_layer_grad_sigma"] = rel(dv_grad, sgd.grad)
    # LatentRendering: same module without the process group
    pg, latent.process_group = latent.process_group, None
    emb = embed.detach().requires_grad_(True)
    latent.zero_grad(set_to_none=True)
    ro = latent(emb)
    ro.backward(grad_embed)
    latent.process_group = pg
    # the sharded step returns this rank's rows of grad_embed: compare them with the same rows of the full gradient
    from vidar_b200 import sharding
    a0, a1 = sharding.shard_range(GRID[1] * GRID[2], rank, world)
    out["latent_grad_embed_rows"] = rel(gemb, emb.grad.view(-1, EMBED)[a0:a1])
    worst = torch.tensor([max(out.values())], device=dev)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX, group=grp)
    out["max_over_ranks"] = float(worst.item())
    out["tolerance"] = 1e-4
    out["ok"] = bool(out["max_over_ranks"] <= 1e-4)
    return out


# ------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU path for MSDA (multi_scale_deformable_attn_pytorch formula) and
# the C port of the ray-caster (the reference has no CPU ray-caster), on a bounded sample.
# ------------------------------------------------------------------------------------------
class CpuArm:
    """The reference's CPU formulas for the step on a bounded SAMPLE: the same fraction f of every stage's
    units, so a sample-step is f of the job and  rays/s = f * 30000 / t_sample  (ms_per_step is the measured
    time of the sample-step, not an extrapolation):
      MSDA fwd+bwd     torch CPU grid_sample formula (= mmcv's multi_scale_deformable_attn_pytorch, the
                       reference's own CPU path), all 6 cameras, f * 40000 queries each (every camera pays the
                       cost of touching its 31.6 MB value / grad_value);
      LatentRendering  reference formula (torch CPU) on f * 40000 BEV cells;
      head sampler+CE  reference formula (torch CPU) on f * 30000 rays;
      dvr.render + dvxlr layer   C/OpenMP port (oracle/dvr_ref.c) on f * 30000 rays.
    The number of torch threads is calibrated once (more threads than ~32 is slower for these ops on
    many-core hosts)."""

    def __init__(self):
        self.full = sca_like_inputs(torch.device("cpu"), cams=NUM_CAMS, Q=BEV_Q, seed=0)
        g = torch.Generator().manual_seed(3)
        mk = lambda f: f(1, GRID[1], GRID[2], GRID[0], generator=g)
        self.lat = (mk(torch.randn), mk(torch.randn), mk(torch.rand))
        self.rays = ray_inputs()
        self.threads = self._calibrate_threads()

    def _calibrate_threads(self):
        cores = os.cpu_count() or 1
        best, best_t = cores, None
        for n in sorted({min(cores, c) for c in (8, 16, 32, 64, cores)}):
            torch.set_num_threads(n)
            self._msda(250, cams=1)                       # warm
            t = self._msda(500, cams=1)
            if best_t is None or t < best_t:
                best, best_t = n, t
        torch.set_num_threads(best)
        return best

    def _msda(self, q, cams=NUM_CAMS):
        from oracle import msda_ref
        d = self.full
        lo = (BEV_Q - q) // 2
        t0 = time.perf_counter()
        for c in range(cams):
            v = d["value"][c:c + 1].detach().requires_grad_(True)
            loc = d["loc"][c:c + 1, lo:lo + q].detach().contiguous().requires_grad_(True)
            aw = d["attn"][c:c + 1, lo:lo + q].detach().contiguous().requires_grad_(True)
            out = msda_ref.msda_grid_sample(v, d["shapes"], loc, aw)
            out.backward(d["grad_out"][c:c + 1, lo:lo + q].contiguous())
        return time.perf_counter() - t0

    def _latent(self, cells):
        from oracle import latent_render_ref as lr
        occ, feat, probmap = self.lat
        t0 = time.perf_counter()
        o, f = occ.detach().requires_grad_(True), feat.detach().requires_grad_(True)
        p, q = lr.latent_core(o, f, LR_GRID_NUM, 0.5, 1e-3, "sigmoid", cells=slice(0, cells), prob_map=probmap)
        (p.sum() + q.sum()).backward()
        return time.perf_counter() - t0

    def _ray_ce(self, rays_n):
        from oracle import ray_head_ref as rr
        sigma, origin, points, tindex = self.rays
        t0 = time.perf_counter()
        s = torch.from_numpy(sigma[0]).requires_grad_(True)
        tot = 0
        for f in range(FRAMES):
            sel = np.flatnonzero(tindex[0] == f)[: max(1, rays_n // FRAMES)]
            lg, ln, vd = rr.sample_frame(s[f], torch.from_numpy(origin[0, f]), torch.from_numpy(points[0][sel]), WAYPOINTS, 1.0)
            tot = tot - torch.log_softmax(lg[vd], -1)[:, 0].sum()
        tot.backward()
        return time.perf_counter() - t0

    def _render(self, rays_n):
        from oracle import dvr_ref
        sigma, origin, points, tindex = self.rays
        t0 = time.perf_counter()
        pts, ti = np.ascontiguousarray(points[:, :rays_n]), np.ascontiguousarray(tindex[:, :rays_n])
        dvr_ref.render(sigma, origin, pts, ti, "l2")
        pred, _ = dvr_ref.dvxlr_forward(sigma, origin, pts, ti)                       # the dvxlr autograd layer
        dvr_ref.dvxlr_autograd_backward(sigma, origin, pts, ti, np.ones_like(pred))
        return time.perf_counter() - t0

    def step(self, f):
        """One pass over fraction f of every stage -> (seconds, per-stage seconds)."""
        parts = {"msda": self._msda(max(8, int(BEV_Q * f))), "latent_render": self._latent(max(8, int(GRID[1] * GRID[2] * f))),
                 "ray_ce": self._ray_ce(max(FRAMES, int(RAYS * f))), "dvr_render": self._render(max(1, int(RAYS * f)))}
        return sum(parts.values()), parts

    def run(self, steps, warmup, budget_s, full_step=False):
        """`warmup` untimed + `steps` timed sample-steps within about `budget_s` seconds of CPU work.
        -> dict(f, seconds per sample-step (list), per-stage seconds, optional measured full step)."""
        self.step(0.01)                                                # first touch of every buffer / code path
        t1, _ = self.step(0.02)                                        # two-point calibration t(f) = a + b f
        t2, _ = self.step(0.08)
        b = max((t2 - t1) / 0.06, 1e-6)
        a = max(t1 - 0.02 * b, 0.0)
        per_step = budget_s / max(steps + warmup, 1)
        f = float(min(1.0, max(0.02, (per_step - a) / b)))
        for _ in range(max(warmup - 1, 0)):
            self.step(f)
        res = [self.step(f) for _ in range(steps)]
        out = {"f": f, "t": [r[0] for r in res], "parts": {k: float(np.mean([r[1][k] for r in res])) for k in res[0][1]}}
        if full_step:
            out["full_step_s"] = self.step(1.0)[0]
        return out

    def describe(self, r):
        from oracle import dvr_ref
        f = r["f"]
        txt = (f"each step = fraction f={f:.3f} of every stage on {self.threads} torch threads / {dvr_ref.num_threads()} OpenMP "
               f"threads: MSDA fwd+bwd (torch CPU grid_sample formula = the reference's CPU path) 6 cameras x {int(BEV_Q * f)} "
               f"queries; LatentRendering core (reference formula) {int(GRID[1] * GRID[2] * f)} cells; head ray sampler+CE "
               f"(reference formula) {int(RAYS * f)} rays; C/OpenMP port of dvr.render and of the dvxlr layer {int(RAYS * f)} rays.  Mean seconds per "
               "sample-step by stage: " + ", ".join(f"{k}={v:.2f}" for k, v in r["parts"].items())
               + f"; rays/s = f*{RAYS}/t_sample")
        if "full_step_s" in r:
            txt += f"; ONE full-size step (f=1) measured afterwards: {r['full_step_s']:.1f} s = {RAYS / r['full_step_s']:.0f} rays/s"
        return txt


def cpu_baseline(sample_only=False, steps=2, warmup=1, budget_s=20.0):
    arm = CpuArm()
    r = arm.run(steps, warmup, budget_s)
    t = float(np.mean(r["t"]))
    return {"value": r["f"] * RAYS / t, "unit": "rays/s", "cores": arm.threads, "kind": "port", "estimated": r["f"] < 1.0,
            "sample_fraction": r["f"], "sample_ms_per_step": t * 1e3, "sample": arm.describe(r)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm()
    # the sampled steps stay within ~2 minutes; one honest full-size step is measured after them
    r = arm.run(args.steps, args.warmup, budget_s=float(os.environ.get("VIDAR_REF_BUDGET_S", "110")),
                full_step=os.environ.get("VIDAR_REF_FULL_STEP", "1") == "1")
    t = float(np.mean(r["t"]))
    value = r["f"] * RAYS / t
    sample = arm.describe(r)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic (same generator as the GPU arm)",
        "config": bench_config(args.gpus), "estimated": r["f"] < 1.0, "sample_fraction": r["f"],
        "note": "ms_per_step is the measured time of one SAMPLE step (fraction f of the job); value = f*30000 rays / that time",
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": arm.threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if "full_step_s" in r:
        line["full_step_measured_ms"] = r["full_step_s"] * 1e3
        line["full_step_rays_per_s"] = RAYS / r["full_step_s"]
    _emit(json.dumps(line))


# ------------------------------------------------------------------------------------------
# BASELINE.json configs[3]: the synthetic ViDAR-RN101 pre-training step (vidar_b200/pretrain.py)
# ------------------------------------------------------------------------------------------
PRETRAIN_WORKLOAD = ("configs[3]: ViDAR-RN101 pre-training step, 1 sample: 4 frames (3 history no-grad + current) x 6 cams x "
                     "3x928x1600 -> RN101+FPN(4 lvls, 256ch) -> 6-layer BEV encoder (TSA, SCA, LatentRendering@layer2, FFN; "
                     "200x200 BEV) -> 3 future frames x 3-layer decoder -> 5 head frames x ray CE + dense Chamfer losses on "
                     "40000 LiDAR-like rays; backward, gradient sync, clip, AdamW")


def _eager_reference_ops():
    """`--workload pretrain --impl reference`: MSDA and the LatentRendering core through the reference's torch formulas on the GPU
    (mmcv's multi_scale_deformable_attn_pytorch / latent_rendering.py statements, as restated in oracle/),
    the rest of the graph unchanged -- the same-box eager baseline of the two hot paths inside the step."""
    from oracle import latent_render_ref, msda_ref
    from vidar_b200.modules import deform_attn, latent_rendering

    def msda_eager(value, shapes, lsi, loc, attn, im2col_step):
        return msda_ref.msda_grid_sample(value, shapes, loc, attn)
    deform_attn.msda_apply = msda_eager
    act = {0: "exp", 1: "sigmoid"}

    def core_eager(occ, feat, grid_num, grid_step, eps, act_id, group=None):
        return latent_render_ref.latent_core(occ, feat, grid_num, grid_step, eps, act[act_id])
    latent_rendering.latent_render_core = core_eager


def run_pretrain(args):
    import torch.distributed as dist

    from vidar_b200 import _lib, pretrain
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    grp = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        grp = dist.group.WORLD
    row_sharded = bool(getattr(args, "row_sharded", False)) and world > 1
    model, opt = pretrain.build(dev, grp, row_sharded=row_sharded)
    eager = args.impl == "reference"
    if eager:
        _eager_reference_ops()
        for layer in model.encoder:
            layer.cross_attn.fuse_rebatch = False
            layer.cross_attn.deformable_attention.fuse_epilogue = False
            if layer.latent_render is not None:
                layer.latent_render.fuse_projections = False
    sample = pretrain.synthetic_sample(dev)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        loss, _ = pretrain.train_step(model, opt, sample, grp)
    sync()
    sampler.mark_begin()
    n0 = _lib.launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        loss, _ = pretrain.train_step(model, opt, sample, grp)
    t1.record()
    sync()
    sampler.mark_end()
    launches = _lib.launch_count() - n0
    ms = t0.elapsed_time(t1) / args.steps
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    _, stages = pretrain.train_step(model, opt, sample, grp, record=True)       # one more step with per-stage events
    clocks = sampler.stop() if rank == 0 else None
    peak_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    if rank == 0:
        agg = {}
        for name, v in stages:
            key = name.split(".")[-1] if name.startswith("hist") else name
            key = ("history." + key) if name.startswith("hist") else key
            agg[key] = agg.get(key, 0.0) + float(v)
        _emit(json.dumps({
            "metric": "ms/step (synthetic ViDAR-RN101 pre-training step: forward + backward + grad sync + AdamW)",
            "value": ms, "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (cuDNN convolutions may use TF32, as in the reference's default PyTorch settings)",
            "data": "synthetic (N(0,1) frames, nuScenes-like 6-camera rig, LiDAR-like rays)", "samples_per_s": 1e3 / ms,
            "config": {"workload": PRETRAIN_WORKLOAD, "ops": "eager reference formulas (MSDA, LatentRendering core)" if eager else "vidar_b200 CUDA ops",
                       "sharding": ("single GPU" if world == 1 else
                                    "one sample over all ranks: cameras (backbone, SCA) and BEV rows (SCA output, LatentRendering) sharded, rest replicated"
                                    + ("; encoder row-wise stages (TSA, norms, FFN) on the rank's BEV rows" if row_sharded else ""))},
            "impl": "reference (eager torch formulas of the two hot paths, same GPU)" if eager else "ours",
            "stage_ms": agg, "loss": float(loss), "peak_mem_gb": peak_gb, "clocks": clocks, "gpu_launches": int(launches)}))
    if world > 1:
        dist.destroy_process_group()


def _finish(world):
    """End of a multi-rank run.  With a captured CUDA graph that contains NCCL kernels, tearing the process group
    down (or the interpreter's exit handlers) was seen to hang for minutes AFTER the JSON line was out (8 and 4
    ranks, gpurun r2h): every result is already written, so the ranks leave without running destructors."""
    if world > 1:
        import torch.distributed as dist
        # nobody leaves before rank 0 has written the line (a rank that disappears early could be noticed by the
        # peers' NCCL watchdog); the barrier is an ordinary collective, which is not what hung
        guard = threading.Timer(30.0, lambda: os._exit(0))      # every result is out: never wait on teardown for long
        guard.daemon = True
        guard.start()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def _emit(line):
    """The JSON line is the ONLY thing this process writes to the real stdout."""
    os.write(_REAL_STDOUT, (line + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    # libraries (NCCL's version banner, extension loaders) print to fd 1: park it on stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="launch the timed steps eagerly instead of replaying a CUDA graph")
    ap.add_argument("--row-sharded", dest="row_sharded", action="store_true",
                    help="--workload pretrain, N > 1: TSA / norms / FFN of the encoder on the rank's BEV rows (EncoderLayer.forward_rows)")
    ap.add_argument("--workload", default="hotpath", choices=["hotpath", "pretrain"],
                    help="hotpath: BASELINE configs[1]+[2] (the headline line); pretrain: configs[3], the synthetic ViDAR-RN101 step "
                         "(--impl reference there = the same graph with the reference's eager torch formulas for MSDA / LatentRendering, on the GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32; "
                         f"an output of more than {DUMP_SAMPLE} elements as a fixed, seeded sample of that many)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload, args.impl, args.gpus) != ("hotpath", "ours", 1):
        ap.error("--dump-outputs writes the single-GPU hot path's outputs (--workload hotpath --impl ours --gpus 1)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload == "pretrain":
        run_pretrain(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
