"""Point-cloud forecasting metrics on the device: Chamfer-inner, ray L1 and ray AbsRel per (sample, frame).

The reference scores ViDAR in `ViDAR.forward_test` (projects/mmdet3d_plugin/bevformer/detectors/vidar.py:389-502)
with per-(sample, frame) boolean masks, `.cpu().numpy()` copies and a numpy ray clamp
(bevformer/utils/eval_utils.py, bevformer/utils/e2e_predictor_utils.py:146-184).  Here:

  evaluate_rays                      the whole metric stage of a decoded batch -> [bs, F, 4] device tensor,
                                     no host sync (csrc/eval.cu + the nearest-neighbour kernel)
  compute_chamfer_distance_inner     drop-in for e2e_predictor_utils.py:173-184
  compute_ray_errors                 drop-in for eval_utils.compute_ray_errors -> (l1, absrel)
  ret_dict_from_metrics              the `{'frame.i': {...}}` dict forward_test returns (vidar.py:450-497)

CUDA tensors only, like everything else in this package.
"""
import numpy as np
import torch

from . import _lib
from .chamfer import knn_points

# columns of the metrics tensor
CHAMFER, L1, ABSREL, COUNT = 0, 1, 2, 3
_RAISED = {-1.0: "Origin and the end point should not be identical (a degenerate ray reached the eval-box clamp)",
           -2.0: "a ray that meets the eval box could not be clamped into it (assert touches_volume)"}


def _gather(origin, points, tindex, gt_dist, pred_dist, pc_range, num_frames, eval_within_grid):
    """vidar_eval_gather -> dict of the padded per-segment lists and counts [4, N] (device)."""
    bs, M = points.shape[:2]
    N = bs * num_frames
    dev = points.device
    f = dict(device=dev, dtype=torch.float32)
    out = dict(pred_in=torch.empty((N, M, 3), **f), gt_in=torch.empty((N, M, 3), **f),
               pred_sph=torch.empty((N, M, 3), **f), pred_dhat=torch.empty((N, M), **f),
               gt_sph=torch.empty((N, M, 3), **f), gt_pts=torch.empty((N, M, 3), **f),
               counts=torch.empty((4, N), dtype=torch.int64, device=dev))
    rng = np.ascontiguousarray(np.asarray(pc_range, np.float64).astype(np.float32))
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vidar_eval_gather(
            _lib.ptr(origin), _lib.ptr(points), _lib.ptr(tindex), _lib.ptr(gt_dist), _lib.ptr(pred_dist),
            rng.ctypes.data, int(bool(eval_within_grid)), _lib.ptr(out["pred_in"]), _lib.ptr(out["gt_in"]),
            _lib.ptr(out["pred_sph"]), _lib.ptr(out["pred_dhat"]), _lib.ptr(out["gt_sph"]), _lib.ptr(out["gt_pts"]),
            _lib.ptr(out["counts"]), bs, M, num_frames, _lib.stream_ptr(dev)))
    return out


def _ray_errors(origin, pred_dhat, gt_pts, nn_idx, cham_fwd, cham_bwd, counts):
    N, Mp = pred_dhat.shape
    Mg = gt_pts.shape[1]
    out = torch.empty((N, 4), dtype=torch.float64, device=gt_pts.device)
    with torch.cuda.device(gt_pts.device):
        _lib.check(_lib.lib().vidar_eval_ray_errors(
            _lib.ptr(origin), _lib.ptr(pred_dhat), _lib.ptr(gt_pts), _lib.ptr(nn_idx), _lib.ptr(cham_fwd),
            _lib.ptr(cham_bwd), _lib.ptr(counts), _lib.ptr(out), N, Mp, Mg, _lib.stream_ptr(gt_pts.device)))
    return out


def _require_cuda(name, t):
    if not (torch.is_tensor(t) and t.is_cuda):
        raise RuntimeError(f"{name} must be a CUDA tensor")


def _f32(name, t, shape_dims):
    _require_cuda(name, t)
    if t.dim() != shape_dims:
        raise ValueError(f"{name}: expected {shape_dims} dimensions, got shape {tuple(t.shape)}")
    return t.float().contiguous()


def evaluate_rays(origin, points, tindex, gt_dist, pred_dist, pc_range, num_frames, eval_within_grid=False):
    """Metrics of every (sample, frame) of a decoded batch, without a host sync.

    origin [bs, F, 3] (metres), points [bs, M, 3] (metres, NaN padding), tindex [bs, M] (frame index, -1
    padding), gt_dist / pred_dist [bs, M] (metres): the padded tensors `ViDARRayHead.get_point_cloud_prediction`
    decodes.  The rays of frame t are those with tindex == t and gt_dist > 0 (and inside pc_range with
    `eval_within_grid`), the clouds those of `get_rendered_pcds`.
    -> [bs, F, 4] float64 = (chamfer-inner, l1, absrel, count): `compute_chamfer_distance_inner(pred, gt,
    pc_range)`, `compute_ray_errors(pred, gt, origin)` and the number of GT rays longer than 1 cm.  A count
    of -1 / -2 marks a segment on which the reference raises (degenerate ray / assert(touches_volume)); the
    consumer that reads the tensor raises RuntimeError there (`ret_dict_from_metrics`, `check_metrics`)."""
    origin = _f32("origin", origin, 3)
    points = _f32("points", points, 3)
    tindex = _f32("tindex", tindex, 2)
    gt_dist = _f32("gt_dist", gt_dist, 2)
    pred_dist = _f32("pred_dist", pred_dist, 2)
    bs, M = points.shape[:2]
    F = int(num_frames)
    if origin.shape[:2] != (bs, F) or tindex.shape != (bs, M) or gt_dist.shape != (bs, M) or pred_dist.shape != (bs, M):
        raise ValueError(f"evaluate_rays: shapes do not agree: origin {tuple(origin.shape)} (want [{bs}, {F}, 3]), "
                         f"points {tuple(points.shape)}, tindex {tuple(tindex.shape)}, gt_dist {tuple(gt_dist.shape)}, "
                         f"pred_dist {tuple(pred_dist.shape)}")
    if bs == 0 or F == 0:
        return torch.empty((bs, F, 4), dtype=torch.float64, device=points.device)
    if M == 0:      # no ray at all: Chamfer 0.0, 0 / 0 ray errors, count 0
        out = torch.zeros((bs, F, 4), dtype=torch.float64, device=points.device)
        out[..., L1:ABSREL + 1] = float("nan")
        return out
    g = _gather(origin, points, tindex, gt_dist, pred_dist, pc_range, F, eval_within_grid)
    c = g["counts"]
    fwd = knn_points(g["pred_in"], g["gt_in"], lengths1=c[0], lengths2=c[1])
    bwd = knn_points(g["gt_in"], g["pred_in"], lengths1=c[1], lengths2=c[0])
    nn = knn_points(g["gt_sph"], g["pred_sph"], lengths1=c[3], lengths2=c[2])
    out = _ray_errors(origin.view(bs * F, 3), g["pred_dhat"], g["gt_pts"], nn.idx[..., 0].contiguous(),
                      fwd.dists[..., 0].contiguous(), bwd.dists[..., 0].contiguous(), c)
    return out.view(bs, F, 4)


def check_metrics(metrics_host):
    """Raise RuntimeError where the reference would have raised (count column -1 / -2)."""
    m = np.asarray(metrics_host)
    bad = np.argwhere(m[..., COUNT] < 0)
    if bad.size:
        where = tuple(int(i) for i in bad[0])
        raise RuntimeError(f"{_RAISED.get(float(m[where + (COUNT,)]), 'evaluation error')} at segment {where}")


def ret_dict_from_metrics(metrics, start_idx=0):
    """[bs, F, 4] metrics -> forward_test's ret_dict (vidar.py:450-497): for every frame, the Chamfer / L1 / AbsRel
    of the batch elements summed in batch order (Chamfer as a Python float, L1 / AbsRel as float32 like the
    reference's numpy scalars) and count = number of batch elements.  One device -> host copy."""
    m = metrics.detach().cpu().numpy() if torch.is_tensor(metrics) else np.asarray(metrics)
    check_metrics(m)
    bs, F = m.shape[:2]
    ret = {}
    for f in range(F):
        cd, l1, ar = 0, np.float32(0), np.float32(0)
        for b in range(bs):
            cd += float(np.float32(m[b, f, CHAMFER]))
            l1 = l1 + np.float32(m[b, f, L1])
            ar = ar + np.float32(m[b, f, ABSREL])
        ret[f"frame.{f + start_idx}"] = dict(count=bs, chamfer_distance=cd, l1_error=l1, absrel_error=ar)
    return ret


def _cloud(name, pcd):
    _require_cuda(name, pcd)
    if pcd.dim() != 2 or pcd.shape[1] != 3:
        raise ValueError(f"{name}: expected [N, 3], got {tuple(pcd.shape)}")
    return pcd.float().contiguous()


def _cloud_lists(pcd, origin, pc_range):
    """The gather kernel on one cloud (every point its own ray, no distance rescaling)."""
    n = pcd.shape[0]
    if n == 0:
        pcd = torch.full((1, 3), float("nan"), device=pcd.device)
        tix = torch.full((1, 1), -1.0, device=pcd.device)
    else:
        tix = torch.zeros((1, n), device=pcd.device)
    return _gather(origin.view(1, 1, 3), pcd[None].contiguous(), tix, None, None, pc_range, 1, False)


def compute_chamfer_distance_inner(pred_pcd, gt_pcd, pc_range):
    """e2e_predictor_utils.py:173-184: Chamfer distance of the points of both clouds inside pc_range; 0.0 when
    either side is empty, else a 0-d CUDA tensor (the reference returns the same two types)."""
    pred_pcd, gt_pcd = _cloud("pred_pcd", pred_pcd), _cloud("gt_pcd", gt_pcd)
    o = torch.zeros(3, device=pred_pcd.device)
    p = _cloud_lists(pred_pcd, o, pc_range)
    g = _cloud_lists(gt_pcd, o, pc_range)
    n_p, n_g = p["counts"][0], g["counts"][1]
    if int(n_p) == 0 or int(n_g) == 0:
        return 0.0
    fwd = knn_points(p["pred_in"], g["gt_in"], lengths1=n_p.view(1), lengths2=n_g.view(1))
    bwd = knn_points(g["gt_in"], p["pred_in"], lengths1=n_g.view(1), lengths2=n_p.view(1))
    counts = torch.stack([n_p, n_g, torch.zeros_like(n_p), torch.zeros_like(n_p)]).view(4, 1)
    out = _ray_errors(o.view(1, 3), p["pred_dhat"], g["gt_pts"], torch.zeros((1, g["gt_pts"].shape[1]), dtype=torch.int64,
                      device=o.device), fwd.dists[..., 0].contiguous(), bwd.dists[..., 0].contiguous(), counts)
    return out[0, CHAMFER].float()


def compute_ray_errors(pred_pcd, gt_pcd, origin, device=None):
    """eval_utils.compute_ray_errors(pred_pcd, gt_pcd, origin, device) -> (l1_error, absrel_error) as Python
    floats.  `device` is accepted for the reference's signature; the tensors' device is used."""
    pred_pcd, gt_pcd = _cloud("pred_pcd", pred_pcd), _cloud("gt_pcd", gt_pcd)
    _require_cuda("origin", origin)
    origin = origin.float().reshape(3).contiguous()
    p = _cloud_lists(pred_pcd, origin, [0.0] * 6)
    g = _cloud_lists(gt_pcd, origin, [0.0] * 6)
    counts = torch.stack([torch.zeros_like(p["counts"][2]), torch.zeros_like(p["counts"][2]),
                          p["counts"][2], g["counts"][3]]).view(4, 1)
    nn = knn_points(g["gt_sph"], p["pred_sph"], lengths1=counts[3], lengths2=counts[2])
    out = _ray_errors(origin.view(1, 3), p["pred_dhat"], g["gt_pts"], nn.idx[..., 0].contiguous(), None, None, counts)
    m = out.cpu().numpy()
    check_metrics(m)
    return float(np.float32(m[0, L1])), float(np.float32(m[0, ABSREL]))
