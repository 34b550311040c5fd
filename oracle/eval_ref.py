"""CPU oracle for the point-cloud forecasting metrics.  TEST INFRASTRUCTURE.

numpy restatement (float32 throughout, like the reference's arrays under numpy >= 2) of
  * eval_utils `clamp` / `_clamp` / `spherical_projection` / `compute_ray_errors`
    (projects/mmdet3d_plugin/bevformer/utils/eval_utils.py), with `oracle.knn_ref.nn` as the
    nearest neighbour in (azimuth, elevation, 1) space,
  * e2e_predictor_utils `compute_chamfer_distance_inner` (utils/e2e_predictor_utils.py:146-184),
  * ViDARHeadBase.get_rendered_pcds (dense_heads/vidar_head_base.py:344-389), per (sample, frame).
Pinned against the reference's own functions run on CPU: tests/golden/eval.npz via tools/make_golden_eval.py.
One divergence, shared with the product: a frame with GT rays but no predicted ray beyond 1 cm gives NaN ray
errors here, where the reference fails with an IndexError."""
import numpy as np

from . import knn_ref

EVAL_BOX = np.float32([-70.0, -70.0, -4.5, 70.0, 70.0, 4.5])
# inside_volume widens the box by 0.02 (in float64) and compares in the array's dtype
SLACK_BOX = np.float32([-70.0 - 0.02, -70.0 - 0.02, -4.5 - 0.02, 70.0 + 0.02, 70.0 + 0.02, 4.5 + 0.02])


def _within(p, box):
    p = np.asarray(p, np.float32)
    return np.all((box[:3] <= p) & (p <= box[3:]), axis=-1)


def _norm(v):
    """sqrt of the squared components summed left to right, float32."""
    return np.sqrt(v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1] + v[..., 2] * v[..., 2])


def _sorted_plane_distances(q, d, sign):
    """[n, 6] distances from q [n, 3] along sign * d to the eval-box planes, MAX_VALUE where the direction component
    is close to 0, ascending (what happens at a plane depends on its distance only, so ties need no order)."""
    cols = []
    for a in range(3):
        close = np.isclose(d[:, a], 0.0)
        den = d[:, a] if sign > 0 else -d[:, a]
        for bound in (EVAL_BOX[a], EVAL_BOX[a + 3]):
            with np.errstate(divide="ignore", invalid="ignore"):
                cols.append(np.where(close, 1e8, (bound - q[:, a]) / den))
    return np.sort(np.stack(cols, 1).astype(np.float32), axis=1)


def clamp(pcd, origin):
    """eval_utils.clamp(pcd, origin, return_invalid_mask=True) -> (origins, points, invalid)."""
    pts = np.array(pcd, np.float32).reshape(-1, 3)
    o = np.asarray(origin, np.float32).reshape(3)
    origins = np.zeros_like(pts) + o
    outer = ~_within(pts, EVAL_BOX)
    if outer.any():
        p = pts[outer]
        e = p - o
        if np.any(np.all(e == 0, axis=1)):
            raise RuntimeError("origin and end point of a ray are identical")
        length = _norm(e)
        d = e / length[:, None]
        new_o = np.zeros_like(p) + o
        o_inside = bool(_within(o, SLACK_BOX))
        hit = np.full(p.shape[0], o_inside)
        if not o_inside:                                    # enter the box from outside
            t = _sorted_plane_distances(np.broadcast_to(o, p.shape), d, 1)
            for i in range(p.shape[0]):
                for k in range(6):
                    if t[i, k] + np.float32(1e-4) >= 0:
                        x = o + t[i, k] * d[i]
                        if _within(x, SLACK_BOX):
                            hit[i] = True
                            new_o[i] = x
                            if t[i, k] > length[i]:
                                p[i] = x
                            break
        t = _sorted_plane_distances(p, d, -1)               # from the (possibly moved) end point, backwards
        for i in range(p.shape[0]):
            if not hit[i]:
                new_o[i] = np.inf
                p[i] = np.inf
            elif not _within(p[i], SLACK_BOX):
                for k in range(6):
                    if t[i, k] + np.float32(1e-4) >= 0:
                        x = p[i] + t[i, k] * (-d[i])
                        if _within(x, SLACK_BOX):
                            p[i] = x
                            break
                else:
                    raise AssertionError("ray meets the eval box but cannot be clamped into it")
        pts[outer] = p
        origins[outer] = new_o
    invalid = np.all(np.isinf(pts), axis=1) | np.all(np.isnan(pts), axis=1)
    return origins, pts, invalid


def spherical(pcd, origin):
    """(azimuth, elevation, range) of pcd - origin."""
    q = np.asarray(pcd, np.float32).reshape(-1, 3) - np.asarray(origin, np.float32).reshape(1, 3)
    return np.arctan2(q[:, 0], q[:, 1]), np.arctan2(q[:, 2], q[:, 1]), _norm(q)


def ray_errors_detail(pred_pcd, gt_pcd, origin, nn=None):
    """compute_ray_errors -> dict(l1, absrel, count, idx): idx = nearest predicted ray (index among the predicted
    rays longer than 1 cm) of every GT ray longer than 1 cm.  `nn(gt_sph, pred_sph) -> idx` replaces the
    nearest-neighbour search (default `knn_ref.nn`)."""
    pred = np.asarray(pred_pcd, np.float32).reshape(-1, 3)
    gt = np.asarray(gt_pcd, np.float32).reshape(-1, 3)
    o = np.asarray(origin, np.float32).reshape(3)
    az_p, el_p, d_p = spherical(pred, o)
    az_g, el_g, d_g = spherical(gt, o)
    keep_p, keep_g = d_p > 1e-2, d_g > 1e-2
    count = int(keep_g.sum())
    sph_p = np.stack([az_p[keep_p], el_p[keep_p], np.ones(int(keep_p.sum()), np.float32)], 1)
    sph_g = np.stack([az_g[keep_g], el_g[keep_g], np.ones(count, np.float32)], 1)
    d_p, gt = d_p[keep_p], gt[keep_g]
    if count and not d_p.size:
        return dict(l1=np.float32(np.nan), absrel=np.float32(np.nan), count=count, idx=np.zeros(count, np.int64))
    if not count:
        idx = np.zeros(0, np.int64)
    else:
        idx = knn_ref.nn(sph_g[None], sph_p[None])[1][0] if nn is None else np.asarray(nn(sph_g, sph_p))
    v = gt - o
    unit = v / np.sqrt((v ** 2).sum(axis=1, keepdims=True))
    interp = o + d_p[idx][:, None] * unit
    g_o, g_p, invalid = clamp(gt, o)
    _, i_p, _ = clamp(interp, o)
    g_o, g_p, i_p = g_o[~invalid], g_p[~invalid], i_p[~invalid]
    dc = np.sqrt(((g_p - g_o) ** 2).sum(axis=1))
    ok = dc > 0.01
    eucl = np.sqrt(((g_p[ok] - i_p[ok]) ** 2).sum(axis=1))
    with np.errstate(invalid="ignore", divide="ignore"):
        l1 = eucl.sum() / np.float32(count)
        absrel = (eucl / dc[ok]).sum() / np.float32(count)
    return dict(l1=np.float32(l1), absrel=np.float32(absrel), count=count, idx=idx)


def compute_ray_errors(pred_pcd, gt_pcd, origin):
    r = ray_errors_detail(pred_pcd, gt_pcd, origin)
    return r["l1"], r["absrel"]


def compute_chamfer_distance_inner(pred_pcd, gt_pcd, pc_range):
    """0.0 when either cloud has no point inside pc_range, else the mean of both directions' mean squared NN distance."""
    box = np.asarray(pc_range, np.float64).astype(np.float32)
    pred = np.asarray(pred_pcd, np.float32).reshape(-1, 3)
    gt = np.asarray(gt_pcd, np.float32).reshape(-1, 3)
    pred, gt = pred[_within(pred, box)], gt[_within(gt, box)]
    if pred.shape[0] == 0 or gt.shape[0] == 0:
        return 0.0
    fwd = knn_ref.nn(pred[None], gt[None])[0][0].sum()
    bwd = knn_ref.nn(gt[None], pred[None])[0][0].sum()
    return np.float32((fwd / np.float32(pred.shape[0]) + bwd / np.float32(gt.shape[0])) / np.float32(2.0))


def rendered_pcds(origin, points, tindex, dist, mask_dist, pc_range=None, eval_within_grid=False):
    """get_rendered_pcds: pcds[b][t] = origin_t + unit(points - origin_t) * dist for the rays of frame t with
    mask_dist > 0 (and inside pc_range with eval_within_grid)."""
    origin, points = np.asarray(origin, np.float32), np.asarray(points, np.float32)
    out = []
    for b in range(origin.shape[0]):
        cur = []
        for t in range(origin.shape[1]):
            m = (np.asarray(tindex[b]) == t) & (np.asarray(mask_dist[b]) > 0)
            if eval_within_grid:
                m &= _within(points[b], np.asarray(pc_range, np.float64).astype(np.float32))
            r = points[b][m] - origin[b, t]
            r = r / np.sqrt((r ** 2).sum(1, keepdims=True))
            cur.append(origin[b, t] + r * np.asarray(dist[b], np.float32)[m][:, None])
        out.append(cur)
    return out


def evaluate_rays(origin, points, tindex, gt_dist, pred_dist, pc_range, eval_within_grid=False):
    """[bs, F, 4] (chamfer-inner, l1, absrel, count) of every (sample, frame), frame by frame like forward_test."""
    pred = rendered_pcds(origin, points, tindex, pred_dist, gt_dist, pc_range, eval_within_grid)
    gt = rendered_pcds(origin, points, tindex, gt_dist, gt_dist, pc_range, eval_within_grid)
    bs, F = np.asarray(origin).shape[:2]
    out = np.zeros((bs, F, 4), np.float64)
    for b in range(bs):
        for t in range(F):
            r = ray_errors_detail(pred[b][t], gt[b][t], np.asarray(origin, np.float32)[b, t])
            out[b, t] = (compute_chamfer_distance_inner(pred[b][t], gt[b][t], pc_range), r["l1"], r["absrel"], r["count"])
    return out
