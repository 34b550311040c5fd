"""Inputs of the evaluation goldens (tests/golden/eval.npz, tools/make_golden_eval.py): predicted / GT clouds in
metres (float32) and the sensor origin of one (sample, frame) each, seeded."""
import numpy as np

PC_RANGE = [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]


def _rays(rng, n, origin, r_lo, r_hi, elev_deg=(-25.0, 12.0)):
    az = rng.uniform(-np.pi, np.pi, n)
    el = np.deg2rad(rng.uniform(*elev_deg, n))
    u = np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], 1)
    r = rng.uniform(r_lo, r_hi, n)
    return u, r


def cases():
    rng = np.random.default_rng(2024)
    out = {}
    # ranges up to 95 m: beyond 51.2 m (Chamfer inner mask), xy beyond 70 m and z beyond +-4.5 m (clamp)
    o = np.array([0.4, -0.3, 1.8])
    u, r = _rays(rng, 300, o, 1.0, 95.0)
    gt = o + u * r[:, None]
    pred = o + u * (r * rng.uniform(0.7, 1.3, 300))[:, None]
    out["mixed"] = (pred, gt, o)
    # rays of at most 1 cm on both sides, and a predicted cloud of another size
    u, r = _rays(rng, 80, o, 2.0, 40.0)
    gt = o + u * r[:, None]
    gt[::9] = o + u[::9] * 0.006
    pu, pr = _rays(rng, 60, o, 2.0, 40.0)
    pred = o + pu * pr[:, None]
    pred[::7] = o + pu[::7] * 0.009
    out["short"] = (pred, gt, o)
    # duplicated directions on both sides: nearest-neighbour ties keep the smallest index
    u, r = _rays(rng, 20, o, 3.0, 60.0)
    uu = np.concatenate([u, u, u[:5]])
    gt = o + uu * np.concatenate([r, r * 1.1, r[:5] * 0.9])[:, None]
    pred = o + uu * np.concatenate([r * 0.8, r * 0.8, r[:5] * 0.8])[:, None]         # exact duplicates
    out["ties"] = (pred, gt, o)
    # origin outside the eval box (above it, and beyond x = 70 m): the entering branch of the clamp
    for name, oo in (("origin_above", np.array([5.0, -3.0, 9.0])), ("origin_far", np.array([82.0, 4.0, 0.5]))):
        tgt = np.concatenate([rng.uniform(-60, 60, (120, 2)), rng.uniform(-8, 3, (120, 1))], 1)
        v = tgt - oo
        d = np.linalg.norm(v, axis=1, keepdims=True)
        gt = oo + v / d * (d * rng.uniform(0.6, 1.4, (120, 1)))
        pred = oo + v / d * (d * rng.uniform(0.6, 1.4, (120, 1)))
        out[name] = (pred, gt, oo)
    # a frame without rays
    out["empty"] = (np.zeros((0, 3)), np.zeros((0, 3)), o)
    # GT entirely outside pc_range (Chamfer inner 0.0), ray errors still defined
    gt = np.concatenate([rng.uniform(-40, 40, (50, 2)), rng.uniform(3.2, 4.4, (50, 1))], 1)      # above z = 3 m
    pred = o + (gt - o) * rng.uniform(0.5, 1.5, (50, 1))
    out["gt_outside_range"] = (pred, gt, o)
    # a degenerate ray: the interpolated point of a 2 cm prediction rounds back onto a far-away origin (the
    # reference raises RuntimeError in the clamp)
    od = np.array([0.0, 0.0, 4194304.0])
    out["degenerate"] = (od[None] + np.array([[0.0, 0.02, 0.0]]), od[None] + np.array([[0.0, 0.0, 1000.0]]), od)
    return {k: tuple(np.asarray(a, np.float32) for a in v) for k, v in out.items()}
