"""Ego motion without a GPU: the numpy oracle and the host statements of vidar_b200/ego.py against goldens made by
the reference's own code (tools/make_golden_ego.py, tests/golden/ego.npz), the synthetic moving-ego queue, argument
validation of the C entry points and the CUDA-only rule."""
import os

import numpy as np
import pytest
import torch

from oracle import ego_ref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ego.npz")
PC_RANGE = [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
ROT_CASES = [f"rot{k}" for k in range(4)]


def _z():
    return np.load(GOLDEN)


def _index_image(H, W):
    return np.arange(1, H * W + 1, dtype=np.float32).reshape(1, H, W)


@pytest.mark.parametrize("case", ROT_CASES)
def test_oracle_rotation_equals_reference_golden(case):
    z = _z()
    H = W = 200
    for b, angle in enumerate(z[f"{case}.angles"]):
        want = z[f"{case}.src_index"][b].astype(np.float32).reshape(H, W)
        out, near, cands = ego_ref.rotate(_index_image(H, W), float(angle), [100, 100])
        np.testing.assert_array_equal(out[0][~near], want[~near])
        assert (cands[:, 0] == want[None]).any(0)[near].all()
        if float(angle) in (0.0, -90.0, 180.0):
            assert not near.any() and np.array_equal(out[0], want)


def test_rotation_theta_equals_oracle():
    from vidar_b200 import ego
    for angle in (0.0, 1e-3, -1e-3, 37.3, -90.0, 180.0, 271.25):
        for hw in ((200, 200), (100, 150)):
            a = ego.rotation_theta(angle, [100, 100], *hw)
            b = ego_ref.rescaled_theta(angle, [100, 100], *hw)
            assert a.dtype == np.float32 and a.shape == (3, 2) and np.array_equal(a, b)


@pytest.mark.parametrize("case", ROT_CASES)
def test_bev_shift_equals_reference_golden(case):
    from vidar_b200 import ego
    z = _z()
    metas = [dict(can_bus=z[f"{case}.can_bus"][b], lidar2global_rotation=z[f"{case}.lidar2global_rotation"][b])
             for b in range(2)]
    got = torch.tensor(ego.bev_shift(metas, (0.512, 0.512), 200, 200), dtype=torch.float32).numpy()
    np.testing.assert_array_equal(got, z[f"{case}.shift"])


def test_shifted_hybrid_reference_points_equal_reference_golden():
    from vidar_b200 import bev_geometry
    z = _z()
    ref_2d = bev_geometry.get_reference_points(50, 50, dim="2d", bs=2, device="cpu")
    shift = torch.from_numpy(z["hybrid.shift"])
    hybrid = torch.stack([ref_2d + shift[:, None, None, :], ref_2d], 1).reshape(4, 2500, 1, 2)
    np.testing.assert_array_equal(hybrid.numpy(), z["hybrid.ref_2d"])


def test_align_bev_coordinates_equals_reference_golden():
    from vidar_b200 import ego
    z = _z()
    keys = ("ref_lidar_to_cur_lidar", "future2ref_lidar_transform", "ref2future_lidar_transform")
    metas = [{k: z[f"dec.{k}"][b] for k in keys} for b in range(2)]
    prev = torch.zeros(2, 1, 600, 4)
    r2h = ego.history_ref_to_previous_transform(prev, 1, [[m] for m in metas])
    np.testing.assert_array_equal(r2h.numpy(), z["dec.ref_to_history0"])
    for k in range(1, 7):
        tgt, aligned, ref2future = ego.align_bev_coordinates(k, r2h, metas, 20, 30, PC_RANGE)
        np.testing.assert_allclose(tgt.numpy(), z[f"dec.{k}.tgt"], rtol=0, atol=1e-7)
        np.testing.assert_allclose(aligned.numpy(), z[f"dec.{k}.aligned"], rtol=0, atol=1e-6)
        r2h = torch.cat([r2h, ref2future.unsqueeze(1)], 1)[:, 1:].contiguous()


@pytest.mark.parametrize("case", ["loss0", "loss1", "loss2", "loss3", "loss4", "test"])
def test_oracle_gt_alignment_equals_reference_golden(case):
    from vidar_b200 import ego
    z = _z()
    keys = ("total_cur2ref_lidar_transform", "total_ref2cur_lidar_transform")
    metas = [{k: z[f"gt.{k}"][b] for k in keys} for b in range(2)]
    src, tgt = z[f"gt.{case}.src"], z[f"gt.{case}.tgt"]
    mats = ego.src_to_tgt_matrices(src, tgt, metas)
    slots = {int(f): s for s, f in enumerate(src)}
    for b in range(2):
        out, origins = ego_ref.align_points(z[f"gt.points{b}"], slots, mats[b])
        order = np.argsort(np.where(out[:, 3] < 0, len(src), out[:, 3]), kind="stable")
        got = out[order][out[order][:, 3] >= 0]
        want = z[f"gt.{case}.out{b}"]
        np.testing.assert_array_equal(got[:, 3], want[:, 3])
        np.testing.assert_allclose(got[:, :3], want[:, :3], rtol=0, atol=1e-6 * np.abs(want[:, :3]).max())
        np.testing.assert_allclose(origins, z[f"gt.{case}.origins"][b], rtol=0, atol=1e-6)


def test_ego_queue_is_self_consistent():
    """A static world point seen in frame k, moved by total_cur2ref[k] @ total_ref2cur[j], lands on its observation
    in frame j; the can_bus deltas agree with the poses."""
    from vidar_b200 import synthetic
    T, future = 4, 4
    q = synthetic.ego_queue(bs=2, T=T, future=future, seed=3, world_points=3000, points_per_frame=3000)
    for b in range(2):
        metas = q["img_metas"][b]
        cur = metas[T - 1]
        c2r, r2c = cur["total_cur2ref_lidar_transform"], cur["total_ref2cur_lidar_transform"]
        assert c2r.shape == (T + future, 4, 4) and np.allclose(c2r[T - 1], np.eye(4))
        # the same static world seen from every pose: a moved point meets an observation of frame j
        pts = q["gt_points"][b].astype(np.float64)
        for k, j in ((0, T - 1), (1, T + 2), (T + future - 1, 2)):
            pk, pj = pts[pts[:, 3] == k, :3], pts[pts[:, 3] == j, :3]
            moved = np.concatenate([pk, np.ones((len(pk), 1))], 1) @ c2r[k] @ r2c[j]
            d = np.sqrt(((moved[:, None, :3] - pj[None]) ** 2).sum(-1)).min(1)
            assert np.median(d) < 1e-4 and (d < 1e-4).mean() > 0.3, (k, j, np.median(d))
        for t in range(1, T):
            m, p = metas[t], metas[t - 1]
            g_t = np.asarray(m["ego2global_translation"]) - np.asarray(p["ego2global_translation"])
            np.testing.assert_allclose(m["can_bus"][:3], g_t, atol=1e-9)
            yaw = lambda q_: np.degrees(2 * np.arctan2(q_[3], q_[0])) % 360       # noqa: E731
            np.testing.assert_allclose(m["can_bus"][-1], yaw(m["ego2global_rotation"]) - yaw(p["ego2global_rotation"]),
                                       atol=1e-9)
            assert m["prev_bev_exists"]
        assert not metas[0]["prev_bev_exists"] and not metas[0]["can_bus"][:3].any()
        # future can_bus: the frame's origin in the previous future frame, and the yaw change
        for k in range(1, future + 1):
            o = np.array([0, 0, 0, 1.0]) @ cur["future2ref_lidar_transform"][k] @ cur["ref2future_lidar_transform"][k - 1]
            np.testing.assert_allclose(cur["future_can_bus"][k][:3], o[:3], atol=1e-9)


def test_entry_points_validate_arguments():
    """Every call returns VIDAR_E_INVALID with a message.  The calls run on a thread of their own: the last-error text
    is per thread, so the test leaves none behind on the main thread."""
    import threading
    errors = []
    t = threading.Thread(target=_run, args=(errors,))
    t.start()
    t.join()
    assert errors == [None], errors


def _run(errors):
    try:
        _validate_arguments()
        errors.append(None)
    except AssertionError as e:        # reported on the main thread
        errors.append(repr(e))


def _validate_arguments():
    import ctypes
    from vidar_b200 import _lib
    L = _lib.lib()
    theta = (ctypes.c_float * 6)()
    assert L.vidar_bev_rotate_forward(None, None, None, 1, 2, 2, 8, None) == 1
    assert b"null pointer" in L.vidar_last_error()
    assert L.vidar_bev_rotate_forward(ctypes.c_void_p(16), ctypes.cast(theta, ctypes.c_void_p), ctypes.c_void_p(64),
                                      1, 0, 2, 8, None) == 1
    assert b"bad sizes" in L.vidar_last_error()
    off = (ctypes.c_int64 * 2)(0, 0)
    slots = (ctypes.c_int32 * 2)(0, 5)
    mats = (ctypes.c_float * 16)()
    args = [ctypes.cast(x, ctypes.c_void_p) for x in (off, slots, mats)]
    assert L.vidar_ego_align_points(None, None, None, 1, None, None, None, 1, 1, None) == 1
    assert b"null pointer" in L.vidar_last_error()
    assert L.vidar_ego_align_points(None, args[0], args[1], 2, args[2], None, ctypes.c_void_p(16), 1, 1, None) == 1
    assert b"slot_of_frame" in L.vidar_last_error()
    assert L.vidar_ego_align_points(None, args[0], args[1], 65, args[2], None, ctypes.c_void_p(16), 1, 1, None) == 1
    assert b"num_frames" in L.vidar_last_error()
    bad = (ctypes.c_int64 * 2)(0, 5)
    assert L.vidar_ego_align_points(None, ctypes.cast(bad, ctypes.c_void_p), args[1], 1, args[2], None,
                                    ctypes.c_void_p(16), 1, 1, None) == 1
    assert b"null pointer" in L.vidar_last_error()


def test_ego_ops_raise_on_cpu_tensors():
    from vidar_b200 import ego
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        ego.rotate_prev_bev(torch.zeros(1, 4, 8), [0.0], [1, 1], 2, 2)
    metas = [dict(total_cur2ref_lidar_transform=np.eye(4)[None], total_ref2cur_lidar_transform=np.eye(4)[None])]
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        ego.align_gt_points([torch.zeros(3, 4)], [0], [0], metas)


def test_align_gt_points_validates_frames():
    from vidar_b200 import ego
    metas = [dict(total_cur2ref_lidar_transform=np.eye(4)[None].repeat(2, 0),
                  total_ref2cur_lidar_transform=np.eye(4)[None].repeat(2, 0))]
    with pytest.raises(ValueError, match="distinct"):
        ego.align_gt_points([torch.zeros(3, 4)], [1, 1], [0, 0], metas)
    with pytest.raises(ValueError, match="target frames"):
        ego.align_gt_points([torch.zeros(3, 4)], [0, 1], [0], metas)
