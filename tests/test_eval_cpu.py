"""The evaluation oracle (oracle/eval_ref.py) against the reference's own eval_utils / e2e_predictor_utils run on CPU
(tests/golden/eval.npz), and the host-side pieces of vidar_b200.evaluation that need no GPU."""
import os

import numpy as np
import pytest
import torch

from oracle import eval_ref
from tests.eval_cases import PC_RANGE, cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "eval.npz")
NAMES = sorted(cases())


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def test_golden_inputs_are_the_cases(golden):
    for name, (pred, gt, origin) in cases().items():
        np.testing.assert_array_equal(golden[f"{name}.pred"], pred)
        np.testing.assert_array_equal(golden[f"{name}.gt"], gt)
        np.testing.assert_array_equal(golden[f"{name}.origin"], origin)


@pytest.mark.parametrize("name", NAMES)
def test_oracle_equals_reference(golden, name):
    pred, gt, origin = golden[f"{name}.pred"], golden[f"{name}.gt"], golden[f"{name}.origin"]
    cd = eval_ref.compute_chamfer_distance_inner(pred, gt, PC_RANGE)
    np.testing.assert_allclose(cd, golden[f"{name}.chamfer"], rtol=1e-6)
    if bool(golden[f"{name}.raises"]):
        with pytest.raises(RuntimeError):
            eval_ref.ray_errors_detail(pred, gt, origin)
        return
    r = eval_ref.ray_errors_detail(pred, gt, origin)
    assert r["count"] == int(golden[f"{name}.count"])
    np.testing.assert_array_equal(r["idx"], golden[f"{name}.idx"])
    np.testing.assert_allclose(r["l1"], golden[f"{name}.l1"], rtol=1e-6, equal_nan=True)
    np.testing.assert_allclose(r["absrel"], golden[f"{name}.absrel"], rtol=1e-6, equal_nan=True)


def test_cases_cover_the_clamp_branches(golden):
    """The goldens exercise what the issue of clamping is about: points beyond the eval box in xy and z, origins
    outside it, rays of at most 1 cm, an empty frame and GT entirely outside pc_range."""
    pred, gt, o = (golden[f"mixed.{k}"] for k in ("pred", "gt", "origin"))
    assert (np.abs(gt[:, :2]) > 70).any() and (np.abs(gt[:, 2]) > 4.5).any() and (np.abs(gt[:, :2]) > 51.2).any()
    for name in ("origin_above", "origin_far"):
        assert not eval_ref._within(golden[f"{name}.origin"], eval_ref.SLACK_BOX)
    assert int(golden["short.count"]) < golden["short.gt"].shape[0]
    assert int(golden["empty.count"]) == 0 and np.isnan(golden["empty.l1"])
    assert float(golden["gt_outside_range.chamfer"]) == 0.0 and np.isfinite(golden["gt_outside_range.l1"])
    idx = golden["ties.idx"]
    assert idx.max() < 20, "duplicated directions: the nearest predicted ray is the first of its duplicates"


def test_cpu_tensors_are_refused():
    from vidar_b200 import evaluation
    p = torch.zeros(4, 3)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        evaluation.compute_chamfer_distance_inner(p, p, PC_RANGE)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        evaluation.compute_ray_errors(p, p, torch.zeros(3), "cpu")
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        evaluation.evaluate_rays(torch.zeros(1, 2, 3), torch.zeros(1, 4, 3), torch.zeros(1, 4), torch.zeros(1, 4),
                                 torch.zeros(1, 4), PC_RANGE, 2)


def test_ret_dict_from_metrics_has_the_reference_structure():
    """vidar.py:450-497: one entry per frame, keys count / chamfer_distance / l1_error / absrel_error, values summed
    over the batch in batch order and count = number of batch elements."""
    from vidar_b200 import evaluation
    rng = np.random.default_rng(0)
    m = rng.uniform(0.1, 3.0, (3, 4, 4))
    m[..., 3] = 100
    ret = evaluation.ret_dict_from_metrics(m, start_idx=0)
    assert list(ret) == [f"frame.{i}" for i in range(4)]
    for f in range(4):
        e = ret[f"frame.{f}"]
        assert set(e) == {"count", "chamfer_distance", "l1_error", "absrel_error"}
        assert e["count"] == 3
        want_cd, want_l1, want_ar = 0, 0, 0
        for b in range(3):                      # the reference's accumulation: Python float / numpy float32
            want_cd += float(np.float32(m[b, f, 0]))
            want_l1 += np.float32(m[b, f, 1])
            want_ar += np.float32(m[b, f, 2])
        assert e["chamfer_distance"] == want_cd and e["l1_error"] == want_l1 and e["absrel_error"] == want_ar
        assert isinstance(e["chamfer_distance"], float) and isinstance(e["l1_error"], np.float32)
    assert list(evaluation.ret_dict_from_metrics(m, start_idx=2)) == [f"frame.{i}" for i in range(2, 6)]


@pytest.mark.parametrize("code", [-1.0, -2.0])
def test_ret_dict_raises_where_the_reference_raises(code):
    from vidar_b200 import evaluation
    m = np.ones((2, 3, 4))
    m[1, 2, 3] = code
    with pytest.raises(RuntimeError, match=r"segment \(1, 2\)"):
        evaluation.ret_dict_from_metrics(m)
