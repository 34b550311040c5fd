"""Golden vectors for the evaluation metrics from the REFERENCE's own code run on CPU here:
utils/eval_utils.py (clamp, _clamp, spherical_projection, compute_ray_errors) loaded from the reference checkout,
and compute_chamfer_distance_inner / compute_chamfer_distance / get_inside_mask of utils/e2e_predictor_utils.py
via tools/ref_shim.load_functions.  chamferdist is the reference's chamfer.py on oracle/_ref/ref_knn_cpu.so, as in
tools/make_golden_knn.py.  Writes tests/golden/eval.npz."""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from oracle import build_ref  # noqa: E402
from tests.eval_cases import PC_RANGE, cases  # noqa: E402

import ref_shim  # noqa: E402

REF_CHAMFER = "/root/reference/third_lib/chamfer_dist/chamferdist/chamferdist"


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    build_ref.build_knn_cpu()
    pkg = types.ModuleType("chamferdist")
    pkg._C = build_ref.load("ref_knn_cpu")
    pkg.__path__ = []
    sys.modules["chamferdist"] = pkg
    ch = _load("chamferdist.chamfer", os.path.join(REF_CHAMFER, "chamfer.py"))
    pkg.ChamferDistance = ch.ChamferDistance
    ev = _load("ref_eval_utils", os.path.join(ref_shim.REF_BEVFORMER, "utils", "eval_utils.py"))
    fns = ref_shim.load_functions(os.path.join("utils", "e2e_predictor_utils.py"),
                                  ("get_inside_mask", "compute_chamfer_distance", "compute_chamfer_distance_inner"))
    fns["compute_chamfer_distance"].__globals__["chamfer_distance"] = ch.ChamferDistance()
    rec = {"pc_range": np.float32(PC_RANGE)}
    for name, (pred, gt, origin) in cases().items():
        rec[f"{name}.pred"], rec[f"{name}.gt"], rec[f"{name}.origin"] = pred, gt, origin
        # the nearest neighbour compute_ray_errors picks, with its own statements
        tp, pp, dp = ev.spherical_projection(pred - origin[None])
        tg, pg, dg = ev.spherical_projection(gt - origin[None])
        sp = np.stack([tp[dp > 1e-2], pp[dp > 1e-2], np.ones(int((dp > 1e-2).sum()), np.float32)], 1)
        sg = np.stack([tg[dg > 1e-2], pg[dg > 1e-2], np.ones(int((dg > 1e-2).sum()), np.float32)], 1)
        rec[f"{name}.count"] = np.int64(sg.shape[0])
        if sg.shape[0] and sp.shape[0]:
            _, (_, idx) = ch.ChamferDistance()(torch.from_numpy(sp[None]), torch.from_numpy(sg[None]), reverse=True,
                                               reduction="mean")
            rec[f"{name}.idx"] = idx[0].numpy().astype(np.int64)
        else:
            rec[f"{name}.idx"] = np.zeros(0, np.int64)
        cd = fns["compute_chamfer_distance_inner"](torch.from_numpy(pred), torch.from_numpy(gt), PC_RANGE)
        rec[f"{name}.chamfer"] = np.float64(cd.item() if torch.is_tensor(cd) else cd)
        try:
            with np.errstate(invalid="ignore", divide="ignore"):
                l1, absrel = ev.compute_ray_errors(pred.copy(), gt.copy(), origin.copy(), "cpu")
            rec[f"{name}.l1"], rec[f"{name}.absrel"] = np.float32(l1), np.float32(absrel)
            rec[f"{name}.raises"] = np.bool_(False)
        except RuntimeError as e:
            print(f"{name}: reference raises RuntimeError: {e}")
            rec[f"{name}.l1"], rec[f"{name}.absrel"] = np.float32(np.nan), np.float32(np.nan)
            rec[f"{name}.raises"] = np.bool_(True)
        print(name, rec[f"{name}.count"], rec[f"{name}.chamfer"], rec[f"{name}.l1"], rec[f"{name}.absrel"])
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "eval.npz"), **rec)


if __name__ == "__main__":
    main()
