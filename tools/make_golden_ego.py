"""Golden vectors for ego motion from the REFERENCE's own code run on CPU here (tools/ref_shim.py):

  rotation / shift   PerceptionTransformer.get_bev_features (modules/transformer.py) with a stub encoder that
                     captures the rotated prev_bev and `shift`; 200 x 200 cells, C = 8, bs 2 with different angles.
                     The input cell value is its index + 1 on every channel, so the output is stored as the map
                     of source index + 1 (0 = zero fill).
  hybrid ref_2d      BEVFormerEncoder.forward (modules/encoder.py) with a stub layer that captures hybird_ref_2d.
  decoder alignment  ViDAR._get_history_ref_to_previous_transform / _align_bev_coordnates (detectors/vidar.py)
                     over a 6-frame roll-out with the queue update of forward_test.
  GT alignment       ViDARHeadV1._get_reference_gt_points (dense_heads/vidar_head_v1.py) for the 5 pred indices of
                     the loss and the src = tgt mapping of get_point_cloud_prediction.

Inputs are `vidar_b200.synthetic.ego_queue` queues.  Writes tests/golden/ego.npz."""
import ast
import functools
import os
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ref_shim  # noqa: E402
from vidar_b200 import synthetic  # noqa: E402

PC_RANGE = [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
ANGLES = [(0.0, 1e-3), (-1e-3, 37.3), (-90.0, 180.0), (-123.456, 71.0)]      # bs 2 per call; the last pair random
ALIGN_BEV = (20, 30)                                                           # non-square


def load_methods(relpath, cls, names, extra):
    """The named methods of class `cls` of a reference file, executed with the file's plain imports + `extra`."""
    path = os.path.join(ref_shim.REF_BEVFORMER, relpath)
    with open(path) as fh:
        tree = ast.parse(fh.read(), filename=path)
    ns = {"__name__": "vidar_ref._methods"}
    for node in tree.body:
        if isinstance(node, (ast.Import, ast.ImportFrom)) and not getattr(node, "level", 0):
            try:
                exec(compile(ast.Module([node], []), path, "exec"), ns)
            except ImportError:
                pass
    ns.update(extra)
    out = {}
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name == cls:
            for fn in node.body:
                if isinstance(fn, ast.FunctionDef) and fn.name in names:
                    fn.decorator_list = []
                    exec(compile(ast.Module([fn], []), path, "exec"), ns)
                    out[fn.name] = ns[fn.name]
    assert set(out) == set(names), (set(names) - set(out))
    return out


class _Capture(nn.Module):
    def __init__(self):
        super().__init__()
        self.kw = None

    def forward(self, *a, **kw):
        self.kw = kw
        return a[0] if a else None


def rotation_goldens(rec):
    from torchvision.transforms.functional import rotate
    get_bev_features = load_methods(os.path.join("modules", "transformer.py"), "PerceptionTransformer",
                                    ("get_bev_features",), dict(rotate=rotate))["get_bev_features"]
    H = W = 200
    C = 8
    for k, (a0, a1) in enumerate(ANGLES):
        q = synthetic.ego_queue(bs=2, T=2, future=1, seed=k)
        metas = [m[1] for m in q["img_metas"]]
        metas[0]["can_bus"][-1], metas[1]["can_bus"][-1] = a0, a1
        pt = nn.Module()
        pt.use_shift, pt.rotate_prev_bev, pt.use_can_bus, pt.use_cams_embeds = True, True, True, True
        pt.rotate_center = [100, 100]
        pt.can_bus_mlp = nn.Linear(18, C)
        pt.cams_embeds = nn.Parameter(torch.zeros(6, C))
        pt.level_embeds = nn.Parameter(torch.zeros(1, C))
        pt.encoder = _Capture()
        idx = torch.arange(1, H * W + 1, dtype=torch.float32)
        prev = idx[None, :, None].repeat(2, 1, C)                                    # [bs, HW, C]
        feats = [torch.zeros(2, 6, C, 2, 2)]
        with torch.no_grad():
            get_bev_features(pt, feats, torch.zeros(H * W, C), H, W, grid_length=(0.512, 0.512),
                                bev_pos=torch.zeros(2, C, H, W), prev_bev=prev, img_metas=metas)
        out = pt.encoder.kw["prev_bev"]                                              # [HW, bs, C]
        assert torch.equal(out, out[..., :1].expand_as(out))
        rec[f"rot{k}.angles"] = np.float64([a0, a1])
        rec[f"rot{k}.src_index"] = out[..., 0].t().numpy().astype(np.uint16)      # [bs, HW], 0 = fill
        rec[f"rot{k}.shift"] = pt.encoder.kw["shift"].numpy()
        rec[f"rot{k}.can_bus"] = np.stack([m_["can_bus"] for m_ in metas])
        rec[f"rot{k}.lidar2global_rotation"] = np.stack([m_["lidar2global_rotation"] for m_ in metas])
        print("rotation", k, a0, a1, "fill", (rec[f"rot{k}.src_index"] == 0).sum(1))


def hybrid_golden(rec):
    fns = load_methods(os.path.join("modules", "encoder.py"), "BEVFormerEncoder",
                       ("forward", "get_reference_points", "point_sampling"), {})
    H, W = 50, 50
    q = synthetic.ego_queue(bs=2, T=2, future=1, seed=7)
    metas = [m[1] for m in q["img_metas"]]
    e = nn.Module()
    e.get_reference_points = fns["get_reference_points"]                          # a staticmethod in the reference
    e.point_sampling = functools.partial(fns["point_sampling"], e)
    e.pc_range, e.num_points_in_pillar, e.return_intermediate = PC_RANGE, 4, False
    e.latent_rendering_lid = None
    e.layers = nn.ModuleList([_Capture()])
    shift = torch.tensor([[0.013, -0.021], [-0.002, 0.0071]])
    C = 8
    with torch.no_grad():
        fns["forward"](e, torch.zeros(H * W, 2, C), torch.zeros(6, 4, 2, C), torch.zeros(6, 4, 2, C), bev_h=H, bev_w=W,
                  bev_pos=torch.zeros(H * W, 2, C), spatial_shapes=torch.tensor([[2, 2]]),
                  level_start_index=torch.tensor([0]), prev_bev=torch.zeros(H * W, 2, C), shift=shift, img_metas=metas)
    rec["hybrid.shift"] = shift.numpy()
    rec["hybrid.ref_2d"] = e.layers[0].kw["ref_2d"].numpy()                      # [bs * 2, Q, 1, 2]
    print("hybrid", rec["hybrid.ref_2d"].shape)


def decoder_goldens(rec):
    ref_shim.install()
    fns = ref_shim.load_functions(os.path.join("utils", "e2e_predictor_utils.py"),
                                  ("get_bev_grids", "bev_grids_to_coordinates", "bev_coords_to_grids"))
    utils = type("U", (), {})()
    utils.get_bev_grids = functools.partial(fns["get_bev_grids"], device="cpu")
    utils.bev_grids_to_coordinates, utils.bev_coords_to_grids = fns["bev_grids_to_coordinates"], fns["bev_coords_to_grids"]
    m = load_methods(os.path.join("detectors", "vidar.py"), "ViDAR",
                     ("_get_history_ref_to_previous_transform", "_align_bev_coordnates"),
                     dict(e2e_predictor_utils=utils))
    H, W = ALIGN_BEV
    self = type("S", (), dict(bev_h=H, bev_w=W, point_cloud_range=PC_RANGE))()
    q = synthetic.ego_queue(bs=2, T=3, future=6, seed=11)
    T = 3
    for key in ("ref_lidar_to_cur_lidar", "future2ref_lidar_transform", "ref2future_lidar_transform"):
        rec[f"dec.{key}"] = np.stack([each[T - 1][key] for each in q["img_metas"]])
    prev = torch.zeros(2, 1, H * W, 4)
    img_metas = [each[T - 1] for each in q["img_metas"]]
    r2h = m["_get_history_ref_to_previous_transform"](self, prev, prev.shape[1], [[each[T - 1]] for each in q["img_metas"]])
    rec["dec.ref_to_history0"] = r2h.numpy()
    for k in range(1, 7):
        tgt, aligned, ref2future = m["_align_bev_coordnates"](self, k, r2h, img_metas)
        rec[f"dec.{k}.tgt"], rec[f"dec.{k}.aligned"] = tgt.numpy(), aligned.numpy()
        r2h = torch.cat([r2h, ref2future.unsqueeze(1)], 1)[:, 1:].contiguous()
    print("decoder alignment", rec["dec.1.aligned"].shape)


def gt_goldens(rec):
    m = load_methods(os.path.join("dense_heads", "vidar_head_v1.py"), "ViDARHeadV1", ("_get_reference_gt_points",), {})
    fn = m["_get_reference_gt_points"]
    T, future = 4, 4
    q = synthetic.ego_queue(bs=2, T=T, future=future, seed=5, points_per_frame=300)
    pts = [torch.from_numpy(p) for p in q["gt_points"]]
    pts[1] = pts[1][pts[1][:, 3] != 5]                                           # sample 1: frame 5 empty
    metas = [each[T - 1] for each in q["img_metas"]]
    for key in ("total_cur2ref_lidar_transform", "total_ref2cur_lidar_transform"):
        rec[f"gt.{key}"] = np.stack([m_[key] for m_ in metas])
    for b in range(2):
        rec[f"gt.points{b}"] = pts[b].numpy()
    hq, ph, valid = T - 1, T - 1, np.arange(4)
    cases = {f"loss{i}": (valid + hq - ph + i, valid + hq) for i in range(5)}
    cases["test"] = (np.arange(5) + hq, np.arange(5) + hq)
    for name, (src, tgt) in cases.items():
        out, origins = fn(None, pts, src, tgt, metas)
        rec[f"gt.{name}.src"], rec[f"gt.{name}.tgt"] = np.int64(src), np.int64(tgt)
        for b in range(2):
            rec[f"gt.{name}.out{b}"] = out[b].numpy()
        rec[f"gt.{name}.origins"] = origins.numpy()
        print("gt", name, [o.shape[0] for o in out])


def main():
    ref_shim.install()          # the mmcv / mmdet names the reference files import
    rec = {}
    rotation_goldens(rec)
    hybrid_golden(rec)
    decoder_goldens(rec)
    gt_goldens(rec)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "ego.npz"), **rec)


if __name__ == "__main__":
    main()
