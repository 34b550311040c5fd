"""The attention modules end to end on the GPU (CUDA MSDA op inside) against goldens produced
by the REFERENCE classes on CPU (tools/make_golden_modules.py).  1e-4 relative fp32."""
import os

import numpy as np
import pytest
import torch

from tests import module_cases as mc
import vidar_b200.modules  # noqa: F401  (registers the classes)
from vidar_b200.registry import build_attention

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "modules.npz")
GOLD_CUSTOM = os.path.join(os.path.dirname(__file__), "golden", "modules_custom.npz")


@pytest.mark.parametrize("kind,cfg,case,seed", [("sca", mc.SCA_CFG, mc.sca_case, 10),
                                                ("tsa", mc.TSA_CFG, mc.tsa_case, 11),
                                                ("pred", mc.PRED_CFG, mc.pred_case, 12)])
def test_module_on_gpu_matches_reference_class(cuda, kind, cfg, case, seed):
    g = np.load(GOLD)
    m = build_attention(cfg)
    m.load_state_dict(mc.seeded_state(m, seed))
    m.eval().to(cuda)
    out, gq, gkv = mc.run_module(m, kind, case(), device=cuda)
    np.testing.assert_allclose(out.cpu().numpy(), g[f"{kind}_out"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(gq.cpu().numpy(), g[f"{kind}_gq"], rtol=1e-4, atol=5e-5)
    np.testing.assert_allclose(gkv[:, ::6].cpu().numpy(), g[f"{kind}_gkv_s6"], rtol=1e-4, atol=5e-5)


@pytest.mark.parametrize("kind,boxes,seed", [("custom", False, 13), ("custom_boxes", True, 14)])
def test_detection_decoder_attention_on_gpu(cuda, kind, boxes, seed):
    g = np.load(GOLD_CUSTOM)
    m = build_attention(mc.CUSTOM_CFG)
    m.load_state_dict(mc.seeded_state(m, seed))
    m.eval().to(cuda)
    out, gq, gkv = mc.run_module(m, kind, mc.custom_case(boxes=boxes), device=cuda)
    np.testing.assert_allclose(out.cpu().numpy(), g[f"{kind}_out"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(gq.cpu().numpy(), g[f"{kind}_gq"], rtol=1e-4, atol=5e-5)
    np.testing.assert_allclose(gkv.cpu().numpy(), g[f"{kind}_gkv"], rtol=1e-4, atol=5e-5)


def test_sca_fused_epilogue_equals_materialised_path(cuda):
    """SpatialCrossAttention through MSDeformableAttention3D with the softmax / sampling-location
    arithmetic inside the kernel (default) vs materialised `sampling_locations` / `attention_weights`."""
    m = build_attention(mc.SCA_CFG)
    m.load_state_dict(mc.seeded_state(m, 10))
    m.eval().to(cuda)
    assert m.deformable_attention.fuse_epilogue
    m.fuse_rebatch = False            # the reference's rebatch data flow: MSDeformableAttention3D is called as a module
    res = []
    for fused in (True, False):
        m.deformable_attention.fuse_epilogue = fused
        m.zero_grad(set_to_none=True)
        out, gq, gkv = mc.run_module(m, "sca", mc.sca_case(), device=cuda)
        res.append((out, gq, gkv, m.deformable_attention.sampling_offsets.weight.grad.clone(),
                    m.deformable_attention.attention_weights.weight.grad.clone()))
    for a, b, w in zip(res[0], res[1], ("out", "grad query", "grad key/value", "grad sampling_offsets.weight",
                                        "grad attention_weights.weight")):
        err = (a - b).abs().max().item()
        assert err <= 2e-5 * b.abs().max().item() + 1e-7, f"{w}: {err:.3e} vs {b.abs().max().item():.3e}"


@pytest.mark.parametrize("bs", [1, 2])
def test_sca_fused_rebatch_equals_reference_data_flow(cuda, bs):
    """SpatialCrossAttention's default path (device-side visible lists, offsets / logits once per pillar,
    rows reduced straight into the BEV slots: vidar_b200/sca.py) against the reference's rebatch /
    index_add_ data flow on the same CUDA op -- output, input gradients and every parameter gradient.

    The two flows compute the sampling offsets with different GEMMs (once per pillar on the tensor cores, once per
    (camera, pillar) row on cuBLAS).  Rounded differently, a sample within an ulp of a pixel-centre line lands on
    either side of it, where d(out)/d(loc) jumps, and through `sampling_offsets` that one sample moves a whole row of
    the query gradient.  So the query and that Linear's parameters are put on dyadic grids (query to 2^-6, weights to
    2^-8), where both GEMMs are exact in fp32: both flows then sample at bit-identical locations."""
    m = build_attention(mc.SCA_CFG)
    sd = mc.seeded_state(m, 10)
    for k in ("deformable_attention.sampling_offsets.weight", "deformable_attention.sampling_offsets.bias"):
        sd[k] = (sd[k] * 256).round() / 256
    m.load_state_dict(sd)
    m.eval().to(cuda)
    assert m.fuse_rebatch
    case = mc.sca_case(bs=bs)
    for k in ("query", "query_pos"):
        case[k] = (case[k] * 64).round() / 64
    res = []
    for fused in (True, False):
        m.fuse_rebatch = fused
        m.zero_grad(set_to_none=True)
        out, gq, gkv = mc.run_module(m, "sca", case, device=cuda)
        res.append([out, gq, gkv] + [p.grad.clone() for _, p in sorted(m.named_parameters())])
    names = ["out", "grad query", "grad key/value"] + [n for n, _ in sorted(m.named_parameters())]
    for a, b, w in zip(res[0], res[1], names):
        err = (a - b).abs().max().item()
        assert err <= 2e-5 * b.abs().max().item() + 1e-7, f"{w}: {err:.3e} vs {b.abs().max().item():.3e}"


def test_sca_default_path_has_no_host_sync(cuda):
    """Forward + backward of the default SpatialCrossAttention path never synchronises with the host
    (the reference syncs on `nonzero()` / max_len in every layer)."""
    m = build_attention(mc.SCA_CFG)
    m.load_state_dict(mc.seeded_state(m, 10))
    m.eval().to(cuda)
    c = {k: (v.to(cuda) if torch.is_tensor(v) else v) for k, v in mc.sca_case().items()}
    q = c["query"].clone().requires_grad_(True)
    kv = c["key"].clone().requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = m(q, kv, kv, query_pos=c["query_pos"], reference_points_cam=c["reference_points_cam"],
                bev_mask=c["bev_mask"], spatial_shapes=c["spatial_shapes"], level_start_index=c["level_start_index"])
        out.backward(c["grad"])
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.isfinite(out).all() and torch.isfinite(q.grad).all()


def test_compact_visible_lists_on_device(cuda):
    from vidar_b200 import sca
    g = torch.Generator().manual_seed(4)
    cams, bs, Q, D = 6, 2, 5000, 4                     # > 1024 pillars: several chunks of the block scan
    mask = torch.rand(cams, bs, Q, D, generator=g) < 0.12
    mask[2] = False
    mask[4] = True
    idx, count, inv = sca.compact_visible(mask.to(cuda))
    hit = mask[:, 0].any(-1)
    for c in range(cams):
        want = hit[c].nonzero().squeeze(-1)
        assert int(count[c]) == want.numel()
        assert torch.equal(idx[c, : want.numel()].cpu().long(), want)
    cnt = mask.any(-1).permute(1, 2, 0).sum(-1).clamp(min=1).float()
    assert torch.equal(inv.cpu(), 1.0 / cnt)
