"""BASELINE.json configs[3]: one ViDAR-RN101 pre-training step on synthetic data, built around the
hot-path modules of this package, with the intra-sample sharding of SURVEY.md 8e.

This is a HARNESS, not a port of the detector: it composes the reference's step
(projects/mmdet3d_plugin/bevformer/detectors/vidar.py:239-387) from
  * a random-init torchvision ResNet-101 (strides 8/16/32; stage 1 frozen, BN in eval mode as in
    vidar_1_8_nusc_3future.py:88-95 -- the reference's DCN in stages 3-4 is out of scope, plain convs) and
    a 4-level FPN (cfg :96-106);
  * the BEV encoder: 6 x [TemporalSelfAttention, LN, SpatialCrossAttention, LN, (LatentRendering in
    layer 2), FFN 256-512-256, LN]  (modules/encoder.py:159-253, encoder_v2.py:52-209, cfg :141-190);
  * the future decoder: 3 x [PredictionMSDeformableAttention (self), LN, PredictionMSDeformableAttention
    (cross to the previous BEV), LN, FFN, LN], rolled out for 3 future frames
    (modules/vidar_decoder.py:25-280, dense_heads/vidar_head_base.py:125-173);
  * the per-layer freespace head and the ray losses of ViDARHeadV1 (dense_heads/vidar_head_v1.py:45-92,
    150-219) through `vidar_b200.head.ViDARRayHead.loss`.
History frames run under no_grad like `obtain_history_bev` (bevformer.py:158-189).

Sharding over a process group (one sample on all ranks -- the reference has replica DDP only):
  * cameras: each camera's image goes through backbone + FPN on ONE rank; a camera whose
    SpatialCrossAttention units are split over two ranks (vidar_b200.sca.unit_plan) has its features
    broadcast inside its 2-rank group (31.6 MB), gradients reduced back to the owner;
  * SpatialCrossAttention: camera-sharded sampling, reduce-scatter of the partial BEV slots, output_proj on
    the rank's rows, ONE all-gather of the BEV grid per layer (modules/deform_attn.py);
  * LatentRendering: BEV rows / cells sharded (modules/latent_rendering.py);
  * everything else (TSA, FFN, norms, decoder, head, loss) is replicated: every rank computes the same
    values and the same gradients, so only parameters that saw sharded data (backbone, FPN, embeddings of
    the camera features, SCA projections) need their gradients summed -- ONE bucketed all-reduce per step
    (`sharding.allreduce_partial_grads`), the counterpart of the reference's DDP all-reduce
    (apis/mmdet_train.py:72-81).
"""
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import bev_geometry, sca, sharding, synthetic
from . import modules as _modules  # noqa: F401  (registers the attention classes)
from .head import ViDARRayHead
from .modules.deform_attn import _linear
from .registry import build_attention

PC_RANGE = [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
EMBED, BEV_H, BEV_W, HEIGHTS = 256, 200, 200, 16


# ------------------------------------------------------------------------------------------------
# image side
# ------------------------------------------------------------------------------------------------
class ImageBackbone(nn.Module):
    """ResNet-101 C3..C5 (strides 8, 16, 32).  frozen_stages=1 and norm_eval=True (cfg :92-94)."""

    def __init__(self):
        super().__init__()
        import torchvision
        r = torchvision.models.resnet101(weights=None)
        self.stem = nn.Sequential(r.conv1, r.bn1, r.relu, r.maxpool)
        self.layer1, self.layer2, self.layer3, self.layer4 = r.layer1, r.layer2, r.layer3, r.layer4
        for m in (self.stem, self.layer1):
            for p in m.parameters():
                p.requires_grad_(False)

    def train(self, mode=True):
        super().train(mode)
        for m in self.modules():                      # norm_eval
            if isinstance(m, nn.BatchNorm2d):
                m.eval()
        return self

    def forward(self, x):
        with torch.no_grad():
            x = self.layer1(self.stem(x))
        c3 = self.layer2(x)
        c4 = self.layer3(c3)
        c5 = self.layer4(c4)
        return c3, c4, c5


class FPN(nn.Module):
    """mmdet FPN(in=[512,1024,2048], out=256, start_level=0, add_extra_convs='on_output', num_outs=4,
    relu_before_extra_convs=True)  (cfg :96-106)."""

    def __init__(self, in_channels=(512, 1024, 2048), out_channels=EMBED):
        super().__init__()
        self.lateral = nn.ModuleList([nn.Conv2d(c, out_channels, 1) for c in in_channels])
        self.out = nn.ModuleList([nn.Conv2d(out_channels, out_channels, 3, padding=1) for _ in in_channels])
        self.extra = nn.Conv2d(out_channels, out_channels, 3, stride=2, padding=1)

    def forward(self, feats):
        lat = [l(f) for l, f in zip(self.lateral, feats)]
        for i in range(len(lat) - 1, 0, -1):
            lat[i - 1] = lat[i - 1] + F.interpolate(lat[i], size=lat[i - 1].shape[-2:], mode="nearest")
        outs = [o(x) for o, x in zip(self.out, lat)]
        outs.append(self.extra(F.relu(outs[-1])))
        return outs


class _ShareCameraFeatures(torch.autograd.Function):
    """Features of a camera whose SCA units are split over two ranks: broadcast from the rank that ran the
    backbone; the co-owner's gradient is reduced back (all-reduce inside the 2-rank group)."""

    @staticmethod
    def forward(ctx, feat, src, group):
        import torch.distributed as dist
        ctx.group = group
        out = feat.contiguous().clone()
        dist.broadcast(out, src=src, group=group)
        return out

    @staticmethod
    def backward(ctx, g):
        import torch.distributed as dist
        g = g.contiguous().clone()
        dist.all_reduce(g, group=ctx.group)
        return g, None, None


# ------------------------------------------------------------------------------------------------
# BEV side
# ------------------------------------------------------------------------------------------------
class FFN(nn.Module):
    """mmcv FFN(embed 256, feedforward 512, 2 fcs, ReLU, dropout 0.1, residual)  (cfg :163-170)."""

    def __init__(self, dims=EMBED, hidden=2 * EMBED, drop=0.1):
        super().__init__()
        self.fc1, self.fc2 = nn.Linear(dims, hidden), nn.Linear(hidden, dims)
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        return x + self.drop(_linear(self.fc2, self.drop(F.relu(_linear(self.fc1, x)))))


class LearnedPositionalEncoding(nn.Module):
    def __init__(self, rows, cols, num_feats=EMBED // 2):
        super().__init__()
        self.row_embed, self.col_embed = nn.Embedding(rows, num_feats), nn.Embedding(cols, num_feats)

    def forward(self, bs):
        h, w = self.row_embed.num_embeddings, self.col_embed.num_embeddings
        x = self.col_embed.weight[None].expand(h, -1, -1)
        y = self.row_embed.weight[:, None].expand(-1, w, -1)
        return torch.cat([x, y], -1).view(1, h * w, -1).expand(bs, -1, -1)      # [bs, Q, C]


class EncoderLayer(nn.Module):
    """BEVFormerLayerV2 (encoder_v2.py:52-209): self_attn, norm, cross_attn, norm, [latent_render], ffn, norm."""

    def __init__(self, latent_render, bev_hw):
        super().__init__()
        self.bev_hw = bev_hw
        self.self_attn = build_attention(dict(type="TemporalSelfAttention", embed_dims=EMBED, num_levels=1))
        self.cross_attn = build_attention(dict(
            type="SpatialCrossAttention", pc_range=PC_RANGE, embed_dims=EMBED,
            deformable_attention=dict(type="MSDeformableAttention3D", embed_dims=EMBED, num_points=8, num_levels=4)))
        self.norms = nn.ModuleList([nn.LayerNorm(EMBED) for _ in range(3)])
        self.ffn = FFN()
        self.latent_render = build_attention(dict(
            type="LatentRendering", embed_dims=EMBED, num_pred_fcs=0, pred_height=HEIGHTS, grid_num=256, grid_step=0.5,
            reduction=16, act="sigmoid")) if latent_render else None

    def forward(self, query, feats, bev_pos, ref_2d, prev_bev, shapes, lsi, ref_cam, bev_mask, bev_shapes, bev_lsi):
        query = self.self_attn(query, prev_bev, prev_bev, None, query_pos=bev_pos, reference_points=ref_2d,
                               spatial_shapes=bev_shapes, level_start_index=bev_lsi)
        query = self.norms[0](query)
        query = self.cross_attn(query, feats, feats, None, reference_points_cam=ref_cam, bev_mask=bev_mask,
                                spatial_shapes=shapes, level_start_index=lsi)
        query = self.norms[1](query)
        if self.latent_render is not None:
            bs, n, c = query.shape
            query = self.latent_render(query.view(bs, self.bev_hw[0], self.bev_hw[1], c)).view(bs, n, c)
        return self.norms[2](self.ffn(query))

    def forward_rows(self, x_full, feats, bev_pos, ref_2d, prev_bev, shapes, lsi, ref_cam, bev_mask, bev_shapes, bev_lsi,
                     group, last):
        """The same layer with the BEV rows sharded over `group` (SURVEY.md 8e: TSA / FFN / norms on the rank's rows,
        value replicated; bs = 1).  `x_full` [1, Q, C] is the replicated layer input; every row-wise stage runs on
        this rank's block only; the full grid is assembled twice: after the first norm (SpatialCrossAttention needs
        every pillar's offsets for its cameras) and at the end (the next layer's TSA samples the whole BEV).  Both
        all-gathers feed sharded consumers, so their backward is a reduce-scatter of partial gradients -- except the
        last layer's, whose consumers (decoder, head) are replicated."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        bs, Q, C = x_full.shape
        lo, hi = sharding.row_range(Q, rank, world)
        q = self.self_attn(x_full[:, lo:hi], prev_bev, prev_bev, None, query_pos=bev_pos[:, lo:hi],
                           reference_points=ref_2d[:, lo:hi], spatial_shapes=bev_shapes, level_start_index=bev_lsi,
                           row_range=(lo, hi))
        q = self.norms[0](q)                                                       # [1, rows, C]
        q_full = sharding.all_gather_rows(q[0], Q, group, grad="sum")[None]
        q = self.cross_attn(q_full, feats, feats, q, reference_points_cam=ref_cam, bev_mask=bev_mask,
                            spatial_shapes=shapes, level_start_index=lsi, rows_out=True, summed_query_grad=True)
        q = self.norms[1](q)                                                       # [rows, C]
        if self.latent_render is not None:
            q = self.latent_render.forward_rows(q, bs, self.bev_hw[0], self.bev_hw[1])
        q = self.norms[2](self.ffn(q))
        return sharding.all_gather_rows(q, Q, group, grad="slice" if last else "sum")[None]


class DecoderLayer(nn.Module):
    """PredictionTransformerLayer (vidar_decoder.py:104-280) without latent rendering (the shipped
    pre-train configs delete it from every decoder layer, SURVEY.md 3.3)."""

    def __init__(self):
        super().__init__()
        self.self_attn = build_attention(dict(type="PredictionMSDeformableAttention", embed_dims=EMBED, num_levels=1))
        self.cross_attn = build_attention(dict(type="PredictionMSDeformableAttention", embed_dims=EMBED, num_levels=1))
        self.norms = nn.ModuleList([nn.LayerNorm(EMBED) for _ in range(3)])
        self.ffn = FFN()

    def forward(self, query, prev_feats, bev_pos, tgt_points, ref_points, bev_shapes, bev_lsi):
        query = self.self_attn(query, None, None, None, query_pos=bev_pos, reference_points=tgt_points,
                               spatial_shapes=bev_shapes, level_start_index=bev_lsi)
        query = self.norms[0](query)
        query = self.cross_attn(query, prev_feats, prev_feats, None, query_pos=bev_pos, reference_points=ref_points,
                                spatial_shapes=bev_shapes, level_start_index=bev_lsi)
        query = self.norms[1](query)
        return self.norms[2](self.ffn(query))

    def forward_rows(self, x_full, prev_feats, bev_pos, tgt_points, ref_points, bev_shapes, bev_lsi, group):
        """The same layer on this rank's block of BEV rows (bs = 1): both attentions sample replicated values (the full
        query grid / the previous BEV) for the rank's rows, norms and FFN are row-wise, ONE all-gather returns the grid
        (backward: reduce-scatter -- `prev_feats` and `bev_pos` must come through `sharding.sum_grad`, replicated
        consumers of the result through `sharding.replicated_view`)."""
        import torch.distributed as dist
        Q = x_full.shape[1]
        lo, hi = sharding.row_range(Q, dist.get_rank(group), dist.get_world_size(group))
        pos = bev_pos[:, lo:hi]
        q = self.self_attn(x_full[:, lo:hi], None, x_full, None, query_pos=pos, reference_points=tgt_points[:, lo:hi],
                           spatial_shapes=bev_shapes, level_start_index=bev_lsi)
        q = self.norms[0](q)
        q = self.cross_attn(q, prev_feats, prev_feats, None, query_pos=pos, reference_points=ref_points[:, lo:hi],
                            spatial_shapes=bev_shapes, level_start_index=bev_lsi)
        q = self.norms[2](self.ffn(self.norms[1](q)))
        return sharding.all_gather_rows(q[0], Q, group, grad="sum")[None]


def run_decoder(layers, query, prev, bev_pos, ref, bev_shapes, bev_lsi, group=None):
    """The future-BEV decoder stack -> (outputs of every layer stacked [inter, bs, Q, C] for the head, last output for
    the next future frame).  `group`: row-sharded layers (`DecoderLayer.forward_rows`); the stacked outputs are then
    (like the returned last output) views for replicated consumers (`sharding.replicated_view`)."""
    inter = []
    if group is None:
        for layer in layers:
            query = layer(query, prev, bev_pos, ref, ref, bev_shapes, bev_lsi)
            inter.append(query)
        return torch.stack(inter), inter[-1]
    query, prev, bev_pos = (sharding.sum_grad(t, group) for t in (query, prev, bev_pos))
    for layer in layers:
        query = layer.forward_rows(query, prev, bev_pos, ref, ref, bev_shapes, bev_lsi, group)
        inter.append(sharding.replicated_view(query, group))
    # the caller's use of the last output (next frame's `prev`, which passes through sum_grad again) is replicated too
    return torch.stack(inter), inter[-1]


class SyntheticViDAR(nn.Module):
    """The pre-training graph of ViDAR-RN101 (3 history frames, 3 future frames, 5 predicted head frames)."""

    def __init__(self, num_cams=6, encoder_layers=6, decoder_layers=3, future_frames=3, history_frames=3,
                 latent_layer=2, bev_hw=(BEV_H, BEV_W), ray_grid_num=512, test_future_frames=6):
        super().__init__()
        self.num_cams, self.future_frames, self.history_frames = num_cams, future_frames, history_frames
        self.test_future_frames = test_future_frames           # roll-outs of forward_test (cfg :18)
        self.bev_h, self.bev_w = bev_hw
        BEV_H, BEV_W = bev_hw          # noqa: N806  (shadows the module defaults below)
        self.backbone, self.neck = ImageBackbone(), FPN()
        self.bev_embedding = nn.Embedding(BEV_H * BEV_W, EMBED)
        self.positional_encoding = LearnedPositionalEncoding(BEV_H, BEV_W)
        self.cams_embeds = nn.Parameter(torch.randn(num_cams, EMBED) * 0.02)
        self.level_embeds = nn.Parameter(torch.randn(4, EMBED) * 0.02)
        self.can_bus_mlp = nn.Sequential(nn.Linear(18, EMBED // 2), nn.ReLU(inplace=True), nn.Linear(EMBED // 2, EMBED),
                                         nn.ReLU(inplace=True), nn.LayerNorm(EMBED))
        self.encoder = nn.ModuleList([EncoderLayer(i == latent_layer, bev_hw) for i in range(encoder_layers)])
        # future head (ViDARHeadV1)
        self.future_bev_embedding = nn.Embedding(BEV_H * BEV_W, EMBED)
        self.future_positional_encoding = LearnedPositionalEncoding(BEV_H, BEV_W)
        self.prev_frame_embedding = nn.Parameter(torch.randn(1, EMBED))
        self.future_can_bus_mlp = nn.Sequential(nn.Linear(18, EMBED // 2), nn.ReLU(inplace=True),
                                                nn.Linear(EMBED // 2, EMBED), nn.ReLU(inplace=True), nn.LayerNorm(EMBED))
        self.decoder = nn.ModuleList([DecoderLayer() for _ in range(decoder_layers)])
        self.pred_frame_num = 1 + history_frames + 1                 # 3 history + current + 1 future per BEV feature (cfg :31-33)
        self.bev_pred_head = nn.ModuleList([nn.Linear(EMBED, self.pred_frame_num * HEIGHTS) for _ in range(decoder_layers)])
        self.ray_head = ViDARRayHead(ray_grid_num=ray_grid_num, ray_grid_step=1.0, use_ce_loss=True, use_dist_loss=False,
                                     use_dense_loss=True, loss_weight=[[1.0]] * (1 + future_frames))
        self.per_frame_loss_weight = (0.1, 0.1, 0.1, 1.0, 1.0)
        self.process_group = None
        self.row_sharded = False
        self.timings = None

    # ---- sharding ------------------------------------------------------------------------------
    def set_process_group(self, group, row_sharded=False):
        """Shard one sample over `group`: cameras (backbone, SpatialCrossAttention), cells (LatentRendering).
        `row_sharded=True` additionally runs every row-wise stage of the encoder (TSA, norms, FFN) on the rank's
        block of BEV rows (`EncoderLayer.forward_rows`; bs = 1, rows divisible by the group size)."""
        import torch.distributed as dist
        self.process_group = group
        self.row_sharded = bool(row_sharded) and group is not None and dist.get_world_size(group) > 1
        world = dist.get_world_size(group) if group is not None else 1
        rank = dist.get_rank(group) if group is not None else 0
        self.plan = sca.unit_plan(world, rank, self.num_cams)
        owners = sca.camera_ranks(world, self.num_cams)
        self.cam_owner = {c: r[0] for c, r in owners.items()}
        self.my_backbone_cams = [c for c, o in self.cam_owner.items() if o == rank]
        self.my_sca_cams = sca.plan_cameras(self.plan)
        self.cam_groups = sca.camera_groups(world, self.num_cams, rank) if world > 1 else {}
        for layer in self.encoder:
            layer.cross_attn.set_process_group(group if world > 1 else None)
            if layer.latent_render is not None:
                layer.latent_render.process_group = group if world > 1 else None
        if world > 1:      # parameters that only see this rank's cameras
            for m in (self.backbone, self.neck):
                sharding.mark_partial(m)
            self.cams_embeds.vidar_partial_grad = True
            self.level_embeds.vidar_partial_grad = True
        for layer in self.encoder:      # row-wise stages see only this rank's rows: partial parameter gradients
            for m in (layer.self_attn, layer.norms, layer.ffn):
                for p_ in m.parameters():
                    p_.vidar_partial_grad = self.row_sharded
        for p_ in self.decoder.parameters():
            p_.vidar_partial_grad = self.row_sharded
        return self

    def _mark(self, name):
        if self.timings is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.timings.append((name, e))

    # ---- image features of one frame -> [cams, K, bs, C] (only this rank's SCA cameras are filled) ----
    def extract_feat(self, img):
        """img [bs, cams, 3, H, W] -> (feat_flatten [cams, K, bs, C], spatial_shapes, level_start_index)."""
        import torch.distributed as dist
        bs = img.shape[0]
        world = dist.get_world_size(self.process_group) if self.process_group is not None else 1
        rank = dist.get_rank(self.process_group) if world > 1 else 0
        mine = self.my_backbone_cams if world > 1 else list(range(self.num_cams))
        per_cam = {}
        if mine:
            x = img[:, mine].reshape(bs * len(mine), *img.shape[2:])
            outs = self.neck(self.backbone(x))
            for i, c in enumerate(mine):
                lv = []
                for lvl, f in enumerate(outs):
                    f = f.view(bs, len(mine), *f.shape[1:])[:, i]                       # [bs, C, h, w]
                    f = f.flatten(2).permute(2, 0, 1)                                    # [hw, bs, C]
                    lv.append(f + self.cams_embeds[c][None, None] + self.level_embeds[lvl][None, None])   # transformer.py:166-172
                per_cam[c] = torch.cat(lv, 0)                                            # [K, bs, C]
            shapes = [tuple(f.shape[-2:]) for f in outs]
        else:
            h, w = img.shape[-2:]
            shapes = [(math.ceil(h / s), math.ceil(w / s)) for s in (8, 16, 32, 64)]
        K = sum(h * w for h, w in shapes)
        feats = img.new_zeros((self.num_cams, K, bs, EMBED))
        pieces = []
        for c in range(self.num_cams):
            f = per_cam.get(c)
            if c in self.cam_groups:                                                      # shared camera
                if f is None:
                    f = img.new_zeros((K, bs, EMBED)).requires_grad_(torch.is_grad_enabled())
                f = _ShareCameraFeatures.apply(f, self.cam_owner[c], self.cam_groups[c])
            pieces.append(f if (f is not None and (world == 1 or c in self.my_sca_cams)) else feats[c])
        feats = torch.stack(pieces, 0)
        spatial_shapes = torch.tensor(shapes, dtype=torch.int64, device=img.device)
        lsi = torch.cat([spatial_shapes.new_zeros(1), (spatial_shapes[:, 0] * spatial_shapes[:, 1]).cumsum(0)[:-1]])
        return feats, spatial_shapes, lsi

    # ---- BEV encoder (transformer.py:102-193 + encoder.py:159-253) ----
    def encode(self, feats, spatial_shapes, lsi, img_metas, can_bus, prev_bev):
        bs = feats.shape[2]
        dev = feats.device
        BEV_H, BEV_W = self.bev_h, self.bev_w          # noqa: N806
        bev_pos = self.positional_encoding(bs)
        query = self.bev_embedding.weight[None].expand(bs, -1, -1) + self.can_bus_mlp(can_bus)[:, None]
        ref_3d = bev_geometry.get_reference_points(BEV_H, BEV_W, PC_RANGE[5] - PC_RANGE[2], 4, dim="3d", bs=bs, device=dev)
        ref_2d = bev_geometry.get_reference_points(BEV_H, BEV_W, dim="2d", bs=bs, device=dev)
        ref_cam, bev_mask = bev_geometry.point_sampling(ref_3d, PC_RANGE, img_metas)
        Q = BEV_H * BEV_W
        hybrid = torch.stack([ref_2d, ref_2d], 1).reshape(bs * 2, Q, 1, 2)          # can_bus zeros: no ego shift
        bev_shapes = torch.tensor([[BEV_H, BEV_W]], device=dev)
        bev_lsi = torch.tensor([0], device=dev)
        rows_mode = getattr(self, "row_sharded", False)
        if rows_mode:
            import torch.distributed as dist
            world = dist.get_world_size(self.process_group)
            if bs != 1 or Q % world != 0:
                raise RuntimeError(f"row-sharded encoder: needs bs == 1 and BEV rows ({Q}) divisible by the group size ({world})")
            # replicated tensors consumed by sharded stages: their gradients are per-rank partial sums
            query = sharding.sum_grad(query, self.process_group)
            bev_pos = sharding.sum_grad(bev_pos, self.process_group)
        for i, layer in enumerate(self.encoder):
            pv = torch.stack([prev_bev if prev_bev is not None else query, query], 1).reshape(bs * 2, Q, EMBED)
            if rows_mode:
                query = layer.forward_rows(query, feats, bev_pos, hybrid, pv, spatial_shapes, lsi, ref_cam, bev_mask,
                                           bev_shapes, bev_lsi, self.process_group, last=i == len(self.encoder) - 1)
            else:
                query = layer(query, feats, bev_pos, hybrid, pv, spatial_shapes, lsi, ref_cam, bev_mask, bev_shapes, bev_lsi)
        return query

    # ---- future decoder (vidar_head_base.py:125-173) ----
    def decode_future(self, prev_bev_input, future_can_bus):
        bs = prev_bev_input.shape[0]
        dev = prev_bev_input.device
        BEV_H, BEV_W = self.bev_h, self.bev_w          # noqa: N806
        bev_pos = self.future_positional_encoding(bs)
        query = self.future_bev_embedding.weight[None] + self.future_can_bus_mlp(future_can_bus)[:, None]
        prev = (prev_bev_input + self.prev_frame_embedding[None, :, None, :]).view(bs, -1, EMBED)
        ref = bev_geometry.get_reference_points(BEV_H, BEV_W, dim="2d", bs=bs, device=dev)      # identity ego motion
        bev_shapes = torch.tensor([[BEV_H, BEV_W]], device=dev)
        bev_lsi = torch.tensor([0], device=dev)
        rows_mode = getattr(self, "row_sharded", False)
        if rows_mode and (bs != 1 or query.shape[1] % torch.distributed.get_world_size(self.process_group) != 0):
            raise RuntimeError("row-sharded decoder: needs bs == 1 and BEV rows divisible by the group size")
        # -> ([inter, bs, Q, C] for the head, the last layer's output for the next future frame)
        return run_decoder(self.decoder, query, prev, bev_pos, ref, bev_shapes, bev_lsi, self.process_group if rows_mode else None)

    def forward_head(self, next_bev_feats):
        """vidar_head_v1.py:64-92: [frames, inter, bs, Q, C] -> [frames, inter, pred_frame, bs, Q, heights]."""
        hist = self.history_frames
        preds = []
        for lvl in range(next_bev_feats.shape[1]):
            p = self.bev_pred_head[lvl](next_bev_feats[:, lvl])
            p = p.view(*p.shape[:-1], HEIGHTS, self.pred_frame_num)
            base = p[..., hist][..., None]
            p = torch.cat([p[..., :hist] + base, base, p[..., hist + 1:] + base], -1)
            preds.append(p.permute(0, 4, 1, 2, 3).contiguous())
        return torch.stack(preds, 1)

    # ---- one training forward (vidar.py:239-387) -> dict of losses ----
    def forward_train(self, img, lidar2img, gt_points, can_bus=None):
        """img [bs, T, cams, 3, H, W] (T-1 history frames + current), lidar2img: host array [bs, cams, 4, 4]
        (it lives in `img_metas` in the reference), gt_points: list over batch of [M, 4] (x, y, z metric,
        frame index 0 = current .. future_frames)."""
        bs, T = img.shape[:2]
        dev = img.device
        can_bus = torch.zeros(bs, 18, device=dev) if can_bus is None else can_bus
        img_metas = [dict(lidar2img=np.asarray(lidar2img[b]), img_shape=[(img.shape[-2], img.shape[-1], 3)]) for b in range(bs)]
        prev_bev = None
        with torch.no_grad():                                                        # obtain_history_bev
            for t in range(T - 1):
                feats, shapes, lsi = self.extract_feat(img[:, t])
                self._mark(f"hist{t}.backbone")
                prev_bev = self.encode(feats, shapes, lsi, img_metas, can_bus, prev_bev)
                self._mark(f"hist{t}.encoder")
        feats, shapes, lsi = self.extract_feat(img[:, T - 1])
        self._mark("cur.backbone")
        ref_bev = self.encode(feats, shapes, lsi, img_metas, can_bus, prev_bev)
        self._mark("cur.encoder")
        inter_num = len(self.bev_pred_head)
        next_bev_feats = [ref_bev.unsqueeze(0).repeat(inter_num, 1, 1, 1)]
        prev_bev_input = ref_bev.unsqueeze(1)
        for _ in range(self.future_frames):
            pred_feat, last = self.decode_future(prev_bev_input, can_bus)
            next_bev_feats.append(pred_feat)
            prev_bev_input = last.unsqueeze(1)                                         # queue length 1 (vidar.py:359-360)
        self._mark("future_decoder")
        next_bev_feats = torch.stack(next_bev_feats, 0)
        next_bev_preds = self.forward_head(next_bev_feats)                              # [F, inter, pred_frame, bs, Q, 16]
        valid_frames = list(range(1 + self.future_frames))
        losses = {}
        for i in range(self.pred_frame_num):                                            # vidar_head_v1.py:179-218
            pred_dict = dict(next_bev_preds=next_bev_preds[:, :, i], valid_frames=valid_frames)
            lw = np.array([[self.per_frame_loss_weight[i]]] * len(valid_frames))
            ld = self.ray_head.loss(pred_dict, gt_points, 0, self.bev_h, self.bev_w, PC_RANGE, pred_frame_num=1 + self.future_frames,
                                    loss_weight=lw)
            for k, v in ld.items():
                losses[f"frame.{i}.{k}"] = v
        self._mark("head+loss")
        return losses

    # ---- one test forward (vidar.py:389-502) -> [ret_dict] of point-cloud forecasting metrics ----
    def forward_test(self, img, lidar2img, gt_points, can_bus=None):
        """img [bs, T, cams, 3, H, W], lidar2img [bs, cams, 4, 4] (host), gt_points: list over batch of [M, 4]
        (x, y, z metric, frame index 0 = current .. test_future_frames).  Every frame is encoded (obtain_history_bev
        in test mode, bevformer.py:217-232), the decoder rolls out `test_future_frames` times with a queue of length 1,
        the head keeps prediction index `history_frames` (vidar_head_v1.py:234) and `ViDARRayHead.evaluate` scores
        every (sample, frame).  Synthetic ego motion is the identity.  -> [ret_dict]."""
        was_training = self.training
        self.eval()
        try:
            with torch.no_grad():
                bs, T = img.shape[:2]
                can_bus = torch.zeros(bs, 18, device=img.device) if can_bus is None else can_bus
                img_metas = [dict(lidar2img=np.asarray(lidar2img[b]), img_shape=[(img.shape[-2], img.shape[-1], 3)])
                             for b in range(bs)]
                prev_bev = None
                for t in range(T):
                    feats, shapes, lsi = self.extract_feat(img[:, t])
                    self._mark(f"frame{t}.backbone")
                    prev_bev = self.encode(feats, shapes, lsi, img_metas, can_bus, prev_bev)
                    self._mark(f"frame{t}.encoder")
                next_bev_feats = [prev_bev.unsqueeze(0).repeat(len(self.bev_pred_head), 1, 1, 1)]
                prev_bev_input = prev_bev.unsqueeze(1)
                for _ in range(self.test_future_frames):
                    pred_feat, last = self.decode_future(prev_bev_input, can_bus)
                    next_bev_feats.append(pred_feat)
                    prev_bev_input = last.unsqueeze(1)
                self._mark("future_decoder")
                next_bev_preds = self.forward_head(torch.stack(next_bev_feats, 0))
                pred_dict = dict(next_bev_preds=next_bev_preds[:, :, self.history_frames],
                                 valid_frames=list(range(1 + self.test_future_frames)))
                self._mark("head")
                ret_dict = self.ray_head.evaluate(pred_dict, gt_points, 0, self.bev_h, self.bev_w, PC_RANGE)
                self._mark("metrics")
        finally:
            self.train(was_training)
        return [ret_dict]


# ------------------------------------------------------------------------------------------------
# synthetic sample + step
# ------------------------------------------------------------------------------------------------
def synthetic_sample(device, frames=4, cams=6, img_hw=synthetic.IMG_HW, rays_per_frame=10000, future_frames=3, seed=0,
                     bev_hw=(BEV_H, BEV_W)):
    """6 x 3 x 928 x 1600 N(0,1) frames, a nuScenes-like rig, LiDAR-like future point clouds (SURVEY.md 8d cfg4)."""
    g = torch.Generator(device=device).manual_seed(seed)
    img = torch.randn(1, frames, cams, 3, img_hw[0], img_hw[1], device=device, generator=g)
    lidar2img = synthetic.camera_rig(cams).numpy()[None]                     # host side, like img_metas
    pts = []
    _, origin, points, tindex = synthetic.dvr_inputs_lidar(M=rays_per_frame * (1 + future_frames), T=1 + future_frames, seed=seed,
                                                           grid=(HEIGHTS, bev_hw[0], bev_hw[1]))
    # voxel units -> metres (inverse of coords_to_voxel_grids)
    p = points[0]
    xyz = np.stack([p[:, 0] / bev_hw[1] * (PC_RANGE[3] - PC_RANGE[0]) + PC_RANGE[0],
                    p[:, 1] / bev_hw[0] * (PC_RANGE[4] - PC_RANGE[1]) + PC_RANGE[1],
                    p[:, 2] / HEIGHTS * (PC_RANGE[5] - PC_RANGE[2]) + PC_RANGE[2]], -1)
    pts.append(torch.from_numpy(np.concatenate([xyz, tindex[0][:, None]], -1).astype(np.float32)).to(device))
    return dict(img=img, lidar2img=lidar2img, gt_points=pts)


def train_step(model, optimizer, sample, group=None, record=False):
    """forward_train + backward + gradient sync of the sharded parameters + clip(35) + AdamW step
    (config :379-388).  -> (loss value tensor, [(stage, ms)] when `record`)."""
    model.timings = [] if record else None
    if record:
        model._mark("start")
    optimizer.zero_grad(set_to_none=True)
    losses = model.forward_train(sample["img"], sample["lidar2img"], sample["gt_points"])
    loss = sum(losses.values())
    loss.backward()
    model._mark("backward")
    if group is not None:
        sharding.allreduce_partial_grads(model, group)
        model._mark("grad_sync")
    torch.nn.utils.clip_grad_norm_([p for p in model.parameters() if p.requires_grad], 35.0)
    optimizer.step()
    model._mark("optimizer")
    stages = None
    if record:
        torch.cuda.synchronize()
        ev = model.timings
        stages = [(ev[i + 1][0], ev[i][1].elapsed_time(ev[i + 1][1])) for i in range(len(ev) - 1)]
    model.timings = None
    return loss.detach(), stages


def build(device, group=None, lr=2e-4, seed=0, row_sharded=False, **model_kwargs):
    torch.manual_seed(seed)
    model = SyntheticViDAR(**model_kwargs).to(device)
    model.set_process_group(group, row_sharded=row_sharded)
    model.train()
    for m in model.modules():                      # dropout off: replicated parts must stay identical over ranks
        if isinstance(m, nn.Dropout):
            m.p = 0.0
    opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=lr, weight_decay=0.01)
    return model, opt
