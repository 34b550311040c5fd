"""Loss / decoding half of the ViDAR head on the CUDA ray kernels.

Mirror of the parts of `ViDARHeadBase` that sit on the hot path -- the future-BEV transformer the
reference class also owns is out of scope (SURVEY.md 2) -- with the reference's method names,
arguments, returned keys and arithmetic
(projects/mmdet3d_plugin/bevformer/dense_heads/vidar_head_base.py):

  _process_gt_points               :219-276   GT point lists -> padded voxel-unit rays + tindex
  loss                             :510-660   'regularization.loss' (CE over 513 ray samples),
                                              'dist.loss', 'loss.dense_voxel' (gumbel decode + Chamfer)
  get_point_cloud_prediction       :662-752   arg-max decode -> predicted / GT point clouds
  get_rendered_pcds                :344-389
  _custom_gumbel_softmax_distance  :754-773

What runs where: the CE term never materialises the [levels, rays, 513] logits
(`ray_head.ce_regularization_loss`, one fused kernel per frame set); the dense term's gumbel decode
is fused with the sampler as well (`ray_head.gumbel_distance`); the distance term samples through
`ray_head.get_grid_features` (CUDA sampler) and then follows the reference's torch statements; Chamfer uses the nearest-neighbour kernel (`chamfer.knn_points`) in
place of mmdet3d's O(N*M) distance matrix (`chamfer_distance`, criterion 'l2', reduction 'mean':
the mean squared NN distance each way); decoding is `ray_head.decode_ray_depth`.
CUDA only, like everything else in this package.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import bev_geometry, chamfer, evaluation, ray_head


def get_inside_mask(points, point_cloud_range):
    """bevformer/utils/e2e_predictor_utils.py:146-160."""
    r = point_cloud_range
    return ((r[0] <= points[..., 0]) & (points[..., 0] <= r[3]) & (r[1] <= points[..., 1]) & (points[..., 1] <= r[4])
            & (r[2] <= points[..., 2]) & (points[..., 2] <= r[5]))


def chamfer_l2_mean(src, dst):
    """mmdet3d.models.losses.chamfer_distance(src, dst) with its defaults (criterion 'l2',
    reduction 'mean', unit weights) -> (loss_src, loss_dst): mean squared distance to the nearest
    neighbour in the other cloud.  src [1,N,3], dst [1,M,3]."""
    a = chamfer.knn_points(src, dst)
    b = chamfer.knn_points(dst, src)
    return a.dists[..., 0].mean(), b.dists[..., 0].mean()


class ViDARRayHead:
    """The ray-supervision logic of ViDARHeadBase (not an nn.Module: it owns no parameters)."""

    def __init__(self, ray_grid_num=1026, ray_grid_step=1.0, use_ce_loss=True, use_dist_loss=False,
                 use_dense_loss=True, dense_loss_weight=1.0, loss_weight=None, eval_within_grid=False):
        self.ray_grid_num = ray_grid_num
        self.ray_grid_step = ray_grid_step
        self.use_ce_loss = use_ce_loss
        self.use_dist_loss = use_dist_loss
        self.use_dense_loss = use_dense_loss
        assert self.use_ce_loss or self.use_dist_loss or self.use_dense_loss
        self.dense_loss_weight = dense_loss_weight
        self.loss_weight = np.array(loss_weight)
        assert self.loss_weight.shape[-1] == 1
        self.eval_within_grid = eval_within_grid
        self.fuse_dense_decode = True     # False: dense term through the materialising sampler + torch statements

    # ------------------------------------------------------------------ ground truth (:219-276)
    def _process_gt_points(self, bev_preds, gt_points, batched_origin_points, valid_frames, start_idx,
                           pred_frame_num, bev_h, bev_w, pc_range):
        valid_frame_num, inter_num, bs, token_num, num_height_pred = bev_preds.shape
        frames = [i for i in range(start_idx, pred_frame_num) if i in valid_frames]
        # The reference selects every frame's points with a boolean mask (a host sync per (batch, frame)),
        # concatenates them in frame order and NaN-pads to the longest sample (:239-262).  Same rays, same
        # order, no sync: a stable sort by the frame's position in `frames`; points of other frames become
        # padding (NaN coordinates, tindex -1) at the tail instead of being dropped -- every consumer skips
        # padded rays, so only the padded length differs (it is the input length, known on the host).
        max_pts = max(int(p.shape[0]) for p in gt_points[:bs])
        pts = bev_preds.new_full((bs, max_pts, 3), float("nan"))
        tindex = bev_preds.new_full((bs, max_pts), -1.0)
        for b in range(bs):
            cur = gt_points[b]
            f = cur[:, -1]
            key = torch.full_like(f, float(len(frames)))
            for r, i in enumerate(frames):
                key = torch.where(f == i, torch.full_like(f, float(r)), key)
            order = torch.argsort(key, stable=True)
            keep = (key[order] < len(frames))
            srt = cur[order]
            pts[b, : cur.shape[0]] = torch.where(keep[:, None], srt[:, :3].to(pts.dtype), pts.new_tensor(float("nan")))
            tindex[b, : cur.shape[0]] = torch.where(keep, srt[:, -1].to(pts.dtype) - start_idx, pts.new_tensor(-1.0))
        if batched_origin_points is None:
            batched_origin_points = torch.zeros((bs, len(valid_frames), 3), dtype=bev_preds.dtype, device=bev_preds.device)
        origin_grids = bev_geometry.coords_to_voxel_grids(batched_origin_points, bev_h=bev_h, bev_w=bev_w,
                                                          pillar_num=num_height_pred, pc_range=pc_range)
        gt_grids = bev_geometry.coords_to_voxel_grids(pts, bev_h=bev_h, bev_w=bev_w, pillar_num=num_height_pred,
                                                      pc_range=pc_range)
        tindex = torch.clamp(tindex, max=valid_frame_num - 1)
        return origin_grids, batched_origin_points, gt_grids, pts, tindex

    # ------------------------------------------------------------------ decode helpers
    def get_rendered_pcds(self, origin, points, tindex, gt_dist, pred_dist, pc_range):
        """:344-389 -> pcds[b][t] = origin_t + unit(points - origin_t) * pred_dist for rays of frame t with gt_dist > 0."""
        bs, num_frames, _ = origin.shape
        pcds = []
        for b in range(bs):
            cur = []
            for t in range(num_frames):
                mask = torch.logical_and(tindex[b] == t, gt_dist[b] > 0.)
                if self.eval_within_grid:
                    mask = torch.logical_and(mask, get_inside_mask(points[b], pc_range))
                p = points[b][mask]
                r = p - origin[b, t].view(1, 3)
                r_norm = r / torch.sqrt((r ** 2).sum(1, keepdims=True))
                cur.append(origin[b, t].view(1, 3) + r_norm * pred_dist[b][mask].view(-1, 1))
            pcds.append(cur)
        return pcds

    def _custom_gumbel_softmax_distance(self, grid_embed, grid_length, gumbels=None):
        """:754-773: sample one waypoint per ray by Gumbel-max, return its length with the gradient of
        `length * P(a waypoint beyond it)` (straight-through on the probability).
        `gumbels`: optional pre-drawn Gumbel(0,1) noise of grid_embed's shape (tests pin the reference's
        CPU draw this way); None draws with the statement F.gumbel_softmax uses, so the generator is
        consumed exactly like in the reference.  The hard one-hot of F.gumbel_softmax is
        `y_hard - y_soft.detach() + y_soft`, whose picked entry is exactly 1.0f and whose other entries are
        exactly 0 in fp32, so `(hard * length).sum(-1)` equals the gather below bit for bit."""
        if gumbels is None:
            gumbels = -torch.empty_like(grid_embed, memory_format=torch.legacy_contiguous_format).exponential_().log()
        pick = (grid_embed + gumbels).softmax(-1).max(-1, keepdim=True)[1]
        sampled = grid_length.gather(-1, pick).squeeze(-1).detach()
        weight = torch.exp(grid_embed - grid_embed.max(-1, keepdim=True)[0])
        beyond = (weight * (grid_length > sampled.unsqueeze(-1)).float()).sum(-1) / weight.sum(-1)
        return (1 - beyond.detach() + beyond) * sampled

    @staticmethod
    def _sigma_volume(level, bs, frames, heights, bev_h, bev_w):
        """[frames, bs, bev_h*bev_w, heights] -> [bs, frames, heights, bev_h, bev_w] (:557-563)."""
        return level.permute(1, 0, 3, 2).contiguous().view(bs, frames, heights, bev_h, bev_w)

    # ------------------------------------------------------------------ loss (:510-660)
    def loss(self, pred_dict, gt_points, start_idx, tgt_bev_h, tgt_bev_w, tgt_pc_range, pred_frame_num,
             img_metas=None, batched_origin_points=None, loss_weight=None, gumbels=None):
        """`gumbels`: optional dict {'dist': noise, 'dense': noise} forwarded to the gumbel decode."""
        valid_frames = pred_dict["valid_frames"]
        sigma = pred_dict["next_bev_preds"][:, -1:].float()     # last intermediate output only (:540); force_fp32
        valid_frame_num, inter_num, bs, token_num, num_height_pred = sigma.shape
        (origin_grids, batched_origin_points, gt_grids, batched_gt_points, gt_tindex) = self._process_gt_points(
            sigma, gt_points, batched_origin_points, valid_frames, start_idx, pred_frame_num, tgt_bev_h, tgt_bev_w,
            tgt_pc_range)
        inter_sigma = [self._sigma_volume(sigma[:, i], bs, valid_frame_num, num_height_pred, tgt_bev_h, tgt_bev_w)
                       for i in range(inter_num)]
        step = self.ray_grid_step
        loss_weight = self.loss_weight if loss_weight is None else loss_weight
        gumbels = gumbels or {}
        loss_dict = dict()
        if self.use_dist_loss:
            r_mask, r_feat, r_w, r_len = ray_head.get_grid_features(origin_grids, gt_grids, gt_tindex, inter_sigma,
                                                                    loss_weight, step, self.ray_grid_num)
            r_pred = self._custom_gumbel_softmax_distance(r_feat + r_mask, r_len[None], gumbels.get("dist"))
            scale = (tgt_pc_range[3] - tgt_pc_range[0]) / tgt_bev_w
            dist_loss = torch.abs(r_pred - r_len[None, :, 0]) * scale
            loss_dict["dist.loss"] = (dist_loss * r_w).sum() / torch.clamp(r_w.sum(), min=1)
        if self.use_ce_loss:
            loss_dict["regularization.loss"] = ray_head.ce_regularization_loss(
                origin_grids, gt_grids, gt_tindex, inter_sigma, loss_weight, step, self.ray_grid_num)
        if self.use_dense_loss:
            tgt = inter_sigma[-1]
            interval = 4
            voxel_grids = bev_geometry.get_bev_grids_3d(tgt_bev_h // interval, tgt_bev_w // interval,
                                                        num_height_pred // interval, bs=bs, device=sigma.device)
            voxel_grids[..., 0] = voxel_grids[..., 0] * tgt_bev_w
            voxel_grids[..., 1] = voxel_grids[..., 1] * tgt_bev_h
            voxel_grids[..., 2] = voxel_grids[..., 2] * num_height_pred
            voxel_grids = voxel_grids.view(bs, -1, 3)
            ones = voxel_grids.new_ones(*voxel_grids.shape[:2]).to(gt_tindex.dtype)
            voxel_grids = torch.cat([voxel_grids for _ in range(valid_frame_num)], 1)
            voxel_tindex = torch.cat([ones * i for i in range(valid_frame_num)], 1)
            if self.fuse_dense_decode:
                # sampler + gumbel decode in one kernel per batch element: the [bs, rays, ray_grid_num]
                # logits / softmax / one-hot tensors are never written.  The noise is drawn with the
                # statement F.gumbel_softmax uses, on the shape its logits would have.
                noise = gumbels.get("dense")
                if noise is None:
                    noise = -torch.empty((bs, voxel_grids.shape[1], self.ray_grid_num), dtype=torch.float32,
                                         device=sigma.device).exponential_().log()
                frame = voxel_tindex[0].to(torch.int32).contiguous()
                dense_dist = torch.stack([
                    ray_head.gumbel_distance(tgt[b], origin_grids[b, :valid_frame_num].contiguous().float(),
                                             voxel_grids[b].contiguous(), frame, self.ray_grid_num, step, noise[b])
                    for b in range(bs)])
            else:
                _, d_feat, _, d_len = ray_head.get_grid_features(
                    origin_grids, voxel_grids, voxel_tindex, [tgt], np.array([[1]] * valid_frame_num), step,
                    self.ray_grid_num, return_as_batch=True)
                d_feat = d_feat[0][..., 1:].contiguous()
                d_len = d_len[..., 1:].contiguous()
                dense_dist = self._custom_gumbel_softmax_distance(d_feat, d_len, gumbels.get("dense"))
            voxel_pcd = self.get_rendered_pcds(origin_grids, voxel_grids, voxel_tindex, dense_dist, dense_dist, tgt_pc_range)
            dense = 0
            for b in range(bs):
                for f in range(valid_frame_num):
                    pred = voxel_pcd[b][f].view(1, -1, 3)
                    gt = gt_grids[b][gt_tindex[b] == f].view(1, -1, 3)
                    m = ((gt[..., 0] < tgt_bev_w - 1) & (gt[..., 0] > 0) & (gt[..., 1] < tgt_bev_h - 1) & (gt[..., 1] > 0)
                         & (gt[..., 2] < num_height_pred - 1) & (gt[..., 2] > 0))
                    gt = gt.squeeze(0)[m.squeeze(0)][None]
                    pred = (pred - origin_grids[b, f:f + 1]) * 0.1
                    gt = (gt - origin_grids[b, f:f + 1]) * 0.1
                    if gt.shape[1] == 0:
                        continue
                    loss_src, loss_tgt = chamfer_l2_mean(pred, gt)
                    dense = dense + ((loss_src + loss_tgt) / 2.) * loss_weight[f, 0]
            dense = dense / (loss_weight.sum() * bs)
            loss_dict["loss.dense_voxel"] = dense * self.dense_loss_weight
        return loss_dict

    # ------------------------------------------------------------------ decode (:662-752)
    def get_point_cloud_prediction(self, pred_dict, gt_points, start_idx, tgt_bev_h, tgt_bev_w, tgt_pc_range,
                                   img_metas=None, batched_origin_points=None):
        batched_origin_points, batched_gt_points, gt_tindex, gt_dist, pred_dist = self._decode_rays(
            pred_dict, gt_points, start_idx, tgt_bev_h, tgt_bev_w, tgt_pc_range, batched_origin_points)
        pred_pcds = self.get_rendered_pcds(batched_origin_points, batched_gt_points, gt_tindex, gt_dist, pred_dist, tgt_pc_range)
        gt_pcds = self.get_rendered_pcds(batched_origin_points, batched_gt_points, gt_tindex, gt_dist, gt_dist, tgt_pc_range)
        return dict(pred_pcds=pred_pcds, gt_pcds=gt_pcds, origin=batched_origin_points)

    # ------------------------------------------------------------------ evaluation (vidar.py:431-497)
    def _decode_rays(self, pred_dict, gt_points, start_idx, tgt_bev_h, tgt_bev_w, tgt_pc_range, batched_origin_points):
        """get_point_cloud_prediction's decode up to the padded per-ray distances (metres)."""
        bev_preds = pred_dict["next_bev_preds"].float()
        valid_frames = pred_dict["valid_frames"]
        pred_frame_num, inter_num, bs, token_num, num_height_pred = bev_preds.shape
        (origin_grids, batched_origin_points, gt_grids, batched_gt_points, gt_tindex) = self._process_gt_points(
            bev_preds, gt_points, batched_origin_points, valid_frames, start_idx, pred_frame_num, tgt_bev_h, tgt_bev_w,
            tgt_pc_range)
        sigma = self._sigma_volume(bev_preds[:, -1], bs, pred_frame_num, num_height_pred, tgt_bev_h, tgt_bev_w)
        pred_dist = torch.zeros_like(gt_grids[..., 0])
        gt_dist = torch.zeros_like(pred_dist)
        for b in range(bs):
            pred_dist[b], gt_dist[b] = ray_head.decode_ray_depth(sigma[b], origin_grids[b], gt_grids[b], gt_tindex[b],
                                                                 self.ray_grid_step, self.ray_grid_num)
        scale = (tgt_pc_range[3] - tgt_pc_range[0]) / tgt_bev_w
        return batched_origin_points, batched_gt_points, gt_tindex, gt_dist * scale, pred_dist * scale

    def evaluate(self, pred_dict, gt_points, start_idx, tgt_bev_h, tgt_bev_w, tgt_pc_range, img_metas=None,
                 batched_origin_points=None):
        """get_point_cloud_prediction's decode, then every (sample, frame) metric on the device
        (`evaluation.evaluate_rays`) -> forward_test's ret_dict {'frame.i': dict(count, chamfer_distance, l1_error,
        absrel_error)}, summed over the batch like vidar.py:450-497.  One host sync, at the end."""
        origin, points, tindex, gt_dist, pred_dist = self._decode_rays(
            pred_dict, gt_points, start_idx, tgt_bev_h, tgt_bev_w, tgt_pc_range, batched_origin_points)
        metrics = evaluation.evaluate_rays(origin, points, tindex, gt_dist, pred_dist, tgt_pc_range, origin.shape[1],
                                           self.eval_within_grid)
        return evaluation.ret_dict_from_metrics(metrics, start_idx)
