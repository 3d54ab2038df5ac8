"""Generates the golden fixtures in this directory by running the UNMODIFIED reference (/root/reference) on CPU
in fp32 through oracle/ref_shim.py.  Run once in the build container:

    python tests/golden/make_goldens.py

The reference tree does not exist on the GPU box, so the outputs (small .pt files) are committed.
"""
import copy
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402

TINY_YOLO_NAS = {
    "in_channels": 3,
    "backbone": {
        "NStageBackbone": {
            "stem": {"YoloNASStem": {"out_channels": 16}},
            "stages": [
                {"YoloNASStage": {"out_channels": 32, "num_blocks": 1, "activation_type": "relu", "hidden_channels": 16, "concat_intermediates": False}},
                {"YoloNASStage": {"out_channels": 48, "num_blocks": 2, "activation_type": "relu", "hidden_channels": 24, "concat_intermediates": False}},
                {"YoloNASStage": {"out_channels": 64, "num_blocks": 1, "activation_type": "relu", "hidden_channels": 32, "concat_intermediates": True}},
                {"YoloNASStage": {"out_channels": 96, "num_blocks": 1, "activation_type": "relu", "hidden_channels": 48, "concat_intermediates": False}},
            ],
            "context_module": {"SPP": {"output_channels": 96, "activation_type": "relu", "k": [5, 9, 13]}},
            "out_layers": ["stage1", "stage2", "stage3", "context_module"],
        }
    },
    "neck": {
        "YoloNASPANNeckWithC2": {
            "neck1": {"YoloNASUpStage": {"out_channels": 48, "num_blocks": 1, "hidden_channels": 24, "width_mult": 1, "depth_mult": 1, "activation_type": "relu", "reduce_channels": True}},
            "neck2": {"YoloNASUpStage": {"out_channels": 32, "num_blocks": 1, "hidden_channels": 16, "width_mult": 1, "depth_mult": 1, "activation_type": "relu", "reduce_channels": True}},
            "neck3": {"YoloNASDownStage": {"out_channels": 48, "num_blocks": 1, "hidden_channels": 24, "activation_type": "relu", "width_mult": 1, "depth_mult": 1}},
            "neck4": {"YoloNASDownStage": {"out_channels": 64, "num_blocks": 1, "hidden_channels": 32, "activation_type": "relu", "width_mult": 1, "depth_mult": 1}},
        }
    },
    "heads": {
        "NDFLHeads": {
            "num_classes": 4,
            "reg_max": 16,
            "heads_list": [
                {"YoloNASDFLHead": {"inter_channels": 32, "width_mult": 0.5, "first_conv_group_size": 0, "stride": 8}},
                {"YoloNASDFLHead": {"inter_channels": 48, "width_mult": 0.5, "first_conv_group_size": 0, "stride": 16}},
                {"YoloNASDFLHead": {"inter_channels": 64, "width_mult": 0.5, "first_conv_group_size": 0, "stride": 32}},
            ],
        }
    },
    "bn_eps": 1e-3,
    "bn_momentum": 0.03,
    "inplace_act": True,
}


def randomize_bn(module, gen):
    for m in module.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data = torch.rand(m.weight.shape, generator=gen) + 0.5
            m.bias.data = torch.randn(m.bias.shape, generator=gen) * 0.1
            m.running_mean.data = torch.randn(m.running_mean.shape, generator=gen) * 0.1
            m.running_var.data = torch.rand(m.running_var.shape, generator=gen) + 0.5


def sd_clone(m):
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def golden_qarepvgg():
    from super_gradients.modules import QARepVGGBlock

    out = {}
    for name, cin, cout, stride, res in [("s1_res", 16, 16, 1, True), ("s2", 8, 24, 2, False)]:
        gen = torch.Generator().manual_seed(1)
        torch.manual_seed(0)
        blk = QARepVGGBlock(cin, cout, stride=stride, use_residual_connection=res)
        randomize_bn(blk, gen)
        for m in blk.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.eps, m.momentum = 1e-3, 0.03
        sd0 = sd_clone(blk)
        x = torch.randn(4, cin, 16, 16, generator=gen, requires_grad=True)
        blk.train()
        y = blk(x)
        gy = torch.randn(y.shape, generator=gen)
        y.backward(gy)
        grads = {k: p.grad.clone() for k, p in blk.named_parameters() if p.grad is not None}
        sd1 = sd_clone(blk)  # running stats after one training forward
        blk.eval()
        with torch.no_grad():
            y_eval = blk(x)
            fused = copy.deepcopy(blk)
            fused.partial_fusion()
            y_partial = fused(x)
            fused.full_fusion()
            y_full = fused(x)
        out[name] = dict(cin=cin, cout=cout, stride=stride, residual=res, sd0=sd0, sd1=sd1, x=x.detach(), y=y.detach(), gy=gy, gx=x.grad.clone(), grads=grads, y_eval=y_eval, y_partial=y_partial, y_full=y_full)
    torch.save(out, os.path.join(HERE, "qarepvgg.pt"))


def golden_conv_blocks():
    from super_gradients.modules import Conv, ConvBNReLU
    from super_gradients.training.models.classification_models.resnet import BasicResNetBlock, Bottleneck
    from super_gradients.training.models.detection_models.csp_darknet53 import SPP

    out = {}
    gen = torch.Generator().manual_seed(2)
    torch.manual_seed(0)
    for name, mod, cin, hw in [
        ("conv3x3_s2", Conv(16, 24, 3, 2, torch.nn.ReLU), 16, 16),
        ("conv1x1", Conv(16, 8, 1, 1, torch.nn.ReLU), 16, 16),
        ("convbnrelu", ConvBNReLU(8, 16, kernel_size=3, stride=1, padding=1, bias=False), 8, 16),
        ("bottleneck_s2", Bottleneck(16, 8, stride=2, expansion=4), 16, 16),
        ("bottleneck_id", Bottleneck(32, 8, stride=1, expansion=4), 32, 16),
        ("basic_s2", BasicResNetBlock(16, 24, stride=2), 16, 16),
        ("spp", SPP(16, 16, (5, 9, 13), torch.nn.ReLU), 16, 16),
    ]:
        randomize_bn(mod, gen)
        sd0 = sd_clone(mod)
        x = torch.randn(4, cin, hw, hw, generator=gen, requires_grad=True)
        mod.train()
        y = mod(x)
        gy = torch.randn(y.shape, generator=gen)
        y.backward(gy)
        grads = {k: p.grad.clone() for k, p in mod.named_parameters() if p.grad is not None}
        sd1 = sd_clone(mod)
        mod.eval()
        with torch.no_grad():
            y_eval = mod(x)
        out[name] = dict(sd0=sd0, sd1=sd1, x=x.detach(), y=y.detach(), gy=gy, gx=x.grad.clone(), grads=grads, y_eval=y_eval)
    torch.save(out, os.path.join(HERE, "conv_blocks.pt"))


def golden_loss():
    from super_gradients.training.losses.functional import bbox_ciou_loss
    from super_gradients.training.losses.ppyolo_loss import GIoULoss, PPYoloELoss, TaskAlignedAssigner
    from super_gradients.training.models.detection_models.pp_yolo_e.pp_yolo_head import generate_anchors_for_grid_cell

    gen = torch.Generator().manual_seed(3)
    B, C, reg_max = 3, 4, 16
    feats = [torch.zeros(B, 1, 8, 8), torch.zeros(B, 1, 4, 4), torch.zeros(B, 1, 2, 2)]
    anchors, anchor_points, nums, stride_tensor = generate_anchors_for_grid_cell(feats, (8, 16, 32), 5.0, 0.5)
    L = sum(nums)
    out = {}
    for case, n_per_img in [("regular", [3, 2, 4]), ("ragged_with_empty", [5, 0, 1]), ("no_targets", [0, 0, 0])]:
        cls_logits = (torch.randn(B, L, C, generator=gen) * 2.0).requires_grad_(True)
        reg_distri = (torch.randn(B, L, 4 * (reg_max + 1), generator=gen) * 1.5).requires_grad_(True)
        rows = []
        for b, n in enumerate(n_per_img):
            for _ in range(n):
                cx, cy = (torch.rand(2, generator=gen) * 40 + 12).tolist()
                w, h = (torch.rand(2, generator=gen) * 30 + 8).tolist()
                rows.append([b, int(torch.randint(0, C, (1,), generator=gen)), cx, cy, w, h])
        targets = torch.tensor(rows, dtype=torch.float32).reshape(-1, 6)
        crit = PPYoloELoss(num_classes=C, use_static_assigner=False)
        raw = (cls_logits, reg_distri, anchors, anchor_points, nums, stride_tensor)
        loss, items = crit(raw, targets)
        loss.backward()
        # assignment of the same inputs (for the assigner kernel)
        with torch.no_grad():
            t = crit._get_targets_for_batched_assigner(targets, batch_size=B)
            pts_s = anchor_points / stride_tensor
            pred_bboxes, _, _ = crit._bbox_decode(pts_s, reg_distri)
            al, ab, asc = TaskAlignedAssigner(topk=13, alpha=1.0, beta=6.0)(
                pred_scores=cls_logits.sigmoid(), pred_bboxes=pred_bboxes * stride_tensor, anchor_points=anchor_points, num_anchors_list=nums,
                gt_labels=t["gt_class"], gt_bboxes=t["gt_bbox"], pad_gt_mask=t["pad_gt_mask"], bg_index=C,
            )  # fmt: skip
        out[case] = dict(
            cls_logits=cls_logits.detach(), reg_distri=reg_distri.detach(), targets=targets, loss=loss.detach(), items=items.detach(),
            g_cls=cls_logits.grad.clone(), g_reg=reg_distri.grad.clone(), assigned_labels=al, assigned_bboxes=ab, assigned_scores=asc,
            gt_class=t["gt_class"], gt_bbox=t["gt_bbox"], pad_gt_mask=t["pad_gt_mask"].float(),
        )  # fmt: skip
    out["anchors"], out["anchor_points"], out["nums"], out["stride_tensor"] = anchors, anchor_points, nums, stride_tensor
    # box losses on random boxes
    p = torch.rand(64, 4, generator=gen) * 10
    p[:, 2:] += p[:, :2] + 0.5
    g = torch.rand(64, 4, generator=gen) * 10
    g[:, 2:] += g[:, :2] + 0.5
    p.requires_grad_(True)
    gl = GIoULoss()(p, g)
    gl.sum().backward()
    g_giou = p.grad.clone()
    p.grad = None
    cl = bbox_ciou_loss(p, g, eps=1e-10)
    cl.sum().backward()
    out["boxes"] = dict(p=p.detach(), g=g, giou=gl.detach(), ciou=cl.detach(), g_giou=g_giou, g_ciou=p.grad.clone())
    torch.save(out, os.path.join(HERE, "loss.pt"))


def golden_atss():
    """Rows L2 (alt) : ATSSAssigner and PPYoloELoss(use_static_assigner=True) on a 128 x 128 input (levels of 256 / 64 / 16 anchors:
    every level holds at least topk = 9 anchors, which torch.topk needs)."""
    from super_gradients.training.losses.ppyolo_loss import ATSSAssigner, PPYoloELoss
    from super_gradients.training.models.detection_models.pp_yolo_e.pp_yolo_head import generate_anchors_for_grid_cell

    gen = torch.Generator().manual_seed(9)
    B, C, reg_max = 3, 5, 16
    feats = [torch.zeros(B, 1, 16, 16), torch.zeros(B, 1, 8, 8), torch.zeros(B, 1, 4, 4)]
    anchors, anchor_points, nums, stride_tensor = generate_anchors_for_grid_cell(feats, (8, 16, 32), 5.0, 0.5)
    L = sum(nums)
    out = {"anchors": anchors, "anchor_points": anchor_points, "nums": nums, "stride_tensor": stride_tensor}
    for case, n_per_img in [("regular", [4, 2, 6]), ("ragged_with_empty", [7, 0, 1]), ("no_targets", [0, 0, 0]), ("crowded", [12, 9, 10])]:
        cls_logits = (torch.randn(B, L, C, generator=gen) * 2.0).requires_grad_(True)
        # predicted distances concentrated around 2.5 strides (the anchor box half-size) so that IoU(gt, prediction) is not negligible
        reg_distri = (torch.randn(B, L, 4 * (reg_max + 1), generator=gen) * 1.0)
        reg_distri[..., 2::17] += 2.0
        reg_distri[..., 3::17] += 2.0
        reg_distri.requires_grad_(True)
        rows = []
        for b, n in enumerate(n_per_img):
            for _ in range(n):
                cx, cy = (torch.rand(2, generator=gen) * 96 + 16).tolist()
                w, h = (torch.rand(2, generator=gen) * (70 if case != "crowded" else 40) + 10).tolist()
                rows.append([b, int(torch.randint(0, C, (1,), generator=gen)), cx, cy, w, h])
        targets = torch.tensor(rows, dtype=torch.float32).reshape(-1, 6)
        crit = PPYoloELoss(num_classes=C, use_static_assigner=True)
        raw = (cls_logits, reg_distri, anchors, anchor_points, nums, stride_tensor)
        loss, items = crit(raw, targets)
        loss.backward()
        with torch.no_grad():
            t = crit._get_targets_for_batched_assigner(targets, batch_size=B)
            pred_bboxes, _, _ = crit._bbox_decode(anchor_points / stride_tensor, reg_distri)
            al, ab, asc = ATSSAssigner(topk=9, num_classes=C)(
                anchor_bboxes=anchors, num_anchors_list=nums, gt_labels=t["gt_class"], gt_bboxes=t["gt_bbox"], pad_gt_mask=t["pad_gt_mask"], bg_index=C,
                pred_bboxes=pred_bboxes * stride_tensor,
            )  # fmt: skip
        out[case] = dict(
            cls_logits=cls_logits.detach(), reg_distri=reg_distri.detach(), targets=targets, loss=loss.detach(), items=items.detach(), g_cls=cls_logits.grad.clone(),
            g_reg=reg_distri.grad.clone(), assigned_labels=al, assigned_bboxes=ab, assigned_scores=asc, gt_class=t["gt_class"], gt_bbox=t["gt_bbox"], pad_gt_mask=t["pad_gt_mask"].float(),
        )  # fmt: skip
        # the focal classification term (use_varifocal_loss=False) behind either assigner, on the same inputs
        for key, static in (("focal_static", True), ("focal_tal", False)):
            cl, rd = cls_logits.detach().clone().requires_grad_(True), reg_distri.detach().clone().requires_grad_(True)
            f_loss, f_items = PPYoloELoss(num_classes=C, use_static_assigner=static, use_varifocal_loss=False)((cl, rd, anchors, anchor_points, nums, stride_tensor), targets)
            f_loss.backward()
            out[case][key] = dict(loss=f_loss.detach(), items=f_items.detach(), g_cls=cl.grad.clone())
            if static:  # same assignment and box terms as the varifocal run: the regression gradient is the one stored above
                assert torch.equal(rd.grad, reg_distri.grad)
            else:
                out[case][key]["g_reg"] = rd.grad.clone()
        print(case, "positives", int((al != C).sum()), "loss", float(loss.detach()), "score sum", float(asc.sum()), "focal", float(out[case]["focal_static"]["loss"]), float(out[case]["focal_tal"]["loss"]))
    torch.save(out, os.path.join(HERE, "atss.pt"))


def golden_pose_nms():
    """YoloNASPosePostPredictionCallback of the unmodified reference on seeded decoded pose outputs."""
    from super_gradients.training.models.pose_estimation_models.yolo_nas_pose.yolo_nas_pose_post_prediction_callback import YoloNASPosePostPredictionCallback

    gen = torch.Generator().manual_seed(9)
    out = {}
    for case, (B, L, J, thr, pre, post) in {
        "regular": (2, 400, 17, 0.5, 1000, 100),
        "topk": (1, 900, 17, 0.2, 300, 50),
        "few_joints": (2, 300, 5, 0.6, 1000, 300),
        "nothing_passes": (1, 100, 17, 2.0, 1000, 100),
    }.items():
        xy = torch.rand(B, L, 2, generator=gen) * 300
        wh = torch.rand(B, L, 2, generator=gen) * 80 + 6
        boxes = torch.cat([xy, xy + wh], -1)
        conf = torch.rand(B, L, 1, generator=gen)
        coords = torch.rand(B, L, J, 2, generator=gen) * 400
        jscores = torch.rand(B, L, J, generator=gen)
        cb = YoloNASPosePostPredictionCallback(pose_confidence_threshold=thr, nms_iou_threshold=0.6, pre_nms_max_predictions=pre, post_nms_max_predictions=post)
        res = cb(((boxes, conf, coords, jscores), None))
        out[case] = dict(boxes=boxes, conf=conf, coords=coords, jscores=jscores,
                         params=dict(pose_confidence_threshold=thr, nms_iou_threshold=0.6, pre_nms_max_predictions=pre, post_nms_max_predictions=post),
                         result=[(r.poses.clone(), r.scores.clone(), r.bboxes_xyxy.clone()) for r in res])
    torch.save(out, os.path.join(HERE, "pose_nms.pt"))


def golden_pose():
    """Rows L7 / L8: YoloNASPoseNDFLHeads decode (through a real yolo_nas_pose_n model at 96x96) and YoloNASPoseLoss value +
    gradients on seeded raw predictions / targets, all from the unmodified reference."""
    from super_gradients.training import models
    from super_gradients.training.losses.yolo_nas_pose_loss import YoloNASPoseLoss

    out = {}
    torch.manual_seed(21)
    m = models.get("yolo_nas_pose_n", num_classes=17).train()
    heads = m.heads
    cap = {}
    for i in (1, 2, 3):
        getattr(heads, f"head{i}").register_forward_hook(lambda mod, inp, o, i=i: cap.__setitem__(i, tuple(t.detach().clone() for t in o)))
    x = torch.randn(2, 3, 96, 96)
    with torch.no_grad():
        decoded, raw = m(x)
    out["decode"] = dict(
        levels=[cap[i] for i in (1, 2, 3)],  # (reg_distri, cls_logit, pose_regression, pose_logits) per level
        strides=tuple(int(s) for s in heads.fpn_strides), reg_max=int(heads.reg_max), cell_offset=float(heads.grid_cell_offset), cell_scale=float(heads.grid_cell_scale),
        pose_offset_multiplier=float(heads.pose_offset_multiplier), compensate=bool(heads.compensate_grid_cell_offset),
        decoded=tuple(t.clone() for t in decoded), raw=tuple(t.clone() if torch.is_tensor(t) else t for t in raw),
    )
    # ---- loss on seeded raw predictions (anchors of a 96x96 image, strides 8/16/32 -> L = 144 + 36 + 9)
    from super_gradients.training.models.detection_models.pp_yolo_e.pp_yolo_head import generate_anchors_for_grid_cell

    gen = torch.Generator().manual_seed(22)
    B, J = 3, 17
    feats = [torch.zeros(B, 1, 96 // s, 96 // s) for s in (8, 16, 32)]
    anchors, anchor_points, nums, stride_tensor = generate_anchors_for_grid_cell(feats, (8, 16, 32), 5.0, 0.5)
    L = anchor_points.shape[0]
    sigmas = [0.026, 0.025, 0.025, 0.035, 0.035, 0.079, 0.079, 0.072, 0.072, 0.062, 0.062, 0.107, 0.107, 0.087, 0.087, 0.089, 0.089]
    boxes, joints, crowd = [], [], []
    for b, n in enumerate((3, 0, 2)):  # an image without targets in the middle
        for k in range(n):
            cx, cy = (torch.rand(2, generator=gen) * 40 + 28).tolist()
            w, h = (torch.rand(2, generator=gen) * 36 + 20).tolist()
            boxes.append([b, cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2])
            jxy = torch.stack([torch.rand(J, generator=gen) * w + cx - w / 2, torch.rand(J, generator=gen) * h + cy - h / 2], -1)
            vis = (torch.rand(J, generator=gen) > 0.3).float() * (1 + (torch.rand(J, generator=gen) > 0.5).float())
            joints.append(torch.cat([torch.full((J, 1), float(b)), jxy, vis[:, None]], -1))
            crowd.append([b, 1.0 if (b == 0 and k == 2) else 0.0])
    targets = (torch.tensor(boxes), torch.stack(joints), torch.tensor(crowd))
    variants = {
        "default": dict(),
        "oks_rescale_bce_giou": dict(classification_loss_type="bce", regression_iou_loss_type="giou", assigner_multiply_by_pose_oks=True, rescale_pose_loss_with_assigned_score=True, pose_classification_loss_type="focal"),
        # recipes/training_hyperparams/coco2017_yolo_nas_pose_train_params.yaml:23-34
        "recipe": dict(classification_loss_weight=1.0, classification_loss_type="focal", regression_iou_loss_type="ciou", iou_loss_weight=2.5, dfl_loss_weight=0.01, pose_cls_loss_weight=1.0,
                       pose_reg_loss_weight=34.0, pose_classification_loss_type="focal", rescale_pose_loss_with_assigned_score=True, assigner_multiply_by_pose_oks=True),
    }
    for name, kw in variants.items():
        cls_logits = (torch.randn(B, L, 1, generator=gen) * 1.5 - 1.0).requires_grad_(True)
        reg_distri = torch.randn(B, L, 68, generator=gen).requires_grad_(True)
        pose_coords = (anchor_points.unsqueeze(0).unsqueeze(2) + torch.randn(B, L, J, 2, generator=gen) * 12).requires_grad_(True)
        pose_logits = torch.randn(B, L, J, generator=gen).requires_grad_(True)
        raw = (cls_logits, reg_distri, pose_coords, pose_logits, anchors, anchor_points, nums, stride_tensor)
        crit = YoloNASPoseLoss(oks_sigmas=sigmas, **kw)
        loss, items = crit((None, raw), targets)
        loss.backward()
        out["loss_" + name] = dict(kw=kw, sigmas=sigmas, targets=targets, raw=tuple(t.detach().clone() if torch.is_tensor(t) else t for t in raw), loss=loss.detach(), items=items.clone(),
                                   grads=tuple(t.grad.clone() for t in (cls_logits, reg_distri, pose_coords, pose_logits)))
    torch.save(out, os.path.join(HERE, "pose.pt"))


def golden_nms():
    from super_gradients.training.models.detection_models.pp_yolo_e import PPYoloEPostPredictionCallback

    gen = torch.Generator().manual_seed(4)
    out = {}
    for case, (B, L, C, thr, topk, maxp, multi, agn) in {
        "multi_small": (2, 300, 4, 0.6, 1000, 300, True, False),
        "multi_topk": (2, 600, 6, 0.3, 200, 50, True, False),
        "multi_vanilla": (1, 2500, 3, 0.5, 1024, 300, True, False),
        "single_label": (2, 500, 5, 0.7, 100, 300, False, False),
        "class_agnostic": (2, 400, 4, 0.7, 1000, 300, True, True),
        "nothing_passes": (2, 100, 3, 2.0, 1000, 300, True, False),
    }.items():
        xy = torch.rand(B, L, 2, generator=gen) * 200
        wh = torch.rand(B, L, 2, generator=gen) * 60 + 4
        boxes = torch.cat([xy, xy + wh], -1)
        scores = torch.rand(B, L, C, generator=gen)
        cb = PPYoloEPostPredictionCallback(score_threshold=thr, nms_threshold=0.65, nms_top_k=topk, max_predictions=maxp, multi_label_per_box=multi, class_agnostic_nms=agn)
        res = cb(((boxes, scores), None))
        out[case] = dict(boxes=boxes, scores=scores, params=dict(score_threshold=thr, nms_threshold=0.65, nms_top_k=topk, max_predictions=maxp, multi_label_per_box=multi, class_agnostic_nms=agn), result=[r.clone() for r in res])
    torch.save(out, os.path.join(HERE, "nms.pt"))


def golden_yolox_nms():
    """Row N3: the reference's non_max_suppression / YoloXPostPredictionCallback on synthetic YoloX-format predictions."""
    from super_gradients.training.models.detection_models.yolo_base import YoloXPostPredictionCallback
    from super_gradients.training.utils.detection_utils import non_max_suppression

    gen = torch.Generator().manual_seed(9)
    out = {}
    for case, (B, A, C, conf, multi, withc, agn) in {
        "multi_conf": (2, 400, 4, 0.35, True, True, False),
        "multi_raw": (2, 300, 3, 0.6, True, False, False),
        "single": (2, 500, 5, 0.45, False, True, False),
        "agnostic": (1, 400, 4, 0.4, True, True, True),
        "one_empty_image": (2, 200, 3, 0.5, True, True, False),
        "nothing_passes": (2, 100, 3, 1.5, True, True, False),
    }.items():
        cxy = torch.rand(B, A, 2, generator=gen) * 200 + 20
        wh = torch.rand(B, A, 2, generator=gen) * 60 + 4
        obj = torch.rand(B, A, 1, generator=gen)
        cls = torch.rand(B, A, C, generator=gen)
        if case == "one_empty_image":
            obj[1] *= 0.4  # below the objectness filter everywhere
        pred = torch.cat([cxy, wh, obj, cls], -1)
        kw = dict(conf_thres=conf, iou_thres=0.6, multi_label_per_box=multi, with_confidence=withc, class_agnostic_nms=agn)
        res = non_max_suppression(pred.clone(), **kw)
        cb = YoloXPostPredictionCallback(conf=conf, iou=0.6, max_predictions=15, with_confidence=withc, class_agnostic_nms=agn, multi_label_per_box=multi)
        res_cb = cb((pred.clone(), None))
        out[case] = dict(pred=pred, kw=kw, result=[None if r is None else r.clone() for r in res], callback=[None if r is None else r.clone() for r in res_cb])
    torch.save(out, os.path.join(HERE, "yolox_nms.pt"))


def golden_processing():
    """Row (f)-N3: the reference's own ComposeProcessing chains (cv2 + numpy) on random uint8 images, and their box post-processing."""
    import numpy as np
    from super_gradients.training.processing import processing as P
    from super_gradients.training.utils.predict import DetectionPrediction, PoseEstimationPrediction

    import hashlib

    rng = np.random.RandomState(12)  # legacy stream: frozen across numpy versions, so the tests regenerate the images instead of storing them
    chains = {
        "yolo_nas_default": (lambda: [P.DetectionLongestMaxSizeRescale(output_shape=(636, 636)), P.DetectionCenterPadding(output_shape=(640, 640), pad_value=114),
                                      P.StandardizeImage(max_value=255.0), P.ImagePermute(permutation=(2, 0, 1))],
                             dict(rescale=(636, 636), keep_aspect=True, pad_shape=(640, 640), pad_value=114, center=True)),
        "pose_default": (lambda: [P.ReverseImageChannels(), P.KeypointsLongestMaxSizeRescale(output_shape=(640, 640)), P.KeypointsBottomRightPadding(output_shape=(640, 640), pad_value=127),
                                  P.StandardizeImage(max_value=255.0), P.ImagePermute(permutation=(2, 0, 1))],
                         dict(rescale=(640, 640), keep_aspect=True, pad_shape=(640, 640), pad_value=127, center=False, reverse=True)),
        "stretch_normalize": (lambda: [P.DetectionRescale(output_shape=(96, 160)), P.StandardizeImage(max_value=255.0), P.NormalizeImage(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225]),
                                       P.ImagePermute(permutation=(2, 0, 1))],
                              dict(rescale=(96, 160), keep_aspect=False, mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])),
    }  # fmt: skip
    out = {}
    for name, (mk, kw) in chains.items():
        cases = []
        for (h, w) in [(427, 640), (640, 480), (333, 500), (1080, 1920), (64, 48), (640, 640)]:
            seed = int(rng.randint(0, 2**31 - 1))
            img = np.random.RandomState(seed).randint(0, 256, (h, w, 3)).astype(np.uint8)
            cp = P.ComposeProcessing(mk())
            pre, metas = cp.preprocess_image(img)
            boxes = np.concatenate([rng.uniform(0, pre.shape[2] / 2, (5, 1)), rng.uniform(0, pre.shape[1] / 2, (5, 1)),
                                    rng.uniform(0, pre.shape[2], (5, 1)), rng.uniform(0, pre.shape[1], (5, 1))], 1).astype(np.float32)
            poses = np.concatenate([rng.uniform(0, pre.shape[2], (5, 4, 1)), rng.uniform(0, pre.shape[1], (5, 4, 1)), rng.uniform(0, 1, (5, 4, 1))], -1).astype(np.float32)
            if name == "pose_default":
                pred = PoseEstimationPrediction(poses=poses.copy(), scores=np.ones(5, np.float32), bboxes_xyxy=boxes.copy(), edge_links=np.zeros((0, 2), int), edge_colors=np.zeros((0, 3), int),
                                                keypoint_colors=np.zeros((4, 3), int), image_shape=pre.shape[1:])
            else:
                pred = DetectionPrediction(bboxes=boxes.copy(), bbox_format="xyxy", confidence=np.ones(5, np.float32), labels=np.zeros(5, np.float32), image_shape=pre.shape[1:])
            post = cp.postprocess_predictions(pred, metas)
            pre_bf16 = torch.from_numpy(np.ascontiguousarray(pre)).to(torch.bfloat16)  # what the model mirrors consume (round to nearest)
            case = dict(image_seed=seed, image_shape=(h, w), pre_shape=tuple(pre.shape), pre_sha256=hashlib.sha256(pre_bf16.view(torch.int16).numpy().tobytes()).hexdigest(),
                        pre_sample=pre_bf16[:, ::37, ::41].clone(), pre_sum=float(pre_bf16.double().sum()),
                        boxes=torch.from_numpy(boxes), boxes_post=torch.from_numpy(np.asarray(post.bboxes_xyxy, dtype=np.float32)))
            if name == "pose_default":
                case.update(poses=torch.from_numpy(poses), poses_post=torch.from_numpy(np.asarray(post.poses, dtype=np.float32)))
            cases.append(case)
        out[name] = dict(kw=kw, cases=cases)
    torch.save(out, os.path.join(HERE, "processing.pt"))


def _metric_scene(gen, n_img, n_cls, hw, max_t, max_p, crowd, normalized):
    """Synthetic NMS output / ground truth of one validation batch: predictions are jittered copies of targets plus clutter."""
    H, W = hw
    targets, crowds, output = [], [], []
    for i in range(n_img):
        nt = int(torch.randint(0, max_t + 1, (1,), generator=gen))
        cxcy = torch.rand(nt, 2, generator=gen) * torch.tensor([W, H]) * 0.8 + torch.tensor([W, H]) * 0.1
        wh = torch.rand(nt, 2, generator=gen) * torch.tensor([W, H]) * 0.3 + 8
        cls = torch.randint(0, n_cls, (nt, 1), generator=gen).float()
        t = torch.cat([torch.full((nt, 1), float(i)), cls, cxcy, wh], 1)
        is_crowd = (torch.rand(nt, generator=gen) < 0.2) if crowd else torch.zeros(nt, dtype=torch.bool)
        boxes = []
        for k in range(nt):
            for _ in range(int(torch.randint(0, 5, (1,), generator=gen))):
                jit = (torch.rand(4, generator=gen) - 0.5) * torch.tensor([0.3, 0.3, 0.4, 0.4])
                cx, cy = (t[k, 2:4] + jit[:2] * t[k, 4:6]).tolist()
                w, h = (t[k, 4:6] * (1 + jit[2:])).tolist()
                c = t[k, 1].item() if torch.rand(1, generator=gen) < 0.85 else float(torch.randint(0, n_cls, (1,), generator=gen))
                boxes.append([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2, 0.0, c])
        n_clutter = int(torch.randint(0, max_p + 1, (1,), generator=gen))
        for _ in range(n_clutter):
            x1, y1 = (torch.rand(2, generator=gen) * torch.tensor([W, H]) * 1.1 - 10).tolist()
            w, h = (torch.rand(2, generator=gen) * 120 + 4).tolist()
            boxes.append([x1, y1, x1 + w, y1 + h, 0.0, float(torch.randint(0, n_cls, (1,), generator=gen))])
        p = torch.tensor(boxes, dtype=torch.float32).reshape(-1, 6)
        if len(p):
            sc = torch.rand(len(p), generator=gen)
            p[:, 4] = sc[torch.argsort(sc, descending=True)]  # NMS output is sorted by confidence
            if len(p) > 3:
                p[-1, 4] = 0.0  # a zero score is dropped by the top-k selection (nonzero())
            assert len(torch.unique(p[:, 4])) == len(p)
        if normalized:
            t[:, [2, 4]] /= W
            t[:, [3, 5]] /= H
        targets.append(t[~is_crowd])
        crowds.append(t[is_crowd])
        output.append(p if len(p) and i != 1 else None)  # image 1: "no prediction"
    return output, torch.cat(targets), torch.cat(crowds)


def golden_detection_metrics():
    """Row (f)-N4: compute_detection_matching (IoUMatching) and compute_detection_metrics on synthetic batches."""
    from super_gradients.training.utils.detection_utils import IoUMatching, IouThreshold, compute_detection_matching, compute_detection_metrics

    gen = torch.Generator().manual_seed(77)
    cases = {}
    specs = {
        "coco_range_crowd": dict(n_img=6, n_cls=5, hw=(320, 416), max_t=9, max_p=40, crowd=True, normalized=True, top_k=12, thr=IouThreshold.MAP_05_TO_095.to_tensor(), score_thres=0.1),
        "single_thr_pixels": dict(n_img=4, n_cls=3, hw=(256, 256), max_t=6, max_p=10, crowd=False, normalized=False, top_k=100, thr=torch.tensor([0.5]), score_thres=0.3),
        "dense": dict(n_img=3, n_cls=2, hw=(640, 640), max_t=30, max_p=150, crowd=True, normalized=True, top_k=100, thr=IouThreshold.MAP_05_TO_095.to_tensor(), score_thres=0.05),
    }
    for name, sp in specs.items():
        batches = []
        info = []
        for b in range(2):
            output, targets, crowds = _metric_scene(gen, sp["n_img"], sp["n_cls"], sp["hw"], sp["max_t"], sp["max_p"], sp["crowd"], sp["normalized"])
            res = compute_detection_matching(
                [None if o is None else o.clone() for o in output], targets.clone(), sp["hw"][0], sp["hw"][1], denormalize_targets=sp["normalized"], device="cpu",
                iou_thresholds=sp["thr"], crowd_targets=crowds.clone() if sp["crowd"] else None, top_k=sp["top_k"], matching_strategy=IoUMatching(sp["thr"]),
            )
            info += res
            batches.append({"output": output, "targets": targets, "crowd_targets": crowds if sp["crowd"] else None, "matching": [tuple(t.clone() for t in r) for r in res]})
        cat = [torch.cat(x, 0) for x in zip(*info)]
        # the recall grid is an input of the golden: torch.linspace's last bit depends on the CPU's SIMD width, and a recall of
        # exactly k / n_targets can sit on a grid point
        recall_thresholds = torch.linspace(0, 1, 101)
        ap, prec, rec, f1, classes, best, best_cls = compute_detection_metrics(*cat, device="cpu", score_threshold=sp["score_thres"], recall_thresholds=recall_thresholds)
        cases[name] = {
            "hw": sp["hw"], "top_k": sp["top_k"], "iou_thresholds": sp["thr"], "normalized": sp["normalized"], "score_thres": sp["score_thres"], "n_cls": sp["n_cls"], "recall_thresholds": recall_thresholds,
            "batches": batches, "metrics": {"ap": ap, "precision": prec, "recall": rec, "f1": f1, "classes": classes, "best_score_threshold": best, "best_per_cls": best_cls},
        }
        print(name, "preds", len(cat[0]), "matched@thr0", int(cat[0][:, 0].sum()), "ignored", int(cat[1][:, 0].sum()), "mAP", float(ap.mean()))
    torch.save(cases, os.path.join(HERE, "detection_metrics.pt"))


def golden_other_configs():
    """BASELINE.json configs 3-5 (YOLO-NAS-M training, ResNet-50 training, YOLO-NAS-POSE-L inference) at reduced resolution: the
    reference's fp32 outputs for its own seeded initialisation (torch.manual_seed(0) before models.get -- the product's
    constructors consume the RNG identically, see tests/test_abi_validation_cpu.py), so only inputs / outputs are stored."""
    from super_gradients.training import models
    from super_gradients.training.losses.ppyolo_loss import PPYoloELoss

    gen = torch.Generator().manual_seed(21)
    out = {}
    # ---- ResNet-50
    torch.manual_seed(0)
    m = models.get("resnet50", num_classes=1000).train()
    x = torch.randn(4, 3, 128, 128, generator=gen).bfloat16().float()  # exactly representable in the product's bf16 input layout
    y = torch.tensor([3, 17, 256, 999])
    logits = m(x)
    loss = torch.nn.functional.cross_entropy(logits, y)
    loss.backward()
    names = ["conv1.weight", "layer1.0.conv1.weight", "layer2.0.shortcut.0.weight", "layer3.5.conv2.weight", "layer4.2.conv3.weight", "linear.weight", "linear.bias", "layer4.2.bn3.weight"]
    params = dict(m.named_parameters())
    grads = {k: params[k].grad.clone() if params[k].grad.numel() < 20000 else params[k].grad.flatten()[:: params[k].grad.numel() // 10000].clone() for k in names}
    grad_norms = {k: float(p.grad.norm()) for k, p in params.items() if p.grad is not None}
    m.eval()
    with torch.no_grad():
        eval_logits = m(x)
    out["resnet50"] = dict(x=x.to(torch.bfloat16), y=y, train_logits=logits.detach(), loss=loss.detach(), grads=grads, grad_norms=grad_norms, eval_logits=eval_logits)
    # NOTE on tolerances: at random initialisation, batch 4 and 4 x 4 final maps the train-mode network is chaotic.  The reference
    # itself, re-run with every Conv2d / BatchNorm2d / ReLU output rounded to bf16 (straight-through forward hooks), moves its
    # logits by 0.16 (relative L2) and leaves the early layers' gradients ~uncorrelated with the fp32 ones (relative L2 1.2-1.3)
    # while the gradient NORMS stay within a few percent.  Hence logits / loss / gradient norms / eval-mode logits are compared,
    # gradient directions only at the classifier.
    print("resnet50 loss", float(loss))
    # ---- YOLO-NAS-M
    torch.manual_seed(0)
    m = models.get("yolo_nas_m", num_classes=80).train()
    x = torch.randn(2, 3, 128, 128, generator=gen).bfloat16().float()
    rows = []
    for b in range(2):
        for _ in range(3):
            cx, cy = (torch.rand(2, generator=gen) * 76 + 26).tolist()
            w, h = (torch.rand(2, generator=gen) * 40 + 10).tolist()
            rows.append([b, int(torch.randint(0, 80, (1,), generator=gen)), cx, cy, w, h])
    targets = torch.tensor(rows, dtype=torch.float32)
    outputs = m(x)
    raw = outputs[1] if isinstance(outputs, tuple) and len(outputs) == 2 else outputs
    loss, items = PPYoloELoss(num_classes=80, use_static_assigner=False)(outputs, targets)
    loss.backward()
    params = dict(m.named_parameters())
    grad_norms = {k: float(p.grad.norm()) for k, p in params.items() if p.grad is not None}
    m.eval()
    with torch.no_grad():
        (eb, es), _ = m(x)
    out["yolo_nas_m"] = dict(x=x.to(torch.bfloat16), targets=targets, cls_logits=raw[0].detach(), reg_distri=raw[1].detach(), loss=loss.detach(), items=items.detach(), grad_norms=grad_norms,
                             eval_boxes=eb, eval_scores=es)  # fmt: skip
    print("yolo_nas_m loss", float(loss.detach()), items)
    # ---- YOLO-NAS-POSE-L
    torch.manual_seed(0)
    m = models.get("yolo_nas_pose_l", num_classes=17).eval()
    x = torch.rand(2, 3, 128, 128, generator=gen).bfloat16().float()
    with torch.no_grad():
        decoded, _raw = m(x)
    out["yolo_nas_pose_l"] = dict(x=x.to(torch.bfloat16), boxes=decoded[0], scores=decoded[1], poses=decoded[2], joint_scores=decoded[3])
    print("pose_l", [tuple(t.shape) for t in decoded])
    torch.save(out, os.path.join(HERE, "other_configs.pt"))


def golden_port_fidelity():
    """The workload of `bench.py --impl reference` / `cpu_baseline` (BASELINE config 2 on a 2-image sample): the UNMODIFIED reference's
    YOLO-NAS-S, loaded with exactly the state the oracle port starts from (oracle.yolo_nas_oracle.random_state(seed 0)) and fed the
    bench's own synthetic batch (bench.synth_batch(2, 123, 640)), one fp32 train-mode forward + PPYoloELoss(TAL) + backward on CPU.
    Only scalars are stored (loss, its components, a checksum of the raw head outputs, per-parameter gradient norms): the test that
    reads this file (tests/test_oracle_golden.py::test_bench_cpu_port_is_the_reference_train_step) times nothing."""
    import bench
    from oracle.yolo_nas_oracle import random_state
    from super_gradients.training import models
    from super_gradients.training.losses.ppyolo_loss import PPYoloELoss

    table = torch.load(os.path.join(HERE, "state_keys.pt"), weights_only=False)
    state = random_state(table["yolo_nas_s"], seed=0)
    m = models.get("yolo_nas_s", num_classes=bench.NCLS)
    missing, unexpected = m.load_state_dict({k: v.clone() for k, v in state.items()}, strict=False)
    assert not unexpected and all("num_batches_tracked" in k or "id_tensor" in k for k in missing), (missing, unexpected)
    m.train()
    x, t = bench.synth_batch(2, 123, 640)
    outputs = m(x)
    raw = outputs[1] if isinstance(outputs, tuple) and len(outputs) == 2 else outputs
    loss, items = PPYoloELoss(num_classes=bench.NCLS, use_static_assigner=False)(outputs, t)
    loss.backward()
    grad_norms = {k: float(p.grad.norm()) for k, p in m.named_parameters() if p.grad is not None}
    out = dict(loss=float(loss.detach()), items=[float(v) for v in items.detach().reshape(-1)], cls_logits_sum=float(raw[0].detach().double().sum()),
               cls_logits_abs=float(raw[0].detach().double().abs().sum()), reg_distri_abs=float(raw[1].detach().double().abs().sum()), grad_norms=grad_norms,
               n_targets=int(t.shape[0]) if torch.is_tensor(t) else len(t))  # fmt: skip
    print("port fidelity: reference loss", out["loss"], out["items"], "params with gradients", len(grad_norms))
    # config 4's CPU arm: ResNet-50 at 224 x 224 on a 4-image sample of the bench's classification batch, the port's own initial state,
    # drop-path off on both sides (the reference draws its masks from the global RNG inside forward; the port's masks are pinned
    # separately by droppath.pt)
    table = torch.load(os.path.join(HERE, "state_keys.pt"), weights_only=False)
    state = random_state(table["resnet50"], seed=0)
    m = models.get("resnet50", num_classes=1000)
    missing, unexpected = torch.nn.Module.load_state_dict(m, {k: v.clone() for k, v in state.items()}, strict=False)  # the reference's override returns None
    assert not unexpected and all("num_batches_tracked" in k for k in missing), (missing, unexpected)
    m.train()
    x, y = bench.synth_cls_batch(4, 123, 224)
    logits = m(x)
    loss = torch.nn.functional.cross_entropy(logits, y)
    loss.backward()
    out["resnet50"] = dict(loss=float(loss.detach()), logits_abs=float(logits.detach().double().abs().sum()),
                           grad_norms={k: float(p.grad.norm()) for k, p in m.named_parameters() if p.grad is not None})
    print("port fidelity: reference resnet50 loss", out["resnet50"]["loss"])
    torch.save(out, os.path.join(HERE, "port_fidelity_2x640.pt"))


def golden_lr_schedules():
    """LR actually in the optimizer at every optimisation step, produced by the reference's own warm-up / scheduler callbacks driven in
    the order of Trainer._train_epoch (epoch-start callbacks, per batch: batch-start callbacks -> optimizer step -> TRAIN_BATCH_STEP
    callbacks, then epoch-end callbacks)."""
    from super_gradients.common.registry.registry import LR_SCHEDULERS_CLS_DICT, LR_WARMUP_CLS_DICT
    from super_gradients.training.utils import HpmStruct
    from super_gradients.training.utils.callbacks import Phase, PhaseContext

    base = dict(lr_mode=None, lr_warmup_epochs=0, lr_warmup_steps=0, lr_cooldown_epochs=0, warmup_initial_lr=None, warmup_mode="LinearEpochLRWarmup", cosine_final_lr_ratio=0.01,
                lr_updates=[], lr_decay_factor=0.1, step_lr_update_freq=None, max_epochs=6, initial_lr=0.1)
    cases = {
        "yolo_nas_recipe": dict(warmup_mode="LinearBatchLRWarmup", warmup_initial_lr=1e-6, lr_warmup_steps=1000, initial_lr=2e-4, lr_mode="CosineLRScheduler", cosine_final_lr_ratio=0.1, max_epochs=4),
        "pose_recipe_like": dict(warmup_mode="LinearBatchLRWarmup", warmup_initial_lr=1e-6, lr_warmup_steps=3, lr_warmup_epochs=2, initial_lr=2e-3, lr_mode="cosine", cosine_final_lr_ratio=0.05),
        "resnet50_like": dict(lr_warmup_epochs=2, lr_mode="CosineLRScheduler", initial_lr=0.1),
        "cifar_like": dict(lr_mode="StepLRScheduler", lr_updates=[2, 4], lr_decay_factor=0.1, initial_lr=0.1),
        "epoch_warmup_given_start_step": dict(lr_warmup_epochs=3, warmup_initial_lr=0.01, lr_mode="step", lr_updates=[4], lr_decay_factor=0.5, initial_lr=0.2),
        "cosine_cooldown": dict(lr_mode="cosine", lr_cooldown_epochs=2, initial_lr=0.05, cosine_final_lr_ratio=0.1),
    }
    out = {}
    loader_len = 5
    for name, kw in cases.items():
        tp = HpmStruct(**{**base, **kw})
        net = torch.nn.Linear(2, 2)
        opt = torch.optim.SGD([{"params": net.parameters(), "name": "default"}], lr=tp.initial_lr)
        common = dict(train_loader_len=loader_len, net=net, training_params=tp, update_param_groups=False, **tp.to_dict())
        cbs = []
        if tp.lr_mode is not None:
            cbs.append(LR_SCHEDULERS_CLS_DICT[tp.lr_mode](**common))
        cbs.append(LR_WARMUP_CLS_DICT[tp.warmup_mode](**common))
        ctx = PhaseContext(epoch=0, batch_idx=0, optimizer=opt, net=net)
        lrs = []

        def fire(phase):
            for cb in cbs:
                if getattr(cb, "phase", None) == phase:
                    cb(ctx)

        for epoch in range(tp.max_epochs):
            ctx.update_context(epoch=epoch, batch_idx=0)
            fire(Phase.TRAIN_EPOCH_START)
            for b in range(loader_len):
                ctx.update_context(batch_idx=b)
                for cb in cbs:
                    if hasattr(cb, "on_train_batch_start") and not hasattr(cb, "phase"):
                        cb.on_train_batch_start(ctx)
                lrs.append(float(opt.param_groups[0]["lr"]))
                fire(Phase.TRAIN_BATCH_STEP)
                fire(Phase.TRAIN_BATCH_END)
            fire(Phase.TRAIN_EPOCH_END)
        out[name] = dict(params={**base, **kw}, loader_len=loader_len, lrs=lrs)
    torch.save(out, os.path.join(HERE, "lr_schedules.pt"))


def golden_param_groups():
    """zero_weight_decay_on_bias_and_bn: which parameters the reference puts in the weight_decay = 0 group
    (training/utils/optimizer_utils.py:32-85), for the tiny YOLO-NAS, the tiny YOLO-NAS-POSE and resnet18_cifar."""
    from super_gradients.training import models
    from super_gradients.training.models.detection_models.yolo_nas.yolo_nas_variants import YoloNAS
    from super_gradients.training.models.pose_estimation_models.yolo_nas_pose.yolo_nas_pose_variants import YoloNASPose
    from super_gradients.training.utils.optimizer_utils import _get_no_decay_param_ids

    out = {}
    ap = copy.deepcopy(TINY_YOLO_NAS)
    nets = {"tiny_yolo_nas": YoloNAS(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=4, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)}
    ap = copy.deepcopy(tiny_pose_arch())
    nets["tiny_yolo_nas_pose"] = YoloNASPose(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=5, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    nets["resnet18_cifar"] = models.get("resnet18_cifar", num_classes=10)
    for name, net in nets.items():
        ids = set(_get_no_decay_param_ids(net))
        out[name] = dict(no_decay=[k for k, p in net.named_parameters() if id(p) in ids], decay=[k for k, p in net.named_parameters() if id(p) not in ids])
    torch.save(out, os.path.join(HERE, "param_groups.pt"))


def golden_collate_decoding():
    """DetectionCollateFN / YoloNASPoseCollateFN (collate_fn/detection_collate_fn.py, yolo_nas_pose_collate_fn.py) and the export
    graph's YoloNASDecodingModule / YoloNASPoseDecodingModule (yolo_nas_variants.py:53-72, yolo_nas_pose_variants.py:54-90) on the
    seeded inputs of tests/test_host_logic.py."""
    sys.path.insert(0, os.path.dirname(HERE))
    import test_host_logic as T
    from super_gradients.training.datasets.pose_estimation_datasets.yolo_nas_pose_collate_fn import YoloNASPoseCollateFN
    from super_gradients.training.models.detection_models.yolo_nas.yolo_nas_variants import YoloNASDecodingModule
    from super_gradients.training.models.pose_estimation_models.yolo_nas_pose.yolo_nas_pose_variants import YoloNASPoseDecodingModule
    from super_gradients.training.utils.collate_fn.detection_collate_fn import DetectionCollateFN

    det_images, det_targets = DetectionCollateFN()(T._collate_samples(0))
    pose_images, pose_targets, _ = YoloNASPoseCollateFN()(T._pose_samples(1))
    boxes, scores, conf, coords, js = T._decoding_inputs(0)
    out = dict(
        det_images=det_images, det_targets=det_targets, pose_images=pose_images, pose_targets=pose_targets,
        det_decoded=YoloNASDecodingModule(100)(((boxes, scores), None)), pose_decoded=YoloNASPoseDecodingModule(64)(((boxes, conf, coords, js), None)),
    )  # fmt: skip
    torch.save(out, os.path.join(HERE, "collate_decoding.pt"))


def golden_tiny_yolo_nas():
    from super_gradients.training.losses.ppyolo_loss import PPYoloELoss
    from super_gradients.training.models.detection_models.yolo_nas.yolo_nas_variants import YoloNAS
    from super_gradients.training.utils import HpmStruct

    gen = torch.Generator().manual_seed(5)
    torch.manual_seed(0)
    ap = copy.deepcopy(TINY_YOLO_NAS)
    m = YoloNAS(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=4, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    randomize_bn(m, gen)
    sd0 = sd_clone(m)
    # 4 x 128 x 128: the deepest feature map is 4 x 4, i.e. 64 samples per channel for the train-mode BatchNorms
    # (with fewer samples the normalisation amplifies bf16 rounding noise of the product path beyond any fixed tolerance)
    x = torch.randn(4, 3, 128, 128, generator=gen)
    targets = torch.tensor([[0, 1, 60.0, 56.0, 48.0, 40.0], [0, 3, 80.0, 88.0, 36.0, 60.0], [1, 0, 40.0, 72.0, 60.0, 44.0], [2, 2, 64.0, 64.0, 80.0, 70.0], [3, 1, 30.0, 90.0, 40.0, 50.0]])
    m.train()
    outs = m(x)
    crit = PPYoloELoss(num_classes=4, use_static_assigner=False)
    loss, items = crit(outs, targets)
    loss.backward()
    grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    sd1 = sd_clone(m)
    m.eval()
    with torch.no_grad():
        (eb, es), raw = m(x)
    live = {k: v for k, v in sd0.items() if "rbr_reparam" not in k}  # dead placeholders are not needed to reproduce
    running = {k: v for k, v in sd1.items() if "running_" in k}
    gsum = {k: (float(g.double().sum()), float(g.double().norm())) for k, g in grads.items()}
    keep = [k for k in grads if k.startswith("backbone.stem") or k.startswith("backbone.stage1.downsample") or k.startswith("heads.head1") or k.startswith("neck.neck2.upsample")]
    torch.save(
        dict(arch=TINY_YOLO_NAS, sd0=live, running1=running, x=x, targets=targets, train_pred_bboxes=outs[0][0].detach(), train_pred_scores=outs[0][1].detach(),
             train_cls_logits=outs[1][0].detach(), train_reg_distri=outs[1][1].detach(), loss=loss.detach(), items=items.detach(),
             grads={k: grads[k] for k in keep}, grad_sums=gsum, eval_pred_bboxes=eb, eval_pred_scores=es,
             param_names=[k for k, _ in m.named_parameters()], state_keys=list(m.state_dict().keys())),
        os.path.join(HERE, "tiny_yolo_nas.pt"),
    )  # fmt: skip


def tiny_pose_arch():
    """TINY_YOLO_NAS backbone + neck with small YoloNASPoseDFLHeads (5 joints; separate stems, joint logits in the class head
    -- the configuration of every shipped YOLO-NAS-POSE variant)."""
    ap = copy.deepcopy(TINY_YOLO_NAS)
    mk = lambda b, p, r, s: {"YoloNASPoseDFLHead": {"bbox_inter_channels": b, "pose_inter_channels": p, "pose_regression_blocks": r, "shared_stem": False, "width_mult": 0.5,
                                                     "pose_conf_in_class_head": True, "pose_block_use_repvgg": False, "first_conv_group_size": 0, "stride": s}}  # noqa: E731
    ap["heads"] = {"YoloNASPoseNDFLHeads": {"num_classes": 5, "reg_max": 16, "pose_offset_multiplier": 1.0, "compensate_grid_cell_offset": True, "inference_mode": False,
                                            "heads_list": [mk(32, 32, 2, 8), mk(48, 64, 2, 16), mk(64, 64, 3, 32)]}}
    return ap


def golden_tiny_yolo_nas_pose():
    """Row L8 end to end: eval-mode forward of a tiny YOLO-NAS-POSE built from the reference classes (random weights and
    BatchNorm running statistics), decoded + raw outputs, and the post-prediction callback on them."""
    from super_gradients.training.models.pose_estimation_models.yolo_nas_pose.yolo_nas_pose_post_prediction_callback import YoloNASPosePostPredictionCallback
    from super_gradients.training.models.pose_estimation_models.yolo_nas_pose.yolo_nas_pose_variants import YoloNASPose

    gen = torch.Generator().manual_seed(15)
    torch.manual_seed(3)
    arch = tiny_pose_arch()
    ap = copy.deepcopy(arch)
    m = YoloNASPose(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=5, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    randomize_bn(m, gen)
    sd0 = sd_clone(m)
    x = torch.randn(2, 3, 96, 96, generator=gen)
    m.eval()
    with torch.no_grad():
        decoded, raw = m(x)
    cb = YoloNASPosePostPredictionCallback(pose_confidence_threshold=0.01, nms_iou_threshold=0.6, pre_nms_max_predictions=100, post_nms_max_predictions=20)
    preds = cb((decoded, raw))
    live = {k: v for k, v in sd0.items() if "rbr_reparam" not in k}
    torch.save(dict(arch=arch, sd0=live, x=x, decoded=tuple(t.clone() for t in decoded), raw=tuple(t.clone() if torch.is_tensor(t) else t for t in raw),
                    cb=dict(pose_confidence_threshold=0.01, nms_iou_threshold=0.6, pre_nms_max_predictions=100, post_nms_max_predictions=20),
                    preds=[(r.poses.clone(), r.scores.clone(), r.bboxes_xyxy.clone()) for r in preds],
                    param_names=[k for k, _ in m.named_parameters()], state_keys=list(m.state_dict().keys())),
               os.path.join(HERE, "tiny_yolo_nas_pose.pt"))  # fmt: skip


def golden_tiny_yolo_nas_pose_train():
    """Row L7 end to end: train-mode forward of the SAME tiny YOLO-NAS-POSE (weights of tiny_yolo_nas_pose.pt), the
    reference YoloNASPoseLoss in the shipped COCO recipe configuration, backward: loss, components, raw head outputs,
    updated BatchNorm statistics, gradient sums of every parameter and full gradients of the layers next to the loss."""
    from super_gradients.training.losses.yolo_nas_pose_loss import YoloNASPoseLoss
    from super_gradients.training.models.pose_estimation_models.yolo_nas_pose.yolo_nas_pose_variants import YoloNASPose

    gen = torch.Generator().manual_seed(15)
    torch.manual_seed(3)
    ap = copy.deepcopy(tiny_pose_arch())
    m = YoloNASPose(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=5, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    randomize_bn(m, gen)
    sd0 = sd_clone(m)
    prev = torch.load(os.path.join(HERE, "tiny_yolo_nas_pose.pt"), weights_only=False)["sd0"]
    assert all(torch.equal(sd0[k], v) for k, v in prev.items()), "must start from the weights of tiny_yolo_nas_pose.pt"
    g2 = torch.Generator().manual_seed(21)
    x = torch.randn(4, 3, 128, 128, generator=g2)
    J = 5
    rows = [(0, 20.0, 24.0, 84.0, 100.0, 0), (0, 60.0, 30.0, 120.0, 90.0, 0), (1, 10.0, 40.0, 70.0, 120.0, 1), (2, 30.0, 20.0, 110.0, 110.0, 0), (3, 48.0, 50.0, 100.0, 118.0, 0)]
    boxes = torch.tensor([[r[0], r[1], r[2], r[3], r[4]] for r in rows])
    crowd = torch.tensor([[float(r[0]), float(r[5])] for r in rows])
    joints = []
    for r in rows:
        xy = torch.rand(J, 2, generator=g2) * torch.tensor([r[3] - r[1], r[4] - r[2]]) + torch.tensor([r[1], r[2]])
        vis = torch.tensor([2.0, 1.0, 0.0, 2.0, 1.0]).roll(int(r[1]) % J)
        joints.append(torch.cat([torch.full((J, 1), float(r[0])), xy, vis[:, None]], 1))
    targets = (boxes, torch.stack(joints), crowd)
    sigmas = [0.026, 0.035, 0.079, 0.072, 0.062]
    kw = dict(classification_loss_weight=1.0, classification_loss_type="focal", regression_iou_loss_type="ciou", iou_loss_weight=2.5, dfl_loss_weight=0.01,
              pose_cls_loss_weight=1.0, pose_reg_loss_weight=34.0, pose_classification_loss_type="focal", rescale_pose_loss_with_assigned_score=True,
              assigner_multiply_by_pose_oks=True)  # fmt: skip
    m.train()
    outs = m(x)
    loss, items = YoloNASPoseLoss(oks_sigmas=sigmas, **kw)(outs, targets)
    loss.backward()
    grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    running = {k: v for k, v in sd_clone(m).items() if "running_" in k}
    gsum = {k: (float(g.double().sum()), float(g.double().norm())) for k, g in grads.items()}
    keep = [k for k in grads if k.startswith("heads.head1") and ("_pred" in k or "pose_convs.1" in k)]
    torch.save(dict(x=x, targets=targets, sigmas=sigmas, kw=kw, loss=loss.detach(), items=items.detach(), raw=tuple(t.detach().clone() for t in outs[1][:4]),
                    running1=running, grads={k: grads[k] for k in keep}, grad_sums=gsum),
               os.path.join(HERE, "tiny_yolo_nas_pose_train.pt"))  # fmt: skip


def golden_state_keys():
    """state_dict keys + shapes of the full-size models (for checkpoint compatibility tests)."""
    from super_gradients.training import models

    out = {}
    for name, nc in [("yolo_nas_s", 80), ("yolo_nas_m", 80), ("yolo_nas_l", 80), ("resnet18_cifar", 10), ("resnet18", 1000), ("resnet50", 1000),
                     ("yolo_nas_pose_n", 17), ("yolo_nas_pose_s", 17), ("yolo_nas_pose_m", 17), ("yolo_nas_pose_l", 17)]:
        torch.manual_seed(0)
        m = models.get(name, num_classes=nc)
        out[name] = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        out[name + "/param_names"] = [k for k, _ in m.named_parameters()]
        if name == "resnet18_cifar":
            # seeded-init fingerprint: used to check that our constructor consumes the RNG identically
            out[name + "/init_sums"] = {k: float(v.double().sum()) for k, v in m.state_dict().items() if v.dtype.is_floating_point}
    torch.save(out, os.path.join(HERE, "state_keys.pt"))


def golden_resnet_cifar_train():
    """config 1: resnet18_cifar, synthetic CIFAR-shape data, bs 64, SGD lr 0.1 m 0.9 wd 1e-4, CE -- the reference's own
    optimizer / loss classes driven step by step (per-step losses are the fixture)."""
    from super_gradients.training import models
    from super_gradients.training.losses.label_smoothing_cross_entropy_loss import CrossEntropyLoss

    torch.manual_seed(0)
    m = models.get("resnet18_cifar", num_classes=10)
    g = torch.Generator().manual_seed(6)
    X = torch.randn(256, 3, 32, 32, generator=g)
    Y = torch.randint(0, 10, (256,), generator=g)
    crit = CrossEntropyLoss()
    decay, no_decay = [], []
    for n, p in m.named_parameters():
        (no_decay if (n.endswith(".bias") or "bn" in n or "shortcut.1" in n) else decay).append(p)
    opt = torch.optim.SGD([{"params": decay, "weight_decay": 1e-4}, {"params": no_decay, "weight_decay": 0.0}], lr=0.1, momentum=0.9)
    losses = []
    m.train()
    for step in range(4):
        xb, yb = X[step * 64 : (step + 1) * 64], Y[step * 64 : (step + 1) * 64]
        out = m(xb)
        loss = crit(out, yb)
        loss = loss[0] if isinstance(loss, tuple) else loss
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    torch.save(dict(losses=losses, data_seed=6), os.path.join(HERE, "resnet18_cifar_train.pt"))


def golden_droppath():
    """Bottleneck / BasicResNetBlock with drop-path (config 4 is specified with droppath_prob 0.05): the reference draws its mask
    inside forward (`x.new_empty((N,1,1,1)).bernoulli_(keep)`); re-seeding and drawing a tensor of the same shape afterwards
    reproduces exactly that mask, which the fixture records as the per-image scale (mask / keep)."""
    from super_gradients.training.models.classification_models.resnet import BasicResNetBlock, Bottleneck

    out = {}
    gen = torch.Generator().manual_seed(12)
    for name, mk, cin, prob in [
        ("bottleneck_s2", lambda p: Bottleneck(16, 8, stride=2, expansion=4, droppath_prob=p), 16, 0.4),
        ("bottleneck_id", lambda p: Bottleneck(32, 8, stride=1, expansion=4, droppath_prob=p), 32, 0.4),
        ("basic_s2", lambda p: BasicResNetBlock(16, 24, stride=2, droppath_prob=p), 16, 0.5),
    ]:
        torch.manual_seed(3)
        mod = mk(prob)
        randomize_bn(mod, gen)
        sd0 = sd_clone(mod)
        x = torch.randn(8, cin, 16, 16, generator=gen, requires_grad=True)
        mod.train()
        torch.manual_seed(77)
        y = mod(x)
        torch.manual_seed(77)
        scale = torch.empty((8, 1, 1, 1)).bernoulli_(1 - prob).div_(1 - prob).reshape(8)
        assert 0 < int((scale == 0).sum()) < 8, "the fixture needs dropped and kept images"
        gy = torch.randn(y.shape, generator=gen)
        y.backward(gy)
        grads = {k: p.grad.clone() for k, p in mod.named_parameters() if p.grad is not None}
        sd1 = sd_clone(mod)
        mod.eval()
        with torch.no_grad():
            y_eval = mod(x)
        out[name] = dict(sd0=sd0, sd1=sd1, x=x.detach(), y=y.detach(), gy=gy, gx=x.grad.clone(), grads=grads, y_eval=y_eval, scale=scale, prob=prob)
    torch.save(out, os.path.join(HERE, "droppath.pt"))


if __name__ == "__main__":
    ref_shim.install()
    which = sys.argv[1:] or ["qarepvgg", "conv_blocks", "loss", "atss", "nms", "yolox_nms", "processing", "detection_metrics", "lr_schedules", "param_groups", "collate_decoding", "pose_nms", "pose", "tiny_yolo_nas", "tiny_yolo_nas_pose", "tiny_yolo_nas_pose_train", "state_keys", "resnet_cifar_train", "other_configs", "port_fidelity"]
    for w in which:
        print("generating", w, flush=True)
        globals()["golden_" + w]()
    print("done")
