"""Host-side logic on CPU: registries / factories / arch params, state-dict compatibility with the reference, target
padding, LR / EMA schedules, flat parameter buffers and the world-size-2 gradient all-reduce (gloo)."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_registry_and_factory_contract():
    from super_gradients_b200.common.factories import DetectionModulesFactory, UnknownTypeException
    from super_gradients_b200.common.registry import ALL_DETECTION_MODULES, ARCHITECTURES, LOSSES, register_model
    from super_gradients_b200.training import models  # noqa: F401  (populates the registries)

    for name in ("yolo_nas_s", "yolo_nas_m", "yolo_nas_l", "resnet18", "resnet18_cifar", "resnet50"):
        assert name in ARCHITECTURES
    for name in ("NStageBackbone", "YoloNASStem", "YoloNASStage", "YoloNASUpStage", "YoloNASDownStage", "YoloNASPANNeckWithC2", "NDFLHeads", "YoloNASDFLHead", "SPP"):
        assert name in ALL_DETECTION_MODULES
    assert "PPYoloELoss" in LOSSES and "ppyoloe_loss" in LOSSES
    with pytest.raises(Exception):  # re-registering a different class under an existing name raises (registry.py:36-41)
        register_model("yolo_nas_s")(type("Other", (), {}))
    f = DetectionModulesFactory()
    assert f.insert_module_param("SPP", "in_channels", 8) == {"SPP": {"in_channels": 8}}
    with pytest.raises(UnknownTypeException):
        f.get({"NoSuchModule": {}})


@pytest.mark.parametrize("name,nc", [("yolo_nas_s", 80), ("yolo_nas_m", 80), ("yolo_nas_l", 80), ("resnet18_cifar", 10), ("resnet18", 1000), ("resnet50", 1000),
                                     ("yolo_nas_pose_n", 17), ("yolo_nas_pose_s", 17), ("yolo_nas_pose_m", 17), ("yolo_nas_pose_l", 17)])  # fmt: skip
def test_state_dict_keys_match_reference(golden, name, nc):
    """Reference checkpoints must load unchanged (SURVEY.md section 5): same keys, shapes and parameter order."""
    from super_gradients_b200.training import models

    g = golden("state_keys")
    torch.manual_seed(0)
    m = models.get(name, num_classes=nc)
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == g[name]
    assert [k for k, _ in m.named_parameters()] == g[name + "/param_names"]
    if name == "resnet18_cifar":  # identical RNG consumption => identical seeded initialisation
        for k, v in m.state_dict().items():
            if v.dtype.is_floating_point:
                assert abs(float(v.double().sum()) - g[name + "/init_sums"][k]) < 1e-9, k


def test_yolo_nas_s_live_parameter_count():
    from super_gradients_b200.training import models
    from super_gradients_b200.training.flat_state import FlatState

    m = models.get("yolo_nas_s", num_classes=80)
    fs = FlatState(m, zero_wd_on_bias_and_bn=True)
    total = sum(p.numel() for p in m.parameters())
    assert total == 19_053_888
    assert abs(fs.n_live - 12.88e6) < 0.01e6  # SURVEY.md D7
    # parameters are views of the flat buffer, decay group first
    name, p = fs.order[0]
    assert p.data_ptr() == fs.params.data_ptr() and p.main_grad.data_ptr() == fs.grads.data_ptr()
    assert all(not n.endswith(".bias") for n, _ in fs.order[:10])
    assert m.backbone.stem.conv.branch_3x3.bn.running_mean.data_ptr() >= fs.buffers.data_ptr()


def test_pad_targets_matches_oracle():
    from oracle import sg_oracle as O
    from super_gradients_b200.training.losses import pad_targets_host

    t = torch.tensor([[2, 1, 30.0, 28.0, 24.0, 20.0], [0, 3, 40.0, 44.0, 18.0, 30.0], [2, 0, 20.0, 36.0, 30.0, 22.0], [0, 2, 0.0, 0.0, 0.0, 0.0]])
    gc, gb, pm = O.pad_targets(t, 3, n_max=4)
    b, l, v = pad_targets_host(t, 3, 4)
    torch.testing.assert_close(b, gb)
    assert torch.equal(l.long(), gc.squeeze(-1)) and torch.equal(v.float(), pm.squeeze(-1))
    b, l, v = pad_targets_host(torch.zeros(0, 6), 2, 1)
    assert b.shape == (2, 1, 4) and int(v.sum()) == 0


def test_schedules_match_reference_formulas():
    from super_gradients_b200.training.sg_trainer import cosine_lr, ema_decay

    # CosineLRScheduler.compute_learning_rate (callbacks.py:506-511)
    for step, total, lr0, r in [(0, 100, 0.1, 0.01), (37, 100, 0.1, 0.01), (100, 100, 2e-4, 0.1)]:
        ref = 0.5 * lr0 * (1.0 + math.cos(step / (total + 1) * math.pi))
        ref = ref * (1 - r) + lr0 * r
        assert abs(cosine_lr(step, total, lr0, r) - ref) < 1e-12
    assert ema_decay("threshold", 0.9997, 5, 100) == min(0.9997, 6 / 15)
    assert ema_decay("constant", 0.99, 5, 100) == 0.99
    assert abs(ema_decay("exp", 0.9999, 50, 100, 15.0) - 0.9999 * (1 - math.exp(-7.5))) < 1e-12


_DDP_SCRIPT = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from super_gradients_b200.training.flat_state import FlatState
dist.init_process_group("gloo", init_method="env://")
rank, world = dist.get_rank(), dist.get_world_size()
torch.manual_seed(0)
net = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 3), torch.nn.BatchNorm2d(4), torch.nn.Conv2d(4, 2, 1))
fs = FlatState(net, zero_wd_on_bias_and_bn=True)
x = torch.full((2, 3, 5, 5), float(rank + 1))
net(x).sum().backward()
for _, p in fs.order:           # plain-autograd gradients are folded into the flat buffer
    p.main_grad.add_(p.grad); p.grad = None
local = fs.grads.clone()
fs.all_reduce_grads(world)      # ONE flat all-reduce of the live gradients
gathered = [torch.zeros_like(local) for _ in range(world)]
dist.all_gather(gathered, local)
assert torch.allclose(fs.grads, sum(gathered)), "flat all-reduce mismatch"
assert fs.n_decay == 4 * 3 * 9 + 2 * 4 and fs.n_live == fs.n_decay + 4 + 4 + 4 + 2
print("rank", rank, "ok")
"""


def test_flat_gradient_allreduce_world2_gloo(tmp_path):
    script = tmp_path / "ddp.py"
    script.write_text(_DDP_SCRIPT)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", "29511", str(script), ROOT],
        capture_output=True, text=True, timeout=240, env=env,
    )  # fmt: skip
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("ok") == 2


def test_step_arena_hands_out_zeroed_non_overlapping_scratch():
    """K.StepArena: the first bracketed step measures demand (plain torch.zeros), later steps sub-allocate 256-byte
    aligned views of one buffer that begin_step() clears; overflow and out-of-step requests fall back to torch.zeros."""
    import torch

    from super_gradients_b200 import kernels as K

    a = K.StepArena()
    assert not a.active and a.zeros((3,), torch.float32, "cpu").sum() == 0  # outside a step: plain tensor
    shapes = [((8, 2, 48), torch.float64), ((32, 3, 3, 32), torch.float32), ((5,), torch.float32), ((3, 96), torch.float64)]
    a.begin_step("cpu")  # step 1: nothing allocated yet, demand is recorded
    first = [a.zeros(s, d, "cpu") for s, d in shapes]
    a.end_step()
    assert a.buf is None and a.need >= sum(t.numel() * t.element_size() for t in first)
    for rep in range(3):
        a.begin_step("cpu")
        assert a.buf is not None
        ts = [a.zeros(s, d, "cpu") for s, d in shapes]
        base = a.buf.data_ptr()
        spans = []
        for t, (s, d) in zip(ts, shapes):
            assert tuple(t.shape) == s and t.dtype == d and float(t.abs().sum()) == 0.0
            off = t.data_ptr() - base
            assert 0 <= off and off % K.StepArena.ALIGN == 0 and off + t.numel() * t.element_size() <= a.buf.numel()
            spans.append((off, off + t.numel() * t.element_size()))
            t.fill_(rep + 1.0)  # dirty it: the next begin_step must clear exactly what this step used
        spans.sort()
        assert all(e0 <= s1 for (_, e0), (s1, _) in zip(spans, spans[1:])), "views overlap"
        huge = a.zeros((a.buf.numel(),), torch.float32, "cpu")  # does not fit: plain tensor, not a view of the arena
        assert not (base <= huge.data_ptr() < base + a.buf.numel())
        a.end_step()
        assert a.high == a.off


def test_tiny_yolo_nas_pose_mirror_has_reference_state_dict(golden):
    """The YoloNASPose mirror built from the fixture's arch has the reference model's state-dict keys, shapes and parameter
    order, and loads the reference state dict (dead rbr_reparam placeholders aside)."""
    import copy

    from super_gradients_b200.training.models.pose_estimation_models import YoloNASPose

    g = golden("tiny_yolo_nas_pose")
    ap = copy.deepcopy(g["arch"])
    m = YoloNASPose(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=5, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    assert list(m.state_dict().keys()) == g["state_keys"]
    assert [k for k, _ in m.named_parameters()] == g["param_names"]
    missing, unexpected = m.load_state_dict(g["sd0"], strict=False)
    assert not unexpected and all("rbr_reparam" in k for k in missing)
    for k, v in g["sd0"].items():
        assert tuple(m.state_dict()[k].shape) == tuple(v.shape), k
    with pytest.raises(Exception):  # no CPU execution path: the product raises instead of falling back
        m.eval()(g["x"])


def test_no_undefined_names_in_any_python_file():
    """No linter ships in the image; tools/undefined_names.py is the stand-in (names read but bound nowhere in the file).  It
    matters most for bench.py / __graft_entry__.py / the GPU tests, whose code paths cannot execute on the CPU box."""
    files = []
    for top in ("bench.py", "__graft_entry__.py"):
        files.append(os.path.join(ROOT, top))
    for sub in ("super_gradients_b200", "tests", "tools", "oracle"):
        for d, _, names in os.walk(os.path.join(ROOT, sub)):
            files += [os.path.join(d, n) for n in names if n.endswith(".py")]
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "undefined_names.py"), *files], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout


@pytest.mark.parametrize("case", ["yolo_nas_recipe", "pose_recipe_like", "resnet50_like", "cifar_like", "epoch_warmup_given_start_step", "cosine_cooldown"])
def test_lr_schedule_reproduces_the_reference_callbacks(golden, case):
    """The LR in the optimizer at every step == traces recorded by driving the reference's LinearBatchLRWarmup / LinearEpochLRWarmup /
    CosineLRScheduler / StepLRScheduler in the order of its training loop (tests/golden/make_goldens.py::golden_lr_schedules),
    including their quirks (cosine values apply from the next step, step milestones from the next epoch, lr_warmup_steps capped
    at the loader length for the warm-up but not for the scheduler's start)."""
    from super_gradients_b200.training.sg_trainer import DEFAULT_TRAINING_PARAMS, lr_schedule

    g = golden("lr_schedules")[case]
    tp = {**DEFAULT_TRAINING_PARAMS, **{k: v for k, v in g["params"].items() if k in DEFAULT_TRAINING_PARAMS}}
    mine = lr_schedule(tp, g["loader_len"])
    assert len(mine) == len(g["lrs"])
    np.testing.assert_allclose(mine, g["lrs"], rtol=1e-12, atol=0)


@pytest.mark.parametrize("name", ["tiny_yolo_nas", "tiny_yolo_nas_pose", "resnet18_cifar"])
def test_zero_weight_decay_groups_match_reference(golden, name):
    """FlatState's decay / no-decay split == the reference's separate_zero_wd_params_groups_for_optimizer on the same architecture
    (the never-used rbr_reparam placeholders aside: they receive no gradient, so no optimizer ever touches them)."""
    import copy

    from super_gradients_b200.training import models
    from super_gradients_b200.training.flat_state import FlatState
    from super_gradients_b200.training.models.detection_models.yolo_nas import YoloNAS
    from super_gradients_b200.training.models.pose_estimation_models import YoloNASPose

    g = golden("param_groups")[name]
    if name == "resnet18_cifar":
        m = models.get("resnet18_cifar", num_classes=10)
    elif name == "tiny_yolo_nas":
        ap = copy.deepcopy(golden("tiny_yolo_nas")["arch"])
        m = YoloNAS(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=4, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    else:
        ap = copy.deepcopy(golden("tiny_yolo_nas_pose")["arch"])
        m = YoloNASPose(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=5, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    fs = FlatState(m, zero_wd_on_bias_and_bn=True)
    decay = [n for n, _ in fs.order if fs.offsets[n][0] < fs.n_decay]
    no_decay = [n for n, _ in fs.order if fs.offsets[n][0] >= fs.n_decay]
    live = lambda names: [n for n in names if "rbr_reparam" not in n]  # noqa: E731
    # membership is the contract (which parameters decay); the ORDER inside the flat buffer is a layout choice -- FlatState moves the
    # BatchNorm parameters of layers that share one GEMM next to each other (sgb_adjacent_tensors), everything else keeps the
    # reference's order
    assert sorted(decay) == sorted(live(g["decay"])) and sorted(no_decay) == sorted(live(g["no_decay"]))
    assert decay == live(g["decay"])  # no adjacency request touches a decaying parameter
    moved = [n for n in no_decay if ".conv2.bn." in n or ".reg_convs.0.seq.bn." in n]
    rest = [n for n in no_decay if n not in moved]
    assert rest == [n for n in live(g["no_decay"]) if n not in moved]
    assert any(n.endswith("alpha") for n in decay) or name == "resnet18_cifar"


def test_replace_input_channels_and_checkpoint_num_classes(tmp_path):
    """models.get(..., checkpoint_path, checkpoint_num_classes, num_input_channels) (model_factory.py:227-254): the checkpoint's head
    is built and loaded first, then replace_head / replace_input_channels; the filter surgery keeps the old channels
    (weight_replacement_utils.py:27-65)."""
    from super_gradients_b200.modules.weight_replacement_utils import replace_conv2d_input_channels
    from super_gradients_b200.training import models

    conv = torch.nn.Conv2d(3, 8, 3, padding=1, bias=True)
    wide, narrow = replace_conv2d_input_channels(conv, 5), replace_conv2d_input_channels(conv, 2)
    assert wide.weight.shape == (8, 5, 3, 3) and torch.equal(wide.weight[:, :3], conv.weight) and wide.weight[:, 3:].abs().sum() > 0
    assert torch.equal(narrow.weight, conv.weight[:, :2]) and narrow.padding == conv.padding and narrow.bias is not None
    assert replace_conv2d_input_channels(conv, 4, fn=lambda c, n: torch.nn.Conv2d(n, c.out_channels, 1)).kernel_size == (1, 1)
    with pytest.raises(ValueError):
        replace_conv2d_input_channels(torch.nn.Conv2d(4, 8, 3, groups=2), 3)

    torch.manual_seed(0)
    r = models.get("resnet18", num_classes=10)
    w0 = r.conv1.weight.detach().clone()
    torch.save({"net": r.state_dict()}, tmp_path / "r18.pth")
    r2 = models.get("resnet18", num_classes=4, checkpoint_path=str(tmp_path / "r18.pth"), checkpoint_num_classes=10, num_input_channels=1)
    assert r2.get_input_channels() == 1 and torch.equal(r2.conv1.weight, w0[:, :1]) and r2.linear.out_features == 4
    assert torch.equal(r2.layer1[0].conv1.weight, r.layer1[0].conv1.weight)  # the rest of the checkpoint is in place

    torch.manual_seed(0)
    y = models.get("yolo_nas_s", num_classes=80, num_input_channels=4)
    assert y.get_input_channels() == 4 == y.in_channels and y.backbone.stem.conv.in_channels == 4
    assert {k: tuple(v.shape) for k, v in y.state_dict().items() if "stem" in k and "3x3.conv.weight" in k}.popitem()[1][1] == 4


def _collate_samples(seed):
    gen = np.random.RandomState(seed)
    return [(gen.rand(16, 24, 3).astype(np.float32), gen.rand(n, 5).astype(np.float32) * 10) for n in (3, 0, 2)]


def _decoding_inputs(seed):
    """Head outputs of 3 images x 400 anchors: boxes, 80 class scores, and the pose head's confidence, 17 joints' coordinates and scores."""
    gen = torch.Generator().manual_seed(seed)
    boxes, scores = torch.rand(3, 400, 4, generator=gen), torch.rand(3, 400, 80, generator=gen)
    return boxes, scores, torch.rand(3, 400, 1, generator=gen), torch.rand(3, 400, 17, 2, generator=gen), torch.rand(3, 400, 17, generator=gen)


def _pose_samples(seed):
    import types

    gen = np.random.RandomState(seed)
    samples = []
    for n in (2, 0, 3):
        samples.append(types.SimpleNamespace(image=gen.randint(0, 255, (32, 48, 3)).astype(np.uint8), mask=np.ones((32, 48), np.float32), bboxes_xywh=gen.rand(n, 4).astype(np.float32) * 20,
                                             joints=gen.rand(n, 5, 3).astype(np.float32) * 30, is_crowd=(gen.rand(n) < 0.5) if n != 3 else None, additional_samples=[1]))  # fmt: skip
    return samples


def test_collate_functions_produce_the_reference_target_formats(golden):
    """DetectionCollateFN (detection_collate_fn.py:10-49) and YoloNASPoseCollateFN / flat_collate_tensors_with_batch_index
    (yolo_nas_pose_collate_fn.py:14-123): the producers of the flat target tensors rows L1 / L7 consume -- equal to the reference's
    outputs (tests/golden/collate_decoding.pt) and accepted by the product's target padding."""
    from super_gradients_b200.common.registry import COLLATE_FUNCTIONS
    from super_gradients_b200.training.datasets.pose_estimation_datasets import YoloNASPoseCollateFN, flat_collate_tensors_with_batch_index, undo_flat_collate_tensors_with_batch_index
    from super_gradients_b200.training.losses.ppyolo_loss import pad_targets_host
    from super_gradients_b200.training.losses.yolo_nas_pose_loss import pad_pose_targets_host
    from super_gradients_b200.training.utils.collate_fn import DatasetItemsException, DetectionCollateFN

    data = _collate_samples(0)
    images, targets = DetectionCollateFN()(data)
    assert images.shape == (3, 3, 16, 24) and images.dtype == torch.float32 and targets.shape == (5, 6) and targets[:, 0].tolist() == [0, 0, 0, 2, 2]
    assert torch.equal(targets[3:, 1:], torch.from_numpy(data[2][1])) and COLLATE_FUNCTIONS["DetectionCollateFN"] is DetectionCollateFN
    boxes, labels, valid = pad_targets_host(targets, 3, 4)
    assert valid.sum(1).tolist() == [3, 0, 2]
    with pytest.raises(DatasetItemsException):
        DetectionCollateFN()([(1, 2, 3)])
    chw = DetectionCollateFN._format_images([np.zeros((3, 8, 8), np.float32)] * 2)
    assert chw.shape == (2, 3, 8, 8)

    flat = flat_collate_tensors_with_batch_index([torch.ones(2, 4, 3), torch.zeros(0, 4, 3), torch.ones(1, 4, 3) * 5])
    assert flat.shape == (3, 4, 4) and flat[:, 0, 0].tolist() == [0, 0, 2]
    parts = undo_flat_collate_tensors_with_batch_index(flat, 3)
    assert [p.shape[0] for p in parts] == [2, 0, 1] and torch.equal(parts[2], torch.ones(1, 4, 3) * 5)
    imgs, (b, j, c), extras = YoloNASPoseCollateFN()(_pose_samples(1))
    assert imgs.shape == (3, 3, 32, 48) and b.shape == (5, 5) and j.shape == (5, 5, 4) and c.shape == (5, 2) and c.dtype == torch.int64
    assert extras["gt_samples"][0].image is None and extras["gt_samples"][0].additional_samples is None
    ref_in = _pose_samples(1)
    assert np.allclose(b[0, 1:].numpy(), np.r_[ref_in[0].bboxes_xywh[0, :2], ref_in[0].bboxes_xywh[0, :2] + ref_in[0].bboxes_xywh[0, 2:]])
    padded = pad_pose_targets_host((b.float(), j.float(), c), 3, 4)
    assert padded[-1].sum(1).tolist() == [2, 0, 3]

    # against the reference's outputs on the same inputs
    g = golden("collate_decoding")
    pi, pt = DetectionCollateFN()(_collate_samples(0))
    assert torch.equal(g["det_images"], pi) and torch.equal(g["det_targets"], pt) and g["det_targets"].dtype == pt.dtype
    pa, (pb, pj, pc), _ = YoloNASPoseCollateFN()(_pose_samples(1))
    ra, (rb, rj, rc) = g["pose_images"], g["pose_targets"]
    assert torch.equal(ra, pa) and torch.equal(rb, pb) and torch.equal(rj, pj) and torch.equal(rc, pc) and rb.dtype == pb.dtype and rc.dtype == pc.dtype


def test_export_decoding_modules_match_the_reference(golden):
    """Row N4: YoloNASDecodingModule (yolo_nas_variants.py:53-72) and YoloNASPoseDecodingModule (yolo_nas_pose_variants.py:54-90),
    the pre-NMS top-k of the export graph, against the reference's modules' outputs on the same random head outputs
    (tests/golden/collate_decoding.pt)."""
    from super_gradients_b200.training.models.detection_models.yolo_nas import YoloNASDecodingModule
    from super_gradients_b200.training.models.pose_estimation_models.yolo_nas_pose.yolo_nas_pose_variants import YoloNASPoseDecodingModule

    gen = torch.Generator().manual_seed(0)
    boxes, scores = torch.rand(2, 50, 4, generator=gen), torch.rand(2, 50, 7, generator=gen)
    b, s = YoloNASDecodingModule(10)(((boxes, scores), None))
    assert b.shape == (2, 10, 4) and s.shape == (2, 10, 7) and (s.max(-1).values.diff(dim=1) <= 0).all()
    conf, coords, js = torch.rand(2, 50, 1, generator=gen), torch.rand(2, 50, 5, 2, generator=gen), torch.rand(2, 50, 5, generator=gen)
    pb, pc, pj = YoloNASPoseDecodingModule(8)(((boxes, conf, coords, js), None))
    assert pb.shape == (2, 8, 4) and pc.shape == (2, 8, 1) and pj.shape == (2, 8, 5, 3) and (pc[:, :, 0].diff(dim=1) <= 0).all()
    k = int(conf[0, :, 0].argmax())
    assert torch.equal(pb[0, 0], boxes[0, k]) and torch.equal(pj[0, 0, :, :2], coords[0, k]) and torch.equal(pj[0, 0, :, 2], js[0, k])
    g = golden("collate_decoding")
    boxes, scores, conf, coords, js = _decoding_inputs(0)
    det, pose = YoloNASDecodingModule(100)(((boxes, scores), None)), YoloNASPoseDecodingModule(64)(((boxes, conf, coords, js), None))
    assert len(det) == len(g["det_decoded"]) and len(pose) == len(g["pose_decoded"])
    for a, b in zip((*g["det_decoded"], *g["pose_decoded"]), (*det, *pose)):
        assert torch.equal(a, b)


def test_flat_state_adjacency_requests_and_checkpoint_remap(tmp_path):
    """FlatState lays tensors that a module asks for (`sgb_adjacent_tensors`) back to back -- parameters, their gradient slots and the
    BatchNorm statistics -- without changing the decay / no-decay membership or anything else's relative order, ignores requests it
    cannot honour (members of different groups), and an optimizer state saved under another layout is restored by name."""
    import torch
    from torch import nn

    from super_gradients_b200.training.flat_state import FlatState, _apply_adjacency

    class Pair(nn.Module):
        def __init__(self):
            super().__init__()
            self.a, self.mid, self.b = nn.BatchNorm2d(8), nn.Conv2d(8, 8, 1), nn.BatchNorm2d(8)

        def sgb_adjacent_tensors(self):
            return [[self.a.weight, self.b.weight], [self.a.bias, self.b.bias], [self.a.running_mean, self.b.running_mean],
                    [self.a.running_var, self.b.running_var], [self.mid.weight, self.a.weight]]  # the last one mixes decay groups: ignored

    def follows(x, y):
        return y.data_ptr() == x.data_ptr() + x.numel() * x.element_size()

    torch.manual_seed(0)
    m = Pair()
    ref = {k: v.clone() for k, v in m.state_dict().items()}
    fs = FlatState(m)
    assert follows(m.a.weight, m.b.weight) and follows(m.a.bias, m.b.bias) and follows(m.a.running_mean, m.b.running_mean) and follows(m.a.running_var, m.b.running_var)
    assert follows(m.a.weight.main_grad, m.b.weight.main_grad) and follows(m.a.bias.main_grad, m.b.bias.main_grad)
    for k, v in m.state_dict().items():  # values untouched by the re-pointing
        assert torch.equal(v, ref[k]), k
    names = [n for n, _ in fs.order]
    assert names[: names.index("a.weight")] == ["mid.weight"]  # the decaying filter first, the no-decay group after it
    assert names.index("b.weight") == names.index("a.weight") + 1 and names.index("b.bias") == names.index("a.bias") + 1
    assert sorted(names) == sorted(n for n, _ in m.named_parameters())
    # the helper alone: groups with a missing member are skipped, followers keep group order
    t = [torch.zeros(1) for _ in range(5)]
    items = list(zip("abcde", t))
    assert [n for n, _ in _apply_adjacency(items, [[t[1], t[4], t[3]], [t[0], torch.zeros(1)]])] == ["a", "b", "e", "d", "c"]
    # optimizer state saved under another flat layout (e.g. a checkpoint written before an adjacency request existed): restored by name
    from types import SimpleNamespace

    from super_gradients_b200.training.sg_trainer import Trainer

    saved_order = sorted(names)  # some other order of the same parameters
    sizes = {n: p.numel() for n, p in m.named_parameters()}
    saved_state = torch.cat([torch.full((sizes[n],), float(i)) for i, n in enumerate(saved_order)])
    step = SimpleNamespace(opt_name="SGD", flat=fs, state=[torch.zeros(fs.n_live)], opt_steps=0, ema_on=False)
    Trainer._restore_training_state(SimpleNamespace(step=step), {"optimizer_state_dict": {"name": "SGD", "flat_order": saved_order, "state": [saved_state], "opt_steps": 7}})
    assert step.opt_steps == 7
    for i, n in enumerate(saved_order):
        off, k = fs.offsets[n]
        assert bool((step.state[0][off : off + k] == float(i)).all()), n
    with pytest.raises(ValueError, match="optimizer"):
        Trainer._restore_training_state(SimpleNamespace(step=step), {"optimizer_state_dict": {"name": "SGD", "flat_order": saved_order[:-1], "state": [saved_state], "opt_steps": 7}})
