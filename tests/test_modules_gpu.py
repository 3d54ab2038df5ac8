"""GPU parity of the drop-in modules (reference constructors / state-dict keys, sm_100a forward+backward) against
fixtures produced by the UNMODIFIED reference in fp32 on CPU (tests/golden/*.pt, see make_goldens.py).

Two comparisons per module:
 (1) TIGHT -- against the CPU oracle in bf16-emulation mode (oracle.sg_oracle.bf16_emulation: the same fp32 arithmetic
     as the pinned oracle, with values rounded to bf16 exactly where the product stores bf16).  This isolates kernel
     errors from the precision choice: relative L2 <= 5e-3 (single block) / 1e-2 (whole graph: 1-ulp flips of bf16
     outputs) for activations, <= 3e-2 for gradients.
 (2) LOOSE -- against the fp32 fixtures produced by the unmodified reference.  The gap is the bf16 precision of the
     product path itself (rounding of operands amplified by the BatchNorm backward); the emulated oracle shows the same
     gap on CPU, e.g. 3.8e-2 for the input gradient of a single QARepVGG block.
(Kernel-level accumulator parity at 1e-3 is asserted in test_kernels_gpu.py with identical bf16 operands.)
"""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"


def l2rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def load_sd(module, sd):
    missing, unexpected = module.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all("rbr_reparam" in k for k in missing), missing


@pytest.mark.parametrize("case", ["s1_res", "s2"])
def test_qarepvgg_block(golden, case):
    from super_gradients_b200.modules import QARepVGGBlock

    g = golden("qarepvgg")[case]
    blk = QARepVGGBlock(g["cin"], g["cout"], stride=g["stride"], use_residual_connection=g["residual"])
    for m in blk.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eps, m.momentum = 1e-3, 0.03
    load_sd(blk, g["sd0"])
    blk.to(DEV).train()
    x = g["x"].to(DEV).bfloat16().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = blk(x)
    y.backward(g["gy"].to(DEV).bfloat16())
    # (1) tight: bf16-emulating oracle
    from oracle import sg_oracle as O

    with O.bf16_emulation():
        pe = {k: v.clone() for k, v in g["sd0"].items()}
        for k in g["grads"]:
            pe[k].requires_grad_(True)
        xe = g["x"].clone().requires_grad_(True)
        ye = O.qarepvgg_forward(O.q(xe), pe, "", g["stride"], g["residual"], "relu", True, 1e-3, 0.03)
        ye.backward(g["gy"].bfloat16().float())
    assert l2rel(y, ye) < 5e-3
    assert l2rel(x.grad, xe.grad) < 2e-2
    params = dict(blk.named_parameters())
    for k, v in g["grads"].items():
        if v.abs().max() < 1e-4 * max(1.0, float(g["gy"].abs().max())):
            # branch_3x3.bn.bias / branch_1x1.bias: exactly zero in exact arithmetic (post_bn removes constants);
            # the reference's value is fp32 round-off noise
            assert float(params[k].grad.abs().max()) <= 1e-3
            continue
        assert l2rel(params[k].grad, pe[k].grad) < 2e-2, k
    # (2) loose: fp32 reference fixture
    assert l2rel(y, g["y"]) < 1e-2
    assert l2rel(x.grad, g["gx"]) < 8e-2
    for k, v in g["grads"].items():
        if v.abs().max() >= 1e-4 * max(1.0, float(g["gy"].abs().max())):
            assert l2rel(params[k].grad, v) < 8e-2, k
    for k, v in g["sd1"].items():
        if "running" in k:
            assert l2rel(blk.state_dict()[k], v) < 1e-2, k
    assert "rbr_reparam.weight" in blk.state_dict() and dict(blk.named_parameters())["rbr_reparam.weight"].grad is None
    # eval (running stats), partial and full fusion
    blk2 = QARepVGGBlock(g["cin"], g["cout"], stride=g["stride"], use_residual_connection=g["residual"])
    for m in blk2.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eps, m.momentum = 1e-3, 0.03
    blk2.load_state_dict(g["sd1"])
    blk2.to(DEV).eval()
    xe = g["x"].to(DEV)
    from super_gradients_b200 import functional as SF

    with torch.no_grad():
        assert l2rel(blk2(SF.to_nhwc(xe)), g["y_eval"]) < 1e-2
        f = copy.deepcopy(blk2)
        f.partial_fusion()
        assert l2rel(f(SF.to_nhwc(xe)), g["y_partial"]) < 1e-2
        f.full_fusion()
        assert l2rel(f(SF.to_nhwc(xe)), g["y_full"]) < 1e-2
        assert "post_bn.weight" not in f.state_dict()


def test_patch_stem_matches_the_two_convolution_path(monkeypatch):
    """The YOLO-NAS stem (QARepVGG 3 -> K, 3 x 3 stride 2 + 1 x 1 stride 2) as ONE 1 x 1 GEMM over gathered patches
    (functional._QARepVGGStem, sgb_stem_patches_f32): same output (1 bf16 ulp: identical products, different fp32 summation order),
    same parameter gradients and running statistics as the two-convolution path, and the oracle's block in bf16-emulation mode."""
    from oracle import sg_oracle as O
    from super_gradients_b200 import functional as SF
    from super_gradients_b200 import lib
    from super_gradients_b200.modules import QARepVGGBlock

    def run(patches, shape):
        monkeypatch.setattr(SF, "STEM_PATCHES", [patches])
        torch.manual_seed(3)
        blk = QARepVGGBlock(3, 48, stride=2, use_residual_connection=False)
        with torch.no_grad():
            for p in blk.parameters():
                p.add_(0.05 * torch.randn_like(p))
        sd0 = {k: v.clone() for k, v in blk.state_dict().items()}
        blk = blk.to(DEV).train()
        x = torch.randn(*shape).bfloat16().float()
        assert SF.stem_patches_supported(blk, x.to(DEV)) == patches
        y = blk(x.to(DEV))
        gy = torch.linspace(-1, 1, y.numel()).reshape(y.shape).bfloat16()
        y.backward(gy.to(DEV))
        torch.cuda.synchronize()
        return x, sd0, gy, y.detach().float().cpu(), {k: p.grad.cpu().clone() for k, p in blk.named_parameters() if p.grad is not None}, {k: v.cpu().clone() for k, v in blk.state_dict().items() if "running" in k}

    for shape in ((2, 3, 64, 96), (3, 3, 70, 54)):  # even and odd sizes (right / bottom border taps)
        x, sd0, gy, y0, g0, r0 = run(False, shape)
        _, _, _, y1, g1, r1 = run(True, shape)
        assert ((y1 - y0).abs() <= y0.abs() * 2**-7 + 1e-3).all(), float((y1 - y0).abs().max())
        assert set(g0) == set(g1)
        for k in g0:
            assert l2rel(g1[k], g0[k]) < 1e-2 or float(g0[k].abs().max()) < 1e-4, (k, l2rel(g1[k], g0[k]))
        for k in r0:
            assert l2rel(r1[k], r0[k]) < 1e-4, k
        with O.bf16_emulation():
            pe = {k: v.clone() for k, v in sd0.items()}
            ye = O.qarepvgg_forward(O.q(x), pe, "", 2, False, "relu", True, 1e-5, 0.1)
        assert l2rel(y1, ye) < 5e-3, l2rel(y1, ye)
    # the patch gather itself, against unfold
    xs = torch.randn(2, 3, 37, 41, device=DEV)
    from super_gradients_b200 import kernels as K

    got = K.stem_patches(xs, 3, 2, 1, 32).float()
    cols = torch.nn.functional.unfold(xs, 3, padding=1, stride=2).reshape(2, 3, 9, 19, 21).permute(0, 2, 1, 3, 4).reshape(2, 27, 19, 21)
    assert torch.equal(got[:, :27], cols.bfloat16().float()) and float(got[:, 27:].abs().max()) == 0.0
    assert lib.load() is not None


def test_resnet_stem_on_patches_matches_the_direct_convolution(monkeypatch):
    """ResNet's 7 x 7 / stride-2 first layer as ONE 1 x 1 GEMM over gathered patches (functional._ConvBnActStem; 147 patch channels
    padded to 160): same output, weight / BatchNorm gradients and running statistics as the direct convolution over the 16-channel-
    padded image (the mma.sync path it replaces), and as fp32 torch on the same bf16-rounded operands; the 7 x 7 gather against unfold."""
    import torch.nn.functional as F

    from super_gradients_b200 import functional as SF
    from super_gradients_b200 import kernels as K
    from super_gradients_b200.training import models

    def run(patches, shape):
        monkeypatch.setattr(SF, "STEM_PATCHES", [patches])
        torch.manual_seed(5)
        net = models.get("resnet18", num_classes=10)
        sd0 = {k: v.clone() for k, v in net.state_dict().items()}
        net = net.to(DEV).train()
        x = torch.randn(*shape).bfloat16().float()
        assert SF.conv_stem_patches_supported(net.conv1, net.bn1, x.to(DEV), True) == patches
        xg = x.to(DEV)
        if patches:
            out = SF.conv_bn_act_stem(xg, net.conv1, net.bn1, act="relu", cache=net._stem_patch_cache)
        else:
            out = net._fused(SF.to_nhwc(xg), net.conv1, net.bn1, "relu", net._stem_cache)
        gy = torch.linspace(-1, 1, out.numel()).reshape(out.shape).bfloat16()
        out.backward(gy.to(DEV))
        torch.cuda.synchronize()
        grads = {k: p.grad.cpu().clone() for k, p in net.named_parameters() if p.grad is not None}
        return x, sd0, gy, out.detach().float().cpu(), grads, {k: v.cpu().clone() for k, v in net.state_dict().items() if k.startswith("bn1.running")}

    for shape in ((2, 3, 64, 96), (3, 3, 70, 54)):
        x, sd0, gy, y0, g0, r0 = run(False, shape)
        _, _, _, y1, g1, r1 = run(True, shape)
        assert ((y1 - y0).abs() <= y0.abs() * 2**-7 + 1e-3).all(), float((y1 - y0).abs().max())
        assert set(g0) == set(g1) == {"conv1.weight", "bn1.weight", "bn1.bias"}
        for k in g0:
            assert l2rel(g1[k], g0[k]) < 1e-2, (k, l2rel(g1[k], g0[k]))
        for k in r0:
            assert l2rel(r1[k], r0[k]) < 1e-4, k
        # fp32 torch on the same bf16 operands
        w = sd0["conv1.weight"].bfloat16().float().requires_grad_(True)
        gam, bet = sd0["bn1.weight"].clone().requires_grad_(True), sd0["bn1.bias"].clone().requires_grad_(True)
        ref = F.relu(F.batch_norm(F.conv2d(x, w, stride=2, padding=3), None, None, gam, bet, True, 0.1, 1e-5))
        ref.backward(gy.float())
        assert l2rel(y1, ref.detach()) < 5e-3, l2rel(y1, ref.detach())
        assert l2rel(g1["conv1.weight"], w.grad) < 2e-2 and l2rel(g1["bn1.weight"], gam.grad) < 1e-2
    xs = torch.randn(2, 3, 37, 41, device=DEV)
    got = K.stem_patches(xs, 7, 2, 3, 160).float()
    cols = F.unfold(xs, 7, padding=3, stride=2).reshape(2, 3, 49, 19, 21).permute(0, 2, 1, 3, 4).reshape(2, 147, 19, 21)
    assert torch.equal(got[:, :147], cols.bfloat16().float()) and float(got[:, 147:].abs().max()) == 0.0


def test_csp_layer_merged_launches_match_the_separate_layers(monkeypatch):
    """On the device: conv1 / conv2 of a CSP layer as ONE GEMM + ONE BatchNorm launch over adjacent parameters with a two-source
    backward (functional._DualConvBnAct, SgbBnDesc.dy2), the bottleneck shortcut's gradient finished in place after cv1's dgrad
    (functional._defer_finish) and the shortcut itself fused into cv2's apply pass (SgbQarepDesc.res) against the same layer with
    every switch off: identical output (per-channel arithmetic, the fused shortcut rounds like the two-pass form), input and parameter
    gradients equal up to the bf16 rounding of one merged dgrad sum; statistics-in-BatchNorm layers included (96 + 96 channels)."""
    from super_gradients_b200 import functional as SF
    from super_gradients_b200.modules import Conv, QARepVGGBlock
    from super_gradients_b200.training.flat_state import FlatState
    from super_gradients_b200.training.models.detection_models.yolo_nas.yolo_stages import YoloNASCSPLayer

    def run(on, cin, hid, shape):
        for name in ("DUAL_CONV", "DEFER_SHORTCUT", "FUSE_SHORTCUT"):
            monkeypatch.setattr(SF, name, [on])
        torch.manual_seed(3)
        net = torch.nn.Sequential(Conv(16, cin, 1, stride=1, activation_type=torch.nn.ReLU), YoloNASCSPLayer(cin, cin, 2, QARepVGGBlock, torch.nn.ReLU, True, True, hidden_channels=hid))
        with torch.no_grad():
            for p in net.parameters():
                p.add_(0.05 * torch.randn_like(p))
        net = net.to(DEV).train()
        flat = FlatState(net)
        assert SF.dual_conv_bn_act_ready(net[1].conv1.conv, net[1].conv1.bn, net[1].conv2.conv, net[1].conv2.bn) == on
        x = torch.randn(*shape).bfloat16().to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        y = net(x)
        gy = torch.linspace(-1, 1, y.numel()).reshape(y.shape).bfloat16().to(DEV)
        y.backward(gy)
        torch.cuda.synchronize()
        return y.detach().float().cpu(), x.grad.float().cpu(), {n: flat.grad_of(n).cpu().clone() for n, _ in flat.order}, flat.buffers.cpu().clone()

    for cin, hid, shape in ((32, 16, (2, 16, 24, 20)), (64, 96, (3, 16, 17, 13))):
        y0, dx0, g0, b0 = run(False, cin, hid, shape)
        y1, dx1, g1, b1 = run(True, cin, hid, shape)
        assert torch.equal(y0, y1), float((y0 - y1).abs().max())
        torch.testing.assert_close(b1, b0, rtol=1e-5, atol=1e-6)
        assert l2rel(dx1, dx0) < 8e-3, l2rel(dx1, dx0)
        scale = max(float(v.norm()) for v in g0.values())
        for k in g0:
            if float(g0[k].norm()) < 1e-4 * scale:
                assert float(g1[k].norm()) < 1e-3 * scale, k
                continue
            assert l2rel(g1[k], g0[k]) < 2e-2, (k, l2rel(g1[k], g0[k]))


def test_backward_reads_a_concat_gradient_slice_in_place():
    """A block whose output feeds a channel concat receives its gradient as a channel SLICE of the concat's gradient buffer.  The
    BatchNorm / QARepVGG backward kernels read that slice in place (SgbBnDesc.dy_pitch, SgbQarepDesc.pitchd) -- round 1 made a
    strided ATen copy per block (31 launches, 0.7 ms of the config-2 step).  Same bits as the dense-gradient path."""
    from super_gradients_b200 import functional as SF
    from super_gradients_b200.modules import Conv, QARepVGGBlock

    torch.manual_seed(5)
    for mk in (lambda: QARepVGGBlock(32, 32, stride=1, use_residual_connection=True), lambda: Conv(32, 32, 3, 1, torch.nn.ReLU)):
        blk = mk().to(DEV).train()
        x0 = torch.randn(2, 32, 20, 20, device=DEV).bfloat16().contiguous(memory_format=torch.channels_last)
        other = torch.randn(2, 16, 20, 20, device=DEV).bfloat16().contiguous(memory_format=torch.channels_last)
        gy = torch.randn(2, 48, 20, 20, device=DEV).bfloat16().contiguous(memory_format=torch.channels_last)
        res = []
        for sliced in (False, True):
            blk.zero_grad(set_to_none=True)
            x = x0.clone().requires_grad_(True)
            y = blk(x)
            if sliced:
                SF.concat([other, y]).backward(gy)
            else:
                y.backward(gy[:, 16:].contiguous(memory_format=torch.channels_last))
            res.append((x.grad.clone(), {k: p.grad.clone() for k, p in blk.named_parameters() if p.grad is not None}))
        assert torch.equal(res[0][0], res[1][0])
        for k in res[0][1]:  # weight gradients are summed with fp32 atomics across pixel splits: equal up to their order
            assert l2rel(res[1][1][k], res[0][1][k]) < 1e-5 or float(res[0][1][k].abs().max()) < 1e-6, (k, l2rel(res[1][1][k], res[0][1][k]))


def _run_block(mod, g, oracle_fn, scale=None):
    from oracle import sg_oracle as O

    load_sd(mod, g["sd0"])
    mod.to(DEV).train()
    if scale is not None:  # drop-path: the block draws its mask from the device RNG; the test injects the reference's recorded one
        mod.drop_path.sample_scale = lambda x: scale.to(DEV) if mod.training else None
    x = g["x"].to(DEV).bfloat16().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = mod(x)
    y.backward(g["gy"].to(DEV).bfloat16())
    params = dict(mod.named_parameters())
    with O.bf16_emulation():
        pe = {k: v.clone() for k, v in g["sd0"].items()}
        for k in g["grads"]:
            pe[k].requires_grad_(True)
        xe = g["x"].clone().requires_grad_(True)
        ye = oracle_fn(O.q(xe), pe)
        ye.backward(g["gy"].bfloat16().float())
    name = type(mod).__name__
    assert l2rel(y, ye) < 5e-3, name
    assert l2rel(x.grad, xe.grad) < 2e-2, name
    for k in g["grads"]:
        assert l2rel(params[k].grad, pe[k].grad) < 3e-2, (name, k)
    for k, v in g["sd1"].items():
        if "running" in k:
            assert l2rel(mod.state_dict()[k], pe[k]) < 1e-3, (name, k)
            assert l2rel(mod.state_dict()[k], v) < 1e-2, (name, k)
        if "num_batches_tracked" in k:
            assert int(mod.state_dict()[k]) == int(v)
    # loose bounds against the fp32 reference fixture
    assert l2rel(y, g["y"]) < 1.5e-2, name
    assert l2rel(x.grad, g["gx"]) < 0.2, name  # max-pool arg-max flips (SPP) make this the loosest block
    mod.eval()
    mod.load_state_dict(g["sd1"])
    with torch.no_grad():
        assert l2rel(mod(x.detach()), g["y_eval"]) < 1.5e-2, name


def test_conv_blocks_bottleneck_spp(golden):
    from oracle import sg_oracle as O
    from super_gradients_b200.modules import Conv, ConvBNReLU
    from super_gradients_b200.training.models.classification_models.resnet import BasicResNetBlock, Bottleneck
    from super_gradients_b200.training.models.detection_models.csp_darknet53 import SPP

    G = golden("conv_blocks")
    _run_block(Conv(16, 24, 3, 2, torch.nn.ReLU), G["conv3x3_s2"], lambda x, p: O.conv_bn_act(x, p, "", 2, 1, "relu", True, 1e-5, 0.1))
    _run_block(Conv(16, 8, 1, 1, torch.nn.ReLU), G["conv1x1"], lambda x, p: O.conv_bn_act(x, p, "", 1, 0, "relu", True, 1e-5, 0.1))
    _run_block(ConvBNReLU(8, 16, kernel_size=3, stride=1, padding=1, bias=False), G["convbnrelu"], lambda x, p: O.conv_bn_act(x, p, "seq.", 1, 1, "relu", True, 1e-5, 0.1))
    _run_block(Bottleneck(16, 8, stride=2, expansion=4), G["bottleneck_s2"], lambda x, p: O.resnet_bottleneck(x, p, "", 2, True, True))
    _run_block(Bottleneck(32, 8, stride=1, expansion=4), G["bottleneck_id"], lambda x, p: O.resnet_bottleneck(x, p, "", 1, False, True))
    _run_block(BasicResNetBlock(16, 24, stride=2), G["basic_s2"], lambda x, p: O.resnet_basic_block(x, p, "", 2, True, True))
    _run_block(SPP(16, 16, (5, 9, 13), torch.nn.ReLU), G["spp"], lambda x, p: O.spp(x, p, "", (5, 9, 13), "relu", True, 1e-5, 0.1))


def _tiny_model(g):
    from super_gradients_b200.training.models.detection_models.yolo_nas import YoloNAS

    ap = copy.deepcopy(g["arch"])
    m = YoloNAS(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=4, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    assert list(m.state_dict().keys()) == g["state_keys"]
    assert [k for k, _ in m.named_parameters()] == g["param_names"]
    load_sd(m, g["sd0"])
    return m.to(DEV)


def test_resnet_blocks_with_drop_path(golden):
    """Config 4 as specified (recipes/imagenet_resnet50.yaml: droppath_prob 0.05): the per-image mask multiply runs inside the
    fused bn + residual + relu kernel and its two backward passes (SgbBnDesc.sample_scale); forward, input gradient, parameter
    gradients and running statistics against the oracle (tight) and the unmodified reference's fixture (loose)."""
    from oracle import sg_oracle as O
    from super_gradients_b200.training.models.classification_models.resnet import BasicResNetBlock, Bottleneck
    from super_gradients_b200.training.utils.regularization_utils import DropPath

    G = golden("droppath")
    for name, mod, fn, args in (
        ("bottleneck_s2", Bottleneck(16, 8, stride=2, expansion=4, droppath_prob=0.4), O.resnet_bottleneck, (2, True)),
        ("bottleneck_id", Bottleneck(32, 8, stride=1, expansion=4, droppath_prob=0.4), O.resnet_bottleneck, (1, False)),
        ("basic_s2", BasicResNetBlock(16, 24, stride=2, droppath_prob=0.5), O.resnet_basic_block, (2, True)),
    ):
        g = G[name]
        _run_block(mod, g, lambda x, p, fn=fn, args=args, g=g: fn(x, p, "", args[0], args[1], True, sample_scale=g["scale"]), scale=g["scale"])
    # the module's own draw: 0 or 1 / keep per image, inactive in eval mode
    dp = DropPath(0.25).to(DEV).train()
    m = dp.sample_scale(torch.zeros(4096, 1, device=DEV))
    vals = m.unique().tolist()
    assert m.shape == (4096,) and len(vals) == 2 and vals[0] == 0.0 and abs(vals[1] - 1 / 0.75) < 1e-6 and 0.2 < float((m == 0).float().mean()) < 0.3
    assert dp.eval().sample_scale(torch.zeros(4, 1, device=DEV)) is None


def test_tiny_yolo_nas_train_step_and_eval(golden):
    """Whole graph (stem, stages, SPP, PAN neck with ConvTranspose, DFL heads, decode, TAL + fused loss, backward)."""
    from oracle import sg_oracle as O
    from oracle.yolo_nas_oracle import YoloNASOracle
    from super_gradients_b200.training.losses import PPYoloELoss

    g = golden("tiny_yolo_nas")
    m = _tiny_model(g)
    m.train()
    (pb, ps), raw = m(g["x"].to(DEV))
    crit = PPYoloELoss(num_classes=4, use_static_assigner=False)
    loss, items = crit(((pb, ps), raw), g["targets"])
    loss.backward()
    params = dict(m.named_parameters())
    live = [k for k in g["param_names"] if "rbr_reparam" not in k]
    # (1) tight: the same graph on the CPU oracle with bf16 emulation
    with O.bf16_emulation():
        pe = {k: v.clone() for k, v in g["sd0"].items()}
        for k in live:
            pe[k].requires_grad_(True)
        (pbe, pse), rawe = YoloNASOracle(g["arch"], pe, training=True).forward(g["x"])
        losse, itemse = O.ppyoloe_loss(rawe, g["targets"], 4)
        losse.backward()
    # Tolerances for the 25-layer graph = 2x the spread between two CPU emulations that differ only in the accumulation
    # precision of the GEMM sums (fp32 vs fp64 before the bf16 store): cls 0.7 %, reg 6.4 %, boxes 0.6 % -- 1-ulp flips of
    # bf16 activations are amplified by the train-mode BatchNorms of the deep 4x4 / 8x8 maps
    # (tests/test_oracle_golden.py::test_bf16_emulation_sensitivity measures that spread).
    assert l2rel(raw[0], rawe[0]) < 1.5e-2 and l2rel(raw[1], rawe[1]) < 0.13
    # scores = sigmoid(logit) with logits around the -4.6 prior bias: d(sigmoid)/sigmoid = (1 - sigmoid) * d(logit), so the
    # RELATIVE score error is the ABSOLUTE logit error, i.e. 1.5e-2 * rms(logit) ~ 7e-2 at the logit tolerance above.
    assert l2rel(ps, pse) < 7e-2 and l2rel(pb, pbe) < 2e-2
    assert abs(float(loss) - float(losse)) <= 5e-2 * abs(float(losse))
    # Gradients: on this graph two CPU emulations that differ only in accumulation precision disagree by a median of 0.51
    # per parameter (discrete top-k assignment + BatchNorm over 4x4 maps; test_bf16_emulation_sensitivity pins that), so
    # the direction check is a sanity bound at 1.5x that spread; the NORMS are well conditioned and checked to 10 % (median).
    # Tight gradient parity is asserted block by block above and kernel by kernel in test_kernels_gpu.py.
    graded = [k for k in live if pe[k].grad is not None and pe[k].grad.norm() > 1e-6]
    errs = sorted((l2rel(params[k].grad, pe[k].grad), k) for k in graded)
    assert errs[len(errs) // 2][0] < 0.75, errs[len(errs) // 2]
    ratios = sorted(abs(float(torch.log(params[k].grad.float().norm().cpu() / pe[k].grad.norm()))) for k in graded)
    assert ratios[len(ratios) // 2] < 0.1, ratios[len(ratios) // 2]
    for k, v in g["running1"].items():
        assert l2rel(m.state_dict()[k], pe[k]) < 5e-2, k
    # anchors / strides are exact
    ref_anchors, ref_points, ref_nums, ref_strides = O.anchors_for_levels([(16, 16), (8, 8), (4, 4)], (8, 16, 32))
    torch.testing.assert_close(raw[2].cpu(), ref_anchors)
    torch.testing.assert_close(raw[3].cpu(), ref_points)
    assert list(raw[4]) == ref_nums
    torch.testing.assert_close(raw[5].cpu(), ref_strides)
    # (2) loose: the fp32 fixture of the unmodified reference
    assert l2rel(raw[1], g["train_reg_distri"]) < 0.2
    assert l2rel(pb, g["train_pred_bboxes"]) < 0.1
    assert abs(float(loss) - float(g["loss"])) <= 0.1 * abs(float(g["loss"]))
    # every live parameter received a gradient; dead placeholders did not (SURVEY.md D7)
    for k, p in params.items():
        assert (p.grad is None) == ("rbr_reparam" in k), k
    # eval mode
    m.eval()
    sd = {**g["sd0"], **g["running1"]}
    m.load_state_dict(sd, strict=False)
    with torch.no_grad():
        (eb, es), _ = m(g["x"].to(DEV))
    with O.bf16_emulation():
        (ebe, ese), _ = YoloNASOracle(g["arch"], {k: v.clone() for k, v in sd.items()}, training=False).forward(g["x"])
    assert l2rel(es, ese) < 3e-2 and l2rel(eb, ebe) < 3e-2
    assert l2rel(es, g["eval_pred_scores"]) < 0.1
    assert l2rel(eb, g["eval_pred_bboxes"]) < 0.1


def test_yolo_nas_s_full_train_step_runs_and_predicts():
    """Config-2 model at reduced batch: forward + loss + backward produce finite values; predict() returns rows."""
    from super_gradients_b200.training import models
    from super_gradients_b200.training.losses import PPYoloELoss

    torch.manual_seed(0)
    m = models.get("yolo_nas_s", num_classes=80).to(DEV)
    m.train()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 3, 320, 320, generator=g).to(DEV)
    rows = []
    for b in range(2):
        for _ in range(4):
            cx, cy = (torch.rand(2, generator=g) * 200 + 60).tolist()
            w, h = (torch.rand(2, generator=g) * 80 + 20).tolist()
            rows.append([b, int(torch.randint(0, 80, (1,), generator=g)), cx, cy, w, h])
    out = m(x)
    assert out[0][0].shape == (2, 2100, 4) and out[1][1].shape == (2, 2100, 68)
    loss, items = PPYoloELoss(num_classes=80, use_static_assigner=False)(out, torch.tensor(rows))
    loss.backward()
    assert torch.isfinite(loss)
    n_live = sum(p.numel() for p in m.parameters() if p.grad is not None)
    assert n_live == 12_880_000 or abs(n_live - 12.88e6) < 0.02e6  # SURVEY.md D7: 12.88 M live of 19.05 M
    assert all(torch.isfinite(p.grad).all() for p in m.parameters() if p.grad is not None)
    preds = m.predict(x, conf=0.01, iou=0.7)
    assert len(preds) == 2 and preds[0].shape[1] == 6


def test_yolo_nas_s_config2_size_loss_parity():
    """Whole-graph parity at CONFIG-2 size (YOLO-NAS-S, 640 x 640, COCO-shape targets; 4 of the 32 images so the CPU oracle stays
    in seconds): raw head outputs, decoded boxes / scores, loss and its three components against
      (1) the whole-graph oracle in bf16-emulation mode (same rounding points as the kernels): the kernels' own error;
      (2) the same oracle in plain fp32 (= the reference's CPU arithmetic): adds the gap bf16 activation STORAGE cannot avoid.
    Unlike the 4 x 4-map tiny fixture the BatchNorms here average >= 1600 positions, so single-ulp flips are not amplified.
    The achieved errors are printed as one JSON object (profiles/r2_config2_parity.json keeps a committed copy)."""
    import json
    import os

    import yaml

    import bench
    from oracle import sg_oracle as O
    from oracle.yolo_nas_oracle import YoloNASOracle
    from super_gradients_b200.training import models
    from super_gradients_b200.training.losses import PPYoloELoss

    torch.manual_seed(0)
    m = models.get("yolo_nas_s", num_classes=80).to(DEV).train()
    sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    x, t = bench.synth_batch(4, 7)
    (pb, ps), raw = m(x.to(DEV))
    loss, items = PPYoloELoss(num_classes=80, use_static_assigner=False)(((pb, ps), raw), t)
    torch.cuda.synchronize()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    arch = yaml.safe_load(open(os.path.join(root, "super_gradients_b200", "recipes", "arch_params", "yolo_nas_s_arch_params.yaml")))
    arch["bn_eps"], arch["bn_momentum"] = float(arch["bn_eps"]), float(arch["bn_momentum"])
    rep = {}
    for mode in ("bf16_emulation", "fp32"):
        with torch.no_grad():
            if mode == "bf16_emulation":
                with O.bf16_emulation():
                    (pbe, pse), rawe = YoloNASOracle(arch, {k: v.clone() for k, v in sd.items()}, training=True).forward(x)
                    losse, itemse = O.ppyoloe_loss(rawe, t, 80)
            else:
                (pbe, pse), rawe = YoloNASOracle(arch, {k: v.clone() for k, v in sd.items()}, training=True).forward(x)
                losse, itemse = O.ppyoloe_loss(rawe, t, 80)
        rep[mode] = {
            "cls_logits": l2rel(raw[0], rawe[0]), "reg_distri": l2rel(raw[1], rawe[1]), "boxes": l2rel(pb, pbe), "scores": l2rel(ps, pse),
            "loss": abs(float(loss) - float(losse)) / abs(float(losse)),
            "items": [abs(float(a) - float(b)) / max(abs(float(b)), 1e-12) for a, b in zip(items.detach().cpu().reshape(-1), itemse.detach().reshape(-1))],
            "loss_value": float(loss), "oracle_loss_value": float(losse),
        }  # fmt: skip
    # (3) the loss kernels on the real graph: the oracle's loss evaluated on the PRODUCT's own head outputs (identical inputs ->
    #     identical assignment): this is the "loss within 1e-3" statement that is well posed.
    raw_cpu = tuple(t.detach().float().cpu() if torch.is_tensor(t) else t for t in raw)
    with torch.no_grad():
        loss_own, items_own = O.ppyoloe_loss(raw_cpu, t, 80)
    rep["loss_kernels_on_own_outputs"] = {"loss": abs(float(loss) - float(loss_own)) / abs(float(loss_own)),
                                          "items": [abs(float(a) - float(b)) / max(abs(float(b)), 1e-12) for a, b in zip(items.detach().cpu().reshape(-1), items_own.reshape(-1))]}  # fmt: skip
    rep["fp32_vs_bf16_emulation_oracles"] = abs(rep["fp32"]["oracle_loss_value"] - rep["bf16_emulation"]["oracle_loss_value"]) / rep["fp32"]["oracle_loss_value"]
    print("config-2-size parity:", json.dumps(rep))
    own = rep["loss_kernels_on_own_outputs"]
    assert own["loss"] < 1e-3 and max(own["items"][:3]) < 1e-3, own
    # End to end the loss is NOT a continuous function of the activations: the task-aligned assigner picks the top-13 anchors per box
    # by score^1 * IoU^6, and at random initialisation neighbouring anchors tie to within bf16 noise, so two implementations that
    # round differently (the two ORACLES differ from each other by 3e-3) assign a few boxes to different anchors.  Measured on B200
    # across builds of this repo: 6.6e-4 ... 4.6e-3 against the emulation, 1.4e-3 ... 2.6e-3 against fp32; bounded here at 1e-2.
    e, f = rep["bf16_emulation"], rep["fp32"]
    assert e["loss"] < 1e-2 and f["loss"] < 1e-2, (e, f)
    # Tensor-level relative L2 after ~100 bf16-stored layers (measured 1.2e-2 / 0.13 / 4.0e-3 / 5.8e-2 vs the emulation: the reg
    # head's logits are near-zero noise at initialisation, which inflates THEIR relative error; the decoded boxes are at 4e-3)
    assert e["cls_logits"] < 2e-2 and e["reg_distri"] < 0.2 and e["boxes"] < 8e-3 and e["scores"] < 9e-2, e
    assert f["cls_logits"] < 3e-2 and f["boxes"] < 1.2e-2, f


def test_resnet18_cifar_training_matches_reference_trajectory(golden):
    """config 1: same seeded init (identical RNG consumption as the reference constructor), same synthetic batches,
    SGD(lr 0.1, m 0.9, wd 1e-4 on conv/linear weights) + CE: per-step losses follow the reference's."""
    from super_gradients_b200.training import models

    g = golden("resnet18_cifar_train")
    torch.manual_seed(0)
    m = models.get("resnet18_cifar", num_classes=10).to(DEV)
    gen = torch.Generator().manual_seed(6)
    X = torch.randn(256, 3, 32, 32, generator=gen)
    Y = torch.randint(0, 10, (256,), generator=gen)
    decay, no_decay = [], []
    for n, p in m.named_parameters():
        (no_decay if (n.endswith(".bias") or "bn" in n or "shortcut.1" in n) else decay).append(p)
    opt = torch.optim.SGD([{"params": decay, "weight_decay": 1e-4}, {"params": no_decay, "weight_decay": 0.0}], lr=0.1, momentum=0.9)
    m.train()
    losses = []
    for step in range(2):
        xb, yb = X[step * 64 : (step + 1) * 64].to(DEV), Y[step * 64 : (step + 1) * 64].to(DEV)
        loss = torch.nn.functional.cross_entropy(m(xb), yb)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert abs(losses[0] - g["losses"][0]) < 2e-2 * g["losses"][0]
    assert abs(losses[1] - g["losses"][1]) < 0.1 * g["losses"][1]


def test_tiny_yolo_nas_pose_eval_and_predict(golden):
    """Row L8 end to end on the GPU: eval-mode YoloNASPose (reference arch + state dict) -> decoded boxes / person scores /
    keypoints / joint scores and raw head outputs against the whole-graph oracle in bf16-emulation mode (tight) and the fp32
    outputs of the unmodified reference (loose); then the post-prediction callback on the product's own outputs against the
    oracle post-processing of the same tensors (exact)."""
    from oracle import sg_oracle as O
    from oracle.yolo_nas_oracle import YoloNASOracle
    from super_gradients_b200.training.models.pose_estimation_models import YoloNASPose, YoloNASPosePostPredictionCallback

    g = golden("tiny_yolo_nas_pose")
    ap = copy.deepcopy(g["arch"])
    m = YoloNASPose(backbone=ap["backbone"], neck=ap["neck"], heads=ap["heads"], num_classes=5, bn_eps=1e-3, bn_momentum=0.03, inplace_act=True, in_channels=3)
    assert list(m.state_dict().keys()) == g["state_keys"]
    load_sd(m, g["sd0"])
    m = m.to(DEV).eval()
    with torch.no_grad():
        decoded, raw = m(g["x"].to(DEV))
    with O.bf16_emulation():
        dec_e, raw_e = YoloNASOracle(g["arch"], {k: v.clone() for k, v in g["sd0"].items()}, training=False).forward(g["x"])
    names = ("boxes", "scores", "pose_coords", "pose_scores")
    for name, a, b in zip(names, decoded, dec_e):
        assert tuple(a.shape) == tuple(b.shape), name
        assert l2rel(a, b) < 3e-2, (name, l2rel(a, b))
    for i in (0, 1, 3):  # person logits, box distributions, joint logits
        assert l2rel(raw[i], raw_e[i]) < 3e-2, (i, l2rel(raw[i], raw_e[i]))
    for i in (4, 5, 7):  # anchors, anchor points, strides are exact
        torch.testing.assert_close(raw[i].cpu(), raw_e[i])
    assert list(raw[6]) == list(raw_e[6])
    for name, a, b in zip(names, decoded, g["decoded"]):  # fp32 reference, loose
        assert l2rel(a, b) < 0.1, (name, l2rel(a, b))
    # post-prediction callback on the product's own decoded tensors: exact against the oracle on the same numbers
    cb = YoloNASPosePostPredictionCallback(**g["cb"])
    preds = cb((decoded, raw))
    ref, _ = O.yolo_nas_pose_postprocess(*(t.cpu() for t in decoded), **g["cb"])
    assert len(preds) == len(ref) and sum(r[0].shape[0] for r in ref) > 0
    for pr, (rposes, rscores, rboxes) in zip(preds, ref):
        np.testing.assert_array_equal(pr.scores.cpu().numpy(), rscores)
        np.testing.assert_array_equal(pr.bboxes_xyxy.cpu().numpy(), rboxes)
        np.testing.assert_array_equal(pr.poses.cpu().numpy(), rposes)
    # the model-level predict() wraps exactly that
    out = m.predict(g["x"].to(DEV), conf=g["cb"]["pose_confidence_threshold"], iou=g["cb"]["nms_iou_threshold"], pre_nms_max_predictions=100, post_nms_max_predictions=20)
    assert [int(o.scores.shape[0]) for o in out] == [r[0].shape[0] for r in ref]
