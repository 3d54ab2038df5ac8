"""Every kernel call the OTHER benchmark configurations make (BASELINE.json configs 3-5: YOLO-NAS-M / -L training, ResNet-50 training,
YOLO-NAS-POSE-L predict) is accepted by the C-ABI's host-side argument validation.

Only YOLO-NAS-S, the tiny fixtures and resnet18_cifar have run on a B200 so far.  Here the models run on the CPU stand-in backend,
and every kernel wrapper call is ALSO forwarded to the real wrapper and the real libsgb200.so entry point with the host tensors'
addresses: without a GPU the entry point either rejects the descriptor (SGB_E_INVALID / SGB_E_UNSUPPORTED -- a shape this
library cannot serve, which would be the first thing to fail on hardware) or gets as far as the first CUDA call and returns
SGB_E_CUDA.  No kernel runs, nothing is read through the pointers on the host."""
import collections
import functools
import os
import re
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import cpu_backend  # noqa: E402
from super_gradients_b200 import kernels as K  # noqa: E402
from super_gradients_b200 import lib as L  # noqa: E402

# the batched filter-refresh / gradient-layout tables are device-resident work lists whose stand-in representation is a Python
# list: nothing to validate through the C entry point
TABLES = {"weight_prepare_batch", "run_weight_prepare_batch", "wgrad_to_oihw_batch_table", "run_wgrad_to_oihw_batch", "qarep_alpha_finish_table", "run_qarep_alpha_finish"}
REAL = {name: getattr(K, name) for name in list(cpu_backend._SUBSET) + list(cpu_backend._TRAINING) if hasattr(K, name) and name not in TABLES}


def without_gpu(test):
    """The tests below pass host tensors' addresses to the real entry points and rely on there being no CUDA device, so that a valid
    call stops at its first CUDA call (SGB_E_CUDA).  Where a GPU is visible such a call would launch kernels on host addresses;
    there the test runs in a child pytest process that sees no GPU (CUDA_VISIBLE_DEVICES empty) and must pass in it."""

    @functools.wraps(test)
    def run(*args, **kwargs):
        if not torch.cuda.is_available():
            return test(*args, **kwargs)
        node = os.environ["PYTEST_CURRENT_TEST"].rsplit(" ", 1)[0]
        out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", node], cwd=os.path.dirname(HERE),
                             env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=850)  # fmt: skip
        assert out.returncode == 0 and re.search(r"\b1 passed\b", out.stdout), out.stdout[-3000:] + out.stderr[-2000:]

    return run


@pytest.fixture
def validating_backend(monkeypatch):
    """Stand-in backend whose every call first goes through the product wrapper + C entry point (validation only)."""
    cpu_backend.install_training(monkeypatch)
    seen, rejected = collections.Counter(), []
    lib = L.load()

    def call(name, *args):
        rc = getattr(lib, name)(*args)
        seen[name] += 1
        if rc in (-1, -2):
            msg = lib.sgb_last_error()
            rejected.append((name, rc, msg.decode() if msg else ""))
        return rc

    monkeypatch.setattr(L, "call", call)
    monkeypatch.setattr(K, "_stream", lambda: None)
    for name, real in REAL.items():
        standin = getattr(K, name)

        def both(*a, _real=real, _standin=standin, _name=name, **k):
            try:
                _real(*a, **k)
            except L.SgbError as e:  # raised by a wrapper's own argument check
                rejected.append((_name, "wrapper", str(e)))
            return _standin(*a, **k)

        monkeypatch.setattr(K, name, both)
    return seen, rejected


def _targets(batch, size, n_cls, per_image=3, seed=0):
    gen = torch.Generator().manual_seed(seed)
    rows = []
    for b in range(batch):
        for _ in range(per_image):
            cx, cy = (torch.rand(2, generator=gen) * size * 0.6 + size * 0.2).tolist()
            w, h = (torch.rand(2, generator=gen) * size * 0.3 + 8).tolist()
            rows.append([b, int(torch.randint(0, n_cls, (1,), generator=gen)), cx, cy, w, h])
    return torch.tensor(rows, dtype=torch.float32)


GOLD = torch.load(os.path.join(HERE, "golden", "other_configs.pt"))  # the reference's fp32 outputs for its seeded initialisation


def l2rel(a, b):
    return float((a.detach().double() - b.detach().double()).norm() / b.detach().double().norm().clamp_min(1e-30))


def _median_log_ratio(mine, ref):
    import math

    r = sorted(abs(math.log(mine[k] / ref[k])) for k in ref if ref[k] > 1e-6 and k in mine and mine[k] > 0)
    return r[len(r) // 2], len(r)


@pytest.mark.parametrize("name", ["yolo_nas_m", "yolo_nas_l"])
@without_gpu
def test_yolo_nas_m_l_train_step_shapes_are_served(validating_backend, name):
    """One AdamW + EMA train step of YOLO-NAS-M / -L at 128 x 128.  For M (config 3) the raw head outputs, the loss components and
    the per-parameter gradient norms are compared with the unmodified reference's (same seeded initialisation)."""
    from super_gradients_b200.training import models
    from super_gradients_b200.training.losses import PPYoloELoss
    from super_gradients_b200.training.sg_trainer import TrainStep

    seen, rejected = validating_backend
    g = GOLD["yolo_nas_m"]
    torch.manual_seed(0)
    m = models.get(name, num_classes=80).train()
    st = TrainStep(m, PPYoloELoss(num_classes=80, use_static_assigner=False), "AdamW", {"weight_decay": 1e-5}, zero_wd_on_bias_and_bn=True, ema=True)
    st.set_hyper_params(2e-4, 0.999)
    loss, items = st.forward_backward(g["x"].float(), g["targets"])
    grad_norms = {n: float(st.flat.grad_of(n).norm()) for n, _ in st.flat.order}
    st.optimizer_step()
    assert torch.isfinite(loss)
    assert not rejected, rejected[:5]
    assert seen["sgb_conv_fprop"] > 100 and seen["sgb_conv_dgrad"] > 100 and seen["sgb_conv_wgrad"] > 100 and seen["sgb_tal_assign"] == 1 and seen["sgb_adamw_step"] >= 1
    if name == "yolo_nas_m":
        assert abs(float(loss) - float(g["loss"])) < 0.05 * float(g["loss"]), (float(loss), float(g["loss"]))
        assert l2rel(items.cpu(), g["items"]) < 0.05
        med, n = _median_log_ratio(grad_norms, g["grad_norms"])
        assert n > 300 and med < 0.1, (med, n)  # bf16 operands vs the fp32 reference
        m.eval()
        with torch.no_grad():
            (eb, es), (cls_logits, reg_distri, *_rest) = m(g["x"].float())
        assert l2rel(eb, g["eval_boxes"]) < 0.03 and l2rel(es, g["eval_scores"]) < 0.03


@without_gpu
def test_resnet50_train_step_shapes_are_served(validating_backend):
    """Config 4's model: train-mode logits, cross-entropy, gradients and eval-mode logits against the reference's."""
    from super_gradients_b200.training import models

    seen, rejected = validating_backend
    g = GOLD["resnet50"]
    torch.manual_seed(0)
    m = models.get("resnet50", num_classes=1000).train()
    logits = m(g["x"].float())
    loss = torch.nn.functional.cross_entropy(logits, g["y"])
    loss.backward()
    assert not rejected, rejected[:5]
    assert seen["sgb_conv_fprop"] >= 53 and seen["sgb_conv_wgrad"] >= 53 and seen["sgb_maxpool_fwd"] == 1 and seen["sgb_avgpool_fwd"] == 1
    # tolerances: see the note in tests/golden/make_goldens.py::golden_other_configs -- the reference itself moves by 0.16 / 1.3
    # (logits / early-layer gradients) under bf16 storage rounding on this fixture; norms and the classifier are well conditioned
    assert l2rel(logits, g["train_logits"]) < 0.35 and abs(float(loss) - float(g["loss"])) < 0.02 * float(g["loss"])
    params = dict(m.named_parameters())
    assert l2rel(params["linear.bias"].grad, g["grads"]["linear.bias"]) < 0.01
    assert l2rel(params["linear.weight"].grad.flatten()[:: params["linear.weight"].grad.numel() // 10000], g["grads"]["linear.weight"]) < 0.35
    med, n = _median_log_ratio({k: float(p.grad.norm()) for k, p in params.items()}, g["grad_norms"])
    assert n > 150 and med < 0.05, (med, n)
    m.eval()
    with torch.no_grad():
        assert l2rel(m(g["x"].float()), g["eval_logits"]) < 0.08


@without_gpu
def test_yolo_nas_pose_l_predict_shapes_are_served(validating_backend):
    """Config 5's model: decoded eval outputs against the reference's, then predict() (NMS path) for the call coverage."""
    from super_gradients_b200.training import models

    seen, rejected = validating_backend
    g = GOLD["yolo_nas_pose_l"]
    torch.manual_seed(0)
    m = models.get("yolo_nas_pose_l", num_classes=17).eval()
    with torch.no_grad():
        (boxes, scores, poses, joint_scores), _raw = m(g["x"].float())
        res = m.predict(g["x"].float(), conf=0.01)
    assert len(res) == 2
    assert not rejected, rejected[:5]
    assert seen["sgb_conv_fprop"] > 100 and seen["sgb_batched_nms"] == 1 and seen["sgb_pose_keypoint_decode"] == 6
    assert l2rel(boxes, g["boxes"]) < 0.03 and l2rel(poses, g["poses"]) < 0.03
    assert l2rel(scores, g["scores"]) < 0.05 and l2rel(joint_scores, g["joint_scores"]) < 0.05


@without_gpu
def test_the_validation_hook_sees_rejections(validating_backend):
    """Negative control: a descriptor the library must refuse is reported, an acceptable one is not."""
    import ctypes

    seen, rejected = validating_backend
    x = torch.zeros(1, 16, 8, 8, dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
    w = torch.zeros(32, 3, 3, 16, dtype=torch.bfloat16)
    K.conv_fprop(x, w, 32, 3, 3, 1, 1)
    assert not rejected and seen["sgb_conv_fprop"] == 1
    d = REAL["conv_fprop"].__globals__["conv_desc"](x, 32, 3, 3, 1, 1)
    d.K = 0
    ep = L.Epilogue()
    L.call("sgb_conv_fprop", ctypes.byref(d), x.data_ptr(), w.data_ptr(), x.data_ptr(), ctypes.byref(ep), None)
    assert len(rejected) == 1 and rejected[0][1] == -1


@without_gpu
def test_new_entry_points_validate_their_descriptors(monkeypatch):
    """sgb_atss_assign / sgb_detection_matching / sgb_focal_cls_fwd_bwd through the product wrappers with host tensors: a valid call
    reaches the first CUDA call (SGB_E_CUDA here), an invalid one is refused with SGB_E_INVALID and the reason."""
    from super_gradients_b200.training.losses.ppyolo_loss import pad_targets_host

    monkeypatch.setattr(K, "require_cuda", lambda t, name="tensor": None)
    monkeypatch.setattr(K, "_stream", lambda: None)
    g = torch.load(os.path.join(HERE, "golden", "atss.pt"))
    c = g["regular"]
    B, Lc, _ = c["cls_logits"].shape
    gb, gl, gv = pad_targets_host(c["targets"], B, 6)
    st = g["stride_tensor"].reshape(-1).contiguous()

    def code(fn):
        with pytest.raises(L.SgbError) as e:
            fn()
        return str(e.value)

    atss = lambda nums, topk=9: K.atss_assign(K.loss_desc(B, Lc, 5, 16, 6, topk=topk), c["reg_distri"], g["anchors"].contiguous(), g["anchor_points"], st, nums, gb, gl, gv, torch.zeros(4, dtype=torch.float64))  # noqa: E731
    assert "code -3" in code(lambda: atss(g["nums"]))
    assert "code -1" in code(lambda: atss([320, 12, 4])) and "at least topk" in code(lambda: atss([320, 12, 4]))
    assert "code -1" in code(lambda: atss([256, 64])) and "code -1" in code(lambda: atss(g["nums"], topk=17))
    match = lambda thr: K.detection_matching(torch.zeros(2, 5, 6), torch.zeros(2, dtype=torch.int32), torch.zeros(2, 3, 5), torch.zeros(2, dtype=torch.int32), None, None, thr, 64, 64)  # noqa: E731
    assert "code -3" in code(lambda: match(torch.tensor([0.5]))) and "code -1" in code(lambda: match(torch.linspace(0.1, 0.9, 33)))
    with pytest.raises(L.SgbError, match="contiguous"):
        K.detection_matching(torch.zeros(2, 5, 6).double(), torch.zeros(2, dtype=torch.int32), torch.zeros(2, 3, 5), torch.zeros(2, dtype=torch.int32), None, None, torch.tensor([0.5]), 64, 64)
    d = K.loss_desc(B, Lc, 5, 16, 6)
    focal = lambda: L.call("sgb_focal_cls_fwd_bwd", __import__("ctypes").byref(d), c["cls_logits"].data_ptr(), gl.data_ptr(), c["cls_logits"].data_ptr(), torch.zeros(4, dtype=torch.float64).data_ptr(), 1.0, 0.25, None, None)  # noqa: E731
    assert "code -3" in code(focal)


@without_gpu
def test_replaced_input_channels_are_served(validating_backend):
    """models.get(..., num_input_channels=N): 1-channel ResNet-18 and 4-channel YOLO-NAS-S forward + backward run, and the first
    layers' (channel-padded) shapes pass the C-ABI validation."""
    from super_gradients_b200.training import models

    seen, rejected = validating_backend
    torch.manual_seed(0)
    r = models.get("resnet18", num_classes=5, num_input_channels=1).train()
    r(torch.randn(2, 1, 64, 64)).sum().backward()
    assert r.conv1.weight.grad is not None and r.conv1.weight.grad.shape[1] == 1 and torch.isfinite(r.conv1.weight.grad).all()
    y = models.get("yolo_nas_s", num_classes=3, num_input_channels=4).eval()
    with torch.no_grad():
        (boxes, scores), _raw = y(torch.randn(1, 4, 64, 64))
    assert tuple(scores.shape) == (1, 84, 3) and torch.isfinite(boxes).all()
    assert not rejected, rejected[:5]
