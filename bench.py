#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric and the other GPU configs of BASELINE.json, one JSON line per run.

    python bench.py --gpus N --steps K --warmup W                 # config 2 (default): the BASELINE metric, our arm
    python bench.py --config {2,3,4,5} ...                         # 3: YOLO-NAS-M train, 4: ResNet-50 train, 5: POSE-L predict()
    python bench.py --impl reference [--config C] --gpus N ...     # the reference's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR                         # also write what the last timed step computed, DIR/<name>.npy

  config 2  YOLO-NAS-S  640x640 train step, 32 images / GPU (fwd + PPYoloELoss/TAL + bwd + AdamW + EMA)      [BASELINE metric]
  config 3  YOLO-NAS-M  640x640 train step, 16 images / GPU (same step; the weak-scaling sweep config)
  config 4  ResNet-50   224x224 train step, 256 images / GPU (drop-path 0.05, cross entropy, SGD momentum; recipes/imagenet_resnet50)
  config 5  YOLO-NAS-POSE-L 640x640 inference: predict(batch_size=64) = fused pre-processing + model + pose-DFL decode + batched NMS

One JSON line on stdout (rank 0).  See DESIGN.md section "Measurement" for how each field is obtained.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NCLS, NBOX = 80, 8
# GFLOP per image: SURVEY.md section 8(d) (train = 3 x 2 x forward GMAC of the train-mode graph; config 5 = 2 x fused inference GMAC)
CONFIGS = {
    2: dict(kind="train_det", model="yolo_nas_s", batch=32, img=640, gflop=101.6, metric="images/sec YOLO-NAS-S 640 bf16 train",
            workload="configs[1]: YOLO-NAS-S 640x640 synthetic COCO-shape train step (fwd + PPYoloELoss/TAL + bwd + AdamW + EMA)", cpu_sample=2),
    3: dict(kind="train_det", model="yolo_nas_m", batch=16, img=640, gflop=282.6, metric="images/sec YOLO-NAS-M 640 bf16 train",
            workload="configs[2]: YOLO-NAS-M 640x640 synthetic COCO-shape train step, 16 images / GPU (fwd + PPYoloELoss/TAL + bwd + AdamW + EMA)", cpu_sample=1),
    4: dict(kind="train_cls", model="resnet50", batch=256, img=224, gflop=24.5, metric="images/sec ResNet-50 224 bf16 train",
            workload="configs[3]: ResNet-50 224x224 synthetic ImageNet-shape train step, 256 images / GPU (drop-path 0.05, cross entropy, SGD momentum)", cpu_sample=16),
    5: dict(kind="predict_pose", model="yolo_nas_pose_l", batch=64, img=640, gflop=144.9, metric="images/sec YOLO-NAS-POSE-L 640 bf16 predict",
            workload="configs[4]: YOLO-NAS-POSE-L 640x640 inference, predict(batch_size=64): pre-processing + model + pose-DFL decode + batched NMS", cpu_sample=2),
}  # fmt: skip
# kept for tools/ that import them
METRIC, WORKLOAD, IMG, BATCH = CONFIGS[2]["metric"], CONFIGS[2]["workload"], 640, 32
TRAIN_GFLOP_PER_IMG = CONFIGS[2]["gflop"]
# dram__bytes_read.sum + dram__bytes_write.sum of the conv family over ONE step from a committed ncu launch list of this command
# (None: not captured for that configuration); the JSON line names the file
NCU_CONV_DRAM = {(2, 32): (17.99e9, "profiles/r2_launches_graph_step.txt")}


def synth_batch(batch, seed, img=640):
    import torch

    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, 3, img, img, generator=g)
    rows = []
    for b in range(batch):
        cxy = torch.rand(NBOX, 2, generator=g) * (img - 200) + 100
        wh = torch.rand(NBOX, 2, generator=g) * 150 + 30
        cls = torch.randint(0, NCLS, (NBOX, 1), generator=g).float()
        rows.append(torch.cat([torch.full((NBOX, 1), float(b)), cls, cxy, wh], 1))
    return x, torch.cat(rows)


def synth_cls_batch(batch, seed, img=224, n_cls=1000):
    import torch

    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, 3, img, img, generator=g), torch.randint(0, n_cls, (batch,), generator=g)


def synth_images_u8(batch, seed, img=640):
    """Raw uint8 H x W x 3 images (what predict() takes) in PINNED host memory, as numpy views."""
    import torch

    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(batch):
        t = torch.randint(0, 256, (img, img, 3), generator=g, dtype=torch.uint8)
        try:
            t = t.pin_memory()
        except Exception:  # no CUDA runtime (CPU dry run)
            pass
        out.append(t.numpy())
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md).

    ONE nvidia-smi process per job (rank 0 samples every GPU of the node), started BEFORE the warm-up steps: spawning it costs
    ~100 ms of NVML initialisation during which driver calls of the benchmark can stall -- round 1 started one process per rank at
    the first timed step, and at N = 8 that stall (eight concurrent NVML initialisations) landed inside the 20-step timed region
    (30.5 ms / step reported against 26.7 ms / step in the e2e loop of the same run, which starts no sampler).  mark() / snapshot()
    select the samples taken between the two barriers of a timed region."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, enabled=True):
        self.index, self.enabled, self.proc, self.lines, self.mark_n = index, enabled, None, [], 0

    def start(self):
        if not self.enabled:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            t0 = time.time()
            while not self.lines and time.time() - t0 < 5.0:  # NVML is up once the first sample arrives
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        self.mark_n = len(self.lines)

    def snapshot(self):
        """Statistics of the samples since mark(): this rank's GPU (`index`) for the clocks, every GPU of the node for the reasons."""
        if not self.enabled:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "sampled by rank 0"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        sm, mx, reasons, others = [], None, set(), []
        for ln in self.lines[self.mark_n :]:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                gpu, clk, cmax = int(f[0]), float(f[1]), float(f[2])
            except ValueError:
                continue
            if gpu == self.index:
                sm.append(clk)
                mx = cmax
            else:
                others.append(clk)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        others.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}
        if others:
            out["other_gpus_sm_mhz"] = {"min": others[0], "median": others[len(others) // 2], "samples": len(others)}
        return out

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            self.proc = None


DUMP_SAMPLE = 1 << 20  # elements kept of an output larger than this (a fixed, seeded sample)


def param_sample(step):
    """The trained parameters (and their EMA) after the step, as a seeded sample taken in parameter-NAME order: two builds whose flat
    parameter layout differs still sample the same elements."""
    import torch

    f = step.flat
    pos = torch.cat([torch.arange(off, off + k) for _, (off, k) in sorted(f.offsets.items())])
    if pos.numel() > DUMP_SAMPLE:
        pos = pos[torch.randperm(pos.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values]
    pos = pos.to(f.params.device)
    out = {"params_sample": f.params[pos]}
    if step.ema_on:
        out["ema_params_sample"] = step.ema_params[pos]
    return out


def dump_outputs(out_dir, arrays):
    """Writes {name: tensor} as out_dir/<name>.npy: float64 stays float64, other floating types become float32, integers float64
    (exact up to 2**53)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu()
        a = a.double() if a.dtype == torch.float64 or not a.is_floating_point() else a.float()
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# =============================================================================================== reference arm (CPU)
def pick_cpu_threads(cores):
    """torch's CPU kernels stop scaling (and on many-socket hosts collapse) long before 128 threads at these sizes, so the
    baseline uses the thread count that is FASTEST on a representative 3x3 convolution fwd + bwd, not blindly all of them."""
    import torch
    import torch.nn.functional as F

    cands = sorted({c for c in (cores, cores // 2, cores // 4, cores // 8, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    x = torch.randn(2, 48, 160, 160, requires_grad=True)
    w = torch.randn(96, 48, 3, 3, requires_grad=True)
    best, best_t = cores, float("inf")
    for c in cands:
        torch.set_num_threads(c)
        F.conv2d(x, w, padding=1).sum().backward()  # warm the thread pool
        t0 = time.perf_counter()
        for _ in range(2):
            F.conv2d(x, w, padding=1).sum().backward()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def _arch_yaml(model):
    import yaml

    arch = yaml.safe_load(open(os.path.join(ROOT, "super_gradients_b200", "recipes", "arch_params", f"{model}_arch_params.yaml")))
    arch["bn_eps"], arch["bn_momentum"] = float(arch["bn_eps"]), float(arch["bn_momentum"])
    return arch


def cpu_step_fn(cfg, sample):
    """One step of the workload in the reference's own arithmetic (oracle port, fp32 CPU) on `sample` images.  Returns a
    zero-argument callable; nothing from the product package is on this path (shapes come from the reference-generated
    tests/golden/state_keys.pt, the architecture from the recipes' yaml)."""
    import torch

    table = torch.load(os.path.join(ROOT, "tests", "golden", "state_keys.pt"), weights_only=False)
    model, img = cfg["model"], cfg["img"]
    if cfg["kind"] == "train_det":
        from oracle.yolo_nas_oracle import random_state, train_step

        state = random_state(table[model], seed=0)
        live = [k for k in table[model + "/param_names"] if "rbr_reparam" not in k]
        arch = _arch_yaml(model)
        x, t = synth_batch(sample, 123, img)
        opt_state = {k: (torch.zeros_like(state[k]), torch.zeros_like(state[k])) for k in live}
        ema = {k: state[k].detach().clone() for k in live}
        it = [0]

        def step():
            it[0] += 1
            _loss, _items, grads = train_step(arch, state, x, t, NCLS, live)
            for k, g in grads.items():  # AdamW + EMA, as in the GPU arm
                m1, m2 = opt_state[k]
                m1.mul_(0.9).add_(g, alpha=0.1)
                m2.mul_(0.999).addcmul_(g, g, value=0.001)
                state[k].mul_(1 - 2e-4 * 1e-5).addcdiv_(m1 / (1 - 0.9 ** it[0]), (m2 / (1 - 0.999 ** it[0])).sqrt_().add_(1e-8), value=-2e-4)
                ema[k].mul_(0.9997).add_(state[k].detach(), alpha=1 - 0.9997)

        return step
    if cfg["kind"] == "train_cls":
        from oracle import resnet_oracle as R
        from oracle.yolo_nas_oracle import random_state

        state = random_state(table[model], seed=0)
        live = list(table[model + "/param_names"])
        x, y = synth_cls_batch(sample, 123, img)
        mom = {k: torch.zeros_like(state[k]) for k in live}
        gen = torch.Generator().manual_seed(5)

        def step():
            _loss, grads = R.train_step(model, state, x, y, live, droppath_prob=0.05, generator=gen)
            for k, g in grads.items():  # SGD momentum 0.9, weight decay 1e-4 on filters (zero on bias / BN), as in the GPU arm
                if state[k].dim() > 1:
                    g = g.add(state[k].detach(), alpha=1e-4)
                mom[k].mul_(0.9).add_(g)
                state[k].add_(mom[k], alpha=-0.1)

        return step
    if cfg["kind"] == "predict_pose":
        import numpy as np

        from oracle import sg_oracle as O
        from oracle.yolo_nas_oracle import YoloNASOracle, random_state

        state = random_state(table[model], seed=0)
        arch = _arch_yaml(model)
        imgs = synth_images_u8(sample, 123, img)

        def step():
            with torch.no_grad():
                batch = torch.stack([torch.from_numpy(O.preprocess_image(im, rescale=(img, img), keep_aspect=True, pad_shape=(img, img), pad_value=127, center=False, reverse=True, max_value=255.0)[0].astype(np.float32)) for im in imgs])
                (boxes, conf, coords, jscores), _raw = YoloNASOracle(arch, state, training=False).forward(batch)
                O.yolo_nas_pose_postprocess(boxes, conf, coords, jscores, pose_confidence_threshold=0.5, nms_iou_threshold=0.7, pre_nms_max_predictions=300, post_nms_max_predictions=100)

        return step
    raise ValueError(cfg["kind"])


def cpu_sample_rate(cfg, threads, max_steps, budget_s):
    """images/sec of the CPU port on a bounded sample: at least one step, more (up to max_steps) only while the time budget allows;
    with >= 2 steps the first (cold) one is excluded.  Returns (images/sec, seconds per step, steps timed, images per step)."""
    import torch

    torch.set_num_threads(threads)
    sample = cfg["cpu_sample"]
    step = cpu_step_fn(cfg, sample)
    times, start = [], time.perf_counter()
    for _ in range(max_steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - start + times[-1] > budget_s:  # another step would overrun the budget
            break
    timed = times[1:] if len(times) > 1 else times
    sec = sum(timed) / len(timed)
    return sample / sec, sec, len(timed), sample, len(times) - len(timed)


def run_reference(args, cfg):
    """The reference's CPU path for the same workload: the oracle port (kind "port": the reference is pure Python on torch CPU
    kernels and /root/reference does not exist on the GPU box; the port's fidelity is what tests/test_oracle_golden.py pins).
    `steps` / `ms_per_step` / `config.images_per_step` describe what was ACTUALLY timed: a bounded sample, not the GPU arm's batch.
    Under torchrun only rank 0 runs: ONE host, whatever N is."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = pick_cpu_threads(cores)
    ips, sec, n, sample, cold = cpu_sample_rate(cfg, threads, max_steps=args.steps + 1, budget_s=float("inf"))  # one cold step + --steps timed
    what = {"train_det": "train step", "train_cls": "train step", "predict_pose": "predict() batch"}[cfg["kind"]]
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": ips, "unit": "images/sec", "n_gpus": args.gpus, "steps": n, "warmup": cold,
        "requested_steps": args.steps, "requested_warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "config": args.config, "per_gpu_batch": cfg["batch"], "global_batch": cfg["batch"], "parallelism": "cpu", "cuda_graph": False,
                   "images_per_step": sample, "same_config": False, "n_gpus_note": "one CPU host regardless of --gpus: compare with the GPU arm at N=1 only",
                   "sample": f"each timed step is a bounded sample of the workload: one {what} on {sample} of the {cfg['batch']} images, fp32 CPU (oracle port)"},
        "cpu_baseline": {"value": ips, "unit": "images/sec", "cores": threads, "kind": "port",
                         "sample": f"{n} timed step(s) of {sample} images x {cfg['img']}x{cfg['img']}, fp32 oracle port, torch CPU threads={threads} (fastest of a sweep up to the host's {cores})"},
        "e2e": {"value": ips, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }  # fmt: skip
    print(json.dumps(line), flush=True)


# =============================================================================================== our arm (GPU)
def _to_dev(obj, dev):
    import torch

    return obj.to(dev) if torch.is_tensor(obj) else tuple(_to_dev(o, dev) for o in obj)


def _pin(obj):
    import torch

    return obj.pin_memory() if torch.is_tensor(obj) else tuple(_pin(o) for o in obj)


def _flat(obj):
    import torch

    return [obj] if torch.is_tensor(obj) else [t for o in obj for t in _flat(o)]


def build_train_workload(cfg, dev, rank, batch):
    """(model, criterion, TrainStep, host batches [(x, targets)], name of the loss-kernel family)."""
    import torch

    from super_gradients_b200.training import models
    from super_gradients_b200.training.sg_trainer import TrainStep

    torch.manual_seed(0)
    nbuf = 4
    if cfg["kind"] == "train_det":
        from super_gradients_b200.training.losses import PPYoloELoss, pad_targets_host

        model = models.get(cfg["model"], num_classes=NCLS).to(dev).train()
        step = TrainStep(model, PPYoloELoss(num_classes=NCLS, use_static_assigner=False), "AdamW", {"weight_decay": 1e-5}, zero_wd_on_bias_and_bn=True, ema=True)
        host = []
        for i in range(nbuf):
            x, t = synth_batch(batch, 1000 * rank + i, cfg["img"])
            host.append((x, tuple(pad_targets_host(t, batch, NBOX))))
    else:
        from super_gradients_b200.training.losses import CrossEntropyLoss

        model = models.get(cfg["model"], arch_params={"droppath_prob": 0.05}, num_classes=1000).to(dev).train()
        step = TrainStep(model, CrossEntropyLoss(), "SGD", {"weight_decay": 1e-4, "momentum": 0.9}, zero_wd_on_bias_and_bn=True, ema=False)
        host = [synth_cls_batch(batch, 1000 * rank + i, cfg["img"]) for i in range(nbuf)]
    return model, step, host


def run_train(args, cfg):
    import torch
    import torch.distributed as dist

    from super_gradients_b200 import kernels as K
    from super_gradients_b200 import lib
    from super_gradients_b200.training.sg_trainer import setup_device

    dev = setup_device()
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    lib.call("sgb_check_device")
    batch = args.batch or cfg["batch"]
    model, step, host = build_train_workload(cfg, dev, rank, batch)
    nbuf = len(host)
    # ---- synthetic data: distinct batches so that consecutive steps do not re-read the same inputs from L2
    host_x = [_pin(x) for x, _ in host]
    host_t = [_pin(t) for _, t in host]
    dev_x = [x.to(dev) for x, _ in host]
    dev_t = [_to_dev(t, dev) for _, t in host]
    ema_decay = 0.9997 if step.ema_on else None

    def lr_at(i):
        return 2e-4 if cfg["kind"] == "train_det" else 0.1

    # ---- count our kernel launches of one eager step (the claim behind `gpu_launches`)
    step.set_hyper_params(lr_at(0), ema_decay)
    lib.LAUNCHES[0] = 0
    step.run(dev_x[0], dev_t[0])
    torch.cuda.synchronize()
    launches_per_step = lib.LAUNCHES[0]

    use_graph = not args.no_graph
    if use_graph:
        try:
            step.capture(dev_x[0], dev_t[0], warmup=2)
        except Exception as e:  # noqa: BLE001
            print(f"[bench] rank {rank}: CUDA graph capture failed ({e!r}); running eagerly", file=sys.stderr)
            step.graph = None
            use_graph = False
        if world > 1:  # all ranks replay the graph or none does
            ok = torch.tensor([1 if use_graph else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok) == 0:
                step.graph = None
                use_graph = False

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- (A) device-resident throughput: `value`
    sampler = ClockSampler(dev.index or 0, enabled=rank == 0)
    sampler.start()  # before the warm-up: its start-up cost must not land in the timed region
    for i in range(args.warmup):
        step.set_hyper_params(lr_at(i), ema_decay)
        step.run(dev_x[i % nbuf], dev_t[i % nbuf])
    prof_range = os.environ.get("SGB_PROFILER_RANGE") == "1"  # `ncu --profile-from-start off`: capture exactly the timed steps

    def timed_region():
        """K steps between barriers, CUDA events, max over ranks; nvidia-smi clocks / throttle reasons sampled meanwhile."""
        barrier()
        sampler.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if prof_range:
            torch.cuda.profiler.start()
        e0.record()
        out = None
        for i in range(args.steps):
            step.set_hyper_params(lr_at(i), ema_decay)
            out = step.run(dev_x[i % nbuf], dev_t[i % nbuf])
        e1.record()
        barrier()
        if prof_range:
            torch.cuda.profiler.stop()
        clocks = sampler.snapshot()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, clocks, out

    ms, clocks, (loss, items) = timed_region()
    # what the last timed step computed, copied before anything else runs (a captured graph's outputs are rewritten by every replay).
    # A re-measured region below continues training, so the outputs are those of the first region: independent of the clocks.
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = {"loss": loss.clone(), "loss_items": items.clone(), **param_sample(step)}
    # a thermally / hardware-throttled region, or clocks pinned far below max without a reason, is measured once more (every
    # rank follows rank 0's verdict: the region contains collectives)
    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(clocks.get("reasons", []))
    pinned = bool(clocks.get("sm_mhz")) and bool(clocks.get("sm_max_mhz")) and clocks["sm_mhz"] < 0.5 * clocks["sm_max_mhz"] and not clocks.get("reasons")
    redo = torch.tensor([1 if (bad or pinned) else 0], device=dev)
    if world > 1:
        dist.broadcast(redo, src=0)
    if int(redo) == 1 and not prof_range:
        first = clocks
        ms, clocks, (loss, _) = timed_region()
        clocks["remeasured_after"] = {"reasons": first.get("reasons"), "sm_mhz": first.get("sm_mhz")}
    sampler.stop()
    final_loss = float(loss)
    value = world * batch * args.steps / (ms / 1e3)

    # ---- (B) end to end through the public step API with HOST (pinned) inputs: H2D of the batch + D2H of the loss
    copy_stream = torch.cuda.Stream()
    stage = [(torch.empty_like(dev_x[0]), _to_dev(host_t[0], dev)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            stage[s][0].copy_(host_x[i % nbuf], non_blocking=True)
            for d, h in zip(_flat(stage[s][1]), _flat(host_t[i % nbuf])):
                d.copy_(h, non_blocking=True)
            ready[s].record(copy_stream)

    for s in range(2):
        consumed[s].record()
    loss_host = torch.zeros(4, dtype=torch.float32).pin_memory()
    e2e_steps = args.steps
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prefetch(0)
    f0.record()
    d2h = 0
    for i in range(e2e_steps):
        if i + 1 < e2e_steps:
            prefetch(i + 1)
        s = i % 2
        torch.cuda.current_stream().wait_event(ready[s])
        step.set_hyper_params(lr_at(i), ema_decay)
        loss, items = step.run(stage[s][0], stage[s][1])
        consumed[s].record()
        items = items.reshape(-1)[:4]
        loss_host[: items.numel()].copy_(items, non_blocking=True)
        d2h = items.numel() * 4
        torch.cuda.current_stream().synchronize()  # the user reads the loss every step
    f1.record()
    barrier()
    ms2 = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([ms2], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms2 = float(t)
    e2e = world * batch * e2e_steps / (ms2 / 1e3)
    h2d = host_x[0].numel() * 4 + sum(t.numel() * t.element_size() for t in _flat(host_t[0]))

    # ---- (C) roofline of the dominant kernel family (implicit-GEMM convolutions): CUDA events around every launch.
    # EVERY rank runs these eager steps (they contain the gradient all-reduce); only rank 0 reports.
    roof = None
    K.PROFILE.clear()
    K.PROFILE_ON[0] = True
    n_prof = 2
    for i in range(n_prof):
        step.set_hyper_params(lr_at(i), ema_decay)
        step._step_eager(dev_x[i % nbuf], dev_t[i % nbuf])
    torch.cuda.synchronize()
    K.PROFILE_ON[0] = False
    barrier()
    if rank == 0:
        roof = conv_roofline(K.PROFILE, n_prof, cfg, batch, ms / args.steps, args.config)

    if rank != 0:
        return
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    cpu = None
    if not args.skip_cpu_baseline and world == 1:
        cpu = cpu_baseline(cfg)
    line = {
        "metric": cfg["metric"], "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {
            "workload": cfg["workload"], "config": args.config, "per_gpu_batch": batch,
            "global_batch": batch * world, "parallelism": f"dp{world}", "cuda_graph": use_graph,
            "l2": f"4 distinct {host_x[0].numel() * 4 / 1e6:.0f} MB input batches rotate (each > 126 MB L2); activations of a step (> 10 GB) never fit L2",
        },
        "e2e": {"value": e2e, "unit": "images/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms2 / e2e_steps},
        "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
        "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "final_loss": final_loss,
        "conv_tflops_whole_step": cfg["gflop"] * 1e9 * batch * world / (ms / args.steps / 1e3) / 1e12,
    }  # fmt: skip
    print(json.dumps(line), flush=True)


def conv_roofline(profile, n_prof, cfg, batch, step_ms, config_id):
    """Roofline object of the convolution family from per-launch CUDA events (kernels.PROFILE) of `n_prof` eager passes."""
    tf_peak, hbm_peak, which = peaks()
    per, conv_bytes = {}, 0.0
    for name, a, b, tag in profile:
        per[name] = per.get(name, 0.0) + a.elapsed_time(b)
        if name.startswith("sgb_conv_") and len(tag) == 7:  # activations in + out of the call (filters are noise)
            N_, H_, W_, C_, K_, _R, s_ = tag
            conv_bytes += 2.0 * N_ * (H_ * W_ * C_ + ((H_ + s_ - 1) // s_) * ((W_ + s_ - 1) // s_) * K_)
    conv_ms = sum(v for k, v in per.items() if k.startswith("sgb_conv")) / n_prof
    conv_bytes /= n_prof
    flops = cfg["gflop"] * 1e9 * batch
    achieved = flops / (conv_ms / 1e3) / 1e12
    traffic, traffic_src = NCU_CONV_DRAM.get((config_id, batch), (None, None))
    return {
        "bound": "tensor", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
        "traffic": traffic, "traffic_source": traffic_src or "not captured for this configuration",
        "kernel": "conv family of one step = one 'launch': conv3x3_halo_kernel / conv1x1_tile_kernel + wgrad3x3_halo_kernel (stride 1), conv_umma_kernel + wgrad_umma_kernel (stride 2, wide 1x1)",
        "peak_source": which, "conv_ms_per_step": conv_ms, "conv_share_of_step": conv_ms / step_ms,
        "timing": "CUDA events around every launch of an eager pass on its launching stream (the in-graph kernels run ~25 % faster: tools/timeline.py)",
        "algorithmic_flops_per_step": flops, "algorithmic_activation_bytes_per_step": conv_bytes,
        "hbm_view": {"achieved_GBps": conv_bytes / (conv_ms / 1e3) / 1e9, "peak_GBps": hbm_peak, "frac": conv_bytes / (conv_ms / 1e3) / 1e9 / hbm_peak,
                     "note": "narrow layers (32..192 channels) are HBM / shared-memory-operand bound, not tensor bound (DESIGN.md section 3)"},
        "per_call_ms": {k: v / n_prof for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:14]},
    }  # fmt: skip


def cpu_baseline(cfg):
    cores = os.cpu_count() or 1
    threads = pick_cpu_threads(cores)
    ips, sec, n, sample, _cold = cpu_sample_rate(cfg, threads, max_steps=2, budget_s=45.0)
    return {"value": ips, "unit": "images/sec", "cores": threads, "kind": "port",
            "sample": f"{n} timed step(s) of {sample} images {cfg['img']}x{cfg['img']}, fp32 oracle port (oracle/), {sec:.1f} s/step, threads={threads} (fastest of a sweep up to {cores})"}  # fmt: skip


def run_predict(args, cfg):
    """Config 5: YOLO-NAS-POSE-L predict(batch_size=64).  `value`: model + decode + NMS callback on a device-resident pre-processed
    batch; `e2e`: model.predict(list of raw uint8 images in pinned host memory) -> results read back to the host, every step.
    Inference shards trivially: under torchrun every rank runs its own replica on its own images (no collective)."""
    import torch
    import torch.distributed as dist

    from super_gradients_b200 import kernels as K
    from super_gradients_b200 import lib
    from super_gradients_b200.training import models
    from super_gradients_b200.training.sg_trainer import setup_device

    dev = setup_device()
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    lib.call("sgb_check_device")
    batch, img = args.batch or cfg["batch"], cfg["img"]
    torch.manual_seed(0)
    model = models.get(cfg["model"], num_classes=17).to(dev).eval()
    # random-init person scores sit at the prior (~0.01): a low threshold keeps the NMS busy like a trained model's crowd scene does
    kw = dict(conf=0.01, iou=0.7, pre_nms_max_predictions=300, post_nms_max_predictions=100)
    cb = model.get_post_prediction_callback(**kw)
    nbuf = 3
    raw = [synth_images_u8(batch, 1000 * rank + i, img) for i in range(nbuf)]
    from super_gradients_b200.training.processing import default_yolo_nas_pose_coco_processing_params

    proc = default_yolo_nas_pose_coco_processing_params()["image_processor"]
    dev_x = [proc.preprocess_batch(r, dev)[0] for r in raw]  # bf16 NHWC model inputs, resident

    def gpu_step(x):
        with torch.no_grad():
            return cb.forward_batched(model(x))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lib.LAUNCHES[0] = 0
    gpu_step(dev_x[0])
    torch.cuda.synchronize()
    launches_per_step = lib.LAUNCHES[0]
    sampler = ClockSampler(dev.index or 0, enabled=rank == 0)
    sampler.start()
    for i in range(args.warmup):
        gpu_step(dev_x[i % nbuf])
    barrier()
    sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = gpu_step(dev_x[i % nbuf])
    e1.record()
    barrier()
    clocks = sampler.snapshot()
    sampler.stop()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    value = world * batch * args.steps / (ms / 1e3)
    kept = float(out[3].float().mean())

    # ---- end to end: the public call, host images in, host results out
    for i in range(2):
        model.predict(raw[i % nbuf], batch_size=batch, **kw)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    d2h = 0
    for i in range(args.steps):
        res = model.predict(raw[i % nbuf], batch_size=batch, **kw)
        host_res = [(r.poses.cpu(), r.scores.cpu(), r.bboxes_xyxy.cpu()) for r in res]
        d2h = sum(t.numel() * t.element_size() for r in host_res for t in r)
    f1.record()
    barrier()
    ms2 = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([ms2], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms2 = float(t)
    e2e = world * batch * args.steps / (ms2 / 1e3)
    h2d = sum(im.nbytes for im in raw[0])

    # ---- per-launch events: conv family (tensor roofline) and the memory-bound decode / NMS kernels
    K.PROFILE.clear()
    K.PROFILE_ON[0] = True
    n_prof = 3
    for i in range(n_prof):
        gpu_step(dev_x[i % nbuf])
    torch.cuda.synchronize()
    K.PROFILE_ON[0] = False
    if rank != 0:
        return
    if args.dump_outputs:  # the last timed step's device-resident result (forward_batched)
        dump_outputs(args.dump_outputs, dict(zip(("rows", "poses", "anchor_index", "count"), out)))
    roof = conv_roofline(K.PROFILE, n_prof, cfg, batch, ms / args.steps, args.config)
    per = {}
    for name, a, b, _tag in K.PROFILE:
        per[name] = per.get(name, 0.0) + a.elapsed_time(b) / n_prof
    _tf, hbm_peak, _w = peaks()
    L, J = sum((img // s) ** 2 for s in (8, 16, 32)), 17
    nms_bytes = batch * L * (4 + 1) * 4  # boxes + person score read once (fp32); the kept rows written are noise
    dec_bytes = batch * L * ((4 * 17 + 1 + 3 * J) * 2 + (4 + 1 + 3 * J) * 4)  # bf16 head maps read, fp32 decoded tensors written
    mem = {}
    for name, byts in (("sgb_batched_nms", nms_bytes), ("sgb_dfl_decode", batch * L * ((4 * 17 + 1) * 2 + 5 * 4)), ("sgb_pose_keypoint_decode", batch * L * (3 * J * 2 + 3 * J * 4))):
        if name in per:
            mem[name] = {"us_per_batch": per[name] * 1e3, "algorithmic_bytes": byts, "GBps": byts / (per[name] / 1e3) / 1e9, "frac_of_hbm_peak": byts / (per[name] / 1e3) / 1e9 / hbm_peak}
    roof["memory_bound_kernels"] = mem
    roof["decode_plus_nms_ms_per_batch"] = sum(v for k, v in per.items() if k in ("sgb_batched_nms", "sgb_dfl_decode", "sgb_pose_keypoint_decode"))
    roof["decode_algorithmic_bytes"] = dec_bytes
    cpu = None
    if not args.skip_cpu_baseline and world == 1:
        cpu = cpu_baseline(cfg)
    line = {
        "metric": cfg["metric"], "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": cfg["workload"], "config": args.config, "per_gpu_batch": batch, "global_batch": batch * world, "parallelism": f"replicas{world}", "cuda_graph": False,
                   "nms": {**kw, "mean_kept_per_image": kept},
                   "l2": f"{nbuf} distinct {dev_x[0].numel() * 2 / 1e6:.0f} MB input batches rotate; a forward pass streams > 20 GB of activations"},
        "e2e": {"value": e2e, "unit": "images/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms2 / args.steps,
                "api": "model.predict(list of uint8 HxWx3 images in pinned host memory, batch_size=64) -> poses / scores / boxes copied to the host"},
        "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
        "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        "conv_tflops_whole_step": cfg["gflop"] * 1e9 * batch * world / (ms / args.steps / 1e3) / 1e12,
    }  # fmt: skip
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the configuration's)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
    elif cfg["kind"] == "predict_pose":
        run_predict(args, cfg)
    else:
        run_train(args, cfg)
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
