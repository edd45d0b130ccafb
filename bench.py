#!/usr/bin/env python
"""bench.py -- images/sec of the hot path on B200, BASELINE.json's metric.

    python bench.py [--config hg_fpd] --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU implementation of the same workload
    python bench.py ... --dump-outputs DIR    # also write what the last timed step computed, as DIR/<name>.npy

--config (default hg_fpd = BASELINE.json configs[1] at N=1, configs[2] at N>1):
    hg_fpd     student hourglass s4 f128 + frozen teacher s8 f256, FPD loss, 256x256, batch 32/GPU        (configs[1], [2])
    hg_mse_s1  hourglass s1 f64, plain MSE (function.train semantics), 256x256, batch 2                    (configs[0])
    hrnet_fpd  pose_hrnet w32 student + frozen w48 teacher, FPD loss, 256x192, batch 24/GPU                (configs[3])
    hg_infer   hourglass s4 f128 forward + flip test + arg-max decode + box NMS, 256x256, batch 128        (configs[4])

One JSON line on stdout (rank 0). A training "step" = student fwd + teacher fwd + fused FPD loss + student bwd + gradient
all-reduce (N>1) + Adam on one batch; an inference "step" = both forwards of the flip test + merge + arg-max + NMS on one
batch. `value`: inputs resident in HBM; `e2e`: pinned-host inputs copied H2D and results read back D2H inside the timed
region. The CPU legs (`cpu_baseline`, `--impl reference`) run the reference's own modules from oracle/_ref/ (oracle port
if that directory is absent) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NS = types.SimpleNamespace
MPII_FLIP_PAIRS = [[0, 5], [1, 4], [2, 3], [10, 15], [11, 14], [12, 13]]   # lib/dataset/mpii.py:32

# FLOP per image: BASELINE.md section 2 (conv MACs x 2; train = 3x student forward, teacher forward-only)
CONFIGS = {
    "hg_fpd": dict(
        workload="hourglass FPD train: student s4 f128 + frozen teacher s8 f256, 256x256, batch 32/GPU",
        family="hourglass", student=(128, 4), teacher=(256, 8), batch=32, H=256, W=256, J=16, lr=2.5e-4,
        flop_per_image=79.633e9, kind="train",
        # dominant kernel shape: the teacher's 3x3 128->128 @64x64 (18 launches/step = 38.7 % of the teacher's MACs)
        roof=dict(cin=128, cout=128, k=3, h=64, w=64)),
    "hg_mse_s1": dict(
        workload="hourglass s1 f64 train, MSE only (function.train), 256x256, batch 2",
        family="hourglass", student=(64, 1), teacher=None, batch=2, H=256, W=256, J=16, lr=2.5e-4,
        flop_per_image=2.369e9, kind="train",
        roof=dict(cin=32, cout=32, k=3, h=64, w=64)),
    "hrnet_fpd": dict(
        workload="pose_hrnet FPD train: student w32 + frozen teacher w48, 256x192, batch 24/GPU",
        family="hrnet", student=32, teacher=48, batch=24, H=256, W=192, J=17, lr=1e-3,
        flop_per_image=77.254e9, kind="train",
        # 3x3 48->48 @64x48: 64 launches per teacher forward, the largest single share of the step's MACs
        roof=dict(cin=48, cout=48, k=3, h=64, w=48)),
    "hg_infer": dict(
        workload="hourglass s4 f128 inference: forward + flip test + arg-max decode + box NMS(1024), 256x256, batch 128",
        family="hourglass", student=(128, 4), teacher=None, batch=128, H=256, W=256, J=16, lr=0.0,
        flop_per_image=15.629e9, kind="infer",
        roof=dict(cin=64, cout=64, k=3, h=64, w=64)),
    # --- beyond BASELINE.json (SURVEY 8 f4): the third registered model family, as experiments/mpii/resnet/res50_256x256_*
    "res50_mse": dict(
        workload="pose_resnet-50 (3 x 256-filter 4x4 deconv head) train, MSE only (function.train), 256x256, batch 32/GPU",
        family="resnet", student=50, teacher=None, batch=32, H=256, W=256, J=16, lr=1e-3,
        flop_per_image=3 * 2 * 7234125824.0, kind="train",
        # 3x3 128->128 @32x32 (layer2 conv2, 4 launches) stands for the body's 3x3 convolutions
        roof=dict(cin=128, cout=128, k=3, h=32, w=32)),
    # --- diagnostics (not BASELINE configs): the two halves of hg_fpd on their own
    "diag_student": dict(
        workload="[diagnostic] hourglass s4 f128 train, MSE only, 256x256, batch 32 (the student half of hg_fpd)",
        family="hourglass", student=(128, 4), teacher=None, batch=32, H=256, W=256, J=16, lr=2.5e-4,
        flop_per_image=23.44e9, kind="train", roof=dict(cin=64, cout=64, k=3, h=64, w=64)),
    "diag_teacher": dict(
        workload="[diagnostic] hourglass s8 f256 forward only (no flip), 256x256, batch 32 (the teacher half of hg_fpd)",
        family="hourglass", student=(256, 8), teacher=None, batch=32, H=256, W=256, J=16, lr=0.0,
        flop_per_image=56.189e9, kind="infer", flip=False, roof=dict(cin=128, cout=128, k=3, h=64, w=64)),
}
CONV_H_3X3_DRAM_BYTES = 89.88e6   # dram__bytes_read + write, conv_tc_h 3x3 128->128 @64x64 B=32: profiles/r2_prof_conv_h_3x3.md


def cfg(f, s, j=16):
    return NS(MODEL=NS(EXTRA=NS(NUM_FEATURES=f, NUM_STACKS=s, NUM_BLOCKS=1), NUM_JOINTS=j))


class _Cfg(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


def _wrap(d):
    return _Cfg({k: _wrap(v) for k, v in d.items()}) if isinstance(d, dict) else d


def resnet_cfg(num_layers, j=16):
    """experiments/mpii/resnet/res*_256x256_d256x3_adam_lr1e-3.yaml, MODEL.EXTRA."""
    return NS(MODEL=NS(NUM_JOINTS=j, INIT_WEIGHTS=False, PRETRAINED='', EXTRA=NS(
        NUM_LAYERS=num_layers, DECONV_WITH_BIAS=False, NUM_DECONV_LAYERS=3, NUM_DECONV_FILTERS=[256, 256, 256],
        NUM_DECONV_KERNELS=[4, 4, 4], FINAL_CONV_KERNEL=1)))


def hrnet_cfg(w, j=17):
    """experiments/fpd_coco/hrnet/w{32,48}_256x192_adam_lr1e-3.yaml, MODEL.EXTRA (hrnet_template.yaml:52-90)."""
    def stage(nmod, chans):
        return dict(NUM_MODULES=nmod, NUM_BRANCHES=len(chans), BLOCK='BASIC', NUM_BLOCKS=[4] * len(chans),
                    NUM_CHANNELS=chans, FUSE_METHOD='SUM')
    return _wrap(dict(MODEL=dict(NUM_JOINTS=j, INIT_WEIGHTS=False, PRETRAINED='', EXTRA=dict(
        PRETRAINED_LAYERS=['*'], FINAL_CONV_KERNEL=1, STAGE2=stage(1, [w, 2 * w]), STAGE3=stage(4, [w, 2 * w, 4 * w]),
        STAGE4=stage(3, [w, 2 * w, 4 * w, 8 * w])))))


def synthetic_batch(B, seed, H=256, W=256, J=16):
    """SURVEY.md 8d: N(0,1) images, reference-style Gaussian targets (sigma 2, 13x13, peak 1), 0/1 weights."""
    import numpy as np
    import torch
    rng = np.random.RandomState(seed)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 3, H, W, generator=g)
    h, w = H // 4, W // 4
    t = np.zeros((B, J, h, w), np.float32)
    xs = np.arange(13, dtype=np.float32)
    gauss = np.exp(-((xs[None] - 6) ** 2 + (xs[:, None] - 6) ** 2) / 8.0)
    for b in range(B):
        for j in range(J):
            mx, my = rng.randint(0, w), rng.randint(0, h)
            x0, y0 = mx - 6, my - 6
            gx0, gx1 = max(0, -x0), min(x0 + 13, w) - x0
            gy0, gy1 = max(0, -y0), min(y0 + 13, h) - y0
            t[b, j, max(0, y0):min(y0 + 13, h), max(0, x0):min(x0 + 13, w)] = gauss[gy0:gy1, gx0:gx1]
    tw = (rng.rand(B, J, 1) > 0.2).astype(np.float32)
    return x, torch.from_numpy(t), torch.from_numpy(tw)


def synthetic_boxes(n, seed, W=256):
    """SURVEY.md 8d NMS input: x1,y1 ~ U(0,W), w,h ~ U(8,128), score ~ U(0,1); returned sorted by score descending."""
    import numpy as np
    rng = np.random.RandomState(seed)
    x1, y1 = rng.uniform(0, W, n), rng.uniform(0, W, n)
    d = np.stack([x1, y1, x1 + rng.uniform(8, 128, n), y1 + rng.uniform(8, 128, n), rng.uniform(0, 1, n)], 1).astype(np.float32)
    return d[d[:, 4].argsort()[::-1]].copy()


def workload_config(name, world, batch):
    c = CONFIGS[name]
    # identical in both arms (GPU and `--impl reference`), so that a driver comparing the two lines sees one configuration
    return {"workload": c["workload"], "name": name, "global_batch": batch * world, "per_gpu_batch": batch,
            "parallelism": "dp%d" % world,
            "l2": "per-step working set (activations: several GB) exceeds the 126 MB L2; no flush needed"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [q.strip() for q in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx = float(p[2])
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------------
# CPU legs: the reference's own modules (oracle/_ref) on the host cores -- cpu_baseline and --impl reference.
# The ONLY place bench.py touches oracle/.
# --------------------------------------------------------------------------------------------------
# Fastest (batch per step, threads) of the reference's CPU path on the B200 box's host (128 schedulable CPUs, Xeon 8562Y+),
# from the committed sweep profiles/r2_cpu_thread_sweep.txt (tools/cpu_thread_sweep.py): more threads or larger batches
# are SLOWER per image there (hg_fpd: 6.7 img/s at B=4 / 16 threads, 3.0 at B=8, 1.6 at B=32; 1.1 with 64 threads), so the
# CPU legs run the sample size and thread count the reference is fastest with. FPD_CPU_THREADS / --batch override.
CPU_BEST = {"hg_fpd": (4, 16), "hg_mse_s1": (2, 8), "hrnet_fpd": (8, 16), "hg_infer": (8, 16), "res50_mse": (8, 16)}


def cpu_threads(name=None):
    n = int(os.environ.get("FPD_CPU_THREADS", "0"))
    if n:
        return n
    best = CPU_BEST.get(name, (0, 16))[1]
    return min(best, len(os.sched_getaffinity(0)))


class CpuReference:
    """Builds the reference modules for a config and exposes one() = one step of the reference loop on the CPU."""

    def __init__(self, name, batch, as_written=False, seed=0):
        import torch
        from oracle import ref_modules as R
        c = CONFIGS[name]
        self.c, self.B, self.kind = c, batch, ("reference" if R.available() else "port")
        self.threads = cpu_threads(name)
        torch.set_num_threads(self.threads)
        torch.manual_seed(seed)
        self.as_written = as_written
        if self.kind == "reference":
            if c["family"] == "hourglass":
                mk = lambda fs: R.hourglass().get_pose_net(R.hg_cfg(fs[0], fs[1], c["J"]), True)   # noqa: E731
            elif c["family"] == "resnet":
                mk = lambda n: R.pose_resnet().get_pose_net(R.resnet_cfg(n, c["J"]), False)        # noqa: E731
            else:
                mk = lambda w: R.pose_hrnet().get_pose_net(R.hrnet_cfg(w), False)                  # noqa: E731
            self.student = mk(c["student"])
            self.teacher = mk(c["teacher"]) if c["teacher"] is not None else None
            self.crit = R.loss().JointsMSELoss(use_target_weight=True)
        else:
            self._port_init(c)
        self.x, self.target, self.tw = synthetic_batch(batch, 0, c["H"], c["W"], c["J"])
        if c["kind"] == "train":
            params = list(self.student.parameters()) if self.kind == "reference" else list(self.params.values())
            self.opt = torch.optim.Adam(params, lr=c["lr"])        # lib/utils/utils.py:69-73
            if self.kind == "reference":
                self.student.train()
                if self.teacher is not None:
                    self.teacher.eval()
        else:
            self.student.eval()
            self.boxes = synthetic_boxes(1024, 1)
            if self.kind == "reference":
                inf, tr, ns = R.decode()
                self.dec = (inf.get_max_preds, tr.flip_back, ns["nms"])
            else:
                from oracle import decode_oracle as D
                self.dec = (D.get_max_preds, D.flip_back, D.nms)

    def _port_init(self, c):
        """oracle port (hourglass only): functional restatement driven from a state_dict."""
        import fpd_b200  # noqa: F401
        from fpd_b200.lib.models import hourglass as H
        if c["family"] != "hourglass":
            raise RuntimeError("oracle/_ref is absent and the oracle port of the CPU step covers the hourglass only")
        self.s_sd = {k: v.clone() for k, v in H.get_pose_net(cfg(*c["student"]), True).state_dict().items()}
        self.params = {k: v.requires_grad_(True) for k, v in self.s_sd.items() if v.is_floating_point() and "running" not in k}
        self.s_sd.update(self.params)
        self.t_sd = None
        if c["teacher"] is not None:
            self.t_sd = {k: v.clone() for k, v in H.get_pose_net(cfg(*c["teacher"]), False).state_dict().items()}
        self.student = types.SimpleNamespace(eval=lambda: None)

    def one(self):
        import torch
        c = self.c
        if c["kind"] == "infer":
            return self._infer()
        if self.kind == "port":
            return self._port_train()
        # lib/core/function.py:44-63 (train) / :119-147 (fpd_train), statement for statement (no .cuda())
        outputs = self.student(self.x)
        if self.teacher is not None:
            if self.as_written:      # function.py:120-121: the teacher is neither frozen nor detached
                toutput = self.teacher(self.x)
            else:
                with torch.no_grad():
                    toutput = self.teacher(self.x)
            if isinstance(toutput, list):
                toutput = toutput[-1]
        outs = outputs if isinstance(outputs, list) else [outputs]
        pose = self.crit(outs[0], self.target, self.tw)
        kd = self.crit(outs[0], toutput, self.tw) if self.teacher is not None else None
        for o in outs[1:]:
            pose += self.crit(o, self.target, self.tw)
            if kd is not None:
                kd += self.crit(o, toutput, self.tw)
        loss = pose if kd is None else (1 - 0.5) * pose + 0.5 * kd
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return loss.item()

    def _port_train(self):
        import torch
        from oracle import hourglass_oracle as O
        outs = O.hourglass_net(self.s_sd, self.x, self.c["student"][1], training=True)
        tout = None
        if self.t_sd is not None:
            with torch.no_grad():
                tout = O.hourglass_net(self.t_sd, self.x, self.c["teacher"][1], training=False)[-1]
        loss, _, _ = O.fpd_loss(outs, self.target, self.tw, tout, 0.5)
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return loss.item()

    def _forward(self, x):
        if self.kind == "port":
            from oracle import hourglass_oracle as O
            return O.hourglass_net(self.s_sd, x, self.c["student"][1], training=False)
        return self.student(x)

    def _infer(self):
        """function.py:212-240 + inference.get_max_preds + numpy nms, on the CPU."""
        import numpy as np
        import torch
        get_max_preds, flip_back, nms = self.dec
        with torch.no_grad():
            out = self._forward(self.x)
            out = out[-1] if isinstance(out, list) else out
            xf = torch.from_numpy(np.flip(self.x.numpy(), 3).copy())
            of = self._forward(xf)
            of = of[-1] if isinstance(of, list) else of
            of = torch.from_numpy(flip_back(of.numpy(), MPII_FLIP_PAIRS).copy())
            of[:, :, :, 1:] = of.clone()[:, :, :, 0:-1]
            out = (out + of) * 0.5
        preds, maxvals = get_max_preds(out.numpy())
        keep = nms(self.boxes, 0.6)
        return float(maxvals.sum()) + len(keep)


def time_cpu(name, batch, steps, warmup, max_seconds, as_written=False):
    ref = CpuReference(name, batch, as_written=as_written)
    for _ in range(warmup):
        ref.one()
    t0 = time.perf_counter()
    n = 0
    while n < steps and (n == 0 or time.perf_counter() - t0 < max_seconds):
        ref.one()
        n += 1
    dt = time.perf_counter() - t0
    return batch * n / dt, n, ref.threads, ref.kind


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation on the SAME config, K steps after W warm-ups, each step one
    batch of the configured size (a bounded sample of the workload: one batch per step, K steps)."""
    if rank != 0:
        return
    name = args.config
    c = CONFIGS[name]
    # one step = one bounded sample of the workload: the batch size the CPU path is FASTEST with on this host (CPU_BEST)
    B = args.batch or CPU_BEST[name][0]
    ips, n, threads, kind = time_cpu(name, B, args.steps, args.warmup, max_seconds=float(os.environ.get("FPD_CPU_MAX_S", "900")))
    sample = ("%s: the reference's own lib/models + lib/core/loss modules (oracle/_ref), loop body of lib/core/function.py, "
              "teacher under no_grad, %d images per step (the sample size and thread count the CPU path is fastest with, "
              "profiles/r2_cpu_thread_sweep.txt), %d timed steps after %d warm-up, fp32, %d threads" % (
                  kind, B, n, args.warmup, threads))
    line = {"impl": "reference", "metric": "images/sec", "value": ips, "unit": "images/s", "n_gpus": args.gpus,
            "steps": n, "warmup": args.warmup, "ms_per_step": 1000.0 * B / ips, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(name, args.gpus, c["batch"]),
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if c["kind"] == "train" and c["teacher"] is not None and os.environ.get("FPD_CPU_AS_WRITTEN", "0") != "0":
        ips2, n2, _, _ = time_cpu(name, B, max(1, args.steps // 2), 1, 600.0, as_written=True)
        line["cpu_baseline"]["as_written"] = {"value": ips2, "steps": n2,
                                              "note": "teacher back-propagated as in function.py:120-121,146"}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def time_dominant_kernel(B, roof):
    """Live CUDA-event timing of the dominant kernel (conv_tc_h_kernel<f16>: tcgen05 kind::f16 implicit-GEMM conv, halo
    tile fetched + BN/ReLU-transformed + split once per channel block, taps as shifted copies into TMEM) on the config's
    heaviest shape, 3xFP16. Eight launches per timed region over four rotating input/output sets (larger than the 126 MB
    L2 at the bench batch sizes, plus an explicit L2 flush before each group), replayed from a CUDA graph so that host
    launch cost is not in the region -- the same way the kernel runs inside the step."""
    import torch
    from fpd_b200 import ops
    H, W, Cin, Cout, k = roof["h"], roof["w"], roof["cin"], roof["cout"], roof["k"]
    g = torch.Generator(device="cuda").manual_seed(0)
    xs = [torch.randn(B, H, W, Cin, device="cuda", generator=g) for _ in range(4)]
    ys = [torch.empty(B, H, W, Cout, device="cuda") for _ in range(4)]
    w = torch.randn(Cout, Cin, k, k, device="cuda", generator=g) * 0.03
    w_hi, w_lo = ops.weight_prep_f16(w)
    mean = torch.zeros(Cin, device="cuda")
    scale = torch.ones(Cin, device="cuda")
    shift = torch.zeros(Cin, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def launch(i):
        ops.conv2d_tc_h(xs[i % 4], w_hi, w_lo, k, mean=mean, scale=scale, shift=shift, relu=True, out=ys[i % 4])
    for i in range(4):
        launch(i)
    torch.cuda.synchronize()
    reps, per, tot = 5, 8, 0.0
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            for i in range(per):
                launch(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for _ in range(reps):
        flush.zero_()  # L2 flush before each timed group
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    ms = tot / (reps * per)
    flops = 2.0 * B * H * W * Cin * Cout * k * k
    return ms, flops


DUMP_MAX_ELEMS = 4 << 20     # per array: at most 16 MB, so that one dump stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy: float32 as it is, anything else (integer indices) as float64, which holds
    it exactly. An array of more than DUMP_MAX_ELEMS entries is flattened and reduced to a fixed sample of that many: the
    same seeded, sorted index set on every run, so that dumps of two builds compare entry for entry."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu()
        if a.numel() > DUMP_MAX_ELEMS:
            pick = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            a = a.reshape(-1)[pick]
        a = a.numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def build_models(name, dev):
    import torch
    import fpd_b200  # noqa: F401
    c = CONFIGS[name]
    torch.manual_seed(0)
    if c["family"] == "hourglass":
        from fpd_b200.lib.models import hourglass as H
        student = H.get_pose_net(cfg(c["student"][0], c["student"][1], c["J"]), True).to(dev)
        teacher = H.get_pose_net(cfg(c["teacher"][0], c["teacher"][1], c["J"]), False).to(dev) if c["teacher"] else None
    elif c["family"] == "resnet":
        from fpd_b200.lib.models import pose_resnet as H
        student = H.get_pose_net(resnet_cfg(c["student"], c["J"]), False).to(dev)
        teacher = H.get_pose_net(resnet_cfg(c["teacher"], c["J"]), False).to(dev) if c["teacher"] else None
    else:
        from fpd_b200.lib.models import pose_hrnet as H
        student = H.get_pose_net(hrnet_cfg(c["student"], c["J"]), False).to(dev)
        teacher = H.get_pose_net(hrnet_cfg(c["teacher"], c["J"]), False).to(dev) if c["teacher"] else None
    return student, teacher


def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import fpd_b200  # noqa: F401
    from fpd_b200.train_step import FPDTrainStep

    name = args.config
    c = CONFIGS[name]
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch or c["batch"]
    student, teacher = build_models(name, dev)
    if world > 1:  # identical replicas: broadcast rank 0's weights once (no per-step broadcast, unlike DataParallel)
        for t in list(student.parameters()) + list(student.buffers()):
            dist.broadcast(t.data, 0)
    x, target, tw = synthetic_batch(B, 1000 + rank, c["H"], c["W"], c["J"])
    xh, th, wh = x.pin_memory(), target.pin_memory(), tw.pin_memory()
    xd, td, wd = xh.to(dev), th.to(dev), wh.to(dev)
    graph_ok = not args.no_graph
    extra = {}

    if c["kind"] == "train":
        step = FPDTrainStep(student, teacher, alpha=0.5, lr=c["lr"], use_graph=graph_ok)
        try:
            step.step(xd, td, wd, next_x=xd)
        except Exception as exc:            # a shape the graph capture cannot take: measure eagerly and say so
            if not graph_ok:
                raise
            extra["graph_fallback"] = repr(exc)[:200]
            torch.cuda.synchronize()
            student, teacher = build_models(name, dev)
            step = FPDTrainStep(student, teacher, alpha=0.5, lr=c["lr"], use_graph=False)
            graph_ok = False
        run_dev = lambda: step.step(xd, td, wd, next_x=xd)                   # noqa: E731
        loss_host = torch.empty(3, dtype=torch.float32).pin_memory()

        def run_e2e():
            losses = step.step(xh, th, wh, next_x=xh)     # pinned-host batch crosses PCIe inside the step
            loss_host.copy_(losses, non_blocking=False)   # the loss the training loop logs: D2H every step
        h2d = (xh.numel() + th.numel() + wh.numel()) * 4
        d2h = 12
        launches = lambda: int(step.launches_per_step or 0)                  # noqa: E731
        final = lambda: float(loss_host[2])                                   # noqa: E731
        # the step's result: its losses (pose, kd, total), the gradient it applied and the student's weights and BatchNorm
        # running statistics after its update (flat, in module order)
        outputs = lambda: {"losses": step.losses, "grad": step.flat.grad, "weights": step.flat.flat,   # noqa: E731
                           "bn_running": torch.cat([b.reshape(-1) for b in student.buffers() if b.is_floating_point()])}
    else:
        from fpd_b200.infer_step import FlipTestInference
        boxes = torch.from_numpy(synthetic_boxes(1024, 1)).to(dev)
        inf = FlipTestInference(student, MPII_FLIP_PAIRS, shift_heatmap=True, flip_test=c.get("flip", True),
                                use_graph=graph_ok, want_avg=False)
        last = {}

        def run_dev():
            last["r"] = inf(xd, boxes, 0.6)
        idx_host = torch.empty(B, c["J"], dtype=torch.int32).pin_memory()
        max_host = torch.empty(B, c["J"], dtype=torch.float32).pin_memory()
        keep_host = torch.empty(1024, dtype=torch.int32).pin_memory()

        def run_e2e():
            r = inf(xh, boxes, 0.6, next_x=xh)     # the next batch crosses PCIe under this one (same bytes per step)
            idx_host.copy_(r["idx"], non_blocking=True)
            max_host.copy_(r["maxval"], non_blocking=True)
            keep_host.copy_(r["nms_keep"], non_blocking=False)
        h2d = xh.numel() * 4
        d2h = idx_host.numel() * 4 + max_host.numel() * 4 + keep_host.numel() * 4
        launches = lambda: int(getattr(inf, "launches", 0))                  # noqa: E731
        final = lambda: float(max_host.sum())                                # noqa: E731
        outputs = lambda: {"idx": last["r"]["idx"], "maxval": last["r"]["maxval"],                   # noqa: E731
                           "nms_keep": last["r"]["nms_keep"][:int(last["r"]["nms_num"])]}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        run_dev()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total = timed(run_dev, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs())
    ms_step = ms_total / args.steps
    value = world * B / (ms_step / 1000.0)

    # ---- end to end: pinned-host inputs copied H2D every step, result read back D2H every step
    for _ in range(2):
        run_e2e()
    ms_e2e = timed(run_e2e, args.steps) / args.steps
    e2e_value = world * B / (ms_e2e / 1000.0)

    if rank != 0:
        _finish(world, dist)
        return

    peaks, peak_src = measured_peaks()
    conf = workload_config(name, world, B)
    run_info = {"cuda_graph": graph_ok, "final_result": final()}
    run_info.update(extra)
    line = {"metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            # forward + data-gradient convs: 3xFP16 (fp16 hi/lo operand pairs, fp32 accumulate); weight gradients: 3xTF32;
            # both fp32-grade (parity <= 1e-3 against the fp32 reference). FPD_PRECISION=tf32 = single-pass TF32.
            "dtype": "f16x3+tf32x3" if os.environ.get("FPD_PRECISION", "tf32x3") != "tf32" else "tf32",
            "data": "synthetic", "config": conf,
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e},
            "gpu_launches": launches() * args.steps, "clocks": clocks, "run_info": run_info}
    step_frac = value / world * c["flop_per_image"] / 1e12 / peaks["bf16_tflops_sustained"]
    try:
        k_ms, k_flops = time_dominant_kernel(B, c["roof"])
        f16_peak = peaks["bf16_tflops"]  # kind::f16 runs at the bf16 rate; burst figure: the kernel is timed alone
        ach = k_flops / (k_ms * 1e-3) / 1e12
        r = c["roof"]
        line["roofline"] = {"bound": "tensor", "achieved": ach, "peak": f16_peak, "unit": "TFLOP/s",
                            "frac": ach / f16_peak,
                            "traffic": CONV_H_3X3_DRAM_BYTES if (name == "hg_fpd" and B == 32) else None,
                            "kernel": "conv_tc_h_kernel<f16> %dx%d %d->%d @%dx%d B=%d (3xFP16: 3 MMA passes per algorithmic "
                                      "FLOP; executed-MMA fraction of peak = 3 x frac)" % (r["k"], r["k"], r["cin"], r["cout"],
                                                                                           r["h"], r["w"], B),
                            "kernel_ms": k_ms, "peak_source": peak_src + ", kind::f16 = bf16 rate",
                            # best shape above; the whole step's algorithmic conv FLOP/s over the sustained peak:
                            "step_frac_of_f16_peak": step_frac,
                            # launch-weighted average of the dominant kernel over ALL its launches in a step (conv FLOPs of the
                            # step / summed kernel time), from the committed launch list -- see profiles/README.md
                            "frac_launch_weighted": LAUNCH_WEIGHTED.get(name)}
    except Exception as exc:  # never lose the headline line to a side measurement
        line["roofline"] = {"error": repr(exc), "step_frac_of_f16_peak": step_frac}
    if world == 1 and not args.no_cpu_baseline:
        try:
            cb = min(B, CPU_BEST[name][0])
            ips, n, threads, kind = time_cpu(name, cb, steps=4, warmup=1, max_seconds=25.0)
            line["cpu_baseline"] = {"value": ips, "unit": "images/s", "cores": threads, "kind": kind,
                                    "sample": "the reference's own modules on the host cores: %d timed steps of batch %d of the "
                                              "same workload (teacher under no_grad), fp32, %d threads; `--impl reference` "
                                              "runs the full batch" % (n, cb, threads)}
        except Exception as exc:
            line["cpu_baseline"] = {"error": repr(exc)}
    print(json.dumps(line), flush=True)
    _finish(world, dist)


def _finish(world, dist):
    """Leave together and for sure: a last barrier (the other ranks wait for rank 0's side measurements), then a hard exit.
    Interpreter finalisation -- and, with NCCL collectives captured inside live CUDA graphs (FPD_BN_SYNC=1), even
    destroy_process_group() -- has been seen to hang a rank for minutes after its work was done (r2 2-GPU runs), which a
    driver waiting for torchrun to exit would count as the job's time. The OS reclaims the communicators."""
    if world > 1:
        try:
            dist.barrier()
            import torch
            torch.cuda.synchronize()
        except Exception:
            pass
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


# launch-weighted roofline fraction of conv_tc_h_kernel over one whole step (all its launches): conv FLOPs it executes
# in the step / its summed duration / peak. Filled from profiles/<tag>_launches.csv.gz by tools/summarize_profiles.py.
# r2: 2.30 TFLOP of forward + data-gradient convolutions in 24.64 ms summed over its 765 launches (ncu launch list,
# profiles/r2_launches_summary.md: cold caches, serialised; the warm CUPTI sum of profiles/r2_step_cupti.txt gives 0.064)
LAUNCH_WEIGHTED = {"hg_fpd": 0.057}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="hg_fpd", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the config's)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
