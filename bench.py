"""Benchmark of the SC-SfMLearner training hot path (BASELINE.json metric: train-step frames/sec at
256x832 ResNet-18 on 1/2/4/8 B200; warp-loss HBM GB/s).

    python bench.py --gpus N --steps K --warmup W [--config kitti_r18|kitti_r50|nyu_r18]     # our arm (torchrun launches N>1)
                    [--dump-outputs DIR]                                                      # + the last timed step's outputs
    python bench.py --impl reference --gpus N --steps K --warmup W                           # the reference's own CPU path

A "step" is one complete optimisation step (train.py:254-282): 1 + n_ref DispResNet and 2 n_ref PoseResNet
forward/backward calls, fused photometric/geometry/smoothness losses, gradient all-reduce (N>1), Adam, on a synthetic
batch (weak scaling: the per-GPU batch is fixed).  One JSON line is printed by rank 0.

  config kitti_r18 (default, BASELINE configs 2/3): DispResNet18+PoseResNet18, 256x832, 2 refs, 4 frames per GPU
  config kitti_r50 (BASELINE config 4):             DispResNet50+PoseResNet50, 256x832, 2 refs, 2 frames per GPU
  config nyu_r18   (BASELINE config 5):             DispResNet18+PoseResNet18, 256x320, 1 ref,  8 frames per GPU

`value` is measured in the convolution mode --conv-mode (default tf32x3: the tcgen05 split-accumulate mode that meets
the 1e-4 parity contract, tests/test_train_step_gpu.py::test_full_size_benchmarked_step_vs_oracle); the single-product
TF32 figure (cuDNN's default arithmetic) is reported beside it as `tf32`.  Extras in the line: `warp_loss` (CUDA-event
timed loss kernels as HBM GB/s, metric half 2), `gpu_reference` (the unmodified reference step through stock PyTorch/cuDNN
on the same GPU, baseline/ref_driver.py), `cpu_baseline` (the unmodified reference on the host cores).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "sc-sfmlearner-release_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

# name: disp layers, pose layers, H, W, n_ref, per-GPU batch, intrinsics, conv GFLOP per frame of a train step (3x forward,
# SURVEY.md section 8d / BASELINE.md section 4), workload label
CONFIGS = {
    "kitti_r18": dict(dl=18, pl=18, H=256, W=832, n_ref=2, batch=4, kind="kitti", gflop=453.4,
                      label="DispResNet18+PoseResNet18 full train step, batch 4 per GPU, 256x832 synthetic KITTI triplets (configs 2/3)"),
    "kitti_r50": dict(dl=50, pl=50, H=256, W=832, n_ref=2, batch=2, kind="kitti", gflop=953.4,
                      label="DispResNet50+PoseResNet50 full train step, batch 2 per GPU, 256x832 synthetic KITTI triplets (config 4)"),
    "nyu_r18": dict(dl=18, pl=18, H=256, W=320, n_ref=1, batch=8, kind="nyu", gflop=103.2,
                    label="DispResNet18+PoseResNet18 full train step, batch 8 per GPU, 256x320 synthetic NYU pairs, 1 ref (config 5)"),
}
METRIC = {"kitti_r18": "train-step frames/sec at 256x832 ResNet18 (DispResNet18+PoseResNet18, fwd+bwd+losses+Adam)",
          "kitti_r50": "train-step frames/sec at 256x832 ResNet50 (DispResNet50+PoseResNet50, fwd+bwd+losses+Adam)",
          "nyu_r18": "train-step frames/sec at 256x320 ResNet18 (DispResNet18+PoseResNet18, 1 ref, fwd+bwd+losses+Adam)"}
DTYPE = {"fp32": "fp32", "tf32": "tf32", "tf32x3": "tf32x3 (3xTF32 split-accumulate, fp32-level)"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "MEASURED_PEAKS.json (of measured)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "B200_PROFILING.md fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms during the timed region."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_batch(cfg, rank, pinned):
    from scsfm import synth
    tgt, refs, K = synth.triplet(1234 + rank, cfg["batch"], cfg["H"], cfg["W"], cfg["n_ref"], cfg["kind"])
    if pinned:
        tgt, refs, K = tgt.pin_memory(), [r.pin_memory() for r in refs], K.pin_memory()
    return tgt, refs, K


# --------------------------------------------------------------------------------------------------
# reference harness (baseline/ref_driver.py drives the UNMODIFIED reference train.train())
# --------------------------------------------------------------------------------------------------
def usable_cores():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota, not just os.cpu_count()
    (the GPU box reports 128 CPUs but oversubscribing a quota-limited container makes torch crawl)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except (OSError, ValueError):
        pass
    try:
        quota, period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()), int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if quota > 0:
            n = min(n, max(1, quota // period))
    except (OSError, ValueError):
        pass
    return max(1, n)


def run_ref_driver(device, config, steps, warmup, threads=0, budget_s=0.0, extra=(), timeout=900):
    """The unmodified reference loop in its own process (so that the CPU arm can hide the GPU from it).  Returns the
    driver's JSON dict, or {"unavailable": why}."""
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_driver.py"), "--device", device, "--config", config, "--steps", str(steps),
           "--warmup", str(warmup), "--threads", str(threads), "--budget-s", str(budget_s)] + list(extra)
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return {"unavailable": "reference driver timed out after %d s" % timeout}
    for ln in reversed(out.stdout.splitlines()):
        ln = ln.strip()
        if ln.startswith("{") and ln.endswith("}"):
            try:
                return json.loads(ln)
            except ValueError:
                continue
    return {"unavailable": "reference driver failed (rc %d): %s" % (out.returncode, (out.stderr or out.stdout)[-300:].replace("\n", " | "))}


def cpu_oracle_port(cfg, steps, budget_s):
    """Fallback CPU baseline when baseline/_ref is absent: the oracle port of the step (oracle/step.py)."""
    import time
    from oracle import geometry as OGEO
    from oracle import nets as N
    from oracle import step as OS
    from scsfm import synth
    OGEO.USE_LIBRARY_KERNELS = True        # F.grid_sample / F.avg_pool2d, exactly what the reference calls on CPU
    cores = usable_cores()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    disp, pose = N.DispResNet(cfg["dl"]).train(), N.PoseResNet(cfg["pl"]).train()
    opt = OS.make_optimizer(disp, pose, lr=1e-4)
    tgt, refs, K = synth.triplet(1234, cfg["batch"], cfg["H"], cfg["W"], cfg["n_ref"], cfg["kind"])

    def one():
        t0 = time.perf_counter()
        OS.train_step(disp, pose, opt, tgt, refs, K, num_scales=1, with_ssim=1, with_mask=1, with_auto_mask=1, padding_mode="zeros")
        return time.perf_counter() - t0
    probe = one()
    steps = max(1, min(steps, int(budget_s / max(probe, 1e-6))))
    total = sum(one() for _ in range(steps))
    return {"value": round(cfg["batch"] * steps / total, 4), "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": "%d timed step(s) of the oracle port of train.py:259-282 at batch %d (%d torch CPU threads)" % (steps, cfg["batch"], cores),
            "ms_per_step": round(1e3 * total / steps, 1)}


def cpu_baseline(config, cfg, steps, warmup, budget_s):
    """The reference's own train.train() on the host cores (all usable cores, fixed -- no auto-picking), a bounded sample."""
    cores = usable_cores()
    r = run_ref_driver("cpu", config, steps, warmup, threads=cores, budget_s=budget_s)
    if "unavailable" in r:
        base = cpu_oracle_port(cfg, steps, budget_s)
        base["note"] = "baseline/_ref unavailable (%s): oracle port timed instead" % r["unavailable"]
        return base
    return {"value": r["frames_per_s"], "unit": "frames/s", "cores": r["threads"], "kind": "reference",
            "sample": "%d timed step(s) (after %d warm-up) of the UNMODIFIED reference train.train() (train.py:235-299, autograd anomaly "
                      "mode on as shipped) at batch %d, config %s, fp32, torch %s CPU with %d threads (= usable host cores)"
                      % (r["steps"], r["warmup"], r["batch"], config, r["torch"], r["threads"]),
            "ms_per_step": r["ms_per_step"]}


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def input_pipeline_extra(cfg, dev, peaks, iters=20):
    """SURVEY.md 8 row f-3: the training transforms of one batch (flip, zoom-crop, to-tensor, normalise) on the GPU
    (scsfm.augment.GpuAugment: uint8 frames in, normalised float NCHW out) beside the reference's host chain
    (custom_transforms.py through PIL / numpy / torch, per sample, one core -- what each of its `-j 4` loader workers runs)."""
    import random
    import numpy as np
    from scsfm.augment import GpuAugment
    B, H, W, n_img = cfg["batch"], cfg["H"], cfg["W"], cfg["n_ref"] + 1
    g = np.random.default_rng(5)
    low = g.integers(0, 256, (n_img, B, H // 8 + 1, W // 8 + 1, 3)).astype(np.float32)
    frames = np.clip(np.kron(low, np.ones((1, 1, 8, 8, 1), np.float32))[:, :, :H, :W] + g.normal(0, 20, (n_img, B, H, W, 3)), 0, 255).astype(np.uint8)
    K = np.tile(np.array([[0.58 * W, 0, 0.49 * W], [0, 1.92 * H, 0.47 * H], [0, 0, 1]], np.float32), (B, 1, 1))
    h_frames = torch.from_numpy(frames).pin_memory()
    d_frames = h_frames.to(dev)
    aug = GpuAugment(device=dev)
    random.seed(0)
    np.random.seed(0)
    for _ in range(3):
        aug(d_frames, K)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        aug(d_frames, K)
    e1.record()
    torch.cuda.synchronize()
    ms_dev = e0.elapsed_time(e1) / iters
    t0 = time.perf_counter()
    for _ in range(iters):
        out, _k = aug(h_frames, K)
        torch.cuda.synchronize()
    ms_e2e = (time.perf_counter() - t0) * 1e3 / iters
    alg = 15.0 * n_img * B * H * W           # 3 B/pixel uint8 in + 12 B/pixel float32 out
    res = {"frames_per_s": round(B / (ms_dev * 1e-3), 1), "ms_per_batch": round(ms_dev, 4), "gbs": round(alg / (ms_dev * 1e-3) / 1e9, 1),
           "frac_of_hbm_peak": round(alg / (ms_dev * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
           "e2e_frames_per_s": round(B / (ms_e2e * 1e-3), 1), "e2e_ms_per_batch": round(ms_e2e, 4), "h2d_bytes_per_batch": int(frames.size),
           "how": "%d batches of %d samples x %d frames %dx%d; device: CUDA events around the whole call (host draws + 2 small uploads + 2 kernels), "
                  "frames resident; e2e: uint8 frames from pinned host memory, synchronised per batch; algorithmic 15 B/pixel" % (iters, B, n_img, H, W)}
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    try:
        sys.path.insert(0, ref_dir)
        import custom_transforms as T       # the reference's (baseline/_ref: unmodified copy made by __graft_entry__.install_reference)
        chain = T.Compose([T.RandomHorizontalFlip(), T.RandomScaleCrop(), T.ArrayToTensor(), T.Normalize(mean=[0.45] * 3, std=[0.225] * 3)])
        nthreads = torch.get_num_threads()
        torch.set_num_threads(1)
        try:
            t0 = time.perf_counter()
            n = 0
            while n < 8 or time.perf_counter() - t0 < 2.0:
                b = n % B
                chain([frames[i, b].astype(np.float32) for i in range(n_img)], np.copy(K[b]))
                n += 1
            per = (time.perf_counter() - t0) / n
        finally:
            torch.set_num_threads(nthreads)
        res["reference_host_chain"] = {"frames_per_s_per_worker": round(1.0 / per, 1), "ms_per_sample": round(per * 1e3, 3), "samples": n,
                                       "what": "unmodified custom_transforms chain (PIL bicubic + numpy + torch) on one core, decode excluded"}
    except Exception as e:      # noqa: BLE001
        res["reference_host_chain"] = {"unavailable": repr(e)}
    finally:
        if ref_dir in sys.path:
            sys.path.remove(ref_dir)
    return res


def run_ours(args):
    import models
    from scsfm import lib as L
    from scsfm.trainer import Trainer

    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.load()          # fails loudly if libscsfm.so is missing
    h_tgt, h_refs, h_K = synthetic_batch(cfg, rank, pinned=True)
    d_tgt, d_refs, d_K = h_tgt.to(dev), [r.to(dev) for r in h_refs], h_K.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    B = cfg["batch"]

    def make_trainer(mode, overlap=True):
        torch.manual_seed(0)
        disp, pose = models.DispResNet(cfg["dl"], False).to(dev).train(), models.PoseResNet(cfg["pl"], False).to(dev).train()
        return Trainer(disp, pose, lr=1e-4, num_scales=1, with_ssim=1, with_mask=1, with_auto_mask=1, padding_mode="zeros",
                       w1=1.0, w2=0.1, w3=0.5, distributed=world > 1, conv_mode=mode, overlap_nets=overlap and bool(args.overlap_nets),
                       overlap_wgrad=overlap and bool(args.overlap_wgrad))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, before=None):
        """device time of `steps` calls (`before` run, then L2 flushed, ahead of each, outside the events), max over ranks, in ms"""
        evs = []
        barrier()
        for _ in range(steps):
            if before is not None:
                before()
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        barrier()
        total = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        return float(total)

    # The per-family / per-kernel passes run the step SERIALLY (one stream): CUDA events around a launch only measure that
    # kernel when nothing else runs beside it.  The timed region below uses the overlapped step (two networks and the weight
    # gradients on side streams).
    trainer = make_trainer(args.conv_mode, overlap=False)
    # ---- warm-up with full per-family profiling: finds the dominant kernel family and times the loss kernels ------
    trainer.step(d_tgt, d_refs, d_K)          # first step unprofiled: lazy kernel loading, allocations, Adam state
    torch.cuda.synchronize()
    nprof = max(args.warmup, 3)
    L.PROF.update(enabled=True, only=None, events=[])
    for _ in range(nprof):
        flush.zero_()
        trainer.step(d_tgt, d_refs, d_K)
    torch.cuda.synchronize()
    fam = {}
    for family, work, e0, e1, _ in L.PROF["events"]:
        t = fam.setdefault(family, [0.0, 0.0, 0])
        t[0] += e0.elapsed_time(e1); t[1] += work; t[2] += 1
    dominant = max(fam, key=lambda k: fam[k][0])
    breakdown = {k: round(v[0] / nprof, 3) for k, v in sorted(fam.items(), key=lambda kv: -kv[1][0])}
    peaks = load_peaks()
    # metric half 2: the fused warp / loss / stencil kernels as achieved HBM bandwidth (algorithmic bytes of SURVEY.md 8d:
    # pair fwd 32 B/px, pair bwd 44 B/px per pair-direction; smoothness fwd 16, bwd 20 B/px per image) over CUDA-event time
    warp_loss = {}
    for k in ("pair_fwd", "pair_bwd", "smooth_fwd", "smooth_bwd"):
        if k in fam and fam[k][0] > 0:
            gbs = fam[k][1] / (fam[k][0] * 1e-3) / 1e9
            warp_loss[k] = {"gbs": round(gbs, 1), "frac": round(gbs / peaks["hbm_gbs"], 4), "us_per_step": round(1e3 * fam[k][0] / nprof, 1),
                            "bytes_per_step": round(fam[k][1] / nprof)}
    tot_b = sum(fam[k][1] for k in warp_loss)
    tot_t = sum(fam[k][0] for k in warp_loss)
    if tot_t > 0:
        warp_loss["all"] = {"gbs": round(tot_b / (tot_t * 1e-3) / 1e9, 1), "frac": round(tot_b / (tot_t * 1e-3) / 1e9 / peaks["hbm_gbs"], 4)}
        warp_loss["peak_gbs"] = peaks["hbm_gbs"]
        warp_loss["how"] = ("algorithmic bytes (SURVEY.md 8d) / CUDA-event time of the launches inside %d eager steps, L2 flushed before "
                            "each step; each family's time includes its small finalize / statistics launches" % nprof)

    # ---- per-kernel roofline pass: the same step, eager, CUDA events only around the dominant family ------
    L.PROF.update(enabled=True, only={dominant}, events=[])
    ms_eager = timed(lambda: trainer.step(d_tgt, d_refs, d_K), args.steps)
    dom_ms = sum(e[2].elapsed_time(e[3]) for e in L.PROF["events"])
    dom_work = sum(e[1] for e in L.PROF["events"])
    dom_n = len(L.PROF["events"])
    L.PROF.update(enabled=False, only=None, events=[])
    del trainer
    trainer = make_trainer(args.conv_mode)
    initial = trainer.optimizer.snapshot()      # seeded initialisation, no step taken yet
    for _ in range(2):
        trainer.step(d_tgt, d_refs, d_K)

    # ---- timed region: device-resident inputs; the whole step is one CUDA-graph replay ---------
    def capture(tr):
        if args.no_graph:
            return False
        if world == 1:
            tr.capture(d_tgt, d_refs, d_K)
            return True
        try:      # data-parallel step incl. the NCCL all-reduce on the side stream as one CUDA graph; eager on any capture error
            tr.capture(d_tgt, d_refs, d_K, allow_distributed=True)
            ok = torch.ones(1, device=dev)
        except Exception as e:      # noqa: BLE001
            print("rank %d: graph capture of the data-parallel step failed, running eagerly: %r" % (rank, e), file=sys.stderr)
            ok = torch.zeros(1, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)       # every rank must take the same path
        if float(ok) == 0:
            tr.drop_graph()
            return False
        return True
    graphed = capture(trainer)
    # Every timed step starts from the seeded initial parameters and optimizer state, restored ahead of the step, before the L2
    # flush and outside the timed events: the loss reductions and BatchNorm statistics accumulate with atomics, and a chain of
    # Adam steps would carry their last-bit differences into everything after them.  So each timed step is the same work on
    # the same values, run after run, and --dump-outputs can compare two builds output for output.
    reset_launches = [0]

    def reset():
        n0 = L.launch_count()
        trainer.optimizer.restore(initial)
        for n in trainer.optimizer.nets:
            n.refresh_operand_weights()        # the operand mirrors the next step reads (Adam writes them during replays)
        reset_launches[0] += L.launch_count() - n0
    launches0 = L.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    last = []
    ms = timed(lambda: last.append(trainer.step(d_tgt, d_refs, d_K)), args.steps, before=reset)
    clocks = sampler.stop() if rank == 0 else None
    launches = trainer.launches_per_step * args.steps if graphed else (L.launch_count() - launches0 - reset_launches[0])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, last[-1])

    # ---- end to end: pinned host inputs copied in, loss read back, every step ----------------------
    result = torch.empty(4, dtype=torch.float32).pin_memory()

    def make_e2e(tr):
        def e2e_step():
            t = h_tgt.to(dev, non_blocking=True)
            r = [x.to(dev, non_blocking=True) for x in h_refs]
            k = h_K.to(dev, non_blocking=True)
            out = tr.step(t, r, k)
            result.copy_(torch.stack(out), non_blocking=True)
            torch.cuda.current_stream().synchronize()       # the user reads the loss (train.py:277)
        return e2e_step
    e2e_step = make_e2e(trainer)
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    h2d = sum(t.numel() * 4 for t in [h_tgt, h_K] + h_refs)
    frames = B * world * args.steps

    # ---- the single-product TF32 mode beside it (cuDNN's default arithmetic; NOT the parity mode) ---------
    tf32_extra = None
    if args.conv_mode != "tf32" and not args.no_tf32_extra:
        del trainer
        t2 = make_trainer("tf32")
        for _ in range(3):
            t2.step(d_tgt, d_refs, d_K)
        g2 = capture(t2)
        steps2 = max(5, args.steps // 2)
        ms2 = timed(lambda: t2.step(d_tgt, d_refs, d_K), steps2)
        e2 = make_e2e(t2)
        e2()
        ms2e = timed(e2, steps2)
        tf32_extra = {"value": round(B * world * steps2 / (ms2 * 1e-3), 3), "unit": "frames/s", "ms_per_step": round(ms2 / steps2, 3),
                      "e2e": round(B * world * steps2 / (ms2e * 1e-3), 3), "steps": steps2, "cuda_graph": g2,
                      "note": "conv_mode tf32: one TF32 product per MAC (what cuDNN does for the reference by default); parameter "
                              "gradients ~1e-3..1e-2 from fp32, i.e. outside the 1e-4 parity contract -- reported, not the headline"}
        del t2

    if rank != 0:
        finish(world)
        return
    is_conv = dominant.startswith("conv")
    if is_conv:
        achieved = dom_work / (dom_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": round(achieved, 2), "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                "frac": round(achieved / peaks["tflops_sustained"], 5), "traffic": None}
    else:
        achieved = dom_work / (dom_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(achieved / peaks["hbm_gbs"], 5), "traffic": None}
    try:        # measured DRAM traffic per launch of the family's kernels (ncu capture summarised by tools/ncu_summarise.py)
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic_by_family.json")))
        if dominant in tr and args.config == "kitti_r18":
            roof["traffic"] = tr[dominant]["dram_bytes_per_launch"]
            roof["traffic_source"] = tr["_source"]
    except (OSError, ValueError, KeyError):
        pass
    roof.update(kernel=dominant, launches_timed=dom_n, avg_launch_us=round(1e3 * dom_ms / max(dom_n, 1), 2),
                algorithmic_flops_or_bytes_per_launch=round(dom_work / max(dom_n, 1)),
                share_of_step=round(dom_ms / ms_eager, 4), peak_source=peaks["source"],
                share_note="share of the SERIAL eager step (one stream); the timed step overlaps the two networks and the weight gradients",
                note="achieved = ALGORITHMIC FLOPs (2*M*N*K per conv pass, the same count in every conv mode: the 3 split-accumulate "
                     "products of tf32x3 are not counted as extra work) or bytes of the family / its CUDA-event time over the same K "
                     "steps run eagerly (events cannot be recorded inside the replayed CUDA graph); sustained bf16 peak is the "
                     "denominator because the kernel runs inside a long step")
    line = {
        "metric": METRIC[args.config],
        "value": round(frames / (ms * 1e-3), 3), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": nprof + 1, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[args.conv_mode],
        "data": "synthetic", "impl": "ours",
        "config": {"workload": cfg["label"], "name": args.config, "global_batch": B * world, "height": cfg["H"], "width": cfg["W"],
                   "n_ref": cfg["n_ref"], "parallelism": "dp%d" % world, "conv_mode": args.conv_mode,
                   "l2": "flushed (256 MiB write) before every step", "cuda_graph": graphed, "overlap_nets": bool(args.overlap_nets), "overlap_wgrad": bool(args.overlap_wgrad),
                   "serial_eager_ms_per_step": round(ms_eager / args.steps, 3), "loss_flags": "num_scales=1 ssim=1 mask=1 auto_mask=1 zeros"},
        "e2e": {"value": round(frames / (ms_e2e * 1e-3), 3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 16, "ms_per_step": round(ms_e2e / args.steps, 3)},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roof,
        "warp_loss": warp_loss,
        "step_breakdown_ms": breakdown,
        "conv_gflop_per_frame_train": cfg["gflop"],
        "step_tflops": round(cfg["gflop"] * frames / (ms * 1e-3) / 1e3, 2),
    }
    if tf32_extra is not None:
        line["tf32"] = tf32_extra
    if world == 1 and not args.no_gpu_reference:
        # the "existing Blackwell kernel" bar (SURVEY.md 2.3, BASELINE.md 3): the UNMODIFIED reference step through stock
        # PyTorch/cuDNN on this same GPU, as shipped (cudnn.benchmark on, TF32 convolutions allowed, anomaly mode on) and with
        # anomaly mode off
        torch.cuda.empty_cache()
        gref = {}
        for name, extra in (("as_shipped", ["--anomaly", "1"]), ("anomaly_off", ["--anomaly", "0"]),
                            ("anomaly_off_fp32", ["--anomaly", "0", "--tf32", "0"])):
            r = run_ref_driver("cuda", args.config, max(5, min(args.steps, 20)), 3, extra=extra, timeout=600)
            gref[name] = r if "unavailable" in r else {"frames_per_s": r["frames_per_s"], "ms_per_step": r["ms_per_step"], "steps": r["steps"],
                                                       "tf32": r["tf32"], "anomaly": r["anomaly"]}
        gref["what"] = ("unmodified reference train.train() (baseline/_ref, stock torch %s / cuDNN, cudnn.benchmark=True) on the same B200, "
                        "wall clock per iteration incl. its own host syncs and CSV write; inputs resident on the host as in train.py:254-257"
                        % torch.__version__)
        line["gpu_reference"] = gref
    if world == 1 and not args.no_input_pipeline:
        try:
            line["input_pipeline"] = input_pipeline_extra(cfg, dev, peaks)
        except Exception as e:      # noqa: BLE001  (an extra: never lose the bench line over it)
            line["input_pipeline"] = {"error": repr(e)}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args.config, cfg, steps=2, warmup=1, budget_s=30.0)
    print(json.dumps(line), flush=True)
    finish(world)


DUMP_SAMPLE = 1 << 21


def dump_outputs(out_dir, trainer, losses):
    """What the last timed step computed, as float32 .npy files: losses.npy = (total, photo, smooth, geometry), the values
    Trainer.step returns, and per network the parameter gradients of the step (disp_grads.npy, pose_grads.npy), flattened in
    named_parameters order and shapes (the layout train.py checkpoints), each a fixed seeded sample of DUMP_SAMPLE elements
    when larger (16 MiB in all).  The step starts from the seeded initial state (see the timed region), so two runs with the
    same arguments agree to rounding.  The parameters after the Adam update are not written: an element whose gradient is
    rounding noise moves by +-lr either way."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)

    def save(name, t):
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_SAMPLE:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
    save("losses", torch.stack(losses))
    for name, net in (("disp", trainer.disp_net), ("pose", trainer.pose_net)):
        save(name + "_grads", torch.cat([p.grad.reshape(-1) for p in net.parameters() if p.grad is not None]))


def finish(world):
    """End of a multi-rank run.  The captured CUDA graphs hold NCCL kernels: tearing the process group down with them alive
    hangs in the NCCL watchdog (observed on 2 GPUs: the line was printed, then destroy_process_group blocked until the
    10-minute watchdog abort).  All results are out, so leave without the teardown."""
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


# --------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the step, all usable host threads
# --------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    # bounded: each step is a full batch of the workload; stop after ~150 s of timed steps
    base = cpu_baseline(args.config, cfg, steps=args.steps, warmup=max(1, min(args.warmup, 2)), budget_s=150.0)
    line = {
        "metric": METRIC[args.config],
        "value": base["value"], "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic", "impl": "reference",
        "config": {"workload": cfg["label"], "name": args.config, "global_batch": cfg["batch"], "height": cfg["H"], "width": cfg["W"],
                   "n_ref": cfg["n_ref"], "parallelism": "cpu"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="kitti_r18")
    ap.add_argument("--conv-mode", choices=["fp32", "tf32", "tf32x3"], default="tf32x3",
                    help="tf32x3 = tcgen05 convolutions with split-accumulate operands (fp32-level, the 1e-4 parity mode; default); "
                         "tf32 = tcgen05 single TF32 product (cuDNN's default arithmetic); fp32 = exact CUDA-core convolutions")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-tf32-extra", action="store_true")
    ap.add_argument("--no-input-pipeline", action="store_true", help="skip the device-side input transforms extra (SURVEY.md 8 f-3)")
    ap.add_argument("--no-graph", action="store_true", help="time the eager step instead of the CUDA-graph replay")
    ap.add_argument("--overlap-wgrad", type=int, default=1, help="1 (default): weight gradients on a side stream per network (Trainer(overlap_wgrad=True))")
    ap.add_argument("--overlap-nets", type=int, default=1, help="1 (default): PoseResNet on a side stream next to DispResNet (Trainer(overlap_nets=True))")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the losses and parameter gradients of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
