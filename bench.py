#!/usr/bin/env python
"""bench.py -- frames/s of the Deformable-DETR R50 hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one training pass of the hot path over one synthetic batch per GPU:
forward (ResNet-50 -> 4-level input projection -> 6+6 deformable transformer on the sm_100a
MSDeformAttn kernels -> heads) + SetCriterion (Hungarian matching, focal / L1 / GIoU over 6 layers) +
backward + [N>1: NCCL gradient all-reduce through DDP] + grad-clip(0.1) + AdamW, exactly the six hot
lines of the reference's engine.train_one_epoch (src/trackformer/engine.py:126-151).

Workload at N=1: BASELINE.json configs[1] -- 1x3x800x1333, 300 object queries, random-init R50.
Weak scaling: the per-GPU batch stays fixed as N grows; frames are independent units, the only
collective is the gradient all-reduce (+ one scalar for num_boxes).

Output: ONE JSON line on rank 0 (see the driver contract), with
  value     frames/s, inputs already resident in HBM
  e2e       frames/s with the frame copied from pinned host memory and the loss read back every step
  roofline  the dominant own kernel (MSDeformAttn encoder backward), CUDA-event timed per launch inside the
            timed region; achieved = algorithmic bytes / mean launch time vs the measured HBM peak
  roofline_dense / roofline_e2e   tensor-pipe and whole-step rooflines (lower bounds, see the notes in the line)
  variable_gt   the same metric when the ground-truth box count changes every step (two-graph path)
  parity_vs_reference_c2   measured max relative error of logits / boxes against the reference's C2 golden
  cpu_baseline  the reference's pure-PyTorch path (oracle/torch_ref.py driving the same host-side model on
            the host cores), rank 0, N=1 only, bounded sample
`--impl reference` prints the CPU arm as the main line (rank 0 only; other ranks exit 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

H, W = 800, 1333
LEVELS = [(100, 167), (50, 84), (25, 42), (13, 21)]
N_GT = 20


# --------------------------------------------------------------------------------------------- helpers
def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def msda_alg_bytes(kind, dims):
    n, s, m, d, l, lq, p = dims
    if kind == "fwd":
        return 4 * n * (s * m * d + 3 * lq * m * l * p + lq * m * d)
    return 4 * n * (2 * s * m * d + 6 * lq * m * l * p + lq * m * d)


def make_targets(batch, device, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(batch):
        cxcy = torch.rand(N_GT, 2, generator=g) * 0.6 + 0.2
        wh = torch.rand(N_GT, 2, generator=g) * 0.25 + 0.05
        out.append({"boxes": torch.cat([cxcy, wh], 1).to(device),
                    "labels": torch.zeros(N_GT, dtype=torch.int64, device=device)})
    return out


def tensor_peak(tf32: bool):
    """Dense tensor-pipe denominator for the precision actually used: the driver-measured sustained bf16 cuBLAS rate
    (the step is long, MEASURED_PEAKS.json) halved for TF32 (half the bf16 rate on this part); strict fp32 has no
    tensor-pipe roofline."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    bf16 = 1400.0
    src = "fallback 1.4 PFLOP/s bf16 sustained (B200_PROFILING.md)"
    if os.path.exists(p):
        try:
            bf16 = float(json.load(open(p))["bf16_tflops_sustained"])
            src = "MEASURED_PEAKS.json bf16_tflops_sustained"
        except Exception:
            pass
    return (bf16 / 2 if tf32 else None), src + (" / 2 (TF32)" if tf32 else "")


def dense_flops_per_step(step_fn):
    """FLOPs of the dense contractions (convolutions, matmuls, attention products) of ONE training step, counted by
    torch's FlopCounterMode over an eager step (forward + backward; the MSDeformAttn core is not a contraction)."""
    import trackformer_b200.fused_linear as fl
    own = fl._TCGEN05
    fl._TCGEN05 = False                      # count the long-token Linears too (the own kernel is not an aten::mm)
    try:
        from torch.utils.flop_counter import FlopCounterMode
        with FlopCounterMode(display=False) as fc:
            step_fn()
        return float(fc.get_total_flops())
    except Exception:
        return None
    finally:
        fl._TCGEN05 = own


DUMP_PARAM_SAMPLE = 1 << 22


def dump_outputs(out_dir, loss, model):
    """Write what the last timed step handed its caller: loss.npy, and params.npy with the trainable parameters as that
    step's optimizer update left them (the flat optimizer zeroes the gradient once it has used it).  The parameters are
    taken in model order, whatever their memory layout, and a fixed seeded sample of 4 M of them is written (16 MB).
    Inputs, initial weights and dropout masks are seeded, but the step's atomic reductions and autotuned cuDNN algorithms
    are not bit-reproducible, and the optimizer compounds that over the warm-up and timed steps: compare two builds
    against the spread of two runs of one build, not bit for bit."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters() if p.requires_grad]).float()
    n = min(flat.numel(), DUMP_PARAM_SAMPLE)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
    np.save(os.path.join(out_dir, "params.npy"), flat[idx.to(flat.device)].cpu().numpy())


def golden_parity(dev):
    """max relative error of pred_logits / pred_boxes on the C2 golden case (reference classes on CPU, recorded by
    tests/golden/make_golden_model.py) under the dense-math setting of this run."""
    try:
        import numpy as np
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import model_fixtures as mf
        from trackformer_b200.model_factory import build_model, default_args
        gold = np.load(os.path.join(ROOT, "tests", "golden", "model_det_c2_800x1333.npz"))

        def build(tracking, multi_frame, **kw):
            torch.manual_seed(0)
            m, c, _ = build_model(default_args(tracking, multi_frame, device=str(dev), **kw))
            return m, c
        res = mf.run_detection(build, [(800, 1333)], device=dev)
        out = {}
        for k in ("pred_logits", "pred_boxes"):
            out[k] = float(np.abs(res[k] - gold[k]).max() / np.abs(gold[k]).max())
        return out
    except Exception as exc:
        return {"error": repr(exc)}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (rank 0)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None
        self.t0 = self.t1 = None

    def start(self):
        """Launch nvidia-smi (25 ms period).  Call it BEFORE the warm-up: the tool needs a few hundred ms to come up, and
        the default timed region (20 steps) is only ~0.25 s long; `mark_begin` / `mark_end` bracket the timed region."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)                                   # let the sample that covers the end of the region arrive
        self.proc.terminate()
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = self.t1 if self.t1 is not None else float("inf")
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.05]
        window = "timed region"
        if len(rows) < 2:                                  # very short region: take the samples around it as well
            rows = [r for t, r in self.rows if t0 - 0.3 <= t <= t1 + 0.3]
            window = "timed region +-0.3 s"
        sm = [float(r[1]) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_arm(steps, warmup, batch):
    """The reference's pure-PyTorch MSDeformAttn path on the host cores: the same host-side model with the
    oracle's torch restatement of ms_deform_attn_core_pytorch substituted for the CUDA function.  This is the
    one place bench.py executes oracle/ code (as the baseline being timed, never as the product)."""
    from oracle.torch_ref import msda_core_torch
    import trackformer_b200.msda_module as mm
    from trackformer_b200.model_factory import build_model, default_args

    class _CpuFn:
        @staticmethod
        def apply(value, shapes, loc, attn, step):
            return msda_core_torch(value, shapes, loc, attn)

    saved = mm.MSDeformAttnFunction
    mm.MSDeformAttnFunction = _CpuFn
    # all the host threads the CPU path can use (torchrun pins OMP_NUM_THREADS=1 by default): one per physical core
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(max(torch.get_num_threads(), ncpu // 2 if ncpu > 16 else ncpu))
    try:
        torch.manual_seed(0)
        model, criterion, _ = build_model(default_args(device="cpu"))
        model.train()
        criterion.train()
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=2e-4, weight_decay=1e-4)
        g = torch.Generator().manual_seed(1)
        frames = torch.randn(batch, 3, H, W, generator=g)
        targets = make_targets(batch, "cpu", 2)
        wd = criterion.weight_dict

        def step():
            out, tg, _, _, _ = model(frames, targets)
            losses = criterion(out, tg)
            loss = sum(losses[k] * wd[k] for k in losses if k in wd)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, 0.1)
            opt.step()
            return float(loss.detach())

        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
    finally:
        mm.MSDeformAttnFunction = saved
    return batch * steps / dt, dt / steps * 1e3, torch.get_num_threads()


# --------------------------------------------------------------------------------------------- configs[4]
def c5_arm(args, rank, local_rank, world):
    """BASELINE configs[4]: MOT20-crowd shape 3x1080x1920, multi-frame attention (hidden 288, 8 decoder levels), 500 object
    queries + track queries carried over from the previous frame; one train-mode step = previous-frame forward (no grad,
    engine.py / detr_tracking.py:219-262) + matching + track-query injection + current-frame forward + SetCriterion +
    backward + [DDP-style gradient all-reduce] + clip + AdamW.  Eager launch path: the injection bookkeeping draws from the
    host RNG and reads the matching back, exactly like the reference, so this workload is not graph-captured."""
    import datetime
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    tf32 = not args.no_tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cudnn.benchmark = True
    from trackformer_b200 import ext
    from trackformer_b200.model_factory import build_model, default_args
    msda = ext.load()
    torch.manual_seed(0)
    model, criterion, _ = build_model(default_args(tracking=True, multi_frame=True, device=str(dev), num_queries=500))
    model.to(dev).train()
    criterion.to(dev).train()
    h5, w5, n_gt = 1080, 1920, 60
    bpg = args.batch_per_gpu
    g = torch.Generator().manual_seed(1 + rank)
    host = torch.randn(bpg, 2, 3, h5, w5, generator=g).pin_memory()          # (current, previous) frame pairs
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=2e-4, weight_decay=1e-4, fused=True)
    flat = torch.zeros(sum(p.numel() for p in params), device=dev) if world > 1 else None
    wd = criterion.weight_dict

    def targets_for(frames):
        gg = torch.Generator().manual_seed(7 + rank)
        out = []
        for b in range(bpg):
            cxcy = torch.rand(n_gt, 2, generator=gg) * 0.8 + 0.1
            wh = torch.rand(n_gt, 2, generator=gg) * 0.08 + 0.02
            boxes = torch.cat([cxcy, wh], 1).to(dev)
            t = {"boxes": boxes, "labels": torch.zeros(n_gt, dtype=torch.int64, device=dev),
                 "track_ids": torch.arange(n_gt, device=dev), "image_id": torch.tensor([b], device=dev)}
            pt = {k: v.clone() for k, v in t.items()}
            pt["boxes"] = (pt["boxes"] + 0.005).clamp(0.02, 0.98)
            t["prev_target"] = pt
            t["prev_image"] = frames[b, 1]
            out.append(t)
        return out

    def step(frames):
        tg = targets_for(frames)
        out, tg_out, *_ = model(frames[:, 0], tg)
        losses = criterion(out, tg_out)
        loss = sum(losses[k] * wd[k] for k in losses if k in wd)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if world > 1:                                                          # flat all-reduce (DDP's job in the reference)
            grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in params]
            torch._foreach_copy_(list(flat.split([p.numel() for p in params])), [x.reshape(-1) for x in grads])
            dist.all_reduce(flat)
            flat.div_(world)
            for p, chunk in zip(params, flat.split([p.numel() for p in params])):
                p.grad = chunk.view_as(p)
        torch.nn.utils.clip_grad_norm_(params, 0.1)
        opt.step()
        return loss.detach()

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    dev_frames = host.to(dev)
    for _ in range(max(args.warmup, 3)):
        step(dev_frames)

    def timed(fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    last = {}

    def timed_step():
        last["loss"] = step(dev_frames)

    if sampler:
        sampler.mark_begin()
    l0 = msda.launch_count()
    ms_total = timed(timed_step)
    launches = msda.launch_count() - l0
    if sampler:
        sampler.mark_end()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["loss"], model)
    ms_e2e = timed(lambda: float(step(host.to(dev, non_blocking=True)).item()))
    if rank == 0:
        line = {"metric": "frames/sec TrackFormer multi-frame train step 1080x1920 (BASELINE configs[4])",
                "value": bpg * world * args.steps / (ms_total / 1e3), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "tf32+f32" if tf32 else "f32", "data": "synthetic",
                "config": {"workload": f"TrackFormer multi-frame (hidden 288, D = 36, 8 decoder levels), {bpg}x3x{h5}x{w5} per GPU, "
                                       f"500 object queries + track queries of the previous frame, {n_gt} boxes per frame "
                                       "(BASELINE configs[4])", "global_batch": bpg * world, "parallelism": f"dp{world}",
                           "execution": "eager (host-RNG track-query injection like the reference); previous-frame forward + "
                                        "current-frame forward + SetCriterion + backward + clip + torch AdamW(fused)",
                           "l2": "one step streams > 2 GB of activations"},
                "e2e": {"value": bpg * world * args.steps / (ms_e2e / 1e3), "unit": "frames/s",
                        "h2d_bytes_per_step": host.numel() * 4, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches) * world, "clocks": clocks, "roofline": None, "cpu_baseline": None}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------- main
_JSON_OUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL writes its "NCCL version ..." banner
    to stdout whenever NCCL_DEBUG is VERSION or WARN -- NCCL_DEBUG_FILE is only honoured from INFO up), so file
    descriptor 1 is pointed at stderr for the whole run and the line goes out through a private copy of the real one."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    print(json.dumps(line), file=out, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch-per-gpu", type=int, default=1)
    ap.add_argument("--no-tf32", action="store_true", help="strict fp32 GEMMs/convs (default: TF32 tensor cores)")
    ap.add_argument("--no-optimizer", action="store_true")
    ap.add_argument("--torch-adamw", action="store_true", help="torch.optim.AdamW(fused=True) instead of the flat kernel")
    ap.add_argument("--no-graphs", action="store_true", help="eager step instead of CUDA-graph replay")
    ap.add_argument("--two-graphs", action="store_true",
                    help="forward graph + eager loss + backward graph instead of the single full-step graph")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"],
                    help="c2 = BASELINE configs[1] (default; configs[3] with --batch-per-gpu 2 --gpus 8); c5 = configs[4]: "
                         "multi-frame TrackFormer train step at 3x1080x1920, 500 object queries + track queries from the "
                         "previous frame (eager: the track-query injection draws from the host RNG, like the reference)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA arms, not to --impl reference")
    _claim_stdout()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    bpg = args.batch_per_gpu
    workload = f"Deformable-DETR R50 fwd+bwd, {bpg}x3x{H}x{W} per GPU, 300 queries, 4 levels (BASELINE configs[1])"

    # ------------------------------------------------------------------ reference (CPU) arm
    if args.impl == "reference":
        if rank != 0:
            return
        warm = min(args.warmup, 1)
        steps = max(1, min(args.steps, 3))        # bounded sample: ~10-30 s of CPU work per step budget
        fps, ms, cores = cpu_reference_arm(steps, warm, bpg)
        line = {"impl": "reference", "metric": "frames/sec Deformable-DETR R50 800x1333 fwd+bwd", "value": fps,
                "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": workload, "global_batch": bpg * args.gpus, "parallelism": f"dp{args.gpus}",
                           "device": "host CPU cores (reference pure-PyTorch ms_deform_attn path)", "dropout": 0.1,
                           "optimizer": "AdamW + clip_grad_norm 0.1", "weights": "random init", "gt_boxes_per_frame": N_GT,
                           "bounded_sample": f"{steps} timed step(s) of {bpg} frame(s) after {warm} warm-up on rank 0"},
                "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                                 "sample": f"{steps} full train step(s), pure-PyTorch grid_sample MSDeformAttn (oracle/torch_ref.py)"},
                "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return

    # ------------------------------------------------------------------ B200 arm
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    if args.workload == "c5":
        return c5_arm(args, rank, local_rank, world)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # NCCL's banner must not land in front of the JSON line
        # a collective that does not complete within two minutes is a bug, not a slow link: fail fast instead of holding
        # N GPUs for the default ten minutes
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    tf32 = not args.no_tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cudnn.benchmark = True

    from trackformer_b200 import ext, msda_function
    from trackformer_b200.model_factory import build_model, default_args
    from trackformer_b200.train_step import TrainStep
    msda = ext.load()          # raises if the sm_100a extension is missing

    torch.manual_seed(0)       # same seed on every rank -> identical replicas
    model, criterion, _ = build_model(default_args(device=str(dev)))
    model.to(dev).train()
    criterion.to(dev).train()

    g = torch.Generator().manual_seed(1 + rank)
    host_frames = torch.randn(bpg, 3, H, W, generator=g).pin_memory()
    dev_frames = host_frames.to(dev)
    targets = make_targets(bpg, dev, 2 + rank)

    opt_factory = flat = None
    if args.torch_adamw and not args.no_optimizer:
        opt_factory = lambda ps: torch.optim.AdamW(ps, lr=2e-4, weight_decay=1e-4, fused=True)    # noqa: E731
    elif not args.no_optimizer:
        # the reference's three learning-rate groups (src/train.py:100-119), updated by the one-pass clip + AdamW kernel
        from trackformer_b200.flat_adamw import reference_param_groups
        flat = {"groups": reference_param_groups(model)}
    step = TrainStep(model, criterion, opt_factory, max_norm=0.1, use_graphs=not args.no_graphs,
                     example_frames=dev_frames, example_targets=None if args.two_graphs else targets, flat_adamw=flat)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step(dev_frames, targets)

    if os.environ.get("TFB200_PROFILE_STEP") == "1":
        # profiling aid (never a bench value): exactly ONE replayed step between cudaProfilerStart/Stop, for
        #   ncu --profile-from-start off --graph-profiling node --metrics gpu__time_duration.sum ... python bench.py
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        step(dev_frames, targets)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        if sampler:
            sampler.stop()
        return

    # (1) device-resident throughput
    last = {}

    def timed_step():
        last["loss"] = step(dev_frames, targets)

    if sampler:
        sampler.mark_begin()
    ms_total = timed(timed_step, args.steps)
    if sampler:
        sampler.mark_end()
    clocks = sampler.stop() if sampler else None
    value = bpg * world * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:                 # before the regions below move the model on
        dump_outputs(args.dump_outputs, last["loss"], model)

    # (2) end to end: pinned host frame -> device every step, loss read back every step
    #     The copy of step i + 1's frame is started (TrainStep.prefetch: side stream, staging buffer) right after step i
    #     has been enqueued and before its loss is read, so it runs under step i -- the usual data-loader pipelining.
    #     The timed region holds exactly K copies, K steps and K loss reads: the first frame's copy is issued (and
    #     exposed) inside it, nothing is prefetched for a step outside it.
    def e2e_region(k):
        step.prefetch(host_frames)
        for i in range(k):
            loss = step(None, targets)         # consumes the prefetched frame
            if i + 1 < k:
                step.prefetch(host_frames)     # next step's frame, overlapped with this step
            float(loss.item())
    e2e_region(2)
    ms_e2e = timed(lambda: e2e_region(args.steps), 1)
    e2e_value = bpg * world * args.steps / (ms_e2e / 1e3)

    # (2b) the general path: ground-truth box counts that change every step (forward graph + sync-free loss + backward
    #      graph instead of the single full-step graph, whose capture is tied to the box count)
    var_targets = [make_targets(bpg, dev, 100 + i) for i in range(4)]
    for i, tg in enumerate(var_targets):
        for t in tg:
            keep = N_GT - 1 - (i % 3)
            t["boxes"], t["labels"] = t["boxes"][:keep].contiguous(), t["labels"][:keep].contiguous()
    counter = [0]

    def var_step():
        counter[0] += 1
        step(dev_frames, var_targets[counter[0] % len(var_targets)])
    for _ in range(3):
        var_step()
    ms_var = timed(var_step, args.steps)
    var_value = bpg * world * args.steps / (ms_var / 1e3)

    # (3) per-launch timing of the own kernels.  CUDA-graph replays cannot host per-kernel events, so the same
    #     step (same model, same inputs, same kernels) is replayed eagerly with every MSDeformAttn launch bracketed
    #     by CUDA events on the launching stream; the launch counter gives the kernels per step.
    probe = TrainStep(model, criterion, None, use_graphs=False)
    probe(dev_frames, targets)
    # (every rank: the probe step issues the gradient collectives, so all ranks have to take it together)
    dense_flops = dense_flops_per_step(lambda: probe(dev_frames, targets))
    sink = []
    msda_function.set_timing_sink(sink)
    launches0 = msda.launch_count()
    probe_steps = min(args.steps, 5)
    torch.cuda.synchronize(dev)
    for _ in range(probe_steps):
        probe(dev_frames, targets)
    torch.cuda.synchronize(dev)
    launches_per_step = (msda.launch_count() - launches0) // probe_steps       # every kernel of libmsda_b200.so
    if step.flat_optimizer is not None:
        launches_per_step += len(step.flat_optimizer.ranges)                     # clip + AdamW, one launch per lr group
    msda_function.set_timing_sink(None)
    launches = launches_per_step * args.steps

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ------------------------------------------------------------------ roofline of the own kernels
    peak, peak_src = hbm_peak()
    groups = {}
    for kind, dims, a, b in sink:
        role = "enc" if dims[5] == dims[1] else "dec"
        groups.setdefault((kind, role, dims), []).append(a.elapsed_time(b) * 1e3)
    per_kernel = []
    for (kind, role, dims), us in groups.items():
        mean_us = sum(us) / len(us)
        nbytes = msda_alg_bytes(kind, dims)
        per_kernel.append({"kernel": f"msda_{kind}_{role}", "dims_N_S_M_D_L_Lq_P": list(dims), "launches": len(us),
                           "mean_us": round(mean_us, 2), "total_ms_per_step": round(sum(us) / 1e3 / probe_steps, 4),
                           "alg_bytes": nbytes, "achieved_gbs": round(nbytes / mean_us / 1e3, 1),
                           "frac": round(nbytes / mean_us / 1e3 / peak, 4)})
    per_kernel.sort(key=lambda r: -r["total_ms_per_step"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    dom = per_kernel[0] if per_kernel else None
    if dom and os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(dom["kernel"])
    roofline = None
    if dom:
        roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_gbs"], "peak": peak,
                    "unit": "GB/s", "frac": dom["frac"], "traffic": traffic, "peak_source": peak_src,
                    "mean_launch_us": dom["mean_us"], "alg_bytes_per_launch": dom["alg_bytes"],
                    "note": "algorithmic (compulsory) bytes / CUDA-event launch time, every launch bracketed by events in an "
                            "eager replay of the timed step (graph replays cannot host per-kernel events); "
                            "the gather itself is L1-wavefront bound, see DESIGN.md"}
    # second yardstick: the measured L1-data-stage ceiling for gather-shaped LDG.128 requests (tools/l1_gather_peak.py)
    l1_roofline = None
    l1_path = os.path.join(ROOT, "profiles", "l1_gather_peak.json")
    if per_kernel and os.path.exists(l1_path):
        l1_peak = json.load(open(l1_path))["l2_resident_22.8MB"]["gbs"]
        l1_roofline = {"peak_gbs": l1_peak, "peak_source": "profiles/l1_gather_peak.json (gather-shaped LDG.128 probe, "
                       "22.8 MB table = a C2 frame's value)", "kernels": {}}
        for r in per_kernel:
            n, s_, m, d, l, lq, p = r["dims_N_S_M_D_L_Lq_P"]
            gathered = n * lq * m * l * p * 4 * d * 4                       # corner rows read through L1
            if r["kernel"].startswith("msda_bwd"):
                gathered *= 2                                                # + the same rows as vector reductions
            gbs = gathered / r["mean_us"] / 1e3
            l1_roofline["kernels"][r["kernel"]] = {"gathered_bytes": gathered, "achieved_gbs": round(gbs, 1),
                                                   "frac": round(gbs / l1_peak, 4)}
    msda_ms = sum(r["total_ms_per_step"] for r in per_kernel)
    msda_bytes = sum(r["alg_bytes"] * r["launches"] for r in per_kernel) / max(probe_steps, 1)

    # tensor-pipe and end-to-end rooflines (SURVEY 8(d)).  Dense time is bounded from above by "step minus MSDeformAttn"
    # (it still contains every elementwise / normalisation / optimizer pass), so `achieved` is a LOWER bound.
    ms_step = ms_total / args.steps
    tc_peak, tc_src = tensor_peak(tf32)
    roofline_dense = roofline_e2e = None
    if dense_flops:
        per_gpu_flops = dense_flops                                    # one rank's step
        dense_ms = max(ms_step - msda_ms, 1e-6)
        ach = per_gpu_flops / dense_ms / 1e9
        roofline_dense = {"bound": "tensor", "flops_per_step": per_gpu_flops, "time_ms_upper_bound": round(dense_ms, 3),
                          "achieved": round(ach, 1), "unit": "TFLOP/s", "peak": tc_peak, "peak_source": tc_src,
                          "frac": round(ach / tc_peak, 4) if tc_peak else None,
                          "note": "dense FLOPs (FlopCounterMode, fwd+bwd) / (step - MSDeformAttn time): lower bound"}
        if tc_peak:
            ideal_ms = msda_bytes / (peak * 1e6) + per_gpu_flops / (tc_peak * 1e9)
            roofline_e2e = {"ideal_ms": round(ideal_ms, 3), "measured_ms": round(ms_step, 3),
                            "frac": round(ideal_ms / ms_step, 4),
                            "note": "(MSDeformAttn algorithmic bytes / HBM peak + dense FLOPs / tensor peak) / measured step; "
                                    "elementwise, normalisation and optimizer traffic not credited (lower bound)"}
    parity = golden_parity(dev) if world == 1 else None

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            fps, ms, cores = cpu_reference_arm(args.cpu_steps, 1, bpg)
            cpu_baseline = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                            "sample": f"{args.cpu_steps} full train step(s) of {bpg} frame(s) on the host cores with the "
                                      f"pure-PyTorch grid_sample MSDeformAttn (oracle/torch_ref.py), {ms:.0f} ms/step"}
        except Exception as exc:  # the GPU numbers stay valid
            cpu_baseline = {"value": None, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                            "sample": f"failed: {exc!r}"}

    line = {
        "metric": "frames/sec Deformable-DETR R50 800x1333 fwd+bwd", "value": value, "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32+f32" if tf32 else "f32", "data": "synthetic",
        "config": {"workload": workload, "global_batch": bpg * world, "parallelism": f"dp{world}",
                   "dense_math": "TF32 tensor cores (cuDNN / cuBLAS / own tcgen05 Linear), fp32 accumulate" if tf32 else "strict fp32",
                   "msda_math": "fp32 (hand-written sm_100a kernels)", "dropout": 0.1,
                   "optimizer": "none" if args.no_optimizer else ("torch AdamW(fused)" if args.torch_adamw else "flat one-pass AdamW kernel, reference lr groups") + " + clip_grad_norm 0.1",
                   "execution": "eager" if args.no_graphs else
                   ("forward graph + loss (device Hungarian matching, no host sync) + backward graph" if args.two_graphs else
                    "ONE CUDA graph per step: forward + matching cost + device Hungarian matching (csrc/lsa.cu) + loss + "
                    "backward incl. gradient accumulation") + "; flat-buffer gradient all-reduce (NCCL), clip and fused "
                   "AdamW follow the replay",
                   "gpu_launches_note": f"{launches_per_step} own kernel launches per step (12 MSDeformAttn forward + 12 "
                                        "backward, fused residual+LayerNorm, column sums, ReLU+dropout, sampling prep, "
                                        "Hungarian matching, clip+AdamW), replayed from the graph except the optimizer",
                   "weights": "random init", "gt_boxes_per_frame": N_GT,
                   "l2": "no explicit flush: one step streams >1 GB of activations/weights, far above the 126 MB L2"},
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": host_frames.numel() * 4,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                "input_copy": "every step's frame copied from pinned host memory inside the timed region, on a side "
                              "stream under the previous step (TrainStep.prefetch); loss read back every step"},
        "gpu_launches": int(launches) * world,
        "clocks": clocks,
        "roofline": roofline,
        "roofline_dense": roofline_dense,
        "roofline_e2e": roofline_e2e,
        "variable_gt": {"value": var_value, "unit": "frames/s", "ms_per_step": ms_var / args.steps,
                        "note": "ground-truth box count changes every step: forward graph + sync-free loss + backward graph"},
        "parity_vs_reference_c2": parity,
        "diagnostics": {"l1_gather_probe": l1_roofline},
        "msda_kernels": per_kernel,
        "msda_ms_per_step": round(msda_ms, 4),
        "cpu_baseline": cpu_baseline,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
