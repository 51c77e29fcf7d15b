#!/usr/bin/env python
"""bench.py -- throughput of the TA3N hot path on B200 (metric of BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA path through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the unmodified reference on the host cores, rank 0

One "step" = one paired mini-batch (B source + B target videos, T=5, D=2048) through
VideoModel.forward (train mode, dropout 0.5/0.5), the composed loss of the shipped script
(CE + 3 domain CEs + 0.003 * attentive entropy; main.py:446, 508-538, 559-562) and backward to all
parameter gradients (+ the gradient all-reduce when N > 1).  clips per step = 2B per GPU.
The optimizer is outside the metric (BASELINE.json: "fwd+bwd"); the e2e leg includes it.

Prints ONE JSON line on rank 0 (schema: see the task contract).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BETA = (0.75, 0.75, 0.5)       # script_train_val.sh: beta 0.75 0.75 0.5
GAMMA = 0.003
H = 256
D = 2048
METRIC = "video-clips/sec fwd+bwd (B=256,T=5,D=2048)"
print_json = None   # set in main(): writes the one JSON line to the real stdout


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="videos per domain per GPU")
    ap.add_argument("--segments", type=int, default=5)
    ap.add_argument("--classes", type=int, default=12)
    ap.add_argument("--fc_dim", type=int, default=512)
    ap.add_argument("--engine", default=os.environ.get("TA3N_ENGINE", "auto"), choices=["auto", "fp32", "tf32", "tf32x3"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="enqueue the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU budget of the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (its loss and every parameter gradient) as "
                         "DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    return args


# ------------------------------------------------------------------------------------------------
# algorithmic traffic (fp32; every operand read once, every result written once) -- DESIGN.md §5
# ------------------------------------------------------------------------------------------------
def traffic_model(M, T, F, C):
    """bytes per step for the whole path ("scope B") and per GEMM call site."""
    from ta3n_b200.functional import relation_set
    rs = relation_set(T)
    R = T - 1
    S = rs.n_slots
    Wt = sum(s * F * H + H for s in rs.scales)
    Wr = R * (H * H + 3 * H + 2)
    f4 = 4.0
    scope_a = f4 * (3 * M * T * F + 3 * Wt + 3 * Wr + 4 * M * R * H + 2 * (3 * M * R + M * H))
    shared = 2 * M * T * D + 3 * (F * D + F)                       # x read fwd+wgrad, W read 2x, dW written
    frame_disc = 3 * (F * F + 3 * F + 2) + 2 * M * T * F + 2 * M * T * F + 3 * M * T * 2
    video = 3 * (H * H + 3 * H + 2 + C * H + C) + 4 * M * H + 3 * M * (C + 2)
    scope_b = scope_a + f4 * (shared + frame_disc + video)
    n_rel = rs.n_rel
    frame_fwd = M * T * F + F * F + F + M * T * F          # frame-disc hidden GEMM: feat, W1, b1 -> hidden
    video_fwd = M * H + H * H + H + M * H
    w_shared = M * T * F + M * T * D + F * D               # d_pre, x -> dW
    w_trn = n_rel * M * H + M * T * F + Wt
    w_frame = 2 * M * T * F + F * F + M * T * 2 + 2 * F
    w_video = 2 * M * H + H * H + M * 2 + 2 * H + M * C + M * H + C * H
    w_rel = 2 * R * M * H + R * H * H + R * M * 2 + R * 2 * H + R * M * H
    sites = {   # algorithmic bytes of ONE launch of each GEMM call site of the TrainStep launch sequence
        "shared_fc_fwd": f4 * (M * T * D + F * D + F + M * T * F),
        "fwd_batch": f4 * (frame_fwd + M * T * F + Wt + n_rel * M * H),      # frame-disc hidden + TRN relations
        "relattn_fwd": f4 * (M * R * H + R * (H * H + H) + R * M * H),
        "disc_fwd": f4 * video_fwd,
        "disc_dgrad": f4 * (M * T * F + F * F + 2 * M * T * F) + f4 * (M * H + H * H + M * H),   # 2 launches
        "relattn_dgrad": f4 * (R * M * H + R * H * H + M * H + M * R + M * R * H),
        "trn_dgrad": f4 * (n_rel * M * H + Wt + M * T * F),
        "wgrad_all": f4 * (w_shared + w_trn + w_frame + w_video + w_rel),    # every weight gradient of the step
    }
    flops_b = 3 * (2 * M * S * F * H + R * (2 * M * H * H + 4 * M * H)) + \
        3 * (2 * M * T * F * F + 4 * M * T * F + 2 * M * H * H + 4 * M * H + 2 * M * H * C) + 2 * (2 * M * T * D * F)
    return {"scope_a": scope_a, "scope_b": scope_b, "sites": sites, "flops_b": flops_b}


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag.is_set():
                    break
                self.samples.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        if self.proc is not None:
            self.proc.terminate()
        sm, smax, reasons, power = [], 0.0, set(), 0.0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                smax = max(smax, float(s[1]))
                power = max(power, float(s[2]))
                for n, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax or None,
                "power_w_max": power or None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 0))), "measured"
    return 6650.0, 1590.0, "fallback"        # B200_PROFILING.md fallback


DUMP_BYTES = 60_000_000      # payload of --dump-outputs: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Write {name: float32 array} as out_dir/<name>.npy.  When they hold more than DUMP_BYTES, every array is cut to
    the same fraction of its entries, a fixed sample seeded by its size (flattened, in index order), so that the
    files of two runs with the same arguments still correspond entry for entry."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    keep = min(1.0, DUMP_BYTES / total) if total else 1.0
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if keep < 1.0:
            idx = np.random.default_rng(a.size).choice(a.size, int(a.size * keep), replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def pick_engine(requested):
    import ta3n_b200
    if requested == "auto":
        requested = os.environ.get("TA3N_DEFAULT_ENGINE", "tf32x3")      # the library default = the parity-tested engine
    ta3n_b200.set_gemm_engine(requested)
    return requested


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path on the host cores (unmodified classes from
# the oracle/_ref snapshot; the oracle port only if that snapshot is missing)
# ------------------------------------------------------------------------------------------------
def host_cores() -> int:
    """Cores this process may really use: affinity mask and cgroup CPU quota, not os.cpu_count()."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def _reference_step_fn(args):
    """One training step (forward + composed loss + backward) of the UNMODIFIED reference classes on CPU:
    models.VideoModel / TRNmodule / loss.attentive_entropy imported through oracle/ref_shims.py from
    /root/reference (build container) or from the oracle/_ref snapshot made by oracle/build_ref.py (GPU box).
    Protocol of BASELINE.md section 2.  Returns (step, kind) or (None, why)."""
    try:
        import torch

        from oracle import gen_golden, ref_shims
        if ref_shims.models_root() is None:
            return None, "no reference modules (oracle/_ref snapshot missing)"
        ref_models, _, _ = ref_shims.load()
        torch.manual_seed(1234)
        model = ref_models.VideoModel(args.classes, "video", "trn-m", "RGB", train_segments=args.segments,
                                      val_segments=args.segments, add_fc=1, fc_dim=args.fc_dim, dropout_i=0.5,
                                      dropout_v=0.5, partial_bn=False, use_bn="none", ens_DA="none",
                                      use_attn="TransAttn", n_attn=1, use_attn_frame="none", share_params="Y",
                                      verbose=False)
        model.train()
        g = torch.Generator().manual_seed(4321)
        xs = torch.randn(args.batch, args.segments, D, generator=g)
        xt = torch.randn(args.batch, args.segments, D, generator=g)
        labels = torch.arange(args.batch) % args.classes

        def step():
            model.zero_grad(set_to_none=True)
            outs = model(xs, xt, list(BETA), 0, is_train=True, reverse=False)        # main.py:418
            loss = gen_golden.reference_loss(outs, labels)                           # main.py:446, 508-538, 559-562
            loss.backward()                                                          # main.py:576
            return loss

        step()
        return step, "reference"
    except Exception as e:      # the port below is the documented fallback; say why
        return None, f"{type(e).__name__}: {e}"


def _port_step_fn(args):
    import torch  # noqa: F401

    from oracle import ta3n_oracle as orc          # checker / CPU baseline only (never the product path)
    cfg = orc.PathConfig(num_class=args.classes, num_segments=args.segments, fc_dim=args.fc_dim,
                         dropout_i=0.5, dropout_v=0.5)
    params = orc.init_params(cfg, seed=1234)
    xs, xt, labels = orc.synthetic_batch(args.batch, cfg)
    names = orc.used_param_names(params)
    leaves = {k: params[k].clone().requires_grad_(True) for k in names}
    live = dict(params)
    live.update(leaves)

    def step():
        for v in leaves.values():
            v.grad = None
        outs = orc.forward(live, xs, xt, BETA, 0.0, cfg, train=True, reverse=False)
        loss = orc.compose_loss(outs, labels, GAMMA)
        loss.backward()
        return loss

    return step


def cpu_reference_run(args, steps, warmup, budget_s=None):
    import torch

    avail = host_cores()
    step, kind = _reference_step_fn(args)
    why_port = None
    if step is None:
        why_port, kind = kind, "port"
        step = _port_step_fn(args)

    # "all the host threads it can use": eager PyTorch stops scaling (and can collapse) well before
    # 100+ threads on these small GEMMs, so time one step per candidate count and keep the fastest.
    best = None
    for n in sorted({min(c, avail) for c in (8, 16, 32, 64, avail)}):
        torch.set_num_threads(n)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, n)
        if dt > 3.0:
            break
    cores = best[1]
    torch.set_num_threads(cores)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        step()
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s and done >= 3:
            break
    dt = time.perf_counter() - t0
    what = ("the UNMODIFIED reference classes (models.VideoModel + TRNmodule + loss.py via oracle/ref_shims.py)"
            if kind == "reference" else "the oracle port (eager PyTorch CPU restatement of the reference)")
    return {"clips_per_s": done * 2 * args.batch / dt, "ms_per_step": 1e3 * dt / done, "steps": done,
            "cores": cores, "cores_available": avail, "kind": kind, "what": what, "why_port": why_port}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args, args.steps, args.warmup)
    sample = (f"{r['steps']} full steps of {r['what']} at B={args.batch}+{args.batch}, T={args.segments}, D={D}, "
              f"train mode, dropout 0.5/0.5, forward + composed loss + backward")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["clips_per_s"], "unit": "clips/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1, "cpu"), "gemm_engine": "cpu fp32 (ATen/MKL)",
        "cpu_baseline": {"value": r["clips_per_s"], "unit": "clips/s", "cores": r["cores"], "cores_available": r["cores_available"],
                         "kind": r["kind"], "sample": sample, "why_port": r["why_port"]},
        "e2e": {"value": r["clips_per_s"], "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print_json(line)


def workload_config(args, world, engine):
    name = {(256, 5, 12, 512): "cfg2", (512, 5, 30, 512): "cfg5 per GPU", (8, 5, 5, 512): "cfg1",
            (128, 9, 12, 512): "cfg3 without frame attention"}.get((args.batch, args.segments, args.classes, args.fc_dim),
                                                                   "custom")
    return {"workload": f"{name}: B={args.batch} source + {args.batch} target videos per GPU, T={args.segments}, "
                        f"D={D}, fc_dim={args.fc_dim}, {args.classes} classes, TRN-M + TransAttn + RevGrad "
                        f"discriminators (frame/video/relation)",
            "global_batch": 2 * args.batch * world, "per_gpu_clips": 2 * args.batch,
            "api": "ta3n_b200.train.TrainStep (forward + fused loss heads + backward, one CUDA graph)",
            "step": "forward + composed loss + backward to all parameter gradients"
                    + (" + gradient all-reduce (see `allreduce`)" if world > 1 else ""),
            "optimizer": "excluded from value (metric is fwd+bwd); included in e2e",
            "dropout": "0.5/0.5 (product arm: in-kernel counter RNG; reference arm: nn.Dropout)",
            "parallelism": f"dp{world}", "l2": "flushed (256 MiB write) before every timed step",
            "timing": "CUDA events around each step on the launching stream; steps enqueued behind a 20 ms "
                      "device-side spin so host launch gaps are outside the events"}


# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    import ta3n_b200
    from ta3n_b200 import _lib
    from ta3n_b200.loss import ta3n_loss
    from ta3n_b200.models import VideoModel
    from ta3n_b200.train import SGDNesterov, TrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    engine = pick_engine(args.engine)

    B, T, C, F = args.batch, args.segments, args.classes, min(args.fc_dim, D)
    torch.manual_seed(1234)
    model = VideoModel(C, "video", "trn-m", "RGB", train_segments=T, val_segments=T, add_fc=1, fc_dim=args.fc_dim,
                       dropout_i=0.5, dropout_v=0.5, partial_bn=False, use_bn="none", ens_DA="none",
                       use_attn="TransAttn", use_attn_frame="none", share_params="Y", verbose=False).to(dev).train()

    g = torch.Generator().manual_seed(4321 + rank)
    xs_h = torch.randn(B, T, D, generator=g).pin_memory()
    xt_h = torch.randn(B, T, D, generator=g).pin_memory()
    lab_h = (torch.arange(B) % C).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # the public training-step API: forward + fused loss heads + backward in one CUDA graph
    step = TrainStep(model, B, B, BETA, gamma=GAMMA, use_graph=not args.no_graph)
    step.load(xs_h, xt_h, lab_h)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step.run()
    barrier()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)

    # ---- value: inputs resident in HBM, device-timed with CUDA events, L2 flushed before each step
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    # Park the GPU (~20 ms spin) while the host enqueues the first steps: the events then bracket device time
    # only, not the gaps a busy host leaves between a flush and the following graph launch (observed on a shared
    # box: 0.29 -> 0.38 ms/step with identical per-kernel times).
    torch.cuda._sleep(int(20e-3 * 1.9e9))
    for k in range(args.steps):
        flush.fill_(k & 0xFF)
        ev[k][0].record()
        step.run()
        ev[k][1].record()
    barrier()
    if args.dump_outputs and rank == 0:
        # before the e2e leg below, whose optimizer steps move the parameters
        names = {id(p): n for n, p in model.named_parameters()}
        outputs = {"loss": step.loss.cpu().numpy()}
        outputs.update((f"grad.{names[id(p)]}", g.cpu().numpy()) for p, g in zip(step.params, step.grad_views))
        dump_outputs(args.dump_outputs, outputs)
    launches = step.launches_per_step * args.steps
    t_ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([t_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_ms = float(t.item())

    # ---- e2e: host (pinned) inputs -> public API -> loss on the host, optimizer step included.
    # Every step's inputs are copied H2D inside the timed region; the copy of step k+1 is issued on a copy
    # stream while step k computes (double-buffered input slots), as a training loop with a prefetching
    # loader would do.
    # optimizer = the shipped script's: SGD-Nesterov lr 3e-2, momentum 0.9, wd 1e-4, clip_gradient 20 (main.py:83,
    # 578-583), run by the library's fused kernels (inside the graph at N=1, after the all-reduce at N>1)
    pipe = TrainStep(model, B, B, BETA, gamma=GAMMA, use_graph=not args.no_graph, double_buffer=True,
                     optimizer=SGDNesterov(lr=3e-2, momentum=0.9, weight_decay=1e-4, clip_gradient=20.0))
    host_batches = [(xs_h, xt_h, lab_h), (xt_h, xs_h, lab_h)]      # two distinct pinned batches, alternated

    loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event() for _ in range(2)]

    def e2e_loop(n):
        """Every step: H2D of its inputs (prefetched one step ahead), the fused iteration, D2H of its loss.  The
        host reads the loss of step k-1 while step k runs (as a logging training loop does), so a slow host
        does not drain the device queue."""
        pipe.prefetch(*host_batches[0])
        last = None
        for k in range(n):
            pipe.swap()                                   # consume the prefetched slot
            pipe.prefetch(*host_batches[(k + 1) & 1])     # H2D of the next step's inputs, overlapped
            loss = pipe.run()                             # fwd + loss + bwd (+ all-reduce) + clip + SGD step
            loss_host[k & 1].copy_(loss, non_blocking=True)      # D2H of this step's result
            loss_ready[k & 1].record()
            if k > 0:
                loss_ready[(k - 1) & 1].synchronize()
                last = float(loss_host[(k - 1) & 1][0])
        loss_ready[(n - 1) & 1].synchronize()
        return float(loss_host[(n - 1) & 1][0]) if n > 0 else last

    e2e_loop(6)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    for p_, v_ in zip(step.params, step.grad_views):      # `pipe` re-pointed .grad at its own bucket
        p_.grad = v_
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    # what the host link can do: the same pinned buffers copied back to back (explains the e2e number)
    ha, hb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ha.record()
    for _ in range(5):
        pipe.slots[0][0].copy_(xs_h, non_blocking=True)
        pipe.slots[0][1].copy_(xt_h, non_blocking=True)
    hb.record()
    torch.cuda.synchronize()
    h2d_gbps = 5 * 2 * xs_h.numel() * 4 / (ha.elapsed_time(hb) * 1e-3) / 1e9
    clocks = sampler.finish() if sampler else None     # sampled across both timed regions (value and e2e)

    # ---- the drop-in autograd API (VideoModel.forward + torch loss + backward), for reference
    def autograd_step():
        model.zero_grad(set_to_none=True)
        outs = model(step.xs, step.xt, list(BETA), 0, is_train=True, reverse=False)
        ta3n_loss(outs, step.labels, GAMMA).backward()

    for _ in range(3):
        autograd_step()
    barrier()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea.record()
    for _ in range(args.steps):
        autograd_step()
    eb.record()
    barrier()
    autograd_ms = ea.elapsed_time(eb) / args.steps
    for p_, v_ in zip(step.params, step.grad_views):
        p_.grad = v_

    # ---- roofline: per-call-site device time (CUDA events inside the library; eager pass, no graph)
    eager = TrainStep(model, B, B, BETA, gamma=GAMMA, use_graph=False)
    eager.load(xs_h, xt_h, lab_h)
    eager.run()
    _lib.timing_enable(True)
    barrier()
    n_prof = min(args.steps, 10)
    for k in range(n_prof):
        flush.fill_(k & 0xFF)
        eager.run()
    torch.cuda.synchronize()
    rep = _lib.timing_report()
    _lib.timing_enable(False)

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            del step, pipe, eager
            torch.cuda.synchronize()
            dist.destroy_process_group()
        return

    hbm_peak, tf_peak, peak_kind = measured_peaks()
    M = 2 * B
    tm = traffic_model(M, T, F, C)
    step_ms = t_ms / args.steps
    total_site_ms = sum(ms for _, ms in rep.values()) or 1.0
    # dominant GEMM call site; sites within 3 % of the slowest are ranked by their algorithmic bytes (the merged
    # weight-gradient launch and the forward batch are that close and would otherwise swap between runs)
    cand = [k for k in rep if k in tm["sites"]]
    t_max = max((rep[k][1] for k in cand), default=0.0)
    dom = max((k for k in cand if rep[k][1] >= 0.97 * t_max), key=lambda k: tm["sites"][k], default=None)
    roof = None
    if dom:
        cnt, ms = rep[dom]
        per_step_ms = ms / n_prof                      # all launches of this call site in one step
        ach = tm["sites"][dom] / (per_step_ms * 1e-3) / 1e9
        traffic = None
        try:   # DRAM bytes of this call site from the committed `ncu --set full` capture (profiles/)
            with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
                traffic = json.load(f)["dram_bytes_per_step"].get(dom) if (B, T, F, C) == (256, 5, 512, 12) else None
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach / hbm_peak, "traffic": traffic,
                "traffic_source": "profiles/r2_step_full.txt (ncu --set full of one step of this binary, tf32x3 engine: "
                                  "dram__bytes_read+write of the launch)",
                "peak_kind": peak_kind,
                "algorithmic_bytes_per_step": tm["sites"][dom], "kernel_ms_per_step": per_step_ms,
                "share_of_library_time": ms / total_site_ms, "launches_per_step": cnt / n_prof}
    ach_b = tm["scope_b"] / (step_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": world * 2 * B * args.steps / (t_ms * 1e-3), "unit": "clips/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "tf32x3": "tf32x3"}.get(engine, "tf32"),
        "data": "synthetic", "config": workload_config(args, world, engine), "gemm_engine": engine,
        "roofline": roof,
        "roofline_step": {"bound": "hbm", "scope": "whole step (SURVEY 8d scope B)", "achieved": ach_b,
                          "peak": hbm_peak, "unit": "GB/s", "frac": ach_b / hbm_peak,
                          "algorithmic_bytes": tm["scope_b"], "algorithmic_flops": tm["flops_b"],
                          "achieved_tflops": tm["flops_b"] / (step_ms * 1e-3) / 1e12, "peak_kind": peak_kind},
        "kernel_ms_per_step": {k: round(v[1] / n_prof, 5) for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1])},
        "e2e": {"value": world * 2 * B * args.steps / e2e_s, "unit": "clips/s",
                "h2d_bytes_per_step": int(2 * B * T * D * 4 + B * 8), "d2h_bytes_per_step": 4,
                "ms_per_step": 1e3 * e2e_s / args.steps,
                "h2d_link_gbps_measured": h2d_gbps,
                "h2d_ms_per_step_at_link_rate": (2 * B * T * D * 4) / (h2d_gbps * 1e9) * 1e3,
                "optimizer_launches_per_step": 2,
                "includes": "H2D of every step's inputs (pinned host -> device, prefetched one step ahead on a "
                "copy stream), forward, loss, backward, all-reduce, clip_grad_norm + SGD-Nesterov step (fused "
                "kernels of this library), D2H of every step's loss (read by the host one step behind)"},
        "gpu_launches": int(launches), "launches_per_step": int(step.launches_per_step),
        "cuda_graph": not args.no_graph, "autograd_api_ms_per_step": autograd_ms, "clocks": clocks,
        "step_mode": step.mode,
        "allreduce": None if world == 1 else (
            {"kind": "library kernel over " + ("NVSwitch multicast (multimem.ld_reduce / multimem.st)" if step.ar["mc"]
                                               else "NVLink peer memory"),
             "bytes": int(step.flat_grad.numel() * 4), "where": "inside the step's CUDA graph, before the optimizer"}
            if step.ar is not None else {"kind": "NCCL all_reduce (AVG) between two graphs", "bytes": int(step.flat_grad.numel() * 4)}),
    }
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(args, 1000, 2, budget_s=args.cpu_seconds)
        line["cpu_baseline"] = {"value": r["clips_per_s"], "unit": "clips/s", "cores": r["cores"],
                                "cores_available": r["cores_available"], "kind": r["kind"],
                                "ms_per_step": r["ms_per_step"], "why_port": r["why_port"],
                                "sample": f"{r['steps']} full steps (B={B}+{B}) of {r['what']} on the host "
                                          f"cores, ~{args.cpu_seconds:.0f}s budget"}
    print_json(line)
    if world > 1:
        del step, pipe, eager
        torch.cuda.synchronize()
        dist.destroy_process_group()


def main():
    args = parse()
    # The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner to stdout) must
    # not pollute it: route fd 1 to stderr for the whole run and write the JSON line to the real stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real_stdout, "w")
    global print_json
    print_json = lambda line: (out.write(json.dumps(line) + "\n"), out.flush())   # noqa: E731
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
