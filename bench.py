#!/usr/bin/env python
"""bench.py -- encoder images/sec at 1024^2 for the EV-M student (BASELINE.json metric), B200-native path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference|eager_gpu] [--batch B] [--img S] [--dump-outputs DIR]

One "step" = one forward pass of the hot path over one synthetic batch (per GPU):
  ImageStudentEncoder(efficientvit_b1) : [B,3,S,S] fp32 NCHW -> [B,1024,E,E] fp32   (stage1/model.py:188-211)
N > 1 (torchrun): images are sharded across ranks, no data-path collective for the forward (SURVEY.md section 8e)
-> "scaling": "weak"; timing = max over ranks of device time.

Every N (1, 2, 4, 8) also carries `per_n`: the paths north_star shards, each timed max-over-ranks on the device:
  kd_train_step_evm / kd_train_step_rvm   the stage-1 KD training iteration (EV-M: config 2's student side; RV-M, 32 img/GPU:
                                          config 4) WITH the gradient all-reduce of the flat arena inside the timed region
                                          (train_image_encoder_stage1.py:67-72, 215-227), the all-reduce timed alone beside it
  teacher_vit_forward                     SAM3 ViT trunk forward, batch 8/GPU at 1008^2 (the "ViT-H" half of the metric)

Keys beyond the base contract: `roofline` (dominant kernel family by time, measured live with CUDA events on the launch stream,
plus whole-step fractions and the top families), `cpu_baseline` (the oracle port timed on this box's host cores, rank 0, N=1),
`e2e` (pinned host batch -> H2D -> module forward -> D2H of the step's scalar metric, every step), `also` (N=1: the other
encoders, the teacher-embedding dump end to end with its real 85 MB/step D2H, and the PyTorch-eager GPU arm).
`--dump-outputs DIR` (native) writes the embeddings of the last timed step, as the caller receives them, to DIR/embeddings.npy
(fp32; above DUMP_MAX_ELEMS elements a fixed seeded sample of them, in flat-index order): the seeded weights and inputs are the
same on every run with the same arguments, so two builds can be compared output for output.
`--impl reference` times the CPU oracle port (the reference is Python/PyTorch; /root/reference does not exist on the GPU box,
and the oracle is pinned to it by tests/golden) with all host threads.  `--impl eager_gpu` runs the same functional PyTorch
restatement on the GPU -- the reference's eager CUDA path (cuDNN / cuBLAS), as shipped (TF32 + fp16 autocast) and strict fp32.
"""
from __future__ import annotations

import argparse
import datetime
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from types import SimpleNamespace as NS

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "encoder images/sec @1024^2 (EV-M student forward)"
UNIT = "images/s"
DUMP_MAX_ELEMS = 1 << 23          # 32 MB of fp32 per dumped array


def dump_sample(t: torch.Tensor):
    """`t` as fp32 numpy when it has at most DUMP_MAX_ELEMS elements, else the elements at a fixed seeded set of flat indices
    (sorted): the same positions on every run for the same shape."""
    t = t.detach()
    if t.numel() > DUMP_MAX_ELEMS:
        idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).unique()
        t = t.reshape(-1)[idx.to(t.device)]
    return t.float().cpu().numpy()


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def build_student(img, embed, device, backbone="efficientvit_b1"):
    from efficientsam3_b200.stage1.model import build_image_student_model
    cfg = NS(MODEL=NS(BACKBONE=backbone), DATA=NS(IMG_SIZE=img), DISTILL=NS(EMBED_DIM=1024, EMBED_SIZE=embed))
    torch.manual_seed(0)
    m = build_image_student_model(cfg)
    with torch.no_grad():  # random-init weights of the named architecture + non-trivial BN statistics
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_var.uniform_(0.5, 1.5)
                mod.running_mean.normal_(0, 0.1)
                mod.weight.uniform_(0.5, 1.5)
                mod.bias.normal_(0, 0.1)
    return m.to(device).eval()


class Ctx:
    """Rank / device / distributed plumbing shared by every leg."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist_
            self.dist = dist_
            self.dist.init_process_group("nccl", device_id=torch.device("cuda", self.local), timeout=datetime.timedelta(minutes=4))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        if self.dist is None:
            return ms
        t = torch.tensor([ms], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def timed(self, fn, warm, steps):
        """W untimed calls, barrier + synchronize, K calls between CUDA events on the launch stream, barrier + synchronize;
        returns the max over ranks of ms per call."""
        for _ in range(warm):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def all_ok(self, ok: bool) -> bool:
        """True when the leg succeeded on every rank (a rank that failed must not leave the others inside a collective
        of the NEXT leg)."""
        if self.dist is None:
            return ok
        t = torch.tensor([1.0 if ok else 0.0], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)


def run_native(args):
    from efficientsam3_b200 import ops
    cx = Ctx()
    rank, world, dev, dist = cx.rank, cx.world, cx.dev, cx.dist
    B, S, E = args.batch, args.img, args.embed
    model = build_student(S, E, dev)
    if args.graph:
        model.enable_cuda_graphs()

    g = torch.Generator().manual_seed(1234 + rank)
    host = [torch.randn(B, 3, S, S, generator=g).pin_memory() for _ in range(2)]
    x_dev = [h.to(dev) for h in host]  # 2 x 403 MB at B=32,S=1024: each larger than the 126 MB L2
    torch.cuda.synchronize()

    # ---------------------------------------------------------------- device-resident throughput
    for i in range(args.warmup):
        out = model(x_dev[i % 2])
    cx.barrier()
    sampler = ClockSampler(cx.local)
    if rank == 0:
        sampler.start()
    l0 = ops.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = model(x_dev[i % 2])
    e1.record()
    cx.barrier()
    launches = ops.launch_count - l0
    if launches == 0 and getattr(model, "graph_launches_per_step", 0):
        launches = model.graph_launches_per_step * args.steps          # replayed from a CUDA graph: counted at capture
    ms_total = cx.max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        # now: with CUDA graphs `out` is the graph's output buffer, which later replays of the same input buffer overwrite
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "embeddings.npy"), dump_sample(out))
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total / 1e3)

    # ---------------------------------------------------------------- end-to-end (host buffers)
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [torch.empty_like(x_dev[0]) for _ in range(2)]
    metric_host = torch.zeros(1).pin_memory()

    def e2e_pass(nsteps):
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        with torch.cuda.stream(copy_stream):
            stage[0].copy_(host[0], non_blocking=True)
            ready[0].record(copy_stream)
        for i in range(nsteps):
            cur, nxt = i % 2, (i + 1) % 2
            if i + 1 < nsteps:
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(freed[nxt])
                    stage[nxt].copy_(host[nxt], non_blocking=True)
                    ready[nxt].record(copy_stream)
            torch.cuda.current_stream().wait_event(ready[cur])
            y = model(stage[cur])
            freed[cur].record()
            metric_host.copy_(y[:, :, ::8, ::8].abs().mean().reshape(1), non_blocking=True)  # step metric, 4 bytes D2H
            torch.cuda.current_stream().synchronize()  # the caller consumes the metric every step

    e2e_pass(2)
    cx.barrier()
    t0 = time.perf_counter()
    e2e_pass(args.steps)
    cx.barrier()
    e2e_ms = cx.max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)

    # the same end-to-end loop with bf16 images in pinned host memory (half the PCIe bytes; the student's first kernel rounds the
    # image to bf16 operands anyway) -- reported beside the headline e2e, never instead of it
    e2e_bf16 = None
    if rank == 0 and world == 1 and not args.no_also:
        keep_host, keep_stage = host, stage
        try:
            host16 = [h.to(torch.bfloat16).pin_memory() for h in keep_host]
            host, stage = host16, [torch.empty_like(x_dev[0], dtype=torch.bfloat16) for _ in range(2)]
            e2e_pass(2)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e2e_pass(args.steps)
            torch.cuda.synchronize()
            e2e_bf16 = {"value": round(B * args.steps / (time.perf_counter() - t0), 1), "unit": UNIT,
                        "h2d_bytes_per_step": host16[0].numel() * 2, "input": "bf16 NCHW in pinned host memory"}
        except Exception as e:
            e2e_bf16 = {"error": f"{type(e).__name__}: {e}"[:200]}
        finally:
            host, stage = keep_host, keep_stage
    del stage

    # ---------------------------------------------------------------- roofline of the dominant kernel
    roofline, kernel_table = None, None
    if rank == 0:
        roofline, kernel_table = roofline_leg(model, x_dev, ms_step, B, S)
    del x_dev, host
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- the sharded paths, every N (collectives inside: ALL ranks)
    per_n = None
    if not args.no_per_n:
        per_n = per_n_legs(cx, S, E)

    # ---------------------------------------------------------------- the other encoders of the north-star (N = 1, brief)
    also = None
    if rank == 0 and world == 1 and not args.no_also:
        also = other_encoders(dev, S, E)
        if not args.no_eager:
            try:
                torch.cuda.empty_cache()
                pn = per_n or {}
                also["eager_gpu"] = eager_gpu_block(dev, S, E, B, native_img_s=value,
                                                    native_teacher_img_s=(pn.get("teacher_vit_forward") or {}).get("images_per_s"),
                                                    native_kd_ms=(pn.get("kd_train_step_evm") or {}).get("ms_per_step"))
            except Exception as e:
                also["eager_gpu"] = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---------------------------------------------------------------- CPU baseline (rank 0, N = 1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_oracle_throughput(S, E, batch=4, steps=5, warmup=1)

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"EV-M student encoder forward (efficientvit_b1 + 1024-ch head, eval), batch {B}/GPU x "
                                   f"3x{S}x{S} fp32 NCHW -> 1024x{E}x{E} fp32; random-init weights",
                       "batch_per_gpu": B, "global_batch": B * world, "img": S, "embed": E, "parallelism": f"dp{world}",
                       "l2_policy": f"inputs alternate between two {B*3*S*S*4/1e6:.0f} MB buffers (> 126 MB L2)",
                       "launch": "CUDA graph replay" if getattr(model, "graph_launches_per_step", 0) else "host-launched kernel sequence"},
            "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": B * 3 * S * S * 4,
                    "d2h_bytes_per_step": 4,
                    "note": "H2D-inclusive: the 403 MB fp32 batch crosses PCIe inside every timed step (copy stream, double-buffered) and "
                            "bounds this figure; the read-back is the step's 4-byte metric, as in the training loop, which keeps the "
                            "embeddings on the device.  The path whose result really leaves the GPU (teacher dump, 85 MB D2H / step) is "
                            "`also.e2e_teacher_dump`"},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "per_n": per_n, "also": also,
        }
        if e2e_bf16 is not None and also is not None:
            also["e2e_bf16_host_input"] = e2e_bf16
        if kernel_table is not None and args.table:
            with open(args.table, "w") as f:
                f.write("| kernel family | launches/step | ms/step | alg GB/s | alg TFLOP/s |\n|---|---|---|---|---|\n")
                for k, kms, c, kb, kf in kernel_table:
                    f.write(f"| `{k}` | {c} | {kms:.4f} | {kb/1e9/(kms/1e3):.0f} | {kf/1e12/(kms/1e3):.1f} |\n")
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def roofline_leg(model, x_dev, ms_step, B, S):
    from efficientsam3_b200 import ops
    prof = ops.Profiler()
    ops.set_profiler(prof)
    eager_forward = getattr(model, "forward_uncaptured", model)      # per-kernel events need the host-launched sequence
    for i in range(3):
        eager_forward(x_dev[i % 2])
    ops.set_profiler(None)
    agg = prof.summary()
    kernel_table = sorted(((k, v["ms"] / 3, v["calls"] // 3, v["bytes"] / 3, v["flops"] / 3) for k, v in agg.items()),
                          key=lambda r: -r[1])
    pk = _peaks()
    total = sum(r[1] for r in kernel_table)

    def fracs(kms, kbytes, kflops):
        gbs, tfs = kbytes / 1e9 / (kms / 1e3), kflops / 1e12 / (kms / 1e3)
        return gbs, tfs, gbs / pk["hbm"], tfs / pk["tf_sustained"]

    name, kms, calls, kbytes, kflops = kernel_table[0]
    gbs, tfs, frac_hbm, frac_tc = fracs(kms, kbytes, kflops)
    if frac_tc > frac_hbm:
        roofline = {"bound": "tensor", "achieved": round(tfs, 1), "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                    "frac": round(frac_tc, 4), "traffic": None}
    else:
        roofline = {"bound": "hbm", "achieved": round(gbs, 1), "peak": pk["hbm"], "unit": "GB/s",
                    "frac": round(frac_hbm, 4), "traffic": None}
    # DRAM bytes per launch of that kernel from an `ncu --set full` capture (profiles/r*_traffic.json; null if not captured)
    for fn in ("r2_traffic.json", "r1_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", fn)
        if os.path.exists(tpath):
            tr = json.load(open(tpath)).get(name)
            if tr:
                roofline["traffic"] = tr["dram_bytes_per_launch"]     # of the captured launch below, not the family average
                roofline["traffic_launch"] = tr.get("captured_launch")
                roofline["traffic_source"] = "profiles/" + fn
                break
    roofline.update(kernel=name, launches_per_step=calls, ms_per_step=round(kms, 4),
                    share_of_step=round(kms / total, 4), peak_source=pk["src"])
    # every family above 4 % of the step, each against its own binding roof: the step is a flat profile, not one kernel
    fam = []
    for k, ms_, c, kb, kf in kernel_table:
        if ms_ / total < 0.04:
            continue
        g_, t_, fh, ft = fracs(ms_, kb, kf)
        fam.append({"kernel": k, "ms_per_step": round(ms_, 4), "share_of_step": round(ms_ / total, 3),
                    "bound": "tensor" if ft > fh else "hbm", "frac": round(max(fh, ft), 3)})
    roofline["families"] = fam
    # whole-step figures against SURVEY section 8d's per-image algorithmic bytes / flops
    alg_bytes = 110e6 * (S / 1008.0) ** 2 * B
    alg_flops = 40.2e9 * (S / 1008.0) ** 2 * B
    roofline["step"] = {"alg_GB_per_step": round(alg_bytes / 1e9, 3), "hbm_frac": round(alg_bytes / 1e9 / (ms_step / 1e3) / pk["hbm"], 4),
                        "alg_TFLOP_per_step": round(alg_flops / 1e12, 3),
                        "tensor_frac": round(alg_flops / 1e12 / (ms_step / 1e3) / pk["tf_sustained"], 4)}
    return roofline, kernel_table


# --------------------------------------------------------------------------------------------------------------------------------
# per-N legs: what north_star shards over the GPUs of one box
def per_n_legs(cx: Ctx, S, E):
    out = {"world": cx.world,
           "timing": "CUDA events on the launch stream between barrier+synchronize pairs, max over ranks; images/s = world x batch / that"}
    legs = [("kd_train_step_evm", lambda: kd_train_step_leg(cx, S, E, batch=32, steps=3, warm=2, backbone="efficientvit_b1")),
            ("kd_train_step_rvm", lambda: kd_train_step_leg(cx, S, E, batch=32, steps=3, warm=2, backbone="repvit_m1_1")),
            ("teacher_vit_forward", lambda: teacher_leg(cx, batch=8, steps=3, warm=1))]
    for name, fn in legs:
        res, ok = None, True
        try:
            torch.cuda.empty_cache()
            res = fn()
        except Exception as e:  # a rank-local failure (OOM): every rank learns of it below and the remaining legs still line up
            res, ok = {"error": f"{type(e).__name__}: {e}"[:300]}, False
        if not cx.all_ok(ok) and ok:
            res = {"error": "failed on another rank"}
        out[name] = res
    torch.cuda.empty_cache()
    return out


def kd_train_step_leg(cx: Ctx, S, E, batch, steps, warm, backbone="efficientvit_b1"):
    """One stage-1 KD training iteration per call on every rank: train-mode student forward (batch-statistics BN) -> KD loss ->
    native backward -> all-reduce of the flat gradient arena (NCCL over NVLink; skipped at world 1) -> grad-norm clip + fused AdamW
    (stage1/losses.kd_train_step).  Stored-teacher targets as in the reference loop (fp16-rounded)."""
    from efficientsam3_b200 import ops
    from efficientsam3_b200.stage1.losses import kd_train_step
    from efficientsam3_b200.stage1.optim import FlatAdamW
    dev = cx.dev
    m = build_student(S, E, dev, backbone).train()
    opt = FlatAdamW(m, lr=1e-4, weight_decay=0.01)
    g = torch.Generator().manual_seed(99 + cx.rank)
    xs = [torch.randn(batch, 3, S, S, generator=g).to(dev) for _ in range(2)]
    teacher = torch.randn(batch, 1024, E, E, generator=g).half().float().to(dev)
    sizes = [(3, S, S * 3 // 4) if i % 2 == 0 else (3, S * 2 // 3, S) for i in range(batch)]
    state = {"i": 0}

    def step():
        state["loss"] = kd_train_step(m, opt, xs[state["i"] % 2], teacher, sizes, 1.0, 5.0)
        state["i"] += 1

    n0 = ops.launch_count
    ms = cx.timed(step, warm, steps)
    per_step = (ops.launch_count - n0) // (warm + steps)
    res = {"student": backbone, "ms_per_step": round(ms, 2), "images_per_s": round(cx.world * batch / ms * 1e3, 1),
           "batch_per_gpu": batch, "global_batch": batch * cx.world, "img": S, "bn": "batch statistics (per rank, no SyncBN)",
           "loss_rank0": round(float(state["loss"].item()), 3), "es3_launches_per_step": per_step,
           "peak_mem_GB": round(torch.cuda.max_memory_allocated() / 1e9, 1)}
    if cx.dist is not None:
        # the collective alone, same buffer: how much of the step it is, and what is left of it once it overlaps the backward
        ar = cx.timed(lambda: opt.all_reduce_grads(), 2, 10)
        res["allreduce"] = {"ms_alone": round(ar, 3), "bytes": int(opt.numel) * 4, "share_of_step": round(ar / ms, 4),
                            "busbw_GB_s": round(2 * (cx.world - 1) / cx.world * opt.numel * 4 / ar / 1e6, 1),
                            "kernel": "ncclDevKernel_AllReduce_Sum_f32_RING_LL / NVLS (NCCL picks; NCCL_DEBUG=INFO prints it)",
                            "placement": getattr(opt, "overlap_note", "blocking, after the backward returns")}
    del m, opt, xs, teacher
    return res


def teacher_leg(cx: Ctx, batch, steps, warm):
    from efficientsam3_b200.stage1.model import SAM3ImageTeacherEncoder
    torch.manual_seed(0)
    t = SAM3ImageTeacherEncoder(embed_size=72).to(cx.dev)
    x = torch.randn(batch, 3, 1008, 1008, device=cx.dev)
    ms = cx.timed(lambda: t(x), warm, steps)
    pk = _peaks()
    tfs = 5.4 * batch / ms * 1e3                            # SURVEY 8d: 5.4 TFLOP / image -> TFLOP/s on this GPU
    res = {"ms_per_step": round(ms, 2), "images_per_s": round(cx.world * batch / ms * 1e3, 2), "batch_per_gpu": batch, "img": 1008,
           "alg_TFLOP_per_s_per_gpu": round(tfs, 1), "frac_of_sustained_tensor_peak": round(tfs / pk["tf_sustained"], 3)}
    del t, x
    return res


# --------------------------------------------------------------------------------------------------------------------------------
def _time_steps(fn, warm, steps):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def other_encoders(dev, S, E):
    """Device-resident images/s of the other paths the north-star names, same run, short loops (reported beside the
    headline; each has its own parity tests).  Teacher / config 3 run at their native 1008 px (SURVEY.md D2)."""
    from efficientsam3_b200.model.sam1_task import Sam3PointPromptSegmenter
    out = {}
    torch.manual_seed(0)
    rv = build_student(S, E, dev, "repvit_m1_1")
    x = torch.randn(32, 3, S, S, device=dev)
    ms = _time_steps(lambda: rv(x), 2, 5)
    pk = _peaks()
    out["rvm_student_forward"] = {"images_per_s": round(32 / ms * 1e3, 1), "ms_per_step": round(ms, 3), "batch": 32, "img": S,
                                  "hbm_frac_algorithmic": round(350e6 * (S / 1008) ** 2 * 32 / 1e9 / (ms / 1e3) / pk["hbm"], 3)}
    del rv
    tv = build_student(S, E, dev, "tiny_vit_11m")
    ms = _time_steps(lambda: tv(x), 2, 5)
    out["tvm_student_forward"] = {"images_per_s": round(32 / ms * 1e3, 1), "ms_per_step": round(ms, 3), "batch": 32, "img": S,
                                  "hbm_frac_algorithmic": round(247e6 * (S / 1008) ** 2 * 32 / 1e9 / (ms / 1e3) / pk["hbm"], 3)}
    del tv, x
    x = torch.randn(8, 3, 1008, 1008, device=dev)
    seg = Sam3PointPromptSegmenter().to(dev)
    coords = torch.rand(8, 1, 2, device=dev) * 1008
    labels = torch.ones(8, 1, dtype=torch.int32, device=dev)
    ms = _time_steps(lambda: seg.set_image_batch(x).predict_batch(coords, labels, multimask_output=True), 1, 3)
    out["config3_vit_fpn_mask_decoder"] = {"images_per_s": round(8 / ms * 1e3, 2), "ms_per_step": round(ms, 2), "batch": 8,
                                           "img": 1008, "prompt": "1 point / image, multimask"}
    del seg, x
    # optimiser side of the KD step (A20): grad norm + fused AdamW over an EV-M-sized flat arena; HBM streams
    from efficientsam3_b200.stage1.optim import FlatAdamW
    ev = build_student(S, E, dev, "efficientvit_b1")
    for p in ev.parameters():
        p.requires_grad_(True)
    opt = FlatAdamW(ev, lr=1e-3, weight_decay=0.01)
    opt.flat_grad.normal_(0, 1e-3)
    ms = _time_steps(lambda: opt.step(max_norm=5.0), 3, 20)
    gbs = opt.numel * 32 / ms / 1e6     # 4 B (norm) + 28 B (AdamW: read p,g,m,v, write p,m,v) per parameter
    out["kd_optimizer_step_evm"] = {"ms_per_step": round(ms, 4), "params": int(opt.numel), "alg_GB_per_s": round(gbs, 1),
                                    "frac_of_hbm_peak": round(gbs / _peaks()["hbm"], 3)}
    del ev, opt
    torch.cuda.empty_cache()
    legs = [
        # config 2 as BASELINE.json words it: EV-M student + frozen ViT teacher in the loop, batch 32, at the teacher's native 1008 px
        ("config2_online_kd_step", lambda: online_kd_step_leg(dev, batch=32, steps=2, warm=1)),
        # EfficientSAM3 as deployed for the SAM-1 task: EV-M student encoder + SAM2-branch FPN + mask decoder, 1 point / image
        ("efficientsam3_evm_point_prompt", lambda: efficientsam3_point_leg(dev, batch=8)),
        # A21 end to end: pinned host images -> H2D -> teacher forward -> fp16 -> D2H of the embeddings (10.6 MB / image)
        ("e2e_teacher_dump", lambda: teacher_dump_e2e_leg(dev, batch=8, steps=4, warm=1)),
        # the strict (fp32-class) precision mode of the headline model: parity mode, CUDA-core fp32 kernels
        ("strict_mode_evm_forward", lambda: strict_leg(dev, S, E, batch=8)),
    ]
    for name, fn in legs:
        try:
            torch.cuda.empty_cache()
            out[name] = fn()
        except Exception as e:  # never let a side measurement take the headline line down
            out[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
    torch.cuda.empty_cache()
    return out


def strict_leg(dev, S, E, batch):
    from efficientsam3_b200 import ops
    m = build_student(S, E, dev)
    x = torch.randn(batch, 3, S, S, device=dev)

    def fwd():
        with ops.strict_precision():
            return m(x)

    ms = _time_steps(fwd, 1, 3)
    fast = m(x)
    strict = fwd()
    rel = ((fast.double() - strict.double()).norm() / strict.double().norm()).item()
    return {"images_per_s": round(batch / ms * 1e3, 1), "ms_per_step": round(ms, 2), "batch": batch, "img": S,
            "what": "EV-M forward with fp32 activations / weights / FMA accumulation (csrc/strict_f32.cu): embeddings within rtol 1e-4 of the "
                    "reference's fp32 output (tests/test_strict_gpu.py); the bf16 tensor-core mode is the headline",
            "bf16_mode_rel_l2_vs_strict": float(f"{rel:.3e}")}


def teacher_dump_e2e_leg(dev, batch, steps, warm):
    """save_embeddings_one_epoch's data movement (save_embedding_image_stage1.py:86-96) through the native pieces: the batch starts
    in pinned host memory, the fp16 embeddings end in pinned host memory (the writer thread's input); H2D and D2H ride a copy
    stream, double-buffered against the teacher forward."""
    from efficientsam3_b200 import ops
    from efficientsam3_b200.stage1.model import SAM3ImageTeacherEncoder
    torch.manual_seed(0)
    t = SAM3ImageTeacherEncoder(embed_size=72).to(dev)
    host_in = [torch.randn(batch, 3, 1008, 1008).pin_memory() for _ in range(2)]
    n_out = batch * 1024 * 72 * 72
    host_out = [torch.empty(n_out, dtype=torch.float16).pin_memory() for _ in range(2)]
    dev_in = [torch.empty(batch, 3, 1008, 1008, device=dev) for _ in range(2)]
    dev_out = [torch.empty(n_out, device=dev, dtype=torch.float16) for _ in range(2)]
    copy = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()

    def run(n):
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        drained = [torch.cuda.Event() for _ in range(2)]
        with torch.cuda.stream(copy):
            dev_in[0].copy_(host_in[0], non_blocking=True)
            ready[0].record(copy)
        for i in range(n):
            cur, nxt = i % 2, (i + 1) % 2
            main.wait_event(ready[cur])
            if i >= 2:
                main.wait_event(drained[cur])
            out = t(dev_in[cur])
            ops.cast_f32_to_f16(out.contiguous(), out=dev_out[cur])
            done[cur].record(main)
            with torch.cuda.stream(copy):
                if i + 1 < n:
                    dev_in[nxt].copy_(host_in[nxt], non_blocking=True)      # next batch in, under this batch's forward
                    ready[nxt].record(copy)
                copy.wait_event(done[cur])
                host_out[cur].copy_(dev_out[cur], non_blocking=True)
                drained[cur].record(copy)
        copy.synchronize()
        main.synchronize()

    run(warm + 1)
    t0 = time.perf_counter()
    run(steps)
    sec = (time.perf_counter() - t0) / steps
    return {"value": round(batch / sec, 2), "unit": UNIT, "ms_per_step": round(sec * 1e3, 2), "batch": batch, "img": 1008,
            "h2d_bytes_per_step": batch * 3 * 1008 * 1008 * 4, "d2h_bytes_per_step": n_out * 2,
            "what": "pinned host fp32 images -> H2D -> SAM3 ViT trunk -> es3_cast_f32_to_f16 -> D2H fp16 embeddings in pinned host memory"}


def efficientsam3_point_leg(dev, batch):
    from efficientsam3_b200.model_builder import build_efficientsam3_point_segmenter
    seg = build_efficientsam3_point_segmenter("efficientvit", "b1").to(dev)
    x = torch.randn(batch, 3, 1008, 1008, device=dev)
    coords = torch.rand(batch, 1, 2, device=dev) * 1008
    labels = torch.ones(batch, 1, dtype=torch.int32, device=dev)
    ms = _time_steps(lambda: seg.set_image_batch(x).predict_batch(coords, labels, multimask_output=True), 2, 5)
    return {"images_per_s": round(batch / ms * 1e3, 1), "ms_per_step": round(ms, 2), "batch": batch, "img": 1008,
            "what": "EV-M student encoder -> 1024x72x72 -> SAM2-branch FPN -> prompt encoder + TwoWay mask decoder -> 1008^2 masks"}


def online_kd_step_leg(dev, batch, steps, warm):
    from efficientsam3_b200.stage1.losses import kd_train_step_online
    from efficientsam3_b200.stage1.model import SAM3ImageTeacherEncoder
    from efficientsam3_b200.stage1.optim import FlatAdamW
    S, E = 1008, 72
    teacher = SAM3ImageTeacherEncoder(embed_size=E).to(dev)
    m = build_student(S, E, dev).train()
    opt = FlatAdamW(m, lr=1e-4, weight_decay=0.01)
    x = torch.randn(batch, 3, S, S, device=dev)
    sizes = [(3, S, S * 3 // 4) if i % 2 == 0 else (3, S * 2 // 3, S) for i in range(batch)]
    state = {}

    def step():
        state["loss"] = kd_train_step_online(m, teacher, opt, x, sizes, 1.0, 5.0)

    ms = _time_steps(step, warm, steps)
    return {"ms_per_step": round(ms, 1), "images_per_s": round(batch / ms * 1e3, 1), "batch": batch, "img": S, "embed": E,
            "what": "frozen ViT teacher forward (chunks of 8) -> fp16-rounded targets -> EV-M train-mode forward -> KD loss -> backward -> AdamW",
            "loss": round(float(state["loss"].item()), 3), "peak_mem_GB": round(torch.cuda.max_memory_allocated() / 1e9, 1)}


# --------------------------------------------------------------------------------------------------------------------------------
# The reference's PyTorch-eager GPU path: the functional restatement of its modules (oracle/, pinned to the reference by
# tests/golden) run by PyTorch on the same GPU -- cuDNN / cuBLAS / SDPA kernels, none of ours.  A BASELINE arm only.
def _oracle_sd(backbone, S, E, dev):
    from efficientsam3_b200.stage1.model import build_image_student_model
    from oracle.weights import fill_state_dict
    cfg = NS(MODEL=NS(BACKBONE=backbone), DATA=NS(IMG_SIZE=S), DISTILL=NS(EMBED_DIM=1024, EMBED_SIZE=E))
    sd = fill_state_dict(build_image_student_model(cfg).state_dict(), 7)
    return {k: v.to(dev) for k, v in sd.items()}


def _eager_modes():
    """(name, tf32, autocast dtype): 'as shipped' = TF32 on (sam3/sam3/model_builder.py:47-56) + torch.cuda.amp.autocast() fp16
    (stage1/train_image_encoder_stage1.py:199); 'strict' = fp32, TF32 off (the parity oracle on the device)."""
    return [("as_shipped_tf32_fp16_autocast", True, torch.float16), ("strict_fp32", False, None)]


class _EagerMode:
    def __init__(self, tf32, ac):
        self.tf32, self.ac = tf32, ac

    def __enter__(self):
        self.prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark)
        torch.backends.cuda.matmul.allow_tf32 = self.tf32
        torch.backends.cudnn.allow_tf32 = self.tf32
        torch.backends.cudnn.benchmark = True
        self.cm = torch.autocast("cuda", dtype=self.ac) if self.ac is not None else None
        if self.cm is not None:
            self.cm.__enter__()

    def __exit__(self, *exc):
        if self.cm is not None:
            self.cm.__exit__(*exc)
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = self.prev


def eager_gpu_block(dev, S, E, B, native_img_s=None, native_teacher_img_s=None, native_kd_ms=None, steps=10, warm=3):
    from oracle import efficientvit as O
    from oracle import vitdet as OV
    from oracle.kd_loss import kd_loss as oracle_kd_loss
    out = {"what": "functional PyTorch restatement of the reference modules (oracle/, pinned by tests/golden) in PyTorch eager on this GPU: "
                   "cuDNN convolutions, cuBLAS GEMMs, SDPA; cudnn.benchmark on; CUDA events, median-free mean of the timed loop",
           "torch": torch.__version__}
    sd = _oracle_sd("efficientvit_b1", S, E, dev)
    x = torch.randn(B, 3, S, S, device=dev)
    ev = {}
    for name, tf32, ac in _eager_modes():
        with torch.no_grad(), _EagerMode(tf32, ac):
            ms = _time_steps(lambda: O.image_student_encoder(sd, x, E, "b1"), warm, steps)
        ev[name] = {"ms_per_step": round(ms, 3), "images_per_s": round(B / ms * 1e3, 1)}
        if native_img_s:
            ev[name]["native_over_eager"] = round(native_img_s / (B / ms * 1e3), 2)
    out["evm_forward"] = dict(ev, batch=B, img=S)
    # EV-M KD training iteration, reference recipe: autocast forward, fp32 loss, GradScaler, clip_grad_norm_, torch.optim.AdamW
    try:
        kd = {}
        for name, tf32, ac in _eager_modes():
            p = {k: (v.clone().requires_grad_(True) if (v.is_floating_point() and "running" not in k and "num_batches" not in k) else v.clone())
                 for k, v in sd.items()}
            params = [v for v in p.values() if v.requires_grad]
            opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=0.01)
            scaler = torch.amp.GradScaler("cuda", enabled=ac is not None)
            teacher = torch.randn(B, 1024, E, E, device=dev).half().float()
            sizes = [(3, S, S * 3 // 4) if i % 2 == 0 else (3, S * 2 // 3, S) for i in range(B)]

            def step():
                with _EagerMode(tf32, ac), O.bn_batch_stats():
                    preds = O.image_student_encoder(p, x, E, "b1")
                loss, _, _ = oracle_kd_loss(preds.float(), teacher, S, sizes, 1.0)
                scaler.scale(loss).backward()
                scaler.unscale_(opt)
                torch.nn.utils.clip_grad_norm_(params, 5.0)
                scaler.step(opt)
                scaler.update()
                opt.zero_grad(set_to_none=True)

            ms = _time_steps(step, 2, 4)
            kd[name] = {"ms_per_step": round(ms, 2), "images_per_s": round(B / ms * 1e3, 1),
                        "peak_mem_GB": round(torch.cuda.max_memory_allocated() / 1e9, 1)}
            if native_kd_ms:
                kd[name]["native_over_eager"] = round(ms / native_kd_ms, 2)
            del p, params, opt
            torch.cuda.empty_cache()
        out["evm_kd_train_step"] = dict(kd, batch=B, img=S)
    except Exception as e:
        out["evm_kd_train_step"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    del sd, x
    torch.cuda.empty_cache()
    # teacher ViT trunk, batch 8 @ 1008^2
    try:
        from efficientsam3_b200.stage1.model import SAM3ImageTeacherEncoder
        from oracle.weights import fill_state_dict
        pre = "sam3.backbone.vision_backbone.trunk."
        tsd = fill_state_dict({k: v for k, v in SAM3ImageTeacherEncoder(embed_size=72).state_dict().items() if not v.is_complex()}, 5)
        tsd = {k: v.to(dev) for k, v in tsd.items()}
        xt = torch.randn(8, 3, 1008, 1008, device=dev)
        tv = {}
        for name, tf32, ac in _eager_modes():
            with torch.no_grad(), _EagerMode(tf32, ac):
                ms = _time_steps(lambda: OV.vit_trunk(tsd, pre, xt), 1, 3)
            tv[name] = {"ms_per_step": round(ms, 2), "images_per_s": round(8 / ms * 1e3, 2)}
            if native_teacher_img_s:
                tv[name]["native_over_eager"] = round(native_teacher_img_s / (8 / ms * 1e3), 2)
        out["teacher_vit_forward"] = dict(tv, batch=8, img=1008)
    except Exception as e:
        out["teacher_vit_forward"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    torch.cuda.empty_cache()
    return out


def run_eager_gpu(args):
    """`--impl eager_gpu`: one JSON line in the headline's metric / config for the reference's eager CUDA path."""
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    B, S, E = args.batch, args.img, args.embed
    blk = eager_gpu_block(dev, S, E, B, steps=max(args.steps, 3), warm=max(args.warmup, 2))
    shipped = blk["evm_forward"]["as_shipped_tf32_fp16_autocast"]
    line = {"impl": "eager_gpu", "metric": METRIC, "value": shipped["images_per_s"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": shipped["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 autocast + TF32 (as shipped)", "data": "synthetic",
            "config": {"workload": f"EV-M student encoder forward, PyTorch eager on the GPU, batch {B} x 3x{S}x{S}", "img": S, "embed": E,
                       "launched_world": world}, "eager_gpu": blk}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------------------------
def _physical_cores():
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def _keep_malloc_off_mmap():
    """glibc serves every allocation above its mmap threshold (<= 32 MB) with a fresh mmap and returns it with munmap: the
    oracle's intermediates (up to 268 MB each) are then page-faulted in on EVERY pass.  Measured on the GPU box's host
    (scripts/cpu_arm_probe.sh, profiles/r2q_cpu_probe.log): 1.5 img/s in a fresh process vs 6.7 img/s with the heap kept
    (and 5 img/s at the end of the native run, whose heap had grown) -- the bimodal CPU arm of round 1.  mallopt() is the
    in-process form of MALLOC_MMAP_MAX_=0 MALLOC_TRIM_THRESHOLD_=big; it only ever makes the CPU baseline faster."""
    try:
        import ctypes
        libc = ctypes.CDLL("libc.so.6")
        M_TRIM_THRESHOLD, M_TOP_PAD, M_MMAP_MAX = -1, -2, -4
        ok = libc.mallopt(M_MMAP_MAX, 0) and libc.mallopt(M_TRIM_THRESHOLD, 2 ** 31 - 1) and libc.mallopt(M_TOP_PAD, 1 << 28)
        return bool(ok)
    except Exception:
        return False


def cpu_oracle_throughput(S, E, batch, steps, warmup):
    """Times the CPU oracle port (oracle/efficientvit.py; pinned to the reference by tests/golden) on the host's physical cores.
    The only place the native arm touches oracle/ besides the eager-GPU arm -- as a baseline, never as the product path.
    Round 1's figure moved 1.05 -> 4.97 img/s between runs (batch 2, 3 passes, 64 unpinned threads): now batch 4, 5 passes after a
    warm-up, threads = physical cores, min / median / max reported."""
    from oracle import efficientvit as O
    from oracle.weights import fill_state_dict
    from efficientsam3_b200.stage1.model import build_image_student_model
    cfg = NS(MODEL=NS(BACKBONE="efficientvit_b1"), DATA=NS(IMG_SIZE=S), DISTILL=NS(EMBED_DIM=1024, EMBED_SIZE=E))
    sd = fill_state_dict(build_image_student_model(cfg).state_dict(), 7)
    x = torch.randn(batch, 3, S, S, generator=torch.Generator().manual_seed(1))
    heap_kept = _keep_malloc_off_mmap()
    prev = torch.get_num_threads()
    cores = min(_physical_cores(), len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else 1 << 30)
    if os.environ.get("ES3_CPU_THREADS"):
        cores = int(os.environ["ES3_CPU_THREADS"])
    if os.environ.get("ES3_CPU_CUDA_INIT") == "1" and torch.cuda.is_available():
        torch.cuda.init()
        torch.zeros(1, device="cuda")
    torch.set_num_threads(cores)
    try:
        with torch.no_grad():
            for _ in range(warmup):
                O.image_student_encoder(sd, x, E, "b1")
            ts = []
            for _ in range(steps):
                t0 = time.perf_counter()
                O.image_student_encoder(sd, x, E, "b1")
                ts.append(time.perf_counter() - t0)
    finally:
        torch.set_num_threads(prev)
    sec = statistics.median(ts)
    return {"value": round(batch / sec, 3), "unit": UNIT, "cores": cores, "kind": "port",
            "min_median_max": [round(batch / max(ts), 3), round(batch / sec, 3), round(batch / min(ts), 3)],
            "sample": f"{steps} timed passes of batch {batch} x 3x{S}x{S} after {warmup} warm-up (median), PyTorch-CPU fp32 eager oracle port, "
                      f"torch threads = {cores} physical cores, glibc heap kept off mmap = {heap_kept}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if rank != 0:
        return
    S, E = args.img, args.embed
    batch = min(args.batch, 4)
    t0 = time.perf_counter()
    cpu = cpu_oracle_throughput(S, E, batch=batch, steps=max(5, min(args.steps, 8)), warmup=max(1, min(args.warmup, 2)))
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(batch / cpu["value"] * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"EV-M student encoder forward on host CPU (oracle port of the reference modules), "
                               f"bounded sample: batch {batch} x 3x{S}x{S}", "img": S, "embed": E},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": round(time.perf_counter() - t0, 1),
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "eager_gpu"])
    ap.add_argument("--batch", type=int, default=32, help="images per GPU per step")
    ap.add_argument("--img", type=int, default=1024)
    ap.add_argument("--embed", type=int, default=64, help="stage1/config.py:21,50 pair IMG_SIZE 1024 with EMBED_SIZE 64")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-also", action="store_true", help="skip the brief RV-M / teacher / config-3 measurements")
    ap.add_argument("--no-eager", action="store_true", help="skip the PyTorch-eager GPU arm inside `also`")
    ap.add_argument("--no-per-n", action="store_true", help="skip the per-N KD-step / teacher legs")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="launch the eval plan kernel by kernel instead of replaying its CUDA graph")
    ap.add_argument("--table", default=None, help="write the per-kernel-family table (markdown) here")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the embeddings of the last timed step (rank 0; sampled above 32 MB) to DIR/embeddings.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs dumps the native path's outputs (--impl native)")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "eager_gpu":
        run_eager_gpu(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
