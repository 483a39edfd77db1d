"""Device preprocessing (es3_preprocess_images) on SA-1B-shaped inputs; writes one JSON file under profiles/.

  (a) kernel time: 32 seeded uint8 1500x2250 CHW images on the device -> [32,3,1024,1024] fp32, CUDA events over >= 50 calls
      (tap prologue + fused resize).  The 324 MB of input exceed the 126 MB L2, so every call reads them from HBM.
  (b) end to end: pinned uint8 host images (raw 1500x2250, and pre-shrunk to 683x1024) -> H2D -> preprocess -> graphed
      EV-M forward, against today's pinned fp32 [32,3,1024,1024] batch -> H2D -> graphed forward.  Every mode launches step i's
      forward, then prepares batch i+1 on a side stream (host packing overlaps the device work), and the modes alternate in
      one process.
  (c) CPU cost of the reference's loader preprocessing per SA-1B image: torch CPU interpolate(antialias) + norm + pad, on one
      thread and with all cores.

usage: python scripts/preprocess_bench.py [--out profiles/preprocess_bench.json] [--steps 20] [--reps 3]
"""
from __future__ import annotations

import argparse
import json
import os
import platform
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU
B, S, EMBED = 32, 1024, 64
H, W = 1500, 2250       # SA-1B


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor() or "unknown"


def kernel_leg(dev, calls):
    from efficientsam3_b200 import ops
    from efficientsam3_b200.stage1 import transforms as T
    g = torch.Generator(device=dev).manual_seed(0)
    imgs = [torch.randint(0, 256, (3, H, W), generator=g, device=dev, dtype=torch.uint8) for _ in range(B)]
    oh, ow = T.get_preprocess_shape(H, W, S)
    rows = [T.describe(t.data_ptr(), 0, H, W, *t.stride(), (oh, ow)) for t in imgs]
    table, taps, max_out = T.build_table(rows)
    pre = T.ImagePreprocessor(S)
    table_d = torch.from_numpy(table).to(dev)
    affine_d = torch.from_numpy(np.stack([pre._affine[0]] * B)).to(dev)
    out = torch.empty(B, 3, S, S, device=dev)
    in_bytes, out_bytes = B * 3 * H * W, B * 3 * S * S * 4

    def once():
        ops.preprocess_images(table_d, affine_d, S, max_out, taps, in_bytes, out=out)

    for _ in range(5):
        once()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        once()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / calls
    # the whole ImagePreprocessor call on the same device images (host table build + table H2D + the two kernels)
    for _ in range(3):
        pre(imgs, out=out)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        pre(imgs, out=out)
    torch.cuda.synchronize()
    ms_api = (time.perf_counter() - t0) * 1e3 / calls
    gbps = (in_bytes + out_bytes) / (ms * 1e-3) / 1e9
    return {"batch": B, "input": f"{B} x uint8 3x{H}x{W} CHW on the device", "output": f"[{B},3,{S},{S}] fp32",
            "calls_timed": calls, "ms_per_batch": round(ms, 4), "algorithmic_bytes": in_bytes + out_bytes,
            "read_bytes": in_bytes, "write_bytes": out_bytes, "achieved_GBps": round(gbps, 1),
            "share_of_hbm_bound": round(gbps / (HBM_TBPS * 1e3), 3),
            "note": "inputs (324 MB) exceed the 126 MB L2: read from HBM every call",
            "ms_per_batch_python_api": round(ms_api, 4)}


def e2e_leg(dev, steps, reps):
    from bench import build_student
    from efficientsam3_b200.stage1.transforms import ImagePreprocessor, get_preprocess_shape
    model = build_student(S, EMBED, dev)
    model.enable_cuda_graphs()
    g = torch.Generator().manual_seed(1)
    host_f32 = [torch.randn(B, 3, S, S, generator=g).pin_memory() for _ in range(2)]
    raw = [[torch.randint(0, 256, (3, H, W), generator=g, dtype=torch.uint8).pin_memory() for _ in range(B)] for _ in range(2)]
    sh, sw = get_preprocess_shape(H, W, S)
    small = [[torch.randint(0, 256, (3, sh, sw), generator=g, dtype=torch.uint8).pin_memory() for _ in range(B)] for _ in range(2)]
    pre = ImagePreprocessor(S)
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [torch.empty(B, 3, S, S, device=dev) for _ in range(2)]
    metric_host = torch.zeros(1).pin_memory()

    def produce(mode, i, dst):
        if mode == "fp32":
            dst.copy_(host_f32[i % 2], non_blocking=True)
        else:
            pre((raw if mode == "raw_uint8" else small)[i % 2], out=dst)

    def run(mode, nsteps):
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        with torch.cuda.stream(copy_stream):
            produce(mode, 0, stage[0])
            ready[0].record(copy_stream)
        for i in range(nsteps):
            cur, nxt = i % 2, (i + 1) % 2
            torch.cuda.current_stream().wait_event(ready[cur])
            y = model(stage[cur])
            freed[cur].record()
            if i + 1 < nsteps:          # after the forward's launch: host-side packing overlaps the device work
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(freed[nxt])
                    produce(mode, i + 1, stage[nxt])
                    ready[nxt].record(copy_stream)
            metric_host.copy_(y[:, :, ::8, ::8].abs().mean().reshape(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()

    modes = ["fp32", "raw_uint8", "preshrunk_uint8"]
    h2d = {"fp32": B * 3 * S * S * 4, "raw_uint8": B * 3 * H * W, "preshrunk_uint8": B * 3 * sh * sw}
    for m in modes:
        run(m, 3)
    res = {m: [] for m in modes}
    for _ in range(reps):
        for m in modes:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(m, steps)
            res[m].append(B * steps / (time.perf_counter() - t0))
    out = {}
    for m in modes:
        v = res[m]
        out[m] = {"img_per_s_median": round(float(np.median(v)), 1), "img_per_s_runs": [round(x, 1) for x in v],
                  "h2d_bytes_per_step": h2d[m]}
    out["fp32"]["input"] = f"pinned fp32 [{B},3,{S},{S}] (the loader already resized / normalised / padded)"
    out["raw_uint8"]["input"] = f"{B} pinned uint8 3x{H}x{W} (copied straight from their pinned memory)"
    out["preshrunk_uint8"]["input"] = f"{B} pinned uint8 3x{sh}x{sw}"
    out["steps_per_run"], out["model"] = steps, f"EV-M (efficientvit_b1) {S}x{S} eval, CUDA graph"
    return out


def cpu_leg(n_images):
    mean = torch.tensor([123.675, 116.28, 103.53]).view(-1, 1, 1)
    std = torch.tensor([58.395, 57.12, 57.375]).view(-1, 1, 1)
    g = torch.Generator().manual_seed(2)
    imgs = [torch.randint(0, 256, (3, H, W), generator=g, dtype=torch.uint8) for _ in range(n_images)]
    from efficientsam3_b200.stage1.transforms import get_preprocess_shape
    oh, ow = get_preprocess_shape(H, W, S)

    def one(img):
        x = F.interpolate(img[None].float(), (oh, ow), mode="bilinear", align_corners=False, antialias=True).squeeze(0)
        x = (x - mean) / std
        return F.pad(x, (0, S - ow, 0, S - oh))

    res, prev = {}, torch.get_num_threads()
    ncores = os.cpu_count() or 1
    for threads in (1, ncores):
        torch.set_num_threads(threads)
        one(imgs[0])
        t0 = time.perf_counter()
        for im in imgs:
            one(im)
        ms = (time.perf_counter() - t0) * 1e3 / n_images
        res[f"threads_{threads}"] = {"ms_per_image": round(ms, 2), "img_per_s": round(1e3 / ms, 1)}
    torch.set_num_threads(prev)
    one_thread = res["threads_1"]["ms_per_image"]
    res["cpu_model"], res["logical_cpus"] = cpu_model(), ncores
    res["cores_for_650_img_per_s"] = round(650 * one_thread / 1e3, 1)
    res["note"] = ("torch CPU F.interpolate(antialias=True) + norm + pad of one 1500x2250 image (decode excluded); "
                   "cores_for_650_img_per_s = 650 img/s (one GPU's KD step) x single-thread time")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "preprocess_bench.json"))
    ap.add_argument("--calls", type=int, default=100)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-images", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("preprocess_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    from efficientsam3_b200 import _lib
    _lib.init(0)
    result = {"gpu": gpu_info(), "torch": torch.__version__}
    result["a_kernel"] = kernel_leg(dev, args.calls)
    print(json.dumps({"a_kernel": result["a_kernel"]}), flush=True)
    result["b_end_to_end"] = e2e_leg(dev, args.steps, args.reps)
    print(json.dumps({"b_end_to_end": result["b_end_to_end"]}), flush=True)
    result["c_cpu_reference_preprocessing"] = cpu_leg(args.cpu_images)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
