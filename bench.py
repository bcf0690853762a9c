#!/usr/bin/env python
"""bench.py -- headline benchmark of the monai_b200 hot path (sliding-window inference, voxels/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload unet_c2|swin_c3] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one full `SlidingWindowInferer(...)(volume, network)` pass over one synthetic volume.
  value : voxels/s with the volume already resident in HBM (CUDA-event timed, max over ranks)
  e2e   : the same call with a pinned HOST volume: H2D copy + inference + D2H copy of the logits inside the timed region
  roofline / cpu_baseline / clocks / gpu_launches : see DESIGN.md "Measurement"
`--impl reference` times the reference algorithm's CPU path (the oracle port: torch-CPU restatement, all host threads).
`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy (see dump_outputs); inputs and weights are seeded,
so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]
    "unet_c2": dict(
        desc="UNet(16,32,64,128,256; strides 2,2,2,2) sliding-window 256^3 fp16, roi 96^3, overlap 0.5, gaussian",
        vol=(256, 256, 256), roi=(96, 96, 96), overlap=0.5, mode="gaussian", sw_batch=25, net="unet_c2", windows=125,
        flop_per_window=2.96e9,
    ),
    # BASELINE.json configs[2]
    "swin_c3": dict(
        desc="SwinUNETR(feature_size=48) sliding-window 512^3 fp16, roi 96^3, overlap 0.5, gaussian",
        vol=(512, 512, 512), roi=(96, 96, 96), overlap=0.5, mode="gaussian", sw_batch=25, net="swin48", windows=1000,   # 25 divides the window share of 1, 2, 4 and 8 ranks
        flop_per_window=636e9,
    ),
    # BASELINE.json configs[4] (the multi-GPU config; also runnable on one GPU)
    "swin_c5": dict(
        desc="SwinUNETR(feature_size=48) sliding-window 512x512x1024 fp16, roi 96^3, overlap 0.5, gaussian",
        vol=(512, 512, 1024), roi=(96, 96, 96), overlap=0.5, mode="gaussian", sw_batch=25, net="swin48", windows=2100,
        flop_per_window=636e9,
    ),
    # BASELINE.json configs[3]
    "transforms_c4": dict(
        desc="Spacingd(1.25mm->1mm, bilinear) + RandAffined(prob 1, rotate .2, scale .1, translate 5, border) + GaussianSmoothd(sigma 1) on 32 x (1,256^3) fp32 MetaTensors",
        vol=(256, 256, 256), volumes=32, net=None,
    ),
}


DUMP_BUDGET = 32 << 20   # bytes that --dump-outputs writes, all arrays together


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each output as <out_dir>/<name>.npy in float32.  An output with more elements than its share of DUMP_BUDGET allows is
    written as its values at a fixed sample of flat indices, torch.randint(numel, (n,), generator=torch.Generator().manual_seed(0))."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BUDGET // 4 // len(arrays)
    for name, t in arrays.items():
        t = t.detach().as_subclass(torch.Tensor)
        if t.numel() > share:
            idx = torch.randint(t.numel(), (share,), generator=torch.Generator().manual_seed(0))
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


def _quiet_nccl() -> None:
    """Keep stdout to the single JSON line WITHOUT overriding the caller's NCCL_DEBUG: when the driver sets NCCL_DEBUG (to read the
    communicator lines), NCCL's log goes to its own file unless a destination is already configured."""
    if "NCCL_DEBUG" in os.environ:
        os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join(tempfile.gettempdir(), "nccl_%h_%p.log"))
    else:
        os.environ["NCCL_DEBUG"] = os.environ.get("B200_NCCL_DEBUG", "WARN")


def ncu_traffic(kernel: str):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/ncu_traffic.json: kernel ->
    {"dram_bytes_per_launch", "algorithmic_bytes_per_launch", "source"}); None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    try:
        return json.load(open(p)).get(kernel, {}).get("dram_bytes_per_launch")
    except (OSError, ValueError):
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf=d.get("bf16_tflops", 1590.0), tf_sustained=d.get("bf16_tflops_sustained", 1400.0), src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback")


def build_net(kind: str, device, half: bool):
    from weights import fill_state_dict

    if kind == "unet_c2":
        from monai_b200.networks.nets import UNet

        net = UNet(3, 1, 2, (16, 32, 64, 128, 256), (2, 2, 2, 2))
    elif kind == "swin48":
        from monai_b200.networks.nets import SwinUNETR

        net = SwinUNETR(in_channels=1, out_channels=2, feature_size=48)
    else:
        raise ValueError(kind)
    net.load_state_dict(fill_state_dict(net.state_dict(), 1))  # random-init weights of the named architecture
    net = net.eval().to(device)
    return net.half() if half else net


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                stdout=self.f, stderr=subprocess.DEVNULL,
            )
        except OSError:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def run_reference(args, wl):
    """CPU arm: the reference algorithm's CPU path (oracle port), all host threads, fp32."""
    from oracle import networks as onet
    from oracle import sliding_window as osw
    from weights import fill_state_dict

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(min(cores, int(os.environ.get("B200_REF_THREADS", "32"))))
    cores = torch.get_num_threads()
    if wl["net"] == "unet_c2":
        from monai_b200.networks.nets import UNet

        sd = fill_state_dict(UNet(3, 1, 2, (16, 32, 64, 128, 256), (2, 2, 2, 2)).state_dict(), 1)
        vol = wl["vol"]
        fwd = lambda a: onet.unet_forward(sd, torch.from_numpy(a), (2, 2, 2, 2)).numpy()  # noqa: E731
        sample = f"full {vol[0]}x{vol[1]}x{vol[2]} volume ({wl['windows']} windows) per step, fp32"
        scale = 1.0
    else:
        from monai_b200.networks.nets import SwinUNETR

        sd = fill_state_dict(SwinUNETR(in_channels=1, out_channels=2, feature_size=48).state_dict(), 1)
        vol = (144, 144, 96)  # 2x2x1 = 4 windows; cost is linear in windows (BASELINE.md section 3)
        fwd = lambda a: onet.swin_unetr_forward(sd, torch.from_numpy(a)).numpy()  # noqa: E731
        sample = "144x144x96 sub-volume (4 windows) per step, extrapolated linearly to 1000 windows, fp32"
        scale = 4.0 / wl["windows"]
    x = np.random.default_rng(0).standard_normal((1, 1, *vol)).astype(np.float32)
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            osw.sliding_window_inference(x, wl["roi"], 4, fwd, wl["overlap"], wl["mode"])
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
    full_vox = float(np.prod(wl["vol"]))
    sec_full = statistics.mean(times) / scale
    v = full_vox / sec_full
    line = {
        "impl": "reference", "metric": "voxels/sec sliding-window inference", "value": v, "unit": "voxels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_full * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": wl["desc"]},
        "cpu_baseline": {"value": v, "unit": "voxels/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def cpu_baseline_leg(wl, budget_s: float = 20.0) -> dict:
    from oracle import networks as onet
    from oracle import sliding_window as osw
    from weights import fill_state_dict

    cores = os.cpu_count() or 1
    if wl["net"] == "unet_c2":
        from monai_b200.networks.nets import UNet

        sd = fill_state_dict(UNet(3, 1, 2, (16, 32, 64, 128, 256), (2, 2, 2, 2)).state_dict(), 1)
        vol, nwin = (144, 144, 144), 8
        fwd = lambda a: onet.unet_forward(sd, torch.from_numpy(a), (2, 2, 2, 2)).numpy()  # noqa: E731
    else:
        from monai_b200.networks.nets import SwinUNETR

        sd = fill_state_dict(SwinUNETR(in_channels=1, out_channels=2, feature_size=48).state_dict(), 1)
        vol, nwin = (96, 96, 96), 1   # one window (636 GFLOP, ~3 s on a many-core host); windows are independent and equal in cost
        fwd = lambda a: onet.swin_unetr_forward(sd, torch.from_numpy(a)).numpy()  # noqa: E731
    x = np.random.default_rng(0).standard_normal((1, 1, *vol)).astype(np.float32)
    best, best_threads, passes = None, cores, 0
    t_all = time.perf_counter()
    with torch.no_grad():
        # oneDNN/ATen on many-core hosts can lose to a smaller pool on these small windows: take the best thread count
        # 32 threads first (the best pool on the many-core hosts measured so far), wider pools only while the budget lasts
        order = [min(cores, 32), cores] if wl["net"] != "unet_c2" else [min(cores, 32), min(cores, 16), min(cores, 64), cores]
        for threads in list(dict.fromkeys(order)):
            torch.set_num_threads(threads)
            for rep in range(2):
                t0 = time.perf_counter()
                osw.sliding_window_inference(x, wl["roi"], 4, fwd, wl["overlap"], wl["mode"])
                dt = time.perf_counter() - t0
                passes += 1
                if rep == 1 and (best is None or dt < best):
                    best, best_threads = dt, threads
            if time.perf_counter() - t_all > budget_s:
                break
    per_win = best / nwin
    v = float(np.prod(wl["vol"])) / (per_win * wl["windows"])
    return {"value": v, "unit": "voxels/s", "cores": best_threads, "host_cores": cores, "kind": "port",
            "sample": f"{vol[0]}x{vol[1]}x{vol[2]} sub-volume ({nwin} windows, fp32, torch-CPU oracle), {passes} passes over thread counts, best "
                      f"seconds/window extrapolated to {wl['windows']} windows"}


def _transform_pipeline(lazy: bool = False):
    from monai_b200.transforms import Compose, GaussianSmoothd, RandAffined, Spacingd

    pipe = Compose([
        Spacingd(keys=["image"], pixdim=(1.0, 1.0, 1.0), mode="bilinear"),
        RandAffined(keys=["image"], prob=1.0, rotate_range=(0.2,) * 3, scale_range=(0.1,) * 3, translate_range=(5,) * 3, mode="bilinear", padding_mode="border"),
        GaussianSmoothd(keys=["image"], sigma=1.0),
    ], lazy=lazy)   # lazy: Spacingd and RandAffined compose into ONE resample (monai/transforms/lazy/functional.py:84-296)
    pipe.transforms[1].set_random_state(seed=0)
    return pipe


def run_transforms(args, wl):
    """Config C4 (SURVEY.md section 8(d)): the spatial pre-processing pipeline on a batch of volumes; replicas-only across GPUs
    (DESIGN.md section 5), so N ranks each process the full batch and `value` is the aggregate."""
    from monai_b200 import _kernels as K
    from monai_b200 import _lib
    from monai_b200.data import MetaTensor

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _quiet_nccl()
    _lib.load()
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    nvol, shape = wl["volumes"], wl["vol"]
    aff = torch.diag(torch.tensor([1.25, 1.25, 1.25, 1.0], dtype=torch.float64))
    g = torch.Generator().manual_seed(0)
    host = [torch.rand((1, *shape), generator=g).pin_memory() for _ in range(nvol)]
    dev_vols = [h.to(dev) for h in host]
    pipe = _transform_pipeline()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out_host = None

    def step_resident():
        return [pipe({"image": MetaTensor(v, affine=aff)})["image"] for v in dev_vols]

    def step_e2e():
        nonlocal out_host
        for h in host:
            y = pipe({"image": MetaTensor(h.to(dev, non_blocking=True), affine=aff)})["image"]
            if out_host is None:
                out_host = torch.empty(tuple(y.shape), dtype=y.dtype).pin_memory()
            out_host.copy_(y, non_blocking=True)
        return y

    def timed(fn, steps, warmup):
        """Milliseconds of `steps` timed calls of fn and what the last one returned."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ms = 0.0
        for _ in range(steps):
            out = None   # a step's result is released before the next step runs
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            e1.synchronize()
            ms += e0.elapsed_time(e1)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    sampler = ClockSampler(local) if rank == 0 else None
    l0 = _lib.launch_count()
    ms_total, ys = timed(step_resident, args.steps, args.warmup)
    launches = (_lib.launch_count() - l0) * args.steps // (args.steps + args.warmup)
    clocks = sampler.stop() if sampler else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f"image_{i:02d}": y for i, y in enumerate(ys)})
    del ys
    ms_e2e, _ = timed(step_e2e, args.steps, 1)
    K.profile_start()
    y = step_resident()[-1]
    prof = K.profile_stop()
    # the same pipeline with Compose(lazy=True): reported next to the eager (reference default) number, not instead of it
    eager_pipe, pipe = pipe, _transform_pipeline(lazy=True)
    ms_lazy, _ = timed(step_resident, args.steps, 1)
    pipe = eager_pipe
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    pk = peaks()
    nvox = float(np.prod(shape)) * nvol * world
    ms_step = ms_total / args.steps
    name, st = max(prof.items(), key=lambda kv: kv[1]["ms"])
    avg_ms = st["ms"] / max(1, st["n"])
    ach = st.get("bytes", 0.0) / max(1, st["n"]) / (avg_ms * 1e-3) / 1e9
    line = {
        "metric": "voxels/sec spatial transform pipeline (input voxels)", "value": nvox / (ms_step * 1e-3), "unit": "voxels/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "volumes_per_step": nvol, "output_shape": list(y.shape), "l2": "256 MiB flush write between timed steps",
                   "parallelism": f"replicas x{world}" if world > 1 else "single GPU"},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": nvox / (ms_e2e / args.steps * 1e-3), "unit": "voxels/s", "h2d_bytes_per_step": sum(h.numel() * 4 for h in host),
                "d2h_bytes_per_step": int(out_host.numel() * 4 * nvol)},
        "roofline": {"kernel": name, "bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": None,
                     "peak_source": pk["src"], "launches": st["n"], "avg_launch_ms": avg_ms,
                     "share_of_kernel_time": st["ms"] / (sum(v["ms"] for v in prof.values()) or 1.0)},
        "kernels": {k: {"ms": round(v["ms"], 4), "n": v["n"]} for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])[:8]},
        "lazy": {"ms_per_step": ms_lazy / args.steps, "value": nvox / (ms_lazy / args.steps * 1e-3), "unit": "voxels/s",
                 "note": "Compose(lazy=True): Spacingd + RandAffined fused into one resample launch per volume"},
    }
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = transforms_cpu_leg(wl)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def transforms_cpu_leg(wl, volumes: int = 1) -> dict:
    """The oracle's torch-CPU restatement of the same three transforms on `volumes` full-size volumes."""
    from oracle import transforms as otr

    cores = os.cpu_count() or 1
    torch.set_num_threads(min(cores, int(os.environ.get("B200_REF_THREADS", "32"))))
    aff = np.diag([1.25, 1.25, 1.25, 1.0])
    g = torch.Generator().manual_seed(0)
    t0 = time.perf_counter()
    for i in range(volumes):
        img = torch.rand((1, *wl["vol"]), generator=g)
        a, _ = otr.spacing(img, aff, (1.0, 1.0, 1.0))
        b, _ = otr.rand_affine(a, i, (0.2,) * 3, (), (5,) * 3, (0.1,) * 3, None, "bilinear", "border")
        otr.gaussian_smooth(b, 1.0)
    dt = time.perf_counter() - t0
    return {"value": float(np.prod(wl["vol"])) * volumes / dt, "unit": "voxels/s", "cores": torch.get_num_threads(), "host_cores": cores,
            "kind": "port", "sample": f"{volumes} of {wl['volumes']} volumes (1x256^3 fp32 -> 320^3), torch-CPU oracle of the three transforms"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("B200_WORKLOAD", "swin_c3"), choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sw-batch", type=int, default=0, help="override the workload's sw_batch_size")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C2 / C4 lines appended to the default single-GPU run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of the workload's GPU path as DIR/<name>.npy "
                    f"(float32, at most {DUMP_BUDGET >> 20} MiB in all: larger outputs as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if os.environ.get("B200_BENCH_WATCHDOG"):
        import faulthandler

        faulthandler.dump_traceback_later(int(os.environ["B200_BENCH_WATCHDOG"]), exit=True)
    wl = dict(WORKLOADS[args.workload])
    if args.sw_batch > 0:
        wl["sw_batch"] = args.sw_batch
    if args.workload == "transforms_c4":
        if args.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                leg = transforms_cpu_leg(wl, volumes=max(1, min(args.steps, 3)))
                print(json.dumps({"impl": "reference", "metric": "voxels/sec spatial transform pipeline (input voxels)", "value": leg["value"],
                                  "unit": "voxels/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
                                  "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": wl["desc"]},
                                  "cpu_baseline": leg, "e2e": {"value": leg["value"], "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
            return
        return run_transforms(args, wl)
    if args.impl == "reference":
        return run_reference(args, wl)

    from monai_b200 import _kernels as K
    from monai_b200 import _lib
    from monai_b200.inferers import SlidingWindowInferer

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    _quiet_nccl()
    _lib.load()
    net = build_net(wl["net"], dev, half=True)
    # capture the network's CUDA graphs (full batch + this rank's remainder batch) BEFORE NCCL starts its helper
    # threads, so no capture ever runs concurrently with communicator activity
    per_rank = [wl["windows"] * (k + 1) // world - wl["windows"] * k // world for k in range(world)]
    for nb in sorted({wl["sw_batch"]} | {c % wl["sw_batch"] for c in per_rank if c % wl["sw_batch"]}):
        net(torch.zeros((nb, 1, *wl["roi"]), device=dev, dtype=torch.float16))
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    vol = wl["vol"]
    host = torch.randn((1, 1, *vol), generator=torch.Generator().manual_seed(0)).half().pin_memory()
    x_dev = host.to(dev)
    inferer = SlidingWindowInferer(wl["roi"], wl["sw_batch"], wl["overlap"], wl["mode"])
    if world > 1:
        from monai_b200.parallel import ShardedSlidingWindowInferer

        inferer = ShardedSlidingWindowInferer(wl["roi"], wl["sw_batch"], wl["overlap"], wl["mode"])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_resident():
        return inferer(x_dev, net)

    out_host = None
    if world > 1:
        # end to end, the sharded job moves every byte once: a rank uploads only the depth rows its windows read and
        # downloads only the rows of the result it owns (no broadcast of the slabs between GPUs)
        inferer_e2e = ShardedSlidingWindowInferer(wl["roi"], wl["sw_batch"], wl["overlap"], wl["mode"], gather=False)
        plan = inferer_e2e.plan(vol, world)
        (s_lo, s_hi), (o_lo, o_hi) = plan.slab[rank], plan.owned[rank]
        x_e2e = torch.zeros_like(x_dev)
        e2e_bytes = [host[:, :, s_lo:s_hi].numel() * host.element_size(), 0]

    def step_e2e():
        nonlocal out_host
        if world > 1:
            x_e2e[:, :, s_lo:s_hi].copy_(host[:, :, s_lo:s_hi], non_blocking=True)
            y = inferer_e2e(x_e2e, net)
            if out_host is None:
                out_host = torch.empty((*y.shape[:2], o_hi - o_lo, *y.shape[3:]), dtype=y.dtype).pin_memory()
            out_host.copy_(y[:, :, o_lo:o_hi], non_blocking=True)
            return y
        xd = host.to(dev, non_blocking=True)
        y = inferer(xd, net)
        if out_host is None:
            out_host = torch.empty(y.shape, dtype=y.dtype).pin_memory()
        out_host.copy_(y, non_blocking=True)
        return y

    def timed(fn, steps, warmup):
        """Milliseconds of `steps` timed calls of fn and what the last one returned."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ms = 0.0
        for _ in range(steps):
            out = None   # a step's result is released before the next step runs
            flush.fill_(1)  # L2 flush between timed iterations (untimed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            e1.synchronize()
            ms += e0.elapsed_time(e1)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    sampler = ClockSampler(local) if rank == 0 else None
    l0 = _lib.launch_count()
    ms_total, y = timed(step_resident, args.steps, args.warmup)
    launches = (_lib.launch_count() - l0) * args.steps // (args.steps + args.warmup)
    clocks = sampler.stop() if sampler else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"logits": y})
    del y
    ms_e2e, _ = timed(step_e2e, args.steps, 1)

    # per-kernel device time (CUDA events around every C-ABI launch, one extra untimed-for-value pass)
    K.profile_start()   # CUDA-graph replay is bypassed while profiling so every launch is individually timed
    step_resident()
    prof = K.profile_stop()

    # correctness of the sharded job, carried in the line: the gathered multi-GPU result against the single-GPU result of the
    # same volume (rank 0 runs the whole volume alone once, outside every timed region)
    parity = None
    if world > 1:
        y_sh = inferer(x_dev, net).float()
        if rank == 0:
            y_one = SlidingWindowInferer(wl["roi"], wl["sw_batch"], wl["overlap"], wl["mode"])(x_dev, net).float()
            diff = (y_sh - y_one).abs()
            parity = {"max_abs_diff": float(diff.max()), "max_abs": float(y_one.abs().max()), "mismatch_frac_1e-3": float((diff > 1e-3 * y_one.abs().max()).float().mean()),
                      "checksum_sharded": float(y_sh.double().sum()), "checksum_single": float(y_one.double().sum())}
            del y_one, diff
        del y_sh
        torch.cuda.synchronize()
        dist.barrier()

    # bytes moved per step, summed over the ranks (each rank uploads its slab rows and downloads its owned rows)
    h2d_total = e2e_bytes[0] if world > 1 else host.numel() * host.element_size()
    d2h_total = out_host.numel() * out_host.element_size() if out_host is not None else 0
    if dist is not None:
        tb = torch.tensor([float(h2d_total), float(d2h_total)], device=dev, dtype=torch.float64)
        dist.all_reduce(tb)
        h2d_total, d2h_total = float(tb[0].item()), float(tb[1].item())
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    nvox = float(np.prod(vol))
    ms_step = ms_total / args.steps
    pk = peaks()
    top = max(prof.items(), key=lambda kv: kv[1]["ms"]) if prof else (None, None)
    total_kernel_ms = sum(v["ms"] for v in prof.values()) or 1.0
    roofline = None
    if top[0] is not None:
        name, st = top
        flops, byts = st.get("flops", 0.0), st.get("bytes", 0.0)
        avg_ms = st["ms"] / max(1, st["n"])
        if flops and (flops / pk["tf"] / 1e12) >= (byts / pk["hbm"] / 1e9):
            ach = flops / max(1, st["n"]) / (avg_ms * 1e-3) / 1e12
            roofline = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"], "traffic": None}
        else:
            ach = byts / max(1, st["n"]) / (avg_ms * 1e-3) / 1e9
            roofline = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": None}
        roofline.update({"peak_source": pk["src"], "launches": st["n"], "avg_launch_ms": avg_ms, "share_of_kernel_time": st["ms"] / total_kernel_ms})
    line = {
        "metric": "voxels/sec sliding-window inference", "value": nvox / (ms_step * 1e-3), "unit": "voxels/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": wl["desc"], "sw_batch_size": wl["sw_batch"], "windows": wl["windows"], "l2": "256 MiB flush write between timed steps",
                   "accumulate": "fp32", "parallelism": f"depth-shard x{world}" if world > 1 else "single GPU"},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": nvox / (ms_e2e / args.steps * 1e-3), "unit": "voxels/s", "h2d_bytes_per_step": int(h2d_total), "d2h_bytes_per_step": int(d2h_total)},
        "model_tflops": wl["flop_per_window"] * wl["windows"] / (ms_step * 1e-3) / 1e12,
        "roofline": roofline,
        "kernels": {k: {"ms": round(v["ms"], 4), "n": v["n"]} for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])[:12]},
    }
    if roofline is not None:
        roofline["traffic"] = ncu_traffic(roofline["kernel"])
    if parity is not None:
        line["parity_vs_single_gpu"] = parity
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline_leg(wl)
    if world == 1 and args.workload == "swin_c3" and not args.no_secondary:
        line["secondary"] = secondary_lines()
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def secondary_lines() -> dict:
    """BASELINE.json configs[1] (UNet, 256^3) and configs[3] (transform pipeline) measured by this same script in sub-processes, so
    the driver-visible line carries them too (value, ms_per_step, e2e, roofline, cpu_baseline)."""
    out = {}
    for key, extra in (("unet_c2", ["--steps", "10", "--warmup", "3"]), ("transforms_c4", ["--steps", "3", "--warmup", "3"])):
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--workload", key, "--no-secondary", *extra], capture_output=True, text=True, timeout=600)
            js = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            d = json.loads(js[-1])
            out[key] = {k: d.get(k) for k in ("metric", "value", "unit", "ms_per_step", "config", "e2e", "roofline", "cpu_baseline", "gpu_launches", "kernels", "lazy") if k in d}
        except Exception as e:  # pragma: no cover - the headline line must survive a failing side measurement
            out[key] = {"error": f"{type(e).__name__}: {e}"}
    return out


if __name__ == "__main__":
    main()
