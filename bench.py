#!/usr/bin/env python
"""bench.py — images/sec of feather::Net::Forward on synthetic 224x224x3 input (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--model vgg16|resnet50|mobilenet_v1|single_conv]
                    [--batch B_per_gpu] [--precision tf32x3|tf32] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, NCCL)

One "step" = one Forward over one batch.  Default workload = BASELINE.json configs[1]: VGG-16 fp32, batch 64 per
GPU (weak scaling: every rank runs its own 64-image shard; the only collective is the weight broadcast at load).
Prints ONE JSON line on rank 0:
  value         whole-job images/s with the input batches already resident in HBM (CUDA events, max over ranks)
  e2e           same metric through the public API with pinned HOST buffers: H2D of the batch and D2H of the
                softmax output inside the timed region, every step
  roofline      every instrumented launch of one eager Forward, timed with CUDA events on the Net's stream and grouped by
                kernel class; the object describes the class with the largest share of the step (achieved =
                algorithmic direct-conv FLOPs, or algorithmic bytes for HBM-bound classes, / summed duration, against
                MEASURED_PEAKS.json) and lists the others under other_kernels
  cpu_baseline  the unmodified reference (oracle/_ref) on the host cores, bounded sample, rank 0 / N=1 only
`--impl reference` times only that CPU reference arm (no GPU work) and prints the same line shape.
`--dump-outputs DIR` writes, on rank 0, the output blob of the last timed step of each workload as DIR/<model>_<blob>.npy
(float32, batch x C x H x W); the inputs and weights are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

DEFAULT_BATCH = {"vgg16": 64, "resnet50": 128, "mobilenet_v1": 256, "single_conv": 64}
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES_PER_WORKLOAD = 16 << 20  # at most three workloads: 48 MB in all


def env_int(name: str, default: int) -> int:
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peaks() -> tuple[dict, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return json.loads(p.read_text()), "measured"
        except Exception:
            pass
    # fallback stated by /opt/skills/guides/B200_PROFILING.md
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def model_files(model: str, rank: int, barrier) -> tuple[str, str, float, tuple]:
    """Rank 0 writes the synthetic ncnn .param/.bin once per box (random-init weights, fixed seed)."""
    from feathercnn_b200.tools import modelgen
    cache = Path(os.environ.get("FEATHER_BENCH_CACHE", "/tmp/feather_bench_models"))
    prefix = cache / f"{model}_seed0"
    meta = cache / f"{model}_seed0.json"
    if rank == 0 and not (meta.exists() and Path(str(prefix) + ".bin").exists()):
        cache.mkdir(parents=True, exist_ok=True)
        m = modelgen.ZOO[model]()
        m.save(prefix)
        meta.write_text(json.dumps({"flops": m.flops, "input": list(m.shape["data"])}))
    barrier()
    info = json.loads(meta.read_text())
    return str(prefix) + ".param", str(prefix) + ".bin", float(info["flops"]), tuple(info["input"])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed regions (B200_PROFILING.md recipe).

    nvidia-smi needs ~0.1-0.5 s to deliver its first row, longer than a short timed region, so the poller is started
    before the warm-up and only the rows received inside the marked windows (device-resident leg and end-to-end leg,
    both under the same load) are used."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows: list[tuple[float, list[str]]] = []
        self.windows: list[list[float]] = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def begin(self):
        self.windows.append([time.perf_counter(), float("inf")])

    def end(self):
        if self.windows:
            self.windows[-1][1] = time.perf_counter()

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def collect(slack: float):
            sm, mx, reasons = [], [], set()
            for t, r in self.rows:
                if len(r) < 8 or not any(w0 - slack <= t <= w1 + slack for w0, w1 in self.windows):
                    continue
                try:
                    sm.append(float(r[1])); mx.append(float(r[2]))
                except ValueError:
                    continue
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            return sm, mx, reasons

        sm, mx, reasons = collect(0.0)
        how = "inside the timed regions"
        if not sm:  # a region shorter than the polling period: take the rows right around it
            sm, mx, reasons = collect(0.12)
            how = "within 120 ms of the timed regions"
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "sampled": how,
                "window_s": round(sum(min(w1, time.perf_counter()) - w0 for w0, w1 in self.windows), 3)}


def common_config(model: str, batch: int, in_shape, world: int) -> dict:
    """The `config` object shared verbatim by both arms (the driver compares them key by key)."""
    return {"workload": f"{model}_b{batch}_{in_shape[1]}x{in_shape[2]}", "batch_per_gpu": batch,
            "global_batch": batch * world, "input": f"{in_shape[0]}x{in_shape[1]}x{in_shape[2]} fp32 synthetic"}


def cpu_reference_run(param: str, binf: str, batch: int, steps: int, budget_s: float) -> dict:
    """The reference's own CPU Forward on the host cores.

    The reference has no batch dimension (src/blob.cpp:73) and is race-free only at 1 thread (src/net.cpp:38), so a
    "step" (= one batch of `batch` images) is run as independent single-image Forwards spread over P single-thread
    worker processes, P = usable cores (physical cores bounded by the container's CPU quota).  First a 1-process probe
    gives the 1-thread figure (SURVEY.md §8d (i)) and sizes the sample so the run fits `budget_s`."""
    from oracle import cpu_bench
    procs, how = cpu_bench.usable_cores()
    one = cpu_bench.run(param, binf, procs=1, warmup=1, iters=2)
    t1 = one["sec_per_forward_mean"]
    per_worker = -(-batch * steps // procs)  # Forwards per worker for `steps` batches
    est = per_worker * t1 * 1.3
    steps_run = steps
    if est > budget_s:  # bounded sample: fewer batches, and say so in `steps`
        steps_run = max(1, int(steps * budget_s / est))
        per_worker = max(1, -(-batch * steps_run // procs))
    r = cpu_bench.run(param, binf, procs=procs, warmup=1, iters=per_worker)
    ips = r["images_per_s"]
    return {"images_per_s": ips, "procs": r["procs"], "kind": r["kind"], "steps_run": steps_run,
            "forwards_per_worker": per_worker, "timed_images": per_worker * r["procs"],
            "ms_per_step": 1e3 * batch / ips, "sec_per_forward_per_core": r["sec_per_forward_mean"],
            "images_per_s_1thread": 1.0 / t1, "sec_per_forward_1thread": t1, "cores_how": how,
            "sample": (f"{r['procs']} single-thread processes x (1 warm-up + {per_worker} timed) whole-net Forward of the same "
                       f"model, batch 1 each (the reference has no batch dimension); 1-thread probe: 1 process x 2 timed")}


def run_reference(args, rank: int, world: int) -> None:
    if rank != 0:
        return
    param, binf, flops, in_shape = model_files(args.model, 0, lambda: None)
    r = cpu_reference_run(param, binf, args.batch, max(1, args.steps), budget_s=150.0)
    line = {
        "impl": "reference", "metric": "images/sec", "value": r["images_per_s"], "unit": "images/s",
        "n_gpus": args.gpus, "steps": r["steps_run"], "warmup": 1,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(args.model, args.batch, in_shape, max(1, world)),
        "details": {"impl_detail": "unmodified FeatherCNN AVX build (oracle/_ref); one step = one batch of batch_per_gpu "
                                   "images run as independent single-image Forwards, one single-thread process per usable core",
                    "requested_steps": args.steps, "timed_images": r["timed_images"],
                    "forwards_per_worker": r["forwards_per_worker"], "cores_how": r["cores_how"]},
        "cpu_baseline": {"value": r["images_per_s"], "unit": "images/s", "cores": r["procs"], "kind": r["kind"],
                         "sample": r["sample"], "value_1thread": r["images_per_s_1thread"],
                         "sec_per_forward_per_core": r["sec_per_forward_per_core"]},
        "e2e": {"value": r["images_per_s"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


KERNEL_CLASS_NAMES = ["tensor_gemm_ts_kernel (tcgen05 kind::tf32, Winograd/im2col/FC GEMM)",
                      "conv_igemm_kernel (tcgen05 kind::f16 BF16x3 / kind::tf32 implicit-GEMM conv)", "wino_input_kernel",
                      "wino_output_kernel", "pooling_kernel", "depthwise kernels", "element-wise kernels"]


def roofline_leg(net, booster, dev_batches, n_rot, ms_step: float, model: str) -> dict:
    """Every instrumented launch of two eager Forwards, timed with CUDA events on the Net's stream, by kernel class."""
    import ctypes
    lib = booster.fcuda()
    net._lib.fnet_set_cuda_graph(net._h, 0)
    try:
        net.FeedInputDevice(dev_batches[0].data_ptr(), tuple(dev_batches[0].shape))
        net.Forward(); net.Synchronize()
        lib.fcuda_profile_tensor_gemm(1)
        reps = 2
        for i in range(reps):
            d = dev_batches[i % n_rot]
            net.FeedInputDevice(d.data_ptr(), tuple(d.shape))
            net.Forward()
        net.Synchronize()
        peaks, how = measured_peaks()
        # kernels timed inside a long step -> the sustained figures; fallbacks = /opt/skills/guides/B200_PROFILING.md
        tf_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
        hbm_peak = float(peaks.get("hbm_gbs", 6500.0))
        classes = []
        for kind, name in enumerate(KERNEL_CLASS_NAMES):
            ms_t, af, mf, ab, nl = (ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_double(),
                                    ctypes.c_longlong())
            lib.fcuda_profile_collect_kind(kind, ctypes.byref(ms_t), ctypes.byref(af), ctypes.byref(mf),
                                           ctypes.byref(ab), ctypes.byref(nl))
            if nl.value == 0 or ms_t.value <= 0:
                continue
            sec = ms_t.value * 1e-3
            tensor = kind <= 1
            ach = af.value / sec / 1e12 if tensor else ab.value / sec / 1e9
            peak = tf_peak if tensor else hbm_peak
            c = {"kernel": name, "bound": "tensor" if tensor else "hbm", "achieved": ach, "peak": peak,
                 "unit": "TFLOP/s" if tensor else "GB/s", "frac": ach / peak,
                 "launches_per_step": nl.value / reps, "avg_launch_us": 1e3 * ms_t.value / nl.value,
                 "share_of_step": (ms_t.value / reps) / ms_step}
            if tensor:
                c["algorithmic_gflop_per_launch"] = af.value / nl.value / 1e9
                c["algorithmic_gb_per_launch"] = ab.value / nl.value / 1e9
                c["hbm_gbps_at_algorithmic_bytes"] = ab.value / sec / 1e9
                c["tensor_pipe_tflops_issued"] = mf.value / sec / 1e12  # 3 MMAs per product in 3xTF32 mode
            else:
                c["algorithmic_gb_per_launch"] = ab.value / nl.value / 1e9
            classes.append(c)
        lib.fcuda_profile_tensor_gemm(0)
        if not classes:
            return {"error": "no instrumented launches"}
        classes.sort(key=lambda c: -c["share_of_step"])
        roof = dict(classes[0])
        roof["peak_source"] = (f"{how}: " + ("bf16_tflops_sustained" if roof["bound"] == "tensor" else "hbm_gbs") +
                               " (kernel timed inside a long step)")
        roof["traffic"] = None
        for tr in sorted((ROOT / "profiles").glob("r0*_kernel_traffic.json"), reverse=True):
            try:
                v = json.loads(tr.read_text()).get(model, {}).get(roof["kernel"].split()[0])
            except Exception:
                v = None
            if v is not None:
                roof["traffic"] = v
                roof["traffic_source"] = f"profiles/{tr.name} (dram__bytes_read+write per launch, ncu --set full)"
                break
        roof["other_kernels"] = classes[1:]
        return roof
    except Exception as e:  # the roofline leg explains the number, it must never cost the bench line
        return {"error": f"{type(e).__name__}: {e}"[:300]}
    finally:
        lib.fcuda_profile_tensor_gemm(0)


def parity_gate(net, param: str, binf: str, in_shape, batch: int, image_index: int) -> dict:
    """SURVEY.md §8d "parity gate in the same run": image 0 of a batch forwarded through the BENCHMARKED configuration
    (fusion, CUDA graph, bench batch size) against the reference's Forward of the same image, every surviving blob."""
    from feathercnn_b200.tools import modelgen
    from oracle import cpu_bench
    try:
        x0 = modelgen.synthetic_input(in_shape, image_index)
        xb = np.stack([x0] + [modelgen.synthetic_input(in_shape, image_index + 1 + (i % 3)) for i in range(batch - 1)])
        net.Forward(xb)  # FeedInputBatch + Forward; graph key of this shape was captured by the earlier legs or runs eagerly
        names = net.BlobNames()
        ref, kind = cpu_bench.dump_blobs(param, binf, image_index)
        worst, worst_blob, n = 0.0, None, 0
        for b in names:
            if b not in ref:
                continue
            try:
                got = net.Extract(b)[0]
            except Exception:
                continue  # fused away / never materialised
            want = ref[b]
            if got.size != want.size:
                continue
            denom = max(float(np.abs(want).max()), 1e-30)
            e = float(np.abs(got.reshape(want.shape).astype(np.float64) - want).max()) / denom
            n += 1
            if e > worst:
                worst, worst_blob = e, b
        return {"parity_max_rel": worst, "worst_blob": worst_blob, "blobs_compared": n, "tolerance": 1e-3,
                "pass": bool(n > 0 and worst <= 1e-3), "oracle": f"oracle/_ref ({kind})",
                "how": f"image 0 of a batch of {batch}, fusion+graph as benchmarked, max|d|/max|ref| per blob"}
    except Exception as e:
        return {"parity_max_rel": None, "pass": False, "error": f"{type(e).__name__}: {e}"[:300]}


def rotating_batches(batch_bytes: int) -> int:
    """How many input batches the timed steps rotate through: together larger than L2, at least 2, at most 8."""
    return min(8, max(2, -(-int(1.25 * L2_BYTES) // batch_bytes)))


def input_batch(in_shape, B: int, rank: int, n_rot: int, r: int) -> np.ndarray:
    """Rotating batch r of `rank`: four seeded synthetic images repeated to B; step i feeds batch i % n_rot."""
    from feathercnn_b200.tools import modelgen
    base = np.stack([modelgen.synthetic_input(in_shape, (rank * n_rot + r) * 4 + i) for i in range(min(B, 4))])
    return np.resize(base, (B,) + tuple(in_shape))


def dump_output(net, out_name: str, model: str, out_dir: Path) -> None:
    """What the last timed Forward left in the output blob, as a caller would Extract it; past the per-workload byte
    budget only the first images are kept (a fixed sample)."""
    out = np.ascontiguousarray(net.Extract(out_name), np.float32)
    keep = max(1, DUMP_BYTES_PER_WORKLOAD // max(1, out[0].nbytes))
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / f"{model}_{out_name}.npy", out[:keep])


def run_workload(args, model: str, B: int, rank: int, world: int, local_rank: int, barrier, full: bool,
                 cpu_leg: bool) -> dict | None:
    """Loads `model`, times the device-resident and end-to-end legs on every rank; rank 0 returns the result dict."""
    import torch
    import torch.distributed as dist

    from feathercnn_b200 import booster
    from feathercnn_b200 import dist as fdist
    from feathercnn_b200.tools import modelgen

    dev = torch.device(f"cuda:{local_rank}")
    param, binf, flops_per_image, in_shape = model_files(model, rank, barrier)
    t_load = time.perf_counter()
    net = fdist.load_net_distributed(param, binf, local_rank, fusion=not args.no_fusion, cuda_graph=not args.no_graph)
    stream = torch.cuda.Stream(device=dev)
    net.SetStream(stream.cuda_stream)
    t_load = time.perf_counter() - t_load

    batch_bytes = B * int(np.prod(in_shape)) * 4
    n_rot = rotating_batches(batch_bytes)
    host_batches = []
    for r in range(n_rot):
        hb = torch.empty((B,) + tuple(in_shape), dtype=torch.float32).pin_memory()
        hb.copy_(torch.from_numpy(input_batch(in_shape, B, rank, n_rot, r)))
        host_batches.append(hb)
    dev_batches = [hb.to(dev) for hb in host_batches]
    out_name = "prob" if "prob" in net.BlobNames() else sorted(b for b in net.BlobNames() if b != "data")[-1]
    torch.cuda.synchronize(dev)

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident leg ("value") -------------------------------------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    res: dict = {}
    with torch.cuda.stream(stream):
        for i in range(args.warmup + 2 * n_rot):  # per rotating buffer: one eager pass, then the graph capture
            d = dev_batches[i % n_rot]
            net.FeedInputDevice(d.data_ptr(), tuple(d.shape))
            net.Forward()
        net.Synchronize()
        launches = net.launches_per_forward
        barrier()
        torch.cuda.synchronize(dev)
        if sampler:
            sampler.begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            d = dev_batches[i % n_rot]
            net.FeedInputDevice(d.data_ptr(), tuple(d.shape))
            net.Forward()
        e1.record(stream)
        e1.synchronize()
        torch.cuda.synchronize(dev)
        barrier()
        if sampler:
            sampler.end()
        ms_dev = max_over_ranks(e0.elapsed_time(e1))
        if args.dump_outputs and rank == 0:
            dump_output(net, out_name, model, Path(args.dump_outputs))

        if args.lean:
            if sampler:
                sampler.stop()
            return {"lean": True, "model": model, "value": world * B * args.steps / (ms_dev * 1e-3),
                    "ms_per_step": ms_dev / args.steps, "launches_per_step": int(launches)} if rank == 0 else None

        # ---- end-to-end legs: pinned host input -> H2D -> Forward -> D2H of the result, every step ----------
        n, c, h, w = net.BlobShape(out_name)
        host_outs = [torch.empty((n, c, h, w), dtype=torch.float32).pin_memory() for _ in range(2)]
        d2h_bytes = host_outs[0].numel() * 4
        # (a) pipelined (the public SubmitBatch / WaitBatch API): the H2D copy of step i+1 runs on a copy stream
        #     behind an event while step i computes; two batches in flight; every step still pays its own copies
        for i in range(max(4, args.warmup)):
            net.WaitBatch(net.SubmitBatch(host_batches[i % n_rot].data_ptr(), B, out_name, host_outs[i & 1].data_ptr()))
        barrier()
        torch.cuda.synchronize(dev)
        if sampler:
            sampler.begin()
        e0.record(stream)
        t_wall = time.perf_counter()
        prev = None
        for i in range(args.steps):
            t = net.SubmitBatch(host_batches[i % n_rot].data_ptr(), B, out_name, host_outs[i & 1].data_ptr())
            if prev is not None:
                net.WaitBatch(prev)  # the caller holds step i-1's result while step i is in flight
            prev = t
        net.WaitBatch(prev)
        e1.record(stream)
        e1.synchronize()
        t_wall = time.perf_counter() - t_wall
        if sampler:
            sampler.end()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        wall_e2e = max_over_ranks(1e3 * t_wall)
        # (b) serial (README-style Forward(float*) then ExtractBlob, nothing overlapped) for comparison
        for i in range(2):
            net.ForwardBatchHostPtr(host_batches[i % n_rot].data_ptr(), B)
            net.ExtractInto(out_name, host_outs[0].data_ptr())
        torch.cuda.synchronize(dev)
        e0.record(stream)
        ser_steps = max(3, args.steps // 2)
        for i in range(ser_steps):
            net.ForwardBatchHostPtr(host_batches[i % n_rot].data_ptr(), B)
            net.ExtractInto(out_name, host_outs[0].data_ptr())  # D2H + stream sync
        e1.record(stream)
        e1.synchronize()
        ms_serial = max_over_ranks(e0.elapsed_time(e1)) / ser_steps
        clocks = sampler.stop() if sampler else None

        # ---- every rank forwards the SAME batch once: output checksums must agree (weight broadcast -> AttachWeights)
        common = np.stack([modelgen.synthetic_input(in_shape, 900 + (i % 4)) for i in range(min(B, 8))])
        net.Forward(common)
        out_common = net.Extract(out_name)
        digest = float(np.abs(out_common.astype(np.float64)).sum()) + float((out_common.astype(np.float64) ** 2).sum())
        checks = [digest]
        if world > 1:
            t = torch.tensor([digest], device=dev, dtype=torch.float64)
            allc = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allc, t)
            checks = [float(v.item()) for v in allc]
        ranks_agree = all(c == checks[0] for c in checks)

        roof = parity = None
        if rank == 0 and full:
            roof = roofline_leg(net, booster, dev_batches, n_rot, ms_dev / args.steps, model)
            net._lib.fnet_set_cuda_graph(net._h, 0 if args.no_graph else 1)
            parity = parity_gate(net, param, binf, in_shape, B, 0)

    if rank != 0:
        del net
        return None
    total_images = world * B * args.steps
    res = {
        "model": model, "value": total_images / (ms_dev * 1e-3), "unit": "images/s", "ms_per_step": ms_dev / args.steps,
        "config": common_config(model, B, in_shape, world),
        "e2e": {"value": total_images / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": batch_bytes,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": ms_e2e / args.steps,
                "wall_ms_per_step": wall_e2e / args.steps,
                "api": "Net::SubmitBatch / WaitBatch (double-buffered: H2D of step i+1 behind an event while step i computes)",
                "serial_value": world * B / (ms_serial * 1e-3), "serial_ms_per_step": ms_serial},
        "launches_per_step": int(launches), "gpu_launches": int(launches) * args.steps,
        "algorithmic_tflops": (total_images / (ms_dev * 1e-3)) * flops_per_image / 1e12,
        "gflop_per_image": flops_per_image / 1e9, "load_s": round(t_load, 3), "n_rot": n_rot, "batch_bytes": batch_bytes,
        "clocks": clocks, "roofline": roof, "parity": parity,
        "rank_checksums": {"equal": ranks_agree, "values": checks[:8],
                           "what": "sum|p| + sum p^2 of the output for one batch forwarded identically on every rank"},
    }
    if cpu_leg:
        try:
            r = cpu_reference_run(param, binf, B, 1, budget_s=25.0)
            res["cpu_baseline"] = {"value": r["images_per_s"], "unit": "images/s", "cores": r["procs"], "kind": r["kind"],
                                   "sample": r["sample"], "sec_per_forward_per_core": r["sec_per_forward_per_core"],
                                   "value_1thread": r["images_per_s_1thread"], "cores_how": r["cores_how"]}
        except Exception as e:  # the baseline is reported, never required for the GPU number
            res["cpu_baseline"] = {"value": None, "unit": "images/s", "cores": 0, "kind": "unavailable", "sample": str(e)[:200]}
    del net
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default=None, choices=["vgg16", "resnet50", "mobilenet_v1", "single_conv"],
                    help="one workload only (default: VGG-16 headline + ResNet-50 and MobileNet-v1 under `workloads`)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: BASELINE.json config)")
    ap.add_argument("--precision", default="fp32split", choices=["fp32split", "tf32x3", "tf32"],
                    help="fp32split (default): fp32-equivalent split operands, BF16x3 in the implicit GEMM + 3xTF32 in the "
                         "TensorGEMM; tf32x3: 3xTF32 everywhere; tf32: single TF32 MMA (not fp32-equivalent)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-fusion", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--l2-chunk-mb", type=float, default=None)
    ap.add_argument("--lean", action="store_true", help="profiling aid: device-resident leg only (no e2e / roofline / cpu legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output blob of the last timed step of each workload to DIR/<model>_<blob>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    headline = args.model or "vgg16"
    extra = [] if (args.model or args.lean) else ["resnet50", "mobilenet_v1"]
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        args.model = headline
        args.batch = args.batch if args.batch > 0 else DEFAULT_BATCH[headline]
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from feathercnn_b200 import booster

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])

    booster.set_precision({"tf32": booster.PRECISION_TF32, "tf32x3": booster.PRECISION_TF32X3,
                           "fp32split": booster.PRECISION_FP32_SPLIT}[args.precision])
    if args.l2_chunk_mb is not None:
        booster.set_l2_chunk_bytes(int(args.l2_chunk_mb * 1024 * 1024))

    B = args.batch if args.batch > 0 else DEFAULT_BATCH[headline]
    head = run_workload(args, headline, B, rank, world, local_rank, barrier, full=True,
                        cpu_leg=(world == 1 and not args.no_cpu_baseline))
    others = []
    for m in extra:  # BASELINE.json metric names VGG-16 AND ResNet-50; configs[2-4] (config 5 = resnet50 b128/GPU at --gpus 8)
        try:
            r = run_workload(args, m, DEFAULT_BATCH[m], rank, world, local_rank, barrier, full=True,
                             cpu_leg=(world == 1 and not args.no_cpu_baseline))
        except Exception as e:
            r = {"model": m, "error": f"{type(e).__name__}: {e}"[:300]} if rank == 0 else None
        if r is not None:
            others.append(r)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if head.get("lean"):
        print(json.dumps(head), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    cfg = dict(head["config"])
    line = {
        "metric": "images/sec", "value": head["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "tf32" if args.precision == "tf32" else "f32", "data": "synthetic",
        "config": cfg,
        "details": {"parallelism": f"batch-shard x{world} (weights broadcast once over NCCL, no collective in Forward)",
                    "tensor_core_mode": {"fp32split": "fp32-equivalent split operands, fp32 accumulation: BF16x3 (p1*q1 + p1*q2 + "
                                                      "p2*q1, kind::f16) in the implicit GEMM, 3xTF32 in the Winograd / FC TensorGEMM; "
                                                      "accuracy = parity_max_rel",
                                         "tf32x3": "3xTF32 split (fp32-equivalent) in every contraction",
                                         "tf32": "TF32"}[args.precision],
                    "algorithms": "tuned SelectAlgo (reference rule, then Winograd -> implicit GEMM when IC,OC <= 128 and OW >= 28, "
                                  "im2col -> implicit GEMM): Winograd F(6,3)+TensorGEMM / SGECONV implicit GEMM / depthwise",
                    "fusion": not args.no_fusion, "cuda_graph": not args.no_graph,
                    "l2_policy": f"{head['n_rot']} rotating input batches ({head['n_rot'] * head['batch_bytes'] / 2**20:.0f} MiB > L2); "
                                 f"activations per step far exceed the 126 MB L2",
                    "gflop_per_image": head["gflop_per_image"], "load_s": head["load_s"]},
        "clocks": head["clocks"],
        "e2e": head["e2e"],
        "gpu_launches": head["gpu_launches"],
        "launches_per_step": head["launches_per_step"],
        "algorithmic_tflops": head["algorithmic_tflops"],
        "roofline": head["roofline"],
        "cpu_baseline": head.get("cpu_baseline"),
        "parity": head["parity"],
        "parity_max_rel": (head["parity"] or {}).get("parity_max_rel"),
        "rank_checksums": head["rank_checksums"],
        "workloads": [{k: v for k, v in o.items() if k not in ("n_rot", "batch_bytes")} for o in others],
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
