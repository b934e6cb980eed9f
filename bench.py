#!/usr/bin/env python
"""bench.py — CSNet forward throughput on B200 (BASELINE.json configs[1]: csnet-L-x2 inference, bs 256,
224x224, fp16 activation storage / fp32 accumulate), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = whole-job images/s with inputs resident in HBM; `e2e` = the same
through the host-buffer C-ABI call (H2D + program + D2H per step, pinned memory); `roofline` = the dominant
kernel's algorithmic bytes / its live CUDA-event time vs the measured HBM peak; `cpu_baseline` = the oracle
port (same ATen calls the reference makes) timed on this box's host cores on a bounded sample.
`--impl reference` times that CPU implementation as the reference arm.  `--dump-outputs DIR` also writes the logits
of the last timed step (rank 0) to DIR/logits.npy; the inputs are seeded, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec CSNet fwd 224x224"
UNIT = "images/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="infer", choices=["infer", "train", "csf"],
                    help="infer (default, BASELINE configs[1]); train: fwd+bwd+Adam step (configs 3-4 shape, fp32 kernels); "
                         "csf: CSF+Res2Net-50 inference (config 5: bs 64, 352x352, fp16; backbone on torch/cuDNN, head on the engine)")
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    ap.add_argument("--size", type=int, default=224)
    ap.add_argument("--dtype", default="fp16", choices=["fp32", "fp16", "bf16"])
    ap.add_argument("--model", default="csnet-L-x2")
    ap.add_argument("--cpu-sample", type=int, default=16, help="images per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-ops", action="store_true", help="print the per-op time table to stderr")
    ap.add_argument("--train-batch", type=int, default=256, help="images per GPU of the `train` sub-record's step")
    ap.add_argument("--train-recompute", action="store_true",
                    help="train sub-record with ILBlock-granular recompute (Trainer(recompute=True)): ~3x less activation memory, one extra forward")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the train sub-record, the eager-GPU baseline and the extra configs (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the float32 logits of the last timed step to DIR/logits.npy (default mode and impl only)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.mode != "infer"):
        ap.error("--dump-outputs covers the default workload: --impl ours --mode infer")
    return a


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write each array as float32 `path/<name>.npy`.  Above DUMP_BYTES in all, each array is replaced by the same fixed,
    seeded sample of its flattened elements (in index order), so dumps made with the same arguments stay comparable."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    for name, v in arrays.items():
        if total > DUMP_BYTES:
            keep = v.size * DUMP_BYTES // total
            v = v.reshape(-1)[np.sort(np.random.default_rng(0).choice(v.size, keep, replace=False))]
        np.save(os.path.join(path, f"{name}.npy"), v)


def workload_config(a, world):
    return {"workload": f"{a.model} inference, {a.batch} img/GPU x {a.size}x{a.size}, {a.dtype} storage / fp32 accumulate",
            "model_weights": "shipped checkpoint (tests/golden npz)", "per_gpu_batch": a.batch,
            "global_batch": a.batch * world, "size": a.size, "parallelism": f"dp{world} (independent batches, no collective)",
            "l2": "activations of one step (>2 GB) exceed the 126 MB L2; no explicit flush"}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (tests infra) — same torch ATen calls as the reference module, all host threads
# ---------------------------------------------------------------------------------------------------
def cpu_forward_timer(a, n_img):
    import torch

    from oracle import csnet_oracle as O
    from sod100k_b200 import checkpoints, synth

    cfg, sd = checkpoints.load_npz(a.model)
    sd = {k: torch.from_numpy(v) for k, v in sd.items()}
    x = torch.from_numpy(synth.randn_images(n_img, a.size, a.size, 1234))

    def step():
        with torch.no_grad():
            O.csnet_forward(cfg, sd, x)

    # "all the host threads it can use": these are ~400 tiny ATen calls per forward, and oversubscribing a
    # 100+-thread box makes them SLOWER (measured 0.3 img/s at 128 threads vs 8.7 img/s at 8), so pick the
    # best thread count from a short sweep and report it as `cores`.
    ncpu = os.cpu_count() or 1
    best, cores = None, ncpu
    for nt in sorted({t for t in (4, 8, 16, 32, 64, ncpu) if t <= ncpu}):
        torch.set_num_threads(nt)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, nt
    torch.set_num_threads(cores)
    return step, cores


def cpu_baseline(a, budget_s=20.0):
    step, cores = cpu_forward_timer(a, a.cpu_sample)
    step()                                           # warm-up
    times, t_all = [], time.perf_counter()
    while len(times) < 2 or (time.perf_counter() - t_all < budget_s and len(times) < 9):
        t = time.perf_counter()
        step()
        times.append(time.perf_counter() - t)
    med = statistics.median(times)
    return {"value": a.cpu_sample / med, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle/csnet_oracle.py forward (reference's ATen calls, fp32, eval) on {a.cpu_sample} of the "
                      f"{a.size}x{a.size} images, median of {len(times)} runs, torch threads={cores}"}


def run_reference(a, rank):
    if rank != 0:
        return
    step, cores = cpu_forward_timer(a, a.cpu_sample)
    for _ in range(max(1, min(a.warmup, 2))):
        step()
    k = a.steps                                      # each step is a few seconds of CPU work
    t = time.perf_counter()
    for _ in range(k):
        step()
    dt = time.perf_counter() - t
    val = a.cpu_sample * k / dt
    sample = (f"{k} steps x {a.cpu_sample} images of the workload (the CPU path cannot finish {a.batch}-image steps "
              f"in minutes), all {cores} host threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": k,
        "warmup": a.warmup, "ms_per_step": 1e3 * dt / k, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": workload_config(a, a.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(dev)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [v.strip() for v in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def op_bytes(prog, op, n):
    """Algorithmic bytes of ONE op launch: distinct source slices read once + destination written once."""
    from sod100k_b200 import ir

    seen, total = set(), 0
    for q in op.paths:
        key = (q.src, q.c0, q.cin)
        if key in seen:
            continue
        seen.add(key)
        t = prog.tensors[q.src]
        total += q.cin * t.H * t.W * ir.DTYPE_BYTES[t.dtype]
    for t_id in (op.dst, getattr(op, "dst2", -1)):               # a fused ILBlock writes two tensors (hi and lo branch)
        if t_id is None or t_id < 0:
            continue
        d = prog.tensors[t_id]
        total += d.C * d.H * d.W * ir.DTYPE_BYTES[d.dtype]
    return n * total


def gpu_eager_baseline(a, dev, steps=5):
    """BASELINE.md §4: eager PyTorch on the SAME B200 — the oracle's functional forward (exactly the reference module's
    ATen calls: F.conv2d / batch_norm / prelu / pooling / interpolate -> cuDNN / ATen kernels), fp32 and torch.autocast(fp16),
    NCHW as the reference runs.  A measured baseline, not the product: none of our kernels run here."""
    import torch

    from oracle import csnet_oracle as O
    from sod100k_b200 import checkpoints, synth

    cfg, sd = checkpoints.load_npz(a.model)
    sd = {k: torch.from_numpy(v).to(dev) for k, v in sd.items()}
    B, S = a.batch, a.size
    x = torch.from_numpy(synth.randn_images(min(B, 32), S, S, 1234)).repeat((B + 31) // 32, 1, 1, 1)[:B].to(dev)
    out = {}
    for name, ctx in (("fp32", None), ("autocast_fp16", torch.autocast("cuda", dtype=torch.float16))):
        try:
            def step():
                with torch.no_grad():
                    if ctx is None:
                        return O.csnet_forward(cfg, sd, x)
                    with ctx:
                        return O.csnet_forward(cfg, sd, x)
            for _ in range(2):
                step()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"value": B / ms * 1e3, "unit": UNIT, "ms_per_step": ms}
        except Exception as e:                                     # e.g. out of memory at an unusual batch size
            out[name] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    out["what"] = (f"oracle/csnet_oracle.py functional forward (the reference module's own ATen / cuDNN calls) on this GPU, "
                   f"{B} x {S}x{S}, eval, no_grad, device-resident input, {steps} steps after 2 warm-ups")
    return out


def extra_config(a, model_name, size, batch, dev, steps=5):
    """Device-resident img/s of another inference configuration (same kernels, same timing rules), for the `configs` array."""
    import torch

    from sod100k_b200 import checkpoints, ir, roofline, synth

    model, cfg, _ = checkpoints.build_from_npz(model_name)
    model.cuda(dev.index).eval()
    model.set_precision(a.dtype)
    x = torch.from_numpy(synth.randn_images(min(batch, 16), size, size, 1234)).repeat((batch + 15) // 16, 1, 1, 1)[:batch].to(dev)
    with torch.no_grad():
        for _ in range(3):
            model(x)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            model(x)
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    nb = roofline.bytes_per_image(cfg, size, size, ir.DTYPE_BYTES[ir.DTYPE_NAMES[a.dtype]], "block")
    del model
    torch.cuda.empty_cache()
    return {"workload": f"{model_name} inference, {batch} x {size}x{size}, {a.dtype}", "value": batch / ms * 1e3, "unit": UNIT,
            "ms_per_step": ms, "bytes_per_image_block_fused": nb, "achieved_gbs": batch / ms * 1e3 * nb / 1e9}


def train_record(a, world, rank, local, dev, steps=5, warmup=3):
    """fwd + BCE + bwd + [one NCCL all-reduce of the flat gradient bucket] + Adam, images/s over all ranks (max-over-ranks time).
    Every rank runs it (the all-reduce is a collective); rank 0 returns the record."""
    import torch
    import torch.distributed as dist

    from sod100k_b200 import checkpoints, roofline, synth, train_ops
    from sod100k_b200.trainer import Trainer

    model, cfg, _ = checkpoints.build_from_npz(a.model)
    model.cuda(local)
    tr = Trainer(model, lr=1e-4, weight_decay=5e-3, recompute=a.train_recompute)
    B, S = a.train_batch, a.size
    xh = torch.from_numpy(synth.randn_images(B, S, S, 1234 + rank)).pin_memory()
    th = torch.from_numpy(synth.random_masks(B, S, S, 1236 + rank)).pin_memory()
    xd, td = xh.to(dev), th.to(dev)
    stream = torch.cuda.current_stream(dev)

    def timed(fn, k):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(warmup):
        tr.step(xd, td)
    l0 = train_ops.LAUNCHES
    ms = timed(lambda: tr.step(xd, td), steps)
    launches = train_ops.LAUNCHES - l0
    # end to end from pinned host batches: every step copies its inputs (Trainer.step_host: copy stream + two staging slots, so the
    # copy of step k+1 runs under the kernels of step k) and reads one loss back — the PREVIOUS step's, so the host never stalls the queue
    prev = [None]

    def e2e_step():
        loss = tr.step_host(xh, th)
        if prev[0] is not None:
            prev[0].item()
        prev[0] = loss

    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, steps)
    el = roofline.forward_elements(cfg, S, S)
    train_bytes = int(2.51 * el["module"]) * 4                  # 3*sum(I) + 2*sum(O) over modules (SURVEY 8d), fp32 storage
    peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks))["hbm_gbs"]) if os.path.exists(peaks) else 6650.0
    ips, ips_e2e = B * world * steps / (ms * 1e-3), B * world * steps / (ms_e2e * 1e-3)
    bucket_bytes = int(tr.flat.bucket.numel() * 4)
    peak_gib = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    del tr, model
    torch.cuda.empty_cache()
    return {"metric": "images/sec CSNet fwd+BCE+bwd+allreduce+Adam 224x224", "value": ips, "unit": UNIT, "ms_per_step": ms / steps,
            "steps": steps, "warmup": warmup, "per_gpu_batch": B, "global_batch": B * world, "ranks": world, "dtype": "fp32",
            "recompute": bool(a.train_recompute), "peak_memory_GiB": round(peak_gib, 2),
            "collective": "one NCCL all-reduce (sum / world) of the flat fp32 gradient bucket per step" if world > 1 else
                          "none at 1 GPU (the flat gradient bucket is all-reduced when ranks > 1)",
            "allreduce_bytes": bucket_bytes, "gpu_launches": launches,
            "e2e": {"value": ips_e2e, "unit": UNIT, "h2d_bytes_per_step": int((xh.numel() + th.numel()) * 4), "d2h_bytes_per_step": 4},
            "roofline": {"bound": "hbm", "achieved": ips / world * train_bytes / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": ips / world * train_bytes / 1e9 / peak, "bytes_per_image_module_fused_fp32": train_bytes}}


def run_ours(a):
    import torch
    import torch.distributed as dist

    from sod100k_b200 import checkpoints, ir, roofline, runtime, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback of the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    model, cfg, _ = checkpoints.build_from_npz(a.model)
    model.cuda(local).eval()
    model.set_precision(a.dtype)
    eng = model.engine()
    B, S = a.batch, a.size
    base = torch.from_numpy(synth.randn_images(min(B, 32), S, S, 1234 + rank))
    x_host = base.repeat((B + base.shape[0] - 1) // base.shape[0], 1, 1, 1)[:B].contiguous().pin_memory()
    x_dev = x_host.to(dev)
    y_host = torch.empty((B, 1, S, S), dtype=torch.float32).pin_memory()
    plan = eng.plan_for(B, S, S, dev)
    eng.freeze(True)
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    with torch.no_grad():
        last = {}

        def fwd():
            last["logits"] = model(x_dev)

        for _ in range(a.warmup):
            fwd()
        clocks = ClockSampler(local) if rank == 0 else None
        ms = timed(fwd, a.steps)
        clk = clocks.stop() if clocks else None
        outputs = {k: v.cpu().numpy() for k, v in last.items()} if a.dump_outputs and rank == 0 else None
        last.clear()
        # end to end through host buffers (same call a user of the reference-facing API makes)
        e2e_fn = lambda: eng.forward_host(x_host, out=y_host, device=local)
        for _ in range(max(1, a.warmup // 2)):
            e2e_fn()
        ms_e2e = timed(e2e_fn, a.steps)
        # same, with the reference's pre / post-processing on the device (uint8 images in, uint8 maps out: test.py:68-98)
        ms_u8 = None
        if not a.no_extras:
            xu8 = torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8).pin_memory()
            yu8 = torch.empty((B, S, S), dtype=torch.uint8).pin_memory()
            u8_fn = lambda: eng.forward_host_u8(xu8, out=yu8, device=local)
            for _ in range(max(1, a.warmup // 2)):
                u8_fn()
            ms_u8 = timed(u8_fn, a.steps)
        per_op = plan.profile(B, [x_dev.data_ptr(), torch.empty_like(y_host, device=dev).data_ptr()], stream.cuda_stream)
        per_op = [min(u, v) for u, v in zip(per_op, plan.profile(B, [x_dev.data_ptr(), torch.empty_like(y_host, device=dev).data_ptr()], stream.cuda_stream))]

    # train step with the gradient all-reduce: every rank takes part (the one collective of the design)
    train = train_c3 = None
    if not a.no_extras:
        del x_dev
        torch.cuda.empty_cache()
        try:
            train = train_record(a, world, rank, local, dev)
        except Exception as e:
            train = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
        # SURVEY config c3's batch (1024 / GPU) on one GPU: ILBlock-granular recompute, fp32 storage (bf16 storage is not built)
        try:
            import copy
            a3 = copy.copy(a)
            a3.train_batch, a3.train_recompute = 1024, True
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats(dev)
            train_c3 = train_record(a3, world, rank, local, dev, steps=3, warmup=2)
        except Exception as e:
            train_c3 = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    prog = plan.prog
    # dominant KERNEL = the kernel (family) with the largest share of the step; its roofline is aggregated over its launches:
    # (sum of their algorithmic bytes) / (sum of their live CUDA-event durations) == mean bytes per launch / mean launch duration
    kern = [plan.op_kernel(i) for i in range(len(per_op))]
    share = {}
    for k_, t_ in zip(kern, per_op):
        share[k_] = share.get(k_, 0.0) + t_
    dom = max(share, key=share.get)
    dom_ops = [i for i in range(len(per_op)) if kern[i] == dom]
    top = max(dom_ops, key=lambda i: per_op[i])                 # its slowest launch
    dom_bytes = sum(op_bytes(prog, prog.ops[i], B) for i in dom_ops)
    dom_ms = sum(per_op[i] for i in dom_ops)
    top_bytes = op_bytes(prog, prog.ops[top], B)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    dbytes = ir.DTYPE_BYTES[ir.DTYPE_NAMES[a.dtype]]
    net_bytes = roofline.bytes_per_image(cfg, S, S, dbytes, "block")
    ips = B * world * a.steps / (ms * 1e-3)
    ips_e2e = B * world * a.steps / (ms_e2e * 1e-3)
    if a.profile_ops:
        tot = sum(per_op)
        for i in sorted(range(len(per_op)), key=lambda i: -per_op[i])[:25]:
            ob = op_bytes(prog, prog.ops[i], B)
            print(f"{prog.ops[i].name:34s} {per_op[i]:8.3f} ms {100 * per_op[i] / tot:5.1f}%  {ob / per_op[i] / 1e6:8.1f} GB/s",
                  file=sys.stderr)
        print(f"sum of per-op times {tot:.3f} ms vs step {ms / a.steps:.3f} ms", file=sys.stderr)
    # DRAM traffic of the dominant kernel: not measurable without a profiler, so it comes from the committed ncu capture of
    # the same op / batch / size / dtype (profiles/traffic.json, written by scripts/ncu_traffic.sh), or stays null
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        per = [tj.get(f"{a.model}:{prog.ops[i].name}:bs{B}:{S}x{S}:{a.dtype}") for i in dom_ops]
        traffic = sum(per) if all(v is not None for v in per) else None
    out = {
        "metric": METRIC, "value": ips, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": a.dtype, "data": "synthetic", "config": workload_config(a, world), "clocks": clk,
        "e2e": {"value": ips_e2e, "unit": UNIT, "h2d_bytes_per_step": int(x_host.numel() * 4),
                "d2h_bytes_per_step": int(y_host.numel() * 4), "ms_per_step": ms_e2e / a.steps},
        "e2e_u8": None if ms_u8 is None else {
            "value": B * world * a.steps / (ms_u8 * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(B * S * S * 3),
            "d2h_bytes_per_step": int(B * S * S), "ms_per_step": ms_u8 / a.steps,
            "note": "csnet_plan_run_host_u8: uint8 HWC images in, uint8 saliency maps out; normalisation and sigmoid*255 on the device"},
        "gpu_launches": plan.launches * a.steps,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": dom, "kernel_share_of_step": dom_ms / sum(per_op), "kernel_launches_per_step": len(dom_ops),
                     "kernel_ms": dom_ms, "algorithmic_bytes": dom_bytes,
                     "note": "achieved = sum of the kernel's algorithmic bytes over its launches in one step / sum of their CUDA-event times; "
                             "traffic = ncu dram bytes of the same launches (profiles/traffic.json)",
                     "slowest_launch": {"op": prog.ops[top].name, "ms": per_op[top], "algorithmic_bytes": top_bytes,
                                        "achieved": top_bytes / (per_op[top] * 1e-3) / 1e9, "frac": top_bytes / (per_op[top] * 1e-3) / 1e9 / peak},
                     "by_kernel": {k_: {"ms": v_, "share": v_ / sum(per_op)} for k_, v_ in sorted(share.items(), key=lambda kv: -kv[1])},
                     "peak_source": peak_src,
                     "net": {"bytes_per_image_block_fused": net_bytes,
                             "achieved": ips / world * net_bytes / 1e9, "frac": ips / world * net_bytes / 1e9 / peak}},
    }
    if not a.no_extras:
        out["train"] = train
        out["train_c3_batch"] = train_c3
        del plan, eng, model
        torch.cuda.empty_cache()
        out["gpu_eager_baseline"] = gpu_eager_baseline(a, dev)
        out["configs"] = []
        for mname, size, batch in ((a.model, 512, 64), ("csnet-L-x1" if a.model != "csnet-L-x1" else "csnet-L-x2", a.size, a.batch)):
            try:
                out["configs"].append(extra_config(a, mname, size, batch, dev))
            except Exception as e:
                out["configs"].append({"workload": f"{mname} {batch} x {size}x{size}", "unavailable": f"{type(e).__name__}: {e}"[:200]})
        try:                                                      # the 1e-3 parity path (fp32 activations, generic kernels), for the record
            a32 = argparse.Namespace(**vars(a))
            a32.dtype = "fp32"
            c32 = extra_config(a32, a.model, a.size, 64, dev, steps=3)
            c32["note"] = "fp32 storage: the configuration that meets the 1e-3 sigmoid gate (generic kernels)"
            out["configs"].append(c32)
        except Exception as e:
            out["configs"].append({"workload": f"{a.model} fp32 64 x {a.size}x{a.size}", "unavailable": f"{type(e).__name__}: {e}"[:200]})
        for c in out["configs"]:
            if "achieved_gbs" in c:
                c["roofline_net_frac"] = c["achieved_gbs"] / peak
    if not a.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(a)
    if outputs is not None:
        dump_outputs(a.dump_outputs, outputs)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_train(a):
    """Train step throughput (configs 3-4 shape, fp32 activations for now): images/s of forward + BCE + backward +
    [DP: one flat-bucket all-reduce] + fused Adam, inputs resident in HBM; e2e adds the pinned H2D of images + masks
    and the D2H of the loss."""
    import torch
    import torch.distributed as dist

    from sod100k_b200 import checkpoints, roofline, synth
    from sod100k_b200.trainer import Trainer

    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model, cfg, _ = checkpoints.build_from_npz(a.model)
    model.cuda(local)
    tr = Trainer(model, lr=1e-4, weight_decay=5e-3)
    B, S = a.batch, a.size
    xh = torch.from_numpy(synth.randn_images(B, S, S, 1234 + rank)).pin_memory()
    th = torch.from_numpy(synth.random_masks(B, S, S, 1236 + rank)).pin_memory()
    xd, td = xh.to(dev), th.to(dev)
    stream = torch.cuda.current_stream(dev)

    def timed(fn, k):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    step = lambda: tr.step(xd, td)
    e2e = lambda: tr.step(xh.to(dev, non_blocking=True), th.to(dev, non_blocking=True)).item()
    for _ in range(a.warmup):
        step()
    clocks = ClockSampler(local) if rank == 0 else None
    from sod100k_b200 import train_ops
    launches0 = train_ops.LAUNCHES
    ms = timed(step, a.steps)
    train_launches = train_ops.LAUNCHES - launches0          # csnet_train_* kernels of the timed steps (memsets not counted)
    clk = clocks.stop() if clocks else None
    e2e()
    ms_e2e = timed(e2e, a.steps)
    if rank == 0:
        peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak = float(json.load(open(peaks))["hbm_gbs"]) if os.path.exists(peaks) else 6650.0
        el = roofline.forward_elements(cfg, S, S)
        ips, ips_e2e = B * world * a.steps / (ms * 1e-3), B * world * a.steps / (ms_e2e * 1e-3)
        train_bytes = int(2.51 * el["module"]) * 4          # 3*sum(I) + 2*sum(O) over modules (SURVEY 8d), fp32
        print(json.dumps({
            "metric": "images/sec CSNet fwd+bwd+Adam 224x224", "value": ips, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic",
            "config": {"workload": f"{a.model} train step, {B} img/GPU x {S}x{S}, fp32 module-granular kernels",
                       "global_batch": B * world, "parallelism": f"dp{world}: local BN, one flat-bucket all-reduce of "
                       f"{tr.flat.bucket.numel()} fp32 gradients", "l2": "activations exceed L2"},
            "clocks": clk,
            "e2e": {"value": ips_e2e, "unit": UNIT, "h2d_bytes_per_step": int((xh.numel() + th.numel()) * 4), "d2h_bytes_per_step": 4},
            "gpu_launches": train_launches,
            "roofline": {"bound": "hbm", "achieved": ips / world * train_bytes / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": ips / world * train_bytes / 1e9 / peak, "traffic": None,
                         "kernel": "whole train step (module-fused algorithmic bytes, fp32)"}}))
    if world > 1:
        dist.destroy_process_group()


def run_csf(a):
    """Config 5: CSF+Res2Net-50, bs 64, 352x352, fp16, seeded synthetic weights (the reference ships none).  The line splits
    the step into the cuDNN backbone (library) and the CSF head (our kernels): only the head is the product."""
    import torch

    from sod100k_b200 import synth
    from sod100k_b200.networks import csf_res2net

    torch.cuda.set_device(0)
    m = csf_res2net.build_model()
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.synth_state_r(shapes, 21).items()})
    m.cuda().eval().set_precision(a.dtype)
    B, S = (64 if a.batch == 256 else a.batch), (352 if a.size == 224 else a.size)
    x = torch.from_numpy(synth.randn_images(min(B, 8), S, S, 1234)).repeat((B + 7) // 8, 1, 1, 1)[:B].cuda()

    def timed(fn, k):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    with torch.no_grad():
        for _ in range(a.warmup):
            m(x)
        clocks = ClockSampler(0)
        ms = timed(lambda: m(x), a.steps)
        clk = clocks.stop()
        ms_backbone = timed(lambda: m.backbone(x), a.steps)
    ips = B * a.steps / (ms * 1e-3)
    head_ms = (ms - ms_backbone) / a.steps
    peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
    tf = float(json.load(open(peaks))["bf16_tflops"]) if os.path.exists(peaks) else 1590.0
    head_flops = 2 * 8.11e9 * (S / 352.0) ** 2 * B               # SURVEY: 8.11 GMAC per 352x352 image in the head
    print(json.dumps({
        "metric": "images/sec CSF+Res2Net50 fwd 352x352", "value": ips, "unit": UNIT, "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": a.dtype, "data": "synthetic",
        "config": {"workload": f"CSF+Res2Net-50 inference, {B} x {S}x{S}, {a.dtype}; backbone = torch/cuDNN (library), CSF head = engine",
                   "backbone_ms": ms_backbone / a.steps, "head_ms": head_ms, "weights": "seeded synthetic (no checkpoint ships)"},
        "clocks": clk, "gpu_launches": None,
        "roofline": {"bound": "tensor", "achieved": head_flops / (head_ms * 1e-3) / 1e12, "peak": tf, "unit": "TFLOP/s",
                     "frac": head_flops / (head_ms * 1e-3) / 1e12 / tf, "traffic": None, "kernel": "CSF head (all engine kernels)"}}))


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank)
    elif a.mode == "csf":
        run_csf(a)
    elif a.mode == "train":
        if a.batch == 256:
            a.batch = 32
        run_train(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
