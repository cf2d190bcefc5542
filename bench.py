#!/usr/bin/env python
"""bench.py — BASELINE.json's metric: ResNet-50 synthetic-image throughput (images/s) of a
data-parallel TorchJob at N worker-replica GPUs, with the allreduce's achieved bus bandwidth against
the NVLink roofline, next to the reference-style gloo/CPU torchjob on the box's host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|nccl]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
      --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one synthetic batch: forward + backward of ResNet-50
(bf16 parameters/gradients, channels_last, per-GPU batch 256, DDP bucket cap 25 MB -> 3 buckets of
4.1/28.9/18.1 MB) whose gradient buckets are averaged across replicas by libtok8s' fused
cast/scale/allreduce kernels (through torch_on_k8s_b200's DDP comm hook), + SGD step.
Timing: CUDA events, barrier + synchronize on both sides, MAX over ranks; rank 0 prints ONE JSON
line.  `value` has inputs resident in HBM; `e2e` copies every step's batch from pinned host memory
and reads the loss back.  The step's working set (GBs of activations) is far larger than the
126 MB L2, so no explicit L2 flush is needed between iterations (stated in config.l2).
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "resnet50_ddp_images_per_sec"
UNIT = "images/s"
NVLINK_PEAK_GBS = 900.0  # nominal per direction per GPU (BASELINE.md §2 fixes this denominator)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:  # noqa: BLE001
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None,
                "samples": len(sm), "reasons": sorted(reasons)}


RESNET50_BF16_BYTES_PER_STEP = 51114064   # 25,557,032 bf16 gradients (SURVEY.md §8a)


def workload_config(batch: int, world: int) -> dict:
    """`config` of BOTH arms: the workload BASELINE.json's metric is quoted on (configs[1])."""
    return {"workload": "ResNet-50 bf16 synthetic 224x224 images (random-init weights), per-replica "
                        "batch %d, DDP bucket 25MB (4.1/28.9/18.1 MB at iteration 0, rebuilt by DDP "
                        "into 28.3/22.9 MB; 51.1 MB of gradient/step/replica), SGD momentum 0.9, "
                        "channels_last; 1 master + %d workers" % (batch, world - 1),
            "global_batch": batch * world, "parallelism": "dp%d" % world,
            "l2": "step working set (GBs of activations) is larger than the 126 MB L2; no explicit "
                  "flush",
            "allreduce_bytes_per_step": RESNET50_BF16_BYTES_PER_STEP}


# --------------------------------------------------------------------------------------------------
# reference arm: the reference-style gloo/CPU torchjob (oracle/gloo_torchjob.py), timed on the host
# --------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0  # rank 0 alone runs the CPU job; other torchrun ranks exit without work
    from oracle import gloo_torchjob
    n = args.gpus
    cores = gloo_torchjob.effective_cores()
    batch = args.ref_batch
    t0 = time.time()
    # replicas get a container-clean environment (SetClusterSpec variables only): nothing of the
    # launcher that started THIS process (torchrun's agent-store variables, OMP_NUM_THREADS=1) leaks in
    res = gloo_torchjob.run("resnet50", world=n, steps=args.steps, warmup=args.warmup, batch=batch,
                            dtype="bf16", job="bench-ref")
    value = res["images_per_sec"]
    sample = ("each step is a bounded sample of the workload: per-replica batch %d instead of %d "
              "(images/s is per image, the allreduce bytes per step do not depend on the batch); "
              "%d timed + %d warm-up steps, bf16, torchvision resnet50, stock DDP + gloo over "
              "loopback wired per SetClusterSpec, %d replicas x %d threads on %d host cores" %
              (batch, args.batch, args.steps, args.warmup, n, res["threads_per_replica"], cores))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": res["seconds"] / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args.batch, n),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "sample_batch_per_replica": batch, "wall_s": time.time() - t0,
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------------------------------
# our arm (and --impl nccl: the same job with stock DDP + NCCL, for the comparison SURVEY §2.1 names)
# --------------------------------------------------------------------------------------------------
def ints_pattern(n, rank, device):
    """Bucket of replica `rank` with values k/4, |k| <= 8: every partial sum of up to 8 replicas, and
    its product with 1/2, 1/4 or 1/8, is exactly representable in bf16 — any summation order (the
    NVSwitch's included) must produce the same bits."""
    import torch
    i = torch.arange(n, device=device, dtype=torch.int64)
    k = ((i * 1103515245 + (rank + 1) * 12345) >> 8) % 17 - 8
    return k.to(torch.float32) * 0.25


def parity_check(rep, sizes, world, zero_copy, stream):
    """Before anything is timed: the real DDP bucket sizes through the SAME path the hook uses
    (pool buckets, arrival + AUTO exchange, scale 1/N) on exactly representable data; the result
    must equal the closed-form sum bit for bit on every replica."""
    import torch
    import torch.distributed as dist
    dev = rep.device
    ok, algos = True, []
    pow2 = world & (world - 1) == 0
    scale = 1.0 / world if pow2 else 1.0
    for sz in sizes:
        n = sz // 2
        t = rep.comm.symm_empty(n, torch.bfloat16) if zero_copy else \
            torch.empty(n, device=dev, dtype=torch.bfloat16)
        with torch.cuda.stream(stream):
            t.copy_(ints_pattern(n, rep.rank, dev))
            arrived = rep.comm.bucket_arrive(t, scale=scale, stream=stream) if world > 1 else False
            rep.comm.allreduce_bucket(t, t, scale=scale, arrived=arrived, elide=False, stream=stream)
            want = sum(ints_pattern(n, r, dev) for r in range(world)) * scale
            good = torch.equal(t, want.to(torch.bfloat16))
            stream.synchronize()
        rep.comm.status()
        algos.append(rep.comm.last_algo())
        ok = ok and bool(good)
        del t, want
    flag = torch.tensor([1 if ok else 0], device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {"exact": bool(flag.item()), "algo": sorted(set(algos)), "bucket_bytes": list(sizes),
            "scale": scale, "zero_copy": bool(zero_copy),
            "pattern": "k/4, |k|<=8 per replica; expected = closed-form sum * scale, compared "
                       "bit for bit on every replica before timing"}


DUMP_SAMPLE = 1 << 22   # elements kept of each flattened array: 16 MiB per file as float32


def dump_outputs(out_dir, model, loss):
    """What the caller of the last timed step holds afterwards, as float32 .npy files: its loss, the
    averaged gradients (the bucket exchange's output) and the updated parameters.  The two flattened
    arrays of 25.6 M elements are cut to the same fixed, seeded sample of DUMP_SAMPLE elements."""
    import numpy as np
    import torch
    params = list(model.parameters())
    flat = {"grads": torch.cat([p.grad.detach().flatten().float() for p in params]),
            "params": torch.cat([p.detach().flatten().float() for p in params])}
    n = flat["params"].numel()
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float32))
    for name, t in flat.items():
        np.save(os.path.join(out_dir, name + ".npy"), t[idx.to(t.device)].cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback "
                         "(use --impl reference for the gloo/CPU torchjob)")
    from torch_on_k8s_b200.netutil import free_port
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            # convenience: re-launch ourselves under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                   "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
                   "--master-port", str(free_port()), os.path.abspath(__file__)] + sys.argv[1:]
            return subprocess.call(cmd)
        raise SystemExit("bench.py: --gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if "MASTER_PORT" not in os.environ:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(free_port())
    os.environ.setdefault("TOK8S_JOB", "bench-resnet50")

    from torch_on_k8s_b200.worker import init_replica
    from workloads.resnet50 import resnet50

    rep = init_replica(device=local)
    dev = rep.device
    # Dumped outputs are compared between runs and builds, so a dumping run takes cuDNN's
    # deterministic algorithms instead of each run's fastest: tens of bf16 training steps amplify
    # one step's last-bit differences until the weights no longer agree.
    torch.backends.cudnn.benchmark = not args.dump_outputs
    torch.backends.cudnn.deterministic = bool(args.dump_outputs)
    B = args.batch
    nccl_only = args.impl == "nccl"

    def make_job(stock_nccl):
        torch.manual_seed(0)
        model = resnet50().to(dev).to(torch.bfloat16).to(memory_format=torch.channels_last)
        if stock_nccl:   # stock PyTorch: DDP's own reducer + ProcessGroupNCCL allreduce
            from torch.nn.parallel import DistributedDataParallel as DDP
            ddp, hook = DDP(model, device_ids=[dev.index], bucket_cap_mb=25,
                            gradient_as_bucket_view=True), None
        else:
            # world 1: the bucket exchange degenerates to the fused scale/cast with scale 1 on an
            # in-place bucket — an identity the library elides by default.  The bench keeps the launch
            # (TOK_FLAG_NO_ELIDE) so that the hot-path kernel is exercised and measured in-step at
            # N=1 too, as the reference's own hook does (div_(1) + allreduce).
            ddp, hook = rep.wrap(model, bucket_cap_mb=25, record_events=True,
                                 elide_identity=(world > 1))
        opt = torch.optim.SGD(ddp.parameters(), lr=0.01, momentum=0.9)
        return ddp, hook, opt

    lossf = torch.nn.CrossEntropyLoss()
    gen = torch.Generator().manual_seed(1234 + rank)
    n_host = 4  # rotating pinned host batches for the e2e leg
    host_x = [torch.randn(B, 3, 224, 224, generator=gen).to(torch.bfloat16)
              .contiguous(memory_format=torch.channels_last).pin_memory() for _ in range(n_host)]
    host_y = [torch.randint(0, 1000, (B,), generator=gen).pin_memory() for _ in range(n_host)]
    dev_x = host_x[0].to(dev, non_blocking=True)
    dev_y = host_y[0].to(dev, non_blocking=True)

    def make_step(ddp, opt):
        def step(x, y):
            opt.zero_grad(set_to_none=True)
            loss = lossf(ddp(x).float(), y)
            loss.backward()
            opt.step()
            return loss
        return step

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        barrier()
        return float(t.item())

    W = max(args.warmup, 3)
    h2d = host_x[0].numel() * host_x[0].element_size() + host_y[0].numel() * host_y[0].element_size()

    def measure(step):
        """(device-resident ms, e2e ms) over args.steps steps each."""
        ms_dev = timed(lambda i: step(dev_x, dev_y), args.steps)

        def e2e_step(i):
            x = host_x[i % n_host].to(dev, non_blocking=True)
            y = host_y[i % n_host].to(dev, non_blocking=True)
            loss = step(x, y)
            return float(loss.detach().float().item())  # device->host read of the step's result
        for i in range(2):
            e2e_step(i)
        return ms_dev, timed(e2e_step, args.steps)

    def nccl_arm():
        """The same job with stock DDP + NCCL, and the step's buckets through ncclAllReduce back to
        back on an idle GPU (same sizes, same rotation over > L2 as roofline_isolated)."""
        ddp2, _, opt2 = make_job(True)
        step2 = make_step(ddp2, opt2)
        for _ in range(W):
            step2(dev_x, dev_y)
        ms_dev2, ms_e2e2 = measure(step2)
        out = {"value": args.steps * B * world / (ms_dev2 * 1e-3), "unit": UNIT,
               "ms_per_step": ms_dev2 / args.steps,
               "e2e": {"value": args.steps * B * world / (ms_e2e2 * 1e-3), "unit": UNIT,
                       "ms_per_step": ms_e2e2 / args.steps},
               "what": "stock torch DistributedDataParallel + ProcessGroupNCCL (NCCL %s), same model, "
                       "batch, bucket cap, optimizer, steps, in the same process right after our arm"
                       % ".".join(str(v) for v in torch.cuda.nccl.version())}
        del ddp2, opt2, step2
        return out

    if nccl_only:
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        res = nccl_arm()
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            line = {"impl": "nccl", "metric": METRIC, "value": res["value"], "unit": UNIT,
                    "n_gpus": world, "steps": args.steps, "warmup": W,
                    "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                    "config": workload_config(B, world), "clocks": clocks,
                    "e2e": dict(res["e2e"], h2d_bytes_per_step=h2d * world, d2h_bytes_per_step=4 * world),
                    "gpu_launches": 0, "what": res["what"]}
            print(json.dumps(line), flush=True)
        rep.close()
        return 0

    ddp, hook, opt = make_job(False)
    step = make_step(ddp, opt)

    # ---- warm-up (also lets DDP rebuild its buckets after iteration 1) ---------------------------
    for _ in range(W):
        step(dev_x, dev_y)
    barrier()
    warm_ev = hook.drain_events()
    rep.comm.status()
    zero_copy = hook.zero_copy_buckets > 0 and world > 1   # DDP's buckets sit in the symmetric pool
    sizes = list(hook.last_step_bytes) or [e[0] for e in warm_ev[-2:]]   # the rebuilt buckets

    # ---- parity first: the timed kernels on this box, on these bucket sizes ------------------------
    cstream = torch.cuda.Stream(device=dev)
    parity = parity_check(rep, sizes, world, zero_copy, cstream)
    barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = rep.comm.launches()
    ms_dev = timed(lambda i: step(dev_x, dev_y), args.steps)
    launches = rep.comm.launches() - launches0
    ev = hook.drain_events()

    # ---- end-to-end leg: host batch -> device every step, loss read back every step --------------
    def e2e_step(i):
        x = host_x[i % n_host].to(dev, non_blocking=True)
        y = host_y[i % n_host].to(dev, non_blocking=True)
        loss = step(x, y)
        return float(loss.detach().float().item())  # device->host read of the step's result

    for i in range(2):
        e2e_step(i)
    last = {}
    ms_e2e = timed(lambda i: last.__setitem__("loss", e2e_step(i)), args.steps)
    clocks = sampler.stop() if rank == 0 else None
    hook.drain_events()
    rep.comm.status()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ddp, last["loss"])

    # ---- roofline of the dominant kernel of OUR path (the bucket exchange) -----------------------
    # CUDA events on the comm stream around the exchange kernel alone; the 1-warp arrival in front of
    # it (the wait for the slowest replica's backward) is timed separately as arrival_wait_us.
    peaks, peak_kind = measured_peaks()
    wire_bytes = sum(e[0] for e in ev)
    bucket_bytes = sum(e[1] for e in ev)
    ar_ms = sum(e[2] for e in ev)
    wait_ms = sum(e[3] for e in ev)
    n_launch = max(len(ev), 1)
    stats = torch.tensor([wire_bytes, ar_ms, wait_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ar_ms_max = float(stats[1].item())
    wait_ms_max = float(stats[2].item())
    kernel_name = rep.comm.last_algo()
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tr = json.load(f).get(kernel_name, {})
        per = [tr.get(str(sz)) for sz in sizes]
        if per and all(v is not None for v in per):
            traffic = sum(per) / len(per)
    except Exception:  # noqa: BLE001
        traffic = None
    if world == 1:
        # fused scale/cast only: S_in + S_out against HBM
        achieved = (2.0 * bucket_bytes) / (ar_ms_max * 1e-3) / 1e9 if ar_ms_max > 0 else 0.0
        roof = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                "kernel": "tok::%s_kernel<bf16>" % kernel_name,
                "algorithmic_bytes_per_launch": 2.0 * bucket_bytes / n_launch,
                "avg_launch_us": ar_ms_max * 1e3 / n_launch, "peak_source": peak_kind + " hbm_gbs",
                "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu "
                                  "--set full at these bucket sizes (profiles/traffic.json)",
                "note": "world=1 degenerates to the fused scale/cast: bytes = S_in + S_out; one "
                        "launch between two CUDA events, launch latency included.  traffic is about "
                        "S_in alone: the in-place result stays in the 126 MB L2 (written back after "
                        "the kernel), and the kernel is latency-bound at this size (ncu: DRAM at "
                        "~30 % of peak for ~10 us) — ATen's own mul_ takes the same 12.3 us "
                        "back to back on the 28 MB bucket (profiles/r02_local_bench_n1.json)"}
    else:
        algbw = wire_bytes / (ar_ms_max * 1e-3) / 1e9 if ar_ms_max > 0 else 0.0
        busbw = algbw * 2.0 * (world - 1) / world
        roof = {"bound": "nvlink", "achieved": busbw, "peak": NVLINK_PEAK_GBS, "unit": "GB/s",
                "frac": busbw / NVLINK_PEAK_GBS, "traffic": traffic,
                "kernel": "tok::%s_kernel<bf16>" % kernel_name,
                "algbw_gbs": algbw, "algorithmic_bytes_per_launch": wire_bytes / n_launch,
                "avg_launch_us": ar_ms_max * 1e3 / n_launch,
                "arrival_wait_us": wait_ms_max * 1e3 / n_launch,
                "peak_source": "nominal NVLink5 900 GB/s per direction (BASELINE.md §2); measured "
                               "peer copy on this pool is 770 GB/s",
                "traffic_note": "ncu cannot replay a kernel that waits for peer replicas' kernels, so "
                                "there is no dram__bytes capture for the cross-GPU kernels; the "
                                "zero-copy exchange makes no staging pass by construction (reads of "
                                "the bucket by the switch / peers + one write of the result)",
                "note": "busbw = S/t * 2(N-1)/N over the exchange kernels inside the timed steps, "
                        "concurrent with backward; the wait for the slowest replica is the 1-warp "
                        "arrival kernel in front (arrival_wait_us), not part of t; NVLS may exceed 1.0"}

    # ---- the same buckets, exchanged back to back with nothing else on the GPU (kernel quality
    #      without backward competing for HBM/SMs); buffers rotate over > L2 bytes -------------------
    iso = nccl_iso = None
    if sizes:
        el = torch.empty(0, dtype=torch.bfloat16).element_size()
        nsets = max(2, int((160 << 20) / max(sum(sizes), 1)) + 1)

        def mk(sz, pool):
            t = rep.comm.symm_empty(sz // el, torch.bfloat16) if pool else \
                torch.empty(sz // el, device=dev, dtype=torch.bfloat16)
            return t.normal_()
        sets = [[mk(sz, zero_copy) for sz in sizes] for _ in range(min(nsets, 8))]

        def iso_ours(i):
            for t in sets[i % len(sets)]:
                rep.comm.allreduce_bucket(t, t, scale=0.5 if world == 1 else 1.0 / world,
                                          stream=cstream)

        def iso_nccl(i):
            for t in sets[i % len(sets)]:
                dist.all_reduce(t)

        def iso_time(fn, iters=30):
            with torch.cuda.stream(cstream):
                for i in range(5):
                    fn(i)
                cstream.synchronize()
                barrier()
                i0 = torch.cuda.Event(enable_timing=True)
                i1 = torch.cuda.Event(enable_timing=True)
                i0.record(cstream)
                for i in range(iters):
                    fn(i)
                i1.record(cstream)
                cstream.synchronize()
            tt = torch.tensor([i0.elapsed_time(i1)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()), iters

        iso_ms, iters = iso_time(iso_ours)
        rep.comm.status()
        iso_bytes = float(sum(sizes) * iters)
        if world == 1:
            ach = 2.0 * iso_bytes / (iso_ms * 1e-3) / 1e9
            iso = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                   "frac": ach / peaks["hbm_gbs"], "avg_launch_us": iso_ms * 1e3 / (iters * len(sizes))}
        else:
            ach = iso_bytes / (iso_ms * 1e-3) / 1e9 * 2.0 * (world - 1) / world
            iso = {"bound": "nvlink", "achieved": ach, "peak": NVLINK_PEAK_GBS, "unit": "GB/s",
                   "frac": ach / NVLINK_PEAK_GBS, "avg_launch_us": iso_ms * 1e3 / (iters * len(sizes)),
                   "launches_per_bucket": 2 if zero_copy else 1}
            n_ms, n_iters = iso_time(iso_nccl)
            n_ach = float(sum(sizes) * n_iters) / (n_ms * 1e-3) / 1e9 * 2.0 * (world - 1) / world
            nccl_iso = {"achieved": n_ach, "unit": "GB/s", "frac": n_ach / NVLINK_PEAK_GBS,
                        "avg_launch_us": n_ms * 1e3 / (n_iters * len(sizes))}
        iso["bucket_bytes"] = sizes
        iso["kernel"] = rep.comm.last_algo()
        iso["zero_copy"] = bool(zero_copy)
        iso["note"] = ("the step's buckets exchanged back to back on an otherwise idle GPU (arrival "
                       "kernels included), inputs rotated over >126 MB so they are not L2 resident")
        del sets

    # ---- stock DDP + NCCL on the same box, same process, right after (N > 1) -----------------------
    nccl = None
    if world > 1 and not args.no_nccl:
        del ddp, opt, step
        torch.cuda.empty_cache()
        nccl = nccl_arm()
        nccl["isolated_buckets"] = nccl_iso

    if rank != 0:
        rep.close()
        return 0

    images = args.steps * B * world
    value = images / (ms_dev * 1e-3)
    e2e_value = images / (ms_e2e * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": W, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(B, world),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world,
                "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches * world),
        "zero_copy_buckets": bool(zero_copy),
        "parity_check": parity,
        "roofline": roof,
        "roofline_isolated": iso,
    }
    if world == 1:
        line["world1_note"] = ("at world 1 the per-bucket exchange is the fused scale/cast with scale "
                               "1 on an in-place bucket: an identity libtok8s elides by default (no "
                               "launch, no HBM pass).  This run passes TOK_FLAG_NO_ELIDE so that the "
                               "hot-path kernel runs and is measured in-step (gpu_launches counts "
                               "those launches), as the reference's own hook does (div_(1) + "
                               "allreduce)")
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs,
                                "cudnn": "deterministic algorithms, benchmark mode off"}
    if nccl is not None:
        line["nccl"] = nccl
        line["vs_nccl"] = {"step": value / nccl["value"], "e2e": e2e_value / nccl["e2e"]["value"],
                           "isolated_buckets": (nccl_iso["avg_launch_us"] / iso["avg_launch_us"])
                           if (nccl_iso and iso) else None}
    if world == 1 and not args.no_cpu_baseline:
        # bounded sample of the same workload on the host cores: the reference-style gloo job
        from oracle import gloo_torchjob
        cb = gloo_torchjob.run("resnet50", world=1, steps=args.cpu_steps, warmup=1,
                               batch=args.ref_batch, dtype="bf16", job="bench-cpu")
        line["cpu_baseline"] = {
            "value": cb["images_per_sec"], "unit": UNIT, "cores": cb["cores"], "kind": "reference",
            "sample": "%d timed steps (+1 warm-up) of the same ResNet-50 bf16 step at batch %d on "
                      "the host CPU: torchvision model, torch DDP + gloo configured per "
                      "SetClusterSpec, %d threads" %
                      (args.cpu_steps, args.ref_batch, cb["threads_per_replica"])}
    print(json.dumps(line), flush=True)
    rep.close()
    return 0 if parity["exact"] else 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl"])
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch (BASELINE config: 256)")
    ap.add_argument("--ref-batch", type=int, default=32,
                    help="per-replica batch of the CPU arm (bounded sample of the same workload; "
                         "BASELINE.md §3)")
    ap.add_argument("--no-nccl", action="store_true", help="skip the stock DDP+NCCL comparison leg")
    ap.add_argument("--cpu-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as "
                         "DIR/<name>.npy (the run uses cuDNN's deterministic algorithms)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
