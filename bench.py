#!/usr/bin/env python
"""bench.py — distillation hot-path throughput (BASELINE.json metric "distill samples/s"; workload = configs[1]).

One STEP = one pass of the hot path over one synthetic batch per GPU:
    student 5-cell BiFPN stack forward (train-mode BatchNorm) from C3/C4/C5  [B,48,96,96] [B,120,48,48] [B,352,24,24]
  + 3 frozen teacher stacks forward (eval, no_grad)
  + 3 MTA losses (one call per teacher, as the shipped cfg does)  -> loss = 0.005 * sum
  + backward through MTA and the student stack (all BiFPN parameter gradients + dL/dC3..C5)
  + (N > 1) one NCCL all-reduce of the flat student gradient buffer.

    python bench.py [--gpus N --steps K --warmup W] [--dtype f32|bf16] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line (rank 0).  `--impl reference` times the CPU port of the reference algorithm (oracle/) on the
host cores for the same metric; it is the only place besides cpu_baseline where bench.py executes oracle/.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

CC = [48, 120, 352]
C = 112
N_CELLS = 5
N_TEACHERS = 3
W_KD = 0.005
S3 = 96           # P3 resolution of a 768x768 input
POS_PER_SAMPLE = 96 * 96 + 48 * 48 + 24 * 24 + 12 * 12 + 6 * 6


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def synth_inputs(B, gen, dtype=torch.float32):
    return [torch.randn(B, c, S3 >> i, S3 >> i, generator=gen).to(dtype) for i, c in enumerate(CC)]


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (torch CPU fp32 restatement of the reference path), all host threads
# ------------------------------------------------------------------------------------------------------------------
def cpu_state(seed):
    from oracle import mmd_oracle as O
    return O.synth_stack_params(C, CC, N_CELLS, seed)


def cpu_step(student_p, teacher_ps, xs_s, xs_ts):
    from oracle import mmd_oracle as O
    leaf = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v)
            for k, v in student_p.items()}
    xs = [x.detach().clone().requires_grad_(True) for x in xs_s]
    fs = O.bifpn_stack(tuple(xs), leaf, N_CELLS, training=True, stats_out={})
    kd = []
    for tp, xt in zip(teacher_ps, xs_ts):
        with torch.no_grad():
            ft = O.bifpn_stack(tuple(xt), tp, N_CELLS, training=False)
        kd.append(O.mta_loss(fs, [f.detach() for f in ft]))
    kd = torch.stack(kd)
    (W_KD * kd.sum()).backward()
    # optimizer.step() (src/optimization/traditional.py:190) with the shipped recipe's Adam (train_methods.py:825-833)
    torch.optim.Adam([v for v in leaf.values() if v.requires_grad], lr=1e-4, betas=(0.9, 0.999)).step()
    return kd.detach()


def time_cpu(B, steps, warmup):
    torch.set_num_threads(os.cpu_count() or 1)
    gen = torch.Generator().manual_seed(0)
    sp = cpu_state(0)
    tps = [cpu_state(1 + k) for k in range(N_TEACHERS)]
    xs_s = synth_inputs(B, gen)
    xs_ts = [synth_inputs(B, gen) for _ in range(N_TEACHERS)]
    for _ in range(warmup):
        cpu_step(sp, tps, xs_s, xs_ts)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        cpu_step(sp, tps, xs_s, xs_ts)
        ts.append(time.perf_counter() - t0)
    return ts


def run_reference(args, rank):
    """The reference arm: the CPU port of the reference's own implementation of the path (oracle/, pinned against outputs
    of the unmodified reference) on all host threads, SAME step and SAME batch as the CUDA arm.  If K + W steps at that
    batch would not end within a few minutes on this host, the per-step sample is halved until they do (and the line
    says so: config.batch_per_step / config.same_batch_as_cuda_arm)."""
    if rank != 0:
        return
    B = args.batch
    budget_s = 240.0
    t_probe = None
    while True:
        t_probe = sum(time_cpu(B, 1, 0))          # one untimed probe step (also warms the allocator / thread pool)
        if t_probe * (args.steps + args.warmup) <= budget_s or B <= 2:
            break
        B //= 2
    ts = time_cpu(B, args.steps, max(args.warmup - 1, 0))
    total = sum(ts)
    v = B * len(ts) / total
    cores = torch.get_num_threads()
    sample = ("each step = the full hot-path step at batch %d (student fwd+bwd, 3 teacher fwd, 3 MTA calls), oracle port, "
              "torch CPU fp32, %d threads" % (B, cores))
    line = {
        "impl": "reference", "metric": "distill samples/s", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(ts), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_step": B, "batch_per_gpu": B, "cuda_arm_batch_per_gpu": args.batch,
                   "same_batch_as_cuda_arm": B == args.batch},
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


WORKLOAD = ("hot path of cfg3/cfg4 (3-teacher -> student distillation step, batch 32 per GPU, bf16) on the cfg2 microbench "
            "inputs: MTA loss + 5-cell EfficientDet-D2 BiFPN on synthetic pyramid features (C3 48@96^2, C4 120@48^2, "
            "C5 352@24^2 -> 112 ch P3-P7): student fwd+bwd (train BN) + 3 teacher fwd (eval) + 3 MTA calls "
            "[+ flat-gradient NCCL all-reduce for N > 1] + Adam update of the student's parameters; the cfg2 batch (16) is measured in the same run (cfg2_b16)")


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  NVML is read in-process from a background thread
    (a polling `nvidia-smi -lms 100` child was measured to slow this launch-bound step 3-4x through driver contention);
    falls back to one nvidia-smi query per second when pynvml is unavailable."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index, period_s=0.02):
        import threading
        self.sm, self.smax, self.reasons, self.src = [], None, set(), None
        self._stop = threading.Event()
        self._thr = None
        self.p = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {
                "hw_slowdown": pynvml.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": pynvml.nvmlClocksThrottleReasonSwPowerCap,
            }

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for n, b in bits.items():
                            if r & b:
                                self.reasons.add(n)
                    except Exception:
                        pass
                    self._stop.wait(period_s)

            self._thr = threading.Thread(target=loop, daemon=True)
            self._thr.start()
            self.src = "nvml"
        except Exception:
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            try:
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + q,
                                           "--format=csv,noheader,nounits", "-lms", "1000"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.src = "nvidia-smi"
            except OSError:
                self.p = None

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join(timeout=2)
        elif self.p is not None:
            time.sleep(0.15)
            self.p.terminate()
            try:
                out, _ = self.p.communicate(timeout=5)
            except subprocess.TimeoutExpired:
                self.p.kill()
                out, _ = self.p.communicate()
            for ln in out.strip().splitlines():
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    self.sm.append(float(f[1]))
                    self.smax = float(f[2])
                except ValueError:
                    continue
                for n, v in zip(self.NAMES, f[5:9]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock source available"]}
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.smax,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.src}


def algo_bytes_per_step(B, esize, n_teachers=N_TEACHERS):
    """Algorithmic HBM bytes of one step (SURVEY.md 8d): student forward + backward = 3 x forward bytes, each teacher
    forward = 1 x, MTA forward reads every student and teacher map once, MTA backward re-reads the student maps and
    writes their gradient.  30 016 512 elements per sample and 5-cell forward; 12 276 * 112 per sample and pyramid."""
    fwd = 30016512 * esize * B
    pyr = POS_PER_SAMPLE * C * esize * B
    return 3 * fwd + n_teachers * fwd + (1 + n_teachers) * pyr + 2 * pyr


def bind_to_gpu_numa_node(gpu_index):
    """Best effort: run this process on the CPUs of the NUMA node the GPU hangs off BEFORE the pinned staging buffers are
    allocated and first touched (first-touch places their pages on that node), so that the per-step host->device copies
    of N ranks do not all cross the same socket.  Returns a short description for the bench line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if bus.startswith("0000"):
            bus = bus[4:]               # sysfs uses a 4-digit domain, NVML prints 8
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return "numa_node=-1 (single node / not exposed)"
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpulist = f.read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return "numa_node=%d has no CPU this process may use" % node
        os.sched_setaffinity(0, allowed)
        return "bound to NUMA node %d (%d CPUs)" % (node, len(allowed))
    except Exception as e:  # noqa: BLE001
        return "not bound (%s: %s)" % (type(e).__name__, str(e)[:80])


DUMP_SAMPLE = 1 << 20   # elements kept of each input gradient (dL/dC3 alone is 57 MB in fp32 at batch 32)


def dump_outputs(out_dir, kd, step, student, xs):
    """Write what the last timed step handed its caller as out_dir/<name>.npy (float32): the [teacher, level] MTA losses it
    returned, the averaged flat student gradient, dL/dC3..C5 (a fixed, seeded sample of each, in NCHW element order), and
    the student's parameters and BatchNorm running statistics as that step left them.  Gradients and parameters differ
    in the last bits from run to run (atomic accumulation in the backward): compare dumps within a tolerance."""
    import numpy as np
    arrays = {"kd_losses": kd, "student_grad": step.flat_grad,
              "student_params": torch.cat([p.detach().flatten() for p in student.parameters()]),
              "student_bn_stats": torch.cat([b.flatten() for b in student.buffers() if b.is_floating_point()])}
    gen = torch.Generator().manual_seed(0)
    for name, x in zip(("c3", "c4", "c5"), xs):
        g = x.grad.flatten()
        idx = torch.randperm(g.numel(), generator=gen)[:DUMP_SAMPLE].sort().values
        arrays["input_grad_" + name] = g[idx.to(g.device)]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def measure(B, args, rank, world, dev, dtype, min_timed_s, dump_dir=None):
    """Everything measured at one per-GPU batch size: resident (device-timed) step, end-to-end step, per-kernel
    instrumented pass.  Timed regions are blocks of EXACTLY args.steps steps bracketed by barrier + synchronize; blocks are
    repeated until >= min_timed_s seconds have been timed and the MEDIAN block is reported (max over ranks per block).
    With `dump_dir`, rank 0 writes the outputs of the last resident step there (dump_outputs)."""
    import mm_distillnet_b200 as mmd
    from mm_distillnet_b200 import _lib
    esize = 4 if dtype == torch.float32 else 2

    torch.manual_seed(0)   # identical student init on every rank (DDP broadcast-at-start semantics)
    student = mmd.BiFPNStack(*[mmd.BiFPN(C, CC, first_time=(i == 0)) for i in range(N_CELLS)]).to(dev).train()
    teachers = []
    for k in range(N_TEACHERS):
        torch.manual_seed(1 + k)
        teachers.append(mmd.BiFPNStack(*[mmd.BiFPN(C, CC, first_time=(i == 0)) for i in range(N_CELLS)]).to(dev).eval())
    # the shipped recipe's optimizer (configs/mm-distillnet.cfg: Adam, lr 1e-4, b1 0.9, b2 0.999; train_methods.py:825-833) as
    # ONE launch over the flat gradient, inside the step (and inside its captured graph)
    opt = None if args.no_optimizer else mmd.FlatAdam(student.parameters(), lr=1e-4, betas=(0.9, 0.999))
    step = mmd.DistillStep(student, teachers, mmd.MTALoss(T=9.0, p=2.0), w_kd=W_KD, optimizer=opt)

    gen = torch.Generator().manual_seed(1000 + rank)

    def pinned_nhwc(x):   # pinned host staging buffer already in the kernels' NHWC (channels_last) layout
        h = torch.empty(x.shape, dtype=x.dtype, pin_memory=True).contiguous(memory_format=torch.channels_last)
        if not h.is_pinned():
            h = h.pin_memory()
        h.copy_(x)
        return h

    host_s = [pinned_nhwc(x) for x in synth_inputs(B, gen, dtype)]
    host_t = [[pinned_nhwc(x) for x in synth_inputs(B, gen, dtype)] for _ in range(N_TEACHERS)]
    dev_s = [x.to(dev).contiguous(memory_format=torch.channels_last).requires_grad_(True) for x in host_s]
    dev_t = [[x.to(dev).contiguous(memory_format=torch.channels_last) for x in xs] for xs in host_t]
    for x in dev_s:
        x.requires_grad_(True)   # dL/dC3..C5 are part of the path (they feed the student backbone)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_block(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    def timed(fn, steps, before_block=None):
        blocks, total = [], 0.0
        while True:
            if before_block is not None:
                before_block()
            ms = timed_block(fn, steps)
            blocks.append(ms)
            total += ms
            more = torch.tensor([1.0 if (total < 1e3 * min_timed_s and len(blocks) < 200) else 0.0], device=dev)
            if world > 1:
                dist.all_reduce(more, op=dist.ReduceOp.MIN)   # every rank times the same number of blocks
            if more.item() == 0.0:
                break
        return statistics.median(blocks), blocks

    def eager_step():
        for x in dev_s:
            x.grad = None
        return step(dev_s, dev_t)

    # The whole step is captured once into a CUDA graph (DistillStep.capture) and replayed: ~300 launches of a few
    # microseconds each are host-bound otherwise.  --no-graph times the eager path instead.
    use_graph = not args.no_graph
    if use_graph:
        # two graphs over two static input sets: the pipelined feed of the e2e leg copies the next step's inputs straight
        # into the set that is not running (no staging-to-static copy); the resident leg replays one of them
        step.capture(dev_s, dev_t, warmup=max(args.warmup, 3), double_buffer=not args.no_prefetch)

    last_kd = [None]

    def resident_step():
        last_kd[0] = step.replay() if use_graph else eager_step()

    host_loss = torch.empty(N_TEACHERS, 5, dtype=torch.float32).pin_memory()
    e2e_i, e2e_total = [0], [0]

    def e2e_step():
        if use_graph and not args.no_prefetch:
            # pipelined feed: this step's inputs were requested by the previous iteration (or just now for the first one);
            # the copy of the NEXT step's inputs is started right after the replay is enqueued, so it overlaps the replay.
            # Every timed step still copies its own inputs host->device and reads its own result back.
            if e2e_i[0] == 0:
                step.prefetch(host_s, host_t)
            kd = step.replay_prefetched()
            e2e_i[0] += 1
            if e2e_i[0] < e2e_total[0]:
                step.prefetch(host_s, host_t)
        elif use_graph:
            kd = step.replay(host_s, host_t)            # pinned host -> static device buffers, then the graph
        else:
            xs = [x.to(dev, non_blocking=True).requires_grad_(True) for x in host_s]
            kd = step(xs, host_t)                       # teacher inputs are copied host->device inside the call
        host_loss.copy_(kd, non_blocking=False)         # device->host read of the step's result
        return host_loss

    W = max(args.warmup, 3)
    for _ in range(W):
        resident_step()
    sampler = ClockSampler(dev.index) if rank == 0 else None
    ms, blocks = timed(resident_step, args.steps)
    clocks = sampler.stop() if sampler else None
    torch.cuda.synchronize()
    if dump_dir is not None and rank == 0:   # before the legs below run more steps on the same student
        dump_outputs(dump_dir, last_kd[0], step, student, step.graph_inputs() if use_graph else dev_s)
    l0 = mmd.launch_count()   # replayed launches never pass through the library's host-side counter: count one eager step
    eager_step()
    torch.cuda.synchronize()
    launches_per_step = mmd.launch_count() - l0

    # gradient checksum (N > 1: the averaged flat gradient must be the same on every rank)
    checksum = float(step.flat_grad.double().sum().item()) if step.flat_grad is not None else None
    checks = [checksum]
    if world > 1:
        t = torch.tensor([checksum], dtype=torch.float64, device=dev)
        ts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(ts, t)
        checks = [float(x.item()) for x in ts]

    def e2e_reset():
        e2e_i[0], e2e_total[0] = 0, args.steps

    e2e_total[0] = W
    for _ in range(W):
        e2e_step()
    ms_e2e, blocks_e2e = timed(e2e_step, args.steps, before_block=e2e_reset)

    # host->device feed alone (pinned host -> staging set on the copy stream), for the N > 1 e2e discussion
    h2d = (1 + N_TEACHERS) * B * sum(c * (S3 >> i) ** 2 for i, c in enumerate(CC)) * esize
    h2d_gbs = None
    if use_graph and not args.no_prefetch:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cs = step._copy_stream
        with torch.cuda.stream(cs):
            e0.record(cs)
        for _ in range(5):   # back to back on the copy stream (the staging set is free: no replay is pending)
            step.prefetch(host_s, host_t)
        with torch.cuda.stream(cs):
            e1.record(cs)
        barrier()
        h2d_ms = e0.elapsed_time(e1) / 5
        step._prefetched = False
        if world > 1:
            t = torch.tensor([h2d_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            h2d_ms = t.item()
        h2d_gbs = h2d / (h2d_ms * 1e-3) / 1e9

    # per-kernel CUDA-event timing of the same step (separate instrumented EAGER pass: an event pair around every launch;
    # every rank runs it because the step contains the gradient all-reduce; rank 0 reports its own timings)
    _lib.prof_enable(True)
    _lib.prof_collect()
    nprof = min(args.steps, 5)
    for _ in range(nprof):
        eager_step()
    prof = _lib.prof_collect()
    _lib.prof_enable(False)
    barrier()
    roof = None
    if rank == 0:
        peak, peak_src = peaks()
        total_ms = sum(v["ms"] for v in prof.values())
        dom = max(prof, key=lambda k: prof[k]["ms"])
        d = prof[dom]
        ach = d["algo_bytes"] / (d["ms"] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj.get("%s_b%d" % (args.dtype, B), tj.get(args.dtype, {}) if B == 16 else {}).get(dom)
        step_bytes = algo_bytes_per_step(B, esize)
        roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "peak_source": peak_src,
                "avg_launch_us": 1e3 * d["ms"] / d["launches"], "algo_bytes_per_launch": d["algo_bytes"] / d["launches"],
                "share_of_kernel_time": d["ms"] / total_ms,
                # the WHOLE step against the same roofline: algorithmic bytes of the step / graph-replay time per step
                "step": {"algo_bytes": step_bytes, "ms": ms / args.steps,
                         "achieved": step_bytes / (ms / args.steps * 1e-3) / 1e9,
                         "frac": step_bytes / (ms / args.steps * 1e-3) / 1e9 / peak},
                "timing_note": ("per-kernel times: CUDA events around every launch of an eager pass (sum %.3f ms/step); the "
                                "graph replay of the same launches takes %.3f ms/step (launch gaps and event overhead differ): "
                                "shares are of the instrumented sum" % (total_ms / nprof, ms / args.steps)),
                "all_kernels": {k: {"ms_per_step": v["ms"] / nprof, "launches_per_step": v["launches"] / nprof,
                                    "GBps": (v["algo_bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else None,
                                    "frac": (v["algo_bytes"] / (v["ms"] * 1e-3) / 1e9 / peak) if v["ms"] > 0 and v["algo_bytes"] > 0 else None}
                                for k, v in prof.items()}}
    res = {"B": B, "ms": ms, "blocks": blocks, "ms_e2e": ms_e2e, "blocks_e2e": blocks_e2e, "roof": roof, "clocks": clocks,
           "launches_per_step": launches_per_step, "h2d": h2d, "h2d_gbs": h2d_gbs, "checksums": checks,
           "use_graph": use_graph, "esize": esize}
    # release this batch size's graph / arenas before the next one is measured
    del step, student, teachers
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return res


def run_ours(args, rank, world, local_rank):
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the product path has no CPU fallback)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dtype = torch.float32 if args.dtype == "f32" else torch.bfloat16
    B = args.batch
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else "single rank: not bound"
    main_r = measure(B, args, rank, world, dev, dtype, args.min_seconds, args.dump_outputs)
    cfg2 = None
    if B != 16 and not args.no_cfg2:   # BASELINE configs[1]: the microbench batch, same run, shorter timed region
        cfg2 = measure(16, args, rank, world, dev, dtype, min(args.min_seconds, 1.0))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        Bc, Kc, Wc = B, 3, 1     # the same step at the same batch: ~10-30 s of CPU work on the box's host cores
        ts = time_cpu(Bc, Kc, Wc)
        cpu = {"value": Bc * len(ts) / sum(ts), "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "%d timed steps (%d warm-up) of the same step at batch %d on the oracle port (torch CPU fp32, "
                         "all host threads)" % (Kc, Wc, Bc)}

    if rank != 0:
        return
    r = main_r
    steps, ms, ms_e2e = args.steps, r["ms"], r["ms_e2e"]
    line = {
        "metric": "distill samples/s", "value": B * world * steps / (ms * 1e-3), "unit": "samples/s",
        "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": B * world,
                   "parallelism": "dp%d (flat-gradient NCCL all-reduce)" % world if world > 1 else "single GPU",
                   "l2": "inputs larger than L2: the step streams ~%.1f GB of activations (L2 = 126 MB); no flush needed"
                         % (algo_bytes_per_step(B, r["esize"]) / 1e9),
                   "timed_region": "%d blocks of exactly %d steps each (%.2f s timed in total), median block reported; "
                                   "min / max block %.3f / %.3f ms per step"
                                   % (len(r["blocks"]), steps, sum(r["blocks"]) * 1e-3, min(r["blocks"]) / steps,
                                      max(r["blocks"]) / steps),
                   "optimizer": ("none (--no-optimizer: the step ends at the averaged gradients)" if args.no_optimizer else
                                 "Adam, lr 1e-4, betas (0.9, 0.999) — the shipped recipe's (configs/mm-distillnet.cfg) — as one "
                                 "launch over the flat gradient inside the timed step (mmd_adam_step)"),
                   "precision": "activations stored as %s, all arithmetic fp32 (TMEM accumulators, BatchNorm statistics "
                                "in double, fp32 master weights and gradients)" % args.dtype,
                   "launch": "CUDA graph replay of the whole step" if r["use_graph"] else "eager",
                   "e2e_feed": ("pinned host inputs copied on a side stream into the static input set of the graph that is "
                                "NOT running while the previous step replays (DistillStep.capture(double_buffer=True) / "
                                "prefetch / replay_prefetched: two graphs over two input sets, no staging copy); K copies, "
                                "K replays, K (blocking) loss read-backs inside the timed region") if (r["use_graph"] and not args.no_prefetch)
                               else "inputs copied in front of every step"},
        "roofline": r["roof"], "cpu_baseline": cpu,
        "e2e": {"value": B * world * steps / (ms_e2e * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": r["h2d"],
                "d2h_bytes_per_step": N_TEACHERS * 5 * 4, "ms_per_step": ms_e2e / steps,
                "h2d_feed_GBps_per_rank": r["h2d_gbs"], "host_numa": numa,
                "h2d_ms_per_step_alone": (r["h2d"] / (r["h2d_gbs"] * 1e9) * 1e3) if r["h2d_gbs"] else None,
                "bound": ("host feed: the H2D copy of a step alone takes longer than the resident step"
                          if r["h2d_gbs"] and r["h2d"] / (r["h2d_gbs"] * 1e9) * 1e3 > ms / steps else "device step")},
        "gpu_launches": r["launches_per_step"] * steps, "gpu_launches_per_step": r["launches_per_step"],
        "clocks": r["clocks"],
        "grad_checksum": {"per_rank": r["checksums"], "equal_on_all_ranks": len(set(r["checksums"])) == 1},
    }
    if cfg2 is not None:
        line["cfg2_b16"] = {"batch_per_gpu": 16, "value": 16 * world * steps / (cfg2["ms"] * 1e-3), "unit": "samples/s",
                            "ms_per_step": cfg2["ms"] / steps,
                            "e2e": {"value": 16 * world * steps / (cfg2["ms_e2e"] * 1e-3), "ms_per_step": cfg2["ms_e2e"] / steps},
                            "roofline": cfg2["roof"], "gpu_launches_per_step": cfg2["launches_per_step"]}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300, help="timed steps: every timed leg runs exactly this many; the "
                    "default times about 2 s of the batch-32 step (6.6 ms per step on a B200 at a 1000 W power limit), a "
                    "window of a fraction of a second measures clock and scheduler noise as much as the step")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="bf16", choices=["f32", "bf16"],
                    help="activation STORAGE type; arithmetic (accumulators, statistics, weights) is fp32 in both modes. "
                         "bf16 is the tensor-core product path (BASELINE cfg 3), f32 the bit-level parity mode")
    ap.add_argument("--batch", type=int, default=32, help="samples per GPU per step (cfg3/cfg4: 32; cfg2's 16 is measured "
                    "in the same run and reported as cfg2_b16)")
    ap.add_argument("--min-seconds", type=float, default=0.0, help="repeat the timed block of K steps until this many "
                    "seconds have been timed; the median block is reported (default: one block, exactly K timed steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                    "(float32, see dump_outputs) to compare builds on identical inputs, within a tolerance: the backward "
                    "accumulates with atomics, so gradients and updated parameters vary in the last bits from run to run")
    ap.add_argument("--no-cfg2", action="store_true", help="skip the extra cfg2 (batch 16) measurement")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-optimizer", action="store_true", help="end the step at the averaged gradients (no Adam update)")
    ap.add_argument("--no-graph", action="store_true", help="time the eager step instead of the CUDA-graph replay")
    ap.add_argument("--no-prefetch", action="store_true",
                    help="e2e leg: copy each step's inputs synchronously in front of its replay instead of overlapping the "
                         "copy with the previous step's replay")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the CUDA step (--impl ours)")
        run_reference(args, rank)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"    # keep NCCL's version banner out of stdout: rank 0 prints ONE JSON line
        # NCCL prints its version banner on stdout when the communicator is created: keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            torch.cuda.set_device(local_rank)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    if world == 1:
        run_ours(args, rank, world, local_rank)
        return
    # N > 1: the step's CUDA graph holds captured NCCL kernels; tearing the communicator down while it is alive was
    # observed to hang the processes AFTER rank 0 had printed its line (destroy_process_group never returned).  Every
    # rank has passed the last barrier by then, so: flush, synchronise, leave without the NCCL teardown.
    code = 0
    try:
        run_ours(args, rank, world, local_rank)
    except BaseException:
        import traceback
        traceback.print_exc()
        code = 1
    sys.stdout.flush()
    sys.stderr.flush()
    try:
        torch.cuda.synchronize()
    except Exception:
        code = code or 1
    os._exit(code)


if __name__ == "__main__":
    main()
