#!/usr/bin/env python
"""Benchmark of the HAWQ integer forward path on B200 (DESIGN.md §Measurement).

  python bench.py --gpus N --steps K --warmup W            one JSON line: images/s of the quantized ResNet forward
  python bench.py ... --dump-outputs DIR                   also write the logits of the last timed step to DIR/logits.npy
  python bench.py --impl reference ...                     the reference's CPU path (oracle port) on the host cores

A "step" = one forward of the frozen quantized ResNet over one batch of synthetic int8 images per GPU.
Default workload: ResNet-50 W8A8 (bit_config_resnet50_uniform8), batch 128 per GPU (BASELINE.json configs[2]).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "images/sec ResNet-50 W8A8 & W4A4 @batch128, 1/2/4/8xB200; % int-TC roofline"
MACS_PER_IMAGE = {"resnet18": 1.8141e9, "resnet50": 3.8580e9, "resnet101": 7.57e9}
INT8_TC_PEAK_OPS = 4.5e15        # nominal dense int8 tcgen05 peak (op/s); reported for context only
DUMP_LIMIT_BYTES = 64 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--arch", default="resnet50")
    ap.add_argument("--scheme", default="uniform8")
    ap.add_argument("--batch", type=int, default=128, help="images per GPU per step")
    ap.add_argument("--cpu-batch", type=int, default=8, help="images per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-batch8", action="store_true", help="skip the latency-regime leg (batch 8 per GPU) of the JSON line")
    ap.add_argument("--residual-bits", type=int, default=16)
    ap.add_argument("--a4-storage", default="byte", choices=["byte", "packed"],
                    help="HBM container of 4-bit activations: one value per byte (default, consumed directly by the int8 tensor-core kernels) or packed nibbles expanded on chip")
    ap.add_argument("--detail", default="", help="write per-layer timings to this JSON file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the logits of the last timed step to DIR/logits.npy (float32; inputs are seeded, so runs with the same "
                         "arguments see the same images and two builds can be compared output for output)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    return a


def dump_outputs(path, arrays):
    """Write every array as <path>/<name>.npy in float32.  An array over DUMP_LIMIT_BYTES is replaced by a fixed sample of its rows
    (seed 0, in row order), the same in every run."""
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        a = t.to("cpu", torch.float32).numpy()
        if a.nbytes > DUMP_LIMIT_BYTES:
            rows = DUMP_LIMIT_BYTES // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured", d
    return 6650.0, "fallback", {}


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout=10.0):
        """nvidia-smi needs a moment to start: block until the first sample arrived so that the timed region is covered."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples read between t_begin and t_end (perf_counter times of the timed region)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        rows = [r for t, r in self.rows if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end + 0.05)]
        if not rows:
            rows = [r for _, r in self.rows[-3:]]
        for r in rows:
            f = [v.strip() for v in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def usable_cpus(cap=32):
    """Threads the CPU legs may use: scheduler affinity, limited by the cgroup CPU quota (os.cpu_count() reports the host's
    cores inside a container and oversubscribing them makes oneDNN crawl), capped at `cap` (the fp32 convs do not scale further)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path, parse in (("/sys/fs/cgroup/cpu.max", lambda t: None if t.split()[0] == "max" else float(t.split()[0]) / float(t.split()[1])),
                        ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", None)):
        try:
            txt = open(path).read().strip()
            if parse is not None:
                q = parse(txt)
            else:
                quota = float(txt)
                period = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().strip())
                q = quota / period if quota > 0 else None
            if q:
                n = min(n, max(1, int(q)))
            break
        except (OSError, ValueError, IndexError, ZeroDivisionError):
            continue
    return max(1, min(n, cap))


def cpu_forward_rate(arch, scheme, max_batch, steps, warmup, budget_s=25.0, fixed_batch=False):
    """The reference's fake-quant forward (oracle/fakequant.py restatement, pinned bit-exact to the unmodified reference)
    on the usable host cores.  The per-step sample (images per forward) is sized from a 1-image probe so that `steps` timed
    forwards fit in about `budget_s` seconds.  Returns (images/s, threads, seconds per step, images per step)."""
    from oracle import fakequant as fq
    from hawq_b200.bit_config import get_bit_config
    from hawq_b200.synthetic import synthetic_batch, synthetic_float_resnet
    threads = usable_cpus()
    torch.set_num_threads(threads)
    net = synthetic_float_resnet(arch, 0)
    m = fq.FakeQuantResNet(arch, net, get_bit_config(arch, scheme))
    m(synthetic_batch(1, 0))                       # calibration (ranges do not change the amount of work)
    m.freeze()
    x1 = synthetic_batch(1, 1)
    m(x1)                                          # warm-up (allocator, oneDNN primitive cache)
    t0 = time.perf_counter()
    m(x1)
    per_img = time.perf_counter() - t0
    if fixed_batch:      # every step is a full batch of the workload; the budget bounds the number of steps (>= 1)
        batch = max_batch
        steps = max(1, min(steps, int(budget_s / max(per_img * batch * 0.8, 1e-6)) - 1))
    else:
        steps = max(1, min(steps, int(4 * budget_s / max(per_img, 1e-6))))   # a pathologically slow host: fewer steps rather than minutes
        batch = int(max(1, min(max_batch, budget_s / max(steps, 1) / max(per_img, 1e-6))))
    x = synthetic_batch(batch, 1)
    for _ in range(min(warmup, 1)):
        m(x)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        m(x)
        ts.append(time.perf_counter() - t0)
    sec = sum(ts) / len(ts)
    return batch / sec, threads, sec, batch, steps


def run_reference(a):
    """The reference's CPU path on this box's host cores, on OUR arm's workload: every step is one forward of a.batch images
    (the configuration our JSON line names).  The number of timed steps is bounded by a time budget (a batch-128 ResNet-50
    forward takes ~13 s on 16 cores), and the line says how many ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, a.steps)
    warm = max(1, a.warmup)
    ips, threads, sec, cpu_b, steps = cpu_forward_rate(a.arch, a.scheme, a.batch, steps, warm, budget_s=120.0, fixed_batch=True)
    line = {"metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": a.gpus, "steps": steps, "warmup": 1,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32 emulating int8/int4 (reference fake-quant)", "data": "synthetic", "impl": "reference",
            "config": workload_config(a, 1, None),
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
                             "sample": "%d timed step(s) (of the %d requested: bounded by a 120 s budget), each the forward of %d images, through oracle/fakequant.py "
                                       "(torch CPU restatement of the reference forward, bit-exact vs the unmodified reference in the build container)"
                                       % (steps, max(1, a.steps), cpu_b)},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(a, world, detail):
    """`config` of the JSON line; identical keys for both arms (the reference arm runs the same workload on the host cores)."""
    B = a.batch
    return {"workload": "%s_%s_b%d" % (a.arch, a.scheme, B), "arch": a.arch, "bit_config": a.scheme, "batch_per_gpu": B,
            "global_batch": B * world, "input": "synthetic int8 NHWC 224x224x3",
            "parallelism": "dp%d (batch sharded, logits all-gather)" % world if world > 1 else "single GPU"}


# ----------------------------------------------------------------------------------------------- GPU arm
def start_watchdog(seconds, what):
    """A multi-rank run that stops making progress (a collective some rank never enters) must end by itself: after `seconds`
    the process prints why and exits with status 3 instead of waiting for an outer timeout."""
    def fire():
        sys.stderr.write("bench.py watchdog: %s still running after %d s - aborting\n" % (what, seconds))
        sys.stderr.flush()
        os._exit(3)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()
    return t


def run_ours(a):
    import torch.distributed as dist
    import hawq_b200 as hb
    from hawq_b200 import ops
    from hawq_b200.build import build_library
    from hawq_b200.synthetic import synthetic_batch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (the product has no CPU path); use --impl reference for the CPU arm")
    # CPU-side calibration / plan building: share the usable host cores between the ranks of this node
    torch.set_num_threads(max(1, usable_cpus() // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        start_watchdog(int(os.environ.get("HAWQ_BENCH_WATCHDOG_S", "420")), "rank %d of %d" % (rank, world))
    build_library()

    B = a.batch
    from hawq_b200 import qtensor as _qt
    _qt.config.a4_container = 4 if a.a4_storage == "packed" else 8
    q = hb.build_synthetic_qresnet(a.arch, a.scheme, calib_batch=4, calib_seed=0)
    s_in = float(q.quant_input.current_scale())
    # synthetic int8 images: POOL different batches per rank so consecutive steps never see the same input
    POOL = 4
    g = torch.Generator().manual_seed(1234 + rank)
    host_pool = [torch.clamp(torch.round(torch.randn(B, 224, 224, 3, generator=g) / s_in), -128, 127).to(torch.int8).pin_memory()
                 for _ in range(POOL)]
    dev_pool = [t.to(dev) for t in host_pool]
    # N > 1: the one collective of the path (all-gather of the logits, BASELINE config 5) is captured inside the CUDA graph
    eng = hb.compile_model(q, dev_pool[0], residual_bits=a.residual_bits, gather=(world > 1))

    def step(i, src):
        return eng.run_async(src[i % POOL])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput ("value")
    for i in range(max(a.warmup, 3)):
        step(i, dev_pool)
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks is not None:
        clocks.wait_first()
    barrier()
    t_begin = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(a.steps):
        out = step(i, dev_pool)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    flag = int(eng.flag.item())
    last = out.clone() if a.dump_outputs and rank == 0 else None     # later legs replay the same graph into the same buffer
    # ---- end-to-end through the public call with host buffers ("e2e")
    # public call: CompiledModel.run_pipelined(host batches) -> host logits; per step it copies the pinned int8 batch H2D,
    # replays the forward, reads logits + status flags back D2H (checked before the result is handed out)
    def batches(n):
        for i in range(n):
            yield host_pool[i % POOL]
    # (N > 1: the gathered logits stay on the device, as the consumer of a sharded batch would use them; the host reads this
    # rank's shard of the result)
    for _ in eng.run_pipelined(batches(3)):
        pass
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    checksum = 0.0
    for res in eng.run_pipelined(batches(a.steps)):
        checksum += float(res[0, 0])                   # the host really consumes every result
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    clk = clocks.stop(t_begin, time.perf_counter()) if clocks is not None else None

    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])

    # ---- parity of the timed configuration: the logits of one timed batch (CUDA graph, uint16 stream, fused kernels) against an
    # eager run of the same batch on the int32 residual stream without ratio promises (generic saturating kernels)
    # (N > 1: the replay contains the all-gather, so every rank takes part; each checks its own shard, rank 0 reports)
    parity = parity_check(hb, q, eng, dev_pool[0], rank)
    if world > 1:
        ok = torch.tensor([1 if parity["bit_equal"] else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        parity["bit_equal"] = bool(int(ok.item()))
        parity["ranks_checked"] = world
    if rank != 0:
        parity = None
    # ---- roofline leg: per-launch CUDA-event timing of an eager (un-graphed) pass, same stream, same buffers
    roof, detail = None, None
    if rank == 0 and not a.no_roofline:
        roof, detail = roofline_leg(hb, ops, q, dev_pool, a, ms / a.steps)
    # ---- latency regime (the reference's own CPU benchmark runs batch 8): same model, 8 images per GPU per step
    small = None
    if rank == 0 and not a.no_batch8 and B != 8:
        small = small_batch_leg(hb, q, dev, s_in, a, 8)
    cpu = None
    if rank == 0 and not a.no_cpu_baseline:
        ips, threads, sec, cpu_b, _ = cpu_forward_rate(a.arch, a.scheme, a.cpu_batch, 3, 1, budget_s=20.0)
        cpu = {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
               "sample": "3 forwards of %d image(s) (%.2f s each) through oracle/fakequant.py, the torch-CPU restatement of the "
                         "reference's fake-quant forward (the Python reference itself cannot travel to the GPU box)" % (cpu_b, sec)}
    if rank == 0:
        total_imgs = B * world * a.steps
        value = total_imgs / (ms / 1e3)
        macs = MACS_PER_IMAGE.get(a.arch, 0.0)
        line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
                "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int8" if a.scheme == "uniform8" else (("int4 values (%s in HBM) / int8 MMA" if a.scheme == "uniform4" else "mixed int4 (%s in HBM) and int8 / int8 MMA")
                                                                % ("packed nibbles" if a.a4_storage == "packed" else "one per byte")),
                "data": "synthetic",
                "config": dict(workload_config(a, world, detail),
                               l2=("per-step working set (%.1f GB of activations) exceeds the 126 MB L2; %d input batches rotate" % (detail["act_bytes"] / 1e9, POOL)) if detail and detail["act_bytes"] > 2.5e8
                               else "%d input batches rotate; at this batch size the per-step working set is L2-resident (latency-bound regime)" % POOL,
                               residual_stream="uint%d" % a.residual_bits if a.residual_bits == 16 else "int32", cuda_graph=True,
                               a4_storage=a.a4_storage,
                               overflow_flag_seen=bool(flag & 1)),
                "e2e": {"value": total_imgs / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": int(host_pool[0].numel()),
                        "d2h_bytes_per_step": int(B * 1000 * 4 + 4), "ms_per_step": ms_e2e / a.steps,
                        "int32_fallbacks": eng.fallbacks},
                "gpu_launches": eng.gpu_launches * a.steps,
                "clocks": clk,
                "tensor": {"achieved_tops": 2 * macs * value / 1e12, "nominal_int8_peak_tops": INT8_TC_PEAK_OPS / 1e12,
                           "frac_of_nominal": 2 * macs * value / INT8_TC_PEAK_OPS},
                "parity": parity, "roofline": roof, "cpu_baseline": cpu, "batch8": small}
        print(json.dumps(line))
        if last is not None:
            dump_outputs(a.dump_outputs, {"logits": last})
        if a.detail and detail is not None:
            with open(a.detail, "w") as f:
                json.dump(detail, f, indent=1)
    if world > 1:
        # Every rank is done once this barrier returns.  The process ends here: tearing the NCCL communicator down while CUDA
        # graphs that captured its kernels are still alive blocked on the GPU box (seen at N = 2), and nothing is left to clean up.
        barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def small_batch_leg(hb, q, dev, s_in, a, b):
    """The same network at `b` images per step on this GPU (own CUDA graph): device-resident and end-to-end images/s, timed like
    the headline numbers (CUDA events on the launch stream, synchronised on both sides)."""
    g = torch.Generator().manual_seed(99)
    host = [torch.clamp(torch.round(torch.randn(b, 224, 224, 3, generator=g) / s_in), -128, 127).to(torch.int8).pin_memory() for _ in range(4)]
    devs = [t.to(dev) for t in host]
    eng = hb.compile_model(q, devs[0], residual_bits=a.residual_bits)
    steps = max(4 * a.steps, 100)
    for i in range(10):
        eng.run_async(devs[i % 4])
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        eng.run_async(devs[i % 4])
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    flag = int(eng.flag.item())
    for _ in eng.run_pipelined(host[i % 4] for i in range(3)):
        pass
    torch.cuda.synchronize(dev)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    acc = 0.0
    for res in eng.run_pipelined(host[i % 4] for i in range(steps)):
        acc += float(res[0, 0])
    f1.record()
    torch.cuda.synchronize(dev)
    ms2 = f0.elapsed_time(f1)
    return {"batch": b, "n_gpus": 1, "steps": steps, "value": b * steps / (ms / 1e3), "unit": "images/s", "ms_per_step": ms / steps,
            "e2e": {"value": b * steps / (ms2 / 1e3), "unit": "images/s", "ms_per_step": ms2 / steps,
                    "h2d_bytes_per_step": int(host[0].numel()), "d2h_bytes_per_step": int(b * 1000 * 4 + 4)},
            "gpu_launches_per_step": eng.gpu_launches, "overflow_flag_seen": bool(flag & 1),
            "note": "latency-bound regime: the per-step working set is L2-resident, %d kernels per step" % eng.gpu_launches}


def parity_check(hb, q, eng, x, rank=0):
    """Logits of one timed batch through the benchmarked path vs an eager (un-graphed) run of the same batch with int32
    residuals and no ratio promises.  Two independent kernel sets (fused tcgen05 / generic IMMA) must agree bit for bit."""
    from hawq_b200 import qtensor
    from hawq_b200.qtensor import IntActivation, Node
    fast = eng(x).clone()
    n, h, w, c = x.shape
    if fast.shape[0] != n:                 # gathered logits of the whole sharded batch: this rank's shard
        fast = fast[rank * n:(rank + 1) * n]
    with torch.no_grad(), qtensor.engine_mode(residual_bits=32, fast_kernels=False, checked=False):
        ref = q(IntActivation(Node("int", (n, c, h, w), data=x.view(-1), bits=8, signed=True), x.device))
    torch.cuda.synchronize()
    return {"what": "all %d x %d logits of one timed batch: benchmarked path (CUDA graph, fused tcgen05 kernels, uint16 stream) vs eager generic "
                    "kernels on the int32 stream" % tuple(fast.shape),
            "bit_equal": bool(torch.equal(fast, ref)), "rows_checked": int(fast.shape[0])}


def build_digest():
    from hawq_b200.build import OUT
    try:
        return open(OUT + ".stamp").read().strip()[:16]
    except OSError:
        return None


def roofline_leg(hb, ops, q, dev_pool, a, graph_ms_per_step):
    """Per-launch CUDA-event timing of an eager pass (torch current stream = the launching stream) gives every kernel's SHARE of
    the step; the denominator of `achieved` is the graph-timed step of the timed region x that share (the eager event sum exceeds
    the graph-timed step: no PDL overlap, event gaps)."""
    from hawq_b200 import qtensor
    from hawq_b200.qtensor import IntActivation, Node
    peak, which, _ = measured_peaks()
    reps = 5
    rows = {}
    for r in range(reps + 1):
        ops.timer = [] if r > 0 else None
        x = dev_pool[r % len(dev_pool)]
        n, h, w, c = x.shape
        # park the GPU behind a spin kernel while the host enqueues the whole forward (tensor-map encoding makes some launches
        # host-bound): the events then bracket back-to-back GPU execution, not the host's launch pace
        torch.cuda._sleep(int(3e7))
        with torch.no_grad(), qtensor.engine_mode(residual_bits=a.residual_bits, checked=True):
            q(IntActivation(Node("int", (n, c, h, w), data=x.view(-1), bits=8, signed=True), x.device))
        torch.cuda.synchronize()
        if r > 0:
            for i, (name, info, e0, e1) in enumerate(ops.timer):
                rows.setdefault(i, {"kernel": name, "macs": info[0], "bytes": info[1], "ms": []})["ms"].append(e0.elapsed_time(e1))
    ops.timer = None
    layers = []
    agg = {}
    for i in sorted(rows):
        r = rows[i]
        ms = statistics.median(r["ms"])
        layers.append({"i": i, "kernel": r["kernel"], "ms": ms, "macs": r["macs"], "bytes": r["bytes"],
                       "GBps": r["bytes"] / ms / 1e6, "TOPS": 2 * r["macs"] / ms / 1e9})
        g = agg.setdefault(r["kernel"], {"ms": 0.0, "bytes": 0, "macs": 0, "launches": 0})
        g["ms"] += ms; g["bytes"] += r["bytes"]; g["macs"] += r["macs"]; g["launches"] += 1
    total_ms = sum(g["ms"] for g in agg.values())
    scale = graph_ms_per_step / total_ms             # eager event time -> time inside the graph-timed step
    # kernel families: conv_tc (+ its dual-accumulator instantiation) is one template; conv_halo is the in-place 3x3 kernel
    fam = {}
    for k, g in agg.items():
        f = fam.setdefault("conv_tc_kernel" if k.startswith("conv_tc") else ("conv_halo_kernel" if k == "conv_halo" else "conv1x1_kernel" if k == "conv1x1" else "conv_dual_kernel" if k == "conv_dual" else "stem_tc_kernel" if k == "stem_tc" else k),
                           {"ms": 0.0, "bytes": 0, "macs": 0, "launches": 0})
        for key in f:
            f[key] += g[key]
    top = max(fam, key=lambda k: fam[k]["ms"])
    t = fam[top]
    achieved = t["bytes"] / (t["ms"] * scale / 1e3) / 1e9
    # measured DRAM traffic of that kernel: from the ncu pass over this command with THIS build (tools/summarize_ncu.py writes the
    # build digest next to the numbers); a stale or missing entry gives null
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            ent = json.load(f).get("%s:%s:%d" % (a.arch, a.scheme, a.batch))
        if ent and ent.get("build") == build_digest() and top in ent.get("kernels", {}):
            traffic = ent["kernels"][top]["traffic_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        traffic = None
    families = {k: {"launches_per_step": v["launches"], "share_of_step": v["ms"] / total_ms, "ms_in_step": v["ms"] * scale,
                    "algorithmic_GBps": v["bytes"] / (v["ms"] * scale / 1e3) / 1e9, "frac_of_hbm_peak": v["bytes"] / (v["ms"] * scale / 1e3) / 1e9 / peak,
                    "tensor_tops": 2 * v["macs"] / (v["ms"] * scale / 1e3) / 1e12} for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
    step_bytes = sum(g["bytes"] for g in agg.values())
    roof = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": "%s (MEASURED_PEAKS.json hbm_gbs)" % which if which == "measured" else "fallback 6650 GB/s",
            "traffic": traffic, "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, ncu, this build)" if traffic else None,
            "algorithmic_bytes_per_launch": t["bytes"] / t["launches"],
            "launches_per_step": t["launches"], "share_of_step": t["ms"] / total_ms,
            "algorithmic_bytes_per_step": t["bytes"], "avg_launch_ms": t["ms"] * scale / t["launches"],
            "tensor_tops": 2 * t["macs"] / (t["ms"] * scale / 1e3) / 1e12,
            "whole_step": {"algorithmic_bytes": step_bytes, "GBps": step_bytes / (graph_ms_per_step / 1e3) / 1e9,
                           "frac_of_hbm_peak": step_bytes / (graph_ms_per_step / 1e3) / 1e9 / peak},
            "families": families, "eager_event_sum_ms": total_ms, "graph_ms_per_step": graph_ms_per_step,
            "note": "all %d %s launches of one step: sum of algorithmic bytes / (graph-timed ms per step of the timed region x the family's share of "
                    "the per-launch CUDA-event times of an eager pass on the launch stream)" % (t["launches"], top)}
    detail = {"layers": layers, "by_kernel": agg, "act_bytes": step_bytes, "eager_step_ms": total_ms, "graph_ms_per_step": graph_ms_per_step}
    return roof, detail


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
