#!/usr/bin/env python
"""bench.py — the hot path's headline benchmark (BASELINE.json: "GFLOP/s at N=K=M=16384 fp32").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

One step = one MatrixMultiplicationKernel invocation C = A * B (operand preparation + GEMM, or the
configured semiring) over one batch of synthetic matrices through the C-ABI of libmm_b200.so.
For N > 1 (torchrun, one rank per GPU, NCCL) C is cut into an r x c grid of blocks, one per rank
(gemm_hls_b200/multi.py; c = 1 is the plain row-block split), B is broadcast ONCE from rank 0 before the
timed region (no per-step collective, SURVEY.md 8e), every rank multiplies its block each step;
time = max over ranks, value = total ops / time.

Printed JSON line (rank 0): see the contract in the task statement; in addition
  roofline      dominant kernel's achieved rate vs the measured peak (MEASURED_PEAKS.json)
  cpu_baseline  the reference's own Naive<> (oracle/_ref, include/Utility.h:18-42) timed on this
                host's cores on a bounded sample of the same workload (rank 0, N == 1)
  e2e           the same metric through ONE host-pointer call for the whole problem, H2D + D2H inside: mm_gemm_host()
                at N = 1, mm_multi_gemm_host() over all N GPUs (issued by rank 0) at N > 1
`--impl reference` times only the reference CPU path (oracle/_ref; the oracle port if absent).
`--dump-outputs DIR` writes the C of the last timed step to DIR (dump_rows) so that two builds can be compared
output for output: the inputs are drawn from fixed seeds, identical on every run with the same arguments.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (dtype name, map, reduce, n, k, m, BASELINE.json config it is)
    "float16384": ("float", "Multiply", "Add", 16384, 16384, 16384, "configs[1] float 16384^3 tcgen05"),
    "half32768": ("half", "Multiply", "Add", 32768, 32768, 32768, "configs[2] half 32768^3"),
    "double8192": ("double", "Multiply", "Add", 8192, 8192, 8192, "configs[3] double 8192^3"),
    "addmin8192": ("float", "Add", "Min", 8192, 8192, 8192, "configs[4] (add,min) float 8192^3"),
    "uint8_16384": ("uint8_t", "Multiply", "Add", 16384, 16384, 16384, "SURVEY.md 8(f3): uint8_t on tcgen05 kind::i8"),
    "half8192": ("half", "Multiply", "Add", 8192, 8192, 8192, "experiments: with --flags 2 the bit-exact half datapath the half host programs run"),
    "float4096": ("float", "Multiply", "Add", 4096, 4096, 4096, "reduced size, debugging only"),
}
DEFAULT_WORKLOAD = "float16384"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        p["_source"] = "measured"
        return p
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


class ClockSampler:
    """SM clock, board power and clock-event (throttle) reasons DURING the timed region, sampled in-process
    through NVML every ~2 ms (nvidia-smi -lms 200 gave 2-3 samples over a 0.2 s region); falls back to
    polling nvidia-smi when the NVML binding is missing."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, device_index, interval_s=0.002):
        self.idx, self.interval = device_index, interval_s
        self.samples, self.stop_flag, self.thread, self.nvml = [], threading.Event(), None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it lists ordinals
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = self.idx
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                phys = int(vis.split(",")[self.idx])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None
        self.thread = threading.Thread(target=self._pump_nvml if self.nvml else self._pump_smi, daemon=True)
        self.thread.start()

    def _pump_nvml(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((time.perf_counter(), float(sm), float(self.max_sm), pw, int(rs)))
            except Exception:
                pass
            time.sleep(self.interval)

    def _pump_smi(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active"
        while not self.stop_flag.is_set():
            try:
                r = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5)
                f = [x.strip() for x in r.stdout.strip().split(",")]
                self.samples.append((time.perf_counter(), float(f[0]), float(f[1]), float(f[2]), int(f[3], 16)))
            except Exception:
                pass
            time.sleep(0.05)

    def mark(self):
        return time.perf_counter()

    def stop(self, t_begin=None, t_end=None):
        """Summary over the samples taken in [t_begin, t_end] (the timed region; all samples when not given)."""
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=5)
        sel = [x for x in self.samples if (t_begin is None or x[0] >= t_begin) and (t_end is None or x[0] <= t_end)]
        if not sel:
            sel = self.samples
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"], "samples": 0}
        sm = [x[1] for x in sel]
        power = [x[3] for x in sel]
        bits = 0
        for x in sel:
            bits |= x[4]
        return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": max(x[2] for x in sel),
                "power_w_max": max(power), "power_w_avg_under_load": sum(power) / len(power),
                "samples": len(sel), "source": "nvml" if self.nvml else "nvidia-smi",
                "reasons": sorted(k for k, v in self.REASONS.items() if bits & v)}


def gpu_numa_node(index):
    """NUMA node the GPU hangs off (PCI sysfs), or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = "/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]
        node = int(open(path).read())
        return node if node >= 0 else None
    except Exception:
        return None


def node_cpus(node):
    cpus = set()
    try:
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
    except Exception:
        pass
    return cpus


def alloc_host_rows(torch, rows, cols, np_dtype, blocks):
    """Page-locked host matrix whose row-blocks `blocks` = [(r0, r1, gpu index), ...] live on the NUMA node of the GPU
    that will copy them (one pinned allocation from one thread puts every page on one socket; the GPUs of the other
    socket then pull their blocks across the inter-socket link: 416 instead of 950 TFLOP/s end to end at 8 GPUs).
      one block   cudaHostAlloc (torch pin_memory) issued from a thread pinned to the GPU's node
      several     an anonymous mapping (transparent huge pages requested), each block first-touched by a thread
                  pinned to its GPU's node, then cudaHostRegister
    Returns (numpy array, keep-alive object, placement note)."""
    import mmap
    import numpy as np
    nodes = [gpu_numa_node(g) for _, _, g in blocks]

    def pinned(cpus, fn):
        def run():
            if cpus:
                try:
                    os.sched_setaffinity(0, cpus)   # pid 0 = the calling THREAD
                except OSError:
                    pass
            fn()
        t = threading.Thread(target=run)
        t.start()
        t.join()

    if len(blocks) == 1:
        box = {}
        pinned(node_cpus(nodes[0]) if nodes[0] is not None else set(),
               lambda: box.setdefault("t", torch.empty((rows, cols), dtype=torch.from_numpy(np.empty(0, np_dtype)).dtype,
                                                       pin_memory=True)))
        return box["t"].numpy(), box["t"], "cudaHostAlloc from a thread on NUMA node %s" % nodes[0]
    nbytes = rows * cols * np.dtype(np_dtype).itemsize
    m = mmap.mmap(-1, max(nbytes, mmap.PAGESIZE))
    try:
        m.madvise(mmap.MADV_HUGEPAGE)
    except (AttributeError, OSError, ValueError):
        pass
    arr = np.frombuffer(m, dtype=np_dtype, count=rows * cols).reshape(rows, cols)
    for (r0, r1, _), node in zip(blocks, nodes):
        pinned(node_cpus(node) if node is not None else set(), lambda r0=r0, r1=r1: arr[r0:r1].fill(0))
    rc = torch.cuda.cudart().cudaHostRegister(arr.ctypes.data, nbytes, 0)
    rc = int(rc[0]) if isinstance(rc, tuple) else int(rc)
    note = ("registered page-locked, row-blocks first-touched on NUMA nodes %s" % nodes) if rc == 0 else \
           ("cudaHostRegister failed (%d): pageable" % rc)
    return arr, (m if rc == 0 else None), note


def host_threads():
    """Host threads for the reference's CPU path: one per PHYSICAL core this process may run on.

    Naive<> walks a column of B with a stride of M elements: 16384 cache lines (1 MiB) per output element,
    reused by the next 15 columns.  That working set fits one core's private L2 once, not twice, so two
    hyper-threads on a core evict each other (on the 128-thread host of the B200 boxes a float 16384^2 step
    with one row on each of the 128 logical CPUs did not finish within 45 s; one row on one thread takes 5 s)."""
    try:
        allowed = set(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        allowed = None
    cores, cpu, pkg = set(), None, None
    try:
        for line in open("/proc/cpuinfo"):
            key, _, val = line.partition(":")
            key, val = key.strip(), val.strip()
            if key == "processor":
                cpu, pkg = int(val), None
            elif key == "physical id":
                pkg = val
            elif key == "core id" and cpu is not None and (allowed is None or cpu in allowed):
                cores.add((pkg, val))
    except OSError:
        pass
    if cores:
        return len(cores)
    return max(1, len(allowed) if allowed else (os.cpu_count() or 1))


def reference_naive_sample(dtype_name, mp_name, rd_name, a_rows, b, k, m, threads=1):
    """Time the reference's own Naive<> (oracle/_ref) on the rows of C that `a_rows` selects.

    Naive<> is single-threaded as written (include/Utility.h:18-42); C rows are independent, so
    `threads` host threads each run the reference's unmodified routine on their own share of the rows
    (ctypes releases the GIL during the call).  Returns (wall seconds, kind, threads used)."""
    from concurrent.futures import ThreadPoolExecutor
    import oracle as O
    dt = {"float": O.FLOAT, "half": O.HALF, "double": O.DOUBLE, "uint8_t": O.UINT8}[dtype_name]
    mp, rd = getattr(O, mp_name.upper()), getattr(O, rd_name.upper())
    rows = a_rows.shape[0]
    threads = max(1, min(threads, rows))
    bounds = [rows * i // threads for i in range(threads + 1)]
    use_ref = O.ref_available(dt, mp, rd)
    if use_ref:
        O.ref_lib(dt, mp, rd)   # load once, before the threads race for it
    else:
        O.lib()

    def work(i):
        lo, hi = bounds[i], bounds[i + 1]
        if use_ref:
            O.ref_naive(dt, mp, rd, a_rows[lo:hi], b, hi - lo, k, m)
        else:
            O.naive(dt, mp, rd, a_rows[lo:hi], b, hi - lo, k, m, threads=1)

    t0 = time.perf_counter()
    if threads == 1:
        work(0)
    else:
        with ThreadPoolExecutor(max_workers=threads) as ex:
            list(ex.map(work, range(threads)))
    return time.perf_counter() - t0, ("reference" if use_ref else "port"), threads


SAMPLE_COLS = 2048   # columns of C per sampled row of the CPU arm (full K): bounds a step to a few seconds


def cpu_sample_inputs(np_dt, k, m, rows, rng=None, a_rows=None, b=None):
    """The bounded sample both CPU legs time: `rows` rows of C restricted to the first SAMPLE_COLS columns, full K.
    Fixed shape (no adaptive shrinking), so that two runs on the same box time the same work."""
    import numpy as np
    cols = min(SAMPLE_COLS, m)
    if b is None:
        b = rng.uniform(1, 10, size=(k, cols)).astype(np_dt)
    else:
        b = np.ascontiguousarray(b[:, :cols])
    if a_rows is None:
        a_rows = rng.uniform(1, 10, size=(rows, k)).astype(np_dt)
    return a_rows, b, cols


def cpu_sample_text(rows, k, cols, threads):
    return ("%d rows x first %d columns of C, full K (%d x %d x %d per step): the reference's Naive<> "
            "(include/Utility.h:18-42, single-threaded as written) on %d host threads (one per physical core), each "
            "on its own rows; fixed sample, no adaptive shrinking" % (rows, cols, rows, k, cols, threads))


def cpu_baseline_line(dtype_name, mp_name, rd_name, unit, k, m, a_rows_of, b):
    """The `cpu_baseline` object of the B200 arm: the reference's Naive<> on the same bounded sample the
    reference arm times — one row of C per physical core, first SAMPLE_COLS columns, full K."""
    threads = host_threads()
    a_rows, b_s, cols = cpu_sample_inputs(None, k, m, threads, a_rows=a_rows_of(threads), b=b)
    rows = a_rows.shape[0]
    reference_naive_sample(dtype_name, mp_name, rd_name, a_rows, b_s, k, cols, threads)  # warm-up (page faults, library load)
    secs, kind, threads = reference_naive_sample(dtype_name, mp_name, rd_name, a_rows, b_s, k, cols, threads)
    return {"value": 1e-9 * 2.0 * rows * k * cols / secs, "unit": unit, "cores": threads, "kind": kind,
            "seconds": secs, "host_cpus": os.cpu_count(), "sample": cpu_sample_text(rows, k, cols, threads)}


DUMP_BYTES = 64 * 10 ** 6   # --dump-outputs writes at most this much in all


def dump_rows(directory, name, c, budget):
    """Write the device matrix `c` as DIR/<name>.npy in float32 (float64 for double): every row when they fit `budget`
    bytes, otherwise a sample of rows drawn with a fixed seed (the same rows on every run of the same shape).  The
    indices of the written rows go beside it as DIR/<name>_rows.npy (float64, exact)."""
    import numpy as np
    import torch
    wide = torch.float64 if c.dtype == torch.float64 else torch.float32
    n, m = c.shape
    row_bytes = m * torch.empty((), dtype=wide).element_size()
    keep = min(n, (budget - 4096) // (row_bytes + 8))   # 4096: room for the two .npy headers
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name + ".npy"), c[torch.from_numpy(rows).to(c.device)].to(wide).cpu().numpy())
    np.save(os.path.join(directory, name + "_rows.npy"), rows.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--flags", type=int, default=0, help="MM_FLAG_* bits (debugging)")
    ap.add_argument("--tune", default="", help="comma-separated knob=value pairs for mm_context_set_tuning (sweeps)")
    ap.add_argument("--emulate-ranks", type=int, default=0,
                    help="experiments only: time ONE rank's row-block of an R-GPU split on this GPU (N/R rows); "
                         "the printed value is that block's own rate, not a multi-GPU figure")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write C of the last timed step as DIR/c.npy (a fixed row sample when larger than 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dtype_name, mp_name, rd_name, N, K, M, cfg_label = WORKLOADS[args.workload]
    if args.emulate_ranks > 1:
        N = (N + args.emulate_ranks - 1) // args.emulate_ranks
        cfg_label += " — ONE row-block of a %d-GPU split, emulated on one GPU (experiment)" % args.emulate_ranks
        args.no_e2e = args.no_cpu = True
    ops_total = 2.0 * N * K * M
    metric = "GFLOP/s" if (mp_name, rd_name) == ("Multiply", "Add") else "GOp/s"
    metric_name = "%s at N=%d K=%d M=%d %s (%s,%s)" % (metric, N, K, M, dtype_name, mp_name, rd_name)
    # `config` names the workload and nothing run-dependent: both arms print it byte for byte
    from gemm_hls_b200 import multi as partition   # pure-Python host logic (no CUDA needed to import)
    grid_r, grid_c = partition.rank_grid(args.gpus, N, K, M)
    config = {"workload": "%s %dx%dx%d (%s,%s)" % (dtype_name, N, K, M, mp_name, rd_name), "baseline_config": cfg_label,
              "partition": ("C blocks over a %d x %d grid of %d GPU(s): %d row-block(s) x %d column-block(s); a rank holds (and "
                            "prepares, every step) its A row-block and its B column-block; no collective inside a step"
                            % (grid_r, grid_c, args.gpus, grid_r, grid_c)),
              "l2": "inputs (A+B+C = %.2f GB) far larger than the 126 MB L2; no explicit flush" %
                    (1e-9 * {"float": 4, "half": 2, "double": 8, "uint8_t": 1}[dtype_name] * (N * K + K * M + N * M))}

    import numpy as np
    np_dt = {"float": np.float32, "half": np.float16, "double": np.float64, "uint8_t": np.uint8}[dtype_name]

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        # one step = one row of C per physical core (C rows are independent; every thread runs the reference's
        # single-threaded Naive<> on its own row), restricted to the first SAMPLE_COLS columns so that W + K steps
        # end within minutes.  The sample is FIXED: same rows, columns and thread count on every run of a box.
        threads = host_threads()
        rng = np.random.default_rng(5)
        a_rows, b, cols = cpu_sample_inputs(np_dt, K, M, threads, rng=rng)
        kind = "reference"
        for _ in range(args.warmup):
            reference_naive_sample(dtype_name, mp_name, rd_name, a_rows, b, K, cols, threads)
        t = 0.0
        for _ in range(args.steps):
            dt_s, kind, threads = reference_naive_sample(dtype_name, mp_name, rd_name, a_rows, b, K, cols, threads)
            t += dt_s
        value = 1e-9 * 2.0 * threads * K * cols * args.steps / t
        print(json.dumps({
            "impl": "reference", "metric": metric_name, "value": value, "unit": metric, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype_name,
            "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": metric, "cores": threads, "kind": kind,
                             "sample": cpu_sample_text(threads, K, cols, threads)},
            "e2e": {"value": value, "unit": metric, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return 0

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    import gemm_hls_b200 as G

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")  # CPU-side barrier: ranks that wait must not spin on their GPU

    t_dt = {"float": torch.float32, "half": torch.float16, "double": torch.float64, "uint8_t": torch.uint8}[dtype_name]
    dtype = G.DTYPE_FROM_NAME[dtype_name]
    mp, rd = G.OP_FROM_NAME[mp_name], G.OP_FROM_NAME[rd_name]
    es = torch.empty((), dtype=t_dt).element_size()
    tune = {kv.split("=")[0]: int(kv.split("=")[1]) for kv in args.tune.split(",") if kv}

    # Block of this rank.  Outer tiles (n0, m0) of C are fully independent (kernel/Compute.cpp:53-56), so C is cut
    # over a grid_r x grid_c grid of ranks: rank (i, j) computes rows block i x columns block j from A's row-block i and
    # B's column-block j.  grid_c = 1 is SURVEY.md 8e's row-block split with B replicated; a 2-D grid replicates less
    # operand preparation per step (each rank rounds 1/grid_r of A and 1/grid_c of B instead of all of B).
    w = {"float": 16, "half": 32, "double": 8, "uint8_t": 64}[dtype_name]   # columns stay multiples of the 64-byte memory word
    r0, r1, c0, c1 = partition.rank_block(rank, (grid_r, grid_c), N, M, w)
    n_local, m_local = r1 - r0, c1 - c0

    gen = torch.Generator(device=dev)
    gen.manual_seed(5 + rank)
    # synthetic U[1,10) inputs as in the reference recipe (test/TestSimulation.cpp:46-55); half uses
    # U[0,1) so that C stays finite in half (SURVEY.md trap 5)
    lo, hi = (0.0, 1.0) if dtype_name == "half" else ((0.0, 256.0) if dtype_name == "uint8_t" else (1.0, 10.0))

    def draw(shape, g):   # uint8_t: the full value range, so that the modulo-256 wrap-around is exercised
        if dtype_name == "uint8_t":
            return torch.randint(0, 256, shape, generator=g, device=dev, dtype=torch.uint8)
        return (torch.rand(shape, generator=g, device=dev, dtype=torch.float32) * (hi - lo) + lo).to(t_dt)

    a_blk = draw((n_local, K), gen)
    if rank == 0:
        b_full = draw((K, M), gen)
    else:
        b_full = torch.empty((K, M), device=dev, dtype=t_dt)
    extra = {}
    if world > 1:
        partition.broadcast_b(b_full, 0)  # the ONE collective of the path: B over NVLink/NVSwitch
        # reported beside the step time (SURVEY.md 8d): the same broadcast once more, now that the
        # communicator exists, timed on the device, max over ranks
        torch.cuda.synchronize()
        dist.barrier()
        eb0, eb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eb0.record()
        dist.broadcast(b_full, src=0)
        eb1.record()
        torch.cuda.synchronize()
        tb = torch.tensor([eb0.elapsed_time(eb1)], device=dev, dtype=torch.float64)
        dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        extra["broadcast_b"] = {"ms": round(float(tb.item()), 4), "bytes": b_full.numel() * b_full.element_size(),
                                "note": "one NCCL broadcast of B before the timed region (SURVEY.md 8e)"}
    # the kernels take dense matrices (no leading dimension, like the reference): this rank's column-block of B
    # becomes its own contiguous K x m_local array, once, with the broadcast, before the timed region
    b_use = partition.local_b(b_full, c0, c1)
    c_blk = torch.empty((n_local, m_local), device=dev, dtype=t_dt)
    torch.cuda.synchronize()

    ctx = G.Context(local_rank)
    ctx.set_tuning(**tune)
    # a dedicated (non-default) torch stream: its handle is what the C-ABI launches on and what the
    # torch.cuda.Event pairs below are recorded on (the default stream's handle is 0 == "use the
    # context's own stream" in the C-ABI)
    bench_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(bench_stream)
    stream = bench_stream.cuda_stream
    assert stream != 0
    flags = args.flags

    def step():
        ctx.enqueue(dtype, mp, rd, a_blk.data_ptr(), b_use.data_ptr(), c_blk.data_ptr(), n_local, K, m_local,
                    flags=flags, stream=stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.05)
    ctx.set_profiling(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    t_end = time.perf_counter()
    elapsed_ms = ev0.elapsed_time(ev1)
    prep_s, main_s, calls = ctx.profile_read()
    ctx.set_profiling(False)
    clocks = sampler.stop(t_begin, t_end) if sampler else None

    t_max = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t_max.item())
    ms_per_step = elapsed_ms / args.steps
    value = 1e-9 * ops_total / (1e-3 * ms_per_step)  # whole job: all ranks' row-blocks

    # ---- light on-device sanity so that a wrong kernel cannot post a number (not the parity test)
    def check_rows(got_rows, a_rows_t, what, b_t=None):
        ref = a_rows_t.double() @ (b_full if b_t is None else b_t).double()
        if dtype_name == "uint8_t":   # exact: FP64 holds the integer sums (< 2^53); the reference stores them modulo 256
            if not torch.equal(torch.remainder(ref, 256.0), got_rows.double()):
                raise SystemExit("bench.py: %s result check failed (uint8_t rows differ from the exact sums modulo 256)" % what)
            return 0.0
        rel = ((got_rows.double() - ref).abs() / ref.abs().clamp_min(1e-30)).max().item()
        tol = 1e-2 if dtype_name == "half" else 1e-3
        if not (rel <= tol):
            raise SystemExit("bench.py: %s result check failed (max rel err %.3e > %.0e)" % (what, rel, tol))
        return rel

    # (half under MM_FLAG_EXACT accumulates in half like Naive<half>: an FP64 product is not its reference — parity tests are)
    if (mp_name, rd_name) == ("Multiply", "Add") and not (dtype_name == "half" and (flags & 2)):
        rows = torch.tensor([0, n_local // 2, n_local - 1], device=dev)
        extra["check"] = "3 rows of C vs fp64 torch.matmul on device: max rel err %.2e" % check_rows(c_blk[rows], a_blk[rows],
                                                                                                 "device-timed", b_use)
    if args.dump_outputs:   # every rank writes its own block of C
        dump_rows(args.dump_outputs, "c" if world == 1 else "c_rank%d" % rank, c_blk, DUMP_BYTES // world)

    out = None
    if rank == 0:
        peaks = load_peaks()
        path = G.kernel_path(dtype, mp, rd, flags)
        main_avg_s = main_s / max(calls, 1)
        local_ops = 2.0 * n_local * K * m_local
        if path in ("tcgen05_tf32", "tcgen05_f16", "tcgen05_i8"):
            # burst figure when the whole timed region is shorter than the ~1 s it takes the power
            # cap to pull the clocks down, the sustained one for a seconds-long back-to-back loop
            long_run = elapsed_ms > 1500.0
            peak_bf16 = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]) if long_run else peaks["bf16_tflops"]
            peak = {"tcgen05_tf32": peak_bf16 / 2.0, "tcgen05_f16": peak_bf16, "tcgen05_i8": peak_bf16 * 2.0}[path]
            peak_note = ("%s bf16 %s %.1f TF/s%s" % (peaks["_source"], "sustained" if long_run else "burst", peak_bf16,
                         {"tcgen05_tf32": " / 2 (kind::tf32 issues at half the 16-bit rate)", "tcgen05_f16": "",
                          "tcgen05_i8": " x 2 (kind::i8 issues at twice the 16-bit rate; no measured int8 figure in "
                                        "MEASURED_PEAKS.json)"}[path]))
            roof = {"bound": "tensor", "achieved": 1e-12 * local_ops / main_avg_s, "peak": peak, "unit": "TFLOP/s"}
        elif path == "dmma_f64":
            # FP64 DMMA is not in MEASURED_PEAKS.json.  Measured on this pool with a registers-only DMMA loop
            # (scripts/exp_fp64_pipes.cu, profiles/r01_exp_fp64_pipes.jsonl): 37.05-37.13 TF/s at 1965 MHz
            # = 64 FMA/clk/SM; the HGX B200 datasheet's 296 TF / 8 GPUs = 37 TF/s.
            peak = 37.1
            peak_note = ("FP64 tensor (DMMA) 37.1 TF/s: registers-only DMMA loop measured on this pool "
                         "(profiles/r01_exp_fp64_pipes.jsonl); datasheet 37; not in MEASURED_PEAKS.json")
            roof = {"bound": "tensor", "achieved": 1e-12 * local_ops / main_avg_s, "peak": peak, "unit": "TFLOP/s"}
        else:
            peak, peak_note = semiring_peak(dtype_name, mp_name, rd_name, flags)
            roof = {"bound": "cuda_core_issue", "achieved": 1e-12 * local_ops / main_avg_s, "peak": peak, "unit": "TOp/s"}
            if peak == 74.4:
                roof["frac_of_measured_mix"] = roof["achieved"] / 52.5
        roof["frac"] = roof["achieved"] / roof["peak"]
        roof["kernel"] = path
        roof["kernel_ms"] = 1e3 * main_avg_s
        roof["prep_ms"] = 1e3 * prep_s / max(calls, 1)
        roof["prep_note"] = ("exposed operand preparation before the main kernel starts (A's TF32 rounding); B's rounding "
                             "runs concurrently with the GEMM and is inside kernel_ms" if path == "tcgen05_tf32" else "")
        roof["peak_source"] = peak_note
        # DRAM bytes of the dominant kernel: only a figure MEASURED for exactly this workload, GPU count and
        # default tuning (one `ncu --set full` capture per round, profiles/ncu_traffic.json); null otherwise
        roof["algorithmic_bytes"] = es * (n_local * K + K * m_local + n_local * m_local)
        traffic = None
        tr_path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tr_path) and not tune and flags == 0:
            traffic = json.load(open(tr_path)).get("%s@%s@n%d" % (path, args.workload, world))
        roof["traffic"] = traffic
        roof["traffic_ratio"] = (traffic / roof["algorithmic_bytes"]) if traffic else None

        out = {"metric": metric_name, "value": value, "unit": metric, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": {"float": "tf32 tensor-core multiply, f32 accumulate/storage",
                                              "half": "f16 multiply, f32 accumulate", "double": "f64",
                                              "uint8_t": "u8 multiply, s32 accumulate, low byte stored (= the reference's arithmetic modulo 256)"}[dtype_name]
               if (mp_name, rd_name) == ("Multiply", "Add") else "f32",
               "data": "synthetic", "config": config, "clocks": clocks, "roofline": roof,
               # NVML board power during the timed region (the reference's PSU power meter, SURVEY.md 8f)
               "energy": ({"avg_power_w": clocks["power_w_avg_under_load"],
                           "gop_per_joule": value / clocks["power_w_avg_under_load"] / world, "scope": "GPU 0 only"}
                          if clocks and clocks.get("power_w_avg_under_load") else None),
               "gpu_launches": args.steps * G.launch_count(dtype, mp, rd, flags)}
        out.update(extra)
        if tune:
            out["tuning"] = tune

    # ------------------------------------------------------------------ e2e: host buffers through the C-ABI
    # The call a user of the reference makes: ONE blocking MatrixMultiplicationKernel(a, b, c, n, k, m) on host
    # pointers (include/MatrixMultiplication.h:155-171).  Rank 0 issues it for the WHOLE problem; with N > 1 the
    # library splits it over all N GPUs itself (mm_multi_gemm_host: A row-blocks and 1/N of B per GPU over PCIe,
    # B assembled GPU-to-GPU over NVLink, C row-blocks back).  The other ranks wait on the CPU and leave their
    # GPUs idle.
    if not args.no_e2e:
        e2e_steps = max(1, min(args.steps, 3))
        e2e_s = 0.0
        if rank == 0:
            # host matrices: one page-locked array each, its row-blocks placed on the NUMA node of the GPU that copies them
            # (A and C: the GPUs' row-blocks; B: the K-row slices the GPUs upload)
            cuts = [G.multi_partition(world, g, N, K) for g in range(world)]      # the library's own partition rule
            a_np, keep_a, place_a = alloc_host_rows(torch, N, K, np_dt, [(c[0], c[1], g) for g, c in enumerate(cuts)])
            b_np, keep_b, _ = alloc_host_rows(torch, K, M, np_dt, [(c[2], c[3], g) for g, c in enumerate(cuts)])
            c_np, keep_c, _ = alloc_host_rows(torch, N, M, np_dt, [(c[0], c[1], g) for g, c in enumerate(cuts)])
            a_host, b_host, c_host = torch.from_numpy(a_np), torch.from_numpy(b_np), torch.from_numpy(c_np)
            g2 = torch.Generator(device=dev)
            g2.manual_seed(99)
            for i in range(0, N, 2048):   # the other ranks' row-blocks are synthetic too: draw all of A here
                rows_i = min(2048, N - i)
                a_host[i:i + rows_i].copy_(draw((rows_i, K), g2))
            b_host.copy_(b_full)
            torch.cuda.synchronize()
            runner = ctx if world == 1 else G.Multi(world)
            if world > 1:
                runner.set_tuning(**tune)
            runner.gemm_host(dtype, mp, rd, a_np, b_np, N, K, M, flags=flags, out=c_np)  # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                runner.gemm_host(dtype, mp, rd, a_np, b_np, N, K, M, flags=flags, out=c_np)
            e2e_s = (time.perf_counter() - t0) / e2e_steps
            note = ("mm_gemm_host(): page-locked host A, B -> device, kernels, C -> page-locked host; wall clock" if world == 1 else
                    "mm_multi_gemm_host() from rank 0 over all %d GPUs (peer access: %s): per GPU 1/%d of A and of B over "
                    "PCIe, B gathered over NVLink by the library's kernels, C row-blocks back; wall clock"
                    % (world, runner.peer_access, world))
            e2e_check = None
            if (mp_name, rd_name) == ("Multiply", "Add"):
                idx = [0, N // 2 + 1, N - 1]
                e2e_check = check_rows(c_host[idx].to(dev), a_host[idx].to(dev), "e2e")
            out["e2e"] = {"value": 1e-9 * ops_total / e2e_s, "unit": metric,
                          "h2d_bytes_per_step": int(es * (N * K + K * M)), "d2h_bytes_per_step": int(es * N * M),
                          "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s, "note": note, "host_memory": place_a,
                          "check": ("3 rows of the host C vs fp64: max rel err %.2e" % e2e_check) if e2e_check is not None else None}
            if world > 1:
                runner.close()
            if world > 1:
                for arr, keep in ((a_np, keep_a), (b_np, keep_b), (c_np, keep_c)):
                    if keep is not None:
                        torch.cuda.cudart().cudaHostUnregister(arr.ctypes.data)
            del a_host, b_host, c_host
        if world > 1:
            dist.barrier(group=host_group)

    # ------------------------------------------------------------------ cpu_baseline (rank 0, N == 1)
    if out is not None and world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline_line(dtype_name, mp_name, rd_name, metric, K, M,
                                                lambda rows: a_blk[:min(rows, n_local)].cpu().numpy(),
                                                b_full[:, :min(SAMPLE_COLS, M)].cpu().numpy())

    if out is not None:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def semiring_peak(dtype_name, mp_name, rd_name, flags):
    """Derived CUDA-core issue ceiling (DESIGN.md 3.3): one warp instruction per clock and scheduler
    = 148 SMs x 4 x 32 lanes x 1.965 GHz = 37.2e12 lane-instructions/s, 2 ops per element-step.
      float (Add, Min|Max): 1 FADD2 + 1 FMNMX3 per two element-steps = 1.0 slot per step -> 74.4 TOp/s.  MEASURED
        (scripts/exp_pipe_rates.cu, profiles/r02_exp_semiring.md): each of the two instructions alone issues every
        cycle, but their mix needs 1.38 cycles per instruction (1.42 with the kernel's fragment loads): the ceiling this
        instruction mix can reach is 52.5 TOp/s.  `peak` stays the derived 74.4 so that rounds compare; `frac_of_measured_mix`
        is printed beside it.
      anything else (e.g. float (Multiply, Add) under MM_FLAG_EXACT: 1 FMUL2 per two steps + 1 FADD per step):
        1.5 slots per step -> 49.6"""
    fast_minmax = dtype_name == "float" and mp_name == "Add" and rd_name in ("Min", "Max") and not (flags & 2)
    peak = 74.4 if fast_minmax else 49.6
    note = ("derived CUDA-core issue ceiling at 1965 MHz, %s (DESIGN.md 3.3); neither HBM- nor tensor-bound%s"
            % ("1 FADD2 + 1 FMNMX3 per two element-steps" if fast_minmax else "1.5 issue slots per element-step",
               "; measured ceiling of that instruction mix incl. fragment loads: 52.5 TOp/s (profiles/r02_exp_semiring.md)"
               if fast_minmax else ""))
    return peak, note


if __name__ == "__main__":
    sys.exit(main())
