#!/usr/bin/env python
"""bench.py — tasks/sec of the task fan-out hot path on N B200s (contract: DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 1|2|3|4] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch: every pending task of the batch is popped,
deserialised, run through the handler and serialised (one persistent drain kernel per GPU).
Default workload = BASELINE.json configs[1]: 1M x 256-character identity tasks per GPU (weak scaling:
every rank owns its own shard of the pending ring; no data-path collective in the drain).

  value        whole-job tasks/s, batch resident in HBM: W untimed steps, then ONE burst of exactly K timed steps,
               bracketed by a barrier and a synchronise on both sides and timed with CUDA events on the drain stream,
               max over ranks (--sustain-seconds S > 0 repeats the burst until the timed bursts add up to S and takes
               the median burst)
  e2e          the same through the C ABI with HOST buffers: b9_batch_push_async (H2D from pinned memory) + b9_drain (D2H)
  e2e_packed   the same starting from payloads scattered over PAGEABLE memory: b9_batch_push_v (the pack step) + b9_drain
  link         what the host<->device link gives on this box for the e2e byte counts (all ranks at once): e2e's roofline
  roofline     drain kernel: SURVEY.md §8(d) algorithmic bytes / CUDA-event kernel time vs the measured HBM peak
  rebalance    N > 1: skewed ingest (rank 0 holds 2x its share), ONE b9_rebalance (NCCL all-to-all), then the drain
  cpu_baseline the oracle's C port of the reference loop on this box's host cores (rank 0, N = 1), plus the 1-thread rate
               and BASELINE.md's C1 (the Python loop, one process, configs[0])

--dump-outputs DIR writes the records the last timed step handed back (rank 0; with --impl reference, the C port's)
as DIR/<name>.npy, see dump_outputs(). The inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
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

L2_BYTES = 126e6
CONFIGS = {   # BASELINE.json configs[i] -> (handler, total tasks quoted, the GPU count it is quoted on)
    1: ("identity", 1_000_000, 1),
    2: ("crc32", 1_000_000, 1),
    3: ("vadd_f32", 10_000_000, 8),
    4: ("json_sum", 100_000, 4),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS), help="BASELINE.json configs[i]; 1 = the metric's configuration")
    ap.add_argument("--tasks", type=int, default=0, help="tasks per GPU per step (default: the config's total / its GPU count)")
    ap.add_argument("--chars", type=int, default=256)
    ap.add_argument("--handler", default="", help="override the config's handler")
    ap.add_argument("--e2e-steps", type=int, default=120, help="steps of the end-to-end legs (about a second of timed region at one GPU)")
    ap.add_argument("--sustain-seconds", type=float, default=0.0,
                    help="0: one burst of K timed steps; S > 0: bursts of K steps are repeated until their timed regions add up to S")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cancelled", type=float, default=0.0, help="fraction of the resident tasks pushed with B9_TF_CANCELLED")
    ap.add_argument("--skew", type=float, default=1.0, help="N>1 rebalance leg: rank 0 ingests (1+skew)x its fair share; 0 = no rebalance leg")
    ap.add_argument("--adversarial", type=float, default=0.01, help="share of tasks whose string needs escaping (SURVEY.md §8d: 1 %%)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write the last timed step's records to DIR/<name>.npy")
    a = ap.parse_args()
    h, total, g = CONFIGS[a.config]
    if not a.handler:
        a.handler = h
    if not a.tasks:
        a.tasks = total // g
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def usable_cores() -> int:
    """Threads this process can really run at once: the scheduler affinity, capped by the cgroup CPU quota
    (os.cpu_count() reports the machine; a container with a quota of 8 CPUs on a 128-core host loses throughput
    when 128 threads are started)."""
    n = len(os.sched_getaffinity(0))
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def bind_to_gpu_numa_node(local_rank: int) -> str:
    """Run this rank on the CPUs next to its GPU (NVML's ideal affinity), BEFORE any pinned buffer is
    allocated: page-locked memory lands on the allocating thread's NUMA node, and a host<->device copy
    that crosses sockets is slower — it matters for the end-to-end number when 8 ranks share one host."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus near gpu {local_rank}"
    except Exception as e:                      # no NVML / no permission: keep the inherited affinity
        return f"unchanged ({type(e).__name__})"
    return "unchanged"


def kernel_source_hash(handler_index: int = 0) -> str:
    """Identity of a drain kernel of THIS build: sha256 over the SASS of `drain3_kernel<handler_index>` in the library the
    bench loads (cuobjdump; host-side edits of the library and changes to the other handlers' kernels do not change it,
    any change of this kernel does). Falls back to the CUDA sources' text when cuobjdump is missing. Stamps
    profiles/ncu_traffic.json entries."""
    so = os.environ.get("B9GPU_LIB") or os.path.join(ROOT, "beta9_b200", "libb9gpu.so")
    try:
        txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, timeout=120, check=True).stdout
        h = hashlib.sha256()
        found = 0
        for part in txt.split("Function : ")[1:]:
            if f"drain3_kernelILi{handler_index}E" not in part.split("\n", 1)[0]:
                continue
            found += 1
            for ln in part.split("\n"):
                ln = ln.strip()
                if ln.startswith("/*") and ";" in ln:                      # an instruction line (not its encoding word)
                    h.update(ln.split("*/", 1)[1].split(";")[0].strip().encode()); h.update(b"\n")
        if found:
            return "sass:" + h.hexdigest()[:16]
    except Exception:                                                       # noqa: BLE001
        pass
    h = hashlib.sha256()
    d = os.path.join(ROOT, "beta9_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return "src:" + h.hexdigest()[:16]


def workload_key(args, n_tasks) -> str:
    return f"{args.handler}:{n_tasks}:{args.chars}:{args.adversarial}" if args.handler == "identity" else f"{args.handler}:{n_tasks}"


def ncu_traffic(args, n_tasks):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of this workload's drain kernel, from the committed ncu
    capture of the same command (profiles/ncu_traffic.json, written by scripts/ncu_traffic.py on a GPU box). An entry is
    used only if it was captured from the kernel sources of THIS build (src_hash); otherwise (traffic: null, why)."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except (OSError, ValueError):
        return None, "no profiles/ncu_traffic.json"
    e = table.get(workload_key(args, n_tasks))
    if e is None:
        return None, "no capture of this workload"
    mine = kernel_source_hash()
    if e.get("src_hash") != mine:
        return None, f"stale capture (kernels {e.get('src_hash')} != {mine})"
    return e.get("dram_bytes"), f"ncu --set full, {e.get('captured', '?')}, kernels {e.get('src_hash')}"


def workload(args, rank, n=None):
    from beta9_b200 import synth
    n = args.tasks if n is None else n
    if n <= 0:                                # (the skewed leg at N = 2 leaves rank 1 with nothing to ingest)
        return synth.Batch(np.zeros((0, 16), np.uint8), np.zeros(0, np.uint8), np.zeros(1, np.uint64), "empty")
    if args.handler == "identity":
        return synth.strings_batch(n, args.chars, adversarial_frac=args.adversarial, seed=synth.SEED + 1000 * rank)
    if args.handler == "crc32":          # configs[2]: zipf 32..4096-char strings
        return synth.crc_batch(n, seed=synth.SEED + 1000 * rank)
    if args.handler == "vadd_f32":       # configs[3] payload shape: 2 x 32 fp32 as base64
        return synth.vadd_batch(n, seed=synth.SEED + 1000 * rank)
    if args.handler == "json_sum":       # configs[4] payload shape: 1 KB JSON documents
        return synth.json_batch(n, seed=synth.SEED + 1000 * rank)
    raise SystemExit(f"bench: unknown handler {args.handler}")


def workload_name(args, n) -> str:
    if args.handler == "identity":
        return f"configs[{args.config}]: {n} x {args.chars}-char identity tasks per GPU ({100 * args.adversarial:g}% adversarial escapes)"
    return f"configs[{args.config}]: {args.handler}, {n} tasks per GPU"


DUMP_SEED = 20261017
DUMP_RECORDS = 1 << 15
DUMP_LIMIT_BYTES = 60_000_000        # the data of all files; their headers add well under a kilobyte


def dump_outputs(out_dir, task_ids, status, has_result, starts, lengths, blob) -> None:
    """--dump-outputs: records of one step, in record (= task) order, as .npy files in out_dir. A fixed, seeded sample of
    DUMP_RECORDS records (fewer when their result bytes would take the files past DUMP_LIMIT_BYTES):
      record_index [k] float64, task_ids [k, 16], status [k], has_result [k], lengths [k]   float32
      result_bytes [sum of lengths] float32: the sampled records' result bytes one after the other
    Record i's bytes are blob[starts[i] : starts[i] + lengths[i]]. Where they sit in the device's blob follows the order in
    which tiles finished, so those offsets are not written: only what they point at."""
    n = int(status.shape[0])
    idx = np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_RECORDS), replace=False)      # in random order
    keep = int(np.searchsorted(np.cumsum(8 + 4 * (16 + 3) + 4 * lengths[idx].astype(np.int64)), DUMP_LIMIT_BYTES, side="right"))
    idx = np.sort(idx[:keep])
    ln = lengths[idx].astype(np.int64)
    ends = np.cumsum(ln)
    rec = np.repeat(np.arange(keep, dtype=np.int64), ln)
    src = np.asarray(starts, dtype=np.int64)[idx][rec] + (np.arange(int(ends[-1]) if keep else 0, dtype=np.int64) - (ends - ln)[rec])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("record_index", idx.astype(np.float64)), ("task_ids", np.asarray(task_ids)[idx].astype(np.float32)),
                    ("status", status[idx].astype(np.float32)), ("has_result", has_result[idx].astype(np.float32)),
                    ("lengths", ln.astype(np.float32)), ("result_bytes", blob[src].astype(np.float32))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    """--impl reference: the reference's CPU task loop on this box's host cores. The Go gateway and
    the Python runner cannot be built/imported here (no Go toolchain, SDK deps missing), so this is
    the oracle's C port of that loop (oracle/c/b9_oracle.c), multi-threaded over the cores this process may
    use; Redis, Postgres, gRPC and the object store are left out, which flatters the reference."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    from oracle import coracle
    batch = workload(args, 0)
    cores = usable_cores()
    times = []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        o = coracle.run_batch(batch.task_ids, batch.payload, batch.offsets, args.handler, nthreads=cores,
                              out_cap=int(batch.payload.size) + 64)
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, batch.task_ids, o.status, o.has, o.offsets[:-1], np.diff(o.offsets), o.payload)
    total = sum(times)
    v = batch.n * len(times) / total
    # the same loop on ONE thread (a bounded sample): what the port does per core, and how it scales
    sample = batch.slice(0, min(batch.n, 100_000))
    t0 = time.perf_counter()
    coracle.run_batch(sample.task_ids, sample.payload, sample.offsets, args.handler, nthreads=1, out_cap=int(sample.payload.size) + 64)
    v1 = sample.n / (time.perf_counter() - t0)
    line = {
        "impl": "reference", "metric": "tasks_per_sec", "value": v, "unit": "tasks/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8" if args.handler != "vadd_f32" else "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, batch.n) + ", resident in HBM", "handler": args.handler, "tasks_per_gpu": batch.n,
                   "arm": "reference CPU loop (C port of the Go + Python path), one bounded sample of the per-GPU batch per step"},
        "cpu_baseline": {"value": v, "unit": "tasks/s", "cores": cores, "kind": "port",
                         "sample": f"{batch.n} tasks x {len(times)} steps, {cores} threads (sched affinity capped by the cgroup quota; os.cpu_count() = {os.cpu_count()})",
                         "one_thread": v1, "scaling_vs_one_thread": v / v1},
        "e2e": {"value": v, "unit": "tasks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_REAL_STDOUT = None


def _own_stdout():
    """stdout carries exactly ONE line, the JSON result: everything else a library prints there (NCCL's
    version banner, for one) is sent to stderr by pointing fd 1 at fd 2 for the lifetime of the run."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def link_ceiling(torch, h2d_bytes: int, d2h_bytes: int, barrier, reduce_max, reps: int = 5):
    """What the host<->device link gives for one e2e step's byte counts: both directions at once from / to pinned memory on
    two streams, every rank at the same time (they share the host's memory and PCIe root complexes). Plain cudaMemcpyAsync
    through torch — no library code: this is e2e's roofline, not a product path."""
    hin = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
    hout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
    din = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8, device="cuda")
    dout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    best = None
    for r in range(reps + 1):
        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s2):
            hout.copy_(dout, non_blocking=True)
        s1.synchronize(); s2.synchronize()
        dt = reduce_max(time.perf_counter() - t0)
        if r:
            best = dt if best is None else min(best, dt)
    del hin, hout, din, dout
    return best


def main():
    args = parse_args()
    _own_stdout()
    if args.impl == "reference":
        return run_reference(args)
    rank, local_rank, world = dist_env()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the b200 arm has no CPU path")
    torch.cuda.set_device(local_rank)
    affinity = (bind_to_gpu_numa_node(local_rank) if world > 1 and not os.environ.get("B9_BENCH_NO_AFFINITY")
                else "inherited")
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from beta9_b200 import _lib as L
    from beta9_b200.device_queue import DeviceQueue
    batch = workload(args, rank)
    n = batch.n
    in_bytes = int(batch.payload.size)
    dq = DeviceQueue(device=local_rank, ring_bytes=max(1 << 30, 4 * in_bytes), ring_tasks=max(1 << 21, 4 * n),
                     max_drain_tasks=max(1 << 21, 2 * n), max_result_bytes=max(1 << 30, 3 * in_bytes))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ------------------------------------------------------------------ device-resident steps
    n_cancelled = 0
    if args.cancelled > 0:
        fl = (np.random.default_rng(5 + rank).random(batch.n) < args.cancelled).astype(np.uint8)
        n_cancelled = int(fl.sum())
        dq.push_batch(batch.task_ids, batch.payload, batch.offsets, flags=fl)
    else:
        dq.push_batch(batch.task_ids, batch.payload, batch.offsets)
    n_total = int(round(reduce_sum(float(n))))
    for _ in range(args.warmup):
        dq.drain_launch(args.handler, n, peek=True)
    sampler = ClockSampler(local_rank)
    launches0 = dq.stats().kernel_launches
    barrier()
    sampler.start()
    # a burst of EXACTLY K steps: the K launches are enqueued back to back (B9_DRAIN_ASYNC), as a host that pipelines its
    # drains would; a barrier + synchronise brackets every burst; the device time of a burst comes from CUDA events on
    # the drain stream (first step's start -> last step's end), the max over ranks is the burst's time. One burst unless
    # --sustain-seconds asks for more.
    burst_dev, burst_wall = [], []
    timed_total = 0.0
    launches_per_burst = None
    while True:
        k0 = dq.stats().kernel_launches
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            got = dq.drain_launch(args.handler, n, peek=True, wait=False)
        dq.sync()
        dev_s = float(dq.stats().last_drain_kernel_ms) * 1e-3
        barrier()
        wall_s = time.perf_counter() - t0
        assert got == n, (got, n)
        launches_per_burst = dq.stats().kernel_launches - k0
        d = reduce_max(dev_s)
        burst_dev.append(d); burst_wall.append(reduce_max(wall_s))
        timed_total += d
        if timed_total >= args.sustain_seconds or len(burst_dev) >= 2000:
            break
    clocks = sampler.stop()
    launches = dq.stats().kernel_launches - launches0
    if args.dump_outputs and rank == 0:
        last = dq.fetch()                            # the last timed step's records (peek: the batch stays resident)
        dump_outputs(args.dump_outputs, last.task_ids, last.status, last.has_result, last.offsets, last.lengths, last.payload)
        del last
    elapsed = statistics.median(burst_dev)
    wall_elapsed = statistics.median(burst_wall)
    value = n_total * args.steps / elapsed
    k_ms = 1e3 * elapsed / args.steps                # device time per timed step (back to back: the gaps between launches count)
    # drop the resident batch; its records are the reference records of the legs below
    dq.drain_launch(args.handler, n, peek=False)
    res = dq.fetch()
    assert res.n == n - n_cancelled, (res.n, n, n_cancelled)
    assert dq.depth() == 0
    if n_cancelled:
        dq.push_batch(batch.task_ids, batch.payload, batch.offsets)
        res = dq.drain(args.handler, n)
    out_bytes = int(res.lengths.astype(np.int64).sum())      # result bytes proper (the blob also holds <= 15 B of padding per tile)
    blob_bytes = int(res.payload.size)

    # ------------------------------------------------------------------ end to end through the C ABI, host buffers
    # Every step copies that step's inputs host->device from pinned memory and reads that step's result
    # records back device->host. Steps are pipelined the way a gateway would run them: one thread pushes
    # (b9_batch_push_async), one drains, so H2D(k+1) overlaps the kernel and D2H(k) on the full-duplex link.
    # Two input buffer sets alternate; results land in one pinned set.
    pins = []
    for _ in range(2):
        pi = dq.pinned(n * 16); pp = dq.pinned(in_bytes); po = dq.pinned((n + 1) * 8)
        pi.array[:] = batch.task_ids.reshape(-1); pp.array[:] = batch.payload
        po.view(np.uint64, n + 1)[:] = batch.offsets
        pins.append((pi, pp, po))
    cap_bytes = blob_bytes + 4096
    o_ids = dq.pinned(n * 16); o_st = dq.pinned(n); o_has = dq.pinned(n); o_off = dq.pinned(n * 8); o_len = dq.pinned(n * 4); o_pl = dq.pinned(cap_bytes)
    resbuf = L.Results(o_ids.ptr, o_st.ptr, o_has.ptr, o_off.ptr, o_len.ptr, o_pl.ptr, n, cap_bytes, 0, 0, 0, 0, 0.0, 0)
    lib = L.load()
    hid = {"identity": 0, "crc32": 1, "vadd_f32": 2, "json_sum": 3}[args.handler]

    def e2e_push(k):
        pi, pp, po = pins[k & 1]
        rc = lib.b9_batch_push_async(dq._ctx, pi.ptr, pp.ptr, po.ptr, n, None)
        if rc != 0:
            raise SystemExit("push failed: " + L.last_error())

    def e2e_drain():
        r = lib.b9_drain(dq._ctx, hid, n, C.byref(resbuf))
        if r != n:
            raise SystemExit(f"drain returned {r}: " + L.last_error())

    def e2e_run(steps, push):
        # a producer thread pushes, this thread drains — one goroutine per side in the gateway; the library runs the two
        # sides concurrently (INTEGRATION.md §1), so the host-side work of push k+1 (index validation, ring placement) is
        # off the drain's critical path and both DMA directions stay busy. At most two batches are in the ring: buffer
        # set k & 1 is reused only after batch k - 2 has been drained.
        room, ready, err = threading.Semaphore(2), threading.Semaphore(0), []

        def producer():
            try:
                for k in range(steps):
                    room.acquire()
                    push(k)
                    ready.release()
            except BaseException as e:          # noqa: BLE001
                err.append(e); ready.release()
        th = threading.Thread(target=producer, daemon=True)
        th.start()
        for k in range(steps):
            ready.acquire()
            if err:
                raise SystemExit(f"push failed: {err[0]}")
            e2e_drain()
            room.release()
        th.join()

    def check_records():            # the records that came back are the real ones
        e_off = o_off.view(np.uint64, n); e_len = o_len.view(np.uint32, n)
        for i in (0, n // 2, n - 1):
            assert bytes(o_pl.array[int(e_off[i]):int(e_off[i]) + int(e_len[i])]) == res.result(i)

    e2e_run(3, e2e_push)
    s0 = dq.stats()
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.e2e_steps, e2e_push)
    barrier()
    t1 = time.perf_counter()
    s1 = dq.stats()
    e2e_elapsed = reduce_max(t1 - t0)
    e2e_value = n_total * args.e2e_steps / e2e_elapsed
    h2d = (s1.bytes_h2d - s0.bytes_h2d) // args.e2e_steps
    d2h = (s1.bytes_d2h - s0.bytes_d2h) // args.e2e_steps
    check_records()

    # ------------------------------------------------------------------ ... and from scattered pageable payloads: the pack step
    # What a Go gateway holds is [][]byte: n separate payloads somewhere in pageable memory. Here they sit in one pageable
    # blob in a random order (so the gather is a gather); b9_batch_push_v packs them into the context's pinned arenas with
    # its own threads and pushes the arena; the pack of step k+1 runs while step k's DMA, kernel and read-back are in flight.
    lens32 = np.diff(batch.offsets).astype(np.uint32)
    perm = np.random.default_rng(17 + rank).permutation(n)
    where = np.zeros(n, np.uint64)
    where[perm] = np.concatenate([[0], np.cumsum(lens32[perm].astype(np.uint64))[:-1]])
    src_rec = np.repeat(np.arange(n, dtype=np.int64), lens32.astype(np.int64))
    starts = np.asarray(batch.offsets[:-1], dtype=np.int64)
    within = np.arange(in_bytes, dtype=np.int64) - starts[src_rec]
    blob = np.empty(in_bytes + 1, np.uint8)
    blob[where.astype(np.int64)[src_rec] + within] = batch.payload
    del src_rec, within
    ptrs = (np.uint64(blob.ctypes.data) + where).astype(np.uint64)
    ids_pageable = np.ascontiguousarray(batch.task_ids).copy()

    def packed_push(k):
        rc = lib.b9_batch_push_v(dq._ctx, ids_pageable.ctypes.data, ptrs.ctypes.data, lens32.ctypes.data, n, None)
        if rc != 0:
            raise SystemExit("push_v failed: " + L.last_error())

    def packed_run(steps):
        e2e_run(steps, packed_push)             # the producer thread packs + pushes (b9_batch_push_v), this thread drains

    packed_run(3)
    barrier()
    t0 = time.perf_counter()
    packed_run(args.e2e_steps)
    barrier()
    packed_elapsed = reduce_max(time.perf_counter() - t0)
    packed_value = n_total * args.e2e_steps / packed_elapsed
    check_records()
    pack_threads = int(os.environ.get("B9_PACK_THREADS", min(16, os.cpu_count() or 1)))

    # ------------------------------------------------------------------ the link's own ceiling for these byte counts
    link_s = link_ceiling(torch, int(h2d), int(d2h), barrier, reduce_max)
    link = {"seconds_per_step": link_s, "h2d_GBps_per_gpu": h2d / link_s / 1e9, "d2h_GBps_per_gpu": d2h / link_s / 1e9,
            "tasks_per_sec": n_total / link_s, "how": "cudaMemcpyAsync H2D + D2H of one step's bytes at once, pinned memory, two streams, all ranks together, best of 5"}

    # ------------------------------------------------------------------ N > 1: skewed ingest -> ONE NCCL rebalance -> drain
    rebalance_info = None
    if world > 1 and args.skew > 0:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(DeviceQueue.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        dq.comm_init(bytes(idt.cpu().numpy().tobytes()), rank, world)
        # the job's total stays N x n; rank 0 ingests (1 + skew) x n, the other ranks share the rest evenly
        n0 = int(n * (1 + args.skew))
        n_mine = n0 if rank == 0 else (n * world - n0) // (world - 1)
        sk = workload(args, rank, n_mine) if n_mine != n else batch
        total_in = int(round(reduce_sum(float(sk.n))))
        ms, moved, after = [], 0.0, 0
        for rep in range(4):
            dq.push_batch(sk.task_ids, sk.payload, sk.offsets)
            barrier()
            r0 = time.perf_counter()
            info = dq.rebalance()
            torch.cuda.synchronize()
            r_local = time.perf_counter() - r0
            barrier()
            if rep:                                       # the first exchange also sizes the arenas
                ms.append(1e3 * reduce_max(r_local))
            moved = reduce_sum(float(info.bytes_sent))
            after = dq.depth()
            dq.drain_launch(args.handler, after, peek=False)             # the drain after the exchange: every task exactly once
            r = dq.fetch()
            total_after = int(round(reduce_sum(float(r.n_popped))))
            assert total_after == total_in, (total_after, total_in)
        r_ms = statistics.median(ms)
        share = reduce_max(float(after)) / (total_in / world)
        rebalance_info = {"ms": r_ms, "ms_all": ms, "skew": args.skew, "tasks_rank0_before": n0, "tasks_per_rank_fair": total_in // world,
                          "max_share_after": share, "bytes_moved_total": moved, "GBps_total": moved / (r_ms * 1e-3) / 1e9,
                          "how": "wall clock of b9_rebalance (all-gather of counts, plan, grouped ncclSend/ncclRecv, ring append) "
                                 "between barriers, max over ranks, median of 3 after one warm-up exchange"}

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import coracle
        cores = usable_cores()
        best = None
        for _ in range(3):
            c0 = time.perf_counter()
            o = coracle.run_batch(batch.task_ids, batch.payload, batch.offsets, args.handler, nthreads=cores, out_cap=in_bytes + 64)
            dt = time.perf_counter() - c0
            best = dt if best is None else min(best, dt)
        # while we are here: the device answers are the oracle's answers
        assert np.array_equal(o.payload, res.fifo_payload()) and np.array_equal(o.status, res.status)
        sample = batch.slice(0, min(n, 100_000))
        c0 = time.perf_counter()
        coracle.run_batch(sample.task_ids, sample.payload, sample.offsets, args.handler, nthreads=1, out_cap=int(sample.payload.size) + 64)
        v1 = sample.n / (time.perf_counter() - c0)
        # BASELINE.md §2 C1 / §3 row 1: configs[0] (10k x 64-char echo) through the Python loop, one process (= reference workers=1)
        from beta9_b200 import synth
        from oracle.pyoracle.loop import run_task_loop
        echo = synth.strings_batch(10_000, 64)
        c0 = time.perf_counter()
        run_task_loop(echo.tasks(), [bytes(t) for t in echo.task_ids], "identity")
        c1 = echo.n / (time.perf_counter() - c0)
        cpu = {"value": n / best, "unit": "tasks/s", "cores": cores, "kind": "port",
               "sample": f"all {n} tasks of the step, best of 3 passes, {cores} threads (oracle/c/b9_oracle.c; os.cpu_count() = {os.cpu_count()})",
               "one_thread": v1, "scaling_vs_one_thread": (n / best) / v1,
               "c1_python_one_process_configs0": c1}

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        if os.path.exists(peaks_path):
            peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)"
        if args.handler == "identity" and args.chars == 256 and args.adversarial <= 0.01:
            algo = 578.0 * n        # SURVEY.md §8(d): 256 in + 258 out + 2 x 32 B of index/id/header
        else:   # SURVEY.md §8(d): argument bytes as carried + result bytes + 2 x 32 B of index/id/header per task
            algo = float(in_bytes - 28 * n + out_bytes + 64 * n)
        achieved = algo / (k_ms * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic(args, n)
        line = {
            "metric": "tasks_per_sec", "value": value, "unit": "tasks/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps, "wall_ms_per_step": 1e3 * wall_elapsed / args.steps,
            "timing": {"bursts": len(burst_dev), "steps_per_burst": args.steps, "timed_steps": len(burst_dev) * args.steps,
                       "timed_seconds": timed_total,
                       "burst_ms_min_median_max": [1e3 * min(burst_dev), 1e3 * elapsed, 1e3 * max(burst_dev)],
                       "how": "every burst = exactly K steps enqueued back to back (B9_DRAIN_ASYNC), CUDA events on the drain stream, "
                              "barrier + synchronise on both sides, max over ranks; one burst unless --sustain-seconds > 0, then value "
                              "uses the median burst; wall_ms_per_step = host clock over the median burst, barriers included"},
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8" if args.handler != "vadd_f32" else "f32", "data": "synthetic",
            "config": {"workload": workload_name(args, n) + ", resident in HBM",
                       "handler": args.handler, "tasks_per_gpu": n,
                       "parallelism": f"shard{world}" if world > 1 else "single",
                       "cpu_affinity": affinity, "cancelled_tasks_per_gpu": n_cancelled,
                       "l2": f"inputs {in_bytes / 1e6:.0f} MB + outputs {out_bytes / 1e6:.0f} MB per step exceed the 126 MB L2; no flush needed"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": f"b9::drain3_kernel<{args.handler}>",
                         "kernel_ms": k_ms, "kernel_ms_how": "device time of the median burst / K",
                         "algorithmic_bytes_per_task": algo / n, "peak_source": peak_src},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "tasks/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": args.e2e_steps, "ms_per_step": 1e3 * e2e_elapsed / args.e2e_steps,
                    "frac_of_link": e2e_value / link["tasks_per_sec"],
                    "api": "b9_batch_push_async on a producer thread + b9_drain on the main thread, pinned host buffers, at most two batches in the ring"},
            "e2e_packed": {"value": packed_value, "unit": "tasks/s", "ms_per_step": 1e3 * packed_elapsed / args.e2e_steps,
                           "pack_threads": pack_threads, "frac_of_link": packed_value / link["tasks_per_sec"],
                           "api": "b9_batch_push_v (payloads scattered over pageable memory, gathered into pinned arenas by the library) on a producer thread + b9_drain on the main thread"},
            "link": link,
            "gpu_launches": int(launches),
            "gpu_launches_per_burst": int(launches_per_burst),
            "rebalance": rebalance_info,
            "clocks": clocks,
        }
        emit(line)
    for p in [x for t in pins for x in t] + [o_ids, o_st, o_has, o_off, o_len, o_pl]:
        p.free()
    dq.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException as e:      # a rank that fails must not leave its peers waiting in a collective until some outer timeout
        if isinstance(e, SystemExit) and e.code in (0, None):
            raise
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
