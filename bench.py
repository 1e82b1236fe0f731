#!/usr/bin/env python
"""bench.py -- mash.Sketch throughput on B200 (BASELINE.json metric) and the rest of SURVEY.md 8d.

A "step" is one pass of the Sketch hot path over one batch of synthetic reads:
BASELINE configs[1] = 10 M x 150 bp reads, k=21, sketchSize=1000 per GPU (reads are
independent, so N GPUs sketch N x 10 M reads with no data-path collective: weak scaling;
N=8 is configs[3], 80 M reads).

  value      whole-job Gbases/s with the reads resident in HBM (CUDA events, max over ranks)
  e2e        the same metric through the reference-facing C ABI call with HOST buffers
             (pg_mash_sketch_uniform: H2D of the reads, kernels, D2H of the sketches); each rank's
             thread and pinned buffers are bound to its GPU's NUMA node (pg_numa_bind_thread).
             e2e_variants (N=1): pageable buffers, and the shape a Go caller gets (one zero-filled
             4*s-byte Sketches array per read, pageable); host_bw: bare cudaMemcpyAsync D2H / H2D
             from the same pinned buffers, all ranks at once -- the platform cap of e2e
  roofline   algorithmic bytes (L + 4*min(L-k, s) per read, SURVEY 8d) / kernel time vs the
             measured HBM copy peak (MEASURED_PEAKS.json)
  cpu_baseline  C restatement of the Go algorithm (oracle/, "port") on the host cores; thread
             count = best of a small sweep bounded by the schedulable cores (affinity, cgroup quota)
  secondary  (N=1) configs[2] and configs[4] on this GPU: cfg3 sketch (K2), cfg3 all-pairs (K3),
             cfg5 Smith-Waterman (K4) and Tm (K5), each with a parity bit against the oracle on a
             sample and its own CPU baseline
  pipeline   (N>1) the exchange north_star names: cfg4 shape (sketch -> all-gather of the sketches
             -> capped row-block distance) with the all-gather FUSED into the sketch kernel (peer
             stores over NVLink) next to K1 + ncclAllGather, and cfg3 sharded over the ranks (sketch ->
             gather -> row-block all-pairs); in-run assertions: fused == NCCL, and a sample of every
             rank's gathered buffer == the oracle

`--impl reference` times the CPU restatement alone (the Go reference cannot run here:
no Go toolchain, see DESIGN.md) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # oracle_ffi: only the cpu_baseline / parity legs import it

READ_LEN, KMER, SKETCH = 150, 21, 1000
NK = READ_LEN - KMER  # 129 informative words per read
BYTES_PER_READ = READ_LEN + 4 * min(NK, SKETCH)  # 666 (SURVEY 8d)
METRIC = "mash.Sketch Gbases/s"
NVLINK_PEER_PEAK_GBS = 770.0  # measured peer-copy bandwidth per direction, B200_PROFILING.md
DUMP_ROWS = 32768  # --dump-outputs: 32768 x 129 float64 = 34 MB, under 64 MB whatever the world size


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 5)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned: a fixed seeded sample of "
                         f"{DUMP_ROWS} rows of the [reads][{NK}] uint32 sketch array as DIR/sketches.npy (float64, "
                         "every uint32 exact) and the read index of each row as DIR/read_index.npy; under torchrun "
                         "every rank writes its share with a _rank<r> suffix")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.t_load = self.t0 = self.t1 = None  # load start (warm-up), timed region start / end

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        # samples inside the timed region; a region shorter than a few sampling periods falls
        # back to the whole loaded window (warm-up + timed), and says so
        rows = [r for (t, r) in self.rows if self.t0 is not None and self.t0 <= t <= self.t1]
        window = "timed region"
        if len(rows) < 3 and self.t_load is not None:
            rows = [r for (t, r) in self.rows if self.t_load <= t <= self.t1 + 0.05]
            window = "warm-up + timed region (timed region shorter than 3 sampling periods)"
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


# ---- host CPU arm -------------------------------------------------------------------------------
def schedulable_cores() -> int:
    """Cores this process can actually run on: the affinity mask, further capped by a cgroup CPU
    quota (os.cpu_count() reports the machine, not the lease -- the round-1 CPU arm swung 5x between
    boxes because it started 128 threads on a handful of schedulable cores)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def _thread_candidates(cores: int):
    c = sorted({max(1, cores // 4), max(1, cores // 2), cores})
    return c


def _cpu_sample(threads: int, budget_s: float, cap_reads: int = 2_000_000):
    """Choose a sample of the cfg2 workload that the C restatement sketches in ~budget_s seconds
    on `threads` host threads, and generate it ONCE (numpy generation is slower than hashing)."""
    import oracle_ffi
    from poly_b200 import synth

    probe = min(cap_reads, 10_000 * threads)
    reads = synth.independent_reads(probe, READ_LEN)
    off = synth.uniform_offsets(probe, READ_LEN)
    oracle_ffi.sketch_batch_timing(reads[: 1000 * READ_LEN], off[:1001], KMER, SKETCH, 0, threads)  # thread start-up
    t0 = time.perf_counter()
    oracle_ffi.sketch_batch_timing(reads, off, KMER, SKETCH, 0, threads)
    rate = probe / (time.perf_counter() - t0)
    n = int(min(max(rate * budget_s, probe), cap_reads))
    if n > probe:
        reads = synth.independent_reads(n, READ_LEN)
        off = synth.uniform_offsets(n, READ_LEN)
    return reads, off, n


def _cpu_time(reads, off, n, threads: int):
    """One timed pass of the C restatement of mash.go:59-104 (faithful variant: one zeroed
    4*s-byte sketch per read as mash.New does, full re-sort on qualifying insert; static
    parallel-for over reads).  bench.py executes oracle/ only in its CPU legs and parity checks."""
    import oracle_ffi

    t0 = time.perf_counter()
    rc, _ = oracle_ffi.sketch_batch_timing(reads, off, KMER, SKETCH, 0, threads)
    dt = time.perf_counter() - t0
    assert rc == 0
    return dt


def _best_threads(reads, off, n, cores: int):
    """Small sweep: the thread count (<= schedulable cores) with the best rate on this box."""
    sweep = {}
    for t in _thread_candidates(cores):
        m = min(n, max(20_000, n // 4))
        sweep[t] = m * READ_LEN / _cpu_time(reads[: m * READ_LEN], off[: m + 1], m, t) / 1e9
    best = max(sweep, key=sweep.get)
    return best, {str(k): round(v, 4) for k, v in sweep.items()}


def _cpu_desc(n, threads, dt, value, cores, sweep):
    return {"value": value, "unit": "Gbases/s", "cores": threads, "kind": "port", "schedulable_cores": cores,
            "thread_sweep_gbases_per_s": sweep,
            "sample": f"first {n} reads of the 10M x 150bp k=21 s=1000 workload per step; C restatement of the Go algorithm "
                      f"(mash.go:59-104, not Go: no Go toolchain here), static parallel-for over reads on {threads} threads "
                      f"(best of the sweep; {cores} schedulable cores), {dt:.2f} s per step"}


def cpu_reference_leg(budget_s: float):
    cores = schedulable_cores()
    reads, off, n = _cpu_sample(cores, budget_s)
    threads, sweep = _best_threads(reads, off, n, cores)
    dt = min(_cpu_time(reads, off, n, threads) for _ in range(2))
    return _cpu_desc(n, threads, dt, n * READ_LEN / dt / 1e9, cores, sweep), n, dt


def run_reference(args, rank: int, world: int):
    """`--impl reference`: the reference's own CPU implementation of the path.  The Go code
    cannot run here, so this is its C restatement on the schedulable host threads; each step is one
    pass over a bounded sample of the cfg2 workload (same metric / unit / config as our arm)."""
    if rank != 0:
        return
    cores = schedulable_cores()
    steps = args.steps + args.warmup
    reads, off, n = _cpu_sample(cores, max(0.3, min(4.0, 100.0 / max(steps, 1))))
    threads, sweep = _best_threads(reads, off, n, cores)
    times = [_cpu_time(reads, off, n, threads) for _ in range(steps)][args.warmup:]
    tot_t = sum(times)
    value = n * len(times) * READ_LEN / tot_t / 1e9
    sample = _cpu_desc(n, threads, tot_t / len(times), value, cores, sweep)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Gbases/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "configs[1]: 10M x 150bp short reads, k=21, sketchSize=1000 (bounded sample per step)",
                   "reads_per_step": n, "read_len": READ_LEN, "k": KMER, "sketch_size": SKETCH},
        "cpu_baseline": sample,
        "e2e": {"value": value, "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---- helpers shared by the GPU legs ---------------------------------------------------------------
class Ctx:
    pass


def ev_time(fn, iters=1, warm=0):
    """CUDA-event time (ms per iteration) of fn on torch's current stream."""
    import torch

    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    for _ in range(iters):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, out


def max_over_ranks(cx, v: float) -> float:
    import torch
    import torch.distributed as dist

    if cx.world == 1:
        return v
    t = torch.tensor([v], dtype=torch.float64, device=cx.dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def all_true(cx, ok: bool) -> bool:
    import torch
    import torch.distributed as dist

    if cx.world == 1:
        return bool(ok)
    t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=cx.dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


def barrier(cx):
    import torch
    import torch.distributed as dist

    if cx.world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def dump_outputs(cx, d_out, out_dir):
    """--dump-outputs: the same rows of the headline step's result on every run with the same --reads
    (the inputs are counter-based, the sample is seeded), so that two builds can be compared output for output."""
    import numpy as np
    import torch

    m = min(cx.n, DUMP_ROWS // cx.world)
    rows = np.sort(np.random.default_rng(0).choice(cx.n, m, replace=False))
    got = d_out.view(cx.n, NK)[torch.from_numpy(rows).to(cx.dev)].cpu().numpy().view(np.uint32)
    suffix = f"_rank{cx.rank}" if cx.world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"sketches{suffix}.npy"), got.astype(np.float64))
    np.save(os.path.join(out_dir, f"read_index{suffix}.npy"), (rows + cx.rank * cx.n).astype(np.float64))


# ---- e2e ---------------------------------------------------------------------------------------------
def e2e_leg(cx, args, d_in, d_out):
    """The metric through the host-pointer C ABI call, host<->device copies inside the timed region."""
    import numpy as np
    import torch

    L, n, dev = cx.L, cx.n, cx.dev
    h_in = torch.empty(n * READ_LEN, dtype=torch.uint8, pin_memory=True)   # allocated after the NUMA bind
    h_out = torch.empty(n * NK, dtype=torch.int32, pin_memory=True)
    h_in.copy_(d_in)
    torch.cuda.synchronize()
    ksteps = args.e2e_steps or min(args.steps, 5)

    def timed(fn, steps):
        fn()
        barrier(cx)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()  # synchronous: returns when the sketches are in host memory
        barrier(cx)
        return max_over_ranks(cx, time.perf_counter() - t0)

    def pinned_step():
        cx.check(L.pg_mash_sketch_uniform(h_in.data_ptr(), n, READ_LEN, KMER, SKETCH, 0, h_out.data_ptr(), NK, None))

    dt = timed(pinned_step, ksteps)
    e2e = {"value": cx.world * n * READ_LEN * ksteps / dt / 1e9, "unit": "Gbases/s", "h2d_bytes_per_step": n * READ_LEN,
           "d2h_bytes_per_step": n * NK * 4, "steps": ksteps, "ms_per_step": 1e3 * dt / ksteps,
           "api": "pg_mash_sketch_uniform (host buffers, pinned, NUMA-local to the GPU)", "numa_node": cx.numa_node,
           "host_GBps_aggregate": cx.world * n * (READ_LEN + NK * 4) * ksteps / dt / 1e9}
    # the host path and the device path must agree bit for bit
    e2e["matches_device_path"] = all_true(cx, bool(torch.equal(h_out[: 4096 * NK].to(dev), d_out[: 4096 * NK])))

    # platform cap: the same bytes as bare cudaMemcpyAsync on two streams, every rank at once
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def bare(do_h2d, do_d2h):
        def f():
            if do_h2d:
                with torch.cuda.stream(s_in):
                    d_in.copy_(h_in, non_blocking=True)
            if do_d2h:
                with torch.cuda.stream(s_out):
                    h_out.copy_(d_out, non_blocking=True)
            s_in.synchronize(); s_out.synchronize()
        return f

    hb = {}
    for name, a, b, nbytes in (("d2h", False, True, n * NK * 4), ("h2d", True, False, n * READ_LEN), ("both", True, True, n * (READ_LEN + NK * 4))):
        dtb = timed(bare(a, b), 2)
        hb[name + "_GBps_per_gpu"] = nbytes * 2 / dtb / 1e9
        hb[name + "_GBps_aggregate"] = cx.world * nbytes * 2 / dtb / 1e9
    hb["note"] = ("bare cudaMemcpyAsync of one step's bytes from the same pinned buffers on all ranks at once; "
                  "e2e.ms_per_step cannot be below both-direction time = the PCIe / host-memory cap of this box")
    e2e["floor_ms_per_step_from_bare_copies"] = 1e3 * n * (READ_LEN + NK * 4) / (hb["both_GBps_per_gpu"] * 1e9)
    variants = None
    if cx.world == 1:
        # pageable host buffers (what a Go []byte / []uint32 is), same call
        p_in = h_in.numpy().copy()
        p_out = np.empty(n * NK, dtype=np.int32)

        def pageable_step():
            cx.check(L.pg_mash_sketch_uniform(p_in.ctypes.data, n, READ_LEN, KMER, SKETCH, 0, p_out.ctypes.data, NK, None))

        dtp = timed(pageable_step, 2)
        ok_p = bool(np.array_equal(p_out[: 4096 * NK], h_out[: 4096 * NK].numpy()))
        del p_out
        # the shape mash.SketchBatch hands back to Go: a full 4*s-byte Sketches array per read, pageable, on a
        # bounded slice so that the 4 kB/read fits.  (a) PG_SKETCH_PAD_ZERO: the library writes all 4 kB per read
        # (everything a fresh []*Mash costs, into warm memory); (b) PG_SKETCH_TAIL_KEEP into an array the caller
        # zeroed beforehand (outside the timed region): the library's share when the host language already hands out
        # zeroed memory, as Go's make does.  First-touching a FRESH 8 GB slab inside the step costs ~1 s on this box
        # (page faults; measured once, DESIGN.md section 6) -- for any implementation, the CPU reference included.
        m = min(n, 2_000_000)
        g_out = np.empty((m, SKETCH), dtype=np.uint32)

        def go_step():
            cx.check(L.pg_mash_sketch_uniform(p_in.ctypes.data, m, READ_LEN, KMER, SKETCH, 1, g_out.ctypes.data, SKETCH, None))

        dtg = timed(go_step, 2)
        ok_g = bool(np.array_equal(g_out[:4096, :NK].reshape(-1).view(np.int32), h_out[: 4096 * NK].numpy()) and not g_out[:4096, NK:].any())
        g_out[:] = 0

        def keep_step():
            cx.check(L.pg_mash_sketch_uniform(p_in.ctypes.data, m, READ_LEN, KMER, SKETCH, 2, g_out.ctypes.data, SKETCH, None))

        dtk = timed(keep_step, 2)
        ok_k = bool(np.array_equal(g_out[:4096, :NK].reshape(-1).view(np.int32), h_out[: 4096 * NK].numpy()) and not g_out[:4096, NK:].any()
                    and np.array_equal(g_out[-1, :NK].view(np.int32), h_out[(m - 1) * NK: m * NK].numpy()) and not g_out[-1, NK:].any())
        variants = {
            "pageable": {"value": n * READ_LEN * 2 / dtp / 1e9, "unit": "Gbases/s", "ms_per_step": 1e3 * dtp / 2, "matches": ok_p,
                         "api": "pg_mash_sketch_uniform, pageable numpy buffers (a Go []byte / []uint32)"},
            "go_shape": {"value": m * READ_LEN * 2 / dtg / 1e9, "unit": "Gbases/s", "ms_per_step": 1e3 * dtg / 2, "reads": m, "matches": ok_g,
                         "host_array_bytes_per_step": m * SKETCH * 4,
                         "api": "pg_mash_sketch_uniform with PG_SKETCH_PAD_ZERO into a pageable [reads][1000] uint32 array: "
                                "the full Sketches array of every read as mash.SketchBatch returns it (4 kB/read, like the CPU arm's calloc per read)"},
            "go_shape_tail_keep": {"value": m * READ_LEN * 2 / dtk / 1e9, "unit": "Gbases/s", "ms_per_step": 1e3 * dtk / 2, "reads": m, "matches": ok_k,
                                   "host_array_bytes_per_step": m * SKETCH * 4,
                                   "api": "the same array, zeroed by the caller outside the timed region, PG_SKETCH_TAIL_KEEP: only the informative "
                                          "words are written (go/search/mash SketchBatch: one zeroed slab from make, filled in place)"},
        }
        del g_out, p_in
    del h_in, h_out
    return e2e, hb, variants


# ---- secondary configs (N=1) -----------------------------------------------------------------------------
def secondary_leg(cx, clocks_mhz):
    """configs[2] (100k x 10 kbp, k=31, s=2000: sketch + all-pairs) and configs[4] (1M x 25 bp primers vs a
    10 kb template: SW + Tm) on this GPU, device-resident, CUDA events; parity on a sample; CPU beside."""
    import numpy as np
    import oracle_ffi
    import torch

    from poly_b200 import align, synth

    L, dev, st = cx.L, cx.dev, cx.stream
    cores = schedulable_cores()
    out = []
    clk = (clocks_mhz or 1965.0) * 1e6
    # ---- cfg3 sketch (K2) ----
    n, RL, k, s = 100_000, 10_000, 31, 2000
    d_reads = torch.empty(n * RL, dtype=torch.uint8, device=dev)
    cx.check(L.pg_synth_reads_dev(d_reads.data_ptr(), 0, n, RL, synth.SEED_READS, 1, 100, st))
    d_sk = torch.empty((n, s), dtype=torch.int32, device=dev)
    l0 = L.pg_launch_count()
    ms, _ = ev_time(lambda: cx.check(L.pg_mash_sketch_uniform_dev(d_reads.data_ptr(), n, RL, k, s, 0, d_sk.data_ptr(), s, None, st)), iters=3, warm=1)
    launches = (L.pg_launch_count() - l0) // 4
    m = 64
    host_reads = synth.family_reads(m, RL, family=100)
    rc, want = oracle_ffi.sketch_batch(host_reads, synth.uniform_offsets(m, RL), k, s, variant=1)
    parity = rc == 0 and bool(np.array_equal(d_sk[:m].cpu().numpy().view(np.uint32), want))
    # CPU: the faithful variant re-sorts 2000 words on every qualifying insert (mash.go:90,99): ~0.1 s per read
    mc = max(2, min(m, 4 * cores))
    t0 = time.perf_counter(); oracle_ffi.sketch_batch_timing(host_reads[: mc * RL], synth.uniform_offsets(mc, RL), k, s, 0, cores); dtc = time.perf_counter() - t0
    # integer-issue ceiling of the formulation (SURVEY 7.2): murmur3 of a 31-mer with shared block pre-mixes needs
    # >= 7 body rounds x 3 + pre-mix 3 + 3-byte tail 4 + length xor 1 + fmix 8 = 37 thread instructions per k-mer
    inst = 37
    ceiling = 148 * 4 * clk * 32 / inst  # SMs x sub-partitions x issue/clk x lanes / instructions per k-mer
    out.append({"name": "cfg3 sketch (K2)", "config": "configs[2]: 100k x 10 kbp long reads, k=31, sketchSize=2000",
                "kernel": "sketch_thresh_walk_kernel + sketch_thresh_select_kernel (+ sketch_select_walk_kernel over the retry list, empty here)",
                "ms": ms, "value": n * RL / ms / 1e6, "unit": "Gbases/s", "gpu_launches_per_pass": launches,
                "bound": "integer issue (not HBM: 1.8 B/base)", "int_issue_ceiling_gbases_per_s": ceiling / 1e9,
                "int_issue_ceiling_derivation": f"148 SMs x 4 sub-partitions x {clk / 1e6:.0f} MHz x 32 lanes / {inst} instructions per 31-mer "
                                                "(7 body rounds x 3, pre-mix 3, tail 4, len 1, fmix 8); selection work excluded",
                "frac_of_int_issue_ceiling": (n * RL / ms * 1e3) / ceiling, "algorithmic_GBps": n * (RL + 4 * s) / ms / 1e6,
                "frac_of_hbm_peak": n * (RL + 4 * s) / ms / 1e6 / cx.peak, "parity_vs_oracle": parity, "parity_sample": f"first {m} reads, all {s} words",
                "cpu_baseline": {"value": mc * RL / dtc / 1e9, "unit": "Gbases/s", "cores": min(cores, mc), "kind": "port",
                                 "sample": f"{mc} reads, faithful variant (full re-sort per insert, mash.go:87-102), {dtc:.2f} s"}})
    # ---- cfg3 all-pairs (K3) ----
    pairs_unordered = n * (n - 1) // 2
    k3 = cx.all_pairs(d_sk, n, s)
    rows_chk = 4
    sk_host = d_sk[:400].cpu().numpy().view(np.uint32)
    rc, want_same = oracle_ffi.similarity_block(sk_host, 0, rows_chk, 0, 400, 1)
    t0 = time.perf_counter(); oracle_ffi.similarity_block(sk_host, 0, 400, 0, 400, cores); dtc = time.perf_counter() - t0
    k3.update({"name": "cfg3 all-pairs (K3)", "config": "configs[2]: all-pairs Mash distance over the 100k sketches",
               "pairs_unordered": pairs_unordered, "algorithmic_bytes": n * s * 4 + 4 * pairs_unordered,
               "parity_vs_oracle": rc == 0 and cx.all_pairs_check(k3, want_same, rows_chk, 400),
               "parity_sample": f"rows 0..{rows_chk - 1} x columns 0..399 (same-family and cross-family pairs)",
               "cpu_baseline": {"value": 400 * 400 / dtc, "unit": "pairs/s", "cores": cores, "kind": "port",
                                "sample": f"400 x 400 sketches, literal two-pointer walk per pair (mash.go:107-135), {dtc:.2f} s"}})
    k3["algorithmic_GBps"] = k3["algorithmic_bytes"] / k3["ms"] / 1e6
    k3["frac_of_hbm_peak"] = k3["algorithmic_GBps"] / cx.peak
    k3.pop("_result", None)
    out.append(k3)
    torch.cuda.empty_cache()
    k3s = cx.all_pairs_sparse(d_sk, n, s)
    k3s.update({"name": "cfg3 all-pairs, sparse upper-triangle output (K3)", "config": "configs[2]: the same all-pairs pass, returning only the pairs that share a hash",
                "pairs_unordered": pairs_unordered, "algorithmic_bytes": n * s * 4 + 4 * pairs_unordered,
                "parity_vs_oracle": rc == 0 and cx.all_pairs_check(k3s, want_same, rows_chk, 400),
                "parity_sample": f"rows 0..{rows_chk - 1} x columns 0..399, entries with j > i",
                "cpu_baseline": k3["cpu_baseline"]})
    k3s["unordered_pairs_per_s"] = pairs_unordered / k3s["ms"] * 1e3
    k3s.pop("_sparse", None)
    out.append(k3s)
    del d_reads, d_sk
    torch.cuda.empty_cache()
    # ---- cfg5: SW (K4) + Tm (K5) ----
    m, PL, TL = 1_000_000, 25, 10_000
    pr_host = synth.primers(m)
    pr = torch.from_numpy(pr_host).to(dev)
    off = torch.arange(m + 1, dtype=torch.int64, device=dev) * PL
    tpl_host = synth.template(TL)
    tpl = torch.from_numpy(tpl_host).to(dev)
    alpha = align.NewAlphabet(["-", "A", "C", "G", "T"])
    mat = np.array([[0, 0, 0, 0, 0], [0, 3, -3, -3, -3], [0, -3, 3, -3, -3], [0, -3, -3, 3, -3], [0, -3, -3, -3, 3]], dtype=np.int64)
    lut = alpha.byte_lut()
    score = torch.empty(m, dtype=torch.int64, device=dev)
    ec = torch.empty(m, dtype=torch.int32, device=dev)
    ep = torch.empty(m, dtype=torch.int64, device=dev)
    ms, _ = ev_time(lambda: cx.check(L.pg_sw_score_batch_dev(pr.data_ptr(), off.data_ptr(), m, PL, tpl.data_ptr(), TL, 1, lut.ctypes.data, lut.ctypes.data,
                                                            mat.ctypes.data, 5, 5, -2, score.data_ptr(), ec.data_ptr(), ep.data_ptr(), st)), iters=2, warm=1)
    mc = min(m, 256 * cores)
    offs_h = np.arange(mc + 1, dtype=np.uint64) * PL
    t0 = time.perf_counter(); rc, want_sc = oracle_ffi.sw_score_batch(pr_host[: mc * PL], offs_h, tpl_host, lut, lut, mat, -2, cores); dtc = time.perf_counter() - t0
    cells = m * PL * TL
    k4_name = (L.pg_last_kernel() or b"").decode()
    per_cell = 2 if "x2" in k4_name else 4  # 3 DPX add-max + 1 max per DP step; the packed int16 kernel advances two cells per step
    alu_ceiling = 148 * 64 * clk / per_cell  # ALU pipe: 64 lanes/clk/SM
    out.append({"name": "cfg5 Smith-Waterman score (K4)", "config": "configs[4]: 1M x 25 bp primers vs a 10 kb template, +3/-3, gap -2",
                "kernel": k4_name, "ms": ms, "value": cells / ms / 1e9, "unit": "TCUPS",
                "bound": "integer ALU / DPX issue", "alu_issue_ceiling_tcups": alu_ceiling / 1e12,
                "alu_issue_ceiling_derivation": f"148 SMs x 64 ALU lanes x {clk / 1e6:.0f} MHz / {per_cell} ALU-pipe instructions per cell"
                                                + (" (4 per DP step of the 2 x int16 packed kernel, two cells per step)" if per_cell == 2 else ""),
                "frac_of_alu_issue_ceiling": (cells / ms * 1e3) / alu_ceiling,
                "parity_vs_oracle": rc == 0 and bool(np.array_equal(score[:mc].cpu().numpy(), want_sc)) and int(ec.abs().max().item()) == 0,
                "parity_sample": f"first {mc} primers",
                "cpu_baseline": {"value": mc * PL * TL / dtc / 1e12, "unit": "TCUPS", "cores": cores, "kind": "port",
                                 "sample": f"{mc} primers x 10 kb, align.go:171-203 per pair (table scoring), {dtc:.2f} s"}})
    tm = torch.empty(m, dtype=torch.float64, device=dev)
    ms, _ = ev_time(lambda: cx.check(L.pg_tm_batch_dev(pr.data_ptr(), off.data_ptr(), m, 500e-9, 50e-3, 0.0, tm.data_ptr(), None, None, None, st)), iters=10, warm=1)
    offs_all = np.arange(m + 1, dtype=np.uint64) * PL
    t0 = time.perf_counter(); rc, want_tm = oracle_ffi.melting_temp_batch(pr_host, offs_all, cores); dtc = time.perf_counter() - t0
    got_tm = tm.cpu().numpy()
    rel = float(np.max(np.abs(got_tm - want_tm) / np.abs(want_tm)))
    out.append({"name": "cfg5 SantaLucia Tm (K5)", "config": "configs[4]: MeltingTemp of the 1M primers", "kernel": "tm_kernel", "ms": ms,
                "value": m / ms / 1e3, "unit": "Mprimers/s", "bound": "latency / launch (33 MB of traffic)",
                "parity_vs_oracle": rc == 0 and rel <= 1e-6, "parity_sample": f"all {m} primers, max relative difference {rel:.2e} (tolerance 1e-6)",
                "cpu_baseline": {"value": m / dtc / 1e6, "unit": "Mprimers/s", "cores": cores, "kind": "port",
                                 "sample": f"all {m} primers, primers.go:70-128 per primer, {dtc:.2f} s"}})
    return out


# ---- multi-GPU pipeline (N>1) ----------------------------------------------------------------------------
def pipeline_leg(cx, d_in, d_out):
    """The exchange step north_star names, timed max-over-ranks, with in-run parity assertions."""
    import numpy as np
    import oracle_ffi
    import torch
    import torch.distributed as dist

    from poly_b200 import synth
    from poly_b200.dist import GatheredBuffer, ShardPlan, all_gather_rows, cuda_distance_block, cuda_sketch_uniform, fused_sketch_gather

    L, dev, rank, world, n = cx.L, cx.dev, cx.rank, cx.world, cx.n
    res = {}

    def timed(fn):
        barrier(cx)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        return out, max_over_ranks(cx, e0.elapsed_time(e1))

    def oracle_rows(first_read, m, RL, k, s, family):
        reads = synth.family_reads(m, RL, family=family, first_read=first_read) if family else synth.independent_reads(m, RL, first_read=first_read)
        rc, want = oracle_ffi.sketch_batch(reads, synth.uniform_offsets(m, RL), k, s, variant=1)
        assert rc == 0
        return want

    # ---- B: cfg4 shape -- every rank sketches its 10M reads; all-gather of the compact sketches ----
    plan = ShardPlan(n * world, rank, world)
    local_sk = d_out.view(n, NK)  # K1 output of the headline step (reads [rank*n, (rank+1)*n))
    gathered, t_ag = timed(lambda: all_gather_rows(local_sk, plan))
    gathered, t_ag2 = timed(lambda: all_gather_rows(local_sk, plan))
    t_ag = min(t_ag, t_ag2)
    _, t_sk = timed(lambda: cx.check(L.pg_mash_sketch_uniform_dev(d_in.data_ptr(), n, READ_LEN, KMER, SKETCH, 0, d_out.data_ptr(), NK, None, cx.stream)))
    buf = GatheredBuffer(plan, NK)
    fused = lambda: fused_sketch_gather(d_in, READ_LEN, KMER, SKETCH, buf, sync=False)  # noqa: E731
    fused(); barrier(cx)
    _, t_f = timed(fused)
    _, t_f2 = timed(fused)
    t_f = min(t_f, t_f2)
    barrier(cx)
    fused_t = buf.as_tensor()
    # parity 1: the fused buffer equals the NCCL all-gather, whole buffer, on every rank
    eq = all_true(cx, bool(torch.equal(fused_t, gathered)))
    # parity 2: on every rank, the first 256 rows of EVERY rank's block equal the oracle
    ok = True
    for r in range(world):
        want = oracle_rows(r * n, 256, READ_LEN, KMER, SKETCH, 0)[:, :NK]
        ok = ok and bool(np.array_equal(fused_t[r * n: r * n + 256].cpu().numpy().view(np.uint32), want))
    ok = all_true(cx, ok)
    # capped row-block distance over the gathered set (reference semantics: n = 129 < s = 1000 -> unsorted
    # zero-padded sketches -> every pair takes the early-out of mash.go:117: distance 1.0, SURVEY 8e)
    cols_per = min(16384, n)
    rows = min(4096, cols_per)
    sub = torch.zeros((cols_per * world, SKETCH), dtype=torch.int32, device=dev)
    for r in range(world):
        sub[r * cols_per:(r + 1) * cols_per, :NK] = fused_t[r * n: r * n + cols_per]
    same, t_d = timed(lambda: cuda_distance_block(sub, rank * cols_per, rank * cols_per + rows))
    max_same = int(same.max().item())
    # oracle: a few pairs of that block, literal walk
    sub_h = sub[: 8].cpu().numpy().view(np.uint32)
    rc, want_same = oracle_ffi.similarity_block(sub_h, 0, 8, 0, 8, 1)
    same0, _ = timed(lambda: cuda_distance_block(sub, 0, 8))
    ok_d = all_true(cx, rc == 0 and bool(np.array_equal(same0[:, :8].cpu().numpy().view(np.uint32), want_same)))
    out_bytes = (world - 1) * n * NK * 4
    res["cfg4"] = {"config": f"configs[3] shape: {world} x {n} reads of 150 bp, k=21, s=1000; all-gather of the compact sketches ({NK} words/read), "
                             f"then rows [{rows}] x columns [{cols_per * world}] of the pair matrix per rank",
                   "sketch_ms": t_sk, "nccl_allgather_ms": t_ag, "separate_ms": t_sk + t_ag, "fused_sketch_gather_ms": t_f,
                   "fused_speedup_vs_separate": (t_sk + t_ag) / t_f, "bytes_out_per_rank_GB": out_bytes / 1e9,
                   "nvlink_GBps_out_per_rank_fused": out_bytes / t_f / 1e6, "nvlink_GBps_per_rank_nccl": out_bytes / t_ag / 1e6,
                   "nvlink_peer_copy_peak_GBps": NVLINK_PEER_PEAK_GBS, "fused_frac_of_peer_copy_peak": out_bytes / t_f / 1e6 / NVLINK_PEER_PEAK_GBS,
                   "distance_block_ms": t_d, "distance_max_same": max_same,
                   "parity": {"fused_equals_nccl_allgather_all_rows_all_ranks": eq,
                              "every_rank_block_first_256_rows_equal_oracle_on_all_ranks": ok,
                              "distance_sample_equals_oracle": ok_d and max_same == 0}}
    del same, same0, sub, gathered, fused_t
    buf.close()
    torch.cuda.empty_cache()

    # ---- A: cfg3 sharded -- 100k long reads over the ranks: sketch -> gather -> row-block all-pairs ----
    nt, RL, k, s = 100_000, 10_000, 31, 2000
    plan = ShardPlan(nt, rank, world)
    nl = plan.hi - plan.lo
    reads = torch.empty(nl * RL, dtype=torch.uint8, device=dev)
    cx.check(L.pg_synth_reads_dev(reads.data_ptr(), plan.lo, nl, RL, synth.SEED_READS, 1, 100, cx.stream))
    cuda_sketch_uniform(reads, nl, RL, k, s)
    local_sk, t_sk = timed(lambda: cuda_sketch_uniform(reads, nl, RL, k, s))
    gathered, t_ag = timed(lambda: all_gather_rows(local_sk, plan))
    gathered, t_ag = timed(lambda: all_gather_rows(local_sk, plan))
    buf = GatheredBuffer(plan, s)
    fused = lambda: fused_sketch_gather(reads, RL, k, s, buf, sync=False)  # noqa: E731
    fused(); barrier(cx)
    _, t_f = timed(fused)
    barrier(cx)
    fused_t = buf.as_tensor()
    eq = all_true(cx, bool(torch.equal(fused_t, gathered)))
    ok = True
    for r in range(world):
        lo_r = ShardPlan(nt, r, world).lo
        ok = ok and bool(np.array_equal(fused_t[lo_r: lo_r + 8].cpu().numpy().view(np.uint32), oracle_rows(lo_r, 8, RL, k, s, 100)))
    ok = all_true(cx, ok)
    k3 = cx.all_pairs(fused_t, nt, s, plan.lo, plan.hi, timer=timed)
    rows_chk = 2
    sk_host = fused_t[plan.lo: plan.lo + 200].cpu().numpy().view(np.uint32)
    # rows [lo, lo+2) x columns [lo, lo+200): this rank's own families
    rc, want_same = oracle_ffi.similarity_block(sk_host, 0, rows_chk, 0, 200, 1)
    ok_d = all_true(cx, rc == 0 and cx.all_pairs_check(k3, want_same, rows_chk, 200, col0=plan.lo))
    k3.pop("_result", None)
    res["cfg3_sharded"] = {"config": f"configs[2] sharded: {nt} x 10 kbp reads over {world} ranks, k=31, s=2000; gather of the sketches; rank r computes row block r",
                           "sketch_ms": t_sk, "nccl_allgather_ms": t_ag, "fused_sketch_gather_ms": t_f, "gather_GB_recv_per_rank": (nt - nl) * s * 4 / 1e9,
                           "distance": k3, "parity": {"fused_equals_nccl_allgather": eq, "gathered_sample_equals_oracle_on_all_ranks": ok,
                                                      "distance_sample_equals_oracle": ok_d}}
    del fused_t, gathered, reads, local_sk
    buf.close()
    torch.cuda.empty_cache()
    res["parity_all_green"] = all(all(v.values()) for v in (res["cfg4"]["parity"], res["cfg3_sharded"]["parity"]))
    return res


def make_all_pairs(cx):
    """All-pairs matching counts over device-resident sketches through the C ABI; returns timing + a handle
    the parity check reads back.  Rows [r0, r1) (default all) x all columns."""
    import numpy as np
    import torch

    L = cx.L

    def all_pairs(d_sk, n, s, r0=0, r1=None, timer=None):
        r1 = n if r1 is None else r1
        rows = r1 - r0
        d_same = torch.empty((rows, n), dtype=torch.int32, device=cx.dev)
        sk = d_sk if d_sk.is_contiguous() else d_sk.contiguous()

        def run():
            cx.check(L.pg_mash_distance_block_dev(sk.data_ptr(), n, s, r0, r1, d_same.data_ptr(), None, cx.stream))

        l0 = L.pg_launch_count()
        run()  # warm-up: first touch of the output, pool growth
        launches = L.pg_launch_count() - l0
        if timer is None:
            ms, _ = ev_time(run, iters=1)
        else:
            _, ms = timer(run)
        return {"ms": ms, "rows": rows, "cols": n, "value": rows * n / ms / 1e6, "unit": "Gpairs/s (ordered pairs of the row block)",
                "kernel": (L.pg_last_kernel() or b"").decode(), "gpu_launches_per_pass": launches, "output": "dense uint32 [rows][n]",
                "output_bytes": rows * n * 4, "_result": d_same}

    def check(k3, want_same, rows, cols, col0=0):
        if "_sparse" in k3:  # triples -> the dense sample (upper triangle only: j > i)
            di, dj, dc, cnt, r0 = k3["_sparse"]
            i, j, c = (t[:cnt].cpu().numpy().astype(np.int64) for t in (di, dj, dc))
            sel = (i < r0 + rows) & (j >= col0) & (j < col0 + cols)
            got = np.zeros((rows, cols), dtype=np.uint32)
            got[i[sel] - r0, j[sel] - col0] = c[sel].astype(np.uint32)
            want = want_same.copy()
            for a in range(rows):  # entries the sparse upper form does not carry: j <= i
                want[a, : max(0, r0 + a + 1 - col0)] = 0
            return bool(np.array_equal(got, want))
        got = k3["_result"][:rows, col0: col0 + cols].cpu().numpy().view(np.uint32)
        return bool(np.array_equal(got, want_same))

    def all_pairs_sparse(d_sk, n, s, r0=0, r1=None, timer=None, cap=32_000_000):
        r1 = n if r1 is None else r1
        d_i, d_j, d_c = (torch.empty(cap, dtype=torch.int32, device=cx.dev) for _ in range(3))
        d_n = torch.zeros(1, dtype=torch.int64, device=cx.dev)
        sk = d_sk if d_sk.is_contiguous() else d_sk.contiguous()

        def run():
            cx.check(L.pg_mash_distance_sparse_dev(sk.data_ptr(), n, s, r0, r1, 1, d_i.data_ptr(), d_j.data_ptr(), d_c.data_ptr(), cap, d_n.data_ptr(), cx.stream))

        l0 = L.pg_launch_count()
        run()
        launches = L.pg_launch_count() - l0
        if timer is None:
            ms, _ = ev_time(run, iters=1)
        else:
            _, ms = timer(run)
        cnt = int(d_n.item())
        return {"ms": ms, "rows": r1 - r0, "cols": n, "value": (r1 - r0) * n / ms / 1e6, "unit": "Gpairs/s (ordered pairs of the row block covered)",
                "kernel": "bucket_join_kernel + compact_pairs_kernel", "gpu_launches_per_pass": launches,
                "output": "sparse (i, j, same) triples of the pairs with j > i that share a hash", "pairs_listed": cnt, "output_bytes": cnt * 12,
                "fits_capacity": cnt <= cap, "_sparse": (d_i, d_j, d_c, min(cnt, cap), r0)}

    cx.all_pairs_sparse = all_pairs_sparse
    return all_pairs, check


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import numpy as np
    import torch
    import torch.distributed as dist

    from poly_b200 import _lib, synth

    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = _lib.lib()
    _lib.check(L.pg_init(local))
    # NUMA: this rank's thread (and the threads / pinned pages it creates from now on) on the GPU's node
    affinity0 = os.sched_getaffinity(0)
    node = C.c_int(-1)
    L.pg_numa_bind_thread(local, C.byref(node))
    dev = torch.device("cuda", local)
    n = args.reads
    first_read = rank * n  # rank r sketches reads [r*n, (r+1)*n): no data-path collective
    stream = torch.cuda.current_stream().cuda_stream

    cx = Ctx()
    cx.L, cx.dev, cx.rank, cx.world, cx.n, cx.stream, cx.check, cx.numa_node = L, dev, rank, world, n, stream, _lib.check, node.value
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        cx.peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        cx.peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    cx.all_pairs, cx.all_pairs_check = make_all_pairs(cx)

    d_in = torch.empty(n * READ_LEN, dtype=torch.uint8, device=dev)
    d_out = torch.empty(n * NK, dtype=torch.int32, device=dev)
    _lib.check(L.pg_synth_reads_dev(d_in.data_ptr(), first_read, n, READ_LEN, synth.SEED_READS, 0, 0, stream))
    torch.cuda.synchronize()

    def step():
        _lib.check(L.pg_mash_sketch_uniform_dev(d_in.data_ptr(), n, READ_LEN, KMER, SKETCH, 0, d_out.data_ptr(), NK, None, stream))

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)  # let nvidia-smi start streaming
    clocks.t_load = time.time()
    for _ in range(max(args.warmup, 3)):
        step()
    # keep the device loaded for >= 100 ms before the timed region so that the clock samples
    # describe clocks under load (untimed; same kernel)
    barrier(cx)
    t_pre = time.time()
    while time.time() - t_pre < 0.1:
        step()
        torch.cuda.synchronize()
    barrier(cx)
    launches0 = L.pg_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(cx)
    clocks.t0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier(cx)
    clocks.t1 = time.time()
    ms = ev0.elapsed_time(ev1)
    launches = L.pg_launch_count() - launches0
    kernel_name = (L.pg_last_kernel() or b"").decode()
    clk = clocks.stop() if rank == 0 else None
    ms = max_over_ranks(cx, ms)
    ms_per_step = ms / args.steps
    value = world * n * READ_LEN / (ms_per_step * 1e-3) / 1e9  # whole-job Gbases/s

    # in-run parity of the headline result on EVERY rank: head of this rank's shard vs the oracle
    import oracle_ffi
    m = 2048
    rc, want = oracle_ffi.sketch_batch(synth.independent_reads(m, READ_LEN, first_read=first_read), synth.uniform_offsets(m, READ_LEN), KMER, SKETCH, 1, 1)
    got = d_out[: m * NK].cpu().numpy().view(np.uint32).reshape(m, NK)
    headline_parity = all_true(cx, rc == 0 and bool(np.array_equal(got, want[:, :NK])))
    if args.dump_outputs:
        dump_outputs(cx, d_out, args.dump_outputs)

    e2e = host_bw = e2e_variants = None
    if not args.no_e2e:
        e2e, host_bw, e2e_variants = e2e_leg(cx, args, d_in, d_out)

    pipeline = None
    if world > 1 and not args.no_pipeline:
        pipeline = pipeline_leg(cx, d_in, d_out)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    achieved = n * BYTES_PER_READ / (ms_per_step * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj["dram_bytes_per_read"] * n  # per launch, scaled from the ncu capture's reads
            traffic_src = f"profiles/k1_traffic.json: ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of {tj.get('source', 'the committed capture')}, per read x {n} reads (not measured in this run: ncu cannot run inside the timed bench)"
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": cx.peak, "unit": "GB/s", "frac": achieved / cx.peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": kernel_name, "algorithmic_bytes_per_launch": n * BYTES_PER_READ,
                "peak_source": peak_src, "avg_launch_ms": ms_per_step}

    del d_in, d_out
    torch.cuda.empty_cache()
    secondary = None
    if world == 1 and not args.no_secondary:
        os.sched_setaffinity(0, affinity0)  # the CPU baselines of this leg use every schedulable core
        secondary = secondary_leg(cx, clk.get("sm_mhz") if clk else None)

    cpu_baseline = None
    if world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, affinity0)
        cpu_baseline, ns, _ = cpu_reference_leg(8.0)
    if cpu_baseline is not None:
        cpu_baseline["gpu_matches_oracle_on_first_2048_reads"] = headline_parity

    out = {
        "metric": METRIC, "value": value, "unit": "Gbases/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
        "data": "synthetic",
        "config": {"workload": "configs[1]: 10M x 150bp short reads, k=21, sketchSize=1000 per GPU"
                   + (" (x8 = configs[3], 80M reads)" if world == 8 else ""),
                   "reads_per_gpu": n, "read_len": READ_LEN, "k": KMER, "sketch_size": SKETCH,
                   "l2": "inputs (1.5 GB) + outputs (5.2 GB) per step are larger than L2 (126 MB); no explicit flush",
                   "parallelism": f"reads sharded over {world} GPU(s), no data-path collective"},
        "parity": {"head_of_every_rank_shard_equals_oracle": headline_parity},
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "e2e_variants": e2e_variants, "host_bw": host_bw,
        "gpu_launches": int(launches), "clocks": clk, "secondary": secondary, "pipeline": pipeline,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
