#!/usr/bin/env python
"""bench.py -- headline benchmark of the dense-LA hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic input: one bf16 matmul 8192^3 per GPU (BASELINE
config 3; at N GPUs the batch axis [N, 8192, 8192] is sharded one batch per rank -- batched matmul over the batch axis,
no data-path collective, weak scaling).  `value` = whole-job TFLOP/s with operands resident in HBM, timed with CUDA events
on the launching stream, max over ranks.  `e2e` = the same metric through the public API with HOST buffers (pinned H2D of
both operands + D2H of the result inside the timed region, every step).

Secondary objects on the same JSON line cover the other BASELINE configs: `reduce` (f32 sum of 2^28, weak + strong
sharding with an NCCL all-reduce), `matmul_f32_4096`, `batched_bf16_4096`, `reference_equivalent` (what CubeCL's own
wmma / vec4 kernels reach on this GPU), plus `roofline`, `roofline_reduce`, `cpu_baseline`, `clocks`.

--impl reference times the reference's CPU semantics (the oracle port; the Rust reference cannot be built here) on the
host cores, on a bounded sample of the same workload; rank 0 only.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# stdout carries exactly one JSON line: NCCL's own log (the "NCCL version ..." banner that NCCL_DEBUG=VERSION/INFO prints,
# from torch's communicator and from this library's) goes to stderr unless the caller already chose a file
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

N_MM = 8192                      # BASELINE config 3
FLOPS_MM = 2.0 * N_MM ** 3
N_RED = 1 << 28                  # BASELINE config 4
BYTES_RED = N_RED * 4
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    return dict(FALLBACK_PEAKS, bf16_tflops_sustained=1400.0, source="fallback")


def ncu_traffic():
    """Per-launch DRAM traffic of the dominant kernels, from the committed ncu summary of this round (or None)."""
    p = ROOT / "profiles" / "traffic.json"
    return json.loads(p.read_text()) if p.exists() else {}


# ---------------------------------------------------------------------------------------------------- clocks
@contextlib.contextmanager
def near_gpu(index: int):
    """While pinned host buffers are allocated, run on the CPUs NVML reports as local to GPU `index`: the pages are placed on
    that NUMA node (first touch at pin time), so the per-step H2D / D2H copies do not cross the socket interconnect.
    One process per GPU, each next to its own device.  Restores the affinity afterwards; a no-op if NVML cannot tell."""
    old = None
    try:
        nv, h = ClockSampler._handle(index)
        words = (os.cpu_count() + 63) // 64
        mask = nv.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {i * 64 + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        if cpus & allowed and os.environ.get("B200_BENCH_NUMA", "1") != "0":
            old = allowed
            os.sched_setaffinity(0, cpus & allowed)
    except Exception:  # noqa: BLE001
        old = None
    try:
        yield
    finally:
        if old is not None:
            os.sched_setaffinity(0, old)


class ClockSampler:
    """Samples SM clock / power / throttle reasons through NVML from a thread DURING the timed region (the recipe's
    nvidia-smi line needs ~100 ms per sample; a 20-step timed region lasts ~15 ms)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._thr, self.err = index, [], threading.Event(), None, None
        self.max_mhz = None

    _nv = None
    _handles = {}

    @classmethod
    def _handle(cls, index):
        """NVML is initialised once, BEFORE any timed region (nvmlInit alone can take longer than the timed region)."""
        if cls._nv is None:
            import pynvml as nv
            nv.nvmlInit()
            cls._nv = nv
        if index not in cls._handles:
            cls._handles[index] = cls._nv.nvmlDeviceGetHandleByIndex(index)
        return cls._nv, cls._handles[index]

    def _run(self):
        try:
            nv, h = self._handle(self.index)
            reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while True:
                self.rows.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), nv.nvmlDeviceGetPowerUsage(h) / 1000.0, int(reasons(h))))
                if self._stop.is_set():
                    break
                time.sleep(0.001)
        except Exception as e:  # noqa: BLE001
            self.err = str(e)

    def __enter__(self):
        try:
            nv, h = self._handle(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = str(e)
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=5)

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": len(self.rows), "how": "NVML thread, ~1 ms period, started before warm-up"}
        if self.err:
            out["error"] = self.err
        if self.rows:
            busy = [r for r in self.rows if r[1] >= 0.5 * max(x[1] for x in self.rows)] or self.rows   # samples under load
            out["sm_mhz"] = float(np.median([r[0] for r in busy]))
            out["sm_mhz_min"] = float(min(r[0] for r in busy))
            out["power_w_max"] = float(max(r[1] for r in self.rows))
            bits = 0
            for r in busy:
                bits |= r[2]
            out["reasons"] = [nm for bit, nm in self.REASONS.items() if bits & bit]
        return out


def rejected(clocks) -> bool:
    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if bad & set(clocks.get("reasons", [])):
        return True
    sm, mx = clocks.get("sm_mhz"), clocks.get("sm_max_mhz")
    return bool(sm and mx and sm < 0.5 * mx and not clocks.get("reasons"))


# ---------------------------------------------------------------------------------------------------- reference arm
def host_threads() -> int:
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1, which would otherwise cap the CPU arm)."""
    try:
        return max(1, min(256, len(os.sched_getaffinity(0))))
    except AttributeError:
        return max(1, min(256, os.cpu_count() or 1))


_CPU_OPERANDS = {}


def cpu_matmul_sample(seconds_target=12.0):
    """Reference-order CPU matmul (oracle port, all host threads) on a bounded block of C of the 8192^3 problem: every output is
    one serial f32 sum over k (the reference's arithmetic), 4 x 4 outputs carried at once, rhs walked in L2-sized panels."""
    import oracle
    from cubecl_b200 import synth
    threads = host_threads()
    K = N_MM

    def operand(seed, rows):   # bf16-rounded rows of the seeded operand; kept across steps (generating 8192 x 8192 takes seconds)
        have = _CPU_OPERANDS.get(seed)
        if have is None or have.shape[0] < rows:
            have = synth.bf16_bits_to_f32(synth.f32_to_bf16_bits(synth.uniform_f32(seed, rows * K, -1.0, 1.0))).reshape(rows, K)
            _CPU_OPERANDS[seed] = have
        return have[:rows]

    b_nk = operand(4, 512)                                 # 512 rhs columns
    rows = 4 * threads
    a = operand(3, rows)
    oracle.matmul_blocked_f32(a[:threads], b_nk, threads)  # thread pool up, pages touched
    t0 = time.perf_counter()
    oracle.matmul_blocked_f32(a, b_nk, threads)
    dt = time.perf_counter() - t0
    rate = 2.0 * rows * 512 * K / dt                       # FLOP/s on the probe
    # size the sample to ~seconds_target of work: rows first (up to the full 8192), then more rhs columns (up to the full 8192)
    want = seconds_target * rate
    rows_s = int(max(rows, min(N_MM, want / (2.0 * 512 * K))))
    rows_s = max(4 * threads, rows_s // (4 * threads) * (4 * threads))
    cols_s = 512
    if rows_s >= N_MM:
        rows_s = N_MM
        cols_s = int(max(512, min(N_MM, want / (2.0 * N_MM * K)) // 512 * 512))
    a = operand(3, rows_s)
    if cols_s != 512:
        b_nk = operand(4, cols_s)
    t0 = time.perf_counter()
    oracle.matmul_blocked_f32(a, b_nk, threads)
    dt = time.perf_counter() - t0
    flops = 2.0 * rows_s * cols_s * K
    return {"value": flops / dt / 1e12, "unit": "TFLOP/s", "cores": threads, "kind": "port",
            "sample": f"{rows_s}x{cols_s} block of C of the bf16 8192^3 matmul (K=8192 full), reference-order f32 sums (4x4 outputs in flight, "
                      f"64-column rhs panels), {threads} threads, {dt:.1f} s",
            "seconds": dt, "flops": flops}


def cpu_reduce_sample():
    import oracle
    from cubecl_b200 import synth
    threads = host_threads()
    n = 1 << 26
    x = synth.uniform_f32(5, n, 0.0, 1.0)
    t0 = time.perf_counter(); oracle.sum_serial_f32(x); t_serial = time.perf_counter() - t0
    t0 = time.perf_counter(); oracle.sum_blocked_f32(x, threads); t_blocked = time.perf_counter() - t0
    return {"serial_gbs": n * 4 / t_serial / 1e9, "blocked_gbs": n * 4 / t_blocked / 1e9, "cores": threads,
            "sample": "2^26 of the 2^28 f32 elements"}


def run_reference(args):
    e_rank = int(os.environ.get("RANK", "0"))
    if e_rank != 0:
        return
    times, last = [], None
    for i in range(args.warmup + args.steps):
        last = cpu_matmul_sample(seconds_target=max(1.0, 40.0 / (args.warmup + args.steps)))
        if i >= args.warmup:
            times.append(last)
    flops = sum(t["flops"] for t in times)
    secs = sum(t["seconds"] for t in times)
    val = flops / secs / 1e12
    line = {"impl": "reference", "metric": "bf16_matmul_tflops", "value": val, "unit": "TFLOP/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / len(times) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "bf16 matmul 8192x8192x8192 (f32 accumulate), bounded sample per step",
                       "note": "reference = CPU restatement of cubecl's semantics (oracle port); the Rust reference cannot be built here"},
            "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": last["cores"], "kind": "port", "sample": last["sample"]},
            "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------------- parity on the record
def mod8_prefix_sum(n: int) -> int:
    """sum_{i < n} (i % 8), exactly."""
    q, r = divmod(int(n), 8)
    return q * 28 + r * (r - 1) // 2


def check_matmul_samples(c, seed_a, seed_b, out, batches, n, rng, samples=16):
    """Sampled outputs of a device-generated bf16 [B, n, n] x [B, n, n] product against f64 dot products of the operands
    regenerated on the host (counter hash): reads back only the sampled output rows.  Returns (ok, worst scaled error)."""
    from cubecl_b200 import synth
    worst, worst_abs = 0.0, 0.0
    for b in batches:
        ms, ns = rng.integers(0, n, samples), rng.integers(0, n, samples)
        for m, col in zip(ms, ns):
            a_row = synth.uniform_f32(seed_a, n, -1.0, 1.0, start=(b * n + int(m)) * n)
            b_col = synth.uniform_at(seed_b, (b * n + np.arange(n, dtype=np.uint64)) * n + np.uint64(col), -1.0, 1.0)
            a_row = synth.bf16_bits_to_f32(synth.f32_to_bf16_bits(a_row)).astype(np.float64)
            b_col = synth.bf16_bits_to_f32(synth.f32_to_bf16_bits(b_col)).astype(np.float64)
            ref, scale = float(a_row @ b_col), float(np.abs(a_row) @ np.abs(b_col))
            raw = c.read_one(out.handle.offset(((b * n + int(m)) * n + int(col)) * 2, 2))
            got = float(synth.bf16_bits_to_f32(np.frombuffer(raw, dtype=np.uint16))[0])
            worst = max(worst, abs(got - ref) / scale)
            worst_abs = max(worst_abs, abs(got - ref) - abs(ref) * 2.0 ** -8)
    # north star: <= 1e-2 relative for bf16; in fact only the bf16 output rounding (2^-9 relative) and f32 accumulation remain
    return bool(worst <= 1e-2 and worst_abs <= 0.05), worst


DUMP_ROWS = 1024                 # rows of C dumped over all ranks: 1024 x 8192 f32 = 32 MiB


def dump_headline(c, out, rank, world, out_dir):
    """Write what the headline's last timed step left in this rank's bf16 product C (batch `rank` of the [world, 8192, 8192]
    output) as float32: the same seeded sample of DUMP_ROWS // world rows on every run, plus their row indices, so two builds
    given the same arguments can be compared output for output."""
    from cubecl_b200 import synth
    rows = np.sort(np.random.default_rng(0).choice(N_MM, max(1, DUMP_ROWS // world), replace=False))
    got = synth.bf16_bits_to_f32(out.to_numpy(c)[rows])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"matmul_bf16_8192_b{rank}.npy"), got)
    np.save(os.path.join(out_dir, f"matmul_bf16_8192_b{rank}_rows.npy"), rows.astype(np.float64))


def multi_gpu_parity(c, D, dist, e, world, ids, xs, reduce, TensorHandle):
    """Exact checks of the multi-GPU paths, on the record the driver keeps (runtime_tests/all_reduce.rs:5-62 is the model:
    integer-valued data, the reduced value identical on every rank and equal to the closed form):
      * local reduce + NCCL all-reduce + sync_collective, and the fused reduce + NVLink exchange, on rank-dependent extents
        (weak) and on contiguous shards of one 2^28 vector (strong);
      * the fused (key, index) exchange of argmax / argmin with cross-rank ties and NaNs planted at known global indices."""
    out = {}
    r_out = TensorHandle.empty_contiguous(c, [1], "f32")
    a_out = TensorHandle.empty_contiguous(c, [1], "u32")
    # ---- weak: rank r reduces n_r = 2^28 - r * 2^20 elements of (i % 8): local sum 3.5 n_r, every partial sum exact in f32
    n_r = N_RED - e.rank * (1 << 20)
    c.fill_modulo(xs[0].handle, "f32", N_RED, 8)
    view = TensorHandle(xs[0].handle.offset(0, n_r * 4), [n_r], [1], "f32")
    expect = float(sum(mod8_prefix_sum(N_RED - r * (1 << 20)) for r in range(world)))
    reduce.launch(c, view, r_out, None, "sum")
    c.all_reduce(r_out.handle, r_out.handle, "f32", ids, "sum")
    c.sync_collective()
    got_nccl = float(r_out.to_numpy(c)[0])
    got_fused = []
    for _ in range(3):                                    # three epochs: both mailbox parities and a reuse
        reduce.launch_all_reduce(c, view, r_out, ids)
        got_fused.append(float(r_out.to_numpy(c)[0]))
    out["weak_sum"] = {"expect": expect, "nccl": got_nccl, "fused": got_fused, "ok": got_nccl == expect and all(g == expect for g in got_fused)}
    # ---- strong: contiguous shards [lo, hi) of the same vector; shard sums from the closed form
    lo, hi = D.shard_range(N_RED, world, e.rank)
    shard = TensorHandle(xs[0].handle.offset(lo * 4, (hi - lo) * 4), [hi - lo], [1], "f32")
    expect_s = float(mod8_prefix_sum(N_RED))
    reduce.launch(c, shard, r_out, None, "sum")
    local = float(r_out.to_numpy(c)[0])
    c.all_reduce(r_out.handle, r_out.handle, "f32", ids, "sum")
    c.sync_collective()
    got_nccl = float(r_out.to_numpy(c)[0])
    reduce.launch_all_reduce(c, shard, r_out, ids)
    got_f = float(r_out.to_numpy(c)[0])
    out["strong_sum"] = {"expect": expect_s, "local_ok": local == float(mod8_prefix_sum(hi) - mod8_prefix_sum(lo)), "nccl": got_nccl, "fused": got_f,
                         "ok": got_nccl == expect_s and got_f == expect_s and local == float(mod8_prefix_sum(hi) - mod8_prefix_sum(lo))}
    # ---- fused arg exchange: per-rank shards of one logical vector, planted extrema
    per = (1 << 22) + 8
    sv = TensorHandle(xs[1].handle.offset(0, per * 4), [per], [1], "f32")
    c.fill_uniform(sv.handle, "f32", per, 33 + e.rank, -1.0, 1.0)

    def plant(rank, idx, value):
        if e.rank == rank:
            c.write(sv.handle.offset(idx * 4, 4), np.array([value], dtype=np.float32))

    last = world - 1
    cases = {}
    plant(1 % world, 17, 7.0); plant(last, 5, 7.0); plant(last, per - 1, 7.0)         # equal maxima on two ranks: lowest global index
    want = min((1 % world) * per + 17, last * per + 5)
    reduce.launch_arg_all_reduce(c, sv, a_out, ids, e.rank * per, "argmax")
    cases["argmax_ties"] = {"expect": want, "got": int(a_out.to_numpy(c)[0])}
    plant(last, 11, -9.0); plant(0, 4000, -9.0)
    reduce.launch_arg_all_reduce(c, sv, a_out, ids, e.rank * per, "argmin")
    cases["argmin_ties"] = {"expect": 4000, "got": int(a_out.to_numpy(c)[0])}
    plant(last, 3, float("nan")); plant(1 % world, 100, float("nan"))                   # NaN is the extreme; the first one wins
    want = min(last * per + 3, (1 % world) * per + 100)
    for op in ("argmax", "argmin"):
        reduce.launch_arg_all_reduce(c, sv, a_out, ids, e.rank * per, op)
        cases[op + "_nan"] = {"expect": want, "got": int(a_out.to_numpy(c)[0])}
    out["arg_all_reduce"] = dict(cases, ok=all(v["expect"] == v["got"] for v in cases.values()))
    out["ok"] = all(v["ok"] for v in out.values())
    return out


def all_ranks_ok(ok: bool, dist, tdev) -> bool:
    if dist is None:
        return ok
    import torch
    t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=tdev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


# ---------------------------------------------------------------------------------------------------- our arm
def emit(line: dict) -> None:
    """The ONE JSON line of the contract, written to the process's original stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


# stdout carries exactly one JSON line.  Libraries loaded later (NCCL's version banner under NCCL_DEBUG=VERSION, seen on the
# 2-GPU box) print to file descriptor 1 behind Python's back, so fd 1 is pointed at stderr for the whole run and the line goes
# to a private duplicate of the original stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def main():
    import faulthandler
    faulthandler.enable()                # a native fault in any rank leaves a Python stack on stderr instead of a bare signal
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="headline + reduce only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the headline's timed steps, write a fixed sample of rows of its last product to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        return run_reference(args)

    from cubecl_b200 import ComputeClient, TensorHandle, matmul, reduce, synth
    from cubecl_b200 import distributed as D

    e = D.env()
    world = e.world_size
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    dist = None
    tdev = None
    if world > 1:
        import torch
        dist = D.init_process_group("nccl")
        tdev = torch.device("cuda", e.local_rank)

    c = ComputeClient.load(e.local_rank)
    pk = peaks()
    rank0 = e.rank == 0

    def barrier():
        c.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warm):
        """W untimed + exactly `steps` timed launches between barriers; CUDA events on the launching stream; max over ranks."""
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = c.event(), c.event()
        l0 = c.launch_count()
        c.record(e0)
        for _ in range(steps):
            fn()
        c.record(e1)
        ms = c.elapsed_ms(e0, e1)
        c.sync()
        launches = c.launch_count() - l0
        barrier()
        if dist is not None:
            ms = D.max_over_ranks(ms, dist, tdev)
        c.event_destroy(e0); c.event_destroy(e1)
        return ms, launches

    # ------------------------------------------------------------------ headline: bf16 8192^3 per GPU, HBM-resident
    a = TensorHandle.empty_contiguous(c, [N_MM, N_MM], "bf16")
    b = TensorHandle.empty_contiguous(c, [N_MM, N_MM], "bf16")
    o = TensorHandle.empty_contiguous(c, [N_MM, N_MM], "bf16")
    c.fill_uniform(a.handle, "bf16", N_MM * N_MM, 3 + 100 * e.rank, -1.0, 1.0)
    c.fill_uniform(b.handle, "bf16", N_MM * N_MM, 4 + 100 * e.rank, -1.0, 1.0)

    def mm_step():
        matmul.launch(c, a, b, o)

    clocks = None
    for attempt in range(2):
        with ClockSampler(e.local_rank) as cs:
            ms, launches = timed(mm_step, args.steps, args.warmup)
        clocks = cs.summary()
        if not rejected(clocks):
            break
        clocks["remeasured"] = True
    c.flush()
    mm_kernel = c.last_kernel()                       # the entry point the timed launches ran (reported, not assumed)
    if args.dump_outputs:                             # before the rows below overwrite `o`
        dump_headline(c, o, e.rank, world, args.dump_outputs)
    value = world * FLOPS_MM * args.steps / (ms * 1e-3) / 1e12
    per_launch_ms = ms / args.steps
    per_gpu_tflops = FLOPS_MM / (per_launch_ms * 1e-3) / 1e12
    traffic = ncu_traffic()

    line = {
        "metric": "bf16_matmul_tflops", "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_launch_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"bf16 matmul 8192x8192x8192 per GPU (f32 accumulate, bf16 out), batch [{world},8192,8192] sharded over the batch axis",
                   "parallelism": f"batch-shard x{world}, no data-path collective",
                   "l2": "inputs_larger_than_L2 (A+B+C = 384 MiB per GPU vs 126 MB L2)", "rhs_layout": "row-major [K,N]"},
        "gpu_launches": launches * world,
        "roofline": {"bound": "tensor", "achieved": per_gpu_tflops, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": per_gpu_tflops / pk["bf16_tflops"], "traffic": traffic.get("gemm_bf16_8192_dram_bytes"),
                     "traffic_source": "static: dram__bytes_read+write of this kernel from the committed ncu --set full capture (profiles/traffic.json), not observed by this run",
                     "peak_source": pk["source"] + " (cuBLAS bf16 burst)", "kernel": mm_kernel,
                     "algorithmic_flops_per_launch": FLOPS_MM},
        "clocks": clocks,
    }

    # ------------------------------------------------------------------ context: the same kernel held for ~1 s (power-capped regime)
    if not args.quick:
        n_sus = max(200, int(1000.0 / per_launch_ms))
        with ClockSampler(e.local_rank) as cs2:
            ms_sus, _ = timed(mm_step, n_sus, 3)
        cl2 = cs2.summary()
        line["sustained"] = {"value": world * FLOPS_MM * n_sus / (ms_sus * 1e-3) / 1e12, "unit": "TFLOP/s", "launches": n_sus,
                             "seconds": ms_sus * 1e-3, "frac_of_sustained_peak": FLOPS_MM * n_sus / (ms_sus * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
                             "peak_sustained": pk["bf16_tflops_sustained"], "clocks": cl2,
                             "note": "back-to-back launches for ~1 s: the 1 kW power cap pulls SM clocks to ~1.5 GHz (ncu: 1.53 GHz, tensor pipe 94 % active)"}

    # ------------------------------------------------------------------ e2e: host buffers through the public API
    nbytes = N_MM * N_MM * 2
    with near_gpu(e.local_rank):
        hab, hc = c.host_alloc(2 * nbytes), c.host_alloc(nbytes)     # A|B contiguous in pinned memory: one H2D per step
        hab.view(np.uint16)[:] = 0x3F80  # 1.0 in bf16 (contents do not change the work)

    # Pipelined through the public multi-stream API: H2D of step i+1 | matmul of step i | D2H of step i-1 run on three
    # streams over two device slots, ordered by events; every step still copies both operands in and the result out.
    s_h2d, s_d2h = c.create_stream(), c.create_stream()

    def make_slot():
        ab = c.empty(2 * nbytes)
        return (ab, TensorHandle.new_contiguous([N_MM, N_MM], ab.offset(0, nbytes), "bf16"),
                TensorHandle.new_contiguous([N_MM, N_MM], ab.offset(nbytes, nbytes), "bf16"),
                TensorHandle.empty_contiguous(c, [N_MM, N_MM], "bf16"))

    slots = [make_slot(), make_slot()]
    ev = [{k2: c.event() for k2 in ("h2d", "mm", "d2h")} for _ in range(2)]
    for sl in ev:                                  # prime the events so the first waits are satisfied
        c.record(sl["mm"]); c.record(sl["d2h"], s_d2h)

    def e2e_step(i):
        sab_, sa_, sb_, so_ = slots[i % 2]
        e_ = ev[i % 2]
        c.stream_wait_event(s_h2d, e_["mm"])          # slot's operands are free once its previous matmul finished
        c.write_async(sab_, hab, stream=s_h2d)        # both operands (256 MiB) in one copy
        c.record(e_["h2d"], s_h2d)
        c.stream_wait_event(None, e_["h2d"])
        c.stream_wait_event(None, e_["d2h"])          # slot's output was read back
        matmul.launch(c, sa_, sb_, so_)
        c.record(e_["mm"])
        c.stream_wait_event(s_d2h, e_["mm"])
        c.read_async(hc, so_.handle, stream=s_d2h)
        c.record(e_["d2h"], s_d2h)

    def e2e_run(steps):
        barrier()
        c.sync_stream(s_h2d); c.sync_stream(s_d2h)
        e0, e1 = c.event(), c.event()
        c.record(e0, s_h2d)
        for i in range(steps):
            e2e_step(i)
        c.record(e1, s_d2h)
        ms_ = c.elapsed_ms(e0, e1)
        c.sync_stream(s_h2d); c.sync_stream(s_d2h); c.sync()
        barrier()
        if dist is not None:
            ms_ = D.max_over_ranks(ms_, dist, tdev)
        return ms_

    e2e_steps = max(4, min(args.steps, 20))
    e2e_run(3)                                        # warm-up
    ms_e2e = e2e_run(e2e_steps)
    assert hc.view(np.uint16)[0] == 0x4600, "e2e result check failed"  # 8192 = sum of 8192 ones, exact in bf16
    line["e2e"] = {"value": world * FLOPS_MM * e2e_steps / (ms_e2e * 1e-3) / 1e12, "unit": "TFLOP/s",
                   "h2d_bytes_per_step": 2 * nbytes, "d2h_bytes_per_step": nbytes, "ms_per_step": ms_e2e / e2e_steps,
                   "api": "ComputeClient.write_async (A|B, one 256 MiB copy) + matmul.launch + read_async per step from pinned host buffers; 3 streams, 2 device slots, event-ordered"}
    if world > 1:
        # Why e2e scales worse than the kernel: the step is PCIe-bound (256 MiB in + 128 MiB out per GPU per step), and the
        # GPUs of a box share host memory / root complexes.  One rank copying alone vs every rank at once says how much.
        def copy_ms(h2d=True, d2h=False, reps=3):
            """device time of `reps` x (256 MiB H2D on one stream and / or 128 MiB D2H on the other, concurrently)"""
            c.sync_stream(s_h2d); c.sync_stream(s_d2h)
            evs = [c.event() for _ in range(4)]
            c.record(evs[0], s_h2d); c.record(evs[2], s_d2h)
            for _ in range(reps):
                if h2d:
                    c.write_async(slots[0][0], hab, stream=s_h2d)
                if d2h:
                    c.read_async(hc, slots[0][3].handle, stream=s_d2h)
            c.record(evs[1], s_h2d); c.record(evs[3], s_d2h)
            t = max(c.elapsed_ms(evs[0], evs[1]), c.elapsed_ms(evs[2], evs[3])) / reps
            for e_ in evs:
                c.event_destroy(e_)
            return t

        solo = duplex_solo = 0.0
        for r in range(world):
            barrier()
            if e.rank == r:
                solo = copy_ms(True, False)
                duplex_solo = copy_ms(True, True)
        barrier()
        conc = copy_ms(True, False)
        barrier()
        duplex = copy_ms(True, True)
        barrier()
        mx = lambda v: D.max_over_ranks(v, dist, tdev)  # noqa: E731
        solo, conc, duplex_solo, duplex = mx(solo), mx(conc), mx(duplex_solo), mx(duplex)
        line["e2e"]["pcie"] = {"h2d_gbs_one_rank_at_a_time": 2 * nbytes / (solo * 1e-3) / 1e9,
                               "h2d_gbs_all_ranks_at_once": 2 * nbytes / (conc * 1e-3) / 1e9,
                               "h2d_plus_d2h_ms_one_rank_at_a_time": duplex_solo, "h2d_plus_d2h_ms_all_ranks_at_once": duplex,
                               "note": "slowest rank, pinned NUMA-local host buffers.  A pipelined e2e step cannot be shorter than the "
                                       "concurrent 256 MiB H2D + 128 MiB D2H of one step (h2d_plus_d2h_ms_*): when every GPU of the box copies "
                                       "in both directions at once the host side (memory / root complexes) is the limiter, not the kernels"}
    c.destroy_stream(s_h2d); c.destroy_stream(s_d2h)
    del slots
    for h in (hab, hc):
        c.host_free(h)
    c.fill_uniform(a.handle, "bf16", N_MM * N_MM, 3 + 100 * e.rank, -1.0, 1.0)
    c.fill_uniform(b.handle, "bf16", N_MM * N_MM, 4 + 100 * e.rank, -1.0, 1.0)

    # ------------------------------------------------------------------ reduce: f32 sum of 2^28 (1 GiB), weak + strong
    red = {"metric": "f32_reduce_sum_gbs", "unit": "GB/s", "elements": N_RED}
    nbuf = 3                                                 # rotate 3 x 1 GiB so nothing survives in the 126 MB L2
    xs = [TensorHandle.empty_contiguous(c, [N_RED], "f32") for _ in range(nbuf)]
    for i, x in enumerate(xs):
        c.fill_uniform(x.handle, "f32", N_RED, 5 + i + 10 * e.rank, 0.0, 1.0)
    r_out = TensorHandle.empty_contiguous(c, [1], "f32")
    k = [0]
    ids = list(range(world))
    if world > 1:
        uid = D.exchange_unique_id(c.get_unique_id, dist)
        c.ensure_init_collective(ids, uid)

    def red_local():
        k[0] += 1
        reduce.launch(c, xs[k[0] % nbuf], r_out, None, "sum")

    rsteps = max(args.steps, 20)
    ms_r, _ = timed(red_local, rsteps, args.warmup)
    red_kernel = c.last_kernel()
    gbs = BYTES_RED / (ms_r / rsteps * 1e-3) / 1e9
    red["kernel_only_per_gpu"] = gbs
    line["roofline_reduce"] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                               "traffic": traffic.get("reduce_sum_2p28_dram_bytes"),
                               "traffic_source": "static: committed ncu --set full capture (profiles/traffic.json)",
                               "peak_source": pk["source"] + " (copy, read+write)",
                               "kernel": red_kernel, "algorithmic_bytes_per_launch": BYTES_RED,
                               "note": "3 rotating 1 GiB inputs (nothing served from L2); consecutive launches on the stream overlap through "
                                       "programmatic dependent launch (the next launch streams while this one's last block finishes) -- "
                                       "reduce.pdl=off costs ~3 us per launch"}
    # argmax over the same 2^28 elements (north star: bit-exact argmax indices): its own roofline, same bytes
    a_out = TensorHandle.empty_contiguous(c, [1], "u32")

    def arg_local():
        k[0] += 1
        reduce.launch(c, xs[k[0] % nbuf], a_out, None, "argmax")

    ms_a, _ = timed(arg_local, rsteps, args.warmup)
    arg_kernel = c.last_kernel()
    gbs_a = BYTES_RED / (ms_a / rsteps * 1e-3) / 1e9
    line["roofline_argmax"] = {"bound": "hbm", "achieved": gbs_a, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs_a / pk["hbm_gbs"],
                               "traffic": None, "peak_source": pk["source"] + " (copy, read+write)", "kernel": arg_kernel,
                               "algorithmic_bytes_per_launch": BYTES_RED, "config": "argmax of 2^28 f32 (1 GiB), 3 rotating buffers"}
    parity = {}
    # exact-integer check of the headline reduce on every rank (BASELINE config 4 pattern: sum of i % 8 = 939,524,096)
    c.fill_modulo(xs[2].handle, "f32", N_RED, 8)
    reduce.launch(c, xs[2], r_out, None, "sum")
    reduce.launch(c, xs[2], a_out, None, "argmax")
    parity["reduce_2p28"] = {"sum": float(r_out.to_numpy(c)[0]), "expect": float(mod8_prefix_sum(N_RED)), "argmax": int(a_out.to_numpy(c)[0]), "argmax_expect": 7}
    parity["reduce_2p28"]["ok"] = parity["reduce_2p28"]["sum"] == parity["reduce_2p28"]["expect"] and parity["reduce_2p28"]["argmax"] == 7
    if world > 1:
        D.connect_p2p(c, dist)
        parity.update(multi_gpu_parity(c, D, dist, e, world, ids, xs, reduce, TensorHandle))
        parity.pop("ok", None)
        for i, x in enumerate(xs):                            # the parity patterns are not the timed data: restore it
            c.fill_uniform(x.handle, "f32", N_RED, 5 + i + 10 * e.rank, 0.0, 1.0)
    else:
        c.fill_uniform(xs[2].handle, "f32", N_RED, 5 + 2 + 10 * e.rank, 0.0, 1.0)
    if world > 1:
        def red_weak():                                       # 2^28 per GPU, local sum + all-reduce of one f32
            red_local()
            c.all_reduce(r_out.handle, r_out.handle, "f32", ids, "sum")
            c.sync_collective()

        ms_w, _ = timed(red_weak, rsteps, args.warmup)
        red["weak"] = {"value": world * BYTES_RED / (ms_w / rsteps * 1e-3) / 1e9, "ms_per_step": ms_w / rsteps,
                       "config": "2^28 f32 per GPU, outer-axis shard + NCCL all-reduce(4 B)"}
        lo, hi = D.shard_range(N_RED, world, e.rank)
        shard = TensorHandle(xs[0].handle.offset(lo * 4, (hi - lo) * 4), [hi - lo], [1], "f32")

        def red_strong():                                     # 2^28 total, 2^28/N per GPU
            reduce.launch(c, shard, r_out, None, "sum")
            c.all_reduce(r_out.handle, r_out.handle, "f32", ids, "sum")
            c.sync_collective()

        ms_s, _ = timed(red_strong, rsteps, args.warmup)
        red["strong"] = {"value": BYTES_RED / (ms_s / rsteps * 1e-3) / 1e9, "ms_per_step": ms_s / rsteps,
                         "config": "2^28 f32 total, contiguous outer-axis shards + NCCL all-reduce(4 B); latency-bound"}
        red["value"] = red["weak"]["value"]
        # fused: local reduce + exchange of the scalar through NVLink peer memory in ONE kernel (no NCCL on the data path)
        try:
            D.connect_p2p(c, dist)

            def red_weak_fused():
                k[0] += 1
                reduce.launch_all_reduce(c, xs[k[0] % nbuf], r_out, ids)

            ms_wf, _ = timed(red_weak_fused, rsteps, args.warmup)
            c.flush()
            red["weak_fused"] = {"value": world * BYTES_RED / (ms_wf / rsteps * 1e-3) / 1e9, "ms_per_step": ms_wf / rsteps,
                                 "config": "2^28 f32 per GPU, reduce + NVLink mailbox all-reduce fused in one kernel"}
            ms_sf, _ = timed(lambda: reduce.launch_all_reduce(c, shard, r_out, ids), rsteps, args.warmup)
            c.flush()
            # where the strong-scaled step goes: the kernel's own clock around the exchange (publish -> all peers seen) and
            # around the last block's grid stage, from a few extra launches with reduce.debug=1 (not the timed ones)
            c.set_option("reduce.debug", 1)
            xch = []
            for _ in range(8):
                reduce.launch_all_reduce(c, shard, r_out, ids)
                xch.append(c.reduce_debug())
            c.set_option("reduce.debug", 0)
            xch_us = float(np.median([w[0] for w in xch[2:]])) / 1e3
            stage_us = float(np.median([w[1] for w in xch[2:]])) / 1e3
            if dist is not None:
                xch_us = D.max_over_ranks(xch_us, dist, tdev)
            local_us = BYTES_RED / world / (gbs * 1e9) * 1e6
            red["strong_fused"] = {"value": BYTES_RED / (ms_sf / rsteps * 1e-3) / 1e9, "ms_per_step": ms_sf / rsteps,
                                   "config": "2^28 f32 total, 2^28/N per GPU, fused exchange",
                                   "exchange_us": xch_us, "grid_stage_us": stage_us, "local_stream_us_at_n1_rate": local_us,
                                   "limiter": "latency: per step = HBM stream of the shard + kernel ramp/tail + the exchange "
                                              "(exchange_us includes waiting for the slowest rank's launch, i.e. inter-process skew)"}
            red["value"] = max(red["value"], red["weak_fused"]["value"])
        except Exception as ex:  # noqa: BLE001
            red["fused_error"] = str(ex)
    else:
        red["value"] = gbs
    # reduce e2e at N=1 (1 GiB pinned H2D + 4 B D2H)
    if world == 1 and not args.quick:
        with near_gpu(e.local_rank):
            hx = c.host_alloc(BYTES_RED)
            hr = c.host_alloc(4)
        hx.view(np.float32)[:] = 1.0

        def red_e2e():
            c.write_async(xs[0].handle, hx)
            reduce.launch(c, xs[0], r_out, None, "sum")
            c.read_async(hr, r_out.handle)

        ms_re, _ = timed(red_e2e, 3, 1)
        assert hr.view(np.float32)[0] == float(N_RED)
        red["e2e"] = {"value": BYTES_RED / (ms_re / 3 * 1e-3) / 1e9, "unit": "GB/s", "h2d_bytes_per_step": BYTES_RED, "d2h_bytes_per_step": 4}
        c.host_free(hx); c.host_free(hr)
    del xs
    c.memory_cleanup()
    line["reduce"] = red

    # ------------------------------------------------------------------ other BASELINE configs (N-independent per GPU)
    def other_configs():
        if not args.quick:
            extra_steps = max(5, min(args.steps, 10))
            n4 = 4096
            # config 5: batched bf16, 8 x 4096^3 per GPU (B = 8N sharded over the batch axis)
            ab = TensorHandle.empty_contiguous(c, [8, n4, n4], "bf16")
            bb = TensorHandle.empty_contiguous(c, [8, n4, n4], "bf16")
            ob = TensorHandle.empty_contiguous(c, [8, n4, n4], "bf16")
            c.fill_uniform(ab.handle, "bf16", 8 * n4 * n4, 6 + 100 * e.rank, -1.0, 1.0)    # this rank's 8 batches of the global B = 8N
            c.fill_uniform(bb.handle, "bf16", 8 * n4 * n4, 7 + 100 * e.rank, -1.0, 1.0)
            ms_b, _ = timed(lambda: matmul.launch(c, ab, bb, ob), extra_steps, 3)
            ok_b, worst_b = check_matmul_samples(c, 6 + 100 * e.rank, 7 + 100 * e.rank, ob, (0, 3, 7), n4, np.random.default_rng(100 + e.rank))
            parity["batched_matmul"] = {"ok": ok_b, "worst_scaled_err": worst_b, "kernel": c.last_kernel(),
                                        "samples": "16 outputs in each of batches 0, 3, 7 of this rank's shard vs f64 dot products of host-regenerated operands"}
            line["batched_bf16_4096"] = {"value": world * 8 * 2.0 * n4 ** 3 * extra_steps / (ms_b * 1e-3) / 1e12, "unit": "TFLOP/s",
                                         "config": f"B={8 * world} x 4096^3 bf16, 8 batches per GPU, batch-axis shard, no collective"}
            del ab, bb, ob
            # config 2: f32 4096^3 on the tensor pipes: hybrid (default; tf32 product + two bf16 cross terms, ~2^-20), 3xTF32, plain tf32
            af = TensorHandle.empty_contiguous(c, [n4, n4], "f32")
            bf = TensorHandle.empty_contiguous(c, [n4, n4], "f32")
            of = TensorHandle.empty_contiguous(c, [n4, n4], "f32")
            c.fill_uniform(af.handle, "f32", n4 * n4, 1, -1.0, 1.0)
            c.fill_uniform(bf.handle, "f32", n4 * n4, 2, -1.0, 1.0)
            f32res = {}
            f32err = {}
            rng_f = np.random.default_rng(7)
            ms_i, ns_i = rng_f.integers(0, n4, 16), rng_f.integers(0, n4, 16)
            a_rows = np.stack([synth.uniform_f32(1, n4, -1.0, 1.0, start=int(m) * n4) for m in ms_i]).astype(np.float64)
            b_cols = np.stack([synth.uniform_at(2, np.arange(n4, dtype=np.uint64) * n4 + int(cc), -1.0, 1.0) for cc in ns_i]).astype(np.float64)
            f64_s, abs_s = a_rows @ b_cols.T, np.abs(a_rows) @ np.abs(b_cols).T
            for mode in ("hybrid", "3xtf32", "tf32"):
                c.set_option("gemm.f32", mode)
                ms_f, _ = timed(lambda: matmul.launch(c, af, bf, of), extra_steps, 3)
                f32res[mode] = world * 2.0 * n4 ** 3 * extra_steps / (ms_f * 1e-3) / 1e12
                got_s = of.to_numpy(c)[np.ix_(ms_i, ns_i)].astype(np.float64)
                f32err[mode] = float(np.max(np.abs(got_s - f64_s) / abs_s))
            c.set_option("gemm.f32", "hybrid")
            line["matmul_f32_4096"] = {"unit": "TFLOP/s (f32-equivalent 2*N^3)", "hybrid_default": f32res["hybrid"], "3xtf32": f32res["3xtf32"],
                                       "tf32": f32res["tf32"], "max_err_over_sum_abs_256_samples": f32err}
            parity["matmul_f32_4096"] = {"ok": bool(f32err["hybrid"] <= 1e-5 and f32err["3xtf32"] <= 1e-5 and f32err["tf32"] <= 1e-3),
                                         "worst_scaled_err": f32err}
            del af, bf, of
            # widening row (SURVEY 8f-4): fp8 e4m3 8192^3 -> bf16 on the same kernel (kind::f8f6f4)
            a8 = TensorHandle.empty_contiguous(c, [N_MM, N_MM], "f8e4m3")
            b8 = TensorHandle.empty_contiguous(c, [N_MM, N_MM], "f8e4m3")
            c.fill_uniform(a8.handle, "f8e4m3", N_MM * N_MM, 8, -1.0, 1.0)
            c.fill_uniform(b8.handle, "f8e4m3", N_MM * N_MM, 9, -1.0, 1.0)
            ms_8, _ = timed(lambda: matmul.launch(c, a8, b8, o), extra_steps, 3)
            line["matmul_fp8_8192"] = {"value": world * FLOPS_MM * extra_steps / (ms_8 * 1e-3) / 1e12, "unit": "TFLOP/s",
                                       "config": "fp8 e4m3 x e4m3 -> bf16, f32 accumulate, 8192^3 per GPU"}
            # same box, same operands: the 512x256 pair tile vs the 256x256 double-accumulator tile (bf16: auto picks the
            # former; fp8: forced, to decide its default)
            c.set_option("gemm.variant", "2sm_n256")
            ms_bn, _ = timed(mm_step, extra_steps, 3)
            ms_8n, _ = timed(lambda: matmul.launch(c, a8, b8, o), extra_steps, 3)
            c.set_option("gemm.variant", "auto")
            line["tile_variants_8192"] = {"unit": "TFLOP/s", "bf16_2sm_n256": world * FLOPS_MM * extra_steps / (ms_bn * 1e-3) / 1e12,
                                          "fp8_2sm_n256": world * FLOPS_MM * extra_steps / (ms_8n * 1e-3) / 1e12,
                                          "note": "gemm.variant forced to the 256x256 double-accumulator tile; the headline and matmul_fp8_8192 (auto) run the 512x256 pair tile 2sm_m512"}
            # widening row (SURVEY 8f-4): block-scaled MX formats -- tcgen05 kind::mxf8f6f4 / kind::mxf4, ue8m0 scale per 32 K,
            # row-major scales as the reference's scaled MMA takes them (the two packing passes run inside the timed call)
            import numpy as _np
            sc = TensorHandle.from_numpy(c, _np.full((N_MM, N_MM // 32), 127, _np.uint8), "ue8m0")
            ms_m8, _ = timed(lambda: matmul.launch_scaled(c, a8, b8, sc, sc, o), extra_steps, 3)
            a4 = TensorHandle(a8.handle, [N_MM, N_MM // 2], [N_MM // 2, 1], "f4e2m1x2")   # the same bytes read as packed e2m1
            b4 = TensorHandle(b8.handle, [N_MM, N_MM // 2], [N_MM // 2, 1], "f4e2m1x2")
            ms_m4, _ = timed(lambda: matmul.launch_scaled(c, a4, b4, sc, sc, o), extra_steps, 3)
            # NVFP4: the same packed e2m1 operands with an e4m3 scale byte per 16 elements of K (kind::mxf4nvf4)
            sc16 = TensorHandle.from_numpy(c, _np.full((N_MM, N_MM // 16), 0x38, _np.uint8), "f8e4m3")
            ms_nv, _ = timed(lambda: matmul.launch_scaled(c, a4, b4, sc16, sc16, o, scale_block=16), extra_steps, 3)
            line["matmul_block_scaled_8192"] = {
                "unit": "TFLOP/s", "mxfp8_e4m3": world * FLOPS_MM * extra_steps / (ms_m8 * 1e-3) / 1e12,
                "mxfp4_e2m1": world * FLOPS_MM * extra_steps / (ms_m4 * 1e-3) / 1e12,
                "nvfp4_e2m1": world * FLOPS_MM * extra_steps / (ms_nv * 1e-3) / 1e12,
                "kernel": c.last_kernel(),
                "config": "8192^3 per GPU -> bf16, row-major scales for both operands (ue8m0 per 32 elements of K; nvfp4: e4m3 per 16), the two "
                          "scale-packing passes run inside the timed call; scale atoms reach TMEM through the dedicated copy thread"}
            del a8, b8, a4, b4, sc, sc16
            # what CubeCL's own kernels reach on this GPU (hand-written from its emit rules; SURVEY 8d)
            if world == 1:
                scratch = c.empty(1024)
                ops = [0.0]

                def wm():
                    ops[0] = c.probe_wmma("bf16", 2048, scratch)

                ms_p, _ = timed(wm, 5, 2)
                uops = [0.0]

                def um():
                    uops[0] = c.probe_umma(8192, scratch)

                ms_u, _ = timed(um, 5, 2)
                buf = c.empty(512 << 20)
                c.fill_modulo(buf, "f32", (512 << 20) // 4, 8)
                ms_m, _ = timed(lambda: c.probe_memread(buf, 512 << 20, scratch), 10, 2)
                line["tcgen05_probe_tflops"] = uops[0] * 5 / (ms_u * 1e-3) / 1e12
                line["reference_equivalent"] = {"wmma_bf16_probe_tflops": ops[0] * 5 / (ms_p * 1e-3) / 1e12,
                                                "vec4_read_probe_gbs": (512 << 20) * 10 / (ms_m * 1e-3) / 1e9,
                                                "note": "compute_cmma.rs / memory_read.rs kernels as CubeCL would JIT them for sm_100a (wmma, 128-bit loads)"}
                del buf

    try:
        other_configs()
    except Exception as ex:  # noqa: BLE001  (secondary rows must never cost the headline line)
        line["secondary_error"] = repr(ex)
        try:
            c.flush()
        except Exception:  # noqa: BLE001
            pass

    # ------------------------------------------------------------------ parity object (every rank checks its own shard; all must agree)
    try:
        matmul.launch(c, a, b, o)
        ok_h, worst_h = check_matmul_samples(c, 3 + 100 * e.rank, 4 + 100 * e.rank, o, (0,), N_MM, np.random.default_rng(7 + e.rank), samples=24)
        parity["headline_matmul"] = {"ok": ok_h, "worst_scaled_err": worst_h, "samples": "24 outputs of this rank's 8192^3 product vs f64 dot products"}
    except Exception as ex:  # noqa: BLE001
        parity["headline_matmul"] = {"ok": False, "error": repr(ex)}
    local_ok = all(v.get("ok", False) for v in parity.values()) and "secondary_error" not in line
    parity["ok"] = all_ranks_ok(local_ok, dist, tdev)
    parity["ranks_checked"] = world
    line["parity"] = parity

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1 only)
    if rank0 and world == 1:
        try:
            cb = cpu_matmul_sample(12.0)
            cb.pop("flops"); cb.pop("seconds")
            line["cpu_baseline"] = cb
            line["reduce"]["cpu_baseline"] = cpu_reduce_sample()
        except Exception as ex:  # noqa: BLE001
            line["cpu_baseline"] = {"error": str(ex)}
    try:
        c.sync()
    except Exception as ex:  # noqa: BLE001  (a fault in a secondary row must not cost the measured headline)
        line["final_sync_error"] = repr(ex)
    if rank0:
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if not line["parity"]["ok"]:
        sys.stderr.write("bench.py: PARITY FAILURE: " + json.dumps(line["parity"]) + "\n")
        sys.exit(1)                      # a wrong result (on any rank) or a broken secondary row is not a benchmark result


if __name__ == "__main__":
    main()
