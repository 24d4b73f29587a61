#!/usr/bin/env python
"""bench.py -- SSA events/sec and ABC sims/sec of the B200 backend, one rank per GPU.

A "step" is one pass of the hot path over one batch of replicates.  The default line is BASELINE.json
configs[1] (C2: b1=1.5, grow 1 cell with 1 copy to 1e6 cells, 1e4 replicates per GPU, final ecDNA
distribution + mean/frequency/entropy; weak scaling) and carries, next to it:
  "abc"     the metric's second half: BASELINE configs[3] (C4) at FULL size - 1e6 prior draws over
            (b1, d0, d1), 1e5-cell birth-death runs, distances + accept fused in the kernel epilogue -
            STRONG-scaled over the ranks, accepted draws packed on the device and all-gathered by the
            library over NCCL; with its own roofline, cpu_baseline and e2e;
  "strong"  C2, C3, C5 strong-scaled over the ranks (their 1e4 / 1e4 / 1e3 replicates in total).

  python bench.py [--gpus N] [--steps K] [--warmup W]                 # this framework
  python bench.py --workload C4                                       # the ABC line on its own
  python bench.py --impl reference [--gpus N] --steps K --warmup W    # CPU restatement, all host cores
  python bench.py --dump-outputs DIR                                  # + the last timed step's results as DIR/*.npy

Every step simulates a different index range, so nothing is reused; a 256 MiB buffer is rewritten
before every step (L2 flush).  The index ranges and seeds depend on the arguments only, so two builds run
with the same arguments can be compared output for output with --dump-outputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (SimulationOptions kwargs, replicates, description)
    "C1": (dict(b0=1.0, b1=1.0, cells=100_000), 100, "neutral, 1e5 cells, 100 replicates"),
    "C2": (dict(b0=1.0, b1=1.5, cells=1_000_000), 10_000, "b1=1.5, 1e6 cells, 1e4 replicates, final distribution + mean/frequency/entropy"),
    "C3": (dict(b0=1.0, b1=1.2, d0=0.3, d1=0.3, cells=100_000), 10_000, "birth-death d0=d1=0.3 b1=1.2, 1e5 cells, 1e4 replicates, dynamics"),
    "C4": (dict(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=100_000), 1_000_000, "ABC: 1e6 prior draws b1~U(1,2), d0,d1~U(0,0.5), 1e5-cell birth-death runs, target = run at (1.4,0.2,0.2)"),
    "C5": (dict(b0=1.0, b1=1.0, cells=10_000_000, initial={50: 1}), 1_000, "neutral, k0=50, 1e7 cells, 1e3 replicates"),
}
WANT = ("stop_reason", "nminus", "nplus", "time", "n_events", "kmax", "mean", "frequency", "entropy", "variance",
        "hist")
ABC_THRESHOLDS = (0.05, 0.1, 0.1, 0.1)
ABC_BINS = 256
DUMP_BYTES = 64_000_000  # --dump-outputs: all files together, .npy headers included


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--replicates", type=int, default=0, help="replicates per GPU per step (0 = the config's)")
    ap.add_argument("--tile-width", type=int, default=0)
    ap.add_argument("--smem-bins", type=int, default=0)
    ap.add_argument("--state", default="auto", choices=["auto", "smem", "hbm"])
    ap.add_argument("--slice-events", type=lambda v: int(v, 0), default=0,
                    help="time-slice length in events (0 = automatic, 0xFFFFFFFF = never)")
    ap.add_argument("--abc-draws", type=int, default=1_000_000, help="prior draws of the ABC leg, in total over all ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-abc", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (at most 64 MB)")
    return ap.parse_args()


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.proc, self.lines = gpu, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU legs: the reference-layout C++ restatement (oracle/), the only place bench.py executes oracle code
# ------------------------------------------------------------------------------------------------
def _oracle_opts(m, ob, kw, seed=26, fast=True):
    o = m.SimulationOptions(save_snapshots=False, seed=seed, **kw)
    return o, ob.make_opts(b0=o.b0, b1=o.b1, d0=o.d0, d1=o.d1, segregation=o.segregation, state=ob.STATE_VECTOR,
                           rng=ob.RNG_RAND, max_cells=o.max_cells, max_time=float(o.years), seed=o.seed,
                           initial=o.distribution)


def cpu_port(workload, seconds, n_threads=0, idx0=260):
    """The CPU restatement of the reference (per-cell vector state, ChaCha8, ziggurat, BINV/BTPE),
    replicates over all host threads with a dynamic queue (rayon par_iter, main.rs:221-224), built as its own
    -O3 -march=native target (oracle/Makefile: libecdna_oracle_fast.so)."""
    import _pkg
    import oracle_binding as ob
    m = _pkg.load()
    ob.use_fast_build()
    kw = WORKLOADS[workload][0]
    o, oo = _oracle_opts(m, ob, kw)
    cores = n_threads or os.cpu_count() or 1
    if workload == "C4":
        return cpu_abc(m, ob, o, oo, seconds, cores)
    # calibrate with one replicate per thread, then size the sample for ~`seconds`
    t0 = time.perf_counter()
    r = ob.run_batch(oo, idx0, cores, cores)
    t1 = time.perf_counter() - t0
    n = int(max(cores, min(cores * 4096, cores * seconds / max(t1, 1e-3))))
    t0 = time.perf_counter()
    r = ob.run_batch(oo, idx0 + cores, n, cores)
    dt = time.perf_counter() - t0
    return {"events": int(r.total_events), "seconds": dt, "replicates": n, "cores": cores,
            "events_per_sec": r.total_events / dt, "sims_per_sec": n / dt}


def abc_priors_numpy(n, seed=12345):
    """Synthetic C4 priors for the CPU leg (same shape as the device's Philox draws): b1~U(1,2), d0,d1~U(0,0.5)."""
    rng = np.random.default_rng(seed)
    r = np.empty((n, 4), dtype=np.float32)
    r[:, 0] = 1.0
    r[:, 1] = rng.uniform(1.0, 2.0, n)
    r[:, 2] = rng.uniform(0.0, 0.5, n)
    r[:, 3] = rng.uniform(0.0, 0.5, n)
    return r


def cpu_abc(m, ob, o, oo, seconds, cores, draws=None):
    """C4 on the CPU: prior draws -> reference-layout replicates -> the four distances + accept per draw."""
    target = ob.run(ob.make_opts(b0=o.b0, b1=o.b1, d0=o.d0, d1=o.d1, state=ob.STATE_HIST, rng=ob.RNG_PHILOX,
                                 max_cells=o.max_cells, max_time=float(o.years), seed=o.seed, run_idx=260),
                    hist_cap=512).hist
    if draws is None:
        probe = 8 * cores
        t0 = time.perf_counter()
        ob.abc_batch(oo, 10_000_000, probe, abc_priors_numpy(probe, 1), target, ABC_THRESHOLDS, cores)
        t1 = max(time.perf_counter() - t0, 1e-3)
        draws = int(max(1000, min(200_000, probe * seconds / t1)))
    rates = abc_priors_numpy(draws)
    idx0 = 20_000_000
    t0 = time.perf_counter()
    r = ob.abc_batch(oo, idx0, draws, rates, target, ABC_THRESHOLDS, cores)
    dt = time.perf_counter() - t0
    return {"events": int(r.total_events), "seconds": dt, "replicates": draws, "cores": cores,
            "events_per_sec": r.total_events / dt, "sims_per_sec": draws / dt, "accepted": int(r.accept.sum()),
            "batch": r, "rates": rates, "first_index": idx0}


def reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on all host cores.  The Rust
    binary cannot be built in this image (no cargo, crates not vendored), so this times the
    reference-layout C++ restatement (oracle/), each step a bounded sample of the same workload."""
    if rank != 0:
        return
    import _pkg
    import oracle_binding as ob
    m = _pkg.load()
    ob.use_fast_build()
    kw, reps, desc = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    o, oo = _oracle_opts(m, ob, kw)
    abc = args.workload == "C4"
    per_step = max(1.0, min(15.0, 100.0 / max(1, args.steps + args.warmup)))
    if abc:
        c = cpu_abc(m, ob, o, oo, per_step, cores)  # calibration pass; its size is the step size
        n = c["replicates"]
        step = lambda i: cpu_abc(m, ob, o, oo, per_step, cores, draws=n)  # noqa: E731
    else:
        t0 = time.perf_counter()
        ob.run_batch(oo, 100, cores, cores)  # calibration: one replicate per thread
        t1 = max(time.perf_counter() - t0, 1e-3)
        n = int(max(cores, min(reps, cores * per_step / t1)))

        def step(i):
            t0 = time.perf_counter()
            r = ob.run_batch(oo, o.idx_begin + i * n, n, cores)
            return {"events": int(r.total_events), "seconds": time.perf_counter() - t0, "batch": r,
                    "first_index": o.idx_begin + i * n}
    for w in range(args.warmup):
        step(w)
    events, tot_t = 0, 0.0
    for s in range(args.steps):
        r = step(args.warmup + s)
        tot_t += r["seconds"]
        events += r["events"]
    if args.dump_outputs:
        b = r["batch"]
        cols = ("distance", "accept", "n_events", "stop") if abc else ("stop", "nminus", "nplus", "time", "n_events")
        rows = {c: (getattr(b, c), getattr(b, c).dtype) for c in cols}
        if abc:
            rows["prior_rates"] = (r["rates"], np.float32)
        dump_outputs(args.dump_outputs, rows, r["first_index"])
    metric, unit = ("abc_sims_per_sec", "sims/s") if abc else ("ssa_events_per_sec", "events/s")
    v = (n * args.steps / tot_t) if abc else events / tot_t
    sample = (f"{n} {'prior draws' if abc else 'replicates'} of {args.workload} per step over {cores} host threads "
              "(reference-layout C++ restatement: per-cell u16 vector, ChaCha8, ziggurat, BINV/BTPE, -O3 -march=native; "
              "the Rust reference cannot be built here)")
    line = {
        "impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps,
        "higher_is_better": True, "scaling": "strong" if abc else "weak", "vs_baseline": None, "dtype": "u32",
        "data": "synthetic", "config": {"workload": f"{args.workload}: {desc}", "replicates_per_step": n},
        "events_per_sec": events / tot_t,
        "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# the GPU legs
# ------------------------------------------------------------------------------------------------
class Env:
    pass


def setup(args):
    import torch
    import torch.distributed as dist
    import _pkg
    e = Env()
    e.torch, e.dist = torch, dist
    e.rank = int(os.environ.get("RANK", "0"))
    e.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    e.world = int(os.environ.get("WORLD_SIZE", "1"))
    e.m = m = _pkg.load()
    if e.local_rank == 0:
        m.build()  # no-op when the prebuilt library matches the sources; only one rank may ever compile
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: libecdna_b200.so has no CPU path")
    torch.cuda.set_device(e.local_rank)
    e.dev = torch.device("cuda", e.local_rank)
    if e.world > 1:
        dist.init_process_group("nccl", device_id=e.dev)
        dist.barrier()  # the library is in place before any rank loads it
    e.ctx = m.Context(e.local_rank)
    if e.world > 1:
        # the library's own communicator (NCCL over NVLink) for the one exchange step of the path; the
        # 128-byte id travels through the launcher's process group
        ident = torch.zeros(m.COMM_ID_BYTES, dtype=torch.uint8, device=e.dev)
        if e.rank == 0:
            ident = torch.tensor(list(m.comm_unique_id()), dtype=torch.uint8, device=e.dev)
        dist.broadcast(ident, 0)
        e.ctx.comm_init(bytes(ident.cpu().numpy().tobytes()), e.rank, e.world)
    # one explicit stream for everything that is timed (the legacy default stream is the NULL handle, which the
    # library reads as "use the context's own stream")
    e.tstream = torch.cuda.Stream(e.dev)
    torch.cuda.set_stream(e.tstream)
    e.stream = e.tstream.cuda_stream
    assert e.stream != 0
    e.flush = torch.empty(256 << 20, dtype=torch.uint8, device=e.dev)  # > 126 MB L2
    e.state_mode = {"auto": m.STATE_AUTO, "smem": m.STATE_SMEM, "hbm": m.STATE_HBM}[args.state]
    return e


def barrier(e):
    if e.world > 1:
        e.dist.barrier()
    e.torch.cuda.synchronize(e.dev)


def reduce_max_sum(e, ms, count):
    t = e.torch.tensor([ms], dtype=e.torch.float64, device=e.dev)
    c = e.torch.tensor([float(count)], dtype=e.torch.float64, device=e.dev)
    if e.world > 1:
        e.dist.all_reduce(t, op=e.dist.ReduceOp.MAX)
        e.dist.all_reduce(c, op=e.dist.ReduceOp.SUM)
    return float(t.item()), float(c.item())


def gather_floats(e, x):
    """One float per rank, on every rank (diagnostics: which rank set the max)."""
    t = e.torch.tensor([float(x)], dtype=e.torch.float64, device=e.dev)
    if e.world == 1:
        return [float(x)]
    parts = [e.torch.zeros_like(t) for _ in range(e.world)]
    e.dist.all_gather(parts, t)
    return [float(p.item()) for p in parts]


def dump_outputs(d, rows, first_index, extra=None, rank=0, world=1):
    """--dump-outputs: result columns as DIR/<name>.npy, floats as float32, integers as float64 (exact below 2**53).
    `rows` maps a name to (tensor or array, numpy dtype of its elements); row i of every column belongs to
    replicate (or prior draw) first_index + i, and replicate_index.npy holds that index for each row written.
    Columns that would exceed DUMP_BYTES together are cut to the same fixed, seeded sample of rows, in index
    order.  `extra` (host arrays written whole) counts against the same budget.  With several ranks, rank r
    writes DIR/rank<r>/."""
    if world > 1:
        d = os.path.join(d, f"rank{rank}")
    os.makedirs(d, exist_ok=True)
    extra = {k: np.asarray(v) for k, v in (extra or {}).items()}
    extra = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in extra.items()}
    n = len(next(iter(rows.values()))[0])

    def row_bytes(x, dtype):
        return int(np.prod(x.shape[1:], dtype=np.int64)) * (4 if np.dtype(dtype) == np.float32 else 8)
    per_row = 8 + sum(row_bytes(x, dt) for x, dt in rows.values())
    budget = DUMP_BYTES - sum(v.nbytes for v in extra.values()) - 4096 * (len(rows) + len(extra) + 1)  # headers
    keep = np.arange(n)
    if per_row * n > budget:
        keep = np.sort(np.random.default_rng(0).choice(n, max(budget // per_row, 1), replace=False))
    out = dict(extra, replicate_index=(first_index + keep).astype(np.float64))
    for name, (x, dtype) in rows.items():
        if hasattr(x, "index_select"):  # a torch tensor: sample on its device, then copy
            import torch
            x = x.index_select(0, torch.from_numpy(keep).to(x.device)).cpu().numpy()
        else:
            x = np.asarray(x)[keep]
        x = x.view(dtype)
        out[name] = x if x.dtype in (np.float32, np.float64) else x.astype(np.float64)
    for name, x in out.items():
        np.save(os.path.join(d, name + ".npy"), x)


def result_dtypes(m):
    return {name: dtype for name, dtype, _ in m.RESULT_FIELDS}


def oracle_check(e, opts, tensors, idx0, picks, dyn=None):
    """Replicates of the batch that was just timed against the CPU oracle (the specification of the native
    stream), bit for bit: stop reason, counts, events, f32 clock bits, final distribution.  Outside the timed
    region.  This is the checker, not the thing measured."""
    import oracle_binding as ob
    m = e.m
    ok, checked = True, []
    host = {k: v[picks].cpu().numpy() for k, v in tensors.items() if k in ("stop_reason", "nminus", "nplus", "time", "n_events", "kmax", "hist", "dyn", "dyn_count")}
    for j, i in enumerate(picks):
        kw = dict(dyn_points=dyn["dyn_points"], dyn_dt=dyn["dyn_dt"]) if dyn else {}
        oo = ob.make_opts(b0=opts.b0, b1=opts.b1, d0=opts.d0, d1=opts.d1, segregation=opts.segregation,
                          state=ob.STATE_HIST, rng=ob.RNG_PHILOX, max_cells=opts.max_cells, max_time=float(opts.years),
                          seed=opts.seed, run_idx=idx0 + int(i), initial=opts.distribution, **kw)
        ref = ob.run(oo, hist_cap=host["hist"].shape[1])
        same = (int(host["stop_reason"][j]) & 0xFF) == ref.stop_reason and int(host["n_events"][j]) == ref.n_events
        same = same and int(host["nminus"][j]) == ref.nminus and int(host["nplus"][j]) == ref.nplus
        same = same and np.float32(host["time"][j]).view(np.uint32) == np.float32(ref.time).view(np.uint32)
        same = same and int(host["kmax"][j]) == ref.kmax
        same = same and np.array_equal(host["hist"][j].astype(np.int64) & 0xFFFFFFFF, ref.hist.astype(np.int64))
        if dyn and same:
            n = ref.dyn_count
            same = int(host["dyn_count"][j]) == n and np.array_equal(host["dyn"][j][:n].view(np.uint32), ref.dyn[:n].view(np.uint32))
        ok = ok and bool(same)
        checked.append(int(idx0 + int(i)))
    del m
    return {"bit_exact_vs_oracle": ok, "replicate_indices": checked}


def ssa_leg(e, args, workload, reps, steps, warmup, idx_base, check=0, sample_clocks=False):
    """`steps` timed passes of `reps` replicates of `workload` on this rank; returns the measurements."""
    m, torch = e.m, e.torch
    kw, _, desc = WORKLOADS[workload]
    opts = m.SimulationOptions(save_snapshots=False, runs=reps, **kw)
    stride = 512
    dyn = dict(dyn_points=300, dyn_dt=0.1) if workload == "C3" else {}
    want = WANT + (("dyn", "dyn_count") if dyn else ())
    knobs = dict(tile_width=args.tile_width, smem_bins=args.smem_bins, state_mode=e.state_mode, hist_stride=stride,
                 slice_events=args.slice_events, **dyn)
    res_struct, tensors = m.device_results(torch, reps, want + ("sum_k", "n_div", "n_death"),
                                           dyn_points=dyn.get("dyn_points", 0), hist_stride=stride, device=e.dev)

    def step(i):
        # every step and every rank simulates its own index range
        idx0 = idx_base + i * 10_000_000
        e.flush.zero_()
        e.ctx.run_device(opts, reps, idx0, res_struct, stream=e.stream, **knobs)
        return idx0

    for i in range(warmup):
        step(i)
    barrier(e)
    sampler = None
    if sample_clocks:
        sampler = ClockSampler(e.local_rank)
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    events = alg_bytes = 0
    kernel_ms = []
    barrier(e)
    e0.record()
    last_idx0 = 0
    for i in range(steps):
        last_idx0 = step(warmup + i)
        # per-launch kernel time from the library's own CUDA events on the launching stream
        t = e.ctx.timing()
        kernel_ms.append(t.kernel_ms)
        events += t.total_events
        alg_bytes += t.alg_bytes
    e1.record()
    barrier(e)
    ms = e0.elapsed_time(e1)
    out = Env()
    out.clocks = sampler.stop() if sampler else None
    out.last = e.ctx.timing()
    out.ms_all, out.events_all = reduce_max_sum(e, ms, events)
    out.ms_per_rank = gather_floats(e, ms / steps)
    out.kernel_ms_per_rank = gather_floats(e, float(np.mean(kernel_ms)))
    out.value = out.events_all / (out.ms_all * 1e-3)
    out.events, out.alg_bytes, out.kernel_ms, out.steps = events, alg_bytes, float(np.mean(kernel_ms)), steps
    out.opts, out.knobs, out.want, out.desc, out.reps = opts, knobs, want, desc, reps
    out.tensors, out.last_idx0 = tensors, last_idx0
    out.kmax = int(tensors["kmax"].max().item())
    # ---- what was simulated, outside the timed region: invariants on every replicate of the last step ... ----
    stops = tensors["stop_reason"].cpu().numpy() & 0xFF
    cells = (tensors["nminus"] + tensors["nplus"]).cpu().numpy()
    inv = bool(np.all(tensors["hist"].sum(dim=1).cpu().numpy() == cells))
    if not opts.birth_death:
        inv = inv and bool(np.all(stops == m.STOP_MAX_CELLS) and np.all(cells == opts.max_cells))
    out.results = {"invariants_ok": inv}
    # ---- ... and a real oracle comparison of `check` of its replicates ----
    if check:
        picks = sorted(set(int(x) for x in np.linspace(0, reps - 1, check)))
        out.results.update(oracle_check(e, opts, tensors, last_idx0, picks, dyn or None))
    return out


def pinned_alloc(torch):
    """Result columns in page-locked host memory (the caller owns its buffers; a pinned one copies at full speed)."""
    tmap = {np.uint32: torch.int32, np.uint64: torch.int64, np.float32: torch.float32, np.uint8: torch.uint8}
    keep = []

    def alloc(shape, dtype):
        t = torch.zeros(shape, dtype=tmap[dtype], pin_memory=True)
        keep.append(t)
        return t.numpy().view(dtype)
    alloc.keep = keep
    return alloc


def e2e_ssa(e, leg, steps, idx_base):
    """End to end through the host-buffer C ABI call (what a reference-side FFI caller sees): host buffers in
    and out (page-locked, reused from step to step), host<->device copies inside the timed region, every step."""
    ctx = e.ctx
    alloc = pinned_alloc(e.torch)
    host = e.m.Results(leg.reps, 0, leg.knobs.get("dyn_points", 0), leg.knobs["hist_stride"], leg.want, alloc=alloc)
    ctx.run(leg.opts, n_runs=leg.reps, idx_begin=idx_base, want=leg.want, results=host, **leg.knobs)  # library buffers
    barrier(e)
    t0 = time.perf_counter()
    ev2 = h2d = d2h = 0
    for i in range(steps):
        r = ctx.run(leg.opts, n_runs=leg.reps, idx_begin=idx_base + (i + 1) * 10_000_000, want=leg.want, results=host,
                    **leg.knobs)
        ev2 += int(r.n_events.sum())  # host read of the step's result
        h2d, d2h = r.timing.h2d_bytes, r.timing.d2h_bytes
    barrier(e)
    dt = time.perf_counter() - t0
    dt_all, n_all = reduce_max_sum(e, dt, ev2)
    return {"value": n_all / dt_all, "unit": "events/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "steps": steps, "api": "ecdna_b200_run (page-locked host buffers; copies inside the timed region)"}


def roofline_block(leg, workload, clocks):
    """SURVEY 8(d): the state lives in shared memory, so the binding resource of the SSA kernel is the SM's
    warp-instruction issue rate (bound "issue"); HBM is idle by design.  Reported: the issue fraction (primary),
    the flat-histogram model bandwidth the judge's formula asks for (hbm_model), and measured DRAM traffic."""
    peak, peak_src = measured_peak()
    k_ms = leg.kernel_ms
    alg_per_launch = leg.alg_bytes / leg.steps
    model_gbs = alg_per_launch / (k_ms * 1e-3) / 1e9
    traffic = inst_per_event = src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(workload)
        if tj and leg.last.tile_width == tj.get("tile_width"):
            traffic, inst_per_event, src = tj.get("bytes"), tj.get("warp_inst_per_event"), tj.get("source")
    except Exception:
        pass
    sm_hz = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
    issue_peak = 148 * 4 * sm_hz
    events_per_launch = leg.events / leg.steps
    r = {"bound": "issue", "unit": "Gwarp-inst/s", "peak": issue_peak / 1e9, "achieved": None, "frac": None,
         "traffic": traffic, "kernel": f"ssa_kernel<{leg.last.tile_width},smem>", "kernel_ms_per_launch": k_ms,
         "events_per_launch": events_per_launch,
         "hbm_model": {"achieved": model_gbs, "peak": peak, "unit": "GB/s", "frac": model_gbs / peak,
                       "peak_source": peak_src, "alg_bytes_per_launch": alg_per_launch,
                       "alg_bytes_per_event": leg.alg_bytes / max(leg.events, 1),
                       "note": "SURVEY 8(d) flat-histogram bytes (4K + 24 + 16 per division, K = kmax+1 at that "
                               "event) / kernel time: how fast a flat HBM histogram would have to stream to keep "
                               "up.  The histogram lives in shared memory; real DRAM traffic is `traffic` bytes "
                               "per launch (ncu, profiles/traffic.json)"},
         "note": "achieved = warp-instructions per event (STATIC: from the committed ncu capture of this launch "
                 "configuration, profiles/traffic.json) x events/s measured live; peak = 148 SMs x 4 schedulers x "
                 "the SM clock sampled during the run"}
    if inst_per_event:
        issued = inst_per_event * events_per_launch / (k_ms * 1e-3)
        r.update({"achieved": issued / 1e9, "frac": issued / issue_peak, "warp_inst_per_event": inst_per_event,
                  "source": src})
    return r


def abc_leg(e, args, draws_total, with_cpu, with_e2e, steps=1, warmup=3, dump=None):
    """BASELINE config 4 at full size, STRONG-scaled: rank r owns a contiguous block of the prior draws; priors
    drawn on the device, 1e5-cell birth-death runs, distances + accept in the kernel epilogue, accepted draws
    packed into records on the device and all-gathered by the library (two ncclAllGather in one group).
    The host waits once per pass, before the simulation is enqueued (run_device fetches the 2 KB target
    distribution to compute its statistics and CDF); simulation, packing and exchange then follow each other on
    the stream without any host synchronisation up to the final event.  `steps` timed passes over fresh prior
    draws follow `warmup` untimed ones; `dump` is the --dump-outputs directory for the last timed pass."""
    m, torch, ctx = e.m, e.torch, e.ctx
    kw, _, desc = WORKLOADS["C4"]
    opts = m.SimulationOptions(save_snapshots=False, runs=draws_total, **kw)
    # synthetic target: one run at the "true" parameters
    tgt = ctx.run(opts, n_runs=1, idx_begin=260, want=("hist",), hist_stride=512).hist[0].astype(np.uint64)
    tgt_d = torch.from_numpy(tgt.astype(np.int64)).to(e.dev)
    idx0, n = m.rank_range(opts.idx_begin, draws_total, e.rank, e.world)
    n_max = m.rank_range(opts.idx_begin, draws_total, 0, e.world)[1]
    want = ("stop_reason", "n_events", "nminus", "nplus", "kmax", "abc_distance", "abc_accept", "mean", "frequency",
            "entropy", "hist")
    rs, t = m.device_results(torch, n, want, hist_stride=ABC_BINS, device=e.dev)
    rates_d = torch.empty((n, 4), dtype=torch.float32, device=e.dev)
    cap = max(1024, n_max // 4)
    words = m.record_words(ABC_BINS)
    rec_d = torch.zeros((cap, words), dtype=torch.int32, device=e.dev)
    cnt_d = torch.zeros(1, dtype=torch.int32, device=e.dev)
    all_rec_d = torch.zeros((e.world, cap, words), dtype=torch.int32, device=e.dev) if e.world > 1 else rec_d
    all_cnt_d = torch.zeros(e.world, dtype=torch.int32, device=e.dev) if e.world > 1 else cnt_d
    kwr = dict(rates_per_run=rates_d, abc_target=tgt_d, abc_thresholds=ABC_THRESHOLDS, hist_stride=ABC_BINS,
               tile_width=args.tile_width, slice_events=args.slice_events)

    marks = [torch.cuda.Event(enable_timing=True) for _ in range(5)]

    def one_pass(count, shift):
        # priors -> simulation + fused epilogue -> pack -> all-gather; all enqueued on one stream
        e.flush.zero_()
        marks[0].record()
        ctx.abc_draw_priors_device(26, idx0 + shift, count, rates_d.data_ptr(), stream=e.stream)
        marks[1].record()
        ctx.run_device(opts, count, idx0 + shift, rs, stream=e.stream, **kwr)
        marks[2].record()
        ctx.abc_pack(rs, rates_d.data_ptr(), (opts.b0, opts.b1, opts.d0, opts.d1), idx0 + shift, count, ABC_BINS,
                     ABC_BINS, cap, rec_d.data_ptr(), cnt_d.data_ptr(), stream=e.stream)
        marks[3].record()
        if e.world > 1:
            ctx.abc_allgather(rec_d.data_ptr(), cnt_d.data_ptr(), ABC_BINS, cap, all_rec_d.data_ptr(),
                              all_cnt_d.data_ptr(), stream=e.stream)
        marks[4].record()

    # warm-up: one pass at full size (every library buffer reaches its final size: no allocation in the timed
    # passes), then reduced ones (kernels, the communicator)
    for w in range(warmup):
        one_pass(n if w == 0 else min(n, 32768), 500_000_000 + w * 2_000_000)
    barrier(e)
    sampler = ClockSampler(e.local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(e)
    events = 0
    e0.record()
    for s in range(steps):
        if s:  # the previous pass's events (the next run_device waits for the stream anyway)
            events += ctx.timing().total_events
        one_pass(n, s * draws_total)
    e1.record()
    barrier(e)
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    tm = ctx.timing()
    events += tm.total_events
    phases = {"priors_ms": marks[0].elapsed_time(marks[1]), "simulate_ms": marks[1].elapsed_time(marks[2]),
              "ssa_kernel_ms": tm.kernel_ms, "pack_ms": marks[2].elapsed_time(marks[3]),
              "allgather_ms": marks[3].elapsed_time(marks[4])}
    ms_all, events_all = reduce_max_sum(e, ms, events)
    counts = all_cnt_d.cpu().numpy().astype(np.int64)
    merged = m.merge_gathered(all_rec_d.cpu().numpy().view(np.uint32), counts, cap, ABC_BINS)
    rec = m.decode_records(merged, ABC_BINS)
    acc_local = int(t["abc_accept"].sum().item())
    stops = np.bincount(t["stop_reason"].cpu().numpy() & 0xFF, minlength=5)
    ok = bool(len(rec["idx"]) == counts.sum() and np.all(np.diff(rec["idx"].astype(np.int64)) > 0) and
              counts[e.rank] == acc_local and np.all(rec["distance"][:, 0] <= ABC_THRESHOLDS[0]))
    post = rec["rates"][:, 1:].mean(axis=0).tolist() if len(rec["idx"]) else None
    if dump:
        dt = result_dtypes(m)
        rows = {k: (v, dt[k]) for k, v in t.items()}
        rows["prior_rates"] = (rates_d, np.float32)
        dump_outputs(dump, rows, idx0 + (steps - 1) * draws_total, extra={"accepted_index": rec["idx"]},
                     rank=e.rank, world=e.world)

    leg = Env()
    leg.kernel_ms, leg.alg_bytes, leg.events, leg.steps, leg.last = tm.kernel_ms, tm.alg_bytes, tm.total_events, 1, tm
    out = {"metric": "abc_sims_per_sec", "value": draws_total * steps / (ms_all * 1e-3), "unit": "sims/s",
           "n_gpus": e.world, "scaling": "strong", "higher_is_better": True, "steps": steps, "warmup": warmup,
           "ms": ms_all / steps, "events_per_sec": events_all / (ms_all * 1e-3),
           "config": {"workload": f"C4: {desc}", "draws_total": draws_total, "draws_this_rank": n, "cells": opts.max_cells,
                      "thresholds": list(ABC_THRESHOLDS), "tile_width": tm.tile_width, "grid_blocks": tm.grid_blocks,
                      "record_words": words, "record_capacity_per_rank": cap,
                      "exchange": "ecdna_b200_abc_pack + ecdna_b200_abc_allgather (NCCL, 2 collectives in one group)"
                                  if e.world > 1 else "ecdna_b200_abc_pack (one rank: nothing to exchange)",
                      "l2": "256 MiB buffer rewritten before every pass"},
           "phases_this_rank": phases,
           "accepted_total": int(counts.sum()), "accepted_per_rank": counts.tolist(), "gather_ok": ok,
           "posterior_mean_b1_d0_d1": post, "stops_this_rank": stops.tolist(), "clocks": clocks,
           "gpu_launches": steps * (tm.kernel_launches + 8), "roofline": roofline_block(leg, "C4", clocks)}

    if with_e2e:
        # end to end through the host-buffer call: host prior draws in (16 B/draw), every draw's distances,
        # accept flag and summary out ("save all, filter later", abc.md:57-71), copies inside the timed region
        rates_h = ctx.abc_draw_priors(seed=26, idx_begin=idx0 + 700_000_000, n_runs=n)
        hw = ("stop_reason", "n_events", "nminus", "nplus", "abc_distance", "abc_accept", "mean", "frequency", "entropy")
        alloc = pinned_alloc(torch)
        host = m.Results(n, 0, 0, ABC_BINS, hw, alloc=alloc)
        rates_p = alloc(rates_h.shape, np.float32)
        rates_p[:] = rates_h
        kwh = dict(kwr, rates_per_run=rates_p, abc_target=tgt)
        ctx.run(opts, n_runs=n, idx_begin=idx0 + 600_000_000, want=hw, results=host, **kwh)  # library buffers at full size
        barrier(e)
        t0 = time.perf_counter()
        r = ctx.run(opts, n_runs=n, idx_begin=idx0 + 700_000_000, want=hw, results=host, **kwh)
        n_acc = int(r.abc_accept.sum())  # host read of the step's result
        barrier(e)
        dt = time.perf_counter() - t0
        dt_all, _ = reduce_max_sum(e, dt, n)
        out["e2e"] = {"value": draws_total / dt_all, "unit": "sims/s", "h2d_bytes_per_step": int(r.timing.h2d_bytes),
                      "d2h_bytes_per_step": int(r.timing.d2h_bytes), "steps": 1, "accepted_this_rank": n_acc,
                      "api": "ecdna_b200_run (page-locked host buffers: prior draws in, per-draw distances/accept/summary out)"}
    if with_cpu and e.rank == 0 and e.world == 1:
        c = cpu_port("C4", args.cpu_seconds)
        out["cpu_baseline"] = {"value": c["sims_per_sec"], "unit": "sims/s", "cores": c["cores"], "kind": "port",
                               "events_per_sec": c["events_per_sec"],
                               "sample": f"{c['replicates']} prior draws of C4 ({c['events']} events, {c['seconds']:.1f} s, "
                                         f"{c['accepted']} accepted) over {c['cores']} host threads; reference-layout C++ "
                                         "restatement + the four distances per draw"}
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    e = setup(args)
    m = e.m

    if args.workload == "C4":  # the ABC line on its own
        a = abc_leg(e, args, args.abc_draws, not args.no_cpu_baseline, not args.no_e2e, steps=args.steps,
                    warmup=args.warmup, dump=args.dump_outputs)
        if rank == 0:
            line = {"metric": a["metric"], "value": a["value"], "unit": a["unit"], "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup,
                    "ms_per_step": a["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "u32", "data": "synthetic"}
            line.update({k: v for k, v in a.items() if k not in line})
            print(json.dumps(line), flush=True)
        if world > 1:
            e.dist.destroy_process_group()
        return

    kw, reps_cfg, desc = WORKLOADS[args.workload]
    reps = args.replicates or reps_cfg
    opts0 = m.SimulationOptions(save_snapshots=False, **kw)
    check = {"C1": 3, "C2": 2, "C3": 4, "C5": 1}[args.workload]
    leg = ssa_leg(e, args, args.workload, reps, args.steps, args.warmup, opts0.idx_begin + rank * reps, check=check,
                  sample_clocks=True)
    if args.dump_outputs:
        dt = result_dtypes(m)
        dump_outputs(args.dump_outputs, {k: (v, dt[k]) for k, v in leg.tensors.items()}, leg.last_idx0,
                     rank=rank, world=world)
    del leg.tensors
    e2e = None if args.no_e2e else e2e_ssa(e, leg, args.steps, opts0.idx_begin + 5_000_000_000 + rank * reps)
    roofline = roofline_block(leg, args.workload, leg.clocks)

    abc = None
    if not args.no_abc:
        abc = abc_leg(e, args, args.abc_draws, not args.no_cpu_baseline, not args.no_e2e)

    strong = None
    if not args.no_strong:
        # the replicates of each config in TOTAL, split over the ranks (what the reference's rayon loop does
        # with more workers, main.rs:214-225); batches this small cannot fill one GPU, let alone eight
        strong = {}
        for w in ("C2", "C3", "C5"):
            total = WORKLOADS[w][1]
            o = m.SimulationOptions(save_snapshots=False, **WORKLOADS[w][0])
            b, c = m.rank_range(o.idx_begin + 3_000_000_000, total, rank, world)
            if w == args.workload and world == 1 and reps == total:
                strong[w] = {"value": leg.value, "unit": "events/s", "ms": leg.ms_all / leg.steps, "replicates_total": total,
                             "tile_width": leg.last.tile_width, "note": "same measurement as the headline"}
                continue
            s = ssa_leg(e, args, w, max(c, 1), 1, 1, b)
            strong[w] = {"value": s.value, "unit": "events/s", "ms": s.ms_all, "replicates_total": total,
                         "replicates_this_rank": c, "tile_width": s.last.tile_width,
                         "grid_blocks": s.last.grid_blocks}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            c = cpu_port(args.workload, args.cpu_seconds)
            cpu = {"value": c["events_per_sec"], "unit": "events/s", "cores": c["cores"], "kind": "port",
                   "sample": f"{c['replicates']} replicates of {args.workload} ({c['events']} events, "
                             f"{c['seconds']:.1f} s) over {c['cores']} host threads; reference-layout C++ "
                             "restatement (vector state, ChaCha8, ziggurat, BINV/BTPE; -O3 -march=native)"}
        last = leg.last
        line = {
            "metric": "ssa_events_per_sec", "value": leg.value, "unit": "events/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": leg.ms_all / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {desc}", "replicates_per_gpu_per_step": reps,
                       "events_per_step": leg.events_all / args.steps, "tile_width": last.tile_width,
                       "smem_bins": last.smem_bins, "state": args.state, "grid_blocks": last.grid_blocks,
                       "block_threads": last.block_threads, "blocks_per_sm": last.blocks_per_sm, "kmax": leg.kmax,
                       "spilled": last.n_spilled, "ms_per_step_per_rank": leg.ms_per_rank,
                       "kernel_ms_per_rank": leg.kernel_ms_per_rank,
                       "l2": "256 MiB buffer rewritten before every step; each step simulates fresh replicate "
                             "indices", "results_ok": leg.results},
            "e2e": e2e, "gpu_launches": args.steps * last.kernel_launches, "clocks": leg.clocks, "roofline": roofline,
            "cpu_baseline": cpu, "abc": abc, "strong": strong,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        e.dist.destroy_process_group()


if __name__ == "__main__":
    main()
