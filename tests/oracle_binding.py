"""ctypes binding of the CPU oracle (oracle/libecdna_oracle.so).

TEST INFRASTRUCTURE: imported only by tests/, __graft_entry__.smoke() and bench.py's CPU legs.
The product package (ecdna-evo_b200/) never imports this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_ORACLE_DIR = os.path.join(_ROOT, "oracle")
_SO = os.path.join(_ORACLE_DIR, "libecdna_oracle.so")

EV_BIRTH_NMINUS, EV_BIRTH_NPLUS, EV_DEATH_NMINUS, EV_DEATH_NPLUS = 0, 1, 2, 3
SEG_DETERMINISTIC, SEG_BINOMIAL_NO_UNEVEN, SEG_BINOMIAL, SEG_BINOMIAL_NO_NMINUS = 0, 1, 2, 3
STOP_NO_INDIVIDUALS, STOP_MAX_ITERS, STOP_MAX_TIME, STOP_MAX_CELLS = 0, 1, 2, 3
STOP_ABSORBING, STOP_COPY_OVERFLOW, STOP_HIST_OVERFLOW, STOP_REPLAY_END, STOP_REPLAY_BAD = 4, 5, 6, 7, 8
STATE_VECTOR, STATE_HIST = 0, 1
RNG_RAND, RNG_PHILOX, RNG_REPLAY = 0, 1, 2

REPLAY_DTYPE = np.dtype(
    [("dt", "<f4"), ("k", "<u2"), ("k1", "<u2"), ("event", "u1"), ("pad", "u1", (3,))], align=False
)
assert REPLAY_DTYPE.itemsize == 12


class Opts(C.Structure):
    _fields_ = [
        ("b0", C.c_float), ("b1", C.c_float), ("d0", C.c_float), ("d1", C.c_float),
        ("segregation", C.c_uint32), ("state", C.c_uint32), ("rng", C.c_uint32), ("bd_count_mode", C.c_uint32),
        ("max_cells", C.c_uint64), ("max_iter", C.c_uint64), ("max_time", C.c_float), ("birth_death", C.c_uint32),
        ("seed", C.c_uint64), ("run_idx", C.c_uint64),
        ("n_init", C.c_uint32), ("init_k", C.c_void_p), ("init_c", C.c_void_p),
        ("n_snap", C.c_uint32), ("snap_cells", C.c_void_p),
        ("dyn_points", C.c_uint32), ("dyn_dt", C.c_float),
        ("replay_in", C.c_void_p), ("replay_len", C.c_uint64),
        ("u64_in", C.c_void_p), ("u64_in_len", C.c_uint64),
    ]


class Out(C.Structure):
    _fields_ = [
        ("stop_reason", C.c_uint32), ("kmax", C.c_uint32),
        ("nminus", C.c_uint64), ("nplus", C.c_uint64), ("n_events", C.c_uint64),
        ("time", C.c_float), ("n_snap_taken", C.c_uint32),
        ("hash", C.c_uint64), ("chain", C.c_uint64),
        ("sum_k", C.c_uint64), ("n_div", C.c_uint64), ("n_death", C.c_uint64),
        ("dyn_count", C.c_uint32),
        ("hist_cap", C.c_uint32), ("hist", C.c_void_p),
        ("trace_out", C.c_void_p), ("trace_cap", C.c_uint64), ("trace_len", C.c_uint64),
        ("traj_out", C.c_void_p), ("traj_cap", C.c_uint64),
        ("snap_hist", C.c_void_p), ("snap_cells_out", C.c_void_p), ("snap_time", C.c_void_p),
        ("dyn_out", C.c_void_p),
        ("u64_out", C.c_void_p), ("u64_cap", C.c_uint64), ("u64_len", C.c_uint64),
    ]


_SOURCES = ("ecdna_oracle.cpp", "ecdna_oracle.h", "Makefile")


def build(force=False):
    """The checker, built in oracle/ when it is missing or older than its sources (__graft_entry__.build()
    leaves it built, so a built tree is only read)."""
    src = [os.path.join(_ORACLE_DIR, f) for f in _SOURCES]
    stale = not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in src)
    if force or stale:
        subprocess.run(["make", "-s", "-C", _ORACLE_DIR] + (["-B"] if force else []) + ["libecdna_oracle.so"],
                       check=True, capture_output=True)
    return _SO


_lib = None
_so_fast = None


def use_fast_build():
    """bench.py's CPU legs time the -O3 -march=native build of the same source; tests never call this.
    -march=native code must be compiled on the host that runs it, so it is compiled once per process, from a
    copy of the sources in a temporary directory: the checkout may be read-only."""
    global _lib, _so_fast
    if _so_fast is None:
        import atexit
        import shutil
        import tempfile
        d = tempfile.mkdtemp(prefix="ecdna_oracle_fast_")
        atexit.register(shutil.rmtree, d, True)
        for f in _SOURCES:
            shutil.copy(os.path.join(_ORACLE_DIR, f), d)
        subprocess.run(["make", "-s", "-C", d, "libecdna_oracle_fast.so"], check=True, capture_output=True)
        _so_fast, _lib = os.path.join(d, "libecdna_oracle_fast.so"), None


def lib():
    global _lib
    if _lib is None:
        if _so_fast is None:
            build()
        L = C.CDLL(_so_fast or _SO)
        L.orc_run.argtypes = [C.POINTER(Opts), C.POINTER(Out)]
        L.orc_run.restype = C.c_int
        L.orc_run_batch.argtypes = [C.POINTER(Opts), C.c_uint64, C.c_uint64, C.c_int] + [C.c_void_p] * 6 + [
            C.c_uint32, C.c_void_p]
        L.orc_run_batch.restype = C.c_uint64
        L.orc_abc_batch.argtypes = [C.POINTER(Opts), C.c_uint64, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32,
                                    C.POINTER(C.c_float), C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_abc_batch.restype = C.c_uint64
        L.orc_stats.argtypes = [C.c_void_p, C.c_uint32] + [C.POINTER(C.c_float)] * 4
        L.orc_ks_distance.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
        L.orc_ks_distance.restype = C.c_float
        L.orc_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_chacha8_u64.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
        L.orc_chacha_block.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p]
        L.orc_seed_from_u64.argtypes = [C.c_uint64, C.c_void_p]
        L.orc_neg_log_u24.argtypes = [C.c_uint32]
        L.orc_neg_log_u24.restype = C.c_float
        L.orc_binomial_half_philox.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
        L.orc_binomial_half_philox.restype = C.c_uint32
        L.orc_pick_philox.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64]
        L.orc_pick_philox.restype = C.c_uint64
        L.orc_rand_binomial.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_double, C.c_uint64, C.c_void_p]
        L.orc_rand_exp1_f32.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
        L.orc_rand_gen_range.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
        L.orc_apply_event.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64] + [
            C.POINTER(C.c_uint32)] * 4
        L.orc_apply_event.restype = C.c_int
        L.orc_segregate.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                    C.POINTER(C.c_uint32)]
        L.orc_segregate.restype = C.c_int
        L.orc_subsample.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]
        L.orc_subsample.restype = None
        L.orc_hist_weight.argtypes = [C.c_uint32]
        L.orc_hist_weight.restype = C.c_uint64
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data if a is not None else None


class Result:
    pass


def make_opts(b0=1.0, b1=1.0, d0=0.0, d1=0.0, segregation=SEG_BINOMIAL, state=STATE_HIST, rng=RNG_PHILOX,
              max_cells=1000, max_iter=1_000_000_000, max_time=None, seed=26, run_idx=260, initial=None,
              snapshots=None, dyn_points=0, dyn_dt=0.1, replay=None, bd_count_mode=0, u64_in=None):
    """Mirror of SimulationOptions (main.rs:28-44) + Options (clap_app.rs:204-209)."""
    if max_time is None:
        max_time = float(int(np.log2(np.float32(max_cells)) + np.float32(4.0)))  # clap_app.rs:151
    initial = initial or {1: 1}  # clap_app.rs:188-191
    keep = {}
    keep["init_k"] = np.array(list(initial.keys()), dtype=np.uint16)
    keep["init_c"] = np.array(list(initial.values()), dtype=np.uint64)
    keep["snap"] = np.array(sorted(snapshots) if snapshots else [], dtype=np.uint64)
    keep["replay"] = np.ascontiguousarray(replay) if replay is not None else None
    o = Opts()
    o.b0, o.b1, o.d0, o.d1 = b0, b1, d0, d1
    o.segregation, o.state, o.rng, o.bd_count_mode = segregation, state, rng, bd_count_mode
    o.max_cells, o.max_iter, o.max_time = max_cells, max_iter, max_time
    o.birth_death = 1 if (d0 > 0 or d1 > 0) else 0
    o.seed, o.run_idx = seed, run_idx
    o.n_init, o.init_k, o.init_c = len(keep["init_k"]), _ptr(keep["init_k"]), _ptr(keep["init_c"])
    o.n_snap, o.snap_cells = len(keep["snap"]), _ptr(keep["snap"]) if len(keep["snap"]) else None
    o.dyn_points, o.dyn_dt = dyn_points, dyn_dt
    if keep["replay"] is not None:
        o.replay_in, o.replay_len = _ptr(keep["replay"]), len(keep["replay"])
    if u64_in is not None:
        keep["u64_in"] = np.ascontiguousarray(u64_in, dtype=np.uint64)
        o.u64_in, o.u64_in_len = _ptr(keep["u64_in"]), len(keep["u64_in"])
    o._keep = keep
    return o


def run(opts, hist_cap=4096, trace_cap=0, traj_cap=0, u64_cap=0):
    out = Out()
    r = Result()
    r.hist = np.zeros(hist_cap, dtype=np.uint64)
    out.hist_cap, out.hist = hist_cap, _ptr(r.hist)
    if trace_cap:
        r.trace = np.zeros(trace_cap, dtype=REPLAY_DTYPE)
        out.trace_out, out.trace_cap = _ptr(r.trace), trace_cap
    if traj_cap:
        r.traj = np.zeros((traj_cap, 4), dtype=np.uint64)
        out.traj_out, out.traj_cap = _ptr(r.traj), traj_cap
    if u64_cap:
        r.u64 = np.zeros(u64_cap, dtype=np.uint64)
        out.u64_out, out.u64_cap = _ptr(r.u64), u64_cap
    if opts.n_snap:
        r.snap_hist = np.zeros((opts.n_snap, hist_cap), dtype=np.uint64)
        r.snap_cells = np.zeros(opts.n_snap, dtype=np.uint64)
        r.snap_time = np.zeros(opts.n_snap, dtype=np.float32)
        out.snap_hist, out.snap_cells_out, out.snap_time = _ptr(r.snap_hist), _ptr(r.snap_cells), _ptr(r.snap_time)
    if opts.dyn_points:
        r.dyn = np.zeros((opts.dyn_points, 5), dtype=np.float32)
        out.dyn_out = _ptr(r.dyn)
    rc = lib().orc_run(C.byref(opts), C.byref(out))
    if rc != 0:
        raise RuntimeError(f"orc_run failed: {rc}")
    for f in ("stop_reason", "kmax", "nminus", "nplus", "n_events", "time", "n_snap_taken", "hash", "chain", "sum_k",
              "n_div", "n_death", "dyn_count", "trace_len", "u64_len"):
        setattr(r, f, getattr(out, f))
    if u64_cap:
        r.u64 = r.u64[: min(r.u64_len, u64_cap)]
    if trace_cap:
        r.trace = r.trace[: min(r.trace_len, trace_cap)]
    if traj_cap:
        r.traj = r.traj[: min(r.n_events, traj_cap)]
    return r


def run_batch(opts, idx_begin, n_runs, n_threads=0, hist_cap=0, rates=None):
    r = Result()
    r.nminus = np.zeros(n_runs, dtype=np.uint64)
    r.nplus = np.zeros(n_runs, dtype=np.uint64)
    r.time = np.zeros(n_runs, dtype=np.float32)
    r.n_events = np.zeros(n_runs, dtype=np.uint64)
    r.stop = np.zeros(n_runs, dtype=np.uint32)
    r.hist = np.zeros((n_runs, hist_cap), dtype=np.uint64) if hist_cap else None
    rates_c = np.ascontiguousarray(rates, dtype=np.float32) if rates is not None else None
    r.total_events = lib().orc_run_batch(C.byref(opts), idx_begin, n_runs, n_threads, _ptr(r.nminus), _ptr(r.nplus),
                                         _ptr(r.time), _ptr(r.n_events), _ptr(r.stop), _ptr(r.hist), hist_cap,
                                         _ptr(rates_c))
    return r


def abc_batch(opts, idx_begin, n_runs, rates, target, thresholds, n_threads=0, hist_cap=512):
    """orc_abc_batch: prior draws -> replicates -> the four ABC distances and the accept flag per draw."""
    r = Result()
    r.distance = np.zeros((n_runs, 4), dtype=np.float32)
    r.accept = np.zeros(n_runs, dtype=np.uint8)
    r.n_events = np.zeros(n_runs, dtype=np.uint64)
    r.stop = np.zeros(n_runs, dtype=np.uint32)
    rates_c = np.ascontiguousarray(rates, dtype=np.float32)
    tgt = np.ascontiguousarray(target, dtype=np.uint64)
    thr = (C.c_float * 4)(*thresholds)
    r.total_events = lib().orc_abc_batch(C.byref(opts), idx_begin, n_runs, n_threads, _ptr(rates_c), _ptr(tgt), len(tgt), thr,
                                         hist_cap, _ptr(r.distance), _ptr(r.accept), _ptr(r.n_events), _ptr(r.stop))
    return r


def stats(hist):
    h = np.ascontiguousarray(hist, dtype=np.uint64)
    m, f, e, v = C.c_float(), C.c_float(), C.c_float(), C.c_float()
    lib().orc_stats(_ptr(h), len(h), C.byref(m), C.byref(f), C.byref(e), C.byref(v))
    return m.value, f.value, e.value, v.value


def subsample(hist, want, seed, run_idx, j):
    """into_subsampled (main.rs:110-123) as the library's native mode defines it."""
    h = np.ascontiguousarray(hist, dtype=np.uint64)
    out = np.zeros_like(h)
    lib().orc_subsample(_ptr(h), len(h), int(want), int(seed), int(run_idx), int(j), _ptr(out))
    return out


def ks_distance(h1, h2):
    a = np.ascontiguousarray(h1, dtype=np.uint64)
    b = np.ascontiguousarray(h2, dtype=np.uint64)
    return lib().orc_ks_distance(_ptr(a), len(a), _ptr(b), len(b))


def philox(ctr, key):
    c = np.array(ctr, dtype=np.uint32)
    k = np.array(key, dtype=np.uint32)
    o = np.zeros(4, dtype=np.uint32)
    lib().orc_philox4x32_10(_ptr(c), _ptr(k), _ptr(o))
    return o
