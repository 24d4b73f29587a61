"""ecdna_evo_b200 -- host-side binding of libecdna_b200.so (include/ecdna_b200.h).

The shared library is the product: a hand-written sm_100a kernel behind a C ABI that replaces the
per-replicate closure of the reference (src/main.rs:55-211).  This module is plumbing only: ctypes
structures, numpy/torch buffer management, and a mirror of the reference's option handling
(src/clap_app.rs) and file layout (src/lib.rs:27-45, src/process.rs:31-55) so tests read like the
reference's.  There is NO CPU fallback: if the library is missing or no B200 is visible, calls raise.

The directory is named `ecdna-evo_b200`; import it with `_pkg.load()` (repo root) which registers
it as the module `ecdna_evo_b200`.
"""
import ctypes as C
import json
import os

import numpy as np

from .build import LIB_PATH, build, build_debug  # noqa: F401
from .shard import gather_accepted, rank_range  # noqa: F401
from .abc import (ABC_FIELDS, REC_HEADER, SMC_FIELDS, abc_rows, decode_records, merge_gathered,  # noqa: F401
                  record_words, write_abc_csv, write_abc_smc)

ABI_VERSION = 3
EV_BIRTH_NMINUS, EV_BIRTH_NPLUS, EV_DEATH_NMINUS, EV_DEATH_NPLUS = 0, 1, 2, 3
SEG_DETERMINISTIC, SEG_BINOMIAL_NO_UNEVEN, SEG_BINOMIAL, SEG_BINOMIAL_NO_NMINUS = 0, 1, 2, 3
SEGREGATION_NAMES = {  # --segregation values, clap_app.rs:232-238
    "deterministic": SEG_DETERMINISTIC, "binomial-no-uneven": SEG_BINOMIAL_NO_UNEVEN,
    "binomial": SEG_BINOMIAL, "binomial-no-nminus": SEG_BINOMIAL_NO_NMINUS,
}
STOP_NO_INDIVIDUALS, STOP_MAX_ITERS, STOP_MAX_TIME, STOP_MAX_CELLS = 0, 1, 2, 3
STOP_ABSORBING, STOP_COPY_OVERFLOW, STOP_HIST_OVERFLOW, STOP_REPLAY_END, STOP_REPLAY_BAD = 4, 5, 6, 7, 8
STOP_NAMES = ["NoIndividualsLeft", "MaxItersReached", "MaxTimeReached", "MaxIndividualsReached",
              "AbsorbingStateReached", "CopyNumberOverflow", "HistogramOverflow", "ReplayExhausted",
              "ReplayInconsistent"]
FLAG_HIST_TRUNCATED, FLAG_SPILLED = 0x100, 0x200
RNG_PHILOX, RNG_REPLAY, RNG_UNIFORMS = 0, 1, 2
STATE_AUTO, STATE_SMEM, STATE_HBM = 0, 1, 2
WANT_DIGEST = 0x1
MAX_ITER = 1_000_000_000  # main.rs:23
MAX_CELLS = 1_000_000_000  # main.rs:25

REPLAY_DTYPE = np.dtype([("dt", "<f4"), ("k", "<u2"), ("k1", "<u2"), ("event", "u1"), ("pad", "u1", (3,))])


class ParamsT(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32),
        ("b0", C.c_float), ("b1", C.c_float), ("d0", C.c_float), ("d1", C.c_float),
        ("segregation", C.c_uint32),
        ("max_cells", C.c_uint64), ("max_iter", C.c_uint64), ("max_time", C.c_float),
        ("seed", C.c_uint64), ("bd_count_mode", C.c_uint32),
        ("n_init", C.c_uint32), ("init_k", C.c_void_p), ("init_c", C.c_void_p),
        ("n_snapshots", C.c_uint32), ("snapshot_cells", C.c_void_p),
        ("rates_per_run", C.c_void_p),
        ("rng_mode", C.c_uint32), ("replay", C.c_void_p), ("replay_offsets", C.c_void_p),
        ("dyn_points", C.c_uint32), ("dyn_dt", C.c_float),
        ("abc_enabled", C.c_uint32), ("abc_target_hist", C.c_void_p), ("abc_target_len", C.c_uint32),
        ("abc_thresholds", C.c_float * 4),
        ("state_mode", C.c_uint32), ("tile_width", C.c_uint32), ("smem_bins", C.c_uint32),
        ("max_copies", C.c_uint32), ("hist_stride", C.c_uint32), ("flags", C.c_uint32),
        ("spill_records", C.c_uint32), ("replay_u64", C.c_void_p), ("slice_events", C.c_uint32),
        ("n_subsamples", C.c_uint32), ("subsample_cells", C.c_void_p),
    ]


# (name, dtype, trailing shape as a function of (n_snapshots, dyn_points, hist_stride, n_subsamples))
RESULT_FIELDS = [
    ("stop_reason", np.uint32, lambda s, d, h, u: ()), ("nminus", np.uint64, lambda s, d, h, u: ()),
    ("nplus", np.uint64, lambda s, d, h, u: ()), ("time", np.float32, lambda s, d, h, u: ()),
    ("n_events", np.uint64, lambda s, d, h, u: ()), ("kmax", np.uint32, lambda s, d, h, u: ()),
    ("mean", np.float32, lambda s, d, h, u: ()), ("frequency", np.float32, lambda s, d, h, u: ()),
    ("entropy", np.float32, lambda s, d, h, u: ()), ("variance", np.float32, lambda s, d, h, u: ()),
    ("abc_distance", np.float32, lambda s, d, h, u: (4,)), ("abc_accept", np.uint8, lambda s, d, h, u: ()),
    ("hash", np.uint64, lambda s, d, h, u: ()), ("chain", np.uint64, lambda s, d, h, u: ()),
    ("hist", np.uint32, lambda s, d, h, u: (h,)), ("snap_count", np.uint32, lambda s, d, h, u: ()),
    ("snap_cells", np.uint64, lambda s, d, h, u: (s,)), ("snap_time", np.float32, lambda s, d, h, u: (s,)),
    ("snap_hist", np.uint32, lambda s, d, h, u: (s, h)), ("dyn_count", np.uint32, lambda s, d, h, u: ()),
    ("dyn", np.float32, lambda s, d, h, u: (d, 5)), ("sum_k", np.uint64, lambda s, d, h, u: ()),
    ("n_div", np.uint32, lambda s, d, h, u: ()), ("n_death", np.uint32, lambda s, d, h, u: ()),
    ("sub_hist", np.uint32, lambda s, d, h, u: (u, h)),
]


class ResultsT(C.Structure):
    _fields_ = [(name, C.c_void_p) for name, _, _ in RESULT_FIELDS]


class ResultSizesT(C.Structure):
    _fields_ = [(name, C.c_uint64) for name, _, _ in RESULT_FIELDS]


def query_sizes(params, n_runs):
    """ecdna_b200_query_sizes: bytes behind every result pointer for a batch (no GPU needed)."""
    out = ResultSizesT()
    rc = lib().ecdna_b200_query_sizes(C.byref(params), n_runs, C.byref(out))
    if rc != 0:
        raise EcdnaB200Error(f"ecdna_b200_query_sizes: status {rc}")
    return {name: getattr(out, name) for name, _, _ in RESULT_FIELDS}


class SparseT(C.Structure):
    """ecdna_b200_sparse_t"""
    _fields_ = [("final_dist", C.c_void_p), ("snap_dist", C.c_void_p), ("sub_dist", C.c_void_p), ("arena", C.c_void_p),
                ("arena_words", C.c_uint64), ("arena_used", C.c_uint64)]


# ecdna_b200_dist_t (40 bytes)
DIST_DTYPE = np.dtype([("cells", np.uint64), ("nminus", np.uint64), ("offset", np.uint64), ("time", np.float32),
                       ("k_len", np.uint32), ("k_min", np.uint16), ("flags", np.uint16), ("reserved", np.uint32)])
DIST_TAKEN, DIST_TRUNCATED = 1, 2
ERR_ARENA = 7


class Sparse:
    """Caller-owned buffers of the sparse return: one descriptor per distribution and the arena of occupied bins."""

    def __init__(self, n_runs, n_snapshots, n_subsamples, arena_words):
        self.struct = SparseT()
        self.final_dist = np.zeros(n_runs, dtype=DIST_DTYPE)
        self.snap_dist = np.zeros((n_runs, n_snapshots), dtype=DIST_DTYPE)
        self.sub_dist = np.zeros((n_runs, n_subsamples), dtype=DIST_DTYPE)
        self.struct.final_dist = self.final_dist.ctypes.data
        if n_snapshots:
            self.struct.snap_dist = self.snap_dist.ctypes.data
        if n_subsamples:
            self.struct.sub_dist = self.sub_dist.ctypes.data
        self.resize(arena_words)

    def resize(self, arena_words):
        self.arena = np.zeros(max(int(arena_words), 1), dtype=np.uint32)
        self.struct.arena = self.arena.ctypes.data
        self.struct.arena_words = int(arena_words)

    @property
    def arena_used(self):
        return int(self.struct.arena_used)

    def dense(self, desc, stride):
        """The dense form of the distributions `desc` (any shape): [..., stride] with [0] = cells without ecDNA."""
        flat = desc.reshape(-1)
        out = np.zeros((flat.size, stride), dtype=np.uint32)
        for i, d in enumerate(flat):
            out[i, 0] = d["nminus"]
            n, k0, off = int(d["k_len"]), int(d["k_min"]), int(d["offset"])
            out[i, k0:k0 + n] = self.arena[off:off + n]
        return out.reshape(desc.shape + (stride,))


class TimingT(C.Structure):
    _fields_ = [
        ("kernel_ms", C.c_float), ("total_ms", C.c_float), ("kernel_launches", C.c_uint32),
        ("tile_width", C.c_uint32), ("smem_bins", C.c_uint32), ("grid_blocks", C.c_uint32),
        ("block_threads", C.c_uint32), ("blocks_per_sm", C.c_uint32),
        ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("total_events", C.c_uint64),
        ("alg_bytes", C.c_uint64), ("n_spilled", C.c_uint32), ("slice_events", C.c_uint32),
        ("n_slices", C.c_uint64), ("n_idle_spells", C.c_uint64), ("n_finished", C.c_uint64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


EXPORTED_SYMBOLS = [
    "ecdna_b200_create", "ecdna_b200_destroy", "ecdna_b200_last_error", "ecdna_b200_abi_version", "ecdna_b200_run",
    "ecdna_b200_run_device", "ecdna_b200_get_timing", "ecdna_b200_abc_draw_priors",
    "ecdna_b200_plan", "ecdna_b200_abc_draw_priors_device", "ecdna_b200_abc_pack", "ecdna_b200_abc_allgather",
    "ecdna_b200_comm_unique_id", "ecdna_b200_comm_init", "ecdna_b200_comm_release",
    "ecdna_b200_multi_create", "ecdna_b200_multi_destroy", "ecdna_b200_multi_device_count",
    "ecdna_b200_multi_last_error", "ecdna_b200_multi_run", "ecdna_b200_multi_get_timing", "ecdna_b200_query_sizes",
    "ecdna_b200_run_sparse", "ecdna_b200_sparse_fetch", "ecdna_b200_multi_run_sparse", "ecdna_b200_multi_sparse_fetch",
    "ecdna_b200_abc_smc_propose", "ecdna_b200_abc_smc_weights", "ecdna_b200_abc_smc",
]
ERR_INTERNAL, ERR_COMM = 5, 6
SMC_STATUS = ["reached", "max_generations", "budget"]  # ECDNA_B200_SMC_*


class SmcOptionsT(C.Structure):
    """ecdna_b200_smc_options_t"""
    _fields_ = [("population", C.c_uint32), ("quantile", C.c_double), ("max_generations", C.c_uint32),
                ("max_simulations", C.c_uint64), ("idx_begin", C.c_uint64), ("chunk", C.c_uint64),
                ("b1_range", C.c_float * 2), ("d0_range", C.c_float * 2), ("d1_range", C.c_float * 2)]


# (name, dtype, trailing shape) of the per-particle and per-generation outputs of ecdna_b200_smc_result_t
SMC_PARTICLE_FIELDS = [("idx", np.uint64, ()), ("parent_idx", np.uint64, ()), ("rates", np.float32, (4,)),
                       ("distance", np.float32, (4,)), ("weight", np.float64, ()), ("cells", np.uint64, ())]
SMC_GENERATION_FIELDS = [("epsilon", np.float32, ()), ("consumed", np.uint64, ()), ("simulated", np.uint64, ()),
                         ("ess", np.float64, ()), ("time_ms", np.float32, (3,))]


class SmcResultT(C.Structure):
    """ecdna_b200_smc_result_t"""
    _fields_ = [(n, C.c_void_p) for n, _, _ in SMC_PARTICLE_FIELDS + SMC_GENERATION_FIELDS] + [
        ("generations", C.c_uint32), ("status", C.c_uint32)]
COMM_ID_BYTES = 128

_lib = None


def plan(n_runs, tile_width=0, slice_events=0, sm_count=148, max_blocks_per_sm=None):
    """ecdna_b200_plan: (lanes, blocks_per_sm, tiles, sliced) the library would launch a batch with."""
    out = [C.c_uint32() for _ in range(4)]
    if max_blocks_per_sm is None:  # what fits on a B200 with the default 256-bin window
        probe = [C.c_uint32() for _ in range(4)]
        lib().ecdna_b200_plan(n_runs, tile_width, slice_events, sm_count, 1, *[C.byref(x) for x in probe])
        max_blocks_per_sm = {1: 3, 2: 3, 4: 5}.get(probe[0].value, 4)
    rc = lib().ecdna_b200_plan(n_runs, tile_width, slice_events, sm_count, max_blocks_per_sm, *[C.byref(x) for x in out])
    if rc != 0:
        raise EcdnaB200Error(f"ecdna_b200_plan: status {rc}")
    return out[0].value, out[1].value, out[2].value, bool(out[3].value)


def lib():
    """Load libecdna_b200.so; raise loudly if it has not been built (no fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a). "
                               "There is no CPU fallback.")
        L = C.CDLL(os.environ.get("ECDNA_B200_LIB", LIB_PATH))  # (the override is for A/B experiments)
        L.ecdna_b200_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.ecdna_b200_destroy.argtypes = [C.c_void_p]
        L.ecdna_b200_destroy.restype = None
        L.ecdna_b200_last_error.argtypes = [C.c_void_p]
        L.ecdna_b200_last_error.restype = C.c_char_p
        L.ecdna_b200_run.argtypes = [C.c_void_p, C.POINTER(ParamsT), C.c_uint64, C.c_uint64, C.POINTER(ResultsT)]
        L.ecdna_b200_run_device.argtypes = [C.c_void_p, C.POINTER(ParamsT), C.c_uint64, C.c_uint64,
                                            C.POINTER(ResultsT), C.c_void_p]
        L.ecdna_b200_get_timing.argtypes = [C.c_void_p, C.POINTER(TimingT)]
        L.ecdna_b200_plan.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32] + [C.POINTER(C.c_uint32)] * 4
        L.ecdna_b200_abc_draw_priors.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_float,
                                                 C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float),
                                                 C.c_void_p]
        L.ecdna_b200_abc_draw_priors_device.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_float,
                                                        C.POINTER(C.c_float), C.POINTER(C.c_float),
                                                        C.POINTER(C.c_float), C.c_void_p, C.c_void_p]
        L.ecdna_b200_abc_pack.argtypes = [C.c_void_p, C.POINTER(ResultsT), C.c_void_p, C.POINTER(C.c_float), C.c_uint64,
                                          C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                          C.c_void_p]
        L.ecdna_b200_abc_allgather.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                               C.c_void_p, C.c_void_p]
        L.ecdna_b200_comm_unique_id.argtypes = [C.c_void_p]
        L.ecdna_b200_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.ecdna_b200_multi_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
        L.ecdna_b200_multi_destroy.argtypes = [C.c_void_p]
        L.ecdna_b200_multi_destroy.restype = None
        L.ecdna_b200_multi_device_count.argtypes = [C.c_void_p]
        L.ecdna_b200_multi_last_error.argtypes = [C.c_void_p]
        L.ecdna_b200_multi_last_error.restype = C.c_char_p
        L.ecdna_b200_multi_run.argtypes = [C.c_void_p, C.POINTER(ParamsT), C.c_uint64, C.c_uint64, C.POINTER(ResultsT)]
        L.ecdna_b200_multi_get_timing.argtypes = [C.c_void_p, C.POINTER(TimingT)]
        L.ecdna_b200_query_sizes.argtypes = [C.POINTER(ParamsT), C.c_uint64, C.POINTER(ResultSizesT)]
        L.ecdna_b200_run_sparse.argtypes = [C.c_void_p, C.POINTER(ParamsT), C.c_uint64, C.c_uint64, C.POINTER(ResultsT),
                                            C.POINTER(SparseT)]
        L.ecdna_b200_sparse_fetch.argtypes = [C.c_void_p, C.POINTER(SparseT)]
        L.ecdna_b200_multi_run_sparse.argtypes = L.ecdna_b200_run_sparse.argtypes
        L.ecdna_b200_multi_sparse_fetch.argtypes = [C.c_void_p, C.POINTER(SparseT)]
        L.ecdna_b200_abc_smc_propose.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p,
                                                 C.c_uint32, C.POINTER(C.c_double)] + [C.POINTER(C.c_float)] * 3 + [
                                                     C.c_void_p, C.c_void_p]
        L.ecdna_b200_abc_smc_weights.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                                 C.POINTER(C.c_double)] + [C.POINTER(C.c_float)] * 3 + [C.c_void_p]
        L.ecdna_b200_abc_smc.argtypes = [C.c_void_p, C.POINTER(ParamsT), C.POINTER(SmcOptionsT), C.POINTER(SmcResultT)]
        L.ecdna_b200_comm_release.argtypes = [C.c_void_p]
        L.ecdna_b200_comm_release.restype = None
        _lib = L
    return _lib


def comm_unique_id():
    """ecdna_b200_comm_unique_id: 128 bytes rank 0 hands to every rank (ncclUniqueId)."""
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    rc = lib().ecdna_b200_comm_unique_id(buf)
    if rc != 0:
        raise EcdnaB200Error(f"ecdna_b200_comm_unique_id: status {rc} (6 = NCCL not available)")
    return bytes(buf)


class EcdnaB200Error(RuntimeError):
    pass


# --------------------------------------------------------------------------------------------
# mirror of the reference's option handling
# --------------------------------------------------------------------------------------------
def years_from_cells(cells):
    """clap_app.rs:151: years = (log2(cells as f32) + 4) as u64."""
    return int(np.float32(np.log2(np.float32(cells))) + np.float32(4.0))


def build_snapshots_from_cells(n_snapshots, cells):
    """clap_app.rs:121-134: 1, 1+dx, ..., cells with dx = cells / (n-1)."""
    dx = cells // (n_snapshots - 1)
    x = [1] * n_snapshots
    for i in range(1, n_snapshots - 1):
        x[i] = x[i - 1] + dx
    x[-1] = cells
    return x


def build_snapshots(cells, snapshots=None):
    """clap_app.rs:102-119: user list or the 11 default sizes, sorted ascending."""
    return sorted(snapshots if snapshots is not None else build_snapshots_from_cells(11, cells))


def _f32_to_string(x):
    """Rust's f32 Display (shortest round-trip repr, no exponent, integers without '.0')."""
    x = np.float32(x)
    if np.isinf(x):
        return "inf" if x > 0 else "-inf"
    if np.isnan(x):
        return "NaN"
    s = np.format_float_positional(x, unique=True, trim="-")
    return s


def create_filename_birth_death(rates, idx):
    """lib.rs:27-36."""
    r = [_f32_to_string(v).replace(".", "dot") for v in rates]
    return f"{r[0]}b0_{r[1]}b1_{r[2]}d0_{r[3]}d1_{idx}idx"


def create_filename_pure_birth(rates, idx):
    """lib.rs:38-45."""
    r = [_f32_to_string(v).replace(".", "dot") for v in rates]
    return f"{r[0]}b0_{r[1]}b1_0d0_0d1_{idx}idx"


def save(path2dir, filename, time, hist):
    """process.rs:31-55: <dir>/<cells>cells/ecdna/<t>years/<filename>.json, JSON histogram
    (dynamics.md:7-8).  `hist` is dense with hist[0] = cells without ecDNA."""
    hist = np.asarray(hist)
    cells = int(hist.sum())
    timepoint = f"{float(np.float32(time)):.1f}".replace(".", "dot") + "years"
    d = os.path.join(path2dir, f"{cells}cells", "ecdna", timepoint)
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, filename + ".json")
    with open(path, "w") as f:
        json.dump({str(k): int(c) for k, c in enumerate(hist) if c}, f)
    return path


class SimulationOptions:
    """SimulationOptions (main.rs:28-44) with the defaults Cli::build derives (clap_app.rs:136-230)."""

    def __init__(self, b0=1.0, b1=1.0, d0=None, d1=None, cells=None, years=None, seed=26, runs=12,
                 segregation="binomial", initial=None, snapshots=None, path2dir=None, subsamples=None,
                 save_snapshots=True):
        if cells is not None and years is not None:
            raise ValueError("--years and --cells are mutually exclusive (clap group 'stop')")
        if years is not None:  # clap_app.rs:142-147
            self.max_cells, self.years = MAX_CELLS, int(years)
        else:  # clap_app.rs:148-157
            self.max_cells = 1000 if cells is None else int(cells)
            self.years = years_from_cells(self.max_cells)
        self.b0, self.b1 = float(b0), float(b1)
        self.d0 = 0.0 if d0 is None else float(d0)  # clap_app.rs:165-174
        self.d1 = 0.0 if d1 is None else float(d1)
        self.birth_death = self.d0 > 0 or self.d1 > 0
        self.seed, self.runs = int(seed), int(runs)
        self.segregation = SEGREGATION_NAMES[segregation] if isinstance(segregation, str) else int(segregation)
        self.distribution = dict(initial) if initial else {1: 1}  # clap_app.rs:188-191
        self.snapshots = build_snapshots(self.max_cells, snapshots) if save_snapshots else []
        self.max_iter = MAX_ITER
        self.path2dir = path2dir
        self.subsamples = subsamples

    @property
    def idx_begin(self):
        return self.seed * 10  # main.rs:214

    def filename(self, idx):
        if self.birth_death:
            return create_filename_birth_death([self.b0, self.b1, self.d0, self.d1], idx)
        return create_filename_pure_birth([self.b0, self.b1], idx)


class Context:
    """One GPU (ecdna_b200_ctx)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = lib().ecdna_b200_create(device, C.byref(self._h))
        if rc != 0:
            raise EcdnaB200Error(f"ecdna_b200_create(device={device}) failed with status {rc} "
                                 "(3 = no sm_100 device; the library has no CPU path)")
        self.device = device

    def close(self):
        if self._h:
            lib().ecdna_b200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise EcdnaB200Error(f"status {rc}: {lib().ecdna_b200_last_error(self._h).decode()}")

    def make_params(self, opts, n_runs, rates_per_run=None, replay=None, replay_offsets=None, dyn_points=0,
                    dyn_dt=0.1, abc_target=None, abc_thresholds=(0.05, 0.1, 0.1, 0.1), state_mode=STATE_AUTO,
                    tile_width=0, smem_bins=0, max_copies=0, hist_stride=0, digest=False, bd_count_mode=0,
                    snapshots=True, spill_records=0, replay_u64=None, slice_events=0, subsamples=None):
        keep = {}
        p = ParamsT()
        p.abi_version = ABI_VERSION
        p.b0, p.b1, p.d0, p.d1 = opts.b0, opts.b1, opts.d0, opts.d1
        p.segregation = opts.segregation
        p.max_cells, p.max_iter, p.max_time = opts.max_cells, opts.max_iter, float(opts.years)
        p.seed, p.bd_count_mode = opts.seed, bd_count_mode
        keep["init_k"] = np.array(list(opts.distribution.keys()), dtype=np.uint16)
        keep["init_c"] = np.array(list(opts.distribution.values()), dtype=np.uint64)
        p.n_init, p.init_k, p.init_c = len(keep["init_k"]), keep["init_k"].ctypes.data, keep["init_c"].ctypes.data
        snaps = list(opts.snapshots) if snapshots else []
        keep["snap"] = np.array(snaps, dtype=np.uint64)
        p.n_snapshots = len(snaps)
        p.snapshot_cells = keep["snap"].ctypes.data if snaps else None
        if rates_per_run is not None:
            keep["rates"] = rates_per_run
            p.rates_per_run = _addr(rates_per_run)
        if replay is not None:
            keep["replay"], keep["replay_off"] = replay, replay_offsets
            p.rng_mode, p.replay, p.replay_offsets = RNG_REPLAY, _addr(replay), _addr(replay_offsets)
        if replay_u64 is not None:
            keep["replay_u64"], keep["replay_off"] = replay_u64, replay_offsets
            p.rng_mode, p.replay_u64, p.replay_offsets = RNG_UNIFORMS, _addr(replay_u64), _addr(replay_offsets)
        p.dyn_points, p.dyn_dt = dyn_points, dyn_dt
        if abc_target is not None:
            keep["abc"] = abc_target
            p.abc_enabled, p.abc_target_hist, p.abc_target_len = 1, _addr(abc_target), len(abc_target)
            for i in range(4):
                p.abc_thresholds[i] = abc_thresholds[i]
        p.state_mode, p.tile_width, p.smem_bins = state_mode, tile_width, smem_bins
        p.max_copies, p.hist_stride = max_copies, hist_stride
        p.flags = WANT_DIGEST if digest else 0
        p.spill_records = spill_records
        p.slice_events = slice_events
        subs = list(opts.subsamples or []) if subsamples is None else list(subsamples)
        if subs:  # main.rs:110-123
            keep["subs"] = np.array(subs, dtype=np.uint64)
            p.n_subsamples, p.subsample_cells = len(subs), keep["subs"].ctypes.data
        p._keep = keep
        return p

    def run(self, opts, n_runs=None, idx_begin=None, want=("stop_reason", "nminus", "nplus", "time", "n_events",
                                                           "kmax", "hist"), results=None, **kw):
        """ecdna_b200_run: host buffers in and out (what a reference-side FFI caller does).  `results`: a
        Results object to reuse (e.g. one whose arrays live in pinned host memory)."""
        n_runs = opts.runs if n_runs is None else n_runs
        idx_begin = opts.idx_begin if idx_begin is None else idx_begin
        p = self.make_params(opts, n_runs, **kw)
        stride = p.hist_stride or 512
        res = results if results is not None else Results(n_runs, p.n_snapshots, p.dyn_points, stride, want, p.n_subsamples)
        assert res.n_runs == n_runs
        self._check(lib().ecdna_b200_run(self._h, C.byref(p), idx_begin, n_runs, C.byref(res.struct)))
        res.timing = self.timing()
        return res

    _run_sparse_fn, _sparse_fetch_fn = "ecdna_b200_run_sparse", "ecdna_b200_sparse_fetch"

    def run_sparse(self, opts, n_runs=None, idx_begin=None, want=("stop_reason", "nminus", "nplus", "time", "n_events",
                                                                  "kmax"), arena_words=None, **kw):
        """ecdna_b200_run_sparse: the distributions come back as descriptors + one arena of occupied bins
        (res.sparse).  arena_words=None: a first guess, then ecdna_b200_sparse_fetch with the size the library
        reports (the two-call pattern; the batch is not simulated again)."""
        n_runs = opts.runs if n_runs is None else n_runs
        idx_begin = opts.idx_begin if idx_begin is None else idx_begin
        p = self.make_params(opts, n_runs, **kw)
        res = Results(n_runs, p.n_snapshots, p.dyn_points, p.hist_stride or 512, want, p.n_subsamples)
        sp = Sparse(n_runs, p.n_snapshots, p.n_subsamples, 0 if arena_words is None else arena_words)
        rc = getattr(lib(), self._run_sparse_fn)(self._h, C.byref(p), idx_begin, n_runs, C.byref(res.struct), C.byref(sp.struct))
        res.refetched = False
        if rc == ERR_ARENA and arena_words is None:
            sp.resize(sp.arena_used)
            rc = getattr(lib(), self._sparse_fetch_fn)(self._h, C.byref(sp.struct))
            res.refetched = True
        self._check(rc)
        res.sparse = sp
        res.timing = self.timing()
        return res

    def run_device(self, opts, n_runs, idx_begin, results_struct, stream=None, **kw):
        """ecdna_b200_run_device: outputs (and bulk inputs) are device pointers; asynchronous."""
        p = self.make_params(opts, n_runs, **kw)
        self._check(lib().ecdna_b200_run_device(self._h, C.byref(p), idx_begin, n_runs, C.byref(results_struct),
                                                C.c_void_p(stream) if stream else None))
        return p

    def timing(self):
        t = TimingT()
        self._check(lib().ecdna_b200_get_timing(self._h, C.byref(t)))
        return t

    def abc_draw_priors(self, seed, idx_begin, n_runs, b0=1.0, b1_range=(1.0, 2.0), d0_range=(0.0, 0.5),
                        d1_range=(0.0, 0.5)):
        out = np.zeros((n_runs, 4), dtype=np.float32)
        r1, r2, r3 = (C.c_float * 2)(*b1_range), (C.c_float * 2)(*d0_range), (C.c_float * 2)(*d1_range)
        self._check(lib().ecdna_b200_abc_draw_priors(self._h, seed, idx_begin, n_runs, b0, r1, r2, r3,
                                                     out.ctypes.data))
        return out

    def abc_draw_priors_device(self, seed, idx_begin, n_runs, rates_dev_ptr, b0=1.0, b1_range=(1.0, 2.0),
                               d0_range=(0.0, 0.5), d1_range=(0.0, 0.5), stream=None):
        r1, r2, r3 = (C.c_float * 2)(*b1_range), (C.c_float * 2)(*d0_range), (C.c_float * 2)(*d1_range)
        self._check(lib().ecdna_b200_abc_draw_priors_device(self._h, seed, idx_begin, n_runs, b0, r1, r2, r3,
                                                            C.c_void_p(rates_dev_ptr),
                                                            C.c_void_p(stream) if stream else None))

    def abc_smc_propose(self, seed, idx_begin, n, prev_rates, cum_weights, sigma, b1_range=(1.0, 2.0),
                        d0_range=(0.0, 0.5), d1_range=(0.0, 0.5)):
        """ecdna_b200_abc_smc_propose: (rates [n][4] f32, parent [n] u32) of draws idx_begin .. idx_begin + n - 1,
        proposed from the population prev_rates [M][4] with cumulative weights cum_weights [M] (f64)."""
        prev = np.ascontiguousarray(prev_rates, dtype=np.float32).reshape(-1, 4)
        cum = np.ascontiguousarray(cum_weights, dtype=np.float64)
        assert len(cum) == len(prev)
        rates, parent = np.zeros((n, 4), dtype=np.float32), np.zeros(n, dtype=np.uint32)
        self._check(lib().ecdna_b200_abc_smc_propose(self._h, seed, idx_begin, n, prev.ctypes.data, cum.ctypes.data,
                                                     len(prev), (C.c_double * 3)(*sigma), *_ranges(b1_range, d0_range,
                                                                                                  d1_range),
                                                     rates.ctypes.data, parent.ctypes.data))
        return rates, parent

    def abc_smc_weights(self, new_rates, prev_rates, prev_weights, sigma, b1_range=(1.0, 2.0), d0_range=(0.0, 0.5),
                        d1_range=(0.0, 0.5)):
        """ecdna_b200_abc_smc_weights: normalised importance weights [N] (f64) of new_rates [N][4] against the
        population prev_rates [M][4] with weights prev_weights [M]."""
        new = np.ascontiguousarray(new_rates, dtype=np.float32).reshape(-1, 4)
        prev = np.ascontiguousarray(prev_rates, dtype=np.float32).reshape(-1, 4)
        w = np.ascontiguousarray(prev_weights, dtype=np.float64)
        assert len(w) == len(prev)
        out = np.zeros(len(new), dtype=np.float64)
        self._check(lib().ecdna_b200_abc_smc_weights(self._h, new.ctypes.data, len(new), prev.ctypes.data, w.ctypes.data,
                                                     len(prev), (C.c_double * 3)(*sigma),
                                                     *_ranges(b1_range, d0_range, d1_range), out.ctypes.data))
        return out

    def abc_pack(self, results_struct, rates_dev_ptr, base_rates, idx_begin, n_runs, hist_stride, rec_bins, capacity,
                 records_dev_ptr, count_dev_ptr, stream=None):
        """ecdna_b200_abc_pack: accepted draws -> fixed-stride records on the device, in index order."""
        base = (C.c_float * 4)(*base_rates)
        self._check(lib().ecdna_b200_abc_pack(self._h, C.byref(results_struct),
                                              C.c_void_p(rates_dev_ptr) if rates_dev_ptr else None, base, idx_begin,
                                              n_runs, hist_stride, rec_bins, capacity, C.c_void_p(records_dev_ptr),
                                              C.c_void_p(count_dev_ptr), C.c_void_p(stream) if stream else None))

    def comm_init(self, unique_id, rank, world):
        """ecdna_b200_comm_init: join the NCCL communicator of the GPUs that share a batch."""
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(unique_id)
        self._check(lib().ecdna_b200_comm_init(self._h, buf, rank, world))

    def abc_allgather(self, records_dev_ptr, count_dev_ptr, rec_bins, capacity, all_records_dev_ptr, all_counts_dev_ptr,
                      stream=None):
        """ecdna_b200_abc_allgather: counts + record blocks of every rank, two ncclAllGather in one group."""
        self._check(lib().ecdna_b200_abc_allgather(self._h, C.c_void_p(records_dev_ptr), C.c_void_p(count_dev_ptr),
                                                   rec_bins, capacity, C.c_void_p(all_records_dev_ptr),
                                                   C.c_void_p(all_counts_dev_ptr),
                                                   C.c_void_p(stream) if stream else None))


class MultiContext(Context):
    """Several GPUs of one box from one process (ecdna_b200_multi): the index range is cut into contiguous
    blocks, one per GPU; outputs are identical to a one-GPU run of the same range."""

    def __init__(self, devices=None):
        self._h = C.c_void_p()
        arr = (C.c_int * len(devices))(*devices) if devices else None
        rc = lib().ecdna_b200_multi_create(arr, len(devices) if devices else 0, C.byref(self._h))
        if rc != 0:
            raise EcdnaB200Error(f"ecdna_b200_multi_create failed with status {rc} (3 = no sm_100 device)")
        self.n_devices = lib().ecdna_b200_multi_device_count(self._h)

    def close(self):
        if self._h:
            lib().ecdna_b200_multi_destroy(self._h)
            self._h = C.c_void_p()

    def _check(self, rc):
        if rc != 0:
            raise EcdnaB200Error(f"status {rc}: {lib().ecdna_b200_multi_last_error(self._h).decode()}")

    _run_sparse_fn, _sparse_fetch_fn = "ecdna_b200_multi_run_sparse", "ecdna_b200_multi_sparse_fetch"

    def run(self, opts, n_runs=None, idx_begin=None, want=("stop_reason", "nminus", "nplus", "time", "n_events",
                                                           "kmax", "hist"), **kw):
        n_runs = opts.runs if n_runs is None else n_runs
        idx_begin = opts.idx_begin if idx_begin is None else idx_begin
        p = self.make_params(opts, n_runs, **kw)
        res = Results(n_runs, p.n_snapshots, p.dyn_points, p.hist_stride or 512, want, p.n_subsamples)
        self._check(lib().ecdna_b200_multi_run(self._h, C.byref(p), idx_begin, n_runs, C.byref(res.struct)))
        res.timing = self.timing()
        return res

    def timing(self):
        t = TimingT()
        self._check(lib().ecdna_b200_multi_get_timing(self._h, C.byref(t)))
        return t

    def abc_smc(self, opts, target, thresholds, population, quantile=0.5, max_generations=10,
                max_simulations=10_000_000, b1_range=(1.0, 2.0), d0_range=(0.0, 0.5), d1_range=(0.0, 0.5), chunk=0,
                idx_begin=None, **kw):
        """ecdna_b200_abc_smc over the GPUs of this handle.  Returns a dict: the per-particle arrays of
        SMC_PARTICLE_FIELDS as [generations][population][...], the per-generation arrays of SMC_GENERATION_FIELDS,
        "generations", "status" (one of SMC_STATUS) and "options" (what write_abc_smc records)."""
        idx_begin = opts.idx_begin if idx_begin is None else idx_begin
        p = self.make_params(opts, 1, abc_target=np.ascontiguousarray(target, dtype=np.uint64),
                             abc_thresholds=thresholds, snapshots=False, **kw)
        o = SmcOptionsT()
        o.population, o.quantile, o.max_generations = population, quantile, max_generations
        o.max_simulations, o.idx_begin, o.chunk = max_simulations, idx_begin, chunk
        o.b1_range[:], o.d0_range[:], o.d1_range[:] = b1_range, d0_range, d1_range
        r = SmcResultT()
        out = {}
        G, M = max(int(max_generations), 1), max(int(population), 1)
        for name, dtype, tail in SMC_PARTICLE_FIELDS:
            out[name] = np.zeros((G, M) + tail, dtype=dtype)
            setattr(r, name, out[name].ctypes.data)
        for name, dtype, tail in SMC_GENERATION_FIELDS:
            out[name] = np.zeros((G,) + tail, dtype=dtype)
            setattr(r, name, out[name].ctypes.data)
        self._check(lib().ecdna_b200_abc_smc(self._h, C.byref(p), C.byref(o), C.byref(r)))
        g = int(r.generations)
        out = {k: v[:g] for k, v in out.items()}
        out["generations"], out["status"] = g, SMC_STATUS[r.status]
        out["options"] = {"seed": int(opts.seed), "idx_begin": int(idx_begin), "population": int(population),
                          "quantile": float(quantile), "max_generations": int(max_generations),
                          "max_simulations": int(max_simulations), "b1_range": [float(np.float32(x)) for x in b1_range],
                          "d0_range": [float(np.float32(x)) for x in d0_range],
                          "d1_range": [float(np.float32(x)) for x in d1_range],
                          "thresholds": [float(np.float32(x)) for x in thresholds]}
        return out


def _ranges(*ranges):
    return [(C.c_float * 2)(*r) for r in ranges]


def _addr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return int(a)


class Results:
    """Caller-owned host buffers for ecdna_b200_results_t."""

    def __init__(self, n_runs, n_snapshots, dyn_points, hist_stride, want, n_subsamples=0, alloc=None):
        """alloc(shape, dtype) -> ndarray: where the columns live (default: np.zeros; bench.py passes an allocator
        of page-locked memory)."""
        self.struct = ResultsT()
        self.n_runs = n_runs
        alloc = alloc or (lambda shape, dtype: np.zeros(shape, dtype=dtype))
        for name, dtype, shape in RESULT_FIELDS:
            if name not in want:
                continue
            tail = shape(n_snapshots, dyn_points, hist_stride, n_subsamples)
            if any(t == 0 for t in tail):
                continue
            arr = alloc((n_runs,) + tail, dtype)
            setattr(self, name, arr)
            setattr(self.struct, name, arr.ctypes.data)

    @property
    def stop(self):
        return self.stop_reason & 0xFF


def device_results(torch, n_runs, want, n_snapshots=0, dyn_points=0, hist_stride=512, device="cuda", n_subsamples=0):
    """Allocate the result columns as torch tensors on the GPU and return (struct, tensors)."""
    tmap = {np.uint32: torch.int32, np.uint64: torch.int64, np.float32: torch.float32, np.uint8: torch.uint8}
    s = ResultsT()
    tensors = {}
    for name, dtype, shape in RESULT_FIELDS:
        if name not in want:
            continue
        tail = shape(n_snapshots, dyn_points, hist_stride, n_subsamples)
        if any(t == 0 for t in tail):
            continue
        t = torch.zeros((n_runs,) + tail, dtype=tmap[dtype], device=device)
        tensors[name] = t
        setattr(s, name, t.data_ptr())
    return s, tensors
