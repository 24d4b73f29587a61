/*
 * ecdna_b200.h -- C ABI of libecdna_b200.so, the B200 (sm_100a) backend for ecdna-evo's hot path.
 *
 * The reference has no FFI; its seam is the per-replicate closure `run_simulations(idx)`
 * (reference src/main.rs:55-211) that rayon maps over idx in [seed*10, seed*10+runs)
 * (main.rs:214-225).  One call of ecdna_b200_run() replaces that closure for a whole index range:
 * it takes the fields of SimulationOptions (main.rs:28-44) and gives back, per replicate, what the
 * closure produces: the stop reason, (nminus, nplus), the clock (main.rs:205-210) and the ecDNA
 * distributions that `save` (src/process.rs:31-55) would have written -- at the end of the run
 * (main.rs:100-109) and at every snapshot size (process.rs:122-145, 267-290).  Writing the JSON
 * files stays on the host side (INTEGRATION.md).
 *
 * Plain C: fixed-width integers, f32 rates (they are f32 in the reference and appear in file
 * names), caller-owned buffers, int status codes, no exceptions, no aborts.
 */
#ifndef ECDNA_B200_H
#define ECDNA_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ECDNA_B200_ABI_VERSION 3

/* status codes returned by every entry point */
enum {
  ECDNA_B200_OK = 0,
  ECDNA_B200_ERR_BAD_PARAMS = 1,  /* see ecdna_b200_last_error() */
  ECDNA_B200_ERR_CUDA = 2,        /* a CUDA call failed; never falls back to the CPU */
  ECDNA_B200_ERR_NO_DEVICE = 3,   /* no sm_100 device: the library refuses to run */
  ECDNA_B200_ERR_ALLOC = 4,
  ECDNA_B200_ERR_INTERNAL = 5,    /* the library lost track of a replicate (results incomplete); a bug */
  ECDNA_B200_ERR_COMM = 6,        /* NCCL is missing or a collective failed */
  ECDNA_B200_ERR_ARENA = 7        /* sparse return: the caller's arena is too small; the descriptors were written,
                                     sparse->arena_used holds the words needed: ecdna_b200_sparse_fetch() */
};

/* sosa reaction order, main.rs:140-145; live variants of EcDNAEvent, process.rs:20-29 */
enum {
  ECDNA_B200_EV_BIRTH_NMINUS = 0, ECDNA_B200_EV_BIRTH_NPLUS = 1,
  ECDNA_B200_EV_DEATH_NMINUS = 2, ECDNA_B200_EV_DEATH_NPLUS = 3
};

/* --segregation, src/clap_app.rs:232-238 (same order as SegregationOptions) */
enum {
  ECDNA_B200_SEG_DETERMINISTIC = 0, ECDNA_B200_SEG_BINOMIAL_NO_UNEVEN = 1,
  ECDNA_B200_SEG_BINOMIAL = 2, ECDNA_B200_SEG_BINOMIAL_NO_NMINUS = 3
};

/* per-run stop reason: sosa::StopReason as printed at main.rs:205-210, plus the conditions the
   reference turns into a panic (reported per run so one bad replicate does not kill the batch) */
enum {
  ECDNA_B200_STOP_NO_INDIVIDUALS = 0,
  ECDNA_B200_STOP_MAX_ITERS = 1,
  ECDNA_B200_STOP_MAX_TIME = 2,
  ECDNA_B200_STOP_MAX_CELLS = 3,
  ECDNA_B200_STOP_ABSORBING = 4,      /* cells left but all propensities zero */
  ECDNA_B200_STOP_COPY_OVERFLOW = 5,  /* k*2 overflows u16: src/proliferation.rs:63-67 panics */
  ECDNA_B200_STOP_HIST_OVERFLOW = 6,  /* copy number beyond params.max_copies */
  ECDNA_B200_STOP_REPLAY_END = 7,     /* replay stream exhausted before a stop rule fired */
  ECDNA_B200_STOP_REPLAY_BAD = 8      /* replay record inconsistent with the population */
};
/* bit set in stop_reason when the final histogram did not fit hist_stride bins */
#define ECDNA_B200_FLAG_HIST_TRUNCATED 0x100u
/* bit set when the replicate's histogram left shared memory for the HBM arena */
#define ECDNA_B200_FLAG_SPILLED 0x200u

enum {
  ECDNA_B200_RNG_PHILOX = 0,   /* native: Philox4x32-10 keyed (seed, replicate, event), Gillespie's direct
                                  method (one exponential + one uniform per event; stream v2, DESIGN.md 3.3) */
  ECDNA_B200_RNG_REPLAY = 1,   /* decision stream {event, dt, k, k1}: drives the histogram kernel */
  ECDNA_B200_RNG_UNIFORMS = 2  /* the reference generator's raw u64 stream: re-runs the replicate on the
                                  reference's own per-cell layout (verification mode, one thread per
                                  replicate; outputs: stop_reason, nminus, nplus, time, n_events, kmax,
                                  hash, chain, hist, sum_k, n_div, n_death; no snapshots/dynamics/ABC) */
};
enum { ECDNA_B200_STATE_AUTO = 0, ECDNA_B200_STATE_SMEM = 1, ECDNA_B200_STATE_HBM = 2 };

/* ecdna_b200_params_t.flags */
#define ECDNA_B200_WANT_DIGEST 0x1u /* maintain the histogram hash and the per-event chain digest */
#define ECDNA_B200_KEEP_ORDER 0x2u  /* start the replicates in index order (default with per-run rates: the ones
                                       expected to run longest first, which shortens the tail of the batch;
                                       results never depend on the order) */

/* one record of the replay stream: the decisions of one iteration of sosa::simulate, in the order
   the reference takes them (waiting time, event, cell picked, first daughter). 12 bytes. */
typedef struct {
  float dt;       /* NextReaction.time, added to the clock at process.rs:184/336 */
  uint16_t k;     /* copies of the cell removed at proliferation.rs:57 / 126-133, else 0 */
  uint16_t k1;    /* first value returned by Segregate::ecdna_segregation (segregation.rs:75-84) */
  uint8_t event;  /* ECDNA_B200_EV_* */
  uint8_t pad[3];
} ecdna_b200_replay_event_t;

/* The run parameters: SimulationOptions (main.rs:28-44) flattened. */
typedef struct {
  uint32_t abi_version;  /* ECDNA_B200_ABI_VERSION */
  float b0, b1, d0, d1;  /* main.rs:31-34; d0=d1=0 is the pure-birth process (clap_app.rs:165-200) */
  uint32_t segregation;  /* ECDNA_B200_SEG_* */
  uint64_t max_cells;    /* options.max_cells, clap_app.rs:208; must be < 2^32 */
  uint64_t max_iter;     /* options.max_iter_time.iter (MAX_ITER, main.rs:23); must be < 2^32 */
  float max_time;        /* options.max_iter_time.time, clap_app.rs:205 */
  uint64_t seed;         /* --seed, clap_app.rs:63-64 */
  uint32_t bd_count_mode; /* 0: max_cells counts cells (documented CLI meaning, clap_app.rs:59-61);
                             1: counts sosa's population array, which process.rs:339-344 fills with
                             [n-,n+,n-,n+] for the birth-death process (SURVEY 8c R1) */

  /* initial distribution (clap_app.rs:177-192): sparse histogram, k == 0 is the ecDNA- count */
  uint32_t n_init;
  const uint16_t* init_k;
  const uint64_t* init_c;

  /* snapshot sizes (clap_app.rs:102-134), ascending; may be NULL/0 */
  uint32_t n_snapshots;
  const uint64_t* snapshot_cells;

  /* optional per-run rates [n_runs][4] = b0,b1,d0,d1: the ABC prior draws (abc.md:44-52) */
  const float* rates_per_run;

  /* random source */
  uint32_t rng_mode;                       /* ECDNA_B200_RNG_* */
  const ecdna_b200_replay_event_t* replay; /* all runs' records, concatenated */
  const uint64_t* replay_offsets;          /* [n_runs + 1] record offsets into `replay` */

  /* dynamics (CHANGELOG.md:34-40): dyn_points samples at multiples of dyn_dt of Gillespie time */
  uint32_t dyn_points;
  float dyn_dt;

  /* ABC epilogue (abc.md:38-55): distances to a target distribution and the accept flag */
  uint32_t abc_enabled;
  const uint64_t* abc_target_hist; /* dense, [0] = cells without ecDNA */
  uint32_t abc_target_len;
  float abc_thresholds[4];         /* ks(ecdna), rel. mean, rel. entropy, rel. frequency */

  /* engine knobs (0 = default) */
  uint32_t state_mode;  /* ECDNA_B200_STATE_* */
  uint32_t tile_width;  /* lanes per replicate: 32 (a warp), 16, 8, 4, 2 or 1 (2, 1: native random source only);
                           0 = the widest tile that keeps the batch within about one warp per SM scheduler
                           (<= 592 replicates: 32, <= 1184: 16, <= 2368: 8, <= 6156: 4, more: 1 - a lane per
                           replicate - when the initial copy numbers are <= 16, else 2) */
  uint32_t smem_bins;   /* histogram bins per replicate held in shared memory (rounded up to 128);
                           0 = 512, or 256 for 4- and 2-lane tiles when the initial copy numbers are <= 16 */
  uint32_t max_copies;  /* largest copy number the HBM arena holds (<= 65535) */
  uint32_t hist_stride; /* bins per output histogram */
  uint32_t flags;       /* ECDNA_B200_WANT_* */
  uint32_t spill_records; /* parked replicates whose state is saved for the HBM launch (others restart);
                             0 = default (32768), 0xFFFFFFFF = none */
  /* RNG_UNIFORMS: every u64 the reference's ChaCha8Rng (main.rs:57-58) handed out, all runs back to
     back; replay_offsets[n_runs + 1] then counts u64 */
  const uint64_t* replay_u64;
  /* Time slicing.  A batch that is somewhat larger than the number of replicates the GPU runs at its
     most efficient occupancy (rayon's for_each over a range that is not a multiple of the worker
     count, main.rs:221-224) is run with that many tiles; every slice_events events a replicate makes
     room for the one that waits longest.  Results do not depend on it.  0 = automatic,
     0xFFFFFFFF = never, otherwise the slice length in events (rounded up to a power of two). */
  uint32_t slice_events;
  /* --subsamples (clap_app.rs, main.rs:110-123): after the final state of every replicate, one
     sample of subsample_cells[j] cells drawn without replacement from it (a size >= the population
     gives the population).  At most 65535 sizes; may be NULL/0. */
  uint32_t n_subsamples;
  const uint64_t* subsample_cells;
} ecdna_b200_params_t;

/* Per-run outputs.  Every pointer is optional (NULL = not wanted) and caller-owned.
   For ecdna_b200_run they are host pointers, for ecdna_b200_run_device device pointers. */
typedef struct {
  uint32_t* stop_reason; /* [n]  ECDNA_B200_STOP_* | ECDNA_B200_FLAG_* */
  uint64_t* nminus;      /* [n]  final_state[0], main.rs:124-128 */
  uint64_t* nplus;       /* [n]  final_state[1] */
  float* time;           /* [n]  process.time */
  uint64_t* n_events;    /* [n]  iterations of sosa::simulate */
  uint32_t* kmax;        /* [n]  largest copy number that ever occurred */
  float* mean;           /* [n]  summary statistics of the final distribution (SURVEY 8c R8) */
  float* frequency;
  float* entropy;
  float* variance;
  float* abc_distance;   /* [n][4] ks, rel.mean, rel.entropy, rel.frequency */
  uint8_t* abc_accept;   /* [n] */
  uint64_t* hash;        /* [n]  digest of the final histogram (WANT_DIGEST) */
  uint64_t* chain;       /* [n]  chained digest of the state after every event (WANT_DIGEST) */
  uint32_t* hist;        /* [n][hist_stride] final distribution, [0] = nminus */
  uint32_t* snap_count;  /* [n]  snapshots taken */
  uint64_t* snap_cells;  /* [n][n_snapshots] */
  float* snap_time;      /* [n][n_snapshots] */
  uint32_t* snap_hist;   /* [n][n_snapshots][hist_stride] */
  uint32_t* dyn_count;   /* [n] */
  float* dyn;            /* [n][dyn_points][5] nminus, nplus, mean, variance, entropy */
  uint64_t* sum_k;       /* [n]  sum over ecDNA+ events of the live histogram width (roofline) */
  uint32_t* n_div;       /* [n]  ecDNA+ divisions */
  uint32_t* n_death;     /* [n]  ecDNA+ deaths */
  uint32_t* sub_hist;    /* [n][n_subsamples][hist_stride] the subsampled distributions, [0] = cells without ecDNA */
} ecdna_b200_results_t;

/* Bytes a caller must provide behind every pointer of ecdna_b200_results_t for a batch of n_runs replicates
   (same member order; 0 = that output does not exist for these parameters, e.g. snap_hist without snapshots).
   The two-call pattern of the boundary: ecdna_b200_query_sizes -> the caller allocates -> ecdna_b200_run. */
typedef struct {
  uint64_t stop_reason, nminus, nplus, time, n_events, kmax, mean, frequency, entropy, variance, abc_distance,
      abc_accept, hash, chain, hist, snap_count, snap_cells, snap_time, snap_hist, dyn_count, dyn, sum_k, n_div,
      n_death, sub_hist;
} ecdna_b200_result_sizes_t;

/* what the last run on a context measured (CUDA events on the context's stream) */
typedef struct {
  float kernel_ms;         /* the SSA kernel alone */
  float total_ms;          /* copies + kernel, host-buffer entry point only */
  uint32_t kernel_launches; /* 1, or 2 when the HBM launch for parked replicates was enqueued */
  uint32_t tile_width, smem_bins, grid_blocks, block_threads, blocks_per_sm;
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t total_events;   /* sum of n_events */
  uint64_t alg_bytes;      /* SURVEY 8(d) flat-histogram model summed over all events */
  uint32_t n_spilled;      /* replicates that moved to the HBM arena */
  uint32_t slice_events;   /* slice length the launch used; 0 = it did not time-slice */
  uint64_t n_slices;       /* times a replicate made room for another one */
  uint64_t n_idle_spells;  /* times a tile of a sliced launch found nothing to run and looked again later */
  uint64_t n_finished;     /* replicates that went through the epilogue; != n_runs is ECDNA_B200_ERR_INTERNAL */
} ecdna_b200_timing_t;

typedef struct ecdna_b200_ctx ecdna_b200_ctx;

/* One context per process and GPU.  `device` is the CUDA ordinal. */
int ecdna_b200_create(int device, ecdna_b200_ctx** out);
void ecdna_b200_destroy(ecdna_b200_ctx* ctx);
const char* ecdna_b200_last_error(const ecdna_b200_ctx* ctx);
int ecdna_b200_abi_version(void);

/* Sizes of the per-run outputs for `params` and n_runs (no GPU needed, no context). */
int ecdna_b200_query_sizes(const ecdna_b200_params_t* params, uint64_t n_runs, ecdna_b200_result_sizes_t* sizes);

/* What the library would do with a batch (no GPU needed; the same code run plans its launch with):
   lanes per replicate, blocks of 128 threads per SM, tiles (replicates resident at once) and whether
   the launch is time-sliced, for a device with sm_count SMs on which max_blocks_per_sm blocks of the
   kernel fit (B200: 148 SMs; 5 for 4-lane tiles with 256 bins, 3 for 2-lane tiles).
   tile_width / slice_events as in ecdna_b200_params_t (0 = automatic). */
int ecdna_b200_plan(uint64_t n_runs, uint32_t tile_width, uint32_t slice_events, uint32_t sm_count,
                    uint32_t max_blocks_per_sm, uint32_t* lanes, uint32_t* blocks_per_sm, uint32_t* tiles,
                    uint32_t* sliced);

/* Replaces main.rs:55-211 for idx in [idx_begin, idx_begin + n_runs).  Host buffers in and out;
   blocking; host<->device copies happen inside. */
int ecdna_b200_run(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* params, uint64_t idx_begin, uint64_t n_runs,
                   const ecdna_b200_results_t* results);

/* Same, but `results` (and params->rates_per_run, replay, replay_offsets, abc_target_hist when
   given) are DEVICE pointers and the work is enqueued on `cuda_stream` (a cudaStream_t, NULL =
   the context's own stream) without a final synchronisation. */
int ecdna_b200_run_device(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* params, uint64_t idx_begin,
                          uint64_t n_runs, const ecdna_b200_results_t* results, void* cuda_stream);

/* Waits for everything enqueued by the context and fills `t` from its CUDA events. */
int ecdna_b200_get_timing(ecdna_b200_ctx* ctx, ecdna_b200_timing_t* t);

/* ABC prior draws (SURVEY 8d C4): rates[i] = {b0, U(lo1,hi1), U(lo_d0,hi_d0), U(lo_d1,hi_d1)} from
   Philox keyed (seed, idx_begin + i); device kernel, host output. */
int ecdna_b200_abc_draw_priors(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n_runs, float b0,
                               const float b1_range[2], const float d0_range[2], const float d1_range[2],
                               float* rates_out /* [n_runs][4], host */);

/* Same draws, left on the device: `rates_dev` is a device buffer [n_runs][4]; enqueued on `cuda_stream`
   (NULL = the context's stream) without a synchronisation. */
int ecdna_b200_abc_draw_priors_device(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n_runs, float b0,
                                      const float b1_range[2], const float d0_range[2], const float d1_range[2],
                                      float* rates_dev, void* cuda_stream);

/* ---- several GPUs of one box from one process (the reference's rayon loop, main.rs:214-225) ----
   The index range of a batch is cut into contiguous blocks, one per GPU, each driven by its own host
   thread and context; the blocks' results are written into the caller's arrays at the block's offset, so
   the outputs are identical to a one-GPU run of the same range.  devices == NULL / n_devices == 0: every
   visible sm_100 device. */
typedef struct ecdna_b200_multi ecdna_b200_multi;
int ecdna_b200_multi_create(const int* devices, int n_devices, ecdna_b200_multi** out);
void ecdna_b200_multi_destroy(ecdna_b200_multi* m);
int ecdna_b200_multi_device_count(const ecdna_b200_multi* m);
const char* ecdna_b200_multi_last_error(const ecdna_b200_multi* m);
/* ecdna_b200_run over all GPUs of `m` (host buffers in and out; blocking) */
int ecdna_b200_multi_run(ecdna_b200_multi* m, const ecdna_b200_params_t* params, uint64_t idx_begin, uint64_t n_runs,
                         const ecdna_b200_results_t* results);
/* times of the slowest block, counts summed over the blocks */
int ecdna_b200_multi_get_timing(ecdna_b200_multi* m, ecdna_b200_timing_t* t);

/* ---- sparse return of the distributions ----
   The reference writes one JSON map {copy number: cells} per saved state (process.rs:31-55), whose size follows the
   copy numbers that occur, not a fixed stride.  The dense columns hist / snap_hist / sub_hist cost hist_stride words
   per distribution on the host and over PCIe whatever they hold (C2 with the default eleven snapshots: 12 x 4 KiB per
   replicate for ~60 occupied bins each).  The sparse return gives, per distribution, one descriptor and the bins
   k_min .. k_min + k_len - 1 (first to last occupied copy number >= 1) in one flat arena of 32-bit words; the
   distributions are measured, laid out (prefix sum) and packed on the device, and only descriptors + arena cross
   the bus.  bin 0 (cells without ecDNA) lives in the descriptor: it is far from the window of a population whose
   copy numbers grew. */
typedef struct {
  uint64_t cells;   /* cells of this distribution: nminus + the bins of the window */
  uint64_t nminus;  /* cells without ecDNA (bin 0 of the dense form) */
  uint64_t offset;  /* first word of the window in the arena */
  float time;       /* the clock when it was taken (snapshot: process.rs:122-145; final state and samples: the end) */
  uint32_t k_len;   /* bins stored; 0: no cell carries ecDNA */
  uint16_t k_min;   /* copy number of the first stored bin */
  uint16_t flags;   /* ECDNA_B200_DIST_* */
  uint32_t reserved;
} ecdna_b200_dist_t;
#define ECDNA_B200_DIST_TAKEN 0x1u     /* 0: a snapshot size the replicate never reached (everything else is 0 too) */
#define ECDNA_B200_DIST_TRUNCATED 0x2u /* the replicate carries ECDNA_B200_FLAG_HIST_TRUNCATED: bins beyond hist_stride are missing */

/* caller-owned; every descriptor pointer is optional */
typedef struct {
  ecdna_b200_dist_t* final_dist; /* [n]               the final distributions (main.rs:100-109) */
  ecdna_b200_dist_t* snap_dist;  /* [n][n_snapshots]  the snapshots, in the order of params.snapshot_cells */
  ecdna_b200_dist_t* sub_dist;   /* [n][n_subsamples] the samples of --subsamples (main.rs:110-123) */
  uint32_t* arena;               /* [arena_words] */
  uint64_t arena_words;          /* capacity of `arena` in 32-bit words (may be 0 to ask for the size only) */
  uint64_t arena_used;           /* out: words the batch needs */
} ecdna_b200_sparse_t;

/* ecdna_b200_run with the distributions returned sparsely: results->hist / snap_hist / sub_hist may be NULL (they
   are still filled when given); every other column of `results` as in ecdna_b200_run.  hist_stride still bounds the
   copy numbers a distribution can hold (on the device only).  When sparse->arena_words < sparse->arena_used the
   descriptors are written, the arena is not, and the call returns ECDNA_B200_ERR_ARENA: the packed batch stays on
   the device until the context's next run, and ecdna_b200_sparse_fetch copies it into a large enough arena without
   simulating again. */
int ecdna_b200_run_sparse(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* params, uint64_t idx_begin, uint64_t n_runs,
                          const ecdna_b200_results_t* results, ecdna_b200_sparse_t* sparse);
int ecdna_b200_sparse_fetch(ecdna_b200_ctx* ctx, ecdna_b200_sparse_t* sparse);
/* the same over all GPUs of `m`: every GPU packs its block, the blocks follow each other in the arena in index
   order and the descriptors' offsets are absolute */
int ecdna_b200_multi_run_sparse(ecdna_b200_multi* m, const ecdna_b200_params_t* params, uint64_t idx_begin,
                                uint64_t n_runs, const ecdna_b200_results_t* results, ecdna_b200_sparse_t* sparse);
int ecdna_b200_multi_sparse_fetch(ecdna_b200_multi* m, ecdna_b200_sparse_t* sparse);

/* ---- the one exchange step of the path: all-gather of the accepted ABC draws (abc.md:57-78) ----
   A record is ECDNA_B200_ABC_REC_HEADER + rec_bins 32-bit words:
     [0..1] replicate index (lo, hi)   [2..5] b0, b1, d0, d1 (f32 bits)   [6..9] the four distances (f32 bits)
     [10] mean  [11] frequency  [12] entropy (f32 bits)   [13] cells   [14] kmax   [15] stop_reason
     [16..] the final distribution, rec_bins bins ([16] = cells without ecDNA)                               */
#define ECDNA_B200_ABC_REC_HEADER 16u
#define ECDNA_B200_COMM_ID_BYTES 128

/* Packs the accepted draws (abc_accept != 0) of a batch whose result columns live on the device into
   records, in index order, on `cuda_stream`; *count_dev (device) receives the number of accepted draws,
   which may exceed `capacity` (then only the first `capacity` records were written).  rates_dev: the
   per-run rates [n_runs][4] on the device, or NULL (then base_rates[4] goes into every record). */
int ecdna_b200_abc_pack(ecdna_b200_ctx* ctx, const ecdna_b200_results_t* results_dev, const float* rates_dev,
                        const float base_rates[4], uint64_t idx_begin, uint64_t n_runs, uint32_t hist_stride,
                        uint32_t rec_bins, uint32_t capacity, uint32_t* records_dev, uint32_t* count_dev,
                        void* cuda_stream);

/* Communicator over the GPUs that share a batch: NCCL (NVLink 5 / NVSwitch inside one box), loaded with
   dlopen("libnccl.so.2") on first use.  One process per GPU: rank 0 calls _unique_id, the caller gets
   the 128 bytes to every rank (MPI, the launcher's rendezvous, a file ...) and every rank calls _comm_init.
   ecdna_b200_destroy releases it. */
int ecdna_b200_comm_unique_id(uint8_t id[ECDNA_B200_COMM_ID_BYTES]);
int ecdna_b200_comm_init(ecdna_b200_ctx* ctx, const uint8_t id[ECDNA_B200_COMM_ID_BYTES], int rank, int world);
void ecdna_b200_comm_release(ecdna_b200_ctx* ctx);

/* All-gather of the packed records: every rank contributes its count and a block of `capacity` records;
   all_counts_dev [world] and all_records_dev [world][capacity][record] (device) receive them in rank order.
   Two ncclAllGather calls in one group on `cuda_stream`; no host synchronisation. */
int ecdna_b200_abc_allgather(ecdna_b200_ctx* ctx, const uint32_t* records_dev, const uint32_t* count_dev,
                             uint32_t rec_bins, uint32_t capacity, uint32_t* all_records_dev,
                             uint32_t* all_counts_dev, void* cuda_stream);

/* ---- ABC-SMC: sequential Monte Carlo ABC (ABC population Monte Carlo) over (b1, d0, d1) ----
   Generation 0 is rejection ABC on the uniform prior box of ecdna_b200_abc_draw_priors: its first M valid draws.
   Generation t+1 proposes from the weighted population t: a parent picked by weight, then every free parameter
   perturbed by a Gaussian truncated to the box, sigma_k^2 = 2 x the weighted variance of parameter k in
   population t (Beaumont, Cornuet, Marin, Robert 2009, Biometrika 96:983); its particles are weighted by
   1 / sum_j W_j prod_k phi((theta_ik - theta_jk) / sigma_k) / Z_j with Z_j the truncation normaliser of parent j
   (ibid.; the uniform prior cancels).  The tolerance eps (a factor on every user threshold thr_j > 0) follows the
   quantile schedule eps_{t+1} = min(eps_t, max(1, rho_(ceil(alpha M)))) of the scalar distances
   rho = max_j d_j / thr_j (Del Moral, Doucet, Jasra 2012, Stat. Comput. 22:1009) and the run ends after the first
   generation at eps = 1, where acceptance is the rejection rule of the kernel's epilogue.  DESIGN.md section 9.
   A range with lo == hi fixes that parameter: it is never perturbed and has no factor in the weights. */

/* Proposals for draws idx_begin .. idx_begin + n - 1 (device kernel; host buffers in and out; blocking).
   Draw i picks parent = the first j with cum_weights[j] > u * cum_weights[M-1] (u in [0,1), 53 bits of Philox
   keyed (seed, i) in a domain of its own) and perturbs every free parameter k (lo < hi, sigma[k] > 0) by
   z = Phi^-1(Phi(a) + u' (Phi(b) - Phi(a))), a, b = the box edges in sigma units around the parent, in f64;
   no rejection loop.  prev_rates [M][4] (b0, b1, d0, d1), cum_weights [M] (f64, non-decreasing, last > 0),
   rates_out [n][4] (column 0 and fixed parameters copied from the parent), parent_out [n] (0 .. M-1). */
int ecdna_b200_abc_smc_propose(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n,
                               const float* prev_rates, const double* cum_weights, uint32_t M, const double sigma[3],
                               const float b1_range[2], const float d0_range[2], const float d1_range[2],
                               float* rates_out, uint32_t* parent_out);

/* Importance weights of new_rates [N][4] against the population prev_rates [M][4] with weights prev_weights [M]
   (f64) and kernel widths sigma[3]: all-pairs sum on the device in a fixed order (no atomics: bit-identical run to
   run); weights_out [N] (f64) are normalised to sum to 1.  Host buffers; blocking. */
int ecdna_b200_abc_smc_weights(ecdna_b200_ctx* ctx, const float* new_rates, uint32_t N, const float* prev_rates,
                               const double* prev_weights, uint32_t M, const double sigma[3], const float b1_range[2],
                               const float d0_range[2], const float d1_range[2], double* weights_out);

enum { ECDNA_B200_SMC_REACHED = 0, ECDNA_B200_SMC_MAX_GENERATIONS = 1, ECDNA_B200_SMC_BUDGET = 2 };

typedef struct {
  uint32_t population;      /* M >= 1 particles per generation */
  double quantile;          /* alpha in (0, 1): eps_{t+1} is the ceil(alpha M)-th smallest rho of generation t */
  uint32_t max_generations; /* >= 1, generation 0 included */
  uint64_t max_simulations; /* draw indices all generations may consume together; 0 = no limit */
  uint64_t idx_begin;       /* index of the first draw (the CLI: seed * 10) */
  uint64_t chunk;           /* draws per ecdna_b200_multi_run call; 0 = sized from the acceptance rate.
                               Results do not depend on it (nor on the number of GPUs) */
  float b1_range[2], d0_range[2], d1_range[2]; /* the uniform prior box, lo <= hi */
} ecdna_b200_smc_options_t;

/* Caller-owned; [G][M] below means [max_generations][population]; every pointer is optional (NULL = not wanted). */
typedef struct {
  uint64_t* idx;        /* [G][M] draw index of the particle (its SSA stream and its proposal stream) */
  uint64_t* parent_idx; /* [G][M] draw index of the parent; UINT64_MAX in generation 0 */
  float* rates;         /* [G][M][4] b0, b1, d0, d1 */
  float* distance;      /* [G][M][4] ks, rel. mean, rel. entropy, rel. frequency */
  double* weight;       /* [G][M] normalised importance weights */
  uint64_t* cells;      /* [G][M] nminus + nplus at the end of the run */
  float* epsilon;       /* [G] tolerance factor of the generation (+inf in generation 0) */
  uint64_t* consumed;   /* [G] draw indices used: up to and including the M-th accepted draw */
  uint64_t* simulated;  /* [G] draws simulated, including those past the M-th acceptance */
  double* ess;          /* [G] effective sample size 1 / sum W_i^2 */
  float* time_ms;       /* [G][3] host clock: simulation, proposal, weights */
  uint32_t generations; /* out: generations completed */
  uint32_t status;      /* out: ECDNA_B200_SMC_* */
} ecdna_b200_smc_result_t;

/* The ABC-SMC loop over every GPU of `m`.  params: b0, the process, the stop rule, the ABC target and the user
   thresholds (abc_enabled set, at least one threshold >= 0, rates_per_run NULL); params->seed keys every stream.
   Draw i is simulated as replicate i (its SSA stream is the one rejection ABC gives index i) through
   ecdna_b200_multi_run in chunks; proposals and weights run on the first GPU.  A draw is accepted when the
   epilogue accepts it at thresholds thr_j * eps (thr_j > 0; others unchanged) and it is valid: stop code neither
   COPY_OVERFLOW nor HIST_OVERFLOW, no FLAG_HIST_TRUNCATED (copy numbers below params->hist_stride), finite rho.
   Ends with status REACHED after the first generation at eps = 1, MAX_GENERATIONS, or BUDGET when the next
   generation would pass max_simulations (the generations before it are returned; not an error). */
int ecdna_b200_abc_smc(ecdna_b200_multi* m, const ecdna_b200_params_t* params, const ecdna_b200_smc_options_t* options,
                       ecdna_b200_smc_result_t* result);

/* ---- ABC-SMC with correlated perturbation kernels (DESIGN.md section 9) ----
   COMPONENT: the kernel above (one Gaussian per parameter).  MVN: N(theta_j, Sigma), Sigma = 2 x the weighted
   covariance of the population.  OLCM (Filippi, Barnes, Cornebise, Stumpf 2013, SAGMB 12:87): N(theta_j, Sigma_j),
   Sigma_j = C + (m - theta_j)(m - theta_j)^T, m and C the weighted mean and covariance of the particles with
   rho <= eps_{t+1}.  Both are truncated to the box by sequential conditioning over the free parameters in the order
   b1, d0, d1 with L = chol(Sigma) (f64): coordinate t is N(c_t + sum_{l<t} L_tl e_l, L_tt^2) truncated to [lo, hi]
   by inverse CDF (in log space beyond 5 sds), e_t = (theta_t - its mean) / L_tt; no rejection loop.  The density
   prod_t phi(e_t) / (L_tt (Phi(b_t) - Phi(a_t))) with e = L^-1 (theta - c) is exact.  Draw i uses the Philox
   words of ecdna_b200_abc_smc_propose, so a diagonal Sigma gives its proposals bit for bit. */
enum { ECDNA_B200_SMC_KERNEL_COMPONENT = 0, ECDNA_B200_SMC_KERNEL_MVN = 1, ECDNA_B200_SMC_KERNEL_OLCM = 2 };

/* cov: packed lower triangles (s11, s21, s22, s31, s32, s33) over (b1, d0, d1), f64; n_cov = 1 (shared) or M (one
   per parent).  A parameter is free when lo < hi and its variance is > 0 in every Sigma (0 in every Sigma fixes it;
   anything else is an error).  Rows/columns of fixed parameters are ignored; a non-finite entry or a Sigma that is
   not positive definite over the free ones -> ERR_BAD_PARAMS.  Otherwise as ecdna_b200_abc_smc_propose. */
int ecdna_b200_abc_smc_propose_cov(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n,
                                   const float* prev_rates, const double* cum_weights, uint32_t M, const double* cov,
                                   uint32_t n_cov, const float b1_range[2], const float d0_range[2],
                                   const float d1_range[2], float* rates_out, uint32_t* parent_out);

/* Importance weights of new_rates [N][4] under the kernels of ecdna_b200_abc_smc_propose_cov: all-pairs sum in a
   fixed order as ecdna_b200_abc_smc_weights (bit-identical run to run); weights_out [N] normalised to sum to 1. */
int ecdna_b200_abc_smc_weights_cov(ecdna_b200_ctx* ctx, const float* new_rates, uint32_t N, const float* prev_rates,
                                   const double* prev_weights, uint32_t M, const double* cov, uint32_t n_cov,
                                   const float b1_range[2], const float d0_range[2], const float d1_range[2],
                                   double* weights_out);

typedef struct {
  uint32_t kernel;      /* ECDNA_B200_SMC_KERNEL_* */
  uint32_t reserved[3]; /* 0 */
} ecdna_b200_smc_kernel_t;

/* ecdna_b200_abc_smc with a choice of kernel (NULL = COMPONENT, which is ecdna_b200_abc_smc byte for byte).  Sigma is
   usable when every Cholesky pivot L_tt >= 2^-12 (hi_t - lo_t); each generation falls back OLCM -> MVN -> COMPONENT
   to the first usable one.  kernel_used [max_generations], optional: UINT32_MAX for generation 0, else the
   ECDNA_B200_SMC_KERNEL_* that proposed and weighted the generation. */
int ecdna_b200_abc_smc_ex(ecdna_b200_multi* m, const ecdna_b200_params_t* params, const ecdna_b200_smc_options_t* options,
                          const ecdna_b200_smc_kernel_t* kernel, ecdna_b200_smc_result_t* result, uint32_t* kernel_used);

#ifdef __cplusplus
}
#endif
#endif
