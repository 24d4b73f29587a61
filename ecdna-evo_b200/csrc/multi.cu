// multi.cu -- one batch over several GPUs of one box from ONE process: the reference maps the whole index
// range over all of rayon's workers (src/main.rs:214-225); here the range is cut into contiguous blocks, one
// per GPU, each driven by its own host thread and context, and every block's results land directly in the
// caller's arrays at the block's offset.  Replicates are independent: no data-path collective.
#include <thread>
#include <vector>

#include "engine.cuh"

using namespace ecdna;

namespace {
// contiguous block of [0, n) owned by part r of `parts` (the first parts take the remainder)
void block_of(uint64_t n, int r, int parts, uint64_t* begin, uint64_t* count) {
  const uint64_t base = n / (uint64_t)parts, rem = n % (uint64_t)parts;
  *begin = (uint64_t)r * base + std::min<uint64_t>((uint64_t)r, rem);
  *count = base + ((uint64_t)r < rem ? 1 : 0);
}
}  // namespace

extern "C" {

int ecdna_b200_multi_create(const int* devices, int n_devices, ecdna_b200_multi** out) {
  if (!out) return ECDNA_B200_ERR_BAD_PARAMS;
  *out = nullptr;
  std::vector<int> devs;
  if (devices && n_devices > 0) devs.assign(devices, devices + n_devices);
  else {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return ECDNA_B200_ERR_NO_DEVICE;
    for (int d = 0; d < count; ++d) {
      cudaDeviceProp prop;
      if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major == 10) devs.push_back(d);
    }
    if (devs.empty()) return ECDNA_B200_ERR_NO_DEVICE;
  }
  ecdna_b200_multi* m = new ecdna_b200_multi();
  for (int d : devs) {
    ecdna_b200_ctx* c = nullptr;
    const int rc = ecdna_b200_create(d, &c);
    if (rc != ECDNA_B200_OK) {
      for (ecdna_b200_ctx* x : m->ctx) ecdna_b200_destroy(x);
      delete m;
      return rc;
    }
    m->ctx.push_back(c);
  }
  m->last_begin.assign(m->ctx.size(), 0);
  m->last_count.assign(m->ctx.size(), 0);
  *out = m;
  return ECDNA_B200_OK;
}

void ecdna_b200_multi_destroy(ecdna_b200_multi* m) {
  if (!m) return;
  for (ecdna_b200_ctx* c : m->ctx) ecdna_b200_destroy(c);
  delete m;
}

int ecdna_b200_multi_device_count(const ecdna_b200_multi* m) { return m ? (int)m->ctx.size() : 0; }
const char* ecdna_b200_multi_last_error(const ecdna_b200_multi* m) { return m ? m->err.c_str() : "no context"; }

int ecdna_b200_multi_run(ecdna_b200_multi* m, const ecdna_b200_params_t* params, uint64_t idx_begin, uint64_t n_runs,
                         const ecdna_b200_results_t* results) {
  if (!m || !params || !results || n_runs == 0) {
    if (m) m->err = "bad multi-GPU run request";
    return ECDNA_B200_ERR_BAD_PARAMS;
  }
  const int parts = (int)std::min<uint64_t>(m->ctx.size(), n_runs);
  const uint32_t stride = params->hist_stride ? params->hist_stride : 512u;
  std::vector<int> rcs(parts, ECDNA_B200_OK);
  std::vector<std::thread> workers;
  m->sp_valid = false;  // (a dense run replaces whatever sparse batch the devices still held)
  for (size_t g = 0; g < m->ctx.size(); ++g) m->last_count[g] = 0;
  for (int g = 0; g < parts; ++g) {
    uint64_t b, c;
    block_of(n_runs, g, parts, &b, &c);
    m->last_begin[g] = b;
    m->last_count[g] = c;
    workers.emplace_back([=, &rcs]() {
      ecdna_b200_params_t p = *params;
      ecdna_b200_results_t r = *results;
      for (int col = 0; col < C_COUNT; ++col) {  // every column of this block starts b replicates in
        void** slot = col_slot(&r, col);
        if (*slot) *slot = (char*)*slot + col_bytes(col, params, stride) * b;
      }
      if (p.rates_per_run) p.rates_per_run += 4 * b;
      if (p.replay_offsets) p.replay_offsets += b;  // (offsets stay absolute into the shared stream)
      rcs[g] = ecdna_b200_run(m->ctx[g], &p, idx_begin + b, c, &r);
    });
  }
  for (std::thread& t : workers) t.join();
  for (int g = 0; g < parts; ++g)
    if (rcs[g] != ECDNA_B200_OK) {
      m->err = "device " + std::to_string(m->ctx[g]->device) + ": " + ecdna_b200_last_error(m->ctx[g]);
      return rcs[g];
    }
  return ECDNA_B200_OK;
}

// Sparse return over all GPUs: every GPU simulates, measures and lays out its block (phase 1); the blocks' arena
// needs give every block its base in the caller's arena; every GPU then packs and copies its block there (phase 2).
int ecdna_b200_multi_run_sparse(ecdna_b200_multi* m, const ecdna_b200_params_t* params, uint64_t idx_begin,
                                uint64_t n_runs, const ecdna_b200_results_t* results, ecdna_b200_sparse_t* sparse) {
  if (!m || !params || !sparse || n_runs == 0) {
    if (m) m->err = "bad multi-GPU run request";
    return ECDNA_B200_ERR_BAD_PARAMS;
  }
  static const ecdna_b200_results_t none{};
  if (!results) results = &none;
  m->sp_valid = false;
  const int parts = (int)std::min<uint64_t>(m->ctx.size(), n_runs);
  const uint32_t stride = params->hist_stride ? params->hist_stride : 512u;
  std::vector<int> rcs(parts, ECDNA_B200_OK);
  std::vector<std::thread> workers;
  m->sp_words.assign(m->ctx.size(), 0);
  for (size_t g = 0; g < m->ctx.size(); ++g) m->last_count[g] = 0;
  for (int g = 0; g < parts; ++g) {
    uint64_t b, c;
    block_of(n_runs, g, parts, &b, &c);
    m->last_begin[g] = b;
    m->last_count[g] = c;
    workers.emplace_back([=, &rcs]() {
      ecdna_b200_params_t p = *params;
      ecdna_b200_results_t r = *results;
      for (int col = 0; col < C_COUNT; ++col) {
        void** slot = col_slot(&r, col);
        if (*slot) *slot = (char*)*slot + col_bytes(col, params, stride) * b;
      }
      if (p.rates_per_run) p.rates_per_run += 4 * b;
      if (p.replay_offsets) p.replay_offsets += b;
      rcs[g] = sparse_prepare(m->ctx[g], &p, idx_begin + b, c, &r, &m->sp_words[g]);
    });
  }
  for (std::thread& t : workers) t.join();
  for (int g = 0; g < parts; ++g)
    if (rcs[g] != ECDNA_B200_OK) {
      m->err = "device " + std::to_string(m->ctx[g]->device) + ": " + ecdna_b200_last_error(m->ctx[g]);
      return rcs[g];
    }
  m->sp_snap = params->n_snapshots;
  m->sp_sub = results->sub_hist || params->n_subsamples ? params->n_subsamples : 0;
  m->sp_valid = true;
  return ecdna_b200_multi_sparse_fetch(m, sparse);
}

int ecdna_b200_multi_sparse_fetch(ecdna_b200_multi* m, ecdna_b200_sparse_t* sparse) {
  if (!m || !sparse) return ECDNA_B200_ERR_BAD_PARAMS;
  if (!m->sp_valid) { m->err = "no sparse batch on the devices: call ecdna_b200_multi_run_sparse first"; return ECDNA_B200_ERR_BAD_PARAMS; }
  uint64_t total = 0;
  std::vector<uint64_t> base(m->ctx.size(), 0);
  for (size_t g = 0; g < m->ctx.size(); ++g) { base[g] = total; total += m->last_count[g] ? m->sp_words[g] : 0; }
  sparse->arena_used = total;
  const bool fits = total == 0 || (sparse->arena && sparse->arena_words >= total);
  std::vector<int> rcs(m->ctx.size(), ECDNA_B200_OK);
  std::vector<std::thread> workers;
  for (size_t g = 0; g < m->ctx.size(); ++g) {
    if (m->last_count[g] == 0) continue;
    workers.emplace_back([=, &rcs]() {
      const uint64_t b = m->last_begin[g];
      rcs[g] = sparse_fetch(m->ctx[g], sparse->final_dist ? sparse->final_dist + b : nullptr,
                            sparse->snap_dist ? sparse->snap_dist + b * m->sp_snap : nullptr,
                            sparse->sub_dist ? sparse->sub_dist + b * m->sp_sub : nullptr, fits ? sparse->arena : nullptr, base[g]);
    });
  }
  for (std::thread& t : workers) t.join();
  for (size_t g = 0; g < m->ctx.size(); ++g)
    if (rcs[g] != ECDNA_B200_OK) {
      m->err = "device " + std::to_string(m->ctx[g]->device) + ": " + ecdna_b200_last_error(m->ctx[g]);
      return rcs[g];
    }
  if (!fits) {
    m->err = "the batch needs an arena of " + std::to_string(total) + " words, the caller gave " + std::to_string(sparse->arena ? sparse->arena_words : 0);
    return ECDNA_B200_ERR_ARENA;
  }
  return ECDNA_B200_OK;
}

int ecdna_b200_multi_get_timing(ecdna_b200_multi* m, ecdna_b200_timing_t* t) {
  if (!m || !t) return ECDNA_B200_ERR_BAD_PARAMS;
  ecdna_b200_timing_t sum{};
  bool first = true;
  for (size_t g = 0; g < m->ctx.size(); ++g) {
    if (m->last_count[g] == 0) continue;
    ecdna_b200_timing_t x;
    const int rc = ecdna_b200_get_timing(m->ctx[g], &x);
    if (rc != ECDNA_B200_OK) { m->err = ecdna_b200_last_error(m->ctx[g]); return rc; }
    if (first) { sum = x; first = false; continue; }
    // the batch takes as long as its slowest block; counts add up
    sum.kernel_ms = std::max(sum.kernel_ms, x.kernel_ms);
    sum.total_ms = std::max(sum.total_ms, x.total_ms);
    sum.kernel_launches += x.kernel_launches;
    sum.grid_blocks += x.grid_blocks;
    sum.h2d_bytes += x.h2d_bytes; sum.d2h_bytes += x.d2h_bytes;
    sum.total_events += x.total_events; sum.alg_bytes += x.alg_bytes;
    sum.n_spilled += x.n_spilled; sum.n_slices += x.n_slices; sum.n_idle_spells += x.n_idle_spells;
    sum.n_finished += x.n_finished;
  }
  *t = sum;
  return ECDNA_B200_OK;
}

}  // extern "C"
