// pb_api.cu — the C ABI of libpersia_b200.so (include/persia_b200.h): object lifetime, argument checks,
// kernel sequencing.  No torch types, no allocation on the hot path after the first call of a given size.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "pb_kernels.cuh"

using namespace pb;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define PB_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(PB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));               \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

uint32_t next_pow2(uint64_t v) {
  uint64_t p = 1;
  while (p < v) p <<= 1;
  return (uint32_t)p;
}

// rand 0.8 UniformFloat::new: shrink the scale until the largest draw stays below `hi`
float uniform_scale(float lo, float hi) {
  float scale = hi - lo;
  uint32_t mb = (0xFFFFFFFFu >> 9) | 0x3f800000u;
  float max_rand;
  std::memcpy(&max_rand, &mb, 4);
  max_rand -= 1.0f;
  if (!(hi > lo)) return 0.0f;
  while (!(scale * max_rand + lo < hi)) {
    uint32_t b;
    std::memcpy(&b, &scale, 4);
    b -= 1;
    std::memcpy(&scale, &b, 4);
  }
  return scale;
}

}  // namespace

struct pb_table {
  int device = 0;
  pb_table_cfg cfg{};
  OptimDev op{};
  bool has_op = false;
  HyperDev hy{};
  bool has_hy = false;
  TableDev d{};
  bool allocated = false;
  uint32_t* scratch = nullptr;  // index cells of a single-request call
  uint32_t scratch_cap = 0;
  // Adam: accumulated (beta1^t, beta2^t) per feature group, keyed by index prefix (optim.rs:99-131, 155-197)
  // (the pairs live on the device: a captured backward advances them on every replay)
  std::vector<uint64_t> adam_keys;  // position = pair number; pair PB_ADAM_KEYS-1 serves pb_update
  float* adam_dev = nullptr;
  // capacity policy (pb_table_set_eviction): 0 = refuse admissions when full
  uint32_t evict_every = 0, evict_low = 0, evict_target = 0, evict_keep = 2;
  uint32_t train_calls = 0;
  uint32_t* evict_ws = nullptr;
  uint32_t pending_batches = 0;  // training forwards whose backward has not been enqueued yet
};

struct pb_ctx {
  int device = 0;
  uint32_t max_occ = 0, max_out = 0;
  pb_slots_cfg slots{};
  bool has_slots = false;
  // forward -> backward state (the EW's post_forward_buffer entry, mod.rs:1087-1098): the batch's distinct signs,
  // where each lives, the occurrence lists and the work lists of the backward (pb_kernels.cuh BatchDev)
  BatchDev b{};
  size_t set_cells = 0;
  bool set_dirty = false;  // the scratch set still holds the last batch's cells
  uint32_t* occ_outrow = nullptr;
  uint32_t* row_off = nullptr;
  bool multi_id = false;
  uint32_t n_occ = 0, batch = 0;
  uint32_t* dev_tick = nullptr;  // request number of the pending forward (device side, CUDA-graph safe)
  uint32_t occ_off[PB_MAX_SLOTS + 1];
  bool pending = false;
  pb_table* pending_table = nullptr;  // the table whose rows the pending batch refers to (eviction spares them)
  // slots of one feature group take turns in the backward (mod.rs:720-822): round of every slot
  uint32_t n_rounds = 1;
  uint8_t round_of[PB_MAX_SLOTS];
  // backward workspace
  uint32_t* nan_tick = nullptr;
  float* vw_stage = nullptr;
  size_t vw_stage_floats = 0;
  float* hot_stage = nullptr;  // [b.hot_cap][hot_stage_stride(dim)] reduced gradients of the hot items
  size_t hot_stage_floats = 0;
  cudaStream_t side = nullptr;  // hot items run beside the main stream during pb_backward
  cudaStream_t side2 = nullptr;  // scratch-set clearing and the warm items, beside the cold ones
  cudaEvent_t ev_fork = nullptr, ev_nan = nullptr, ev_join = nullptr, ev_join2 = nullptr;
  // raw slot (pb_forward_raw / pb_backward_raw): allocated on first use
  uint32_t* occ_cell = nullptr;
  RawWork raw{};
  bool raw_ready = false, raw_pending = false;
  float* raw_stage = nullptr;
  size_t raw_stage_floats = 0;
};

namespace {

int ensure_alloc(pb_table* t) {
  if (t->allocated) return PB_OK;
  if (!t->has_op) return fail(PB_ERR_STATE, "optimizer not registered (OptimizerNotFoundError)");
  uint32_t dim = t->cfg.dim;
  uint32_t state = 0;
  switch (t->op.kind) {
    case PB_OPT_ADAGRAD: state = dim; break;
    case PB_OPT_ADAGRAD_VW: state = 1; break;
    case PB_OPT_ADAM: state = 2 * dim; break;
    default: state = 0;
  }
  TableDev& d = t->d;
  d.dim = dim;
  d.state_floats = state;
  d.stride = (dim + state + 3u) & ~3u;
  if (t->cfg.capacity >= 0xFFFFFFF0ull) return fail(PB_ERR_INVALID, "capacity must be < 2^32 - 16 rows per shard");
  d.capacity = (uint32_t)t->cfg.capacity;
  uint64_t want = (uint64_t)d.capacity + d.capacity / 2;
  if (want < 1024) want = 1024;
  if (want > (1ull << 31)) return fail(PB_ERR_INVALID, "capacity too large for a 2^31-cell index");
  d.n_cells = next_pow2(want);
  d.cell_mask = d.n_cells - 1;
  d.bucket_mask = d.n_cells / BUCKET - 1;
  PB_CUDA(cudaMalloc(&d.cells, sizeof(Cell) * ((size_t)d.n_cells + N_SPECIAL)));
  PB_CUDA(cudaMalloc(&d.rows, sizeof(float) * (size_t)d.capacity * d.stride));
  PB_CUDA(cudaMalloc(&d.counters, sizeof(uint32_t) * CTR_COUNT));
  PB_CUDA(cudaMalloc(&d.row_tick, sizeof(uint32_t) * (size_t)d.capacity));
  PB_CUDA(cudaMemset(d.row_tick, 0, sizeof(uint32_t) * (size_t)d.capacity));
  PB_CUDA(cudaMemset(d.counters, 0, sizeof(uint32_t) * CTR_COUNT));
  launch_fill_cells(d.cells, (uint64_t)d.n_cells + N_SPECIAL, 0);
  d.free_rows = nullptr;
  PB_CUDA(cudaDeviceSynchronize());
  t->allocated = true;
  return PB_OK;
}

int ensure_scratch(pb_table* t, uint32_t n) {
  if (n <= t->scratch_cap) return PB_OK;
  if (t->scratch) cudaFree(t->scratch);
  t->scratch = nullptr;
  t->scratch_cap = 0;
  uint32_t cap = next_pow2(n);
  PB_CUDA(cudaMalloc(&t->scratch, sizeof(uint32_t) * (size_t)cap));
  t->scratch_cap = cap;
  return PB_OK;
}

// Between two training requests: release the least recently used rows when free storage runs low.
int maybe_evict(pb_table* t, cudaStream_t st) {
  if (!t->evict_every || (++t->train_calls % t->evict_every)) return PB_OK;
  if (!t->d.free_rows) {
    PB_CUDA(cudaMalloc(&t->d.free_rows, sizeof(uint32_t) * (size_t)t->d.capacity));
    PB_CUDA(cudaMalloc(&t->evict_ws, sizeof(uint32_t) * (3 + 1024)));
  }
  // rows of batches whose gradients are still to come are never released: a row used by a pending batch was
  // refreshed by its forward, i.e. at most `pending_batches` requests ago
  const uint32_t keep = t->evict_keep > t->pending_batches + 1 ? t->evict_keep : t->pending_batches + 1;
  launch_evict(t->d, t->evict_low, t->evict_target, keep, t->evict_ws, st);
  return PB_OK;
}

int ready_for_training(pb_table* t) {
  if (!t->has_op) return fail(PB_ERR_STATE, "optimizer not registered (OptimizerNotFoundError)");
  if (!t->has_hy) return fail(PB_ERR_STATE, "embedding server not configured (NotConfiguredError)");
  return PB_OK;
}

// pair number of a feature group (keyed by its index prefix); -1 when the table is out of pairs
int adam_index(pb_table* t, uint64_t prefix) {
  for (size_t i = 0; i < t->adam_keys.size(); ++i)
    if (t->adam_keys[i] == prefix) return (int)i;
  if (t->adam_keys.size() + 1 >= PB_ADAM_KEYS) return -1;
  t->adam_keys.push_back(prefix);
  return (int)t->adam_keys.size() - 1;
}

SlotsDev no_slots() {
  SlotsDev s;
  std::memset(&s, 0, sizeof(s));
  s.n_slots = 1;
  s.spacing = ~0ULL;
  s.spacing_bits = 64;
  return s;
}

int make_slots(const pb_slots_cfg& cfg, const uint32_t* h_occ_off, SlotsDev& s) {
  std::memset(&s, 0, sizeof(s));
  if (cfg.n_slots == 0 || cfg.n_slots > PB_MAX_SLOTS) return fail(PB_ERR_INVALID, "n_slots must be in 1..PB_MAX_SLOTS");
  s.n_slots = cfg.n_slots;
  s.spacing = cfg.prefix_bit > 0 ? ((1ULL << (64 - cfg.prefix_bit)) - 1) : ~0ULL;
  s.spacing_bits = 64 - cfg.prefix_bit;
  for (uint32_t i = 0; i < cfg.n_slots; ++i) {
    s.prefix[i] = cfg.prefix[i];
    s.sqrt_scaling[i] = cfg.sqrt_scaling[i];
    s.occ_off[i] = h_occ_off[i];
  }
  s.occ_off[cfg.n_slots] = h_occ_off[cfg.n_slots];
  s.uniform = cfg.n_slots ? (h_occ_off[cfg.n_slots] - h_occ_off[0]) / cfg.n_slots : 0;
  for (uint32_t i = 0; i <= cfg.n_slots && s.uniform; ++i)
    if (h_occ_off[i] != i * s.uniform) s.uniform = 0;
  return PB_OK;
}

void drop_pending(pb_ctx* c) {
  if (c->pending && c->pending_table && c->pending_table->pending_batches) c->pending_table->pending_batches--;
  c->pending = false;
  c->pending_table = nullptr;
}

}  // namespace

extern "C" {

const char* pb_last_error(void) { return g_err.c_str(); }
int pb_version(void) { return 100; }
uint64_t pb_launch_count(void) { return launch_count(); }
int pb_profile_enable(int family_mask) {
  profile_enable((uint32_t)family_mask);
  return PB_OK;
}
int pb_profile_read(double* h_ms, uint64_t* h_count, int n) {
  if (!h_ms || !h_count || n <= 0) return fail(PB_ERR_INVALID, "bad argument");
  PB_CUDA(cudaDeviceSynchronize());
  profile_read(h_ms, h_count, n < FAM_COUNT ? n : FAM_COUNT);
  for (int i = FAM_COUNT; i < n; ++i) {
    h_ms[i] = 0;
    h_count[i] = 0;
  }
  return PB_OK;
}

int pb_table_create(int device, const pb_table_cfg* cfg, pb_table** out) {
  if (!cfg || !out) return fail(PB_ERR_INVALID, "null argument");
  if (cfg->dim == 0 || cfg->dim > 4096) return fail(PB_ERR_INVALID, "dim must be in 1..4096");
  if (cfg->capacity == 0) return fail(PB_ERR_INVALID, "capacity must be > 0");
  int ndev = 0;
  PB_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(PB_ERR_INVALID, "no such CUDA device");
  pb_table* t = new pb_table();
  t->device = device;
  t->cfg = *cfg;
  *out = t;
  return PB_OK;
}

int pb_table_destroy(pb_table* t) {
  if (!t) return PB_OK;
  DeviceGuard g(t->device);
  if (t->allocated) {
    cudaDeviceSynchronize();
    cudaFree(t->d.cells);
    cudaFree(t->d.rows);
    cudaFree(t->d.counters);
    cudaFree(t->d.row_tick);
    if (t->d.free_rows) cudaFree(t->d.free_rows);
    if (t->evict_ws) cudaFree(t->evict_ws);
  }
  if (t->scratch) cudaFree(t->scratch);
  if (t->adam_dev) cudaFree(t->adam_dev);
  delete t;
  return PB_OK;
}

int pb_table_set_optimizer(pb_table* t, const pb_optim_cfg* c) {
  if (!t || !c) return fail(PB_ERR_INVALID, "null argument");
  if (c->kind < PB_OPT_SGD || c->kind > PB_OPT_ADAM) return fail(PB_ERR_INVALID, "unknown optimizer kind");
  if (t->allocated && c->kind != t->op.kind)
    return fail(PB_ERR_STATE, "optimizer kind cannot change once rows are resident (row layout is fixed)");
  t->op.kind = c->kind;
  t->op.lr = c->lr;
  t->op.wd = c->wd;
  t->op.mom = c->g_square_momentum;
  t->op.init_acc = c->initialization;
  t->op.eps = c->eps;
  t->op.b1 = c->beta1;
  t->op.b2 = c->beta2;
  if (!t->has_op && c->kind == PB_OPT_ADAM) {  // AdamPowerOfBetas starts at (beta1, beta2) for every feature group (optim.rs:118-124)
    DeviceGuard g(t->device);
    t->adam_keys.clear();
    if (!t->adam_dev) PB_CUDA(cudaMalloc(&t->adam_dev, sizeof(float) * 2 * PB_ADAM_KEYS));
    launch_adam_fill(t->adam_dev, c->beta1, c->beta2, 0);
    PB_CUDA(cudaDeviceSynchronize());
  }
  t->has_op = true;
  return PB_OK;
}

int pb_table_configure(pb_table* t, const pb_hyper_cfg* c) {
  if (!t || !c) return fail(PB_ERR_INVALID, "null argument");
  t->hy.lo = c->init_lower;
  t->hy.scale = uniform_scale(c->init_lower, c->init_upper);
  t->hy.admit_p = c->admit_probability;
  t->hy.enable_wb = c->enable_weight_bound;
  t->hy.wb = c->weight_bound;
  t->has_hy = true;
  return PB_OK;
}

int pb_table_spill(pb_table* t, uint64_t want_free, uint32_t keep_batches, uint64_t* d_signs, float* d_entries, uint32_t max_n,
                   uint32_t* d_count, void* stream) {
  if (!t || !d_count || (max_n && (!d_signs || !d_entries))) return fail(PB_ERR_INVALID, "null argument");
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (!t->d.free_rows) {
    PB_CUDA(cudaMalloc(&t->d.free_rows, sizeof(uint32_t) * (size_t)t->d.capacity));
    PB_CUDA(cudaMalloc(&t->evict_ws, sizeof(uint32_t) * (3 + 1024)));
  }
  if (want_free > t->d.capacity) want_free = t->d.capacity;
  const uint32_t keep = keep_batches > t->pending_batches + 1 ? keep_batches : t->pending_batches + 1;
  PB_CUDA(cudaMemsetAsync(d_count, 0, sizeof(uint32_t), st));
  launch_spill(t->d, (uint32_t)want_free, keep, t->evict_ws, d_signs, d_entries, max_n, d_count, st);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_table_set_eviction(pb_table* t, uint32_t check_every, uint64_t low_water, uint64_t target_free, uint32_t keep_batches) {
  if (!t) return fail(PB_ERR_INVALID, "null argument");
  if (check_every && (target_free < low_water || target_free > t->cfg.capacity))
    return fail(PB_ERR_INVALID, "need low_water <= target_free <= capacity");
  t->evict_every = check_every;
  t->evict_low = (uint32_t)low_water;
  t->evict_target = (uint32_t)target_free;
  t->evict_keep = keep_batches;
  return PB_OK;
}

int pb_table_entry_len(pb_table* t, uint32_t* h_out) {
  if (!t || !h_out) return fail(PB_ERR_INVALID, "null argument");
  if (!t->has_op) return fail(PB_ERR_STATE, "optimizer not registered");
  uint32_t dim = t->cfg.dim;
  *h_out = dim + (t->op.kind == PB_OPT_ADAGRAD ? dim : t->op.kind == PB_OPT_ADAGRAD_VW ? 1 : t->op.kind == PB_OPT_ADAM ? 2 * dim : 0);
  return PB_OK;
}

int pb_table_counters(pb_table* t, uint64_t h_out[5], void* stream) {
  if (!t || !h_out) return fail(PB_ERR_INVALID, "null argument");
  h_out[0] = h_out[1] = h_out[2] = h_out[3] = h_out[4] = 0;
  if (!t->allocated) return PB_OK;
  DeviceGuard g(t->device);
  uint32_t c[CTR_COUNT];
  PB_CUDA(cudaMemcpyAsync(c, t->d.counters, sizeof(c), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  PB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  h_out[0] = c[CTR_ADMIT] - c[CTR_EVICT];  // resident rows
  h_out[1] = c[CTR_MISS];
  h_out[2] = c[CTR_GRAD_MISS];
  h_out[3] = c[CTR_FULL];
  h_out[4] = c[CTR_ERR];
  return PB_OK;
}

int pb_table_size(pb_table* t, uint64_t* h_out, void* stream) {
  if (!t || !h_out) return fail(PB_ERR_INVALID, "null argument");
  uint64_t c[5];
  int rc = pb_table_counters(t, c, stream);
  if (rc) return rc;
  *h_out = c[0];
  return PB_OK;
}

int pb_table_clear(pb_table* t, void* stream) {
  if (!t) return fail(PB_ERR_INVALID, "null argument");
  if (!t->allocated) return PB_OK;
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  launch_fill_cells(t->d.cells, (uint64_t)t->d.n_cells + N_SPECIAL, st);
  PB_CUDA(cudaMemsetAsync(t->d.counters, 0, sizeof(uint32_t) * CTR_COUNT, st));
  PB_CUDA(cudaMemsetAsync(t->d.row_tick, 0, sizeof(uint32_t) * (size_t)t->d.capacity, st));
  return PB_OK;
}

int pb_lookup(pb_table* t, const uint64_t* d_signs, uint32_t n, int training, float* d_out, void* stream) {
  if (!t || (n && (!d_signs || !d_out))) return fail(PB_ERR_INVALID, "null argument");
  if (training) {
    int rc = ready_for_training(t);
    if (rc) return rc;
  } else if (!t->has_op) {  // nothing can be resident yet: zeros
    DeviceGuard g(t->device);
    PB_CUDA(cudaMemsetAsync(d_out, 0, sizeof(float) * (size_t)n * t->cfg.dim, (cudaStream_t)stream));
    return PB_OK;
  }
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = ensure_alloc(t);
  if (rc) return rc;
  if ((rc = ensure_scratch(t, n))) return rc;
  SlotsDev sl = no_slots();
  if (training) {
    if ((rc = maybe_evict(t, st))) return rc;
    launch_begin_batch(t->d, nullptr, nullptr, st);
    launch_probe(MODE_TRAIN, false, t->d, t->hy, t->op, sl, d_signs, n, t->scratch, st);
  } else {
    launch_probe(MODE_FIND, false, t->d, t->hy, t->op, sl, d_signs, n, t->scratch, st);
  }
  launch_gather(t->d, t->scratch, n, d_out, st);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_update(pb_table* t, const uint64_t* d_signs, const float* d_grads, uint32_t n, void* stream) {
  if (!t || (n && (!d_signs || !d_grads))) return fail(PB_ERR_INVALID, "null argument");
  int rc = ready_for_training(t);
  if (rc) return rc;
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = ensure_alloc(t))) return rc;
  if ((rc = ensure_scratch(t, n))) return rc;
  SlotsDev sl = no_slots();
  launch_probe(MODE_FIND, false, t->d, t->hy, t->op, sl, d_signs, n, t->scratch, st);
  const float* pair = nullptr;
  if (t->op.kind == PB_OPT_ADAM) {  // get_batch_level_state: one power step per request (optim.rs:155-197)
    AdamKeys k{};
    k.idx[0] = (uint8_t)(PB_ADAM_KEYS - 1);
    k.n = 1;
    launch_adam_advance(t->adam_dev, k, t->op.b1, t->op.b2, st);
    pair = t->adam_dev + 2 * (PB_ADAM_KEYS - 1);
  }
  launch_update_direct(t->d, t->op, t->hy, t->scratch, d_grads, n, pair, st);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_set_rows(pb_table* t, const uint64_t* d_signs, const float* d_entries, uint32_t n, void* stream) {
  if (!t || (n && (!d_signs || !d_entries))) return fail(PB_ERR_INVALID, "null argument");
  if (!t->has_op) return fail(PB_ERR_STATE, "optimizer not registered: entry length unknown");
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = ensure_alloc(t);
  if (rc) return rc;
  if ((rc = ensure_scratch(t, n))) return rc;
  SlotsDev sl = no_slots();
  launch_probe(MODE_SET, false, t->d, t->hy, t->op, sl, d_signs, n, t->scratch, st);
  launch_copy_entries(true, t->d, t->scratch, n, const_cast<float*>(d_entries), nullptr, st);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_get_rows(pb_table* t, const uint64_t* d_signs, uint32_t n, float* d_entries, uint8_t* d_found, void* stream) {
  if (!t || (n && (!d_signs || !d_entries))) return fail(PB_ERR_INVALID, "null argument");
  if (!t->has_op) return fail(PB_ERR_STATE, "optimizer not registered: entry length unknown");
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = ensure_alloc(t);
  if (rc) return rc;
  if ((rc = ensure_scratch(t, n))) return rc;
  SlotsDev sl = no_slots();
  launch_probe(MODE_FIND, false, t->d, t->hy, t->op, sl, d_signs, n, t->scratch, st);
  launch_copy_entries(false, t->d, t->scratch, n, d_entries, d_found, st);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_table_export_signs(pb_table* t, uint64_t* d_signs, uint32_t* d_recency, uint32_t max_n, uint32_t* d_count,
                          void* stream) {
  if (!t || !d_count || (max_n && (!d_signs || !d_recency))) return fail(PB_ERR_INVALID, "null argument");
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (!t->allocated) {
    PB_CUDA(cudaMemsetAsync(d_count, 0, sizeof(uint32_t), st));
    return PB_OK;
  }
  launch_export_signs(t->d, d_signs, d_recency, max_n, d_count, st);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_add_prefix(const uint64_t* d_ids, uint32_t n, const uint32_t* h_slot_occ_off, const uint64_t* h_prefix,
                  uint32_t n_slots, uint32_t prefix_bit, uint64_t* d_out, void* stream) {
  if (n && (!d_ids || !d_out)) return fail(PB_ERR_INVALID, "null argument");
  if (!h_slot_occ_off || !h_prefix) return fail(PB_ERR_INVALID, "null argument");
  pb_slots_cfg cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  cfg.n_slots = n_slots;
  cfg.prefix_bit = prefix_bit;
  if (n_slots == 0 || n_slots > PB_MAX_SLOTS) return fail(PB_ERR_INVALID, "n_slots must be in 1..PB_MAX_SLOTS");
  for (uint32_t i = 0; i < n_slots; ++i) cfg.prefix[i] = h_prefix[i];
  SlotsDev sl;
  int rc = make_slots(cfg, h_slot_occ_off, sl);
  if (rc) return rc;
  launch_add_prefix(sl, d_ids, n, d_out, (cudaStream_t)stream);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_shard_of(const uint64_t* d_signs, uint32_t n, uint32_t R, uint32_t* d_shard, void* stream) {
  if (n && (!d_signs || !d_shard)) return fail(PB_ERR_INVALID, "null argument");
  if (R == 0) return fail(PB_ERR_INVALID, "replica size must be > 0");
  launch_shard_of(d_signs, n, R, d_shard, nullptr, (cudaStream_t)stream);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_farmhash64(const uint64_t* d_in, uint32_t n, uint64_t* d_out, void* stream) {
  if (n && (!d_in || !d_out)) return fail(PB_ERR_INVALID, "null argument");
  launch_shard_of(d_in, n, 1, nullptr, d_out, (cudaStream_t)stream);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_hash_stack(const uint64_t* d_ids, uint32_t n, uint32_t rounds, uint64_t embedding_size, uint64_t* d_out, void* stream) {
  if (n && (!d_ids || !d_out)) return fail(PB_ERR_INVALID, "null argument");
  if (rounds == 0 || embedding_size == 0) return fail(PB_ERR_INVALID, "hash_stack_rounds and embedding_size must be > 0");
  launch_hash_stack(d_ids, n, rounds, embedding_size, d_out, (cudaStream_t)stream);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

uint64_t pb_partition_workspace(uint32_t n) { return partition_workspace_bytes(n); }

int pb_partition_by_shard(const uint64_t* d_signs, uint32_t n, uint32_t R, uint32_t* d_perm, uint32_t* d_counts,
                          void* d_work, uint64_t work_bytes, void* stream) {
  if ((n && (!d_signs || !d_perm)) || !d_counts || !d_work) return fail(PB_ERR_INVALID, "null argument");
  if (R == 0 || R > 256) return fail(PB_ERR_INVALID, "replica size must be in 1..256");
  if (work_bytes < pb_partition_workspace(n)) return fail(PB_ERR_CAPACITY, "workspace smaller than pb_partition_workspace(n)");
  launch_partition_by_shard(d_signs, n, R, d_perm, d_counts, (uint32_t*)d_work, (cudaStream_t)stream);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_ctx_create(int device, uint32_t max_occurrences, uint32_t max_out_rows, pb_ctx** out) {
  if (!out || max_occurrences == 0 || max_out_rows == 0) return fail(PB_ERR_INVALID, "bad argument");
  if (max_occurrences > (1u << 24)) return fail(PB_ERR_INVALID, "at most 2^24 id occurrences per batch");
  DeviceGuard g(device);
  pb_ctx* c = new pb_ctx();
  c->device = device;
  c->max_occ = max_occurrences;
  c->max_out = max_out_rows;
  std::memset(c->round_of, 0, sizeof(c->round_of));
  const size_t n = max_occurrences;
  c->set_cells = 2 * n + 2 * PB_MAX_SLOTS;  // region of slot s: 2*n_s + 1 cells and the reserved one
  cudaError_t e = cudaSuccess;
  auto A = [&](void** p, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(p, bytes);
  };
  A((void**)&c->b.set, sizeof(DCell) * c->set_cells);
  A((void**)&c->b.occ_set, 4 * n);
  A((void**)&c->b.item_cell, 4 * n);
  A((void**)&c->b.seg_occ, 4 * n);
  A((void**)&c->b.cold, 8 * n);
  A((void**)&c->b.warm, 16 * (n / 2 + 1));
  c->b.giant_cap = n / PB_GIANT_MIN + 1;
  c->b.hot_cap = n / (PB_WARM_MAX + 1) + 1 + c->b.giant_cap;
  A((void**)&c->b.hot, 16 * (size_t)c->b.hot_cap);
  c->b.hot_words = (uint32_t)(n < 4096 ? 4096 : n);  // 32 bits of pool per id occurrence the context can hold
  A((void**)&c->b.hot_bits, 4 * (size_t)c->b.hot_words);
  A((void**)&c->b.cnt, 4 * BC_COUNT);
  A((void**)&c->occ_cell, 4 * n);
  A((void**)&c->occ_outrow, 4 * n);
  A((void**)&c->row_off, 4 * ((size_t)max_out_rows + 1));
  A((void**)&c->nan_tick, 4 * PB_MAX_SLOTS);
  A((void**)&c->dev_tick, 4);
  if (e == cudaSuccess) e = cudaMemset(c->nan_tick, 0, 4 * PB_MAX_SLOTS);
  if (e == cudaSuccess) e = cudaMemset(c->dev_tick, 0, 4);
  if (e == cudaSuccess) e = cudaMemset(c->b.cnt, 0, 4 * BC_COUNT);
  if (e == cudaSuccess) e = cudaMemset(c->b.hot_bits, 0, 4 * (size_t)c->b.hot_words);
  if (e == cudaSuccess) {
    launch_fill_set(c->b.set, c->set_cells, 0);
    e = cudaDeviceSynchronize();
  }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->side2, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_join2, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_nan, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    pb_ctx_destroy(c);
    return fail(PB_ERR_CUDA, std::string("pb_ctx_create: ") + cudaGetErrorString(e));
  }
  *out = c;
  return PB_OK;
}

int pb_ctx_destroy(pb_ctx* c) {
  if (!c) return PB_OK;
  DeviceGuard g(c->device);
  cudaDeviceSynchronize();
  drop_pending(c);
  void* ptrs[] = {c->b.set,   c->b.occ_set, c->b.item_cell, c->b.seg_occ, c->b.cold, c->b.warm, c->b.hot, c->b.hot_bits, c->b.cnt,
                  c->occ_cell, c->occ_outrow, c->row_off, c->nan_tick, c->vw_stage, c->hot_stage, c->dev_tick, c->raw.set,
                  c->raw.occ_set, c->raw.flag, c->raw.rank, c->raw.tiles, c->raw.distinct_cell, c->raw.counts, c->raw_stage};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  if (c->side) cudaStreamDestroy(c->side);
  if (c->side2) cudaStreamDestroy(c->side2);
  if (c->ev_join2) cudaEventDestroy(c->ev_join2);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_nan) cudaEventDestroy(c->ev_nan);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  delete c;
  return PB_OK;
}

int pb_ctx_set_slots(pb_ctx* c, const pb_slots_cfg* cfg) {
  if (!c || !cfg) return fail(PB_ERR_INVALID, "null argument");
  if (cfg->n_slots == 0 || cfg->n_slots > PB_MAX_SLOTS) return fail(PB_ERR_INVALID, "n_slots must be in 1..PB_MAX_SLOTS");
  if (cfg->prefix_bit == 0 || cfg->prefix_bit > 63)  // parse_embedding_config asserts > 0 (config lib.rs:624-627)
    return fail(PB_ERR_INVALID, "feature_index_prefix_bit must be in 1..63");
  c->slots = *cfg;
  c->has_slots = true;
  // two slots with the same prefix share a key space (one feature group): a sign may sit in both, and the reference
  // steps it once per slot, in slot order (mod.rs:720-822).  Slot s runs in round = number of earlier slots of its group.
  c->n_rounds = 1;
  for (uint32_t i = 0; i < cfg->n_slots; ++i) {
    uint32_t r = 0;
    for (uint32_t k = 0; k < i; ++k)
      if (cfg->prefix[i] == cfg->prefix[k]) ++r;
    c->round_of[i] = (uint8_t)r;
    if (r + 1 > c->n_rounds) c->n_rounds = r + 1;
  }
  return PB_OK;
}

int pb_ctx_batch_stats(pb_ctx* c, uint32_t h_out[6], void* stream) {
  if (!c || !h_out) return fail(PB_ERR_INVALID, "null argument");
  DeviceGuard g(c->device);
  uint32_t w[BC_PEER];
  PB_CUDA(cudaMemcpyAsync(w, c->b.cnt, sizeof(w), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  PB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  h_out[0] = w[BC_ITEMS];
  h_out[1] = w[BC_COLD];
  h_out[2] = w[BC_WARM];
  h_out[3] = w[BC_HOT] + w[BC_HUGE] + w[BC_GIANT];
  h_out[4] = w[BC_SEG];
  h_out[5] = c->n_occ;
  return PB_OK;
}

int pb_forward(pb_table* t, pb_ctx* c, const uint64_t* d_ids, uint32_t n_occ, const uint32_t* d_row_off,
               const uint32_t* h_slot_occ_off, uint32_t batch, int training, void* d_out_f16, void* stream) {
  if (!t || !c || !h_slot_occ_off || !d_out_f16 || (n_occ && !d_ids)) return fail(PB_ERR_INVALID, "null argument");
  if (!c->has_slots) return fail(PB_ERR_STATE, "pb_ctx_set_slots not called");
  if (t->device != c->device) return fail(PB_ERR_INVALID, "table and context live on different devices");
  if (batch > 65535) return fail(PB_ERR_BATCH, "batch size cannot be larger than 65535");
  uint32_t S = c->slots.n_slots;
  uint64_t n_out = (uint64_t)S * batch;
  if (n_occ > c->max_occ || n_out > c->max_out) return fail(PB_ERR_CAPACITY, "batch exceeds the context's capacity");
  if (!d_row_off && n_occ != n_out) return fail(PB_ERR_INVALID, "row offsets are required unless every sample has one id per slot");
  if (h_slot_occ_off[0] != 0 || h_slot_occ_off[S] != n_occ) return fail(PB_ERR_INVALID, "slot offsets do not span the id array");
  for (uint32_t s = 0; s < S; ++s)
    if (h_slot_occ_off[s] > h_slot_occ_off[s + 1]) return fail(PB_ERR_INVALID, "slot offsets must ascend");
  int rc;
  if (training) {
    if ((rc = ready_for_training(t))) return rc;
  } else if (!t->has_op) {
    DeviceGuard g(t->device);
    PB_CUDA(cudaMemsetAsync(d_out_f16, 0, 2 * n_out * t->cfg.dim, (cudaStream_t)stream));
    return PB_OK;
  }
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = ensure_alloc(t))) return rc;
  SlotsDev sl;
  if ((rc = make_slots(c->slots, h_slot_occ_off, sl))) return rc;
  // a batch whose gradients never came (or an inference request) leaves its cells in the scratch set: empty it first
  if (c->set_dirty) {
    launch_clear_items(c->b, st);
    c->set_dirty = false;
  }
  if (c->pending) launch_clear_hot_bits(c->b, st);  // its hot items' bitmaps were never consumed
  drop_pending(c);  // like an expired post_forward_buffer entry (mod.rs:991-1029)
  if (training) {
    if ((rc = maybe_evict(t, st))) return rc;
  }
  launch_begin_batch(t->d, training ? c->dev_tick : nullptr, c->b.cnt, st, training != 0);
  c->b.n = n_occ;
  launch_dedup(sl, c->b, d_ids, st);
  launch_probe_items(training != 0, t->d, t->hy, t->op, sl, c->b, st);
  launch_gather_items(t->d, sl, c->b, d_row_off, (uint32_t)n_out, batch, training != 0, d_out_f16, st);
  if (training) {
    c->n_occ = n_occ;
    c->batch = batch;
    c->multi_id = d_row_off != nullptr;
    std::memcpy(c->occ_off, h_slot_occ_off, sizeof(uint32_t) * (S + 1));
    if (d_row_off) {
      PB_CUDA(cudaMemcpyAsync(c->row_off, d_row_off, 4 * (n_out + 1), cudaMemcpyDeviceToDevice, st));
      launch_expand_rows(c->row_off, (uint32_t)n_out, c->occ_outrow, st);
    }
    c->pending = true;
    c->pending_table = t;
    t->pending_batches++;
    c->set_dirty = true;  // emptied beside the backward (or by the next forward)
  } else {
    launch_clear_items(c->b, st);
  }
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_backward(pb_table* t, pb_ctx* c, const void* const* h_grads, int is_f16, const float* h_scale,
                int32_t* d_slot_status, void* stream) {
  if (!t || !c || !h_grads) return fail(PB_ERR_INVALID, "null argument");
  if (!c->pending) return fail(PB_ERR_STATE, "no forward batch is pending in this context (backward_ref_id not found)");
  if (c->pending_table != t) return fail(PB_ERR_INVALID, "the pending batch was looked up in another table");
  int rc = ready_for_training(t);
  if (rc) return rc;
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t S = c->slots.n_slots;
  SlotsDev sl;
  if ((rc = make_slots(c->slots, c->occ_off, sl))) return rc;
  GradsDev gr;
  std::memset(&gr, 0, sizeof(gr));
  for (uint32_t s = 0; s < S; ++s) {
    gr.ptr[s] = h_grads[s];
    float sc = h_scale ? h_scale[s] : 1.0f;
    gr.do_scale[s] = std::fabs(sc - 1.0f) > 1.1920929e-07f;
    float inv = 1.0f / sc;
    if (gr.do_scale[s] && !std::isfinite(inv)) return fail(PB_ERR_INVALID, "scale on gradient must be finite");
    gr.inv_scale[s] = inv;
  }
  AdamKeys adam_keys{};
  if (t->op.kind == PB_OPT_ADAM) {  // get_batch_level_state: one power step per request and feature group
    AdamKeys keys{};
    for (uint32_t s = 0; s < S; ++s) {
      if (!h_grads[s]) continue;
      const int k = adam_index(t, c->slots.prefix[s]);
      if (k < 0) return fail(PB_ERR_CAPACITY, "more feature groups than Adam beta-power pairs");
      gr.pow_idx[s] = (uint8_t)k;
      bool done = false;
      for (uint32_t i = 0; i < keys.n; ++i) done |= keys.idx[i] == (uint8_t)k;
      if (!done) keys.idx[keys.n++] = (uint8_t)k;
    }
    gr.adam_pow = t->adam_dev;
    adam_keys = keys;  // advanced below, once the NaN marks of this request are known
  }
  float* vw = nullptr;
  if (t->op.kind == PB_OPT_ADAGRAD_VW) {
    size_t need = (size_t)c->n_occ * t->d.dim;
    if (need > c->vw_stage_floats) {
      PB_CUDA(cudaStreamSynchronize(st));
      if (c->vw_stage) cudaFree(c->vw_stage);
      c->vw_stage = nullptr;
      c->vw_stage_floats = 0;
      PB_CUDA(cudaMalloc(&c->vw_stage, sizeof(float) * need));
      c->vw_stage_floats = need;
    }
    vw = c->vw_stage;
  }
  const size_t hot_need = (size_t)c->b.hot_cap * hot_stage_stride(t->d.dim);
  if (hot_need > c->hot_stage_floats) {
    PB_CUDA(cudaStreamSynchronize(st));
    if (c->hot_stage) cudaFree(c->hot_stage);
    c->hot_stage = nullptr;
    c->hot_stage_floats = 0;
    PB_CUDA(cudaMalloc(&c->hot_stage, sizeof(float) * hot_need));
    c->hot_stage_floats = hot_need;
  }
  ReduceArgs a;
  std::memset(&a, 0, sizeof(a));
  a.b = c->b;
  a.b.n = c->n_occ;
  a.occ_outrow = c->multi_id ? c->occ_outrow : nullptr;
  a.row_off = c->multi_id ? c->row_off : nullptr;
  a.tick_ptr = c->dev_tick;
  a.nan_tick = c->nan_tick;
  a.vw_stage = vw;
  a.hot_stage = c->hot_stage;
  a.hot_stride = hot_stage_stride(t->d.dim);
  a.batch = c->batch;
  a.quiet_miss = 0;
  auto set_round = [&](uint32_t r) {
    a.round = r;
    std::memset(a.round_mask, 0, sizeof(a.round_mask));
    for (uint32_t s = 0; s < S; ++s)
      if (c->round_of[s] == r) a.round_mask[s >> 5] |= 1u << (s & 31);
  };
  // One round (no shared feature groups, the usual case): the hot items' sums (the long pole) start on `side` at once,
  // beside the NaN scan, and their steps follow the verdict; warm items run on side2 beside the cold ones.  Several
  // rounds: one kernel after another, round by round (the items of a round are distinct rows, whatever their list).
  const bool one = c->n_rounds == 1 && !profiling();  // (timed alone when the bench instruments a family)
  PB_CUDA(cudaEventRecord(c->ev_fork, st));
  PB_CUDA(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
  PB_CUDA(cudaStreamWaitEvent(c->side2, c->ev_fork, 0));
  if (c->set_dirty) {  // nothing in the backward reads the scratch set
    launch_clear_items(c->b, c->side2);
    c->set_dirty = false;
  }
  if (one) {
    set_round(0);
    launch_reduce_hot(t->d, sl, gr, is_f16 != 0, a, c->side);
  }
  uint32_t elems = c->batch * t->d.dim;
  launch_nan_scan(gr, S, elems, is_f16 != 0, c->dev_tick, c->nan_tick, d_slot_status, st);
  if (adam_keys.n) launch_adam_advance(t->adam_dev, adam_keys, t->op.b1, t->op.b2, st, &gr, S, c->dev_tick, c->nan_tick);
  PB_CUDA(cudaEventRecord(c->ev_nan, st));
  PB_CUDA(cudaStreamWaitEvent(c->side, c->ev_nan, 0));
  PB_CUDA(cudaStreamWaitEvent(c->side2, c->ev_nan, 0));
  for (uint32_t r = 0; r < c->n_rounds; ++r) {
    set_round(r);
    if (!one) launch_reduce_hot(t->d, sl, gr, is_f16 != 0, a, st);
    launch_step_hot(t->d, t->op, t->hy, sl, gr, a, one ? c->side : st);
    launch_reduce_items(t->d, t->op, t->hy, sl, gr, is_f16 != 0, a, st, one ? c->side2 : st, false);
  }
  PB_CUDA(cudaEventRecord(c->ev_join, c->side));
  PB_CUDA(cudaStreamWaitEvent(st, c->ev_join, 0));
  PB_CUDA(cudaEventRecord(c->ev_join2, c->side2));
  PB_CUDA(cudaStreamWaitEvent(st, c->ev_join2, 0));
  drop_pending(c);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

// ---- the sharded path: R GPUs of one box -------------------------------------------------------------
struct pb_xchg {
  int device = 0;
  uint32_t dim = 0;
  XchgDev d{};
  uint32_t* mem = nullptr;  // epoch | waited | own_cnt | err | own_row | uwin
  UCell* ucell = nullptr;   // rows of the step's requests (owner side)
  uint64_t* akeys = nullptr;  // Adam: the table's feature-group prefixes on the device
  uint32_t* apresent = nullptr;
  float* apow = nullptr;
  size_t akeys_uploaded = 0;
  bool u_dirty = false;     // a training lookup filled ucell and its update has not run (abandoned batch)
};

namespace {
uint64_t round256(uint64_t v) { return (v + 255u) & ~(uint64_t)255u; }
void xchg_layout(uint32_t R, uint32_t cap, uint32_t dim, int rows_f32, uint64_t off[5]) {
  off[0] = round256((uint64_t)XC_WORDS * PB_MAX_RANKS * 4);                        // sign
  off[1] = off[0] + round256((uint64_t)R * cap * 8);                               // row
  off[2] = off[1] + round256((uint64_t)R * cap * dim * (rows_f32 ? 4 : 2));        // grad
  off[3] = off[2] + round256((uint64_t)R * cap * dim * 4);                         // gok
  off[4] = off[3] + round256((uint64_t)R * cap * 4);                               // end
}
}  // namespace

uint64_t pb_xchg_bytes(uint32_t R, uint32_t cap, uint32_t dim, int rows_f32) {
  if (R == 0 || R > PB_MAX_RANKS || cap == 0 || dim == 0) return 0;
  uint64_t off[5];
  xchg_layout(R, cap, dim, rows_f32, off);
  return off[4];
}

int pb_xchg_create(int device, uint32_t R, uint32_t rank, uint32_t cap, uint32_t dim, int rows_f32,
                   const uint64_t* h_peer_base, pb_xchg** out) {
  if (!out || !h_peer_base || R == 0 || R > PB_MAX_RANKS || rank >= R || cap == 0 || dim == 0)
    return fail(PB_ERR_INVALID, "bad argument");
  if ((uint64_t)R * cap >= 0xFFFFFFF0ull) return fail(PB_ERR_INVALID, "R * cap must stay below 2^32 - 16");
  for (uint32_t q = 0; q < R; ++q)
    if (!h_peer_base[q] || (h_peer_base[q] & 255u)) return fail(PB_ERR_INVALID, "receive areas must be mapped and 256-byte aligned");
  DeviceGuard g(device);
  pb_xchg* x = new pb_xchg();
  x->device = device;
  x->dim = dim;
  uint64_t off[5];
  xchg_layout(R, cap, dim, rows_f32, off);
  XchgDev& d = x->d;
  std::memset(&d, 0, sizeof(d));
  for (uint32_t q = 0; q < R; ++q) d.base[q] = h_peer_base[q];
  d.off_sign = off[0];
  d.off_row = off[1];
  d.off_grad = off[2];
  d.off_gok = off[3];
  d.R = R;
  d.rank = rank;
  d.cap = cap;
  d.row_f32 = rows_f32 ? 1 : 0;
  const size_t words = XC_WORDS + (size_t)XC_WORDS * PB_MAX_RANKS + PB_MAX_RANKS + 4 + 2 * (size_t)R * cap;
  cudaError_t e = cudaMalloc(&x->mem, 4 * words);
  if (e == cudaSuccess) e = cudaMemset(x->mem, 0, 4 * words);
  uint32_t ucells = 1024;
  while ((size_t)ucells < 2 * (size_t)R * cap) ucells <<= 1;
  if (e == cudaSuccess) e = cudaMalloc(&x->ucell, sizeof(UCell) * (size_t)ucells);
  if (e == cudaSuccess) e = cudaMalloc(&x->akeys, sizeof(uint64_t) * PB_ADAM_KEYS);
  if (e == cudaSuccess) e = cudaMalloc(&x->apresent, sizeof(uint32_t) * PB_MAX_RANKS * (PB_ADAM_KEYS / 32));
  if (e == cudaSuccess) e = cudaMemset(x->apresent, 0, sizeof(uint32_t) * PB_MAX_RANKS * (PB_ADAM_KEYS / 32));
  if (e == cudaSuccess) e = cudaMalloc(&x->apow, sizeof(float) * 2 * PB_MAX_RANKS * PB_ADAM_KEYS);

  if (e != cudaSuccess) {
    delete x;
    return fail(PB_ERR_CUDA, std::string("pb_xchg_create: ") + cudaGetErrorString(e));
  }
  d.epoch = x->mem;
  d.waited = d.epoch + XC_WORDS;
  d.own_cnt = d.waited + (size_t)XC_WORDS * PB_MAX_RANKS;
  d.err = d.own_cnt + PB_MAX_RANKS;
  d.own_row = d.err + 4;
  d.uwin = d.own_row + (size_t)R * cap;
  d.ucell = x->ucell;
  d.ucells = ucells;
  d.akeys = x->akeys;
  d.apresent = x->apresent;
  d.apow = x->apow;
  launch_uclear(d, nullptr);
  PB_CUDA(cudaDeviceSynchronize());
  *out = x;
  return PB_OK;
}

int pb_xchg_destroy(pb_xchg* x) {
  if (!x) return PB_OK;
  DeviceGuard g(x->device);
  cudaDeviceSynchronize();
  if (x->mem) cudaFree(x->mem);
  if (x->ucell) cudaFree(x->ucell);
  if (x->akeys) cudaFree(x->akeys);
  if (x->apresent) cudaFree(x->apresent);
  if (x->apow) cudaFree(x->apow);
  delete x;
  return PB_OK;
}

int pb_xchg_status(pb_xchg* x, uint32_t h_out[2], void* stream) {
  if (!x || !h_out) return fail(PB_ERR_INVALID, "null argument");
  DeviceGuard g(x->device);
  PB_CUDA(cudaMemcpyAsync(h_out, x->d.err, 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  PB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return PB_OK;
}

int pb_forward_sharded(pb_table* t, pb_ctx* c, pb_xchg* x, const uint64_t* d_ids, uint32_t n_occ, const uint32_t* d_row_off,
                       const uint32_t* h_slot_occ_off, uint32_t batch, int training, void* d_out_f16, void* stream,
                       int phases) {
  if (phases == 0) phases = PB_PHASE_ALL;
  const bool all = phases == PB_PHASE_ALL;
  if (!t || !c || !x || !h_slot_occ_off || !d_out_f16 || (n_occ && !d_ids)) return fail(PB_ERR_INVALID, "null argument");
  if (!c->has_slots) return fail(PB_ERR_STATE, "pb_ctx_set_slots not called");
  if (t->device != c->device || t->device != x->device) return fail(PB_ERR_INVALID, "table, context and exchange live on different devices");
  if (x->dim != t->cfg.dim) return fail(PB_ERR_INVALID, "the exchange was sized for another embedding dim");
  if (batch > 65535) return fail(PB_ERR_BATCH, "batch size cannot be larger than 65535");
  if (c->n_rounds != 1) return fail(PB_ERR_INVALID, "slots sharing a feature group are not supported on the sharded path");
  if (d_row_off && !x->d.row_f32) return fail(PB_ERR_INVALID, "ragged layouts need an exchange created with f32 rows");
  uint32_t S = c->slots.n_slots;
  uint64_t n_out = (uint64_t)S * batch;
  if (n_occ > c->max_occ || n_out > c->max_out) return fail(PB_ERR_CAPACITY, "batch exceeds the context's capacity");
  if (!d_row_off && n_occ != n_out) return fail(PB_ERR_INVALID, "row offsets are required unless every sample has one id per slot");
  if (h_slot_occ_off[0] != 0 || h_slot_occ_off[S] != n_occ) return fail(PB_ERR_INVALID, "slot offsets do not span the id array");
  for (uint32_t s = 0; s < S; ++s)
    if (h_slot_occ_off[s] > h_slot_occ_off[s + 1]) return fail(PB_ERR_INVALID, "slot offsets must ascend");
  int rc;
  // every rank serves lookups whether or not its own batch trains: the shard must be usable (a collective call)
  if ((rc = ready_for_training(t))) return rc;
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = ensure_alloc(t))) return rc;
  SlotsDev sl;
  if ((rc = make_slots(c->slots, h_slot_occ_off, sl))) return rc;
  if (phases & PB_PHASE_SEND) {
    if (c->set_dirty) {
      launch_clear_items(c->b, st);
      c->set_dirty = false;
    }
    if (c->pending) launch_clear_hot_bits(c->b, st);
    drop_pending(c);
    if (training) {
      if ((rc = maybe_evict(t, st))) return rc;
    }
    launch_begin_batch(t->d, training ? c->dev_tick : nullptr, c->b.cnt, st, training != 0);
    c->b.n = n_occ;
    launch_dedup(sl, c->b, d_ids, st);
    launch_route_items(training != 0, sl, c->b, x->d, st);               // requester: signs -> owners' areas
    if (all) launch_signal_wait(x->d, XC_FLAG_SIGN, c->b.cnt + BC_PEER, st);  // (one launch when no phase split is asked for)
    else launch_signal(x->d, XC_FLAG_SIGN, c->b.cnt + BC_PEER, st);
  }
  if (phases & PB_PHASE_SERVE) {
    if (!all) launch_wait(x->d, XC_FLAG_SIGN, -1, st);
    if (training && x->u_dirty) launch_uclear(x->d, st);  // a training batch whose gradients never came left its rows noted
    launch_owner_lookup(training != 0, t->d, t->hy, t->op, x->d, st);    // owner: rows -> requesters' areas
    if (training) x->u_dirty = true;
    if (all) launch_signal_wait(x->d, XC_FLAG_ROW, nullptr, st);
    else launch_signal(x->d, XC_FLAG_ROW, nullptr, st);
  }
  if (!(phases & PB_PHASE_FINISH)) {
    PB_CUDA(cudaGetLastError());
    return PB_OK;
  }
  if (!all) launch_wait(x->d, XC_FLAG_ROW, -1, st);
  launch_expand_items(t->d, sl, c->b, x->d, d_row_off, (uint32_t)n_out, batch, training != 0, d_out_f16, st);
  if (training) {
    c->n_occ = n_occ;
    c->batch = batch;
    c->multi_id = d_row_off != nullptr;
    std::memcpy(c->occ_off, h_slot_occ_off, sizeof(uint32_t) * (S + 1));
    if (d_row_off) {
      PB_CUDA(cudaMemcpyAsync(c->row_off, d_row_off, 4 * (n_out + 1), cudaMemcpyDeviceToDevice, st));
      launch_expand_rows(c->row_off, (uint32_t)n_out, c->occ_outrow, st);
    }
    c->pending = true;
    c->pending_table = t;
    t->pending_batches++;
    c->set_dirty = true;
  } else {
    launch_clear_items(c->b, st);
  }
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_backward_sharded(pb_table* t, pb_ctx* c, pb_xchg* x, const void* const* h_grads, int is_f16, const float* h_scale,
                        int32_t* d_slot_status, void* stream, int phases) {
  if (phases == 0) phases = PB_PHASE_ALL;
  if (!t || !c || !x || !h_grads) return fail(PB_ERR_INVALID, "null argument");
  if (!c->pending) return fail(PB_ERR_STATE, "no forward batch is pending in this context (backward_ref_id not found)");
  if (c->pending_table != t) return fail(PB_ERR_INVALID, "the pending batch was looked up in another table");
  int rc = ready_for_training(t);
  if (rc) return rc;
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t S = c->slots.n_slots;
  SlotsDev sl;
  if ((rc = make_slots(c->slots, c->occ_off, sl))) return rc;
  GradsDev gr;
  std::memset(&gr, 0, sizeof(gr));
  for (uint32_t s = 0; s < S; ++s) {
    gr.ptr[s] = h_grads[s];
    float sc = h_scale ? h_scale[s] : 1.0f;
    gr.do_scale[s] = std::fabs(sc - 1.0f) > 1.1920929e-07f;
    float inv = 1.0f / sc;
    if (gr.do_scale[s] && !std::isfinite(inv)) return fail(PB_ERR_INVALID, "scale on gradient must be finite");
    gr.inv_scale[s] = inv;
  }
  if (phases & PB_PHASE_SEND) {
  PB_CUDA(cudaEventRecord(c->ev_fork, st));
  PB_CUDA(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
  if (c->set_dirty) {
    launch_clear_items(c->b, c->side);
    c->set_dirty = false;
  }
  launch_nan_scan(gr, S, c->batch * t->d.dim, is_f16 != 0, c->dev_tick, c->nan_tick, d_slot_status, st);  // per slot, on the requester (mod.rs:731-746)
  PB_CUDA(cudaEventRecord(c->ev_nan, st));
  PB_CUDA(cudaStreamWaitEvent(c->side, c->ev_nan, 0));
  PB_CUDA(cudaStreamWaitEvent(c->side2, c->ev_nan, 0));
  ReduceArgs a;
  std::memset(&a, 0, sizeof(a));
  a.b = c->b;
  a.b.n = c->n_occ;
  a.occ_outrow = c->multi_id ? c->occ_outrow : nullptr;
  a.row_off = c->multi_id ? c->row_off : nullptr;
  a.tick_ptr = c->dev_tick;
  a.nan_tick = c->nan_tick;
  a.batch = c->batch;
  a.round = 0;
  for (uint32_t s = 0; s < S; ++s) a.round_mask[s >> 5] |= 1u << (s & 31);
  a.x = x->d;
  PB_CUDA(cudaStreamWaitEvent(c->side2, c->ev_nan, 0));
  // requester: gradients -> owners' areas
  launch_reduce_hot(t->d, sl, gr, is_f16 != 0, a, profiling() ? st : c->side, true);
  launch_reduce_items(t->d, t->op, t->hy, sl, gr, is_f16 != 0, a, st, profiling() ? st : c->side2, true);
  PB_CUDA(cudaEventRecord(c->ev_join, c->side));
  PB_CUDA(cudaStreamWaitEvent(st, c->ev_join, 0));
  PB_CUDA(cudaEventRecord(c->ev_join2, c->side2));
  PB_CUDA(cudaStreamWaitEvent(st, c->ev_join2, 0));
  if (phases == PB_PHASE_ALL && t->op.kind != PB_OPT_ADAGRAD_VW) launch_signal_wait(x->d, XC_FLAG_GRAD, nullptr, st);
  else launch_signal(x->d, XC_FLAG_GRAD, nullptr, st);
  }
  if (!(phases & PB_PHASE_SERVE)) {
    PB_CUDA(cudaGetLastError());
    return PB_OK;
  }
  if (t->op.kind == PB_OPT_ADAGRAD_VW) {  // (needs the whole gradient's dot per step) one request after another
    for (uint32_t src = 0; src < x->d.R; ++src) {
      launch_wait(x->d, XC_FLAG_GRAD, (int)src, st);
      launch_owner_update(t->d, t->op, t->hy, x->d, src, st);
    }
    launch_uclear(x->d, st);
  } else {  // owner: the R requests in one launch, every row stepped in rank order
    if (phases != PB_PHASE_ALL) launch_wait(x->d, XC_FLAG_GRAD, -1, st);
    if (t->op.kind == PB_OPT_ADAM) {  // every request advances the beta powers of the feature groups it holds here
      for (uint32_t s = 0; s < S; ++s)
        if (adam_index(t, c->slots.prefix[s]) < 0) return fail(PB_ERR_CAPACITY, "more feature groups than Adam beta-power pairs");
      if (x->akeys_uploaded != t->adam_keys.size()) {  // (first steps only: not inside a graph capture)
        PB_CUDA(cudaStreamSynchronize(st));
        PB_CUDA(cudaMemcpy(x->akeys, t->adam_keys.data(), sizeof(uint64_t) * t->adam_keys.size(), cudaMemcpyHostToDevice));
        x->akeys_uploaded = t->adam_keys.size();
      }
      x->d.n_akeys = (uint32_t)t->adam_keys.size();
      x->d.amask = ~sl.spacing;
      launch_owner_adam(x->d, t->adam_dev, t->op.b1, t->op.b2, st);
    }
    launch_owner_update_all(t->d, t->op, t->hy, x->d, st);
  }
  x->u_dirty = false;
  drop_pending(c);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

// ---- raw slots ------------------------------------------------------------------------------------
static int ensure_raw(pb_ctx* c) {
  if (c->raw_ready) return PB_OK;
  RawWork& w = c->raw;
  size_t n = c->max_occ;
  size_t m = n > c->max_out ? n : c->max_out;
  uint32_t cells = next_pow2(2 * (uint64_t)n < 1024 ? 1024 : 2 * (uint64_t)n);
  w.set_mask = cells - 1;
  PB_CUDA(cudaMalloc(&w.set, sizeof(RawCell) * ((size_t)cells + 1)));
  PB_CUDA(cudaMalloc(&w.occ_set, 4 * n));
  PB_CUDA(cudaMalloc(&w.flag, 4 * m));
  PB_CUDA(cudaMalloc(&w.rank, 4 * m));
  PB_CUDA(cudaMalloc(&w.tiles, 4 * (size_t)raw_scan_tiles((uint32_t)m)));
  PB_CUDA(cudaMalloc(&w.distinct_cell, 4 * n));
  PB_CUDA(cudaMalloc(&w.counts, 8));
  PB_CUDA(cudaMemset(w.counts, 0, 8));
  c->raw_ready = true;
  return PB_OK;
}

int pb_forward_raw(pb_table* t, pb_ctx* c, const uint64_t* d_ids, uint32_t n_occ, const uint32_t* d_row_off,
                   uint32_t batch, uint32_t sample_fixed_size, int training, void* d_table_f16, int64_t* d_index,
                   int64_t* d_non_empty, uint32_t* d_sample_id_num, uint32_t* d_counts, void* stream) {
  if (!t || !c || !d_table_f16 || !d_index || !d_non_empty || !d_sample_id_num || !d_counts || (n_occ && !d_ids))
    return fail(PB_ERR_INVALID, "null argument");
  if (!c->has_slots || c->slots.n_slots != 1) return fail(PB_ERR_STATE, "a raw context serves exactly one slot (pb_ctx_set_slots)");
  if (t->device != c->device) return fail(PB_ERR_INVALID, "table and context live on different devices");
  if (batch > 65535) return fail(PB_ERR_BATCH, "batch size cannot be larger than 65535");
  if (sample_fixed_size == 0) return fail(PB_ERR_INVALID, "sample_fixed_size must be positive");
  if (n_occ > c->max_occ || batch > c->max_out || (uint64_t)batch * sample_fixed_size > (1ull << 31))
    return fail(PB_ERR_CAPACITY, "batch exceeds the context's capacity");
  if (!d_row_off && n_occ != batch) return fail(PB_ERR_INVALID, "row offsets are required unless every sample has one id");
  int rc;
  if (training) {
    if ((rc = ready_for_training(t))) return rc;
  } else if (!t->has_op) {
    return fail(PB_ERR_STATE, "optimizer not registered (OptimizerNotFoundError)");
  }
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = ensure_alloc(t))) return rc;
  if ((rc = ensure_raw(c))) return rc;
  const uint32_t occ_off[2] = {0, n_occ};
  SlotsDev sl;
  if ((rc = make_slots(c->slots, occ_off, sl))) return rc;
  sl.uniform = 0;
  if (training) {
    if ((rc = maybe_evict(t, st))) return rc;
    launch_begin_batch(t->d, c->dev_tick, nullptr, st);
    launch_probe(MODE_TRAIN, true, t->d, t->hy, t->op, sl, d_ids, n_occ, c->occ_cell, st);
  } else {
    launch_probe(MODE_FIND, true, t->d, t->hy, t->op, sl, d_ids, n_occ, c->occ_cell, st);
  }
  const uint32_t* occ_sample = nullptr;
  if (d_row_off) {
    PB_CUDA(cudaMemcpyAsync(c->row_off, d_row_off, 4 * ((size_t)batch + 1), cudaMemcpyDeviceToDevice, st));
    launch_expand_rows(c->row_off, batch, c->occ_outrow, st);
    occ_sample = c->occ_outrow;
  }
  launch_raw_forward(t->d, sl, d_ids, n_occ, d_row_off ? c->row_off : nullptr, occ_sample, batch, sample_fixed_size,
                     c->occ_cell, c->raw, d_table_f16, (long long*)d_index, (long long*)d_non_empty, d_sample_id_num, st);
  PB_CUDA(cudaMemcpyAsync(d_counts, c->raw.counts, 8, cudaMemcpyDeviceToDevice, st));
  if (training) {
    c->n_occ = n_occ;
    c->batch = batch;
    c->raw_pending = true;
  }
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

int pb_backward_raw(pb_table* t, pb_ctx* c, const void* d_grad, int is_f16, float scale, int32_t* d_status,
                    void* stream) {
  if (!t || !c) return fail(PB_ERR_INVALID, "null argument");
  if (!c->raw_pending) return fail(PB_ERR_STATE, "no raw forward batch is pending in this context (backward_ref_id not found)");
  int rc = ready_for_training(t);
  if (rc) return rc;
  DeviceGuard g(t->device);
  cudaStream_t st = (cudaStream_t)stream;
  c->raw_pending = false;
  GradsDev gr;
  std::memset(&gr, 0, sizeof(gr));
  gr.ptr[0] = d_grad;
  if (!d_grad) {  // add_skipped_gradient
    if (d_status) launch_slot_status(gr, 1, c->dev_tick, c->nan_tick, d_status, st);
    return PB_OK;
  }
  const bool do_scale = std::fabs(scale - 1.0f) > 1.1920929e-07f;
  const float inv = 1.0f / scale;
  if (do_scale && !std::isfinite(inv)) return fail(PB_ERR_INVALID, "scale on gradient must be finite");
  const float* pair = nullptr;
  if (t->op.kind == PB_OPT_ADAM) {  // one power step per request and feature group (optim.rs:155-197)
    const int k = adam_index(t, c->slots.prefix[0]);
    if (k < 0) return fail(PB_ERR_CAPACITY, "more feature groups than Adam beta-power pairs");
    AdamKeys keys{};
    keys.idx[0] = (uint8_t)k;
    keys.n = 1;
    launch_adam_advance(t->adam_dev, keys, t->op.b1, t->op.b2, st);
    pair = t->adam_dev + 2 * k;
  }
  const uint32_t dim = t->d.dim;
  launch_raw_nan(d_grad, is_f16 != 0, c->raw.counts, dim, c->dev_tick, c->nan_tick, st);
  if (d_status) launch_slot_status(gr, 1, c->dev_tick, c->nan_tick, d_status, st);
  const float* g32 = (const float*)d_grad;
  if (is_f16 || do_scale) {
    size_t need = (size_t)c->n_occ * dim;
    if (need > c->raw_stage_floats) {
      PB_CUDA(cudaStreamSynchronize(st));
      if (c->raw_stage) cudaFree(c->raw_stage);
      c->raw_stage = nullptr;
      c->raw_stage_floats = 0;
      size_t cap = (size_t)c->max_occ * dim;
      PB_CUDA(cudaMalloc(&c->raw_stage, sizeof(float) * cap));
      c->raw_stage_floats = cap;
    }
    launch_raw_stage(d_grad, is_f16 != 0, c->raw.counts, dim, inv, do_scale, c->raw_stage, st);
    g32 = c->raw_stage;
  }
  launch_update_direct(t->d, t->op, t->hy, c->raw.distinct_cell, g32, c->n_occ, pair, st, c->raw.counts,
                       c->dev_tick, c->nan_tick);
  PB_CUDA(cudaGetLastError());
  return PB_OK;
}

}  // extern "C"

// debugging aid (not in include/persia_b200.h): device buffer of 4 u64 per hot item that k_reduce_hot stamps
namespace pb { void set_hot_trace(unsigned long long* p); }
extern "C" void pb_debug_hot_trace(void* d_buf) { pb::set_hot_trace(reinterpret_cast<unsigned long long*>(d_buf)); }
