// pb_update.cu — the NaN rule of the backward (A8), pb_update's direct optimizer step and Adam's batch-level state.
// The batched reduce + step is pb_reduce.cu.  SURVEY.md §8a.
#include "pb_optim.cuh"

namespace pb {

// ------------------------------------------------------------------------------------------------
// A8 (NaN rule): a slot whose gradient holds any NaN is skipped whole (mod.rs:731-746).
// status[s] = tick when a NaN was seen (no reset needed between batches).
//
// A pure streaming read.  Each slot's gradient is cut into tiles of NAN_THREADS x NAN_LOADS 16-byte vectors; the grid
// (a few blocks per SM) strides over the tiles of all slots, and a thread has the NAN_LOADS loads of its tile in flight
// together.  The scan runs beside k_reduce_hot, one 256-thread block of <= 224 registers per SM, which leaves 8192
// registers and no spare shared memory: __maxnreg__(32) keeps a scan block small enough to fit next to it.
// A value is NaN iff its magnitude bits exceed those of inf, so one running unsigned max of the magnitudes (per 16-bit
// half for f16: __vmaxu2) decides the whole tile.  Elements before the first 16-byte boundary of a slot and after the
// last whole vector are checked one by one by the slot's first tile.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t NAN_THREADS = 256;
constexpr uint32_t NAN_LOADS = 4;  // 16-byte loads in flight per thread
constexpr uint32_t NAN_TILE = NAN_THREADS * NAN_LOADS;  // vectors per tile

template <bool F16>
__global__ void __maxnreg__(32) k_nan_scan(GradsDev gr, uint32_t n_slots, uint32_t elems_per_slot, uint32_t tiles_per_slot,
                                           const uint32_t* __restrict__ tick_ptr, uint32_t* __restrict__ nan_tick) {
  constexpr uint32_t ES = F16 ? 2u : 4u, EV = 16u / ES;  // bytes per element, elements per vector
  constexpr uint32_t MAG = F16 ? 0x7fff7fffu : 0x7fffffffu;
  const uint32_t n_tiles = n_slots * tiles_per_slot;
  for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {  // (uniform over the block)
    const uint32_t s = t / tiles_per_slot, tile = t - s * tiles_per_slot;
    const unsigned char* base = reinterpret_cast<const unsigned char*>(gr.ptr[s]);
    if (!base) continue;  // skipped slot: nothing to read
    const uint32_t head = min(elems_per_slot, ((16u - (uint32_t)(reinterpret_cast<uintptr_t>(base) & 15u)) & 15u) / ES);
    const uint32_t nv = (elems_per_slot - head) / EV;
    const uint4* p = reinterpret_cast<const uint4*>(base + head * ES);
    uint32_t m = 0;  // running max of the magnitudes
    if (tile == 0) {  // the elements outside the whole vectors: [0, head) and [head + nv * EV, elems)
      const uint32_t body_end = head + nv * EV;
      for (uint32_t e = threadIdx.x; e < head + (elems_per_slot - body_end); e += NAN_THREADS) {
        const uint32_t k = e < head ? e : body_end + (e - head);
        const uint32_t x = F16 ? reinterpret_cast<const uint16_t*>(base)[k] : reinterpret_cast<const uint32_t*>(base)[k];
        m = F16 ? __vmaxu2(m, x & 0x7fffu) : max(m, x & MAG);
      }
    }
    const uint32_t j0 = tile * NAN_TILE + threadIdx.x;
    uint4 v[NAN_LOADS];
#pragma unroll
    for (uint32_t u = 0; u < NAN_LOADS; ++u) {
      const uint32_t j = j0 + u * NAN_THREADS;
      v[u] = j < nv ? p[j] : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (uint32_t u = 0; u < NAN_LOADS; ++u) {
      if (F16) {
        m = __vmaxu2(m, __vmaxu2(__vmaxu2(v[u].x & MAG, v[u].y & MAG), __vmaxu2(v[u].z & MAG, v[u].w & MAG)));
      } else {
        m = max(m, max(max(v[u].x & MAG, v[u].y & MAG), max(v[u].z & MAG, v[u].w & MAG)));
      }
    }
    const bool bad = F16 ? ((m & 0xffffu) > 0x7c00u || (m >> 16) > 0x7c00u)  // (h & 0x7fff) > 0x7c00: 0x7c00 is inf
                         : m > 0x7f800000u;                                   // isnan
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) nan_tick[s] = *tick_ptr;
  }
}

__global__ void k_slot_status(GradsDev gr, uint32_t n_slots, const uint32_t* __restrict__ tick_ptr,
                              const uint32_t* __restrict__ nan_tick, int32_t* __restrict__ status) {
  uint32_t s = threadIdx.x;
  const uint32_t tick = *tick_ptr;
  if (s < n_slots) status[s] = !gr.ptr[s] ? 1 : (nan_tick[s] == tick ? 2 : 0);
}

// pb_update: distinct signs with explicit f32 gradients (update_gradient_mixed, PS mod.rs:359-427).
template <int VEC, int G>
__global__ void __launch_bounds__(256) k_update_direct(TableDev t, OptimDev op, HyperDev hy,
                                                       const uint32_t* __restrict__ occ_cell,
                                                       const float* __restrict__ grads, uint32_t n,
                                                       const float* __restrict__ adam_pair,
                                                       const uint32_t* __restrict__ n_ptr,
                                                       const uint32_t* __restrict__ tick_ptr,
                                                       const uint32_t* __restrict__ nan_tick) {
  uint32_t gid = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  uint32_t lane = threadIdx.x % G;
  if (n_ptr) n = *n_ptr;
  if (gid >= n) return;
  if (nan_tick && nan_tick[0] == *tick_ptr) return;  // NaN rule: the whole gradient is dropped
  uint32_t h = occ_cell[gid];
  uint32_t row = (h < t.n_cells + N_SPECIAL) ? t.cells[h].row : ROW_NONE;
  if (row >= t.capacity) {
    if (lane == 0) atomicAdd(&t.counters[CTR_GRAD_MISS], 1u);
    return;
  }
  float* prow = t.rows + (size_t)row * t.stride;
  const uint32_t nvec = t.dim / VEC;
  StepCtx sc;
  sc.vw_state = (op.kind == PB_OPT_ADAGRAD_VW) ? prow[t.dim] : 0.0f;
  sc.r1 = sc.r2 = 0.0f;
  if (op.kind == PB_OPT_ADAM) {
    sc.r1 = __fdiv_rn(1.0f, __fsub_rn(1.0f, adam_pair[0]));
    sc.r2 = __fdiv_rn(1.0f, __fsub_rn(1.0f, adam_pair[1]));
  }
  const float* g0 = grads + (size_t)gid * t.dim;
  for (uint32_t c = lane; c < nvec; c += G) {
    float g[VEC];
    load_vec<VEC>(g0 + c * VEC, g);
    RowElems<-1, VEC> rc;
    rc.load(prow, c * VEC, t, op);
    rc.step(c * VEC, g, t, op, hy, sc);
    rc.store(prow, c * VEC, t, op);
  }
  if (op.kind == PB_OPT_ADAGRAD_VW && lane == 0) {
    float gs = __fdiv_rn(vw_dot(g0, t.dim), (float)t.dim);
    prow[t.dim] = __fadd_rn(__fmul_rn(sc.vw_state, op.mom), gs);
  }
}

// ------------------------------------------------------------------------------------------------
// launchers (host)
// ------------------------------------------------------------------------------------------------
void launch_nan_scan(const GradsDev& gr, uint32_t n_slots, uint32_t elems_per_slot, bool f16, const uint32_t* tick,
                     uint32_t* nan_tick, int32_t* status, cudaStream_t st) {
  const uint32_t nv = elems_per_slot / (f16 ? 8u : 4u);
  const uint32_t tiles_per_slot = nv ? cdiv(nv, NAN_TILE) : 1u;
  uint32_t grid = n_slots * tiles_per_slot;
  if (grid > 148u * 4u) grid = 148u * 4u;  // blocks stride over the tiles
  if (f16) PB_LAUNCH_F(FAM_NAN, k_nan_scan<true>, grid, NAN_THREADS, 0, st, gr, n_slots, elems_per_slot, tiles_per_slot, tick, nan_tick);
  else PB_LAUNCH_F(FAM_NAN, k_nan_scan<false>, grid, NAN_THREADS, 0, st, gr, n_slots, elems_per_slot, tiles_per_slot, tick, nan_tick);
  if (status) PB_LAUNCH(k_slot_status, 1, PB_MAX_SLOTS, 0, st, gr, n_slots, tick, nan_tick, status);
}

// Adam's batch-level state (optim.rs:99-131, 155-197): one (beta1^t, beta2^t) pair per feature group, kept on the
// device so that a captured backward advances it on every replay.
__global__ void k_adam_fill(float* pow, float b1, float b2) {
  uint32_t i = threadIdx.x;
  if (i < PB_ADAM_KEYS) {
    pow[2 * i] = b1;
    pow[2 * i + 1] = b2;
  }
}
// gr / tick / nan_tick (optional): a feature group advances only if one of its slots is applied by this request — a slot
// skipped for a NaN gradient sends nothing to the parameter server (mod.rs:731-746), so it cannot advance the powers
__global__ void k_adam_advance(float* pow, AdamKeys keys, float b1, float b2, GradsDev gr, uint32_t n_slots,
                               const uint32_t* __restrict__ tick, const uint32_t* __restrict__ nan_tick) {
  uint32_t i = threadIdx.x;
  if (i < keys.n) {
    bool applied = nan_tick == nullptr;
    if (!applied) {
      const uint32_t now = *tick;
      for (uint32_t s = 0; s < n_slots; ++s) applied |= gr.ptr[s] && gr.pow_idx[s] == keys.idx[i] && nan_tick[s] != now;
    }
    if (applied) {
      float* p = pow + 2u * keys.idx[i];
      p[0] = __fmul_rn(p[0], b1);
      p[1] = __fmul_rn(p[1], b2);
    }
  }
}
void launch_adam_fill(float* pow, float b1, float b2, cudaStream_t st) { PB_LAUNCH(k_adam_fill, 1, PB_ADAM_KEYS, 0, st, pow, b1, b2); }
void launch_adam_advance(float* pow, const AdamKeys& keys, float b1, float b2, cudaStream_t st, const GradsDev* gr,
                         uint32_t n_slots, const uint32_t* tick, const uint32_t* nan_tick) {
  GradsDev none{};
  if (keys.n) PB_LAUNCH(k_adam_advance, 1, PB_MAX_SLOTS, 0, st, pow, keys, b1, b2, gr ? *gr : none, n_slots, tick, gr ? nan_tick : nullptr);
}

void launch_slot_status(const GradsDev& gr, uint32_t n_slots, const uint32_t* tick, const uint32_t* nan_tick,
                        int32_t* status, cudaStream_t st) {
  PB_LAUNCH(k_slot_status, 1, PB_MAX_SLOTS, 0, st, gr, n_slots, tick, nan_tick, status);
}

void launch_update_direct(const TableDev& t, const OptimDev& op, const HyperDev& hy, const uint32_t* occ_cell,
                          const float* grads, uint32_t n, const float* adam_pair, cudaStream_t st,
                          const uint32_t* n_ptr, const uint32_t* tick, const uint32_t* nan_tick) {
  if (!n) return;
  int vec, G;
  vec_group(t.dim, vec, G);
  uint32_t grid = cdiv((uint64_t)n * G, 256);
#define PB_U(V, GG)                                                                                          \
  if (vec == V && G == GG)                                                                                   \
    PB_LAUNCH_F(FAM_UPDATE, (k_update_direct<V, GG>), grid, 256, 0, st, t, op, hy, occ_cell, grads, n, adam_pair, n_ptr, \
                tick, nan_tick);
  PB_U(4, 1) PB_U(4, 2) PB_U(4, 4) PB_U(4, 8) PB_U(4, 16) PB_U(4, 32)
  PB_U(1, 1) PB_U(1, 2) PB_U(1, 4) PB_U(1, 8) PB_U(1, 16) PB_U(1, 32)
#undef PB_U
}

}  // namespace pb
