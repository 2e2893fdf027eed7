// pb_reduce.cu — backward of the batched path: per distinct sign, the in-order gradient segment reduce (A8) fused with
// the optimizer step and weight bound on the resident row (A9).  SURVEY.md §8a.
//
// Reference: update_all_batched_gradients (embedding_worker_service/mod.rs:703-872) reduces, per slot and distinct
// sign, the gradients of the samples holding the sign — sequentially, in the order FeatureBatch::new listed them
// (ascending sample) — and update_gradient_mixed (embedding_parameter_service/mod.rs:359-427) performs one optimizer
// step per (slot, sign) with the sum.  f32 addition is not associative, so the order is kept exactly, for any
// multiplicity: results are bit-identical to the reference's whatever a sign's popularity.
//
// The forward left three work lists (pb_dedup.cu): cold items (one occurrence — nothing to reduce), warm items
// (2..PB_WARM_MAX occurrences, list unsorted) and hot items (more: the head of the Zipf curve and every sign of a
// tiny-cardinality slot, thousands of occurrences each).
//   k_reduce_cold   a lane group per item: two independent loads (row, gradient), step, store — light on registers, the
//                   whole chip's worth of groups resident.
//   k_reduce_warm   a lane group per item: the group sorts the item's <= 32 occurrences in shared memory (rank by
//                   counting), then adds them in order.
//   k_reduce_hot    persistent; a CTA per item.  The occurrences are put in order from a bitmap over the slot's
//                   samples (a counting sort that costs B/32 words); producer warps stream the gradient rows into a
//                   shared-memory ring, chain warps add them in order — a dependent FADD chain fed from shared memory,
//                   which is the floor for a strictly sequential sum — and store the sum to the hot stage.  It reads no
//                   NaN verdict, so it runs beside the NaN scan.
//   k_step_hot      a warp per hot item, after the NaN verdict: the optimizer step with the staged sum.
#include <cstdlib>

#include "pb_optim.cuh"

namespace pb {

// ------------------------------------------------------------------------------------------------
// shared pieces
// ------------------------------------------------------------------------------------------------
struct ItemSrc {  // where an item's gradients come from
  const void* gbase;    // the slot's gradient tensor [batch, dim]
  uint32_t slot_row0;   // slot * batch
  float inv_scale;
  bool do_scale, do_sqrt, plain;
};

__device__ __forceinline__ ItemSrc item_src(const SlotsDev& sl, const GradsDev& gr, const ReduceArgs& a, uint32_t slot) {
  ItemSrc s;
  s.gbase = gr.ptr[slot];
  s.slot_row0 = slot * a.batch;
  s.inv_scale = gr.inv_scale[slot];
  s.do_scale = gr.do_scale[slot];
  s.do_sqrt = sl.sqrt_scaling[slot];
  s.plain = !a.occ_outrow && !s.do_scale && !s.do_sqrt;
  return s;
}

// output row (= gradient row) of an occurrence and its sample's sqrt factor (mirror of the forward scaling without
// its max(.,1), mod.rs:757-768)
__device__ __forceinline__ uint32_t occ_out_row(const ReduceArgs& a, uint32_t occ) {
  return a.occ_outrow ? a.occ_outrow[occ] : occ;
}
__device__ __forceinline__ GradPrep grad_prep(const ItemSrc& s, const ReduceArgs& a, uint32_t orow) {
  GradPrep p;
  p.inv_scale = s.inv_scale;
  p.do_scale = s.do_scale;
  p.do_sqrt = s.do_sqrt;
  p.sqrt_f = 1.0f;
  if (s.do_sqrt) {
    uint32_t cnt = a.row_off ? a.row_off[orow + 1] - a.row_off[orow] : 1u;
    p.sqrt_f = __fdiv_rn(1.0f, __fsqrt_rn((float)cnt));
  }
  return p;
}

// N consecutive gradient elements of one output row starting at element e0, converted to f32 and clamped
template <int N, bool F16>
__device__ __forceinline__ void load_grad_elems(float (&g)[N], const void* gbase, size_t row_elem0, uint32_t e0) {
  if (F16) {
    const __half* gp = reinterpret_cast<const __half*>(gbase) + row_elem0 + e0;
    if (N % 4 == 0) {
#pragma unroll
      for (int q = 0; q < N / 4; ++q) {
        uint2 raw = *reinterpret_cast<const uint2*>(gp + 4 * q);
        // +-inf -> +-65504 (persia-common lib.rs:163-180), two halves per instruction; finite halves are inside already
        const __half2 lim = __floats2half2_rn(65504.0f, 65504.0f);
        __half2 h0 = __hmin2(__hmax2(*reinterpret_cast<__half2*>(&raw.x), __hneg2(lim)), lim);
        __half2 h1 = __hmin2(__hmax2(*reinterpret_cast<__half2*>(&raw.y), __hneg2(lim)), lim);
        float2 x = __half22float2(h0), y = __half22float2(h1);
        g[4 * q] = x.x; g[4 * q + 1] = x.y; g[4 * q + 2] = y.x; g[4 * q + 3] = y.y;
      }
    } else {
#pragma unroll
      for (int q = 0; q < N; ++q) g[q] = clamp_f16(__half2float(gp[q]));
    }
  } else {
    const float* gp = reinterpret_cast<const float*>(gbase) + row_elem0 + e0;
    if (N % 4 == 0) {
#pragma unroll
      for (int q = 0; q < N / 4; ++q) {
        float4 x = *reinterpret_cast<const float4*>(gp + 4 * q);
        g[4 * q] = x.x; g[4 * q + 1] = x.y; g[4 * q + 2] = x.z; g[4 * q + 3] = x.w;
      }
    } else {
#pragma unroll
      for (int q = 0; q < N; ++q) g[q] = gp[q];
    }
  }
}

template <int N>
__device__ __forceinline__ void add_prepared(float (&acc)[N], const float (&g)[N], const GradPrep& p, bool plain) {
  if (plain) {
#pragma unroll
    for (int q = 0; q < N; ++q) acc[q] = __fadd_rn(acc[q], g[q]);
  } else {
#pragma unroll
    for (int q = 0; q < N; ++q) acc[q] = __fadd_rn(acc[q], p(g[q]));
  }
}

// sum of the gradients of occurrences pos(0..cnt-1) (already in ascending order), elements [e0, e0+N).
// Batches of 8 / 4 occurrences have all their loads issued together; the adds stay sequential.
template <int N, bool F16, typename POS>
__device__ __forceinline__ void reduce_sorted(float (&acc)[N], const ItemSrc& s, const ReduceArgs& a, const TableDev& t,
                                              uint32_t cnt, uint32_t e0, POS pos) {
#pragma unroll
  for (int q = 0; q < N; ++q) acc[q] = 0.0f;
  uint32_t k = 0;
  for (; k + 8 <= cnt; k += 8) {
    uint32_t orow[8];
    float g[8][N];
#pragma unroll
    for (int u = 0; u < 8; ++u) orow[u] = occ_out_row(a, pos(k + u));
#pragma unroll
    for (int u = 0; u < 8; ++u) load_grad_elems<N, F16>(g[u], s.gbase, (size_t)(orow[u] - s.slot_row0) * t.dim, e0);
#pragma unroll
    for (int u = 0; u < 8; ++u) add_prepared<N>(acc, g[u], grad_prep(s, a, orow[u]), s.plain);
  }
  if (k + 4 <= cnt) {
    uint32_t orow[4];
    float g[4][N];
#pragma unroll
    for (int u = 0; u < 4; ++u) orow[u] = occ_out_row(a, pos(k + u));
#pragma unroll
    for (int u = 0; u < 4; ++u) load_grad_elems<N, F16>(g[u], s.gbase, (size_t)(orow[u] - s.slot_row0) * t.dim, e0);
#pragma unroll
    for (int u = 0; u < 4; ++u) add_prepared<N>(acc, g[u], grad_prep(s, a, orow[u]), s.plain);
    k += 4;
  }
  for (; k < cnt; ++k) {
    const uint32_t orow = occ_out_row(a, pos(k));
    float g[N];
    load_grad_elems<N, F16>(g, s.gbase, (size_t)(orow - s.slot_row0) * t.dim, e0);
    add_prepared<N>(acc, g, grad_prep(s, a, orow), s.plain);
  }
}

// sharded requester: where the reduced gradient of the item with target = owner * cap + k goes (the owner's receive
// area, slot [this rank][k]) and its apply / skip word
__device__ __forceinline__ float* send_grad_ptr(const XchgDev& x, uint32_t target, uint32_t dim) {
  const uint32_t q = target / x.cap, k = target % x.cap;
  return reinterpret_cast<float*>(x.base[q] + x.off_grad) + ((size_t)x.rank * x.cap + k) * dim;
}
__device__ __forceinline__ uint32_t* send_gok_ptr(const XchgDev& x, uint32_t target) {
  const uint32_t q = target / x.cap, k = target % x.cap;
  return reinterpret_cast<uint32_t*>(x.base[q] + x.off_gok) + ((size_t)x.rank * x.cap + k);
}

// slots whose gradient is skipped or holds a NaN (mod.rs:731-746), or that this launch does not step, as a bit mask.
// with_nan = false: only what the host knows (no gradient, not this round) — the NaN verdict is not read, so the kernel
// need not wait for the scan.
__device__ __forceinline__ void build_dead_mask(uint32_t* dead, const GradsDev& gr, const ReduceArgs& a, uint32_t n_slots,
                                                bool with_nan = true) {
  if (threadIdx.x < PB_MAX_SLOTS / 32) dead[threadIdx.x] = 0u;
  __syncthreads();
  const uint32_t tick = with_nan ? *a.tick_ptr : 0u;
  for (uint32_t s = threadIdx.x; s < PB_MAX_SLOTS; s += blockDim.x) {
    const bool off = s >= n_slots || !gr.ptr[s] || (with_nan && a.nan_tick[s] == tick) ||
                     !((a.round_mask[s >> 5] >> (s & 31)) & 1u);
    if (off) atomicOr(&dead[s >> 5], 1u << (s & 31));
  }
  __syncthreads();
}
__device__ __forceinline__ bool slot_dead(const uint32_t* dead, uint32_t slot) { return (dead[slot >> 5] >> (slot & 31)) & 1u; }

// ------------------------------------------------------------------------------------------------
// cold and warm items
// ------------------------------------------------------------------------------------------------
// one item through the generic path: sorted occurrence list pos(0..cnt-1)
// sharded requester: the reduced gradient of one item goes to its owner (update_all_batched_gradients ends with one
// (signs, gradients) request per parameter server, mod.rs:813-857)
template <int VEC, bool F16, typename POS>
__device__ __forceinline__ void send_item(const TableDev& t, const SlotsDev& sl, const GradsDev& gr, const ReduceArgs& a,
                                          uint32_t target, uint32_t slot, uint32_t cnt, uint32_t lane, uint32_t G, POS pos) {
  float* dst = send_grad_ptr(a.x, target, t.dim);
  const uint32_t nvec = t.dim / VEC;
  const ItemSrc src = item_src(sl, gr, a, slot);
  for (uint32_t c = lane; c < nvec; c += G) {
    float acc[VEC];
    reduce_sorted<VEC, F16>(acc, src, a, t, cnt, c * VEC, pos);
    store_vec<VEC>(dst + c * VEC, acc);
  }
  if (lane == 0) *send_gok_ptr(a.x, target) = 1u;
}

template <int VEC, bool F16, int KIND, typename POS>
__device__ __forceinline__ void step_item(const TableDev& t, const OptimDev& op, const HyperDev& hy, const SlotsDev& sl,
                                          const GradsDev& gr, const ReduceArgs& a, uint32_t row, uint32_t slot,
                                          uint32_t cnt, uint32_t lane, uint32_t G, uint32_t gmask, float* stage, POS pos) {
  float* prow = t.rows + (size_t)row * t.stride;
  const uint32_t nvec = t.dim / VEC;
  const ItemSrc src = item_src(sl, gr, a, slot);
  const StepCtx sc = step_ctx(prow, t, op, gr, slot);
  for (uint32_t c = lane; c < nvec; c += G) {
    RowElems<KIND, VEC> rc;
    rc.load(prow, c * VEC, t, op);  // in flight while the gradients are fetched and summed
    float acc[VEC];
    reduce_sorted<VEC, F16>(acc, src, a, t, cnt, c * VEC, pos);
    if (KIND == PB_OPT_ADAGRAD_VW) store_vec<VEC>(stage + c * VEC, acc);
    rc.step(c * VEC, acc, t, op, hy, sc);
    rc.store(prow, c * VEC, t, op);
  }
  if (KIND == PB_OPT_ADAGRAD_VW) {  // state = state*mom + dot(g,g)/dim (optim.rs:280-283)
    __syncwarp(gmask);              // the staged gradient of every lane of the group is visible to lane 0
    if (lane == 0) {
      float gs = __fdiv_rn(vw_dot(stage, t.dim), (float)t.dim);
      prow[t.dim] = __fadd_rn(__fmul_rn(sc.vw_state, op.mom), gs);
    }
    __syncwarp(gmask);
  }
}

// ---- warm items: one lane group per item; the group sorts the item's <= 32 occurrences (rank by counting), then adds
// them in order.  Items are assigned statically (a shared work counter would be thousands of same-address atomics).
template <int VEC, bool F16, int KIND, bool SEND>
__global__ void __launch_bounds__(256, 3) k_reduce_warm(TableDev t, OptimDev op, HyperDev hy, SlotsDev sl, GradsDev gr,
                                                     ReduceArgs a, uint32_t G) {
  __shared__ uint32_t dead[PB_MAX_SLOTS / 32];
  __shared__ uint32_t sortbuf[64][2 * PB_WARM_MAX];  // per lane group (G >= 4): unsorted | sorted occurrences
  const uint32_t n_warm = a.b.cnt[BC_WARM], n_cold = a.b.cnt[BC_COLD];
  if (blockIdx.x * (blockDim.x / G) >= n_warm) return;  // whole block
  build_dead_mask(dead, gr, a, sl.n_slots);
  const uint32_t lane = threadIdx.x % G, grp = threadIdx.x / G, wl = threadIdx.x & 31;
  const uint32_t gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (wl / G * G));
  uint32_t* raw = sortbuf[grp];
  uint32_t* srt = raw + PB_WARM_MAX;
  // the grid holds a few blocks per SM; a group strides over the list (its length lives on the device)
  for (uint32_t w = blockIdx.x * (blockDim.x / G) + grp; w < n_warm; w += gridDim.x * (blockDim.x / G)) {
    __syncwarp(gmask);  // the previous item's sorted list is no longer read
    const uint4 d = a.b.warm[w];
    const uint32_t row = d.x, base = d.y, cnt = d.z;
    for (uint32_t l = lane; l < cnt; l += G) raw[l] = a.b.seg_occ[base + l];
    __syncwarp(gmask);
    for (uint32_t l = lane; l < cnt; l += G) {  // occurrences are distinct numbers
      const uint32_t p = raw[l];
      uint32_t r = 0;
      for (uint32_t m = 0; m < cnt; ++m) r += raw[m] < p;
      srt[r] = p;
    }
    __syncwarp(gmask);
    const uint32_t slot = slot_of_occ(sl, srt[0]);
    if (SEND) {
      if (row == ROW_NONE) continue;  // the item found no room in its owner's segment (flagged in k_route_items)
      if (slot_dead(dead, slot)) {
        if (lane == 0) *send_gok_ptr(a.x, row) = 0u;
      } else {
        send_item<VEC, F16>(t, sl, gr, a, row, slot, cnt, lane, G, [&](uint32_t k) { return srt[k]; });
      }
      continue;
    }
    if (slot_dead(dead, slot)) continue;
    if (row >= t.capacity) {
      if (lane == 0 && !a.quiet_miss) atomicAdd(&t.counters[CTR_GRAD_MISS], 1u);  // gradient_id_miss_count (PS mod.rs:401-403)
      continue;
    }
    float* stage = a.vw_stage ? a.vw_stage + (size_t)(n_cold + w) * t.dim : nullptr;
    step_item<VEC, F16, KIND>(t, op, hy, sl, gr, a, row, slot, cnt, lane, G, gmask, stage, [&](uint32_t k) { return srt[k]; });
  }
}

// ---- cold items (one occurrence — the majority): nothing to reduce.  One lane group per item, nothing but two
// independent loads (row, gradient), the step and the store; light on registers so that the whole chip's worth of
// groups is resident and the loads of many rows are in flight.
template <int VEC, bool F16, int KIND, bool SEND>
__global__ void __launch_bounds__(256) k_reduce_cold(TableDev t, OptimDev op, HyperDev hy, SlotsDev sl, GradsDev gr,
                                                     ReduceArgs a, uint32_t G) {
  __shared__ uint32_t dead[PB_MAX_SLOTS / 32];
  const uint32_t n_cold = a.b.cnt[BC_COLD];
  if (blockIdx.x * (blockDim.x / G) >= n_cold) return;  // whole block
  build_dead_mask(dead, gr, a, sl.n_slots);
  const uint32_t lane = threadIdx.x % G, wl = threadIdx.x & 31;
  const uint32_t gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (wl / G * G));
  const uint32_t nvec = t.dim / VEC;
  // the grid holds a few blocks per SM; a group strides over the list (its length lives on the device)
  for (uint32_t w = blockIdx.x * (blockDim.x / G) + threadIdx.x / G; w < n_cold; w += gridDim.x * (blockDim.x / G)) {
    const uint2 d = a.b.cold[w];
    const uint32_t slot = slot_of_occ(sl, d.y);
    const ItemSrc src = item_src(sl, gr, a, slot);
    const uint32_t orow = occ_out_row(a, d.y);
    const GradPrep prep = grad_prep(src, a, orow);
    const size_t gelem = (size_t)(orow - src.slot_row0) * t.dim;
    if (SEND) {
      if (d.x == ROW_NONE) continue;
      const bool off = slot_dead(dead, slot);
      if (lane == 0) *send_gok_ptr(a.x, d.x) = off ? 0u : 1u;
      if (off) continue;
      float* dst = send_grad_ptr(a.x, d.x, t.dim);
      for (uint32_t c = lane; c < nvec; c += G) {
        float g[VEC], acc[VEC];
        load_grad_elems<VEC, F16>(g, src.gbase, gelem, c * VEC);
#pragma unroll
        for (int q = 0; q < VEC; ++q) acc[q] = 0.0f;
        add_prepared<VEC>(acc, g, prep, src.plain);
        store_vec<VEC>(dst + c * VEC, acc);
      }
      continue;
    }
    if (slot_dead(dead, slot)) continue;
    if (d.x >= t.capacity) {
      if (lane == 0 && !a.quiet_miss) atomicAdd(&t.counters[CTR_GRAD_MISS], 1u);
      continue;
    }
    if (KIND == PB_OPT_ADAGRAD_VW) {  // needs the whole reduced gradient staged for the dot
      const uint32_t occ = d.y;
      step_item<VEC, F16, KIND>(t, op, hy, sl, gr, a, d.x, slot, 1u, lane, G, gmask, a.vw_stage + (size_t)w * t.dim,
                                [&](uint32_t) { return occ; });
      continue;
    }
    float* prow = t.rows + (size_t)d.x * t.stride;
    StepCtx sc;
    sc.vw_state = sc.r1 = sc.r2 = 0.0f;
    if (KIND == PB_OPT_ADAM) sc = step_ctx(prow, t, op, gr, slot);
    for (uint32_t c = lane; c < nvec; c += G) {
      RowElems<KIND, VEC> rc;
      float g[VEC], acc[VEC];
      rc.load(prow, c * VEC, t, op);
      load_grad_elems<VEC, F16>(g, src.gbase, gelem, c * VEC);
#pragma unroll
      for (int q = 0; q < VEC; ++q) acc[q] = 0.0f;  // the reference adds into a zeroed row (-0 -> +0)
      add_prepared<VEC>(acc, g, prep, src.plain);
      rc.step(c * VEC, acc, t, op, hy, sc);
      rc.store(prow, c * VEC, t, op);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// hot items: counting-sort order, then producer warps -> shared-memory ring of PREPARED rows -> chain warp(s)
//
// A strictly sequential f32 sum costs one dependent FADD per row and element whatever else happens (measured: 6.6
// cycles per row for a warp that does nothing but LDS + FADD, scripts/ubench/hot_ubench.cu); the head of the Zipf curve
// and the signs of a tiny slot have thousands of rows.  A lone warp sustains only an instruction every ~2 cycles, so
// everything that is not that FADD is taken off the chain and spread over the block's other warps:
//   order      The forward already set one bit per occurrence in the item's bitmap over its slot's samples (hot_bits,
//              k_gather_items) — a counting sort that costs B/32 words.  Here the words are loaded (and zeroed for the
//              next batch), prefix-summed and expanded into the ascending list of sample numbers in shared memory.
//              (Items that found no room in the bitmap pool come with an unsorted occurrence list and set the bits here.)
//   producers  (HOT_WARPS - CH warps) take chunks of R consecutive occurrences round robin: 16-byte loads of the
//              gradient rows straight from global memory, eight in flight per lane, then the EW's value preparation
//              (f16 -> f32 with +-inf clamped, 1/scale, sqrt factor; mod.rs:751-778) and the f32 values go to the
//              chunk's ring slot; every lane arrives on the slot's `full` mbarrier.  The common case (one id per
//              sample, no scaling) has its own lean loop: ~25 instructions per 16 bytes is what bounds a producer.
//   chain      (CH warps, 32 * EPL columns each) waits for the slot and adds its rows in order: one LDS and EPL
//              dependent FADDs per row — nothing else — then arrives on `empty`; finally it stores the sum to the item's
//              row of the hot stage (k_step_hot steps it once the NaN verdict is known) or, sharded, to the owner.
// Measured alternatives (profiles/r2_hot_ubench_*.txt): cp.async.bulk of the rows into a raw ring + converter warps is
// bound by the copy engine's issue rate (~60 cycles per 128-byte copy and SM), a single warp doing load + convert + add
// by the instruction stream (~40 cycles per row).
// ------------------------------------------------------------------------------------------------
constexpr uint32_t HOT_WIN = 8192;   // samples per bitmap window
constexpr uint32_t HOT_WORDS = HOT_WIN / 32;
constexpr uint32_t HOT_THREADS = 256;
constexpr uint32_t HOT_WARPS = HOT_THREADS / 32;
constexpr uint32_t HOT_MAX_SLOTS = 8;      // ring slots
constexpr uint32_t HOT_COLS = 512;         // columns per pass (4 chain warps x 128)
constexpr uint32_t WAIT_SPINS = 1u << 22;  // bounded waits: a lost completion voids the batch (CTR_ERR) instead of hanging the GPU

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t spins = 0; spins < WAIT_SPINS; ++spins) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return true;
  }
  return false;
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long now;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
  return now;
}
// non-blocking: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}

// +-inf -> +-65504 (persia-common lib.rs:163-180), two halves per instruction; finite halves are inside already
__device__ __forceinline__ __half2 clamp_h2(__half2 v) {
  const __half2 lim = __floats2half2_rn(65504.0f, 65504.0f);
  return __hmin2(__hmax2(v, __hneg2(lim)), lim);
}

struct HotGeom {
  uint32_t cols;      // columns of this pass
  uint32_t stride;    // floats per ring row (cols rounded up to 4)
  uint32_t R;         // rows per ring slot (chunk): one or two halves of R1 rows
  uint32_t R1;        // rows a producer prepares at a time (its lanes describe them: <= 32)
  uint32_t S;         // ring slots
  uint32_t rowbytes;  // bytes of a gradient row
  uint32_t lean;      // the producers' lean loop applies (16-byte vectors, power-of-two vectors per row <= 32)
  uint32_t CH;        // chain warps
  uint32_t vec;       // producer mode: 1 = 16-byte loads (8 halves / 4 floats), 0 = element by element
  uint32_t vshift;    // log2(vectors per row) when that is a power of two, else 32
};

// one chunk: rows k0 .. k0+nv-1 of the sorted list, columns [col0, col0+cols) -> prepared f32 in the ring slot.
// Vector mode: R * (vectors per row) <= 256, i.e. at most eight 16-byte loads per lane, all issued before the first
// conversion; vector v = j * 32 + lane of the chunk is row v / nvr, vector v % nvr of the row (POW2: by shift and
// mask).  Rows nv .. the next multiple of four are written as zeros: the chain adds whole groups of four rows, and
// x + (+0) = x for every x the accumulator can hold (it starts at +0, so it is never -0).
template <bool F16, bool POW2>
__device__ __forceinline__ void produce_vec(float* slot, const HotGeom& g, const ItemSrc& src, uint32_t my_row, float my_f,
                                            uint32_t nv, uint32_t col0, uint32_t dim, uint32_t lane) {
  constexpr uint32_t EV = F16 ? 8u : 4u;  // elements per 16-byte vector
  const unsigned char* gcol = reinterpret_cast<const unsigned char*>(src.gbase) + (size_t)col0 * (F16 ? 2u : 4u);
  const uint32_t rowbytes = dim * (F16 ? 2u : 4u);
  const uint32_t nvr = g.cols / EV, total = g.R1 * nvr, nv4 = (nv + 3u) & ~3u;
  uint4 raw[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t v = (uint32_t)j * 32u + lane;
    const uint32_t r = POW2 ? v >> g.vshift : v / nvr, c = POW2 ? v & (nvr - 1u) : v % nvr;
    const uint32_t grow = __shfl_sync(0xffffffffu, my_row, r & 31u);
    raw[j] = make_uint4(0u, 0u, 0u, 0u);
    if (v < total && r < nv) raw[j] = __ldg(reinterpret_cast<const uint4*>(gcol + (size_t)grow * rowbytes + c * 16u));
  }
  const bool prep = src.do_scale || src.do_sqrt;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t v = (uint32_t)j * 32u + lane;
    const uint32_t r = POW2 ? v >> g.vshift : v / nvr, c = POW2 ? v & (nvr - 1u) : v % nvr;
    float f = 1.0f;
    if (prep) f = __shfl_sync(0xffffffffu, my_f, r & 31u);
    if (v >= total || r >= nv4) continue;
    float x[EV];
    if constexpr (F16) {
      const __half2* h = reinterpret_cast<const __half2*>(&raw[j]);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float2 y = __half22float2(clamp_h2(h[q]));
        x[2 * q] = y.x;
        x[2 * q + 1] = y.y;
      }
    } else {
      x[0] = __uint_as_float(raw[j].x); x[1] = __uint_as_float(raw[j].y);
      x[2] = __uint_as_float(raw[j].z); x[3] = __uint_as_float(raw[j].w);
    }
    if (prep) {
      if (src.do_scale) {
#pragma unroll
        for (uint32_t q = 0; q < EV; ++q) x[q] = __fmul_rn(x[q], src.inv_scale);
      }
      if (src.do_sqrt) {
#pragma unroll
        for (uint32_t q = 0; q < EV; ++q) x[q] = __fmul_rn(x[q], f);
      }
    }
    float4* dst = reinterpret_cast<float4*>(slot + (size_t)r * g.stride + c * EV);
    dst[0] = make_float4(x[0], x[1], x[2], x[3]);
    if constexpr (F16) dst[1] = make_float4(x[4], x[5], x[6], x[7]);
  }
}

template <bool F16>
__device__ __forceinline__ void produce_chunk(float* slot, const HotGeom& g, const ItemSrc& src, const ReduceArgs& a,
                                              const uint16_t* sorted, uint32_t k0, uint32_t nv, uint32_t wbase,
                                              uint32_t col0, uint32_t dim, uint32_t lane) {
  // per row of the chunk (lane = row): gradient row number and the sample's sqrt factor
  uint32_t my_row = 0;
  float my_f = 0.0f;  // (zero rows stay zero)
  if (lane < nv) {
    const uint32_t orow = occ_out_row(a, wbase + sorted[k0 + lane]);
    my_row = orow - src.slot_row0;
    my_f = src.do_sqrt ? grad_prep(src, a, orow).sqrt_f : 1.0f;
  }
  if (g.vec) {
    if (g.vshift < 32u) produce_vec<F16, true>(slot, g, src, my_row, my_f, nv, col0, dim, lane);
    else produce_vec<F16, false>(slot, g, src, my_row, my_f, nv, col0, dim, lane);
  } else {
    const unsigned char* gbytes = reinterpret_cast<const unsigned char*>(src.gbase);
    const uint32_t nv4 = min(g.R1, (nv + 3u) & ~3u), total = nv4 * g.cols;
    for (uint32_t i0 = 0; i0 < total; i0 += 32u) {  // uniform trip count: the shuffles are warp-wide
      const uint32_t i = i0 + lane;
      const bool ok = i < total;
      const uint32_t r = ok ? i / g.cols : 0u, c = ok ? i % g.cols : 0u;
      const uint32_t grow = __shfl_sync(0xffffffffu, my_row, r);
      const float f = __shfl_sync(0xffffffffu, my_f, r);
      if (!ok) continue;
      float x = 0.0f;
      if (r < nv) {
        const size_t e = (size_t)grow * dim + col0 + c;
        x = F16 ? clamp_f16(__half2float(reinterpret_cast<const __half*>(gbytes)[e])) : reinterpret_cast<const float*>(gbytes)[e];
        if (src.do_scale) x = __fmul_rn(x, src.inv_scale);
        if (src.do_sqrt) x = __fmul_rn(x, f);
      }
      slot[(size_t)r * g.stride + c] = x;
    }
  }
}

// the producers' lean loop: one id per sample (the gradient row of sample b is row b), no scaling.  Vector j of a lane is
// row (j * 32 + lane) >> vshift of the chunk, 16-byte vector (j * 32 + lane) & (nvr - 1) of the row; the row number comes
// straight from the sorted list.  Rows nv .. the next multiple of four are written as zeros (see produce_vec).  Split in
// two so that a producer has its NEXT chunk's loads in flight while it converts this one.
__device__ __forceinline__ void lean_load(uint4 (&raw)[8], const HotGeom& g, const unsigned char* gcol0, const uint16_t* sorted,
                                          uint32_t nv, uint32_t lane) {
  const uint32_t nvr_mask = (1u << g.vshift) - 1u;
  const uint32_t r0 = lane >> g.vshift, rstep = 32u >> g.vshift;
  const unsigned char* gc = gcol0 + (lane & nvr_mask) * 16u;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t r = (uint32_t)j * rstep + r0;
    raw[j] = make_uint4(0u, 0u, 0u, 0u);
    if (r < nv) raw[j] = __ldg(reinterpret_cast<const uint4*>(gc + (size_t)sorted[r] * g.rowbytes));
  }
}
template <bool F16>
__device__ __forceinline__ void lean_store(float* slot, const uint4 (&raw)[8], const HotGeom& g, uint32_t nv, uint32_t lane) {
  constexpr uint32_t EV = F16 ? 8u : 4u;
  const uint32_t nvr_mask = (1u << g.vshift) - 1u, nv4 = (nv + 3u) & ~3u;
  const uint32_t r0 = lane >> g.vshift, rstep = 32u >> g.vshift;
  float* sc = slot + (lane & nvr_mask) * EV;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t r = (uint32_t)j * rstep + r0;
    if (r >= nv4) continue;  // (r grows with j: past the chunk's rows)
    float4* dst = reinterpret_cast<float4*>(sc + (size_t)r * g.stride);
    if constexpr (F16) {
      const __half2* h = reinterpret_cast<const __half2*>(&raw[j]);
      const float2 y0 = __half22float2(clamp_h2(h[0])), y1 = __half22float2(clamp_h2(h[1]));
      const float2 y2 = __half22float2(clamp_h2(h[2])), y3 = __half22float2(clamp_h2(h[3]));
      dst[0] = make_float4(y0.x, y0.y, y1.x, y1.y);
      dst[1] = make_float4(y2.x, y2.y, y3.x, y3.y);
    } else {
      dst[0] = make_float4(__uint_as_float(raw[j].x), __uint_as_float(raw[j].y), __uint_as_float(raw[j].z), __uint_as_float(raw[j].w));
    }
  }
}

// the chain's straight-line block: RB rows loaded, then added in order.  (A loop with the loads and adds of different
// groups interleaved under branches measured 18 cycles per row, this 6.6: the compiler must see the loads far ahead.)
template <int EPL, int RB>
__device__ __forceinline__ void chain_block(float (&acc)[EPL], const float* rp, uint32_t stride) {
  float v[RB][EPL];
#pragma unroll
  for (int u = 0; u < RB; ++u) RowElems<-1, EPL>::template ld<EPL>(rp + (size_t)u * stride, v[u]);
#pragma unroll
  for (int u = 0; u < RB; ++u) {
#pragma unroll
    for (int q = 0; q < EPL; ++q) acc[q] = __fadd_rn(acc[q], v[u][q]);
  }
}

// entry of `hot` of the h-th hot item in reduce order: the giants, the huge ones (both listed from the list's end), the rest
__device__ __forceinline__ uint32_t hot_entry(const BatchDev& b, uint32_t h, uint32_t n_giant, uint32_t n_huge) {
  return h < n_giant ? b.hot_cap - 1u - h
                     : (h < n_giant + n_huge ? b.hot_cap - 1u - b.giant_cap - (h - n_giant) : h - n_giant - n_huge);
}

template <int EPL, bool F16, bool SEND>
__global__ void __launch_bounds__(HOT_THREADS, 1) k_reduce_hot(TableDev t, SlotsDev sl, GradsDev gr, ReduceArgs a, HotGeom geo,
                                                              unsigned long long* trace) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint32_t dead[PB_MAX_SLOTS / 32];
  __shared__ uint32_t s_item, s_nwin;
  __shared__ uint32_t bitmap[HOT_WORDS], wpre[HOT_WORDS];
  __shared__ uint16_t sorted[HOT_WIN];
  __shared__ __align__(8) uint64_t bars[2 * HOT_MAX_SLOTS];  // full[0..8), empty[8..16)
  float* ring = reinterpret_cast<float*>(smem_raw);                     // [S][R][stride] prepared rows
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // PW producers share S slots: PW <= S keeps a producer from running two rounds ahead of the chain (the parity of a
  // slot's barrier only tells odd rounds from even ones)
  const uint32_t CH = geo.CH, PW = min(HOT_WARPS - CH, geo.S);
  if (tid == 0) {
    for (uint32_t s = 0; s < HOT_MAX_SLOTS; ++s) {
      mbar_init(smem_u32(bars + s), 32u);                       // every lane of the producing warp
      mbar_init(smem_u32(bars + HOT_MAX_SLOTS + s), 32u * CH);  // every lane of every chain warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // sending: the owner is told whether to apply, which needs the NaN verdict; staging: k_step_hot decides
  build_dead_mask(dead, gr, a, sl.n_slots, SEND);  // ends with __syncthreads
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + HOT_MAX_SLOTS);
  const uint32_t n_giant = a.b.cnt[BC_GIANT], n_huge = a.b.cnt[BC_HUGE];  // the longest chains first
  const uint32_t n_hot = a.b.cnt[BC_HOT] + n_huge + n_giant;
  uint32_t* next = a.b.cnt + BC_NEXT + PB_MAX_SLOTS + a.round;
  const uint32_t n_pass = (t.dim + HOT_COLS - 1u) / HOT_COLS;
  uint32_t it = 0;  // ring chunks so far: producers and chain count the same chunks
  bool failed = false;
  for (;;) {
    __syncthreads();  // s_item, bitmap and sorted are free again
    if (tid == 0) s_item = atomicAdd(next, 1u);
    __syncthreads();
    const uint32_t h = s_item;
    if (h >= n_hot) break;
    if (trace && tid == 0) trace[8 * h] = globaltimer_ns();
    const uint32_t entry = hot_entry(a.b, h, n_giant, n_huge);
    const uint4 d = a.b.hot[entry];
    const uint32_t row = d.x, cnt = d.z, slot = d.w;
    const bool bm_mode = d.y >> 31;
    const uint32_t base = d.y & 0x7FFFFFFFu;  // first bitmap word of the item, or first entry of its occurrence list
    const uint32_t lo = sl.occ_off[slot], hi = sl.occ_off[slot + 1];
    bool skip = false;
    if (SEND) {
      skip = row == ROW_NONE || slot_dead(dead, slot);
      if (row != ROW_NONE && tid == 0) *send_gok_ptr(a.x, row) = slot_dead(dead, slot) ? 0u : 1u;
    } else {
      skip = slot_dead(dead, slot) || row >= t.capacity;  // (k_step_hot counts the miss)
    }
    if (skip) {  // the item's bits must still go back to zero for the next batch
      if (bm_mode)
        for (uint32_t w = tid; w < (hi - lo + 31u) / 32u; w += HOT_THREADS) a.b.hot_bits[base + w] = 0u;
      continue;
    }
    const ItemSrc src = item_src(sl, gr, a, slot);
    float* dst = SEND ? send_grad_ptr(a.x, row, t.dim) : a.hot_stage + (size_t)entry * a.hot_stride;
    for (uint32_t pass = 0; pass < n_pass; ++pass) {
      const uint32_t col0 = pass * HOT_COLS;
      HotGeom g = geo;
      g.cols = min(geo.cols, t.dim - col0);
      if (g.cols != geo.cols) g.vec = g.lean = 0;  // a short last column block goes element by element
      const bool lean = g.lean && src.plain;
      const uint32_t e0 = col0 + (warp * 32u + lane) * EPL;  // chain lanes: EPL columns each
      const bool own = warp < CH && e0 < t.dim;
      float acc[EPL];
#pragma unroll
      for (int q = 0; q < EPL; ++q) acc[q] = 0.0f;
      for (uint32_t wbase = lo; wbase < hi; wbase += HOT_WIN) {
        const uint32_t wend = min(hi, wbase + HOT_WIN);
        const uint32_t n_words = (wend - wbase + 31u) / 32u;
        // ---- the item's occurrences inside this window, ascending
        if (bm_mode) {
          uint32_t* gw = a.b.hot_bits + base + (wbase - lo) / 32u;
          for (uint32_t w = tid; w < HOT_WORDS; w += HOT_THREADS) {
            bitmap[w] = w < n_words ? gw[w] : 0u;
            if (w < n_words && pass + 1 == n_pass) gw[w] = 0u;  // all zero again for the next batch
          }
        } else {
          for (uint32_t w = tid; w < HOT_WORDS; w += HOT_THREADS) bitmap[w] = 0u;
          __syncthreads();
          for (uint32_t k0 = tid; k0 < cnt; k0 += 4 * HOT_THREADS) {  // four loads in flight per thread
            uint32_t p[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) p[u] = k0 + u * HOT_THREADS < cnt ? a.b.seg_occ[base + k0 + u * HOT_THREADS] : 0xFFFFFFFFu;
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (p[u] >= wbase && p[u] < wend) atomicOr(&bitmap[(p[u] - wbase) >> 5], 1u << ((p[u] - wbase) & 31u));
          }
        }
        __syncthreads();
        if (warp == 0) {  // exclusive prefix of the word popcounts: HOT_WORDS / 32 words per lane
          uint32_t c[HOT_WORDS / 32], sum = 0;
#pragma unroll
          for (uint32_t j = 0; j < HOT_WORDS / 32; ++j) {
            c[j] = sum;
            sum += __popc(bitmap[lane * (HOT_WORDS / 32) + j]);
          }
          uint32_t inc = sum;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= (uint32_t)o) inc += y;
          }
#pragma unroll
          for (uint32_t j = 0; j < HOT_WORDS / 32; ++j) wpre[lane * (HOT_WORDS / 32) + j] = inc - sum + c[j];
          if (lane == 31) s_nwin = inc;
        }
        __syncthreads();
        for (uint32_t w = tid; w < HOT_WORDS; w += HOT_THREADS) {
          uint32_t m = bitmap[w], at = wpre[w];
          while (m) {
            sorted[at++] = (uint16_t)(w * 32u + __ffs(m) - 1u);
            m &= m - 1u;
          }
        }
        __syncthreads();
        const uint32_t nwin = s_nwin;
        const uint32_t n_chunks = (nwin + g.R - 1u) / g.R;
        if (trace && tid == 0) trace[8 * h + 1] = globaltimer_ns();
        if (warp >= CH) {
          // ---- producers: chunk c belongs to warp CH + (it % PW)
          const uint32_t me = warp - CH;
          // lean: gradient row of sample b of the slot is row b (+ the window's offset inside the slot)
          const unsigned char* gcol0 = reinterpret_cast<const unsigned char*>(src.gbase) +
                                       ((size_t)(wbase - src.slot_row0) * t.dim + col0) * (F16 ? 2u : 4u);
          // a chunk is one or two halves of R1 rows; a producer has both halves' loads in flight before it converts
          for (uint32_t c = me < PW ? (me + PW - it % PW) % PW : n_chunks; c < n_chunks; c += PW) {  // (warps past PW idle)
            const uint32_t i = it + c, stage = i % g.S, par = (i / g.S) & 1u;
            const uint32_t nv = min(g.R, nwin - c * g.R);
            float* slotp = ring + (size_t)stage * g.R * g.stride;
            const uint16_t* srt = sorted + c * g.R;
            if (lean) {
              // the chunk's parts of R1 rows ping-pong between two register sets: part k + 2 is loaded as soon as part k has
              // been converted, so two parts' loads are always in flight
              uint4 ra[8], rb[8];
              const uint32_t np = (nv + g.R1 - 1u) / g.R1;  // parts of this chunk (<= 4)
              lean_load(ra, g, gcol0, srt, min(g.R1, nv), lane);
              if (np > 1) lean_load(rb, g, gcol0, srt + g.R1, min(g.R1, nv - g.R1), lane);
              if (!failed && !mbar_wait(empty0 + 8u * stage, par ^ 1u)) failed = true;
              lean_store<F16>(slotp, ra, g, min(g.R1, nv), lane);
              if (np > 2) lean_load(ra, g, gcol0, srt + 2u * g.R1, min(g.R1, nv - 2u * g.R1), lane);
              if (np > 1) lean_store<F16>(slotp + (size_t)g.R1 * g.stride, rb, g, min(g.R1, nv - g.R1), lane);
              if (np > 3) lean_load(rb, g, gcol0, srt + 3u * g.R1, min(g.R1, nv - 3u * g.R1), lane);
              if (np > 2) lean_store<F16>(slotp + (size_t)2u * g.R1 * g.stride, ra, g, min(g.R1, nv - 2u * g.R1), lane);
              if (np > 3) lean_store<F16>(slotp + (size_t)3u * g.R1 * g.stride, rb, g, min(g.R1, nv - 3u * g.R1), lane);
            } else {
              if (!failed && !mbar_wait(empty0 + 8u * stage, par ^ 1u)) failed = true;
              for (uint32_t r0 = 0; r0 < nv; r0 += g.R1)
                produce_chunk<F16>(slotp + (size_t)r0 * g.stride, g, src, a, sorted, c * g.R + r0, min(g.R1, nv - r0), wbase, col0, t.dim, lane);
            }
            mbar_arrive(full0 + 8u * stage);
          }
        } else if (n_chunks) {
          // ---- chain: the rows in ascending order, one dependent add per row and element
          long long tw = 0, ta = 0;
          for (uint32_t c = 0; c < n_chunks; ++c) {
            const uint32_t i = it + c;
            const uint32_t nv = min(g.R, nwin - c * g.R), stage = i % g.S, par = (i / g.S) & 1u;
            const long long c0 = trace ? clock64() : 0;
            if (!failed && !mbar_wait(full0 + 8u * stage, par)) failed = true;
            if (trace) { const long long c1 = clock64(); tw += c1 - c0; ta -= c1; }
            if (own) {
              const float* rp = ring + (size_t)stage * g.R * g.stride + (e0 - col0);
              if (nv == g.R && g.R == 64u) {  // whole chunk: straight-line blocks
                chain_block<EPL, 32>(acc, rp, g.stride);
                chain_block<EPL, 32>(acc, rp + (size_t)32u * g.stride, g.stride);
              } else if (nv == g.R && g.R == 32u) {
                chain_block<EPL, 32>(acc, rp, g.stride);
              } else if (nv == g.R && g.R == 16u) {
                chain_block<EPL, 16>(acc, rp, g.stride);
              } else if (nv == g.R && g.R == 8u) {
                chain_block<EPL, 8>(acc, rp, g.stride);
              } else {  // the item's last chunk (the producer padded it with zero rows to a multiple of four)
                for (uint32_t r = 0; r < nv; r += 4) chain_block<EPL, 4>(acc, rp + (size_t)r * g.stride, g.stride);
              }
            }
            mbar_arrive(empty0 + 8u * stage);  // the slot may be refilled
            if (trace) ta += clock64();
          }
          if (trace && tid == 0) { trace[8 * h + 4] = (unsigned long long)tw; trace[8 * h + 5] = (unsigned long long)ta; }
        }
        it += n_chunks;
      }
      if (trace && tid == 0) {
        trace[8 * h + 2] = globaltimer_ns();
        trace[8 * h + 3] = ((unsigned long long)blockIdx.x << 32) | cnt;
      }
      // ---- this pass's columns of the sum (chain warps).  Columns past dim (dim % EPL != 0) were summed from the
      // ring's padding and are dropped here.
      if (own) {
        const uint32_t nq = min((uint32_t)EPL, t.dim - e0);
        if (nq == EPL) RowElems<-1, EPL>::template st<EPL>(dst + e0, acc);
        else for (uint32_t q = 0; q < nq; ++q) dst[e0 + q] = acc[q];
      }
    }
  }
  if (failed && lane == 0) atomicAdd(&t.counters[CTR_ERR], 1u);
}

// ---- the optimizer step of the hot items, once the NaN verdict is known: a warp per item, the reduced gradient from the
// hot stage.  Lane l owns the elements e0 = (l + 32 k) * EPL, EPL at a time and the last ones one by one.  When dim is
// not a multiple of EPL the state arrays (row + dim, row + 2 dim) are not EPL-float aligned: every element goes one by
// one then.  (An element's step depends on its index alone, so the grouping never changes a result.)
template <int EPL>
__global__ void __launch_bounds__(256) k_step_hot(TableDev t, OptimDev op, HyperDev hy, SlotsDev sl, GradsDev gr, ReduceArgs a) {
  __shared__ uint32_t dead[PB_MAX_SLOTS / 32];
  const uint32_t n_giant = a.b.cnt[BC_GIANT], n_huge = a.b.cnt[BC_HUGE];
  const uint32_t n_hot = a.b.cnt[BC_HOT] + n_huge + n_giant;
  const uint32_t per_block = blockDim.x / 32u;
  if (blockIdx.x * per_block >= n_hot) return;  // whole block
  build_dead_mask(dead, gr, a, sl.n_slots);
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t h = blockIdx.x * per_block + threadIdx.x / 32u; h < n_hot; h += gridDim.x * per_block) {
    const uint32_t entry = hot_entry(a.b, h, n_giant, n_huge);
    const uint4 d = a.b.hot[entry];
    const uint32_t row = d.x, slot = d.w;
    if (slot_dead(dead, slot)) continue;
    if (row >= t.capacity) {
      if (lane == 0 && !a.quiet_miss) atomicAdd(&t.counters[CTR_GRAD_MISS], 1u);  // gradient_id_miss_count (PS mod.rs:401-403)
      continue;
    }
    const float* g = a.hot_stage + (size_t)entry * a.hot_stride;
    float* prow = t.rows + (size_t)row * t.stride;
    const StepCtx sc = step_ctx(prow, t, op, gr, slot);
    const bool aligned = t.dim % EPL == 0;
    for (uint32_t e0 = lane * EPL; e0 < t.dim; e0 += 32u * EPL) {
      const uint32_t nq = min((uint32_t)EPL, t.dim - e0);
      if (aligned && nq == EPL) {
        float acc[EPL];
        RowElems<-1, EPL>::template ld<EPL>(g + e0, acc);
        RowElems<-1, EPL> rc;
        rc.load(prow, e0, t, op);
        rc.step(e0, acc, t, op, hy, sc);
        rc.store(prow, e0, t, op);
      } else {
        for (uint32_t q = 0; q < nq; ++q) {
          RowElems<-1, 1> rc;
          float one[1] = {g[e0 + q]};
          rc.load(prow, e0 + q, t, op);
          rc.step(e0 + q, one, t, op, hy, sc);
          rc.store(prow, e0 + q, t, op);
        }
      }
    }
    if (op.kind == PB_OPT_ADAGRAD_VW) {  // state = state*mom + dot(g,g)/dim (optim.rs:280-283)
      __syncwarp();                      // every lane has read the old state (step_ctx)
      if (lane == 0) prow[t.dim] = __fadd_rn(__fmul_rn(sc.vw_state, op.mom), __fdiv_rn(vw_dot(g, t.dim), (float)t.dim));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// launchers (host)
// ------------------------------------------------------------------------------------------------
template <int VEC, bool F16>
static void items_dispatch(const TableDev& t, const OptimDev& op, const HyperDev& hy, const SlotsDev& sl, const GradsDev& gr,
                           const ReduceArgs& a, uint32_t G, cudaStream_t st, cudaStream_t st_warm, bool send) {
  // grids sized for the worst case (every occurrence its own item); blocks past the list lengths return at once
  const uint32_t per_block = 256u / G;
  uint32_t grid_cold = cdiv(a.b.n, per_block), grid_warm = cdiv(a.b.n / 2 + 1, per_block);
  if (grid_cold > 148u * 6u) grid_cold = 148u * 6u;  // groups stride over their list
  if (grid_warm > 148u * 3u) grid_warm = 148u * 3u;
  if (send) {
    PB_LAUNCH_F(FAM_WARM, (k_reduce_warm<VEC, F16, PB_OPT_SGD, true>), grid_warm, 256, 0, st_warm, t, op, hy, sl, gr, a, G);
    PB_LAUNCH_F(FAM_UPDATE, (k_reduce_cold<VEC, F16, PB_OPT_SGD, true>), grid_cold, 256, 0, st, t, op, hy, sl, gr, a, G);
    return;
  }
#define PB_K(KK)                                                                                                   \
  case KK:                                                                                                         \
    PB_LAUNCH_F(FAM_WARM, (k_reduce_warm<VEC, F16, KK, false>), grid_warm, 256, 0, st_warm, t, op, hy, sl, gr, a, G); \
    PB_LAUNCH_F(FAM_UPDATE, (k_reduce_cold<VEC, F16, KK, false>), grid_cold, 256, 0, st, t, op, hy, sl, gr, a, G); \
    break;
  switch (op.kind) { PB_K(PB_OPT_SGD) PB_K(PB_OPT_ADAGRAD) PB_K(PB_OPT_ADAGRAD_VW) PB_K(PB_OPT_ADAM) }
#undef PB_K
}

static unsigned long long* g_hot_trace = nullptr;  // debugging aid: per hot item {start, sorted, summed} globaltimer stamps
void set_hot_trace(unsigned long long* p) { g_hot_trace = p; }

template <int EPL, bool F16, bool SEND>
static void hot_launch(const TableDev& t, const SlotsDev& sl, const GradsDev& gr, const ReduceArgs& a, uint32_t vec,
                       cudaStream_t st) {
  HotGeom g;
  g.cols = t.dim < HOT_COLS ? t.dim : HOT_COLS;
  g.stride = (g.cols + 3u) & ~3u;
  g.CH = (g.cols + 32u * EPL - 1u) / (32u * EPL);
  g.rowbytes = t.dim * (F16 ? 2u : 4u);
  g.vec = vec;
  const uint32_t nvr = g.cols / (F16 ? 8u : 4u);
  g.vshift = 32u;
  if (vec && nvr && !(nvr & (nvr - 1u)))
    for (g.vshift = 0; (1u << g.vshift) < nvr; ++g.vshift) {}
  g.S = HOT_MAX_SLOTS;
  uint32_t slot_bytes = 8192;
  if (getenv("PB_HOT_SLOT_BYTES")) slot_bytes = (uint32_t)atoi(getenv("PB_HOT_SLOT_BYTES"));
  g.R = slot_bytes / (g.stride * 4u);
  if (g.R > 32u) g.R = 32u;  // a chunk's rows are described by the lanes of the producing warp
  if (vec && g.R * nvr > 256u) g.R = 256u / nvr;  // at most eight 16-byte loads per producer lane and chunk
  g.R &= ~3u;  // the chain adds groups of four rows
  if (g.R < 4u) g.R = 4u;
  if (vec && g.R * nvr > 256u) g.vec = 0;  // (rows longer than 64 vectors per pass: element by element)
  g.lean = g.vec && g.vshift <= 5u && t.dim <= HOT_COLS && !a.occ_outrow && !getenv("PB_HOT_NO_LEAN");
  // every chunk costs the chain a barrier round trip (~500 cycles measured) whatever its size: two halves per chunk
  g.R1 = g.R;
  if (!getenv("PB_HOT_ONE_HALF")) {  // 64 rows per chunk where the slot stays within 32 KB
    while (g.R < 64u && 2u * g.R * g.stride * 4u <= 32768u) g.R *= 2u;
    if (g.R * g.stride * 4u > 16384u) g.S = 6;  // 6 x 32 KB (the producers must not outnumber the slots)
  }
  const size_t smem = (size_t)g.S * g.R * g.stride * 4u;
  auto kern = k_reduce_hot<EPL, F16, SEND>;
  static size_t configured[64] = {0};  // per instantiation and device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && smem > configured[dev]) {
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    configured[dev] = smem;
  }
  // one block per SM: a producer keeps two chunks (64 registers of loads) in flight, which needs the whole register
  // file share of a 256-thread block
  uint32_t per_sm = 1;
  if (getenv("PB_HOT_PER_SM")) per_sm = (uint32_t)atoi(getenv("PB_HOT_PER_SM"));
  const uint32_t cap_blocks = cdiv(a.b.n, PB_WARM_MAX + 1);  // at most this many hot items exist
  uint32_t grid = 148u * per_sm;
  if (grid > cap_blocks) grid = cap_blocks ? cap_blocks : 1;
  PB_LAUNCH_F(FAM_HOT, kern, grid, HOT_THREADS, smem, st, t, sl, gr, a, g, g_hot_trace);
}

// chain lanes own 2 columns (one or two chain warps) up to 128 columns, 4 above
static bool hot_epl2(uint32_t dim) { return dim <= 128u && dim % 2u == 0; }

uint32_t hot_stage_stride(uint32_t dim) { return (dim + 3u) & ~3u; }  // whole float4s for the chain lanes' stores

void launch_reduce_hot(const TableDev& t, const SlotsDev& sl, const GradsDev& gr, bool f16, const ReduceArgs& a,
                       cudaStream_t st, bool send) {
  if (!a.b.n) return;
  const uint32_t ev = f16 ? 8u : 4u;  // the producers' 16-byte loads need whole vectors and aligned rows
  uint32_t hv = t.dim % ev == 0 ? 1u : 0u;
  for (uint32_t s = 0; s < sl.n_slots && hv; ++s)
    if (gr.ptr[s] && (reinterpret_cast<uintptr_t>(gr.ptr[s]) & 15u)) hv = 0;
  if (getenv("PB_HOT_NO_VEC")) hv = 0;
#define PB_H(E)                                                 \
  if (send) {                                                   \
    if (f16) hot_launch<E, true, true>(t, sl, gr, a, hv, st);   \
    else hot_launch<E, false, true>(t, sl, gr, a, hv, st);      \
  } else {                                                      \
    if (f16) hot_launch<E, true, false>(t, sl, gr, a, hv, st);  \
    else hot_launch<E, false, false>(t, sl, gr, a, hv, st);     \
  }
  if (hot_epl2(t.dim)) { PB_H(2) } else { PB_H(4) }
#undef PB_H
}

void launch_step_hot(const TableDev& t, const OptimDev& op, const HyperDev& hy, const SlotsDev& sl, const GradsDev& gr,
                     const ReduceArgs& a, cudaStream_t st) {
  if (!a.b.n) return;
  // a warp per item; blocks past the list's length (it lives on the device) return at once
  uint32_t grid = cdiv(cdiv(a.b.n, PB_WARM_MAX + 1), 8u);
  if (grid > 148u * 8u) grid = 148u * 8u;
  if (hot_epl2(t.dim)) PB_LAUNCH(k_step_hot<2>, grid, 256, 0, st, t, op, hy, sl, gr, a);
  else PB_LAUNCH(k_step_hot<4>, grid, 256, 0, st, t, op, hy, sl, gr, a);
}

void launch_reduce_items(const TableDev& t, const OptimDev& op, const HyperDev& hy, const SlotsDev& sl,
                         const GradsDev& gr, bool f16, const ReduceArgs& a, cudaStream_t st, cudaStream_t st_warm,
                         bool send) {
  if (!a.b.n) return;
  int vec, Gi;
  vec_group(t.dim, vec, Gi);
  uint32_t G = (uint32_t)Gi < 4u ? 4u : (uint32_t)Gi;
  if (vec == 4) {
    if (f16) items_dispatch<4, true>(t, op, hy, sl, gr, a, G, st, st_warm, send);
    else items_dispatch<4, false>(t, op, hy, sl, gr, a, G, st, st_warm, send);
  } else {
    if (f16) items_dispatch<1, true>(t, op, hy, sl, gr, a, G, st, st_warm, send);
    else items_dispatch<1, false>(t, op, hy, sl, gr, a, G, st, st_warm, send);
  }
}

}  // namespace pb
