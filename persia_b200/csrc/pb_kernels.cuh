// pb_kernels.cuh — kernel-side parameter blocks and launcher prototypes (internal).
#pragma once
#include <atomic>

#include "pb_common.cuh"

namespace pb {

// per-batch slot table, passed by value in kernel-parameter memory
struct SlotsDev {
  uint64_t prefix[PB_MAX_SLOTS];
  uint32_t occ_off[PB_MAX_SLOTS + 1];  // slot boundaries in the flat id array
  uint8_t sqrt_scaling[PB_MAX_SLOTS];
  uint32_t n_slots;
  uint64_t spacing;  // 2^(64-prefix_bit) - 1
  uint32_t spacing_bits;  // 64 - prefix_bit
  uint32_t uniform;       // occurrences per slot when every slot holds the same number (one id per sample), else 0
};

// per-batch gradient table (GradientBatch, persia-core/src/backward.rs:74-106)
struct GradsDev {
  const void* ptr[PB_MAX_SLOTS];  // nullptr = skipped slot
  float inv_scale[PB_MAX_SLOTS];  // 1/scale_factor
  uint8_t do_scale[PB_MAX_SLOTS]; // |scale-1| > f32::EPSILON (mod.rs:751)
  const float* adam_pow;          // Adam: accumulated (beta1^t, beta2^t) pairs on the device, one per feature group
  uint8_t pow_idx[PB_MAX_SLOTS];  // the slot's pair
};

// ---- the batch context on the device (what the EW keeps in post_forward_buffer, mod.rs:1087-1098) ------------------
// Filled by the forward (dedup -> probe -> gather), consumed by the backward.  A distinct (sign, slot) pair of the
// batch is an "item"; the occurrences of an item with count > 1 are listed in seg_occ[base, base + count) in
// arbitrary order (the reducing kernels put them in ascending order, the reference's summation order).
constexpr uint32_t PB_GIANT_MIN = 1024;  // the few longest chains of a batch: listed in the top giant_cap entries of `hot`
constexpr uint32_t PB_HUGE_MIN = 256;  // hot items above this are the long poles of the backward: they start first
constexpr uint32_t PB_WARM_MAX = 32;  // items of 2..PB_WARM_MAX occurrences are reduced by a lane group, larger ones by a CTA
enum {
  BC_ITEMS = 0,  // distinct items of the batch
  BC_COLD,       // items of one occurrence
  BC_WARM,       // items of 2..PB_WARM_MAX occurrences
  BC_HOT,        // items of more
  BC_SEG,        // entries of seg_occ handed out
  BC_HUGE,       // hot items of more than PB_HUGE_MIN occurrences: listed from the END of `hot`, reduced first
  BC_HOTW,       // words of the hot-item bitmap pool handed out
  BC_GIANT,      // hot items of more than PB_GIANT_MIN occurrences: the very first to be reduced
  BC_PEER = 8,
  BC_NEXT = 24,  // work cursors of the reducing kernels: [round] warm, [PB_MAX_SLOTS + round] hot
  BC_COUNT = BC_NEXT + 2 * PB_MAX_SLOTS
};
struct BatchDev {
  DCell* set;           // scratch set: region of slot s = [2*occ_off[s] + 2*s, +2*n_s + 1), then its reserved cell
  uint32_t* occ_set;    // [n] set cell of every occurrence
  uint32_t* item_cell;  // [n] set cell of every item
  uint32_t* seg_occ;    // [n] occurrence lists
  uint2* cold;          // [n]   (target, occurrence)
  uint4* warm;          // [n/2] (target, base, count, -)
  uint4* hot;           // [n/PB_WARM_MAX] (target, base | bitmap word offset + bit 31, count, slot)
  uint32_t* hot_bits;   // [hot_words] one bit per sample of the slot for hot items in bitmap mode (all zero between batches)
  uint32_t hot_words;
  uint32_t hot_cap;     // entries of `hot`
  uint32_t giant_cap;   // of which the top ones are reserved for the giants (n / PB_GIANT_MIN + 1)
  uint32_t* cnt;        // BC_* words
  uint32_t n;           // id occurrences of the batch
};

// ---- the shard exchange (pb_shard.cu): one endpoint per rank, buffers in peer-mapped memory -----------------------
// Every rank is an embedding worker for its own batches (requester) and parameter server `rank` (owner).  Rank r owns
// one receive area, written by its peers over NVLink with plain stores; `base[q]` is rank q's area as mapped here.
//   ctrl   [XC_WORDS][16] u32   flags (one word per phase and source, written by that source) and sign counts
//   sign   [R][cap] u64         signs requested of this rank, by source
//   row    [R][cap][dim]        rows returned to this rank, by owner (f16, or f32 for ragged layouts)
//   grad   [R][cap][dim] f32    reduced gradients sent to this rank, by source
//   gok    [R][cap] u32         1 = apply the gradient, 0 = the slot was skipped / held a NaN
enum { XC_FLAG_SIGN = 0, XC_FLAG_ROW, XC_FLAG_GRAD, XC_COUNT, XC_WORDS };
constexpr uint32_t PB_MAX_RANKS = 16;
constexpr uint32_t PB_ADAM_KEYS = 256;  // beta-power pairs per table; the last one serves pb_update
// owner side, one step: the distinct rows the R requests touch (k_owner_lookup fills it, k_owner_update_all empties it)
struct __align__(16) UCell {
  uint32_t row;               // ROW_NONE = empty
  uint32_t mask;              // sources that asked for the row
  uint32_t k[PB_MAX_RANKS];   // the row's index in each such source's request
  uint32_t pad[2];
};
struct XchgDev {
  uint64_t base[PB_MAX_RANKS];
  uint64_t off_sign, off_row, off_grad, off_gok;  // byte offsets inside an area (ctrl at 0)
  uint32_t R, rank, cap, row_f32;
  uint32_t* epoch;     // [XC_WORDS] phases signalled so far (device side: CUDA-graph safe)
  uint32_t* waited;    // [XC_WORDS][PB_MAX_RANKS] phases waited for so far, per source
  uint32_t* own_row;   // [R][cap] row of every received sign (forward -> backward)
  uint32_t* own_cnt;   // [R] signs received per source (copied out of ctrl: the next request may overwrite it early)
  uint32_t* err;       // [0] a pair needed more than cap slots, [1] a wait gave up
  UCell* ucell;        // [ucells] rows of the step's requests, hashed by row number
  uint32_t* uwin;      // [R][cap] the cell a request's sign opened (it was the first to ask for the row), else ROW_NONE
  uint32_t ucells;     // a power of two >= 2 R cap
  // Adam on the owner: feature groups (index prefixes) of the table, the groups each request holds, and the (beta1^t,
  // beta2^t) pair every request's signs of a group use (get_batch_level_state, optim.rs:151-197)
  const uint64_t* akeys;  // [n_akeys] prefixes, position = pair number of the table
  uint32_t n_akeys;
  uint64_t amask;         // the prefix bits of a sign
  uint32_t* apresent;     // [R][PB_ADAM_KEYS / 32] groups among the signs request s applies
  float* apow;            // [R][PB_ADAM_KEYS][2]
};

// arguments of the backward kernels (pb_reduce.cu)
struct ReduceArgs {
  BatchDev b;
  const uint32_t* occ_outrow;  // nullptr: one id per sample per slot (output row == occurrence)
  const uint32_t* row_off;
  const uint32_t* tick_ptr;
  const uint32_t* nan_tick;
  float* vw_stage;             // Adagrad vectorwise: one reduced gradient per item
  float* hot_stage;            // [hot_cap][hot_stride] reduced gradient of every hot item (k_reduce_hot -> k_step_hot)
  uint32_t hot_stride;
  uint32_t batch, round, quiet_miss;
  uint32_t round_mask[PB_MAX_SLOTS / 32];  // slots stepped by this launch (slots of one feature group take turns)
  XchgDev x;                   // sharded: the reduced gradient is stored into the owner's receive area instead
};

// raw slots (pb_raw.cu): per-batch scratch set of distinct signs and its workspace
struct RawCell {
  uint64_t key;
  uint32_t first;  // first occurrence of the sign in the flat id array
  uint32_t rank;   // number of the sign among the batch's distinct signs (first-occurrence order)
};
struct RawWork {
  RawCell* set;      // set_mask + 2 cells
  uint32_t set_mask;
  uint32_t* occ_set;        // set cell of every occurrence
  uint32_t* flag;           // scan input / second scan output
  uint32_t* rank;           // scan output
  uint32_t* tiles;          // scan spine
  uint32_t* distinct_cell;  // index cell of every distinct sign (forward -> backward)
  uint32_t* counts;         // [0] distinct signs, [1] ids placed in `index`
};

void launch_fill_cells(Cell* cells, uint64_t n, cudaStream_t st);
void launch_fill_set(DCell* set, uint64_t n, cudaStream_t st);
// bump: a training request (advances the table's batch number and the context's request number)
void launch_begin_batch(const TableDev& t, uint32_t* ctx_tick, uint32_t* batch_cnt, cudaStream_t st, bool bump = true);
void launch_probe(int mode, bool prefix, const TableDev& t, const HyperDev& hy, const OptimDev& op, const SlotsDev& sl,
                  const uint64_t* ids, uint32_t n, uint32_t* occ_cell, cudaStream_t st);
void launch_gather(const TableDev& t, const uint32_t* occ_cell, uint32_t n_out, float* out, cudaStream_t st);
// batched path (pb_dedup.cu)
void launch_dedup(const SlotsDev& sl, const BatchDev& b, const uint64_t* ids, cudaStream_t st);
void launch_probe_items(bool training, const TableDev& t, const HyperDev& hy, const OptimDev& op, const SlotsDev& sl,
                        const BatchDev& b, cudaStream_t st);
void launch_gather_items(const TableDev& t, const SlotsDev& sl, const BatchDev& b, const uint32_t* row_off,
                         uint32_t n_out, uint32_t batch, bool training, void* out_f16, cudaStream_t st);
void launch_clear_items(const BatchDev& b, cudaStream_t st);
void launch_clear_hot_bits(const BatchDev& b, cudaStream_t st);  // of a batch whose backward never came
void launch_copy_entries(bool write, const TableDev& t, const uint32_t* occ_cell, uint32_t n, float* entries,
                         uint8_t* found, cudaStream_t st);
void launch_nan_scan(const GradsDev& gr, uint32_t n_slots, uint32_t elems_per_slot, bool f16, const uint32_t* tick,
                     uint32_t* nan_tick, int32_t* status, cudaStream_t st);
// pb_reduce.cu.  send: sharded requester — a.x names the owners' receive areas, no row is touched here.
// Hot items: their gradient sums go to a.hot_stage (to the owners when sending); the sums read no NaN verdict, so they
// may start before the NaN scan has finished.  launch_step_hot then steps the rows of the applied ones.
void launch_reduce_hot(const TableDev& t, const SlotsDev& sl, const GradsDev& gr, bool f16, const ReduceArgs& a,
                       cudaStream_t st, bool send = false);
void launch_step_hot(const TableDev& t, const OptimDev& op, const HyperDev& hy, const SlotsDev& sl, const GradsDev& gr,
                     const ReduceArgs& a, cudaStream_t st);
uint32_t hot_stage_stride(uint32_t dim);
// cold items on `st`, warm items on `st_warm` (may equal st)
void launch_reduce_items(const TableDev& t, const OptimDev& op, const HyperDev& hy, const SlotsDev& sl,
                         const GradsDev& gr, bool f16, const ReduceArgs& a, cudaStream_t st, cudaStream_t st_warm,
                         bool send = false);
// pb_shard.cu
void launch_route_items(bool training, const SlotsDev& sl, const BatchDev& b, const XchgDev& x, cudaStream_t st);
void launch_signal(const XchgDev& x, int phase, const uint32_t* counts, cudaStream_t st);
void launch_wait(const XchgDev& x, int phase, int src /* -1: every source */, cudaStream_t st);
void launch_signal_wait(const XchgDev& x, int phase, const uint32_t* counts, cudaStream_t st);
void launch_owner_lookup(bool training, const TableDev& t, const HyperDev& hy, const OptimDev& op, const XchgDev& x,
                         cudaStream_t st);
void launch_expand_items(const TableDev& t, const SlotsDev& sl, const BatchDev& b, const XchgDev& x,
                         const uint32_t* row_off, uint32_t n_out, uint32_t batch, bool training, void* out_f16,
                         cudaStream_t st);
void launch_hash_stack(const uint64_t* ids, uint32_t n, uint32_t rounds, uint64_t size, uint64_t* out, cudaStream_t st);
void launch_owner_adam(const XchgDev& x, float* table_pow, float b1, float b2, cudaStream_t st);
void launch_uclear(const XchgDev& x, cudaStream_t st);
void launch_owner_update_all(const TableDev& t, const OptimDev& op, const HyperDev& hy, const XchgDev& x, cudaStream_t st);
void launch_owner_update(const TableDev& t, const OptimDev& op, const HyperDev& hy, const XchgDev& x, uint32_t src,
                         cudaStream_t st);
// n_ptr (optional): the live count on the device (<= n); tick/nan_tick (optional): skip everything when equal
void launch_update_direct(const TableDev& t, const OptimDev& op, const HyperDev& hy, const uint32_t* occ_cell,
                          const float* grads, uint32_t n, const float* adam_pair, cudaStream_t st,
                          const uint32_t* n_ptr = nullptr, const uint32_t* tick = nullptr,
                          const uint32_t* nan_tick = nullptr);
struct AdamKeys {
  uint8_t idx[PB_MAX_SLOTS];
  uint32_t n;
};
void launch_adam_fill(float* pow, float b1, float b2, cudaStream_t st);
void launch_adam_advance(float* pow, const AdamKeys& keys, float b1, float b2, cudaStream_t st, const GradsDev* gr = nullptr,
                         uint32_t n_slots = 0, const uint32_t* tick = nullptr, const uint32_t* nan_tick = nullptr);
uint32_t raw_scan_tiles(uint32_t n);
void launch_raw_forward(const TableDev& t, const SlotsDev& sl, const uint64_t* ids, uint32_t n,
                        const uint32_t* row_off, const uint32_t* occ_sample, uint32_t batch, uint32_t fixed,
                        const uint32_t* occ_cell, const RawWork& w, void* table_f16, long long* index,
                        long long* non_empty, uint32_t* sample_id_num, cudaStream_t st);
void launch_raw_nan(const void* grad, bool f16, const uint32_t* n_distinct, uint32_t dim, const uint32_t* tick,
                    uint32_t* nan_tick, cudaStream_t st);
void launch_raw_stage(const void* grad, bool f16, const uint32_t* n_distinct, uint32_t dim, float inv_scale,
                      bool do_scale, float* out, cudaStream_t st);
void launch_slot_status(const GradsDev& gr, uint32_t n_slots, const uint32_t* tick, const uint32_t* nan_tick,
                        int32_t* status, cudaStream_t st);
uint32_t radix_tile(uint32_t n);
uint32_t radix_hist_words();
uint32_t radix_hist_zero_words(uint32_t n);
void launch_zero_words(uint32_t* p, uint32_t n_words, cudaStream_t st);
uint64_t partition_workspace_bytes(uint32_t n);
void launch_partition_by_shard(const uint64_t* signs, uint32_t n, uint32_t R, uint32_t* perm, uint32_t* counts,
                               uint32_t* work, cudaStream_t st);
void launch_expand_rows(const uint32_t* row_off, uint32_t n_out, uint32_t* occ_outrow, cudaStream_t st);
void launch_add_prefix(const SlotsDev& sl, const uint64_t* ids, uint32_t n, uint64_t* out, cudaStream_t st);
void launch_shard_of(const uint64_t* signs, uint32_t n, uint32_t R, uint32_t* shard, uint64_t* hash, cudaStream_t st);
void launch_export_signs(const TableDev& t, uint64_t* signs, uint32_t* recency, uint32_t max_n, uint32_t* count,
                         cudaStream_t st);
void launch_spill(const TableDev& t, uint32_t want_free, uint32_t keep, uint32_t* ev, uint64_t* signs, float* entries,
                  uint32_t max_n, uint32_t* count, cudaStream_t st);
void launch_evict(const TableDev& t, uint32_t low_water, uint32_t target_free, uint32_t keep, uint32_t* ev, cudaStream_t st);
uint64_t launch_count();
enum { FAM_PROBE = 0, FAM_DEDUP, FAM_GATHER, FAM_NAN, FAM_HOT, FAM_UPDATE, FAM_OTHER, FAM_WARM, FAM_WAIT, FAM_ROUTE, FAM_OWNER, FAM_COUNT };
bool profiling();  // a kernel family is being timed: the backward then runs its kernels one after another
void profile_enable(uint32_t family_mask);
void profile_read(double* ms, uint64_t* count, int n_families);

enum { MODE_FIND = 0, MODE_TRAIN = 1, MODE_SET = 2 };

}  // namespace pb
