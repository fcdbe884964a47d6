// dnz_kernels.cu -- sm_100a kernels of the windowed grouped aggregate.
//
//   k_tile_scan      per-tile byte ranges + timestamp min/max  (RecordBatchWatermark::try_from, utils/time.rs:31-57)
//   k_aggregate      TMA-staged (cp.async.bulk + mbarrier ring) key interning + count/min/max/sum reduction
//                    (GroupedAggWindowFrame::push + group_aggregate_batch, grouped_window_agg_stream.rs:501-605;
//                     DataFusion GroupValues::intern + GroupsAccumulator::update_batch x4)
//   k_aggregate_generic / k_deferred   same arithmetic with direct global loads (bitmaps, unaligned or very long keys,
//                    rows replayed after a table grew)
//   k_emit           pane combine + avg + FilterExec predicate (totalOrder) + stream compaction into Arrow columns
//                    (trigger_windows / evaluate, :220-253, :609-629; continuous/mod.rs:64-89; FilterExec)
//
// No tensor-core work exists on this path (no dense contraction); the kernels are HBM/L2-transaction bound.
#include <algorithm>
#include <cstring>

#include "dnz_device.cuh"

namespace dnz {

// =================================================================================================
// k_tile_scan
// =================================================================================================
__global__ void k_init_minmax(BatchMinMax* mm, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) { mm[i].ts_min = INT64_MAX; mm[i].ts_max = INT64_MIN; mm[i].n_valid = 0; mm[i].key_bytes = 0; mm[i].n_fast = 0; mm[i].n_tiles = 0; }
}

// One warp per tile, SCAN_TILES_PER_CTA consecutive tiles per CTA, four CONSECUTIVE tiles per warp.  The batch that owns the
// CTA's first tile is found by one 32-ary search; warps walk forward from there.  The kernel has to stream 8 B per row and was
// instruction-bound (605 warp instructions per 416-row tile: 64-bit min/max chains, 64-bit shuffles, a 64-bit division), so:
//   * timestamps are reduced as 32-bit offsets from the tile's first timestamp (u = ts - first + 2^31: one 64-bit subtract,
//     an OR of the high words that proves the offsets fit, 32-bit min / max); a tile whose timestamps spread over more than
//     +-24 days takes the 64-bit path
//   * the warp reduction is three REDUX instructions
//   * the pane of the minimum comes from one multiplication by 1 / pane_ms in double precision (exact below 2^53) plus a fix-up
//   * the per-batch results are accumulated over the warp's tiles and flushed with one set of atomics per batch change.
constexpr int SCAN_TILES_PER_CTA = 32;
constexpr int SCAN_TILES_PER_WARP = 4;
__global__ void __launch_bounds__(256, 3) k_tile_scan(const BatchDesc* __restrict__ batches, int64_t n_batches, int64_t n_tiles,
                                                    int64_t pane_ms, double inv_pane_ms, TileDesc* __restrict__ tiles, BatchMinMax* mm, int allow_fast) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ int64_t s_b0;
  const int64_t t0 = (int64_t)blockIdx.x * SCAN_TILES_PER_CTA;
  if (warp == 0) {             // batch that owns tile t0: last b with tile0 <= t0 (tile0 is non-decreasing); 32-ary search by one
    int64_t lo = 0, hi = n_batches;   // warp: 2 dependent load rounds for 1 K batches instead of 10
    while (hi - lo > 1) {
      const int64_t step = (hi - lo + 31) / 32, b = lo + step * lane;
      const bool ok = b < hi && batches[b].tile0 <= t0;
      const unsigned m = __ballot_sync(0xffffffffu, ok) | 1u;
      const int last = 31 - __clz((int)m);
      lo = lo + step * last; hi = min(hi, lo + step);
    }
    if (lane == 0) s_b0 = lo;
  }
  __syncthreads();
  int64_t lo = s_b0;
  // per-batch accumulators of this warp (meaningful in lane 0)
  int64_t acc_b = -1; long long acc_mn = INT64_MAX, acc_mx = INT64_MIN; unsigned long long acc_valid = 0, acc_bytes = 0, acc_fast = 0, acc_tiles = 0;
  auto flush = [&]() {
    if (lane == 0 && acc_b >= 0) {
      BatchMinMax* m = mm + acc_b;
      if (acc_valid) { atomicMin((long long*)&m->ts_min, acc_mn); atomicMax((long long*)&m->ts_max, acc_mx); atomicAdd((unsigned long long*)&m->n_valid, acc_valid); }
      atomicAdd((unsigned long long*)&m->key_bytes, acc_bytes); atomicAdd((unsigned long long*)&m->n_tiles, acc_tiles);
      if (acc_fast) atomicAdd((unsigned long long*)&m->n_fast, acc_fast);
    }
    acc_mn = INT64_MAX; acc_mx = INT64_MIN; acc_valid = acc_bytes = acc_fast = acc_tiles = 0;
  };
  const int64_t tw0 = t0 + (int64_t)warp * SCAN_TILES_PER_WARP;
  for (int64_t t = tw0; t < tw0 + SCAN_TILES_PER_WARP && t < n_tiles; t++) {
    while (lo + 1 < n_batches && batches[lo + 1].tile0 <= t) lo++;
    if (lo != acc_b) { flush(); acc_b = lo; }
    const BatchDesc bd = batches[lo];
    const int64_t row0 = (t - bd.tile0) * TILE;
    const int n = (int)min((int64_t)TILE, bd.n_rows - row0);
    const int32_t o_lane = (lane < 2 && bd.off) ? bd.off[row0 + (lane ? n : 0)] : 0;      // key byte range: in flight while the timestamps stream (no key column: ungrouped)
    long long mn = INT64_MAX, mx = INT64_MIN; int cnt = 0;
    const long long* ts = reinterpret_cast<const long long*>(bd.ts) + row0;
    if (!bd.ts_valid && (reinterpret_cast<uintptr_t>(ts) & 15u) == 0) {
      const longlong2* p = reinterpret_cast<const longlong2*>(ts);
      const int np = n >> 1;
      static_assert(TILE <= 7 * 64, "seven 16 B loads per lane cover a tile");
      // all loads of the tile are issued back to back (a loop with a per-lane trip count ends up in the compiler's serial
      // remainder loop: one dependent round trip per iteration)
      longlong2 v[7];
      const long long first = __ldg(ts);                                    // same address for the whole warp: one transaction
      const long long tail = (n & 1) ? __ldg(ts + n - 1) : first;           // odd row count (last tile of a batch)
#pragma unroll
      for (int k = 0; k < 7; k++) { const int i = lane + 32 * k; v[k] = i < np ? __ldg(p + i) : make_longlong2(first, tail); }
      const long long basem = first - 0x80000000ll;
      uint32_t mn32 = 0xFFFFFFFFu, mx32 = 0u, orhi = 0u;
#pragma unroll
      for (int k = 0; k < 7; k++) {
        const unsigned long long u0 = (unsigned long long)(v[k].x - basem), u1 = (unsigned long long)(v[k].y - basem);
        orhi |= (uint32_t)(u0 >> 32) | (uint32_t)(u1 >> 32);
        mn32 = min(mn32, min((uint32_t)u0, (uint32_t)u1)); mx32 = max(mx32, max((uint32_t)u0, (uint32_t)u1));
      }
      { const unsigned long long ut = (unsigned long long)(tail - basem); orhi |= (uint32_t)(ut >> 32); mn32 = min(mn32, (uint32_t)ut); mx32 = max(mx32, (uint32_t)ut); }
      orhi = __reduce_or_sync(0xffffffffu, orhi);
      if (orhi == 0u) {
        mn32 = __reduce_min_sync(0xffffffffu, mn32); mx32 = __reduce_max_sync(0xffffffffu, mx32);
        mn = basem + (long long)mn32; mx = basem + (long long)mx32;
      } else {                                                             // widely spread timestamps: 64-bit path
#pragma unroll
        for (int k = 0; k < 7; k++) { mn = min(mn, min(v[k].x, v[k].y)); mx = max(mx, max(v[k].x, v[k].y)); }
        mn = min(mn, tail); mx = max(mx, tail);
        for (int o = 16; o; o >>= 1) { mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
      }
      cnt = n;
    } else {
      for (int r = lane; r < n; r += 32) {
        bool ok = bd.ts_valid == nullptr || bit_at(bd.ts_valid, bd.ts_vbit + row0 + r);
        if (ok) { long long v = ts[r]; mn = min(mn, v); mx = max(mx, v); cnt++; }
      }
      for (int o = 16; o; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      }
    }
    const int32_t o0 = __shfl_sync(0xffffffffu, o_lane, 0), o1 = __shfl_sync(0xffffffffu, o_lane, 1);
    if (lane == 0) {
      TileDesc td;
      td.batch = (int32_t)lo; td.row0 = (int32_t)row0; td.n_rows = n; td.flags = 0;
      td.byte0 = o0; td.byte_len = o1 - o0; td.pad = 0;
      td.ts_min = mn; td.ts_max = mx; td.pane_lo = 0;
      if (cnt == 0) td.flags |= TILE_EMPTY;
      else {
        // floor(mn / pane_ms): timestamps in [0, 2^53) (negative ones are rejected by the host before aggregation, and the pane of
        // such a tile is never used); the product is within one unit of the quotient, the remainder test makes it exact
        long long q;
        if (mn >= 0 && mn < (1ll << 53)) {
          q = (long long)((double)mn * inv_pane_ms);
          long long r = mn - q * pane_ms;
          if (r < 0) { q--; r += pane_ms; } else if (r >= pane_ms) { q++; r -= pane_ms; }
        } else q = mn / pane_ms;
        td.pane_lo = q;
        if (mx < (q + 1) * pane_ms) td.flags |= TILE_PANE_UNIFORM;     // == (mx / pane_ms == pane_lo) for ts >= 0
        acc_mn = min(acc_mn, mn); acc_mx = max(acc_mx, mx); acc_valid += (unsigned long long)cnt;
      }
      bool aligned = ((reinterpret_cast<uintptr_t>(bd.ts + row0) | reinterpret_cast<uintptr_t>(bd.val + row0) |
                       reinterpret_cast<uintptr_t>(bd.off + row0) | reinterpret_cast<uintptr_t>(bd.bytes)) & 15u) == 0;
      if (allow_fast && (bd.flags & BATCH_BULK_OK) && aligned && !bd.ts_valid && !bd.val_valid && !bd.key_valid && cnt > 0)
        td.flags |= td.byte_len <= BCAP ? TILE_FAST : (TILE_FAST | TILE_KEYS_GLOBAL);
      tiles[t] = td;
      acc_bytes += (unsigned long long)td.byte_len; acc_tiles += 1;
      if (td.flags & TILE_FAST) acc_fast += 1;
    }
  }
  flush();
}

cudaError_t launch_tile_scan(const BatchDesc* batches, int64_t n_batches, int64_t n_tiles, int64_t pane_ms, TileDesc* tiles,
                             BatchMinMax* minmax, bool allow_fast, cudaStream_t s) {
  if (n_batches <= 0 || n_tiles <= 0) return cudaSuccess;
  k_init_minmax<<<(unsigned)((n_batches + 255) / 256), 256, 0, s>>>(minmax, n_batches);
  k_tile_scan<<<(unsigned)((n_tiles + SCAN_TILES_PER_CTA - 1) / SCAN_TILES_PER_CTA), 256, 0, s>>>(batches, n_batches, n_tiles, pane_ms, 1.0 / (double)pane_ms, tiles, minmax, allow_fast ? 1 : 0);
  return cudaGetLastError();
}

// =================================================================================================
// row application shared by every aggregate path
// =================================================================================================
// Returns false when the row had to be deferred (nothing was modified).
__device__ __forceinline__ bool apply_row(const AggParams& P, uint32_t tile, uint32_t row, int64_t pane, bool val_ok, double v,
                                          uint32_t gid, unsigned long long rowseq) {
  int64_t pi = pane - P.panes.pane0;
  if (pi < 0 || pi >= P.panes.n_panes) return true;           // cannot happen: the host sizes the table from the tile scan
  GroupState* m = P.panes.main[pi];
  GroupState* l = P.panes.late[pi];
  if (!val_ok) {
    unsigned long long* nm = m ? P.panes.nullrows_main[pi] : nullptr;
    unsigned long long* nl = l ? P.panes.nullrows_late[pi] : nullptr;
    if ((m && !nm) || (l && !nl)) { defer_row(P.defer, tile, row, DEFER_NEED_NULLROWS); return false; }
    if (nm) red_add_u64(nm + gid, 1ull);
    if (nl) red_add_u64(nl + gid, 1ull);
    return true;
  }
  unsigned long long* fm = nullptr; unsigned long long* fl = nullptr;
  if (v == 0.0) {
    fm = m ? P.panes.fz_main[pi] : nullptr; fl = l ? P.panes.fz_late[pi] : nullptr;
    if ((m && !fm) || (l && !fl)) { defer_row(P.defer, tile, row, DEFER_NEED_FZ); return false; }
  }
  if (m) state_update(m, fm, gid, v, rowseq);
  if (l) state_update(l, fl, gid, v, rowseq);
  return true;
}

// One row read straight from global memory (bitmaps honoured).
__device__ __forceinline__ void process_row_generic(const AggParams& P, uint32_t tile, const TileDesc& td, const BatchDesc& bd,
                                                    uint32_t r) {
  int64_t row = (int64_t)td.row0 + r;
  if (bd.ts_valid && !bit_at(bd.ts_valid, bd.ts_vbit + row)) return;          // null timestamp: row vanishes (§8a-1)
  int64_t ts = bd.ts[row];
  bool val_ok = !bd.val_valid || bit_at(bd.val_valid, bd.val_vbit + row);
  double v = val_ok ? bd.val[row] : 0.0;
  bool key_ok = !bd.key_valid || bit_at(bd.key_valid, bd.key_vbit + row);
  uint32_t gid;
  if (key_ok) {
    int32_t o0 = bd.off[row], o1 = bd.off[row + 1];
    KeyRef k; load_key<false>(bd.bytes + o0, (uint32_t)(o1 - o0), k);
    gid = dict_lookup(P.dict, k, false);
  } else gid = dict_lookup_null(P.dict);
  if (gid == GID_DEFER_GROUPS) { defer_row(P.defer, tile, r, DEFER_GROUPS_FULL); return; }
  if (gid == GID_DEFER_ARENA) { defer_row(P.defer, tile, r, DEFER_ARENA_FULL); return; }
  int64_t pane = (td.flags & TILE_PANE_UNIFORM) ? td.pane_lo : ts / P.panes.pane_ms;
  unsigned long long rowseq = ((unsigned long long)bd.seq << 32) | (unsigned long long)row;
  apply_row(P, tile, r, pane, val_ok, v, gid, rowseq);
}

__global__ void __launch_bounds__(256) k_aggregate_generic(const __grid_constant__ AggParams P) {
  for (int64_t t = P.tile_begin + blockIdx.x; t < P.tile_end; t += gridDim.x) {
    const TileDesc td = P.tiles[t];
    if (td.flags & TILE_EMPTY) continue;
    const BatchDesc bd = P.batches[td.batch];
    for (uint32_t r = threadIdx.x; r < (uint32_t)td.n_rows; r += blockDim.x) process_row_generic(P, (uint32_t)(t - P.tile_begin), td, bd, r);
  }
}

__global__ void __launch_bounds__(256) k_deferred(const __grid_constant__ AggParams P, uint64_t n_entries, const DeferEntry* entries) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_entries; i += (uint64_t)gridDim.x * blockDim.x) {
    DeferEntry e = entries[i];
    const TileDesc td = P.tiles[P.tile_begin + e.tile];
    const BatchDesc bd = P.batches[td.batch];
    process_row_generic(P, e.tile, td, bd, e.row);
  }
}

// =================================================================================================
// k_aggregate: persistent (two CTAs of 14 warps per SM), warp-specialised.
//
// The last warp is the TMA producer.  It claims tiles from a global counter (stream order), resolves their descriptors,
// and per tile: waits for the ring slot, writes the tile header (row count, key byte base, resolved pane state array +
// hint tag) into shared memory and issues four 1-D bulk copies (timestamps, values, key offsets, key bytes; SASS
// UBLKCP) that complete on the slot's `full` mbarrier.
//
// The other 13 warps consume, one row per thread (26 consumer warps per SM across the two CTAs hide the L2 round trip of
// the probe).  Hot path per row: 3 LDS for value/offsets, 4-5 LDS.32 + funnel shifts + clamp-shift masks for the <= 16 B
// key, a 32-bit hash, ONE 32 B dictionary-slot load (LDG.E.256) that also carries the group's min/max hint; a row whose
// slot holds another key is parked in the warp's retry queue; count and sum are reduced by lane PAIRS: lanes 2j / 2j+1
// update {cnt, sum} of the same row with one red.add.f64 (16 sectors per instruction instead of 32); min / max are reduced
// by the row's own lane for the ~7 % of the rows the hint lets through.  Everything rare (empty or locked slot -> insert,
// keys > 16 B, +-0.0 / non-finite values, tiles spanning panes, late panes) is outlined into __noinline__ helpers so
// that the hot loop stays ~330 SASS instructions per 32 rows (profiles/README.md).
// =================================================================================================
struct __align__(16) StageHdr {   // the consumers read the first two 16 B words with one LDS.128 each (2 wavefronts per tile, not 8)
  int32_t n_rows, flags, a0; uint32_t tag;
  GroupState* mbase;            // main state array of the tile's pane when every row can take the paired path, else nullptr
  uint32_t tile_rel, pane_rel;  // tile index inside the launch; pane index relative to PaneTable::pane0 (when mbase != nullptr)
  long long pane_lo;
  unsigned long long rowseq0;   // (batch arrival seq << 32) | first row of the tile inside its batch
  const uint8_t* gbytes;        // TILE_KEYS_GLOBAL: the batch's key byte buffer (offsets are absolute)
  uint32_t pad[2];
};
static_assert(sizeof(StageHdr) == 64, "header size");
struct __align__(128) Stage {
  long long ts[TILE];
  double val[TILE];
  int32_t off[TILE + 4];
  uint8_t bytes[BCAP + 48];     // a FAST tile stages <= BCAP + 15 bytes; the key loader may over-read 20 B past a key start
  StageHdr hdr;
};
// Per-warp retry queue.  A row whose first probe hit a slot occupied by ANOTHER key does not make its warp loop (the
// slowest of 64 rows would pace the warp: ~3 dependent L2 round trips per tile at 25 % load); it is parked here with its
// next slot index and re-probed 32 rows at a time, so every round trip is a full-warp load.
constexpr int QCAP = 64;             // < 32 carried over + 32 new rows
struct WarpQueue {
  uint4 key[QCAP];                   // inline key words
  uint2 meta[QCAP];                  // x: next slot index, y: key length | pane index (relative to PaneTable::pane0) << 8
  double val[QCAP];
  uint32_t row[QCAP];                // tile (relative to the launch) << 10 | row inside the tile  (deferred-row bookkeeping)
};
static_assert(TILE <= 1024, "row packing");
struct __align__(16) TileFetch {     // what the producer needs to hand one tile to the ring (staged in shared memory, 2 x 32)
  StageHdr h;
  const int64_t* gts; const double* gval; const int32_t* goff; const uint8_t* gby;
  uint32_t nts, noff, nby, pad;
};
struct AggSmem {
  Stage st[STAGES];
  WarpQueue q[CONSUMER_WARPS];
  TileFetch fetch[2][8];
  uint64_t full[STAGES];
  uint64_t empty[STAGES];
};

__device__ __forceinline__ uint32_t round16(uint32_t x) { return (x + 15u) & ~15u; }
__device__ __forceinline__ uint32_t lds32(uint32_t addr) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }

// ---- outlined slow paths ------------------------------------------------------------------------------------------------
// Full dictionary lookup / insert for one staged row (any key length).  Returns the gid (or GID_DEFER_*).
// Out-parameters would live in local memory, and local loads queue behind the scattered traffic in the L1TEX FIFO:
// the slot index comes back packed as (slot << 32) | gid.
__device__ __noinline__ uint64_t agg_probe_slow(const AggParams& P, const uint8_t* key_smem, uint32_t len) {
  KeyRef k; load_key<true>(key_smem, len, k);
  uint32_t slot = 0; uint32_t g = dict_lookup(P.dict, k, true, &slot);
  return ((uint64_t)slot << 32) | g;
}
__device__ __noinline__ uint64_t agg_probe_slow_global(const AggParams& P, const uint8_t* key_gmem, uint32_t len) {
  KeyRef k; load_key<false>(key_gmem, len, k);
  uint32_t slot = 0; uint32_t g = dict_lookup(P.dict, k, false, &slot);
  return ((uint64_t)slot << 32) | g;
}
// Accumulate one staged row through the general per-row path (pane from the timestamp, late panes, +-0.0, ...).
__device__ __noinline__ void agg_apply_slow(const AggParams& P, const StageHdr& h, uint32_t r, long long ts, double v, uint32_t gid) {
  long long pane = (h.flags & TILE_PANE_UNIFORM) ? h.pane_lo : ts / P.panes.pane_ms;
  apply_row(P, h.tile_rel, r, pane, true, v, gid, h.rowseq0 + r);
}
// Lookup / insert of a parked row whose chain ended in an empty or locked slot (inline key rebuilt from its words).
__device__ __noinline__ uint64_t agg_probe_words(const AggParams& P, uint4 kw, uint32_t len) {
  KeyRef k; k.k0 = ((uint64_t)kw.y << 32) | kw.x; k.k1 = ((uint64_t)kw.w << 32) | kw.z; k.len = len; k.ptr = nullptr;
  k.hash = hash_words(kw.x, kw.y, kw.z, kw.w, len);
  uint32_t slot = 0; uint32_t g = dict_lookup(P.dict, k, false, &slot);
  return ((uint64_t)slot << 32) | g;
}
__device__ __noinline__ void agg_tile_generic(const AggParams& P, uint32_t tile_rel, int tid) {
  const TileDesc td = P.tiles[P.tile_begin + tile_rel];
  if (td.flags & TILE_EMPTY) return;
  const BatchDesc bd = P.batches[td.batch];
  for (uint32_t r = tid; r < (uint32_t)td.n_rows; r += CONSUMER_WARPS * 32) process_row_generic(P, tile_rel, td, bd, r);
}

// One full-warp probe round over the top (up to) 32 parked rows.  Rows that resolve are accumulated with scalar
// reductions (count, sum, hint-gated min / max); rows that collide again are pushed back.  Returns the new queue length.
__device__ __noinline__ uint32_t agg_queue_round(const AggParams& P, WarpQueue& Q, uint32_t qcount, int lane, bool use_hints) {
  __syncwarp();
  const uint32_t nb = min(qcount, 32u), base = qcount - nb;
  const bool have = (uint32_t)lane < nb;
  uint4 kw = make_uint4(0, 0, 0, 0); uint2 me = make_uint2(0, 0); uint32_t ro = 0; double v = 0.0;
  bool again = false;
  if (have) {
    kw = Q.key[base + lane]; me = Q.meta[base + lane]; v = Q.val[base + lane]; ro = Q.row[base + lane];
    const uint32_t len = me.y & 0xFFu, pi = me.y >> 8;
    uint64_t sa, sb, sc, sd;
    ld_slot(P.dict.slots + me.x, sa, sb, sc, sd);
    const uint32_t state = (uint32_t)(sd >> 32);
    uint32_t gid = 0, slot = me.x; uint64_t hint = 0; bool done = false;
    if (state - 1u < 0xFFFFFFFEu) {
      if ((uint32_t)sd == len && sa == (((uint64_t)kw.y << 32) | kw.x) && sb == (((uint64_t)kw.w << 32) | kw.z)) { gid = state - 1u; hint = sc; done = true; }
      else { me.x = (me.x + 1u) & P.dict.mask; again = true; }
    } else { const uint64_t gs = agg_probe_words(P, kw, len); gid = (uint32_t)gs; slot = (uint32_t)(gs >> 32); done = true; }
    if (done) {
      if (gid >= GID_DEFER_ARENA) defer_row(P.defer, ro >> 10, ro & 1023u, gid == GID_DEFER_GROUPS ? DEFER_GROUPS_FULL : DEFER_ARENA_FULL);
      else {
        GroupState* s = (P.priv ? P.priv + ((size_t)blockIdx.x * P.panes.n_panes + pi) * P.priv_groups : P.panes.main[pi]) + gid;   // parked rows: plain main pane, v != +-0.0
        const uint32_t tag = (uint32_t)P.panes.tag_main[pi];
        const unsigned long long o = ord_bits((unsigned long long)__double_as_longlong(v));
        const bool okmin = v <= 1.7976931348623157e308, okmax = v >= -1.7976931348623157e308;
        const uint32_t tmin = (uint32_t)((ORD_F64_MAX - o) >> 48), tmax = (uint32_t)((o - ORD_F64_MIN) >> 48);
        uint32_t hmin = 0, hmax = 0;
        const uint32_t htag = (uint32_t)(hint >> 32);
        if (use_hints && htag == tag) { hmin = (uint32_t)(hint >> 16) & 0xFFFFu; hmax = (uint32_t)hint & 0xFFFFu; }
        red_add_f64(&s->cnt, 1.0); red_add_f64(&s->sum, v);
        if (okmin && tmin >= hmin) red_max_u64(&s->minkey, ORD_F64_MAX - o);
        if (okmax && tmax >= hmax) red_max_u64(&s->maxkey, o - ORD_F64_MIN);
        if (use_hints && (int32_t)(htag - tag) <= 0 && ((okmin && tmin > hmin) || (okmax && tmax > hmax))) {
          const uint32_t nmin = okmin ? max(hmin, tmin) : hmin, nmax = okmax ? max(hmax, tmax) : hmax;
          st_relaxed_u64(&P.dict.slots[slot].hint, ((uint64_t)tag << 32) | ((uint64_t)nmin << 16) | (uint64_t)nmax);
        }
      }
    }
  }
  __syncwarp();                                        // every lane has read its entry before the survivors are re-packed
  const uint32_t bal = __ballot_sync(0xffffffffu, again);
  if (again) {
    const uint32_t pos = base + __popc(bal & ((1u << lane) - 1u));
    Q.key[pos] = kw; Q.meta[pos] = me; Q.val[pos] = v; Q.row[pos] = ro;
  }
  return base + __popc(bal);
}

__global__ void __launch_bounds__(AGG_THREADS, 2) k_aggregate(const __grid_constant__ AggParams P) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  AggSmem& S = *reinterpret_cast<AggSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < STAGES; s++) { mbar_init(&S.full[s], 1); mbar_init(&S.empty[s], CONSUMER_WARPS); }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == CONSUMER_WARPS) {
    // ------------------------------------------------------------ producer warp
    // Lanes 0..CLAIM-1 resolve the descriptors of the claimed tiles in parallel (TileDesc -> BatchDesc -> pane table: three
    // dependent global loads that would otherwise serialise per tile) into shared memory; lane 0 then feeds the ring.
    auto fetch = [&](int64_t t, TileFetch& d) {
      StageHdr h; h.mbase = nullptr; h.tag = 0; h.pane_lo = 0; h.rowseq0 = 0; h.n_rows = 0; h.flags = 0; h.a0 = 0; h.tile_rel = 0;
      h.pane_rel = 0; h.gbytes = nullptr; h.pad[0] = h.pad[1] = 0;
      d.nts = d.noff = d.nby = 0;
      if (t < P.tile_end) {
        const TileDesc td = P.tiles[t];
        const BatchDesc& bd = P.batches[td.batch];
        h.n_rows = td.n_rows; h.flags = td.flags; h.pane_lo = td.pane_lo; h.tile_rel = (uint32_t)(t - P.tile_begin);
        h.a0 = (int32_t)(td.byte0 & ~(int64_t)15);
        h.rowseq0 = ((unsigned long long)bd.seq << 32) | (unsigned long long)(uint32_t)td.row0;
        if (td.flags & TILE_FAST) {
          d.gts = bd.ts + td.row0; d.gval = bd.val + td.row0; d.goff = bd.off + td.row0; d.gby = bd.bytes + h.a0;
          d.nts = round16((uint32_t)td.n_rows * 8u); d.noff = round16(((uint32_t)td.n_rows + 1u) * 4u);
          d.nby = (td.flags & TILE_KEYS_GLOBAL) ? 0u : round16((uint32_t)(td.byte0 + td.byte_len - h.a0));
          h.gbytes = bd.bytes;
          if (td.flags & TILE_PANE_UNIFORM) {
            int64_t pi = td.pane_lo - P.panes.pane0;
            if (pi >= 0 && pi < P.panes.n_panes && P.panes.late[pi] == nullptr) {
              h.mbase = P.panes.main[pi]; h.tag = (uint32_t)P.panes.tag_main[pi]; h.pane_rel = (uint32_t)pi;
              if (P.priv && h.mbase) h.mbase = P.priv + ((size_t)blockIdx.x * P.panes.n_panes + pi) * P.priv_groups;
            }
          }
        }
      }
      d.h = h;
    };
    // Tiles are claimed dynamically, CLAIM at a time, in stream order: all CTAs then work within a few hundred tiles of each
    // other, so that two panes are in flight only for ~1 % of the rows around a pane boundary (hints of the older pane are
    // dead once the newer pane's rows arrive) and the tail of the launch balances itself.
    constexpr uint32_t CLAIM = 4;
    const uint32_t n_tiles = (uint32_t)(P.tile_end - P.tile_begin);
    uint32_t it = 0;
    // the NEXT claim (atomic + three dependent descriptor loads, ~4 us) is resolved while the current one feeds the ring
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(P.tile_counter, CLAIM);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base < n_tiles && lane < (int)CLAIM) fetch(P.tile_begin + base + lane, S.fetch[0][lane]);
    int buf = 0;
    while (base < n_tiles) {
      uint32_t nbase = 0;
      if (lane == 0) nbase = atomicAdd(P.tile_counter, CLAIM);
      nbase = __shfl_sync(0xffffffffu, nbase, 0);
      if (nbase < n_tiles && lane < (int)CLAIM) fetch(P.tile_begin + nbase + lane, S.fetch[buf ^ 1][lane]);
      __syncwarp();
      if (lane == 0) {
        for (uint32_t j = 0; j < CLAIM && base + j < n_tiles; j++, it++) {
          const int s = it % STAGES;
          const TileFetch& f = S.fetch[buf][j];
          mbar_wait(&S.empty[s], ((it / STAGES) & 1u) ^ 1u);
          S.st[s].hdr = f.h;
          if (f.h.flags & TILE_FAST) {
            mbar_arrive_expect_tx(&S.full[s], f.nts * 2u + f.noff + f.nby);
            bulk_g2s(S.st[s].ts, f.gts, f.nts, &S.full[s]);
            bulk_g2s(S.st[s].val, f.gval, f.nts, &S.full[s]);
            bulk_g2s(S.st[s].off, f.goff, f.noff, &S.full[s]);
            if (f.nby) bulk_g2s(S.st[s].bytes, f.gby, f.nby, &S.full[s]);
          } else {
            mbar_arrive(&S.full[s]);
          }
        }
      }
      it = __shfl_sync(0xffffffffu, it, 0);
      base = nbase; buf ^= 1;
    }
    if (lane == 0) {                                   // end marker for the consumers
      const int s = it % STAGES;
      mbar_wait(&S.empty[s], ((it / STAGES) & 1u) ^ 1u);
      S.st[s].hdr.flags = TILE_END;
      mbar_arrive(&S.full[s]);
    }
    return;
  }

  // -------------------------------------------------------------- consumer warps: one row per thread
  const DictSlot* const slots = P.dict.slots;
  const uint32_t dmask = P.dict.mask;
  // hints are switched off together with the private pane copies (low cardinality): the copies make every reduction cheap, and
  // hint stores into a few hundred hot dictionary sectors that every SM keeps reading bounce those lines between the two L2
  // partitions (ncu on cfg 1: 57 % of the samples waiting for the probe, LSU pipe 6 % busy)
  const bool use_hints = !(P.flags & AGG_NO_HINTS) && P.priv == nullptr, use_queue = !(P.flags & AGG_NO_QUEUE);
  uint32_t qcount = 0;                 // warp-uniform
  for (uint32_t it = 0;; it++) {
    const int s = it % STAGES;
    mbar_wait(&S.full[s], (it / STAGES) & 1u);
    const Stage& st = S.st[s];
    const StageHdr& H = st.hdr;
    const int4 h0 = *reinterpret_cast<const int4*>(&H.n_rows);            // n_rows, flags, a0, tag
    if (h0.y & TILE_END) break;
    // Everything derived from the thread index is recomputed per tile behind an opaque barrier: hoisted out of the loop
    // these values (lane masks, shuffle sources, queue address) cost registers the 64-register budget does not have, and
    // a spill is a local-memory access that queues behind the scattered traffic in the L1TEX FIFO.
    uint32_t tix = (uint32_t)tid; asm volatile("" : "+r"(tix));
    const int lane = (int)(tix & 31u), odd = (int)(tix & 1u);
    WarpQueue& Q = S.q[tix >> 5];
    if (!(h0.y & TILE_FAST)) {
      agg_tile_generic(P, H.tile_rel, (int)tix);
    } else {
      const uint4 h1 = *reinterpret_cast<const uint4*>(&H.mbase);         // mbase, tile_rel, pane_rel
      const uint32_t r = tix;
      const bool live = r < (uint32_t)h0.x;
      GroupState* const mbase = reinterpret_cast<GroupState*>(((uint64_t)h1.y << 32) | h1.x);
      const double v = st.val[r];
      const int32_t o0 = st.off[r], o1 = st.off[r + 1];
      const bool keys_global = (h0.y & TILE_KEYS_GLOBAL) != 0;          // warp-uniform: the key bytes were not staged
      const uint32_t klen = live ? (uint32_t)(o1 - o0) : 0u, kb = (live && !keys_global) ? (uint32_t)(o0 - h0.z) : 0u;
      const uint32_t addr = smem_u32(st.bytes) + kb, q = addr & ~3u, mis = addr & 3u, sh = mis * 8u;
      uint32_t a[5];
#pragma unroll
      for (int j = 0; j < 4; j++) a[j] = lds32(q + 4u * j);
      a[4] = (mis + klen > 16u) ? lds32(q + 16u) : 0u;                    // a 5th word only when the key straddles it
      // byte mask of word i of a klen-byte key: 0xFFFFFFFF >> clamp(32 - 8 * (klen - 4 i), 0, 32)  (shf.r.clamp saturates at 32)
      const int mb = 32 - 8 * (int)min(klen, (uint32_t)INLINE_KEY);
      const uint32_t w0 = __funnelshift_r(a[0], a[1], sh) & __funnelshift_rc(0xFFFFFFFFu, 0u, (uint32_t)max(mb, 0));
      const uint32_t w1 = __funnelshift_r(a[1], a[2], sh) & __funnelshift_rc(0xFFFFFFFFu, 0u, (uint32_t)max(mb + 32, 0));
      const uint32_t w2 = __funnelshift_r(a[2], a[3], sh) & __funnelshift_rc(0xFFFFFFFFu, 0u, (uint32_t)max(mb + 64, 0));
      const uint32_t w3 = __funnelshift_r(a[3], a[4], sh) & __funnelshift_rc(0xFFFFFFFFu, 0u, (uint32_t)max(mb + 96, 0));
      uint32_t idx = hash_words(w0, w1, w2, w3, klen) & dmask;
      // paired-path row: finite and not +-0.0 (everything else goes through the general per-row path)
      const uint32_t bhi = (uint32_t)__double2hiint(v), blo = (uint32_t)__double2loint(v);
      const bool plain = mbase != nullptr && (bhi & 0x7FF00000u) != 0x7FF00000u && ((bhi << 1) | blo) != 0u;
      uint32_t gid = 0; uint64_t hint = 0;
      bool need_slow = live && (klen > (uint32_t)INLINE_KEY || keys_global), park = false, hit = false;
      // ONE dictionary probe (32 B sector, carries the group's min/max hint)
      if (live && !need_slow) {
        uint64_t sa, sb, sc, sd;
        ld_slot(slots + idx, sa, sb, sc, sd);
        const uint32_t state = (uint32_t)(sd >> 32);
        if (state - 1u < 0xFFFFFFFEu) {                   // occupied and published
          if ((uint32_t)sd == klen && (uint32_t)sa == w0 && (uint32_t)(sa >> 32) == w1 && (uint32_t)sb == w2 && (uint32_t)(sb >> 32) == w3) {
            gid = state - 1u; hint = sc; hit = true;
          } else if (use_queue && plain) { idx = (idx + 1u) & dmask; park = true; }   // chain continues: park, re-probe 32 at a time
          else need_slow = true;
        } else need_slow = true;                          // empty (insert) or locked (insert in flight)
      }
      const uint32_t bal = __ballot_sync(0xffffffffu, park);
      if (bal) {
        if (park) {
          const uint32_t pos = qcount + __popc(bal & ((1u << lane) - 1u));
          Q.key[pos] = make_uint4(w0, w1, w2, w3);
          Q.meta[pos] = make_uint2(idx, klen | (h1.w << 8));
          Q.val[pos] = v;
          Q.row[pos] = (h1.z << 10) | r;
        }
        qcount += __popc(bal);
      }
      if (need_slow) {
        const uint64_t gs = keys_global ? agg_probe_slow_global(P, H.gbytes + o0, klen) : agg_probe_slow(P, st.bytes + kb, klen);
        gid = (uint32_t)gs; idx = (uint32_t)(gs >> 32); hint = 0; hit = true;
      }
      uint32_t pk = 0;
      if (hit) {
        if (gid >= GID_DEFER_ARENA) defer_row(P.defer, h1.z, r, gid == GID_DEFER_GROUPS ? DEFER_GROUPS_FULL : DEFER_ARENA_FULL);
        else if (plain) {
          // hints: top 16 bits of minkey / maxkey follow from the high word of ord(v) alone (no borrow from the low word)
          const uint32_t ohi = (bhi & 0x80000000u) ? ~bhi : (bhi | 0x80000000u);
          const uint32_t tmin = (0xFFEFFFFFu - ohi) >> 16, tmax = (ohi - 0x00100000u) >> 16;
          uint32_t hmin = 0, hmax = 0;
          const uint32_t tag = (uint32_t)h0.w;
          const uint32_t htag = (uint32_t)(hint >> 32);
          if (use_hints && htag == tag) { hmin = (uint32_t)(hint >> 16) & 0xFFFFu; hmax = (uint32_t)hint & 0xFFFFu; }
          // CTAs drift apart by up to a few million rows, so around a pane boundary two panes are in flight: a straggler of
          // the OLDER pane (smaller tag; tags live in [1, 2^31)) never replaces the newer pane's hint -- it just reduces
          if (use_hints && (int32_t)(htag - tag) <= 0 && (tmin > hmin || tmax > hmax))
            st_relaxed_u64(const_cast<uint64_t*>(&slots[idx].hint), ((uint64_t)tag << 32) | ((uint64_t)max(hmin, tmin) << 16) | (uint64_t)max(hmax, tmax));
          // min / max: the hint lets ~7 % of the rows through; they are reduced here, by the row's own lane.  (Parking them in a
          // per-warp queue and reducing 32 at a time was tried in round 2: 0.96 ms instead of 0.92 ms per launch -- the queue
          // bookkeeping costs more than the sparse instructions it saves.)
          const uint32_t olo = (bhi & 0x80000000u) ? ~blo : blo;
          if (tmin >= hmin) red_max_u64(&mbase[gid].minkey, ((unsigned long long)(0xFFEFFFFFu - ohi) << 32) | (uint32_t)~olo);
          if (tmax >= hmax) red_max_u64(&mbase[gid].maxkey, ((unsigned long long)(ohi - 0x00100000u) << 32) | olo);
          pk = gid | (1u << 29);
        } else {
          agg_apply_slow(P, H, r, st.ts[r], v, gid);
        }
      }
      // count and sum by lane pairs: in each of two instructions lanes 2j / 2j+1 update {cnt, sum} of ONE row -- adjacent words of
      // the state sector, 16 sectors per instruction, half the reduction wavefronts of two scalar reductions.  First the rows of
      // the even lanes (the row's own lane adds its value to sum, the odd partner adds 1.0 to cnt), then the rows of the odd
      // lanes: one xor-shuffle of the packed group id serves both (the value never leaves its lane).
      if (mbase != nullptr) {                       // warp-uniform
        const uint32_t pk2 = __shfl_xor_sync(0xffffffffu, pk, 1);
#pragma unroll
        for (int half = 0; half < 2; half++) {
          const bool own = (odd == half);
          const uint32_t p = own ? pk : pk2;
          if (p & (1u << 29)) {
            GroupState* s2 = mbase + (p & 0x1FFFFFFFu);
            red_add_f64(own ? &s2->sum : &s2->cnt, own ? v : 1.0);
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive_relaxed(&S.empty[s]);
    while (qcount >= 32u) qcount = agg_queue_round(P, Q, qcount, lane, use_hints);
  }
  while (qcount > 0u) qcount = agg_queue_round(P, S.q[warp], qcount, lane, use_hints);
}

static int g_agg_smem = 0;
cudaError_t agg_kernel_setup() {
  g_agg_smem = (int)sizeof(AggSmem);
  return cudaFuncSetAttribute(k_aggregate, cudaFuncAttributeMaxDynamicSharedMemorySize, g_agg_smem);
}

int aggregate_grid(int64_t n_tiles, int sm_count) {
  return (int)(n_tiles < (int64_t)sm_count * 2 ? n_tiles : (int64_t)sm_count * 2);          // two persistent CTAs per SM
}
cudaError_t launch_aggregate(const AggParams& p, int sm_count, cudaStream_t s) {
  int64_t n_tiles = p.tile_end - p.tile_begin;
  if (n_tiles <= 0) return cudaSuccess;
  if (!g_agg_smem) { cudaError_t e = agg_kernel_setup(); if (e != cudaSuccess) return e; }
  k_aggregate<<<aggregate_grid(n_tiles, sm_count), AGG_THREADS, g_agg_smem, s>>>(p);
  return cudaGetLastError();
}

// Fold the per-CTA private pane copies into the panes: thread per (pane of the launch, group id).
__global__ void __launch_bounds__(256) k_merge_private(const __grid_constant__ AggParams P, int n_cta) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  const int pi = blockIdx.y;
  if (g >= P.priv_groups) return;
  GroupState* dst = P.panes.main[pi];
  if (!dst) return;
  double cnt = 0.0, sum = 0.0; unsigned long long mn = 0, mx = 0; bool first = true;
  for (int c = 0; c < n_cta; c++) {
    const GroupState s = P.priv[((size_t)c * P.panes.n_panes + pi) * P.priv_groups + g];
    if (s.cnt != 0.0) { sum = first ? s.sum : sum + s.sum; first = false; cnt += s.cnt; }
    mn = max(mn, s.minkey); mx = max(mx, s.maxkey);
  }
  if (cnt == 0.0) return;
  GroupState* d = dst + g;                      // the slow paths may have reduced into the pane concurrently-ordered before: add
  red_add_f64(&d->cnt, cnt); red_add_f64(&d->sum, sum);
  if (mn) red_max_u64(&d->minkey, mn);
  if (mx) red_max_u64(&d->maxkey, mx);
}
cudaError_t launch_merge_private(const AggParams& p, int grid, cudaStream_t s) {
  if (!p.priv || grid <= 0) return cudaSuccess;
  dim3 g((p.priv_groups + 255) / 256, (unsigned)p.panes.n_panes);
  k_merge_private<<<g, 256, 0, s>>>(p, grid);
  return cudaGetLastError();
}
cudaError_t launch_aggregate_generic(const AggParams& p, int sm_count, cudaStream_t s) {
  int64_t n_tiles = p.tile_end - p.tile_begin;
  if (n_tiles <= 0) return cudaSuccess;
  int grid = (int)(n_tiles < (int64_t)sm_count * 8 ? n_tiles : (int64_t)sm_count * 8);
  k_aggregate_generic<<<grid, 256, 0, s>>>(p);
  return cudaGetLastError();
}
cudaError_t launch_deferred(const AggParams& p, const DeferEntry* in, uint64_t n_entries, cudaStream_t s) {
  if (!n_entries) return cudaSuccess;
  uint64_t gb = (n_entries + 255) / 256; int grid = (int)(gb < 148 * 8 ? gb : 148 * 8);
  k_deferred<<<grid, 256, 0, s>>>(p, n_entries, in);
  return cudaGetLastError();
}

// =================================================================================================
// k_aggregate_ungrouped: `.window([], aggs, ..)` -- WindowAggStream in Partial mode (streaming_window.rs:640-828): no key, one
// accumulator set per window.  Pure streaming reduction: a CTA owns a contiguous chunk of tiles, keeps {count, sum, min, max}
// of the pane it is in in registers, and flushes one set of reductions when the pane changes.  Accumulator semantics are those
// of DataFusion's row accumulators, NOT of the grouped ones: count of non-null values, sum by plain addition, min / max over
// IEEE totalOrder (arrow `compute::min/max` + ScalarValue total_cmp: -0.0 < +0.0, NaN above +inf) -- so the state keeps
// maxk = ord(v) and mink = ~ord(v), both reduced with max, zero = "no value" (decided by the count).
// State layout per pane: GroupState[0] = {cnt, sum, mink, maxk}; nullrows[0] counts rows whose value is NULL.
// =================================================================================================
struct UAcc { double cnt, sum; unsigned long long mink, maxk, nulls; };
__device__ __forceinline__ void uacc_add(UAcc& a, bool val_ok, double v) {
  if (!val_ok) { a.nulls++; return; }
  const unsigned long long o = ord_bits(f64_bits(v));
  a.cnt += 1.0; a.sum += v; a.mink = max(a.mink, ~o); a.maxk = max(a.maxk, o);
}
__device__ void uacc_flush(UAcc& a, GroupState* m, GroupState* l, unsigned long long* nm, unsigned long long* nl, double* s_red) {
  // block reduction (256 threads): warp shuffles, then warp 0 over the 8 partials
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 16; o; o >>= 1) {
    a.cnt += __shfl_xor_sync(0xffffffffu, a.cnt, o); a.sum += __shfl_xor_sync(0xffffffffu, a.sum, o);
    a.mink = max(a.mink, __shfl_xor_sync(0xffffffffu, a.mink, o)); a.maxk = max(a.maxk, __shfl_xor_sync(0xffffffffu, a.maxk, o));
    a.nulls += __shfl_xor_sync(0xffffffffu, a.nulls, o);
  }
  unsigned long long* s_u = reinterpret_cast<unsigned long long*>(s_red);
  __syncthreads();
  if (lane == 0) { s_red[warp * 5 + 0] = a.cnt; s_red[warp * 5 + 1] = a.sum; s_u[warp * 5 + 2] = a.mink; s_u[warp * 5 + 3] = a.maxk; s_u[warp * 5 + 4] = a.nulls; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double cnt = 0, sum = 0; unsigned long long mink = 0, maxk = 0, nulls = 0; bool first = true;
    for (int w = 0; w < 8; w++) {
      if (s_red[w * 5] != 0.0) { sum = first ? s_red[w * 5 + 1] : sum + s_red[w * 5 + 1]; first = false; cnt += s_red[w * 5]; }
      mink = max(mink, s_u[w * 5 + 2]); maxk = max(maxk, s_u[w * 5 + 3]); nulls += s_u[w * 5 + 4];
    }
    for (int k = 0; k < 2; k++) {
      GroupState* d = k ? l : m; unsigned long long* dn = k ? nl : nm;
      if (!d) continue;
      if (cnt != 0.0) { red_add_f64(&d->cnt, cnt); red_add_f64(&d->sum, sum); red_max_u64(&d->minkey, mink); red_max_u64(&d->maxkey, maxk); }
      if (nulls && dn) red_add_u64(dn, nulls);
    }
  }
  a.cnt = 0; a.sum = 0; a.mink = 0; a.maxk = 0; a.nulls = 0;
}
__global__ void __launch_bounds__(256) k_aggregate_ungrouped(const __grid_constant__ AggParams P) {
  __shared__ double s_red[8 * 5];
  const int64_t n_tiles = P.tile_end - P.tile_begin;
  const int64_t chunk = (n_tiles + gridDim.x - 1) / gridDim.x;
  const int64_t t0 = P.tile_begin + (int64_t)blockIdx.x * chunk, t1 = min(P.tile_end, t0 + chunk);
  UAcc a; a.cnt = 0; a.sum = 0; a.mink = 0; a.maxk = 0; a.nulls = 0;
  int64_t cur = INT64_MIN;                                  // pane the register accumulators belong to (block-uniform)
  auto flush = [&]() {
    if (cur == INT64_MIN) return;
    const int64_t pi = cur - P.panes.pane0;
    if (pi >= 0 && pi < P.panes.n_panes) uacc_flush(a, P.panes.main[pi], P.panes.late[pi], P.panes.nullrows_main[pi], P.panes.nullrows_late[pi], s_red);
    cur = INT64_MIN;
  };
  for (int64_t t = t0; t < t1; t++) {
    const TileDesc td = P.tiles[t];
    if (td.flags & TILE_EMPTY) continue;
    const BatchDesc bd = P.batches[td.batch];
    const bool uniform = (td.flags & TILE_PANE_UNIFORM) != 0 && bd.ts_valid == nullptr;
    if (uniform && td.pane_lo != cur) { flush(); cur = td.pane_lo; }
    if (!uniform) flush();
    for (int r = threadIdx.x; r < td.n_rows; r += blockDim.x) {
      const int64_t row = (int64_t)td.row0 + r;
      const bool val_ok = !bd.val_valid || bit_at(bd.val_valid, bd.val_vbit + row);
      const double v = val_ok ? __ldg(bd.val + row) : 0.0;
      if (uniform) { uacc_add(a, val_ok, v); continue; }
      // tile spans panes or has NULL timestamps: per-row reductions (rare)
      if (bd.ts_valid && !bit_at(bd.ts_valid, bd.ts_vbit + row)) continue;
      const int64_t pi = bd.ts[row] / P.panes.pane_ms - P.panes.pane0;
      if (pi < 0 || pi >= P.panes.n_panes) continue;
      for (int k = 0; k < 2; k++) {
        GroupState* d = k ? P.panes.late[pi] : P.panes.main[pi]; unsigned long long* dn = k ? P.panes.nullrows_late[pi] : P.panes.nullrows_main[pi];
        if (!d) continue;
        if (!val_ok) { if (dn) red_add_u64(dn, 1ull); continue; }
        const unsigned long long o = ord_bits(f64_bits(v));
        red_add_f64(&d->cnt, 1.0); red_add_f64(&d->sum, v); red_max_u64(&d->minkey, ~o); red_max_u64(&d->maxkey, o);
      }
    }
  }
  flush();
}
// one thread per closed window: combine its panes into one partial state (count +, sum + in ascending pane order, mink / maxk max)
__global__ void k_ungrouped_collect(const UWindow* __restrict__ wins, int n, UState* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const UWindow w = wins[i];
  UState r; r.cnt = 0; r.sum = 0.0; r.mink = 0; r.maxk = 0; r.nulls = 0;
  bool first = true;
  for (int p = 0; p < w.n; p++) {
    if (!w.st[p]) continue;
    const GroupState s = *w.st[p];
    if (s.cnt != 0.0) { r.sum = first ? s.sum : r.sum + s.sum; first = false; r.cnt += (unsigned long long)s.cnt; }
    r.mink = max(r.mink, s.minkey); r.maxk = max(r.maxk, s.maxkey);
    if (w.nr[p]) r.nulls += *w.nr[p];
  }
  out[i] = r;
}
cudaError_t launch_ungrouped_collect(const UWindow* wins, int n, UState* out, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_ungrouped_collect<<<(n + 63) / 64, 64, 0, s>>>(wins, n, out);
  return cudaGetLastError();
}
cudaError_t launch_aggregate_ungrouped(const AggParams& p, int sm_count, cudaStream_t s) {
  const int64_t n_tiles = p.tile_end - p.tile_begin;
  if (n_tiles <= 0) return cudaSuccess;
  k_aggregate_ungrouped<<<(unsigned)std::min<int64_t>(n_tiles, (int64_t)sm_count * 8), 256, 0, s>>>(p);
  return cudaGetLastError();
}

// =================================================================================================
// k_emit: one thread per group id.  Combines the window's panes (count +, sum + in ascending pane order, min/max
// over the ordered keys, first-zero sign), evaluates the post-aggregate predicate with IEEE totalOrder (arrow-ord
// cmp on Float64) and compacts the survivors: warp ballot + block scan -> one 64-bit atomic per block reserves
// (rows, key bytes) contiguously so that the Utf8 offsets stay monotone.
// =================================================================================================
__device__ __forceinline__ bool predicate(int op, long long a, long long b) {
  switch (op) { case 0: return a > b; case 1: return a >= b; case 2: return a < b; case 3: return a <= b; case 4: return a == b; default: return a != b; }
}

// owner hash of a group's key (NULL key: 0 -> rank 0)
__device__ __forceinline__ uint64_t key_hash(const GidKey& gk) {
  if (gk.len == 0xFFFFFFFFu) return 0;
  return gk.len <= (uint32_t)INLINE_KEY ? hash_inline(gk.k0, gk.k1, gk.len) : gk.k0;
}

struct Combined { unsigned long long cnt, nullrows, mnk, mxk, fz; double sum; bool present; };   // cnt: exact integer

__device__ __forceinline__ Combined combine_panes(const EmitParams& P, uint32_t g) {
  Combined c; c.cnt = 0; c.nullrows = 0; c.mnk = 0; c.mxk = 0; c.fz = ~0ull; c.sum = 0.0;
  bool first = true;
  for (int p = 0; p < P.n_panes; p++) {
    const GroupState s = P.panes[p][g];
    if (s.cnt != 0.0) { c.sum = first ? s.sum : c.sum + s.sum; first = false; }   // no "+ 0.0" for absent panes: keeps -0.0 sums exact
    c.cnt += (unsigned long long)s.cnt; c.mnk = max(c.mnk, s.minkey); c.mxk = max(c.mxk, s.maxkey);
    if (P.nullrows[p]) c.nullrows += P.nullrows[p][g];
    if (P.fz[p]) c.fz = min(c.fz, P.fz[p][g]);
  }
  c.present = (c.cnt | c.nullrows) != 0;
  return c;
}

constexpr int EMIT_STAGE = 12288;     // key bytes a block stages in shared memory before one coalesced copy
__global__ void __launch_bounds__(256) k_emit(const __grid_constant__ EmitParams P) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool keep = false; uint32_t klen = 0; Combined c; c.cnt = 0; c.sum = 0; c.mnk = c.mxk = 0; c.fz = ~0ull; c.nullrows = 0; c.present = false;
  GidKey gk; gk.k0 = gk.k1 = 0; gk.len = 0; gk.pad = 0;
  double mn = 0, mx = 0, avg = 0;
  bool agg_ok = false;
  if (P.gate) {                                       // block-uniform
    if ((P.gate[0] | P.gate[4] | P.gate[8]) != 0ull) { if (threadIdx.x == 0 && P.blocked) *P.blocked = 1u; return; }
  }
  const uint32_t n_groups = min(min(*P.dict.n_groups, P.dict.gcap), P.n_groups);
  if (g < n_groups) {
    c = combine_panes(P, g);
    if (c.present) {
      gk = P.dict.gid_key[g];
      klen = gk.len == 0xFFFFFFFFu ? 0u : gk.len;
      keep = P.world <= 1 || (int)(key_hash(gk) % (uint64_t)P.world) == P.rank;
      agg_ok = c.cnt != 0;
      if (agg_ok) {
        unsigned long long bmn = unord_bits(ORD_F64_MAX - c.mnk), bmx = unord_bits(c.mxk + ORD_F64_MIN);
        unsigned long long zsign = (c.fz != ~0ull) ? ((c.fz & 1ull) << 63) : 0ull;
        if ((bmn << 1) == 0) bmn = zsign;             // min is a zero: sign of the first zero seen
        if ((bmx << 1) == 0) bmx = zsign;
        mn = __longlong_as_double((long long)bmn); mx = __longlong_as_double((long long)bmx);
        avg = c.sum / (double)c.cnt;
      }
      if (keep && P.has_filter) {
        long long lit = total_key((unsigned long long)__double_as_longlong(P.filter_lit));
        if (P.filter_col == 0) keep = predicate(P.filter_op, total_key((unsigned long long)__double_as_longlong((double)(long long)c.cnt)), lit);
        else if (!agg_ok) keep = false;               // null predicate drops the row
        else {
          double x = P.filter_col == 1 ? mn : P.filter_col == 2 ? mx : P.filter_col == 3 ? avg : c.sum;
          keep = predicate(P.filter_op, total_key((unsigned long long)__double_as_longlong(x)), lit);
        }
      }
    }
  }
  // block-level exclusive scan of (rows, bytes)
  uint32_t kb = keep ? klen : 0u;
  uint32_t ballot = __ballot_sync(0xffffffffu, keep);
  uint32_t row_pre = __popc(ballot & ((1u << lane) - 1u));
  uint32_t byte_inc = kb;
  for (int o = 1; o < 32; o <<= 1) { uint32_t x = __shfl_up_sync(0xffffffffu, byte_inc, o); if (lane >= o) byte_inc += x; }
  __shared__ uint32_t wrows[8], wbytes[8]; __shared__ unsigned long long base; __shared__ uint32_t s_tb;
  __shared__ __align__(16) uint8_t stage[EMIT_STAGE + 8];
  if (lane == 31) { wrows[warp] = __popc(ballot); wbytes[warp] = byte_inc; }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tr = 0, tb = 0;
    for (int i = 0; i < 8; i++) { uint32_t r = wrows[i], b = wbytes[i]; wrows[i] = tr; wbytes[i] = tb; tr += r; tb += b; }
    unsigned long long res = 0;
    if (tr) res = atomicAdd(P.out.cursor, ((unsigned long long)tr << 32) | tb);
    base = res; s_tb = tb;
    if (tr && ((res >> 32) + tr > P.out.row_cap || (res & 0xFFFFFFFFull) + tb > P.out.byte_cap)) { atomicOr(P.out.overflow, 1u); base = ~0ull; }
  }
  __syncthreads();
  if (base == ~0ull) return;                          // block-uniform
  const EmitOut& O = P.out;
  const uint32_t bbase = (uint32_t)(base & 0xFFFFFFFFull), tb = s_tb;
  const uint32_t boff = bbase + wbytes[warp] + (byte_inc - kb);
  // key bytes: staged in shared memory at their position relative to the block's (4 B aligned-down) output offset, then
  // written with coalesced 32-bit stores (was: one scattered byte store per key byte)
  const bool staged = tb <= (uint32_t)EMIT_STAGE;
  const uint32_t abase = bbase & ~3u;
  if (keep && klen) {
    uint8_t* dst = staged ? stage + (boff - abase) : O.key_bytes + boff;
    if (klen <= (uint32_t)INLINE_KEY) {
      const uint64_t w[2] = {gk.k0, gk.k1};
      for (uint32_t i = 0; i < klen; i++) dst[i] = (uint8_t)(w[i >> 3] >> ((i & 7) * 8));
    } else {
      const uint8_t* src = P.dict.arena + gk.k1;
      for (uint32_t i = 0; i < klen; i++) dst[i] = src[i];
    }
  }
  if (staged && tb) {
    __syncthreads();
    const uint32_t lo = bbase - abase, hi = lo + tb;              // staged byte range [lo, hi)
    const uint32_t w0 = (lo + 3u) >> 2, w1 = hi >> 2;              // full words [w0, w1)
    for (uint32_t w = w0 + threadIdx.x; w < w1; w += 256)
      reinterpret_cast<uint32_t*>(O.key_bytes + abase)[w] = reinterpret_cast<const uint32_t*>(stage)[w];
    if (threadIdx.x == 0) {                                        // ragged edges (neighbouring blocks own the other bytes of these words)
      for (uint32_t b = lo; b < min(w0 * 4u, hi); b++) O.key_bytes[abase + b] = stage[b];
      for (uint32_t b = max(w1 * 4u, min(w0 * 4u, hi)); b < hi; b++) O.key_bytes[abase + b] = stage[b];
    }
  }
  if (!keep) return;
  const uint64_t row = (base >> 32) + wrows[warp] + row_pre;
  O.key_off[row] = (int32_t)boff;
  O.key_valid[row] = gk.len != 0xFFFFFFFFu;
  O.count[row] = (long long)c.cnt;
  O.mn[row] = mn; O.mx[row] = mx; O.avg[row] = avg; O.sum[row] = agg_ok ? c.sum : 0.0;
  O.agg_valid[row] = agg_ok;
  O.wstart[row] = P.wstart; O.wend[row] = P.wend;
}

cudaError_t launch_emit(const EmitParams& p, cudaStream_t s) {
  if (!p.n_groups) return cudaSuccess;
  k_emit<<<(p.n_groups + 255) / 256, 256, 0, s>>>(p);
  return cudaGetLastError();
}

// =================================================================================================
// k_ts_convert: the step BEFORE the path -- canonical event time from a raw column, as array_to_timestamp_array does
// (physical_plan/utils/time.rs:59-94).  Thread per row; blockIdx.y = batch.
//   kind 2  Int64 seconds      ts * 1000
//   kind 3  Utf8, chrono format NaiveDateTime::parse_from_str(s, fmt).and_utc().timestamp_millis()
// Supported specifiers: %Y %m %d %H %M %S %f %.f %3f %6f %9f %.3f %.6f %.9f %F %T %% and literals (whitespace in the format
// matches any run of whitespace).  A string that does not match raises the error flag (the reference unwraps and panics).
// =================================================================================================
__device__ __forceinline__ bool ts_digits(const uint8_t* s, int& i, int n, int min_d, int max_d, long long& out) {
  int d = 0; long long v = 0;
  while (d < max_d && i < n && s[i] >= '0' && s[i] <= '9') { v = v * 10 + (s[i] - '0'); i++; d++; }
  out = v;
  return d >= min_d;
}
__device__ bool ts_parse(const uint8_t* s, int n, const TsFormat& F, long long* out_ms) {
  long long Y = 1970, mo = 1, D = 1, H = 0, Mi = 0, S = 0, nanos = 0;
  int i = 0;
  for (int f = 0; f < F.len; f++) {
    const char c = F.fmt[f];
    if (c == ' ' || c == '\t' || c == '\n') { while (i < n && (s[i] == ' ' || s[i] == '\t' || s[i] == '\n')) i++; continue; }
    if (c != '%') { if (i >= n || s[i] != (uint8_t)c) return false; i++; continue; }
    char sp = F.fmt[++f];
    bool dot = false; int fixed = 0;
    if (sp == '.') { dot = true; sp = F.fmt[++f]; }
    if (sp == '3' || sp == '6' || sp == '9') { fixed = sp - '0'; sp = F.fmt[++f]; }
    long long v = 0;
    switch (sp) {
      case 'Y': { bool neg = false; if (i < n && (s[i] == '-' || s[i] == '+')) { neg = s[i] == '-'; i++; } const bool sg = neg || (i > 0 && s[i - 1] == '+'); if (!ts_digits(s, i, n, 1, sg ? 6 : 4, v)) return false; Y = neg ? -v : v; break; }   // chrono: more than 4 year digits need a sign
      case 'm': if (!ts_digits(s, i, n, 1, 2, v) || v < 1 || v > 12) return false; mo = v; break;
      case 'd': if (!ts_digits(s, i, n, 1, 2, v) || v < 1 || v > 31) return false; D = v; break;
      case 'H': if (!ts_digits(s, i, n, 1, 2, v) || v > 23) return false; H = v; break;
      case 'M': if (!ts_digits(s, i, n, 1, 2, v) || v > 59) return false; Mi = v; break;
      case 'S': if (!ts_digits(s, i, n, 1, 2, v) || v > 60) return false; S = v; break;
      case 'f': {
        if (dot) {                                   // %.f / %.3f ...: optional for %.f, fraction of a second
          if (i < n && s[i] == '.') {
            i++;
            int d0 = i;
            if (!ts_digits(s, i, n, fixed ? fixed : 1, fixed ? fixed : 9, v)) return false;
            int nd = i - d0; for (int k = nd; k < 9; k++) v *= 10;
            while (!fixed && i < n && s[i] >= '0' && s[i] <= '9') i++;      // digits beyond nanoseconds are dropped
            nanos = v;
          } else if (fixed) return false;
        } else if (fixed) {                          // %3f / %6f / %9f: exactly that many fraction digits, no dot
          if (!ts_digits(s, i, n, fixed, fixed, v)) return false;
          for (int k = fixed; k < 9; k++) v *= 10;
          nanos = v;
        } else {                                     // %f: NANOSECONDS as a number (up to 9 digits)
          if (!ts_digits(s, i, n, 1, 9, v)) return false;
          nanos = v;
        }
        break;
      }
      case '%': if (i >= n || s[i] != '%') return false; i++; break;
      default: return false;
    }
  }
  if (i != n) return false;                          // trailing input
  // days from civil (proleptic Gregorian), then seconds
  const long long y = mo <= 2 ? Y - 1 : Y;
  const long long era = (y >= 0 ? y : y - 399) / 400;
  const long long yoe = y - era * 400;
  const long long doy = (153 * (mo + (mo > 2 ? -3 : 9)) + 2) / 5 + D - 1;
  const long long doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
  const long long days = era * 146097 + doe - 719468;
  {   // reject dates that do not exist (31 April, 29 February of a common year)
    const bool leap = (Y % 4 == 0 && Y % 100 != 0) || Y % 400 == 0;
    const int mdays[12] = {31, leap ? 29 : 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31};
    if (D > mdays[mo - 1]) return false;
  }
  long long secs = days * 86400 + H * 3600 + Mi * 60 + (S == 60 ? 59 : S);
  if (S == 60) nanos += 1000000000ll;                // chrono keeps the leap second in the nanosecond field
  *out_ms = secs * 1000 + nanos / 1000000;
  return true;
}
__global__ void __launch_bounds__(256) k_ts_convert(const TsJob* __restrict__ jobs, int kind, const __grid_constant__ TsFormat F, uint32_t* error) {
  const TsJob j = jobs[blockIdx.y];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < j.n; i += (int64_t)gridDim.x * blockDim.x) {
    if (kind == 2) { j.dst[i] = reinterpret_cast<const int64_t*>(j.src)[i] * 1000; continue; }
    const int32_t o0 = j.off[i], o1 = j.off[i + 1];
    long long ms = 0;
    if (!ts_parse(j.bytes + o0, o1 - o0, F, &ms)) { atomicOr(error, 1u); ms = 0; }
    j.dst[i] = ms;
  }
}
cudaError_t launch_ts_convert(const TsJob* jobs, int n_jobs, int64_t max_rows, int kind, const TsFormat& fmt, uint32_t* error, cudaStream_t s) {
  if (n_jobs <= 0 || max_rows <= 0) return cudaSuccess;
  const unsigned gx = (unsigned)std::min<int64_t>((max_rows + 255) / 256, 1024);
  for (int j0 = 0; j0 < n_jobs; j0 += 65535) {
    dim3 grid(gx, (unsigned)std::min(n_jobs - j0, 65535));
    k_ts_convert<<<grid, 256, 0, s>>>(jobs + j0, kind, fmt, error);
  }
  return cudaGetLastError();
}
bool ts_format_supported(const char* fmt) {
  if (!fmt) return false;
  const size_t n = strlen(fmt);
  if (n == 0 || n >= (size_t)TS_FMT_MAX) return false;
  for (size_t f = 0; f < n; f++) {
    if (fmt[f] != '%') continue;
    char sp = fmt[++f];
    if (sp == '.') sp = fmt[++f];
    if (sp == '3' || sp == '6' || sp == '9') { sp = fmt[++f]; if (sp != 'f') return false; }
    if (!strchr("YmdHMSf%", sp) || sp == 0) return false;
  }
  return true;
}

// =================================================================================================
// small utilities
// =================================================================================================
__global__ void k_fill_u64(unsigned long long* p, uint64_t n, unsigned long long v) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}
cudaError_t launch_fill_u64(unsigned long long* p, uint64_t n, unsigned long long v, cudaStream_t s) {
  if (!n) return cudaSuccess;
  uint64_t gb = (n + 255) / 256; int grid = (int)(gb < 148 * 16 ? gb : 148 * 16);
  k_fill_u64<<<grid, 256, 0, s>>>(p, n, v);
  return cudaGetLastError();
}

// Host-pinned -> device gather copy.  CTAs claim 256 KiB pieces of the descriptor list dynamically; every thread keeps
// eight 16 B loads from system memory in flight (PCIe reads need ~100 KB outstanding to reach line rate).
__global__ void __launch_bounds__(256) k_gather_copy(const CopyDesc* __restrict__ descs, uint32_t n, unsigned int* cursor) {
  constexpr uint64_t PIECE = COPY_PIECE;
  __shared__ unsigned int s_desc; __shared__ unsigned long long s_skip;
  const uint64_t total = descs[n - 1].first_piece + (descs[n - 1].bytes + PIECE - 1) / PIECE;
  for (;;) {
    if (threadIdx.x == 0) {
      unsigned int piece = atomicAdd(cursor, 1u);
      uint32_t lo = 0, hi = n - 1;                       // last descriptor whose first_piece <= piece
      if (piece >= total) lo = n;
      else while (lo < hi) { uint32_t mid = (lo + hi + 1) >> 1; if (descs[mid].first_piece <= piece) lo = mid; else hi = mid - 1; }
      s_desc = lo; s_skip = lo < n ? piece - descs[lo].first_piece : 0;
    }
    __syncthreads();
    const uint32_t d = s_desc; const uint64_t skip = s_skip;
    __syncthreads();
    if (d >= n) return;
    const CopyDesc cd = descs[d];
    uint64_t off = skip * PIECE, end = min(cd.bytes, off + PIECE);
    const char* src = (const char*)cd.src; char* dst = (char*)cd.dst;
    if (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0) {
      uint64_t nvec = (end - off) >> 4;
      const int4* s4 = reinterpret_cast<const int4*>(src + off); int4* d4 = reinterpret_cast<int4*>(dst + off);
      uint64_t i = threadIdx.x;
      for (; i + 7 * 256 < nvec; i += 8 * 256) {
        int4 v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = __ldcs(s4 + i + k * 256);
#pragma unroll
        for (int k = 0; k < 8; k++) d4[i + k * 256] = v[k];
      }
      for (; i < nvec; i += 256) d4[i] = __ldcs(s4 + i);
      for (uint64_t b = off + (nvec << 4) + threadIdx.x; b < end; b += 256) dst[b] = src[b];
    } else {
      for (uint64_t b = off + threadIdx.x; b < end; b += 256) dst[b] = src[b];
    }
  }
}
cudaError_t launch_gather_copy(const CopyDesc* descs, uint32_t n, unsigned int* cursor, cudaStream_t s) {
  if (!n) return cudaSuccess;
  k_gather_copy<<<64, 256, 0, s>>>(descs, n, cursor);
  return cudaGetLastError();
}

// re-insert every occupied slot of the old table into the (zeroed) new one; group ids are preserved
__global__ void k_dict_rehash(const DictSlot* old_slots, uint32_t old_cap, DictView nd) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < old_cap; i += (uint64_t)gridDim.x * blockDim.x) {
    DictSlot s = old_slots[i];
    if (s.state == SLOT_EMPTY || s.state == SLOT_LOCKED) continue;
    uint64_t h = s.len <= (uint32_t)INLINE_KEY ? hash_inline(s.k0, s.k1, s.len) : s.k0;
    uint32_t idx = (uint32_t)h & nd.mask;
    for (;;) {
      uint32_t old = atomicCAS(&nd.slots[idx].state, SLOT_EMPTY, SLOT_LOCKED);
      if (old == SLOT_EMPTY) break;
      idx = (idx + 1) & nd.mask;
    }
    DictSlot* d = nd.slots + idx;
    d->k0 = s.k0; d->k1 = s.k1; d->hint = s.hint; d->len = s.len;
    __threadfence();
    d->state = s.state;
  }
}
cudaError_t launch_dict_rehash(const DictSlot* old_slots, uint32_t old_cap, DictView nd, cudaStream_t s) {
  uint64_t gb = ((uint64_t)old_cap + 255) / 256; int grid = (int)(gb < 148 * 16 ? gb : 148 * 16);
  k_dict_rehash<<<grid, 256, 0, s>>>(old_slots, old_cap, nd);
  return cudaGetLastError();
}


// checkpoint restore: re-insert the keys of gid_key[0, n) into an EMPTY table with their original group ids
__global__ void k_dict_restore(DictView d, uint32_t n) {
  for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < n; g += gridDim.x * blockDim.x) {
    const GidKey gk = d.gid_key[g];
    if (gk.len == 0xFFFFFFFFu) { *d.null_gid = g + 1; continue; }
    const uint64_t h = gk.len <= (uint32_t)INLINE_KEY ? hash_inline(gk.k0, gk.k1, gk.len) : gk.k0;
    uint32_t idx = (uint32_t)h & d.mask;
    for (;;) {
      if (atomicCAS(&d.slots[idx].state, SLOT_EMPTY, SLOT_LOCKED) == SLOT_EMPTY) break;
      idx = (idx + 1) & d.mask;
    }
    DictSlot* s = d.slots + idx;
    s->k0 = gk.k0; s->k1 = gk.k1; s->hint = 0; s->len = gk.len;
    __threadfence();
    s->state = g + 1;
  }
}
cudaError_t launch_dict_restore(DictView d, uint32_t n, cudaStream_t s) {
  if (!n) return cudaSuccess;
  k_dict_restore<<<(unsigned)std::min<uint64_t>(((uint64_t)n + 255) / 256, 148 * 16), 256, 0, s>>>(d, n);
  return cudaGetLastError();
}

__global__ void k_clear_hints(DictSlot* slots, uint32_t cap) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) slots[i].hint = 0;
}
cudaError_t launch_clear_hints(DictSlot* slots, uint32_t cap, cudaStream_t s) {
  uint64_t gb = ((uint64_t)cap + 255) / 256; int grid = (int)(gb < 148 * 16 ? gb : 148 * 16);
  k_clear_hints<<<grid, 256, 0, s>>>(slots, cap);
  return cudaGetLastError();
}

}  // namespace dnz
