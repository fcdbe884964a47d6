// dnz_device.cuh -- device helpers: PTX wrappers (mbarrier, cp.async.bulk, wide loads, reductions),
// ordered float keys, key loading / hashing, dictionary probe+insert, per-row state update.
#pragma once
#include "dnz_kernels.h"

namespace dnz {

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Releasing a ring slot only has to order the consumer's shared-memory READS of the slot before the producer's refill;
// those reads have completed once their values were used.  The default .release form also waits for every outstanding
// global reduction of the warp (an L2 round trip per tile).
__device__ __forceinline__ void mbar_arrive_relaxed(uint64_t* bar) {
  asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"     // %3: suspend-time hint (ns): park the warp
      "selp.u32 %0, 1, 0, p;\n\t}"                                          // instead of spinning through issue slots
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP.S.G).
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// one 32 B sector in a single request (SASS: LDG.E.256), always served by L2: slots are written by other SMs
// (atomicCAS + release store) while we probe, and the per-SM L1 is not coherent -- an L1-cached copy of an
// EMPTY/LOCKED slot would make the probe loop spin forever.
__device__ __forceinline__ void ld_slot(const DictSlot* p, uint64_t& a, uint64_t& b, uint64_t& c, uint64_t& d) {
  asm volatile("ld.relaxed.gpu.global.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void red_add_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void red_add_f64(double* p, double v) {
  asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void red_max_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("red.global.max.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void red_min_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("red.global.min.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// ---------------------------------------------------------------- ordered float keys
// ord(): monotone map f64 -> u64 over IEEE totalOrder.  min/max accumulators are kept as distances from the
// DataFusion starting values (f64::MAX for min, f64::MIN for max) so that a zero-filled state IS the start.
constexpr unsigned long long SIGN64 = 0x8000000000000000ull;
constexpr unsigned long long BITS_F64_MAX = 0x7FEFFFFFFFFFFFFFull;
constexpr unsigned long long ORD_F64_MAX = BITS_F64_MAX | SIGN64;        // ord(+MAX)
constexpr unsigned long long ORD_F64_MIN = ~(BITS_F64_MAX | SIGN64);     // ord(-MAX)
__host__ __device__ __forceinline__ unsigned long long ord_bits(unsigned long long b) { return (b & SIGN64) ? ~b : (b | SIGN64); }
__host__ __device__ __forceinline__ unsigned long long unord_bits(unsigned long long o) { return (o & SIGN64) ? (o & ~SIGN64) : ~o; }
// The bits of a double through an opaque move.  Given __double_as_longlong(v), nvcc rewrites ord_bits' `b | SIGN64` into the
// floating-point -|v| (DADD), which turns a NaN into the canonical 0x7FFFFFFFFFFFFFFF and so loses it from a totalOrder max.
// Paths whose min / max see NaN take the bits from here.
__device__ __forceinline__ unsigned long long f64_bits(double v) {
  unsigned long long b;
  asm("mov.b64 %0, %1;" : "=l"(b) : "d"(v));
  return b;
}
// IEEE totalOrder key (arrow-ord cmp on floats == f64::total_cmp)
__host__ __device__ __forceinline__ long long total_key(unsigned long long b) {
  long long s = (long long)b; return s ^ (long long)(((unsigned long long)(s >> 63)) >> 1);
}

// ---------------------------------------------------------------- hashing
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x ^= x >> 32; x *= 0xD6E8FEB86659FD93ull; x ^= x >> 32; x *= 0xD6E8FEB86659FD93ull; x ^= x >> 32; return x;
}
// inline keys (<= 16 B, four zero-padded 32-bit words): 32-bit multiply-xorshift chain -- the slot index needs < 30 bits and
// 64-bit multiplies cost 3-4 IMADs each on the hot path
__host__ __device__ __forceinline__ uint32_t hash_words(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t len) {
  // four INDEPENDENT multiplies (they issue back to back), rotated so that the digits of "sensor_123"-style keys land in
  // different bit ranges, summed, then murmur3's 32-bit finaliser: a shorter dependent chain in front of the dictionary
  // probe than a word-by-word chain, same probe lengths in simulation (1.119 vs 1.117 average at 19 % load)
  uint32_t a = w1 * 0xC2B2AE35u, b = w2 * 0x27D4EB2Fu, c = w3 * 0x165667B1u;
  uint32_t h = w0 * 0x85EBCA6Bu + ((a << 13) | (a >> 19)) + ((b << 21) | (b >> 11)) + ((c << 5) | (c >> 27)) + len * 0x9E3779B1u;
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}
__host__ __device__ __forceinline__ uint64_t hash_inline(uint64_t k0, uint64_t k1, uint32_t len) {
  return hash_words((uint32_t)k0, (uint32_t)(k0 >> 32), (uint32_t)k1, (uint32_t)(k1 >> 32), len);
}

// A key as the dictionary sees it.
struct KeyRef {
  uint64_t k0, k1;       // inline words (long keys: k0 = hash of all bytes)
  uint64_t hash;
  uint32_t len;
  const uint8_t* ptr;    // original bytes (needed only for long keys)
};

// Load up to 16 key bytes from an arbitrarily aligned address using aligned 32-bit loads.
// Reading the aligned words that contain the first / last key byte never leaves their 4 B word, so it is
// safe for both shared and global memory.
template <bool SHARED>
__device__ __forceinline__ uint32_t ld_word(const uint8_t* p) {
  if (SHARED) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p))); return v; }
  return __ldg(reinterpret_cast<const uint32_t*>(p));
}
template <bool SHARED>
__device__ __forceinline__ void load_key(const uint8_t* p, uint32_t len, KeyRef& k) {
  k.len = len; k.ptr = p;
  if (len <= (uint32_t)INLINE_KEY) {
    uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3u);
    const uint8_t* q = p - mis;
    uint32_t nw = (mis + len + 3u) >> 2;            // aligned words holding the key (<= 5)
    uint32_t a[5];
#pragma unroll
    for (int i = 0; i < 5; i++) a[i] = (uint32_t)i < nw ? ld_word<SHARED>(q + 4 * i) : 0u;
    uint32_t w[4];
    uint32_t sh = mis * 8u;
#pragma unroll
    for (int i = 0; i < 4; i++) w[i] = __funnelshift_r(a[i], i < 4 ? a[i + 1] : 0u, sh);
#pragma unroll
    for (int i = 0; i < 4; i++) {                    // zero the bytes past len
      uint32_t lo = 4u * i;
      uint32_t keep = len <= lo ? 0u : (len - lo >= 4u ? 0xFFFFFFFFu : ((1u << ((len - lo) * 8u)) - 1u));
      w[i] &= keep;
    }
    k.k0 = (uint64_t)w[0] | ((uint64_t)w[1] << 32); k.k1 = (uint64_t)w[2] | ((uint64_t)w[3] << 32);
    k.hash = hash_inline(k.k0, k.k1, len);
  } else {
    // long key: two 32-bit multiply-xorshift lanes over its little-endian 32-bit words (aligned loads + funnel shifts; the
    // byte-at-a-time version cost ~250 instructions for a 36 B UUID and was the whole kernel for such streams)
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3u), sh = mis * 8u;
    const uint8_t* q = p - mis;
    const uint32_t nk = (len + 3u) >> 2, nw = (mis + len + 3u) >> 2;
    uint32_t h1 = 0x9E3779B1u * (len + 1u), h2 = 0x85EBCA77u ^ len;
    uint32_t prev = ld_word<SHARED>(q);
    for (uint32_t i = 0; i < nk; i++) {
      const uint32_t next = (i + 1u < nw) ? ld_word<SHARED>(q + 4u * (i + 1u)) : 0u;
      uint32_t w = __funnelshift_r(prev, next, sh);
      prev = next;
      if (i + 1u == nk && (len & 3u)) w &= (1u << ((len & 3u) * 8u)) - 1u;
      h1 = (h1 ^ w) * 0x85EBCA6Bu; h1 ^= h1 >> 15;
      h2 = (h2 + w) * 0xC2B2AE3Du; h2 = (h2 << 13) | (h2 >> 19);
    }
    h1 ^= h2 * 0x27D4EB2Fu; h1 ^= h1 >> 16; h1 *= 0x165667B1u; h1 ^= h1 >> 13;
    h2 ^= h1 * 0x9E3779B1u; h2 ^= h2 >> 15; h2 *= 0x85EBCA6Bu; h2 ^= h2 >> 16;
    const uint64_t h = ((uint64_t)h2 << 32) | h1;
    k.k0 = h; k.k1 = 0; k.hash = h;
  }
}

__device__ __forceinline__ uint8_t ld_key_byte(const uint8_t* p, bool shared) {
  if (shared) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(smem_u32(p))); return (uint8_t)v; }
  return __ldg(p);
}

// ---------------------------------------------------------------- dictionary
enum : uint32_t { GID_DEFER_GROUPS = 0xFFFFFFFEu, GID_DEFER_ARENA = 0xFFFFFFFDu };

// Try to claim `slot` for key k.  Returns gid, or GID_DEFER_* when a table is full, or 0xFFFFFFFF when the CAS was
// lost (caller re-examines the slot).
__device__ __forceinline__ uint32_t dict_try_insert(const DictView& d, DictSlot* slot, uint32_t slot_idx, const KeyRef& k,
                                                   bool key_shared) {
  unsigned long long arena_off = 0;
  if (k.len > (uint32_t)INLINE_KEY) {                // reserve arena space first (a lost race leaks a few bytes)
    unsigned long long need = (k.len + 7ull) & ~7ull;
    arena_off = atomicAdd(d.arena_used, need);
    if (arena_off + need > d.arena_cap) return GID_DEFER_ARENA;
  }
  uint32_t old = atomicCAS(&slot->state, SLOT_EMPTY, SLOT_LOCKED);
  if (old != SLOT_EMPTY) return 0xFFFFFFFFu;
  // group id: one atomicAdd (a CAS loop on this single counter serialises every inserter on the chip).  The counter may
  // run past gcap; ids >= gcap are never used (the rows are deferred) and the host clamps the counter before it grows.
  uint32_t g = atomicAdd(d.n_groups, 1u);
  if (g >= d.gcap) { st_release_u32(&slot->state, SLOT_EMPTY); return GID_DEFER_GROUPS; }
  if (k.len > (uint32_t)INLINE_KEY) {
    for (uint32_t i = 0; i < k.len; i++) d.arena[arena_off + i] = ld_key_byte(k.ptr + i, key_shared);
    slot->k0 = k.k0; slot->k1 = arena_off;
  } else {
    slot->k0 = k.k0; slot->k1 = k.k1;
  }                                                  // slot->hint stays 0 (= no hint) from the zero fill
  slot->len = k.len;
  d.gid_key[g] = GidKey{k.k0, k.len > (uint32_t)INLINE_KEY ? arena_off : k.k1, k.len, 0u};
  atomicAdd(d.key_bytes_total, (unsigned long long)k.len);
  __threadfence();
  st_release_u32(&slot->state, g + 1);
  return g;
}

__device__ __forceinline__ bool dict_long_equal(const DictView& d, uint64_t arena_off, const KeyRef& k, bool key_shared) {
  // word-wise; arena entries are 8 B aligned.  __ldcg: arena bytes of OTHER keys sharing an L1 sector may have been cached
  // before this key was written
  const uint32_t* aw = reinterpret_cast<const uint32_t*>(d.arena + arena_off);
  const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(k.ptr) & 3u), sh = mis * 8u;
  const uint8_t* q = k.ptr - mis;
  const uint32_t nk = (k.len + 3u) >> 2, nw = (mis + k.len + 3u) >> 2;
  uint32_t prev = key_shared ? ld_word<true>(q) : ld_word<false>(q);
  for (uint32_t i = 0; i < nk; i++) {
    const uint32_t next = (i + 1u < nw) ? (key_shared ? ld_word<true>(q + 4u * (i + 1u)) : ld_word<false>(q + 4u * (i + 1u))) : 0u;
    uint32_t w = __funnelshift_r(prev, next, sh), a = __ldcg(aw + i);
    prev = next;
    if (i + 1u == nk && (k.len & 3u)) { const uint32_t m = (1u << ((k.len & 3u) * 8u)) - 1u; w &= m; a &= m; }
    if (w != a) return false;
  }
  return true;
}

// Examine one slot.  Returns: gid (found or inserted) / GID_DEFER_* / 0xFFFFFFFF = keep probing.
// `advance` is set when the probe must move to the next slot (occupied by a different key).
__device__ __forceinline__ uint32_t dict_step(const DictView& d, uint32_t idx, const KeyRef& k, bool key_shared, bool& advance) {
  DictSlot* slot = d.slots + idx;
  uint64_t a, b, hint, w3;
  ld_slot(slot, a, b, hint, w3);
  uint32_t len = (uint32_t)w3, state = (uint32_t)(w3 >> 32);
  advance = false;
  if (state == SLOT_EMPTY) {
    uint32_t g = dict_try_insert(d, slot, idx, k, key_shared);
    return g;                                  // 0xFFFFFFFF: lost the race -> re-read the same slot
  }
  if (state == SLOT_LOCKED) return 0xFFFFFFFFu;  // insert in flight -> re-read
  bool eq;
  if (k.len <= (uint32_t)INLINE_KEY) eq = (len == k.len) && a == k.k0 && b == k.k1;
  else eq = (len == k.len) && a == k.k0 && dict_long_equal(d, b, k, key_shared);
  if (eq) return state - 1;
  advance = true;
  return 0xFFFFFFFFu;
}

__device__ __forceinline__ uint32_t dict_lookup_null(const DictView& d) {
  for (;;) {
    uint32_t s = ld_acquire_u32(d.null_gid);
    if (s != 0 && s != SLOT_LOCKED) return s - 1;
    if (s == 0) {
      uint32_t old = atomicCAS(d.null_gid, 0u, SLOT_LOCKED);
      if (old != 0) continue;
      uint32_t g = atomicAdd(d.n_groups, 1u);
      if (g >= d.gcap) { st_release_u32(d.null_gid, 0u); return GID_DEFER_GROUPS; }
      d.gid_key[g] = GidKey{0ull, 0ull, 0xFFFFFFFFu, 0u};
      __threadfence();
      st_release_u32(d.null_gid, g + 1);
      return g;
    }
  }
}

// full lookup (used by the generic / deferred / merge paths and by the staged kernel's slow path)
__device__ __forceinline__ uint32_t dict_lookup(const DictView& d, const KeyRef& k, bool key_shared, uint32_t* slot_out = nullptr) {
  uint32_t idx = (uint32_t)k.hash & d.mask;
  for (;;) {
    bool adv;
    uint32_t g = dict_step(d, idx, k, key_shared, adv);
    if (g != 0xFFFFFFFFu) { if (slot_out) *slot_out = idx; return g; }
    if (adv) idx = (idx + 1) & d.mask;
    else __nanosleep(100);      // slot locked by an insert in flight (possibly by another lane of this warp): let it finish
  }
}

// ---------------------------------------------------------------- per-row accumulator update
// DataFusion-42 semantics (SURVEY.md §8a-5): count += 1 per non-null value; min: `if cur > v`, max: `if cur < v`
// from f64::MAX / f64::MIN (NaN never replaces, +inf never lowers min's start, -inf never raises max's start,
// the first +-0.0 wins); avg = sum / count.
__device__ __forceinline__ bool value_needs_fz(double v) { return v == 0.0; }

__device__ __forceinline__ void state_update(GroupState* st, unsigned long long* fz, uint32_t gid, double v,
                                             unsigned long long rowseq) {
  GroupState* s = st + gid;
  unsigned long long bits = (unsigned long long)__double_as_longlong(v);
  if (v == 0.0) {                      // both zeros order as +0.0; remember which one came first
    red_min_u64(fz + gid, (rowseq << 1) | (bits >> 63));
    bits = 0ull;
  }
  red_add_f64(&s->cnt, 1.0);
  red_add_f64(&s->sum, v);
  unsigned long long o = ord_bits(bits);
  if (v <= 1.7976931348623157e308) red_max_u64(&s->minkey, ORD_F64_MAX - o);    // false for NaN and +inf
  if (v >= -1.7976931348623157e308) red_max_u64(&s->maxkey, o - ORD_F64_MIN);   // false for NaN and -inf
}

__device__ __forceinline__ void defer_row(const DeferList& dl, uint32_t tile, uint32_t row, uint32_t why) {
  atomicOr(dl.flags, why);
  unsigned long long i = atomicAdd(dl.count, 1ull);
  if (i < dl.cap) dl.entries[i] = DeferEntry{tile, row};
  else atomicOr(dl.flags, (uint32_t)DEFER_LIST_OVERFLOW);
}

__device__ __forceinline__ bool bit_at(const uint8_t* bm, int64_t i) { return (__ldg(bm + (i >> 3)) >> (i & 7)) & 1; }

}  // namespace dnz
