// engine.cu -- CUDA kernels (sm_100a) and the C ABI (include/ibft_verify.h) of the batched verification engine.
//
// Kernels (SURVEY.md §2.2 checklist):
//   k_recover        K1+K2 fused: Keccak-256 of the payload / seal wrap, secp256k1 public-key recovery, address
//                    derivation + compare with msg.From / seal.Signer, validator-set membership, warp-ballot of the
//                    32 verdicts of a warp into one word of the pass/fail bitmap.
//   k_quorum_mark /  K3: resolve every passing item's signer to its validator index and OR it into the group's voted
//   k_quorum_reduce  set; then per group: distinct count, 320-bit weighted voting-power sum, >= quorum threshold
//                    (reference core/validator_manager.go:77-96, :130-135).
//   k_keccak_batch   hash-only batch for IsValidProposalHash (reference core/backend.go:50-51).
// There is no CPU fallback anywhere in this file: without a CUDA device ibft_engine_create fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/ibft_verify.h"
#include "verify_core.cuh"

#include "secp_gtable.inc"

using namespace ibft;

static_assert(sizeof(ibft_sig_item) == 128, "packed item must be 128 bytes");
static_assert(sizeof(ibft_group_desc) == 16, "group descriptor must be 16 bytes");
static_assert(IBFT_GTABLE_WG == IBFT_WG, "regenerate secp_gtable.inc (tools/gen_tables.py) for this IBFT_WG");

#define IBFT_BLOCK 128
#ifndef IBFT_GTAB_SMEM
#define IBFT_GTAB_SMEM (IBFT_WG <= 8 && IBFT_WC == 0)  // with a combined table the recover kernel never reads the small one
#endif
#define IBFT_ITEM_ROW_WORDS 33  // 128-byte item + 1 pad word: conflict-free per-thread reads from shared memory

// ------------------------------------------------------------------------------------------------------------
// device-side tables
// ------------------------------------------------------------------------------------------------------------
__device__ uint32_t g_gtable[IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES];  // filled from IBFT_GTABLE at engine creation

struct slot_dev {
  const uint32_t* keys;    // n x 6 words: address as 5 big-endian words (sorted ascending) + validator index
  const uint64_t* powers;  // n x 4 little-endian limbs, validator-index order
  uint64_t quorum[5];      // floor(2*total/3) + 1
  uint32_t n;
  uint32_t valid;
  // key registry (engine flag IBFT_FLAG_KEY_CACHE; all nullptr otherwise), validator-index order:
  uint32_t* key_state;     // 0 = unknown, 1 = key learned from a successful recovery, 3 = table being built, 2 = comb table built
  uint32_t* key_xy;        // n x 16 words: affine public key
  uint32_t* key_tab;       // n x IBFT_KEYTAB_WORDS: per validator 17 comb positions x 128 entries x 16 words, affine (build_keytab_pos)
  uint32_t* learn_count;   // number of keys learned so far (the host compares it with the number of tables built)
};
#define IBFT_KEY_UNKNOWN 0u
#define IBFT_KEY_LEARNED 1u
#define IBFT_KEY_READY 2u
#define IBFT_KEY_BUILDING 3u  // claimed by a table-build pass (refresh_key_tables_locked)

__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

// binary search of a 20-byte address in a slot's sorted key table; returns validator index or -1
__device__ int lookup_validator(const slot_dev& s, const uint8_t* addr) {
  uint32_t a[5];
#pragma unroll
  for (int i = 0; i < 5; i++)
    a[i] = ((uint32_t)addr[4 * i] << 24) | ((uint32_t)addr[4 * i + 1] << 16) | ((uint32_t)addr[4 * i + 2] << 8) | addr[4 * i + 3];
  int lo = 0, hi = (int)s.n - 1;
  while (lo <= hi) {
    int mid = (lo + hi) >> 1;
    const uint32_t* k = s.keys + 6 * (size_t)mid;
    int cmp = 0;
#pragma unroll
    for (int i = 0; i < 5; i++) {
      uint32_t kv = __ldg(k + i);
      if (cmp == 0 && kv != a[i]) cmp = kv < a[i] ? -1 : 1;
    }
    if (cmp == 0) return (int)__ldg(k + 5);
    if (cmp < 0) lo = mid + 1; else hi = mid - 1;
  }
  return -1;
}

struct group_dev {
  uint32_t voted_off;  // word offset of the group's voted set
  uint32_t n_words;
};

// Where a recover kernel may record a VALID item's vote right away (K2 + the marking half of K3 fused): the group's voted
// set and valid count.  voted == nullptr: no fused marking (device-resident / sharded callers run k_quorum_mark themselves).
struct vote_sink {
  uint32_t* voted;
  uint32_t* n_valid;
  const group_dev* gdev;
};

// validator-set membership at the message's height (reference core/backend.go:44).  Returns false when the item can never
// get verdict 1 (unknown group, unset table, signer not in the set); *v_out = validator index, or -1 when the group has no
// table (IBFT_NO_TABLE) or no groups were given.
__device__ __forceinline__ bool group_member(const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
                                             const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t group,
                                             const uint8_t* signer, int* v_out, uint32_t* slot_out) {
  *v_out = -1;
  *slot_out = IBFT_NO_TABLE;
  if (groups == nullptr) return true;
  if (group >= n_groups) return false;
  uint32_t slot = groups[group].table_slot;
  if (slot == IBFT_NO_TABLE) return true;
  if (slot >= n_slots || !slots[slot].valid) return false;
  int v = lookup_validator(slots[slot], signer);
  if (v < 0) return false;
  *v_out = v;
  *slot_out = slot;
  return true;
}
// the vote of a valid item: same effect as k_quorum_mark on this item
__device__ __forceinline__ void record_vote(const vote_sink& sink, const ibft_group_desc* __restrict__ groups, uint32_t group, int v) {
  if (groups == nullptr || sink.voted == nullptr) return;
  atomicAdd(&sink.n_valid[group], 1u);
  if (v >= 0) atomicOr(&sink.voted[sink.gdev[group].voted_off + ((uint32_t)v >> 5)], 1u << (v & 31));
}
// membership + vote for an item whose signature verified (the latency kernels look the signer up at the end)
__device__ __forceinline__ bool member_and_vote(const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
                                                const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t group,
                                                const uint8_t* signer, const vote_sink& sink, bool record, int* v_out = nullptr,
                                                uint32_t* slot_out = nullptr) {
  int v;
  uint32_t slot;
  bool ok = group_member(groups, n_groups, slots, n_slots, group, signer, &v, &slot);
  if (v_out) *v_out = v;
  if (slot_out) *slot_out = slot;
  if (ok && record) record_vote(sink, groups, group, v);
  return ok;
}
// key registry: remember the public key a successful recovery produced for validator v (first writer wins; concurrent
// writers store the same key)
__device__ __forceinline__ void learn_key(const slot_dev* __restrict__ slots, uint32_t slot, int v, const aff& K) {
  if (slot == IBFT_NO_TABLE || v < 0) return;
  const slot_dev& s = slots[slot];
  if (s.key_state == nullptr || s.key_state[v] != IBFT_KEY_UNKNOWN) return;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    s.key_xy[16 * (size_t)v + i] = K.x.v[i];
    s.key_xy[16 * (size_t)v + 8 + i] = K.y.v[i];
  }
  __threadfence();
  if (atomicCAS(&s.key_state[v], IBFT_KEY_UNKNOWN, IBFT_KEY_LEARNED) == IBFT_KEY_UNKNOWN) atomicAdd(s.learn_count, 1u);
}

// ------------------------------------------------------------------------------------------------------------
// K1 + K2: recover kernel.  One thread per signature; a warp's 32 verdicts become one bitmap word.
// ------------------------------------------------------------------------------------------------------------
#ifndef IBFT_MIN_BLOCKS
#define IBFT_MIN_BLOCKS 3
#endif
// BLOCK = 128 for throughput (12 resident warps/SM at 166 registers); BLOCK = 32 for latency-critical small batches (a
// 10k-validator COMMIT round is only 313 warps: one-warp CTAs spread them over all 148 SMs instead of 79).
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK, (IBFT_MIN_BLOCKS * IBFT_BLOCK) / BLOCK)
k_recover(const ibft_sig_item* __restrict__ items, uint32_t n, const uint8_t* __restrict__ arena, size_t arena_len,
          uint32_t shard_lo, uint32_t shard_hi, const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
          const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t* __restrict__ bitmap,
          uint8_t* __restrict__ recovered, uint8_t* __restrict__ status, const uint32_t* __restrict__ ctable, vote_sink sink,
          const uint32_t* __restrict__ list) {
  // list != nullptr: WORKLIST mode (second pass of the key-registry path): list[0] = count, list[1..] = item indices that the
  // verify pass could not decide; the items are gathered, verdict bits are OR-ed into the bitmap the first pass wrote.
#if IBFT_GTAB_SMEM
  __shared__ uint32_t s_gtab[IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES];
#else
  const uint32_t* s_gtab = g_gtable;  // the table stays in global memory (L1/L2 resident)
#endif
  // Dynamic shared memory, BLOCK x 128 words, used twice: first as the staging area of the CTA's packed tuples (33-word
  // rows), then -- once every thread holds its tuple in registers -- as the per-signature tables {1..8}*R (thread-interleaved).
  extern __shared__ uint32_t s_rtab[];
  uint32_t* s_items = s_rtab;
  const uint32_t tid = threadIdx.x;
#if IBFT_GTAB_SMEM
  // stage the generator window table (shared by every signature of the CTA)
  for (uint32_t i = tid; i < IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES; i += BLOCK) s_gtab[i] = g_gtable[i];
#endif
  // stage this CTA's 128 packed tuples with coalesced 16-byte loads
  const uint32_t base = shard_lo + blockIdx.x * BLOCK;
  if (list == nullptr) {
    const uint4* src = reinterpret_cast<const uint4*>(items + base);
    uint32_t avail = base < shard_hi ? min((uint32_t)BLOCK, shard_hi - base) : 0u;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      uint32_t q = tid + k * BLOCK;  // uint4 index within the CTA's tuple block
      uint32_t row = q >> 3, col = q & 7;
      if (row < avail) {
        uint4 v = __ldg(src + q);
        uint32_t* d = s_items + row * IBFT_ITEM_ROW_WORDS + col * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
      }
    }
  }
  __syncthreads();
  uint32_t idx = base + tid;
  bool active = idx < shard_hi;
  bool ok = false;
  ibft_sig_item it;
  if (list == nullptr) {
    uint32_t* w = reinterpret_cast<uint32_t*>(&it);
    const uint32_t* s = s_items + tid * IBFT_ITEM_ROW_WORDS;
#pragma unroll
    for (int i = 0; i < 32; i++) w[i] = s[i];
  } else {
    const uint32_t t = blockIdx.x * BLOCK + tid;
    active = t < list[0];
    idx = active ? list[1 + t] : 0u;
    const uint4* src = reinterpret_cast<const uint4*>(items + idx);
    uint4* w = reinterpret_cast<uint4*>(&it);
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = __ldg(src + i);
  }
  __syncthreads();  // the staging area becomes the R tables from here on
  if (active) {
    uint8_t addr[20];
#pragma unroll
    for (int i = 0; i < 20; i++) addr[i] = 0;
    resolved_item ri;
    bool have = false;
    IBFT_STAGE(0);
    int st = resolve_item(it, arena, arena_len, ri, &have);  // raw frames are parsed here (IBFT_KIND_WIRE*)
    if (status != nullptr && list == nullptr) status[idx] = (uint8_t)st;
    gtab_view G{s_gtab};
    G.comb = ctable;
    rtab_view T{s_rtab + tid, (uint32_t)BLOCK};
    // the signer is looked up FIRST: an item of an unknown group / a non-member can never get verdict 1 (its signature is
    // still recovered when the caller asked for the recovered addresses)
    int v = -1;
    uint32_t slot = IBFT_NO_TABLE;
    const bool member = have && group_member(groups, n_groups, slots, n_slots, it.group, ri.signer, &v, &slot);
    if (have && (member || recovered != nullptr)) {
      aff K;
      bool rec = ecrecover_address(ri.r, ri.s, ri.v, ri.z, G, T, addr, &K);
      if (!rec) {
#pragma unroll
        for (int i = 0; i < 20; i++) addr[i] = 0;
      }
      ok = rec && member;
#pragma unroll
      for (int i = 0; i < 20; i++) ok = ok && (addr[i] == ri.signer[i]);
      if (ok) learn_key(slots, slot, v, K);
    }
    if (ok) record_vote(sink, groups, it.group, v);
    if (recovered != nullptr) {
#pragma unroll
      for (int i = 0; i < 20; i++) recovered[(size_t)idx * 20 + i] = addr[i];
    }
    if (list != nullptr && ok) atomicOr(&bitmap[idx >> 5], 1u << (idx & 31u));
  }
  if (list != nullptr) return;
  // warp-ballot reduction of the 32 verdicts into one bitmap word (shard bounds are multiples of 32)
  uint32_t word = __ballot_sync(0xFFFFFFFFu, ok);
  if ((tid & 31) == 0 && idx < shard_hi) bitmap[idx >> 5] = word;
}

#if IBFT_WC > 0
// ------------------------------------------------------------------------------------------------------------
// Key-registry path, first pass (engine flag IBFT_FLAG_KEY_CACHE, throughput regime): one thread per signature; a signature
// whose signer's key table is ready is VERIFIED against the key (verify_core.cuh ecdsa_verify_known).  Whatever this pass
// cannot accept -- key not known yet, or the verification rejected -- goes to the worklist and is decided by the recover
// path in a second, dense launch of k_recover (so a warp never walks both window loops, and every verdict is the recover
// path's verdict).  Items that can never be valid (malformed, unknown group, signer not in the set) are settled here.
// ------------------------------------------------------------------------------------------------------------
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK, (IBFT_MIN_BLOCKS * IBFT_BLOCK) / BLOCK)
k_verify_known(const ibft_sig_item* __restrict__ items, uint32_t n, const uint8_t* __restrict__ arena, size_t arena_len,
               uint32_t shard_lo, uint32_t shard_hi, const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
               const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t* __restrict__ bitmap,
               uint8_t* __restrict__ status, const uint32_t* __restrict__ ctable, vote_sink sink, uint32_t* __restrict__ worklist) {
  __shared__ uint32_t s_items[BLOCK * IBFT_ITEM_ROW_WORDS];
  const uint32_t tid = threadIdx.x;
  const uint32_t base = shard_lo + blockIdx.x * BLOCK;
  {
    const uint4* src = reinterpret_cast<const uint4*>(items + base);
    uint32_t avail = base < shard_hi ? min((uint32_t)BLOCK, shard_hi - base) : 0u;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      uint32_t q = tid + k * BLOCK;
      uint32_t row = q >> 3, col = q & 7;
      if (row < avail) {
        uint4 v = __ldg(src + q);
        uint32_t* d = s_items + row * IBFT_ITEM_ROW_WORDS + col * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
      }
    }
  }
  __syncthreads();
  const uint32_t idx = base + tid;
  bool ok = false;
  if (idx < shard_hi) {
    ibft_sig_item it;
    {
      uint32_t* w = reinterpret_cast<uint32_t*>(&it);
      const uint32_t* s = s_items + tid * IBFT_ITEM_ROW_WORDS;
#pragma unroll
      for (int i = 0; i < 32; i++) w[i] = s[i];
    }
    resolved_item ri;
    bool have = false;
    int st = resolve_item(it, arena, arena_len, ri, &have);
    if (status != nullptr) status[idx] = (uint8_t)st;
    int v = -1;
    uint32_t slot = IBFT_NO_TABLE;
    const bool member = have && group_member(groups, n_groups, slots, n_slots, it.group, ri.signer, &v, &slot);
    if (member) {
      bool ready = v >= 0 && slots[slot].key_state != nullptr && slots[slot].key_state[v] == IBFT_KEY_READY;
      if (ready) {
        gtab_view G{g_gtable};
        G.comb = ctable;
        gtab_view Qt{slots[slot].key_tab + (size_t)v * IBFT_KEYTAB_WORDS};
        ok = ecdsa_verify_known(ri, G, Qt);
      }
      if (ok) record_vote(sink, groups, it.group, v);
      else worklist[1 + atomicAdd(&worklist[0], 1u)] = idx;  // key unknown, or rejected: the recover pass decides (the host
                                                             // only takes this path when the shard fits the worklist)
    }
  }
  uint32_t word = __ballot_sync(0xFFFFFFFFu, ok);
  if ((tid & 31) == 0 && idx < shard_hi) bitmap[idx >> 5] = word;
}
#endif

// ------------------------------------------------------------------------------------------------------------
// K1 + K2, latency variant: FOUR LANES PER SIGNATURE.  A 10k-validator COMMIT round is one wave of independent serial
// chains on the throughput kernel (~5.4k dependent field multiplications each); here the quad's lanes share each chain --
// every lane holds the full state, the up-to-four independent products of a group-law level go one per lane and come back
// through shared memory (secp_ec.cuh, exec_quad).  Everything outside the double-scalar multiplication (Keccak, sqrt,
// inversions) is simply replicated: the kernel does ~4x the work of k_recover and is only used when the batch is too small
// to fill the machine anyway.  CTA = 128 threads = 32 signatures = one bitmap word.
// ------------------------------------------------------------------------------------------------------------
#define IBFT_QUAD_SIGS 32
__global__ void __launch_bounds__(4 * IBFT_QUAD_SIGS, 2)
k_recover_quad(const ibft_sig_item* __restrict__ items, uint32_t n, const uint8_t* __restrict__ arena, size_t arena_len,
               uint32_t shard_lo, uint32_t shard_hi, const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
               const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t* __restrict__ bitmap,
               uint8_t* __restrict__ recovered, uint8_t* __restrict__ status, const uint32_t* __restrict__ ctable, vote_sink sink) {
  __shared__ uint32_t s_items[IBFT_QUAD_SIGS * IBFT_ITEM_ROW_WORDS];
  __shared__ uint32_t s_rtab[IBFT_QUAD_SIGS * IBFT_QTAB_WORDS];  // projective (XYZZ) tables {1..8}*R
  __shared__ uint4 s_xb[4 * 4 * IBFT_QUAD_SIGS];  // exec_quad's product exchange buffer (2 parities x 2 halves per thread)
  __shared__ uint32_t s_word;
  const uint32_t tid = threadIdx.x;
  const uint32_t q = tid >> 2;  // signature within the CTA
  const uint32_t base = shard_lo + blockIdx.x * IBFT_QUAD_SIGS;
  {
    const uint4* src = reinterpret_cast<const uint4*>(items + base);
    uint32_t avail = base < shard_hi ? min((uint32_t)IBFT_QUAD_SIGS, shard_hi - base) : 0u;
#pragma unroll
    for (int k = 0; k < 2; k++) {
      uint32_t u = tid + k * 4 * IBFT_QUAD_SIGS;  // uint4 index within the CTA's tuple block (32 tuples x 8)
      uint32_t row = u >> 3, col = u & 7;
      if (row < avail) {
        uint4 v = __ldg(src + u);
        uint32_t* d = s_items + row * IBFT_ITEM_ROW_WORDS + col * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
      }
    }
    if (tid == 0) s_word = 0;
  }
  __syncthreads();
  const uint32_t idx = base + q;
  bool ok = false;
  if (idx < shard_hi) {  // uniform over the quad
    ibft_sig_item it;
    {
      uint32_t* w = reinterpret_cast<uint32_t*>(&it);
      const uint32_t* s = s_items + q * IBFT_ITEM_ROW_WORDS;
#pragma unroll
      for (int i = 0; i < 32; i++) w[i] = s[i];
    }
    exec_quad ex;
    ex.role = (int)(tid & 3u);
    ex.mask = 0xFu << (tid & 28u);
    ex.xb = s_xb;
    ex.par = 0;
    uint8_t addr[20];
    resolved_item ri;
    bool have = false;
    IBFT_STAGE(0);
    int st = resolve_item(it, arena, arena_len, ri, &have);
    gtab_view G{g_gtable};
    G.comb = ctable;
    rtab_view T{s_rtab + q, (uint32_t)IBFT_QUAD_SIGS};
    aff K;
    bool rec = have && ecrecover_address_x(ex, ri.r, ri.s, ri.v, ri.z, G, T, addr, &K);
    if (!rec) {
#pragma unroll
      for (int i = 0; i < 20; i++) addr[i] = 0;
    }
    ok = rec;
#pragma unroll
    for (int i = 0; i < 20; i++) ok = ok && (addr[i] == ri.signer[i]);
    int vi = -1;
    uint32_t vslot = IBFT_NO_TABLE;
    if (ok) ok = member_and_vote(groups, n_groups, slots, n_slots, it.group, ri.signer, sink, ex.leader(), &vi, &vslot);
    if (ok && ex.leader()) learn_key(slots, vslot, vi, K);
    if (ex.leader()) {
      if (status != nullptr) status[idx] = (uint8_t)st;
      if (recovered != nullptr) {
#pragma unroll
        for (int i = 0; i < 20; i++) recovered[(size_t)idx * 20 + i] = addr[i];
      }
      if (ok) atomicOr(&s_word, 1u << q);
    }
  }
  __syncthreads();
  if (tid == 0 && base < shard_hi) bitmap[base >> 5] = s_word;
}

#if IBFT_WC > 0
// ------------------------------------------------------------------------------------------------------------
// K1 + K2, mid-size latency variant: CHAIN warps + one HELPER warp per CTA, one CTA per SM, one warp per scheduler.
// A 10k-validator COMMIT round is 313 warps on the one-thread kernel -- 279 of the 592 schedulers idle while every busy one
// walks the whole serial chain.  Here CTA = 3 chain warps (96 signatures, one per lane) + 1 helper warp that serves all
// three: the helper takes the digest, r^-1, the GLV splits, the square root and u1*G (a comb without doublings) off the
// chain, which only computes u2*R -- on an isomorphic curve, so that it does not have to wait for the root (verify_core.cuh,
// "Split pipeline").  Hand-off through shared memory and named barriers (bar.arrive by the helper, bar.sync by the chain).
// Capacity of one wave: SMs x 96 signatures (14,208 on a B200).
// ------------------------------------------------------------------------------------------------------------
#define IBFT_SPLIT_CHAINS 3
#define IBFT_SPLIT_SIGS (32 * IBFT_SPLIT_CHAINS)
#define IBFT_SLOT_WORDS 28  // [0..4] |k1|, [5..9] |k2| of u2, [10] phase-1 flags, [11..18] y then gx, [19..26] gy, [27] phase-2 flags
                            // (the two phases have their own flag words: the helper may post phase 2 before a chain warp has
                            // read phase 1 -- same bits either way, but two words keep the hand-off free of unordered accesses)
#define IBFT_SPLIT_SMEM ((IBFT_SPLIT_SIGS * (IBFT_ITEM_ROW_WORDS + IBFT_RTAB_WORDS + IBFT_SLOT_WORDS + 8)) * 4)
#define IBFT_SF_VALID 1u   // phase 1: (r, s, v) in range, digits posted
#define IBFT_SF_NEG0 2u
#define IBFT_SF_NEG1 4u
#define IBFT_SF_ROOT 8u    // phase 2: r is an abscissa, y posted
#define IBFT_SF_GINF 16u   // phase 2: u1*G is the point at infinity
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

__global__ void __launch_bounds__(32 * (IBFT_SPLIT_CHAINS + 1), 1)
k_recover_split(const ibft_sig_item* __restrict__ items, uint32_t n, const uint8_t* __restrict__ arena, size_t arena_len,
                uint32_t shard_lo, uint32_t shard_hi, const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
                const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t* __restrict__ bitmap,
                uint8_t* __restrict__ recovered, uint8_t* __restrict__ status, const uint32_t* __restrict__ ctable, vote_sink sink) {
  extern __shared__ uint32_t s_dyn[];
  uint32_t* s_items = s_dyn;                                              // 96 packed tuples, 33-word rows
  uint32_t* s_rtab = s_items + IBFT_SPLIT_SIGS * IBFT_ITEM_ROW_WORDS;     // 96 tables {1..8}*phi(R), signature-interleaved
  uint32_t* s_slot = s_rtab + IBFT_SPLIT_SIGS * IBFT_RTAB_WORDS;          // hand-off slots, word w of signature i at [w*96 + i]
  uint32_t* s_y = s_slot + IBFT_SPLIT_SIGS * IBFT_SLOT_WORDS;             // the root y, 8 words per signature, same interleave
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  const uint32_t base = shard_lo + blockIdx.x * IBFT_SPLIT_SIGS;
  {
    const uint4* src = reinterpret_cast<const uint4*>(items + base);
    uint32_t avail = base < shard_hi ? min((uint32_t)IBFT_SPLIT_SIGS, shard_hi - base) : 0u;
#pragma unroll
    for (int k = 0; k < (IBFT_SPLIT_SIGS * 8) / (32 * (IBFT_SPLIT_CHAINS + 1)); k++) {
      uint32_t u = tid + k * 32 * (IBFT_SPLIT_CHAINS + 1);
      uint32_t row = u >> 3, col = u & 7;
      if (row < avail) {
        uint4 v = __ldg(src + u);
        uint32_t* d = s_items + row * IBFT_ITEM_ROW_WORDS + col * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
      }
    }
  }
  __syncthreads();
  gtab_view G{g_gtable};
  G.comb = ctable;
  if (warp == IBFT_SPLIT_CHAINS) {
    // ------------------------------------------------------------------ helper warp: lane l serves signature 32p + l of
    // every chain warp p.  Order of work = order in which the chains need it:
    //   1a  range checks, ONE scalar inversion for the lane's three signatures (Montgomery's trick), digits of u2 -> posted
    //       while the chains are still building their tables;
    //   1b/2 per pass: digest, digits of u1, square root, u1*G comb, affine -> posted long before the chain's loop ends.
    // Between the steps the lane's per-signature state (r, s, then r^-1) is parked in the result area of the hand-off slot,
    // which phase 2 overwrites only after reading it -- nothing big is carried in registers across the passes.
    uint32_t okmask = 0;
    IBFT_ROLLED
    for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
      const uint32_t i = 32 * p + lane, idx = base + i;
      bool have = false;
      if (idx < shard_hi) {
        ibft_sig_item it;
        uint32_t* w = reinterpret_cast<uint32_t*>(&it);
        const uint32_t* src = s_items + i * IBFT_ITEM_ROW_WORDS;
#pragma unroll
        for (int k = 0; k < 32; k++) w[k] = src[k];
        resolved_item ri;
        resolve_item(it, arena, arena_len, ri, &have, false);
        have = have && split_sig_in_range(ri);
        if (have) {
          sc r = sc_from_be(ri.r), sv = sc_from_be(ri.s);
#pragma unroll
          for (int k = 0; k < 8; k++) {
            s_slot[(11 + k) * IBFT_SPLIT_SIGS + i] = r.v[k];
            s_slot[(19 + k) * IBFT_SPLIT_SIGS + i] = sv.v[k];
          }
        }
      }
      if (have) okmask |= 1u << p;
    }
    {
      // prefix products of the valid r's (an invalid one contributes 1), one inversion, peel backwards
      sc one;
#pragma unroll
      for (int k = 0; k < 8; k++) one.v[k] = k == 0;
      sc rr[IBFT_SPLIT_CHAINS], pre[IBFT_SPLIT_CHAINS];
#pragma unroll
      for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
        rr[p] = one;
        if ((okmask >> p) & 1u) {
#pragma unroll
          for (int k = 0; k < 8; k++) rr[p].v[k] = s_slot[(11 + k) * IBFT_SPLIT_SIGS + 32 * p + lane];
        }
        pre[p] = p ? sc_mul(pre[p - 1], rr[p]) : rr[p];
      }
      sc inv = IBFT_SC_INV(pre[IBFT_SPLIT_CHAINS - 1]);
#pragma unroll
      for (int p = IBFT_SPLIT_CHAINS - 1; p >= 0; p--) {
        sc ri = p ? sc_mul(inv, pre[p - 1]) : inv;
        if (p) inv = sc_mul(inv, rr[p]);
#pragma unroll
        for (int k = 0; k < 8; k++) s_slot[(11 + k) * IBFT_SPLIT_SIGS + 32 * p + lane] = ri.v[k];  // r^-1 replaces r
      }
    }
    IBFT_ROLLED
    for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
      const uint32_t i = 32 * p + lane;
      uint32_t flags = 0;
      if ((okmask >> p) & 1u) {
        sc sv, rinv;
#pragma unroll
        for (int k = 0; k < 8; k++) {
          rinv.v[k] = s_slot[(11 + k) * IBFT_SPLIT_SIGS + i];
          sv.v[k] = s_slot[(19 + k) * IBFT_SPLIT_SIGS + i];
        }
        ecmult_digits dg;
        ecmult_split_into(sc_mul(sv, rinv), dg, 0);
        flags = IBFT_SF_VALID | (dg.kneg[0] ? IBFT_SF_NEG0 : 0u) | (dg.kneg[1] ? IBFT_SF_NEG1 : 0u);
#pragma unroll
        for (int k = 0; k < 5; k++) {
          s_slot[k * IBFT_SPLIT_SIGS + i] = dg.ks[0][k];
          s_slot[(5 + k) * IBFT_SPLIT_SIGS + i] = dg.ks[1][k];
        }
      }
      s_slot[10 * IBFT_SPLIT_SIGS + i] = flags;
      __threadfence_block();
      named_bar_arrive(1 + p, 64);
    }
    IBFT_ROLLED
    for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
      const uint32_t i = 32 * p + lane;
      if ((okmask >> p) & 1u) {
        uint32_t flags = s_slot[10 * IBFT_SPLIT_SIGS + i];
        ibft_sig_item it;
        uint32_t* w = reinterpret_cast<uint32_t*>(&it);
        const uint32_t* src = s_items + i * IBFT_ITEM_ROW_WORDS;
#pragma unroll
        for (int k = 0; k < 32; k++) w[k] = src[k];
        resolved_item ri;
        bool have = false;
        resolve_item(it, arena, arena_len, ri, &have, true);  // this time with the digest
        sc rinv;
#pragma unroll
        for (int k = 0; k < 8; k++) rinv.v[k] = s_slot[(11 + k) * IBFT_SPLIT_SIGS + i];
        ecmult_digits dg;
#pragma unroll
        for (int k = 0; k < 6; k++) dg.ks[0][k] = dg.ks[1][k] = 0;
        dg.kneg[0] = dg.kneg[1] = false;
        split_helper_u1(ri, rinv, dg);
        fe y, gx, gy;
        bool g_inf = false;
        if (split_helper_point(ri, dg, G, y, g_inf, gx, gy)) {
          flags |= IBFT_SF_ROOT | (g_inf ? IBFT_SF_GINF : 0u);
#pragma unroll
          for (int k = 0; k < 8; k++) {
            s_y[k * IBFT_SPLIT_SIGS + i] = y.v[k];
            if (!g_inf) {
              s_slot[(11 + k) * IBFT_SPLIT_SIGS + i] = gx.v[k];
              s_slot[(19 + k) * IBFT_SPLIT_SIGS + i] = gy.v[k];
            }
          }
        }
        s_slot[27 * IBFT_SPLIT_SIGS + i] = flags;
      }
      __threadfence_block();
      named_bar_arrive(1 + IBFT_SPLIT_CHAINS + p, 64);
    }
    return;
  }
  // -------------------------------------------------------------------- chain warp
  const uint32_t i = tid, idx = base + i;  // tid = 32 * warp + lane
  const bool active = idx < shard_hi;
  ibft_sig_item it;
  resolved_item ri;
  bool have = false;
  int st = IBFT_ITEM_OK;
  rtab_view T{s_rtab + i, (uint32_t)IBFT_SPLIT_SIGS};
  fe gz = fe_from_u32(1);  // global Z of the table (ecmult_build_rtable_globalz)
  if (active) {
    uint32_t* w = reinterpret_cast<uint32_t*>(&it);
    const uint32_t* src = s_items + i * IBFT_ITEM_ROW_WORDS;
#pragma unroll
    for (int k = 0; k < 32; k++) w[k] = src[k];
    st = resolve_item(it, arena, arena_len, ri, &have, false);  // fields only: the chain never needs the digest
    if (have) gz = ecmult_build_rtable_globalz(split_chain_point(ri.r), T);  // table on a second isomorphic curve: no inversion
  }
  named_bar_sync(1 + warp, 64);  // the helper has posted the digits of u2
  jac acc;
  acc.x = fe_zero(); acc.y = fe_zero(); acc.z = fe_zero();
  acc.inf = true;
  bool go = false;
  if (active && have) {
    uint32_t flags = s_slot[10 * IBFT_SPLIT_SIGS + i];
    if (flags & IBFT_SF_VALID) {
      ecmult_digits dg;
#pragma unroll
      for (int k = 0; k < 5; k++) {
        dg.ks[0][k] = s_slot[k * IBFT_SPLIT_SIGS + i];
        dg.ks[1][k] = s_slot[(5 + k) * IBFT_SPLIT_SIGS + i];
        dg.ks[2][k] = dg.ks[3][k] = 0;
      }
      dg.ks[0][5] = dg.ks[1][5] = dg.ks[2][5] = dg.ks[3][5] = 0;
      dg.kneg[0] = flags & IBFT_SF_NEG0; dg.kneg[1] = flags & IBFT_SF_NEG1;
      dg.kneg[2] = dg.kneg[3] = false;
      acc = ecmult_streams(dg, G, T, false);
      go = true;
    }
  }
  named_bar_sync(1 + IBFT_SPLIT_CHAINS + warp, 64);  // the helper has posted y and u1*G
  aff K;
  K.x = fe_zero(); K.y = fe_zero();
  uint8_t addr[20];
#pragma unroll
  for (int k = 0; k < 20; k++) addr[k] = 0;
  bool ok = false;
  if (go) {
    uint32_t flags = s_slot[27 * IBFT_SPLIT_SIGS + i];
    if (flags & IBFT_SF_ROOT) {
      fe y, gx, gy;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        y.v[k] = s_y[k * IBFT_SPLIT_SIGS + i];
        gx.v[k] = s_slot[(11 + k) * IBFT_SPLIT_SIGS + i];
        gy.v[k] = s_slot[(19 + k) * IBFT_SPLIT_SIGS + i];
      }
      ok = split_chain_finish(acc, fe_mul(y, gz), (flags & IBFT_SF_GINF) != 0, gx, gy, addr, &K);  // Z' -> Z' * Z_8 * y
    }
  }
  if (active) {
#pragma unroll
    for (int k = 0; k < 20; k++) ok = ok && (addr[k] == ri.signer[k]);
    int vi = -1;
    uint32_t vslot = IBFT_NO_TABLE;
    if (ok) ok = member_and_vote(groups, n_groups, slots, n_slots, it.group, ri.signer, sink, true, &vi, &vslot);
    if (ok) learn_key(slots, vslot, vi, K);
    if (status != nullptr) status[idx] = (uint8_t)st;
    if (recovered != nullptr) {
#pragma unroll
      for (int k = 0; k < 20; k++) recovered[(size_t)idx * 20 + k] = addr[k];
    }
  } else {
    ok = false;
  }
  uint32_t word = __ballot_sync(0xFFFFFFFFu, ok);
  if (lane == 0 && active) bitmap[idx >> 5] = word;
}
#endif

#if IBFT_WC > 0
// ------------------------------------------------------------------------------------------------------------
// Known-key LATENCY variant (engine flag IBFT_FLAG_KEY_CACHE, mid-size rounds): k_recover_split's chain + helper layout, but
// the signature is VERIFIED against the validator's learned key instead of recovered (verify_core.cuh "Verification against a
// KNOWN public key").  The helper warp supplies w = s^-1 (one inversion for the lane's three signatures), the digits of
// u2 = r w, and later the affine u1*G = (z w) G from the comb tables; the chain warp walks u2*Q over the validator's table of
// multiples -- 17 rounds of 8 doublings + at most two additions, no per-signature table, no square root, no address hash --
// adds u1*G and accepts iff the point is exactly R = (r, y) with parity(y) = v.  An accept IS the recover path's verdict 1.
// Everything else that could still be valid -- key not learned yet, or the verification rejected -- goes to the worklist and is
// decided by the recover path (k_recover_qsplit in worklist mode, launched right behind this kernel); items that can never be
// valid (malformed, out of range, unknown group, signer not in the set) are settled here.  A round in which every signature
// verifies (the normal case of consensus) never runs a second chain.
// ------------------------------------------------------------------------------------------------------------
#define IBFT_VSLOT_WORDS 29   // [0..26] as IBFT_SLOT_WORDS, [27] validator index | slot << 16 of the signer, [28] phase-2 flags
#define IBFT_VSPLIT_SMEM ((IBFT_SPLIT_SIGS * (IBFT_ITEM_ROW_WORDS + IBFT_VSLOT_WORDS)) * 4)
#define IBFT_VF_VALID 1u      // digits of u2 posted: the chain runs
#define IBFT_VF_NEG0 2u
#define IBFT_VF_NEG1 4u
#define IBFT_VF_GREADY 8u     // u1*G posted
#define IBFT_VF_GINF 16u
#define IBFT_VF_RECOVER 32u   // member, but the key is not known yet: worklist
__global__ void __launch_bounds__(32 * (IBFT_SPLIT_CHAINS + 1), 1)
k_verify_split(const ibft_sig_item* __restrict__ items, uint32_t n, const uint8_t* __restrict__ arena, size_t arena_len,
               uint32_t shard_lo, uint32_t shard_hi, const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
               const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t* __restrict__ bitmap, uint8_t* __restrict__ status,
               const uint32_t* __restrict__ ctable, vote_sink sink, uint32_t* __restrict__ worklist) {
  extern __shared__ uint32_t s_dyn[];
  uint32_t* s_items = s_dyn;
  uint32_t* s_slot = s_items + IBFT_SPLIT_SIGS * IBFT_ITEM_ROW_WORDS;  // word w of signature i at [w * 96 + i]
  const uint32_t S = IBFT_SPLIT_SIGS;
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  const uint32_t base = shard_lo + blockIdx.x * IBFT_SPLIT_SIGS;
  {
    const uint4* src = reinterpret_cast<const uint4*>(items + base);
    uint32_t avail = base < shard_hi ? min((uint32_t)IBFT_SPLIT_SIGS, shard_hi - base) : 0u;
#pragma unroll
    for (int k = 0; k < (IBFT_SPLIT_SIGS * 8) / (32 * (IBFT_SPLIT_CHAINS + 1)); k++) {
      uint32_t u = tid + k * 32 * (IBFT_SPLIT_CHAINS + 1);
      uint32_t row = u >> 3, col = u & 7;
      if (row < avail) {
        uint4 v = __ldg(src + u);
        uint32_t* d = s_items + row * IBFT_ITEM_ROW_WORDS + col * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
      }
    }
  }
  __syncthreads();
  gtab_view G{g_gtable};
  G.comb = ctable;
  if (warp == IBFT_SPLIT_CHAINS) {
    // ------------------------------------------------------------------ helper warp
    uint32_t okmask = 0;
    IBFT_ROLLED
    for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
      const uint32_t i = 32 * p + lane, idx = base + i;
      uint32_t flags = 0;
      if (idx < shard_hi) {
        ibft_sig_item it;
        uint32_t* w = reinterpret_cast<uint32_t*>(&it);
        const uint32_t* src = s_items + i * IBFT_ITEM_ROW_WORDS;
#pragma unroll
        for (int k = 0; k < 32; k++) w[k] = src[k];
        resolved_item ri;
        bool have = false;
        int st = resolve_item(it, arena, arena_len, ri, &have, false);
        if (status != nullptr) status[idx] = (uint8_t)st;
        have = have && split_sig_in_range(ri);
        int v = -1;
        uint32_t slot = IBFT_NO_TABLE;
        if (have && group_member(groups, n_groups, slots, n_slots, it.group, ri.signer, &v, &slot)) {
          const bool ready = v >= 0 && slots[slot].key_state != nullptr && slots[slot].key_state[v] == IBFT_KEY_READY;
          if (ready) {
            sc r = sc_from_be(ri.r), sv = sc_from_be(ri.s);
#pragma unroll
            for (int k = 0; k < 8; k++) {
              s_slot[(11 + k) * S + i] = sv.v[k];   // s (inverted below), then r
              s_slot[(19 + k) * S + i] = r.v[k];
            }
            s_slot[27 * S + i] = (uint32_t)v | (slot << 16);
            okmask |= 1u << p;
          } else {
            flags = IBFT_VF_RECOVER;               // member whose key is not known (or no table: v < 0): the recover path decides
          }
        }
      }
      s_slot[10 * S + i] = flags;
    }
    {
      // w = s^-1 for the lane's signatures with ONE inversion (Montgomery's trick; an absent one contributes 1)
      sc one;
#pragma unroll
      for (int k = 0; k < 8; k++) one.v[k] = k == 0;
      sc ss[IBFT_SPLIT_CHAINS], pre[IBFT_SPLIT_CHAINS];
#pragma unroll
      for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
        ss[p] = one;
        if ((okmask >> p) & 1u) {
#pragma unroll
          for (int k = 0; k < 8; k++) ss[p].v[k] = s_slot[(11 + k) * S + 32 * p + lane];
        }
        pre[p] = p ? sc_mul(pre[p - 1], ss[p]) : ss[p];
      }
      sc inv = IBFT_SC_INV(pre[IBFT_SPLIT_CHAINS - 1]);
#pragma unroll
      for (int p = IBFT_SPLIT_CHAINS - 1; p >= 0; p--) {
        sc wi = p ? sc_mul(inv, pre[p - 1]) : inv;
        if (p) inv = sc_mul(inv, ss[p]);
#pragma unroll
        for (int k = 0; k < 8; k++) s_slot[(11 + k) * S + 32 * p + lane] = wi.v[k];  // w replaces s
      }
    }
    IBFT_ROLLED
    for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
      const uint32_t i = 32 * p + lane;
      if ((okmask >> p) & 1u) {
        sc w, r;
#pragma unroll
        for (int k = 0; k < 8; k++) {
          w.v[k] = s_slot[(11 + k) * S + i];
          r.v[k] = s_slot[(19 + k) * S + i];
        }
        ecmult_digits dg;
        ecmult_split_into(sc_mul(r, w), dg, 0);
#pragma unroll
        for (int k = 0; k < 5; k++) {
          s_slot[k * S + i] = dg.ks[0][k];
          s_slot[(5 + k) * S + i] = dg.ks[1][k];
        }
        s_slot[10 * S + i] = IBFT_VF_VALID | (dg.kneg[0] ? IBFT_VF_NEG0 : 0u) | (dg.kneg[1] ? IBFT_VF_NEG1 : 0u);
      }
      __threadfence_block();
      named_bar_arrive(1 + p, 64);
    }
    IBFT_ROLLED
    for (uint32_t p = 0; p < IBFT_SPLIT_CHAINS; p++) {
      const uint32_t i = 32 * p + lane;
      if ((okmask >> p) & 1u) {
        ibft_sig_item it;
        uint32_t* wd = reinterpret_cast<uint32_t*>(&it);
        const uint32_t* src = s_items + i * IBFT_ITEM_ROW_WORDS;
#pragma unroll
        for (int k = 0; k < 32; k++) wd[k] = src[k];
        resolved_item ri;
        bool have = false;
        resolve_item(it, arena, arena_len, ri, &have, true);  // this time with the digest
        sc w;
#pragma unroll
        for (int k = 0; k < 8; k++) w.v[k] = s_slot[(11 + k) * S + i];
        fe gx = fe_zero(), gy = fe_zero();
        bool g_inf = false;
        known_helper_u1g(ri, w, G, g_inf, gx, gy);
        uint32_t flags = IBFT_VF_GREADY | (g_inf ? IBFT_VF_GINF : 0u);
#pragma unroll
        for (int k = 0; k < 8; k++) {
          s_slot[(11 + k) * S + i] = gx.v[k];
          s_slot[(19 + k) * S + i] = gy.v[k];
        }
        s_slot[28 * S + i] = flags;
      }
      __threadfence_block();
      named_bar_arrive(1 + IBFT_SPLIT_CHAINS + p, 64);
    }
    return;
  }
  // -------------------------------------------------------------------- chain warp: u2 * Q from the validator's table
  const uint32_t i = tid, idx = base + i;
  const bool active = idx < shard_hi;
  named_bar_sync(1 + warp, 64);  // digits of u2 (and the verdict of the structural checks) are posted
  jac acc;
  acc.x = fe_zero(); acc.y = fe_zero(); acc.z = fe_zero();
  acc.inf = true;
  uint32_t flags = active ? s_slot[10 * S + i] : 0u;
  uint32_t vslot = 0;
  if (flags & IBFT_VF_VALID) {
    ecmult_digits dg;
#pragma unroll
    for (int k = 0; k < 5; k++) {
      dg.ks[0][k] = s_slot[k * S + i];
      dg.ks[1][k] = s_slot[(5 + k) * S + i];
      dg.ks[2][k] = dg.ks[3][k] = 0;
    }
    dg.ks[0][5] = dg.ks[1][5] = dg.ks[2][5] = dg.ks[3][5] = 0;
    dg.kneg[0] = flags & IBFT_VF_NEG0; dg.kneg[1] = flags & IBFT_VF_NEG1;
    dg.kneg[2] = dg.kneg[3] = false;
    vslot = s_slot[27 * S + i];
    const slot_dev& sd = slots[vslot >> 16];
    gtab_view Qt{sd.key_tab + (size_t)(vslot & 0xFFFFu) * IBFT_KEYTAB_WORDS};
    acc = ecmult_streams_known(dg, G, Qt, false);
  }
  named_bar_sync(1 + IBFT_SPLIT_CHAINS + warp, 64);  // u1*G is posted
  bool ok = false;
  if (flags & IBFT_VF_VALID) {
    const uint32_t f2 = s_slot[28 * S + i];
    fe gx, gy;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      gx.v[k] = s_slot[(11 + k) * S + i];
      gy.v[k] = s_slot[(19 + k) * S + i];
    }
    ibft_sig_item it;
    uint32_t* w = reinterpret_cast<uint32_t*>(&it);
    const uint32_t* src = s_items + i * IBFT_ITEM_ROW_WORDS;
#pragma unroll
    for (int k = 0; k < 32; k++) w[k] = src[k];
    resolved_item ri;
    bool have = false;
    resolve_item(it, arena, arena_len, ri, &have, false);
    ok = known_chain_finish(acc, (f2 & IBFT_VF_GINF) != 0, gx, gy, ri);
    if (ok) record_vote(sink, groups, it.group, (int)(vslot & 0xFFFFu));
  }
  // whatever was not accepted but could still be valid goes to the recover pass
  if (active && !ok && (flags & (IBFT_VF_VALID | IBFT_VF_RECOVER))) worklist[1 + atomicAdd(&worklist[0], 1u)] = idx;
  uint32_t word = __ballot_sync(0xFFFFFFFFu, ok);
  if (lane == 0 && active) bitmap[idx >> 5] = word;
}
#endif

#if IBFT_WC > 0
// ------------------------------------------------------------------------------------------------------------
// K1 + K2, small-round latency variant: the two ideas above combined.  CTA = 3 four-lane CHAIN warps (8 signatures each)
// + 1 HELPER warp (one lane per signature, a single pass over the CTA's 24), one CTA per SM, one warp per scheduler.
// The quads walk only u2*phi(R) (XYZZ levels, projective table, no square root, no inversion before the final one);
// the helper supplies the digits of u2 early and y, u1*G later.  Verdict bits are OR-ed into a pre-zeroed bitmap
// (24 signatures per CTA do not align with the 32-bit words).  Capacity of one wave: SMs x 24 signatures.
// ------------------------------------------------------------------------------------------------------------
#define IBFT_QSPLIT_SIGS 24
#ifndef IBFT_QSPLIT_MIN_CTAS
#define IBFT_QSPLIT_MIN_CTAS 1
#endif
__global__ void __launch_bounds__(128, IBFT_QSPLIT_MIN_CTAS)
k_recover_qsplit(const ibft_sig_item* __restrict__ items, uint32_t n, const uint8_t* __restrict__ arena, size_t arena_len,
                 uint32_t shard_lo, uint32_t shard_hi, const ibft_group_desc* __restrict__ groups, uint32_t n_groups,
                 const slot_dev* __restrict__ slots, uint32_t n_slots, uint32_t* __restrict__ bitmap,
                 uint8_t* __restrict__ recovered, uint8_t* __restrict__ status, const uint32_t* __restrict__ ctable, vote_sink sink,
                 const uint32_t* __restrict__ list) {
  // list != nullptr: WORKLIST mode (second pass of the known-key latency path): list[0] = count, list[1..] = item indices; the
  // t-th signature of the grid is item list[1 + t]; CTAs beyond the count leave at once; verdict bits are OR-ed in.
  __shared__ uint32_t s_items[IBFT_QSPLIT_SIGS * IBFT_ITEM_ROW_WORDS];
  __shared__ uint32_t s_idx[IBFT_QSPLIT_SIGS];
  __shared__ uint32_t s_qtab[IBFT_QSPLIT_SIGS * IBFT_QTAB_WORDS];
  __shared__ uint32_t s_slot[IBFT_QSPLIT_SIGS * IBFT_SLOT_WORDS];
  __shared__ uint32_t s_y[IBFT_QSPLIT_SIGS * 8];
  __shared__ uint4 s_xb[4 * 128];
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  const uint32_t base = list ? blockIdx.x * IBFT_QSPLIT_SIGS : shard_lo + blockIdx.x * IBFT_QSPLIT_SIGS;
  const uint32_t limit = list ? list[0] : shard_hi;   // rows [base, limit) of this CTA exist
  if (base >= limit) return;                            // (uniform over the CTA)
  {
    uint32_t avail = min((uint32_t)IBFT_QSPLIT_SIGS, limit - base);
    if (tid < IBFT_QSPLIT_SIGS) s_idx[tid] = tid < avail ? (list ? list[1 + base + tid] : base + tid) : 0xFFFFFFFFu;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 2; k++) {
      uint32_t u = tid + k * 128;
      uint32_t row = u >> 3, col = u & 7;
      if (row < avail) {
        uint4 v = __ldg(reinterpret_cast<const uint4*>(items + s_idx[row]) + col);
        uint32_t* d = s_items + row * IBFT_ITEM_ROW_WORDS + col * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
      }
    }
  }
  __syncthreads();
  gtab_view G{g_gtable};
  G.comb = ctable;
  const uint32_t S = IBFT_QSPLIT_SIGS;
  if (warp == 3) {
    // ---------------------------------------------------------------- helper warp: lane l serves signature l (l < 24)
    const uint32_t i = lane, idx = lane < S ? s_idx[lane] : 0xFFFFFFFFu;
    const bool mine = lane < S && idx != 0xFFFFFFFFu;
    ibft_sig_item it;
    resolved_item ri;
    sc rinv;
    uint32_t flags = 0;
    if (mine) {
      uint32_t* w = reinterpret_cast<uint32_t*>(&it);
      const uint32_t* src = s_items + i * IBFT_ITEM_ROW_WORDS;
#pragma unroll
      for (int k = 0; k < 32; k++) w[k] = src[k];
      bool have = false;
      resolve_item(it, arena, arena_len, ri, &have, false);
      if (have && split_sig_in_range(ri)) {
        rinv = IBFT_SC_INV(sc_from_be(ri.r));
        ecmult_digits dg;
        split_helper_u2(ri, rinv, dg);
        flags = IBFT_SF_VALID | (dg.kneg[0] ? IBFT_SF_NEG0 : 0u) | (dg.kneg[1] ? IBFT_SF_NEG1 : 0u);
#pragma unroll
        for (int k = 0; k < 5; k++) {
          s_slot[k * S + i] = dg.ks[0][k];
          s_slot[(5 + k) * S + i] = dg.ks[1][k];
        }
      }
    }
    if (lane < S) s_slot[10 * S + i] = flags;
    __threadfence_block();
    named_bar_arrive(1, 64); named_bar_arrive(2, 64); named_bar_arrive(3, 64);
    if (flags & IBFT_SF_VALID) {
      bool have = false;
      resolve_item(it, arena, arena_len, ri, &have, true);  // with the digest
      ecmult_digits dg;
#pragma unroll
      for (int k = 0; k < 6; k++) dg.ks[0][k] = dg.ks[1][k] = 0;
      dg.kneg[0] = dg.kneg[1] = false;
      split_helper_u1(ri, rinv, dg);
      fe y, gx, gy;
      bool g_inf = false;
      if (split_helper_point(ri, dg, G, y, g_inf, gx, gy)) {
        flags |= IBFT_SF_ROOT | (g_inf ? IBFT_SF_GINF : 0u);
#pragma unroll
        for (int k = 0; k < 8; k++) {
          s_y[k * S + i] = y.v[k];
          if (!g_inf) {
            s_slot[(11 + k) * S + i] = gx.v[k];
            s_slot[(19 + k) * S + i] = gy.v[k];
          }
        }
      }
      s_slot[27 * S + i] = flags;
    }
    __threadfence_block();
    named_bar_arrive(4, 64); named_bar_arrive(5, 64); named_bar_arrive(6, 64);
    return;
  }
  // ------------------------------------------------------------------ chain warps: four lanes per signature
  const uint32_t q = tid >> 2, idx = s_idx[q];
  const bool active = idx != 0xFFFFFFFFu;
  exec_quad ex;
  ex.role = (int)(tid & 3u);
  ex.mask = 0xFu << (tid & 28u);
  ex.xb = s_xb;
  ex.par = 0;
  ibft_sig_item it;
  resolved_item ri;
  bool have = false;
  int st = IBFT_ITEM_OK;
  fe c = fe_zero();
  qtab_view T{s_qtab + q, S};
  if (active) {
    uint32_t* w = reinterpret_cast<uint32_t*>(&it);
    const uint32_t* src = s_items + q * IBFT_ITEM_ROW_WORDS;
#pragma unroll
    for (int k = 0; k < 32; k++) w[k] = src[k];
    st = resolve_item(it, arena, arena_len, ri, &have, false);
    if (have) ecmult_build_qtable(ex, split_chain_point(ri.r, &c), T);
  }
  named_bar_sync(1 + warp, 64);
  xyzz acc;
  acc.x = fe_zero(); acc.y = fe_zero(); acc.zz = fe_zero(); acc.zzz = fe_zero();
  acc.inf = true;
  bool go = false;
  if (active && have) {
    uint32_t flags = s_slot[10 * S + q];
    if (flags & IBFT_SF_VALID) {
      ecmult_digits dg;
#pragma unroll
      for (int k = 0; k < 5; k++) {
        dg.ks[0][k] = s_slot[k * S + q];
        dg.ks[1][k] = s_slot[(5 + k) * S + q];
        dg.ks[2][k] = dg.ks[3][k] = 0;
      }
      dg.ks[0][5] = dg.ks[1][5] = dg.ks[2][5] = dg.ks[3][5] = 0;
      dg.kneg[0] = flags & IBFT_SF_NEG0; dg.kneg[1] = flags & IBFT_SF_NEG1;
      dg.kneg[2] = dg.kneg[3] = false;
      acc = ecmult_streams_x(ex, dg, G, T, false);
      go = true;
    }
  }
  named_bar_sync(4 + warp, 64);
  aff K;
  K.x = fe_zero(); K.y = fe_zero();
  uint8_t addr[20];
#pragma unroll
  for (int k = 0; k < 20; k++) addr[k] = 0;
  bool ok = false;
  if (go) {
    uint32_t flags = s_slot[27 * S + q];
    if (flags & IBFT_SF_ROOT) {
      fe y, gx, gy;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        y.v[k] = s_y[k * S + q];
        gx.v[k] = s_slot[(11 + k) * S + q];
        gy.v[k] = s_slot[(19 + k) * S + q];
      }
      ok = split_chain_finish_x(ex, acc, c, y, (flags & IBFT_SF_GINF) != 0, gx, gy, addr, &K);
    }
  }
  if (active) {
#pragma unroll
    for (int k = 0; k < 20; k++) ok = ok && (addr[k] == ri.signer[k]);
    int vi = -1;
    uint32_t vslot = IBFT_NO_TABLE;
    if (ok) ok = member_and_vote(groups, n_groups, slots, n_slots, it.group, ri.signer, sink, ex.leader(), &vi, &vslot);
    if (ok && ex.leader()) learn_key(slots, vslot, vi, K);
    if (ex.leader()) {
      if (status != nullptr && list == nullptr) status[idx] = (uint8_t)st;
      if (recovered != nullptr) {
#pragma unroll
        for (int k = 0; k < 20; k++) recovered[(size_t)idx * 20 + k] = addr[k];
      }
      if (ok) atomicOr(&bitmap[idx >> 5], 1u << (idx & 31u));
    }
  }
}
#endif

// ------------------------------------------------------------------------------------------------------------
// K3: quorum
// ------------------------------------------------------------------------------------------------------------

__global__ void k_quorum_mark(const ibft_sig_item* __restrict__ items, uint32_t n, const uint8_t* __restrict__ arena, size_t arena_len,
                              const uint32_t* __restrict__ bitmap,
                              const ibft_group_desc* __restrict__ groups, const group_dev* __restrict__ gdev,
                              uint32_t n_groups, const slot_dev* __restrict__ slots, uint32_t n_slots,
                              uint32_t* __restrict__ voted, uint32_t* __restrict__ n_valid, uint32_t lo, uint32_t hi) {
  uint32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hi || i >= n) return;
  if (!((bitmap[i >> 5] >> (i & 31)) & 1u)) return;
  const ibft_sig_item* it = items + i;
  uint32_t g = it->group;
  if (g >= n_groups) return;
  atomicAdd(&n_valid[g], 1u);
  uint32_t slot = groups[g].table_slot;
  if (slot == IBFT_NO_TABLE || slot >= n_slots || !slots[slot].valid) return;
  uint8_t addr[20];
  ibft_sig_item local = *it;
  if (!item_signer(local, arena, arena_len, addr)) return;
  int v = lookup_validator(slots[slot], addr);
  if (v >= 0) atomicOr(&voted[gdev[g].voted_off + ((uint32_t)v >> 5)], 1u << (v & 31));
}

// multi-GPU: OR the ranks' partial voted sets and add their valid counts (partial layout: voted words, then one count per group)
__global__ void k_quorum_merge(const uint32_t* __restrict__ parts, uint32_t n_parts, uint32_t part_stride, uint32_t voted_words,
                               uint32_t n_groups, uint32_t* __restrict__ voted, uint32_t* __restrict__ n_valid) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= voted_words + n_groups) return;
  uint32_t acc = 0;
  for (uint32_t r = 0; r < n_parts; r++) {
    uint32_t v = parts[(size_t)r * part_stride + i];
    acc = i < voted_words ? (acc | v) : (acc + v);
  }
  if (i < voted_words) voted[i] = acc;
  else n_valid[i - voted_words] = acc;
}

// Multi-GPU exchange WITHOUT a library collective: every rank's (bitmap words | partial voted sets | valid counts) sit in a
// buffer its peers have mapped over NVLink (CUDA IPC); this kernel publishes "my round `epoch` is complete", waits for the
// peers' flags, then reads their words straight out of peer memory -- OR-ing the voted sets, summing the counts, and assembling
// the complete bitmap -- so that the all-gather and the merge are ONE launch (the NCCL path costs a collective launch + the
// merge kernel: ~25-30 us of a 0.5 ms round).  Buffer of rank r: [2 parities][words_per_rank] words, then flags[2].  Rounds
// alternate parities: a rank can only start writing parity p for round e+2 after it has seen every peer's flag for round e+1,
// i.e. after every peer has finished reading round e.  The wait is bounded (spin_limit polls): on timeout the kernel reports
// through *timeout_flag and merges nothing -- it never hangs the device.
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
struct peer_bufs {
  uint32_t* buf[8];  // one node: at most 8 ranks
};
__global__ void k_quorum_exchange(peer_bufs peers, uint32_t world, uint32_t rank, uint32_t words_per_rank, uint32_t bitmap_words,
                                  uint32_t voted_words, uint32_t n_groups, uint32_t epoch, uint32_t spin_limit,
                                  uint32_t* __restrict__ full_bitmap, uint32_t* __restrict__ voted, uint32_t* __restrict__ n_valid,
                                  uint32_t* __restrict__ timeout_flag) {
  __shared__ uint32_t s_ok;
  const uint32_t par = epoch & 1u;
  const size_t flags_off = 2 * (size_t)words_per_rank;
  if (threadIdx.x == 0) {
    if (blockIdx.x == 0) {
      __threadfence_system();  // the verify / mark kernels' writes to my buffer are visible to the peers before the flag is
      st_release_sys(peers.buf[rank] + flags_off + par, epoch);
    }
    uint32_t ok = 1;
    for (uint32_t r = 0; r < world && ok; r++) {
      const uint32_t* f = peers.buf[r] + flags_off + par;
      uint32_t spins = 0;
      while ((int32_t)(ld_acquire_sys(f) - epoch) < 0) {
        if (++spins > spin_limit) { ok = 0; break; }
        __nanosleep(64);
      }
    }
    if (!ok) atomicExch(timeout_flag, 1u);
    s_ok = ok;
  }
  __syncthreads();
  if (!s_ok) return;
  const uint32_t per_rank_bitmap = bitmap_words;  // words [0, bitmap_words) of a rank's buffer: its slice of the bitmap
  const uint32_t total = world * per_rank_bitmap + voted_words + n_groups;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    if (i < world * per_rank_bitmap) {
      const uint32_t r = i / per_rank_bitmap, w = i % per_rank_bitmap;
      full_bitmap[i] = ld_relaxed_sys(peers.buf[r] + (size_t)par * words_per_rank + w);
    } else {
      const uint32_t j = i - world * per_rank_bitmap;  // index into (voted sets | counts)
      uint32_t acc = 0;
      for (uint32_t r = 0; r < world; r++) {
        uint32_t v = ld_relaxed_sys(peers.buf[r] + (size_t)par * words_per_rank + per_rank_bitmap + j);
        acc = j < voted_words ? (acc | v) : (acc + v);
      }
      if (j < voted_words) voted[j] = acc;
      else n_valid[j - voted_words] = acc;
    }
  }
}

// one CTA per group: 320-bit sum of the voting power of the voted validators, compared with the threshold
#define IBFT_REDUCE_THREADS 1024  // one CTA per group; a 10k-validator set is 10 strided passes instead of 40
__global__ void __launch_bounds__(IBFT_REDUCE_THREADS)
k_quorum_reduce(const ibft_group_desc* __restrict__ groups, const group_dev* __restrict__ gdev, uint32_t n_groups,
                const slot_dev* __restrict__ slots, uint32_t n_slots, const uint32_t* __restrict__ voted,
                const uint32_t* __restrict__ n_valid, ibft_group_result* __restrict__ results) {
  __shared__ uint64_t s_sum[IBFT_REDUCE_THREADS][5];
  __shared__ uint32_t s_cnt[IBFT_REDUCE_THREADS];
  uint32_t g = blockIdx.x;
  if (g >= n_groups) return;
  uint32_t slot = groups[g].table_slot;
  bool has_table = slot != IBFT_NO_TABLE && slot < n_slots && slots[slot].valid;
  uint64_t acc[5] = {0, 0, 0, 0, 0};
  uint32_t cnt = 0;
  if (has_table) {
    const slot_dev& s = slots[slot];
    const uint32_t* vw = voted + gdev[g].voted_off;
    for (uint32_t v = threadIdx.x; v < s.n; v += blockDim.x) {
      if ((vw[v >> 5] >> (v & 31)) & 1u) {
        cnt++;
        const uint64_t* p = s.powers + 4 * (size_t)v;
        unsigned long long c = 0;
#pragma unroll
        for (int k = 0; k < 5; k++) {
          unsigned long long add = k < 4 ? p[k] : 0ull;
          unsigned long long t = acc[k] + add;
          unsigned long long c1 = t < add;
          unsigned long long t2 = t + c;
          c1 += t2 < c;
          acc[k] = t2;
          c = c1;
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 5; k++) s_sum[threadIdx.x][k] = acc[k];
  s_cnt[threadIdx.x] = cnt;
  __syncthreads();
  for (uint32_t stride = blockDim.x >> 1; stride > 0; stride >>= 1) {
    if (threadIdx.x < stride) {
      unsigned long long c = 0;
#pragma unroll
      for (int k = 0; k < 5; k++) {
        unsigned long long a = s_sum[threadIdx.x][k], b = s_sum[threadIdx.x + stride][k];
        unsigned long long t = a + b;
        unsigned long long c1 = t < b;
        unsigned long long t2 = t + c;
        c1 += t2 < c;
        s_sum[threadIdx.x][k] = t2;
        c = c1;
      }
      s_cnt[threadIdx.x] += s_cnt[threadIdx.x + stride];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    ibft_group_result r;
#pragma unroll
    for (int k = 0; k < 5; k++) r.power[k] = s_sum[0][k];
    r.n_valid = n_valid[g];
    r.n_distinct = s_cnt[0];
    r.has_quorum = 0;
    r.reserved = 0;
    if (has_table) {
      // power >= quorum ?
      int cmp = 0;
      for (int k = 4; k >= 0; k--) {
        uint64_t q = slots[slot].quorum[k];
        if (cmp == 0 && r.power[k] != q) cmp = r.power[k] < q ? -1 : 1;
      }
      r.has_quorum = cmp >= 0 ? 1u : 0u;
    }
    results[g] = r;
  }
}

// ------------------------------------------------------------------------------------------------------------
// hash-only batch (IsValidProposalHash)
// ------------------------------------------------------------------------------------------------------------
__global__ void k_keccak_batch(const uint8_t* __restrict__ arena, size_t arena_len, const uint32_t* __restrict__ offs,
                               const uint32_t* __restrict__ lens, const uint64_t* __restrict__ rounds, uint32_t n,
                               uint8_t* __restrict__ out) {
  // rounds == nullptr: out[i] = Keccak-256(message i).
  // rounds != nullptr: the proposal hash of this engine's synthetic convention (SURVEY.md §8c), both sponges in ONE launch:
  //                    out[i] = Keccak-256(Keccak-256(rawProposal_i) || u64_be(round_i))   (IsValidProposalHash)
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t h[40];
  if ((size_t)offs[i] + lens[i] > arena_len) {
#pragma unroll
    for (int k = 0; k < 32; k++) h[k] = 0;
  } else {
    keccak256_bytes(arena + offs[i], lens[i], h);
    if (rounds != nullptr) {
      uint64_t r = rounds[i];
#pragma unroll
      for (int k = 0; k < 8; k++) h[32 + k] = (uint8_t)(r >> (8 * (7 - k)));
      uint8_t h2[32];
      keccak256_bytes(h, 40, h2);
#pragma unroll
      for (int k = 0; k < 32; k++) h[k] = h2[k];
    }
  }
#pragma unroll
  for (int k = 0; k < 32; k++) out[(size_t)i * 32 + k] = h[k];
}

// ------------------------------------------------------------------------------------------------------------
// combined generator table (IBFT_WC > 0): entry (d1, d2) = d1*G + d2*lambda*G, computed with the kernel's own scalar
// multiplication as (d1 + d2*lambda mod n) * G and checked against the oracle in tests/test_gpu_primitives.py
// ------------------------------------------------------------------------------------------------------------
#if IBFT_WC > 0
__global__ void __launch_bounds__(64)
k_build_ctable(uint32_t* __restrict__ out) {  // blockIdx.y = comb position: entries scaled by 2^(WC * position)
  __shared__ uint32_t s_gtab[IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES];
  __shared__ uint32_t s_rtab[64 * IBFT_RTAB_WORDS];
  for (uint32_t i = threadIdx.x; i < IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES; i += 64) s_gtab[i] = g_gtable[i];
  __syncthreads();
  size_t e = (size_t)blockIdx.x * 64 + threadIdx.x;
  if (e >= (size_t)IBFT_CTAB_ENTRIES) return;
  int d1 = (int)(e / IBFT_CTAB_D2), d2 = (int)(e % IBFT_CTAB_D2) - (1 << (IBFT_WC - 1));
  const uint32_t lam[8] = {0x1B23BD72u, 0xDF02967Cu, 0x20816678u, 0x122E22EAu, 0x8812645Au, 0xA5261C02u, 0xC05C30E0u, 0x5363AD4Cu};
  sc a, b, l;
#pragma unroll
  for (int i = 0; i < 8; i++) { a.v[i] = 0; b.v[i] = 0; l.v[i] = lam[i]; }
  a.v[0] = (uint32_t)d1;
  b.v[0] = (uint32_t)(d2 < 0 ? -d2 : d2);
  sc t = sc_mul(b, l);
  if (d2 < 0) t = sc_neg(t);
  sc k = sc_add(a, t);
  const uint32_t pos = blockIdx.y;
  if (pos) {
    sc m;
#pragma unroll
    for (int i = 0; i < 8; i++) m.v[i] = 0;
    m.v[(pos * IBFT_WC) / 32] = 1u << ((pos * IBFT_WC) % 32);
    k = sc_mul(k, m);
  }
  uint32_t* o = out + IBFT_GTAB_ENTRY_WORDS * ((size_t)pos * IBFT_CTAB_ENTRIES + e);
  gtab_view G{s_gtab};
  rtab_view T{s_rtab + threadIdx.x, 64u};
  aff g1;
  G.load(0, g1.x, g1.y);
  sc zero;
#pragma unroll
  for (int i = 0; i < 8; i++) zero.v[i] = 0;
  jac P = ecmult_double(k, zero, g1, G, T);
  if (P.inf || fe_is_zero(P.z)) {
#pragma unroll
    for (int i = 0; i < 16; i++) o[i] = 0;  // (0, 0): never looked up
    return;
  }
  fe zi = IBFT_FE_INV(P.z), zi2 = fe_sqr(zi);
  fe x = fe_normalize(fe_mul(P.x, zi2)), y = fe_normalize(fe_mul(P.y, fe_mul(zi2, zi)));
#pragma unroll
  for (int i = 0; i < 8; i++) { o[i] = x.v[i]; o[8 + i] = y.v[i]; }
}
#endif

#if IBFT_WC > 0
// key registry: comb tables for every validator of `slot` whose key has been learned but whose table is missing.  One thread
// per (validator, comb position): 8*pos doublings, 128 additions and 128 inversions each -- a whole 10k-validator set
// (170,000 threads, 21.8 M table entries, 1.39 GB) is built once per validator set; k_keytabs_ready then publishes the tables.
__global__ void __launch_bounds__(64)
k_build_keytabs(const slot_dev* __restrict__ slots, uint32_t slot) {
  const slot_dev& s = slots[slot];
  const uint32_t t = blockIdx.x * 64 + threadIdx.x;
  const uint32_t v = t / IBFT_KEYTAB_POSITIONS, pos = t % IBFT_KEYTAB_POSITIONS;
  if (s.key_state == nullptr || v >= s.n || s.key_state[v] != IBFT_KEY_BUILDING) return;
  aff Q;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    Q.x.v[i] = s.key_xy[16 * (size_t)v + i];
    Q.y.v[i] = s.key_xy[16 * (size_t)v + 8 + i];
  }
  build_keytab_pos(Q, (int)pos, s.key_tab + (size_t)v * IBFT_KEYTAB_WORDS + (size_t)pos * IBFT_KEYTAB_ENTRIES * IBFT_GTAB_ENTRY_WORDS);
}
// state steps around the build, one launch each on the same stream: LEARNED -> BUILDING (claim: the set of validators this pass
// builds is fixed here -- recover kernels of another lane may keep learning keys meanwhile, those wait for the next pass),
// BUILDING -> READY (publish)
__global__ void __launch_bounds__(256)
k_keytabs_step(const slot_dev* __restrict__ slots, uint32_t slot, uint32_t from, uint32_t to) {
  const slot_dev& s = slots[slot];
  const uint32_t v = blockIdx.x * 256 + threadIdx.x;
  if (s.key_state != nullptr && v < s.n && s.key_state[v] == from) s.key_state[v] = to;
}
#endif

#if IBFT_WC > 0
// key registry carry-over (ibft_set_validators): consensus moves to the next height with (mostly) the same validators, and a
// key belongs to an ADDRESS, not to a height.  One CTA per validator of the new table (rank r of its sorted address table):
// look the address up in the donor table; if the donor holds a finished comb table for it, copy key + table (136 KiB, 16-byte
// loads) and publish.  A 10k-validator set is 1.39 GB of device-to-device copy, once per height.
__global__ void __launch_bounds__(256)
k_carry_keys(slot_dev dst, slot_dev src) {
  __shared__ int s_src;
  const uint32_t r = blockIdx.x;
  const uint32_t* k = dst.keys + 6 * (size_t)r;
  const uint32_t v = __ldg(k + 5);
  if (threadIdx.x == 0) {
    int lo = 0, hi = (int)src.n - 1, found = -1;
    while (lo <= hi && found < 0) {
      int mid = (lo + hi) >> 1;
      const uint32_t* q = src.keys + 6 * (size_t)mid;
      int cmp = 0;
#pragma unroll
      for (int i = 0; i < 5; i++) {
        uint32_t a = __ldg(q + i), b = __ldg(k + i);
        if (cmp == 0 && a != b) cmp = a < b ? -1 : 1;
      }
      if (cmp == 0) found = (int)__ldg(q + 5);
      else if (cmp < 0) lo = mid + 1;
      else hi = mid - 1;
    }
    if (found >= 0 && src.key_state[found] != IBFT_KEY_READY) found = -1;
    s_src = found;
  }
  __syncthreads();
  const int sv = s_src;
  if (sv < 0) return;
  const uint4* from = reinterpret_cast<const uint4*>(src.key_tab + (size_t)sv * IBFT_KEYTAB_WORDS);
  uint4* to = reinterpret_cast<uint4*>(dst.key_tab + (size_t)v * IBFT_KEYTAB_WORDS);
  for (uint32_t i = threadIdx.x; i < IBFT_KEYTAB_WORDS / 4; i += 256) to[i] = from[i];
  if (threadIdx.x < 16) dst.key_xy[16 * (size_t)v + threadIdx.x] = src.key_xy[16 * (size_t)sv + threadIdx.x];
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    dst.key_state[v] = IBFT_KEY_READY;
    atomicAdd(dst.learn_count, 1u);
  }
}
#endif

// ------------------------------------------------------------------------------------------------------------
// batched signing (MessageConstructor side)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64)
k_sign(const uint8_t* __restrict__ privkeys, const uint8_t* __restrict__ digests, const uint8_t* __restrict__ nonces, uint32_t n,
       uint8_t* __restrict__ sigs) {
  __shared__ uint32_t s_gtab[IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES];
  __shared__ uint32_t s_rtab[64 * IBFT_RTAB_WORDS];
  for (uint32_t i = threadIdx.x; i < IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES; i += 64) s_gtab[i] = g_gtable[i];
  __syncthreads();
  uint32_t i = blockIdx.x * 64 + threadIdx.x;
  if (i >= n) return;
  uint8_t d[32], z[32], k[32], sig[65];
#pragma unroll
  for (int j = 0; j < 32; j++) { d[j] = privkeys[32 * (size_t)i + j]; z[j] = digests[32 * (size_t)i + j]; }
  gtab_view G{s_gtab};
  rtab_view T{s_rtab + threadIdx.x, 64u};
  bool ok = false;
  if (nonces != nullptr) {
#pragma unroll
    for (int j = 0; j < 32; j++) k[j] = nonces[32 * (size_t)i + j];
    ok = ecdsa_sign(d, z, k, G, T, sig);
  } else {
    // derived nonce: k = Keccak-256(d || z || ctr), ctr = 0, 1, ... until usable (deterministic, unique per (key, digest))
    for (uint32_t ctr = 0; ctr < 4 && !ok; ctr++) {
      uint8_t buf[65];
#pragma unroll
      for (int j = 0; j < 32; j++) { buf[j] = d[j]; buf[32 + j] = z[j]; }
      buf[64] = (uint8_t)ctr;
      keccak256_bytes(buf, 65, k);
      ok = ecdsa_sign(d, z, k, G, T, sig);
    }
  }
#pragma unroll
  for (int j = 0; j < 65; j++) sigs[65 * (size_t)i + j] = ok ? sig[j] : (uint8_t)0;
}

// ------------------------------------------------------------------------------------------------------------
// primitive parity hooks + integer-pipe probes
// ------------------------------------------------------------------------------------------------------------
__global__ void k_debug_op(int op, const uint8_t* a, const uint8_t* b, const uint8_t* c, uint32_t n, uint8_t* out,
                           uint32_t stride) {
#if IBFT_GTAB_SMEM
  __shared__ uint32_t s_gtab[IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES];
  for (uint32_t i = threadIdx.x; i < IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES; i += blockDim.x) s_gtab[i] = g_gtable[i];
  __syncthreads();
#else
  const uint32_t* s_gtab = g_gtable;
#endif
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* pa = a + 32 * (size_t)i;
  const uint8_t* pb = b ? b + 32 * (size_t)i : pa;
  uint8_t* o = out + (size_t)stride * i;
  switch (op) {
    case IBFT_DBG_FE_MUL: fe_to_be(fe_normalize(fe_mul(fe_from_be(pa), fe_from_be(pb))), o); break;
    case IBFT_DBG_FE_SQR: fe_to_be(fe_normalize(fe_sqr(fe_from_be(pa))), o); break;
    case IBFT_DBG_FE_INV: fe_to_be(fe_normalize(IBFT_FE_INV(fe_from_be(pa))), o); break;
    case IBFT_DBG_FE_SQRT: fe_to_be(fe_normalize(fe_sqrt_candidate(fe_from_be(pa))), o); break;
    case IBFT_DBG_FE_ADD: fe_to_be(fe_normalize(fe_add(fe_from_be(pa), fe_from_be(pb))), o); break;
    case IBFT_DBG_FE_SUB: fe_to_be(fe_normalize(fe_sub(fe_from_be(pa), fe_from_be(pb))), o); break;
    case IBFT_DBG_SC_MUL: sc_to_be(sc_mul(sc_from_be(pa), sc_from_be(pb)), o); break;
    case IBFT_DBG_SC_INV: sc_to_be(IBFT_SC_INV(sc_reduce_once(sc_from_be(pa))), o); break;
    case IBFT_DBG_GLV: {
      glv_half h1, h2;
      glv_split(sc_reduce_once(sc_from_be(pa)), h1, h2);
      for (int k = 0; k < 64; k++) o[k] = 0;
      for (int k = 0; k < 5; k++)
        for (int j = 0; j < 4; j++) {
          o[4 * k + j] = (uint8_t)(h1.k[k] >> (8 * j));
          o[24 + 4 * k + j] = (uint8_t)(h2.k[k] >> (8 * j));
        }
      o[20] = h1.neg;
      o[44] = h2.neg;
      break;
    }
    case IBFT_DBG_ECMULT: {
      gtab_view G{s_gtab};
      const uint8_t* pc = c + 64 * (size_t)i;
      aff P;
      P.x = fe_from_be(pc);
      P.y = fe_from_be(pc + 32);
      uint32_t rtab[IBFT_RTAB_WORDS];
      rtab_view T{rtab, 1};
      jac Q = ecmult_double(sc_reduce_once(sc_from_be(pa)), sc_reduce_once(sc_from_be(pb)), P, G, T);
      for (int k = 0; k < 64; k++) o[k] = 0;
      if (!(Q.inf || fe_is_zero(Q.z))) {
        fe zi = IBFT_FE_INV(Q.z), zi2 = fe_sqr(zi);
        fe_to_be(fe_normalize(fe_mul(Q.x, zi2)), o);
        fe_to_be(fe_normalize(fe_mul(Q.y, fe_mul(zi2, zi))), o + 32);
      }
      break;
    }
    default: break;
  }
}

#define PROBE_ITERS 2048
#define PROBE_UNROLL 16
__global__ void k_probe_imad(uint32_t* out, uint32_t a, uint32_t b) {
  uint32_t x[8];
#pragma unroll
  for (int k = 0; k < 8; k++) x[k] = threadIdx.x + k;
  for (int i = 0; i < PROBE_ITERS; i++) {
#pragma unroll
    for (int u = 0; u < PROBE_UNROLL; u++) {
#pragma unroll
      for (int k = 0; k < 8; k++) asm volatile("mad.lo.u32 %0,%0,%1,%2;" : "+r"(x[k]) : "r"(a), "r"(b));
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) s ^= x[k];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_probe_wide(uint32_t* out, uint32_t a, uint32_t b) {
  uint32_t x[4][8];
#pragma unroll
  for (int k = 0; k < 4; k++)
#pragma unroll
    for (int j = 0; j < 8; j++) x[k][j] = threadIdx.x + k + j;
  for (int i = 0; i < PROBE_ITERS; i++) {
#pragma unroll
    for (int u = 0; u < PROBE_UNROLL / 4; u++) {
#pragma unroll
      for (int k = 0; k < 4; k++) {
        asm volatile(
            "mad.lo.cc.u32 %0,%8,%9,%0; madc.hi.cc.u32 %1,%8,%9,%1;"
            "madc.lo.cc.u32 %2,%8,%9,%2; madc.hi.cc.u32 %3,%8,%9,%3;"
            "madc.lo.cc.u32 %4,%8,%9,%4; madc.hi.cc.u32 %5,%8,%9,%5;"
            "madc.lo.cc.u32 %6,%8,%9,%6; madc.hi.u32 %7,%8,%9,%7;"
            : "+r"(x[k][0]), "+r"(x[k][1]), "+r"(x[k][2]), "+r"(x[k][3]), "+r"(x[k][4]), "+r"(x[k][5]), "+r"(x[k][6]),
              "+r"(x[k][7])
            : "r"(a), "r"(b));
      }
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < 4; k++)
#pragma unroll
    for (int j = 0; j < 8; j++) s ^= x[k][j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ------------------------------------------------------------------------------------------------------------
// host side: engine object + C ABI
// ------------------------------------------------------------------------------------------------------------
static thread_local char tl_err[512] = "";
static void set_err(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tl_err, sizeof tl_err, fmt, ap);
  va_end(ap);
}
#define CU(call)                                                                                        \
  do {                                                                                                  \
    cudaError_t _e = (call);                                                                            \
    if (_e != cudaSuccess) {                                                                            \
      set_err("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__);              \
      return IBFT_ERR_CUDA;                                                                             \
    }                                                                                                   \
  } while (0)

struct slot_host {
  bool valid = false;
  uint64_t height = 0;
  uint32_t n = 0;
  uint32_t* d_keys = nullptr;
  uint64_t* d_powers = nullptr;
  uint64_t quorum[5] = {0, 0, 0, 0, 0};
  // key registry (IBFT_FLAG_KEY_CACHE)
  uint32_t* d_key_state = nullptr;
  uint32_t* d_key_xy = nullptr;
  uint32_t* d_key_tab = nullptr;
  uint32_t* d_learn_count = nullptr;
  uint32_t built_count = 0;  // value of *d_learn_count when the tables were last brought up to date
};

struct pending_call {
  bool active = false;
  uint32_t n = 0, n_groups = 0;
  uint32_t* bitmap_out = nullptr;
  ibft_group_result* results_out = nullptr;
  uint8_t* recovered_out = nullptr;
};

// One LANE = everything a host-buffer verify call needs while it is in flight: streams, events, device buffers, pinned
// staging.  The engine has two, so that two handlers do not serialise (the reference runs the COMMIT fan-in, a ROUND_CHANGE
// watcher and the gossip ingress concurrently: core/ibft.go:335-347, :1128):
//   lane 0  full capacity (max_items): bulk handler batches, the async submit/poll/wait API, the device-resident entry points;
//   lane 1  a small lane (IBFT_LANE1_ITEMS) for the ingress coalescer's batches and other small concurrent calls.
// A call holds its lane's mutex from staging to the copy-out; validator tables and the key registry are shared.
#define IBFT_LANES 2
#define IBFT_LANE1_ITEMS 16384u
#define IBFT_LANE1_ARENA (4u << 20)
struct lane {
  std::mutex mu;
  uint32_t cap_items = 0;
  size_t cap_arena = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;       // H2D of chunk k+1 overlaps the recover kernel of chunk k
  std::vector<cudaEvent_t> chunk_ev;
  cudaStream_t lat_stream[4] = {nullptr, nullptr, nullptr, nullptr};  // one round in four pieces: copy + kernel of piece k
  cudaEvent_t lat_ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // overlap the staging of piece k+1 (latency path)
  cudaEvent_t done_ev = nullptr;
  // device
  ibft_sig_item* d_items = nullptr;
  uint8_t* d_arena = nullptr;
  uint32_t* d_bitmap = nullptr;
  uint8_t* d_recovered = nullptr;
  uint8_t* d_status = nullptr;
  uint8_t* h_status = nullptr;
  uint32_t last_status_n = 0;
  ibft_group_desc* d_groups = nullptr;
  group_dev* d_gdev = nullptr;
  ibft_group_result* d_results = nullptr;
  uint32_t* d_voted = nullptr;
  uint32_t* d_nvalid = nullptr;
  size_t voted_words_cap = 0;
  // pinned host staging
  ibft_sig_item* h_items = nullptr;
  uint8_t* h_arena = nullptr;
  uint32_t* h_bitmap = nullptr;
  uint8_t* h_recovered = nullptr;
  ibft_group_desc* h_groups = nullptr;
  group_dev* h_gdev = nullptr;
  ibft_group_result* h_results = nullptr;
  std::vector<group_dev> last_gdev;  // layout of the voted sets of the most recent reduce
  std::vector<ibft_group_desc> last_groups;
  pending_call pending;
  uint32_t* d_worklist = nullptr;  // key-registry path: [0] = count, [1..] = indices left to the recover pass
  cudaEvent_t wl_ev[4] = {nullptr, nullptr, nullptr, nullptr};  // last use of each worklist (orders launches that arrive on different streams)
  uint32_t wl_used = 0;  // bit k: worklist k was filled by the current / last host-buffer call (ibft_debug_last_deferred)
  const uint8_t* dev_arena = nullptr;
  size_t dev_arena_len = 0;
};

struct ibft_engine {
  ibft_engine_params p;
  lane lanes[IBFT_LANES];
  std::atomic<int> last_lane{0};  // lane of the most recently COMPLETED host-buffer call (ibft_last_item_status, ibft_get_voted_bitmap)
  slot_dev* d_slots = nullptr;
  std::vector<slot_host> slots;
  std::vector<slot_dev> slots_shadow;
  std::atomic<uint64_t> launches{0};
  std::atomic<int> recover_path{IBFT_PATH_AUTO};
  std::mutex keys_mu;                  // key registry upkeep (built_count, h_learn_counts)
  uint32_t* d_learn_counts = nullptr;  // key registry: one "keys learned" counter per table slot (read back in one copy)
  uint32_t* h_learn_counts = nullptr;  // pinned
  int sm_count = 148;
  uint32_t* d_ctable = nullptr;  // combined generator table (IBFT_WC > 0)
  cudaFuncAttributes recover_attr{};
  // hashing (ibft_keccak256_batch / ibft_proposal_hash_batch): own lock, own stream, own grow-only scratch -- a hash call
  // never waits for a verify call and never allocates on the per-call path
  std::mutex hash_mu;
  cudaStream_t hash_stream = nullptr;
  uint8_t *hs_arena = nullptr, *hs_h_arena = nullptr, *hs_meta = nullptr, *hs_h_meta = nullptr;
  size_t hs_arena_cap = 0;
  uint32_t hs_n_cap = 0;
};
// every lane, in index order (validator-table replacement and other engine-wide operations)
struct all_lanes_lock {
  ibft_engine* e;
  explicit all_lanes_lock(ibft_engine* e_) : e(e_) { for (auto& L : e->lanes) L.mu.lock(); }
  ~all_lanes_lock() { for (int i = IBFT_LANES - 1; i >= 0; i--) e->lanes[i].mu.unlock(); }
};

extern "C" int ibft_abi_version(void) { return IBFT_ABI_VERSION; }
extern "C" const char* ibft_last_error(void) { return tl_err; }

static void lane_free(lane* L) {
  cudaFree(L->d_status); cudaFreeHost(L->h_status);
  cudaFree(L->d_worklist);
  cudaFree(L->d_items); cudaFree(L->d_arena); cudaFree(L->d_bitmap); cudaFree(L->d_recovered); cudaFree(L->d_groups);
  cudaFree(L->d_gdev); cudaFree(L->d_results); cudaFree(L->d_voted); cudaFree(L->d_nvalid);
  cudaFreeHost(L->h_items); cudaFreeHost(L->h_arena); cudaFreeHost(L->h_bitmap); cudaFreeHost(L->h_recovered);
  cudaFreeHost(L->h_groups); cudaFreeHost(L->h_gdev); cudaFreeHost(L->h_results);
  if (L->done_ev) cudaEventDestroy(L->done_ev);
  for (auto ev : L->chunk_ev) cudaEventDestroy(ev);
  if (L->copy_stream) cudaStreamDestroy(L->copy_stream);
  for (auto ls : L->lat_stream) if (ls) cudaStreamDestroy(ls);
  for (auto ev : L->lat_ev) if (ev) cudaEventDestroy(ev);
  for (auto ev : L->wl_ev) if (ev) cudaEventDestroy(ev);
  if (L->stream) cudaStreamDestroy(L->stream);
}

static void engine_free(ibft_engine* e) {
  if (!e) return;
  cudaSetDevice(e->p.device);
  cudaDeviceSynchronize();
  for (auto& s : e->slots) {
    if (s.d_keys) cudaFree(s.d_keys);
    if (s.d_powers) cudaFree(s.d_powers);
    cudaFree(s.d_key_state); cudaFree(s.d_key_xy); cudaFree(s.d_key_tab);
  }
  for (auto& L : e->lanes) lane_free(&L);
  cudaFree(e->d_ctable);
  cudaFree(e->d_learn_counts);
  cudaFreeHost(e->h_learn_counts);
  cudaFree(e->d_slots);
  if (e->hash_stream) cudaStreamDestroy(e->hash_stream);
  cudaFree(e->hs_arena); cudaFreeHost(e->hs_h_arena); cudaFree(e->hs_meta); cudaFreeHost(e->hs_h_meta);
  delete e;
}

static int lane_alloc(ibft_engine* e, lane* L, uint32_t cap_items, size_t cap_arena) {
  const ibft_engine_params& p = e->p;
  L->cap_items = cap_items;
  L->cap_arena = cap_arena;
  CU(cudaStreamCreateWithFlags(&L->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&L->copy_stream, cudaStreamNonBlocking));
  for (auto& ls : L->lat_stream) CU(cudaStreamCreateWithFlags(&ls, cudaStreamNonBlocking));
  for (auto& ev : L->lat_ev) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  for (auto& ev : L->wl_ev) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&L->done_ev, cudaEventDisableTiming));
  size_t n = cap_items, words = (n + 31) / 32;
  CU(cudaMalloc(&L->d_items, n * sizeof(ibft_sig_item)));
  if (p.flags & IBFT_FLAG_KEY_CACHE)
    CU(cudaMalloc(&L->d_worklist, 4 * (n + 1) * 4));  // four lists: chunks of a large host batch alternate between two streams, the
                                                      // four pieces of a mid-size round (latency path) run side by side
  CU(cudaMalloc(&L->d_arena, std::max<size_t>(cap_arena, 16)));
  CU(cudaMalloc(&L->d_bitmap, std::max<size_t>(words, 1) * 4));
  CU(cudaMalloc(&L->d_recovered, n * 20));
  CU(cudaMalloc(&L->d_status, n));
  CU(cudaHostAlloc(&L->h_status, n, cudaHostAllocDefault));
  CU(cudaMalloc(&L->d_groups, (size_t)p.max_groups * sizeof(ibft_group_desc)));
  CU(cudaMalloc(&L->d_gdev, (size_t)p.max_groups * sizeof(group_dev)));
  CU(cudaMalloc(&L->d_results, (size_t)p.max_groups * sizeof(ibft_group_result)));
  L->voted_words_cap = (size_t)p.max_groups * ((p.max_validators + 31) / 32);
  CU(cudaMalloc(&L->d_voted, std::max<size_t>(L->voted_words_cap, 1) * 4));
  CU(cudaMalloc(&L->d_nvalid, (size_t)p.max_groups * 4));
  CU(cudaHostAlloc(&L->h_items, n * sizeof(ibft_sig_item), cudaHostAllocDefault));
  CU(cudaHostAlloc(&L->h_arena, std::max<size_t>(cap_arena, 16), cudaHostAllocDefault));
  CU(cudaHostAlloc(&L->h_bitmap, std::max<size_t>(words, 1) * 4, cudaHostAllocDefault));
  CU(cudaHostAlloc(&L->h_recovered, n * 20, cudaHostAllocDefault));
  CU(cudaHostAlloc(&L->h_groups, (size_t)p.max_groups * sizeof(ibft_group_desc), cudaHostAllocDefault));
  CU(cudaHostAlloc(&L->h_gdev, (size_t)p.max_groups * sizeof(group_dev), cudaHostAllocDefault));
  CU(cudaHostAlloc(&L->h_results, (size_t)p.max_groups * sizeof(ibft_group_result), cudaHostAllocDefault));
  return IBFT_OK;
}

static int engine_alloc(ibft_engine* e) {
  const ibft_engine_params& p = e->p;
  CU(cudaSetDevice(p.device));
  CU(cudaStreamCreateWithFlags(&e->hash_stream, cudaStreamNonBlocking));
  int rc = lane_alloc(e, &e->lanes[0], p.max_items, p.max_payload_bytes);
  if (rc != IBFT_OK) return rc;
  rc = lane_alloc(e, &e->lanes[1], std::min<uint32_t>(p.max_items, IBFT_LANE1_ITEMS), std::min<size_t>(p.max_payload_bytes, IBFT_LANE1_ARENA));
  if (rc != IBFT_OK) return rc;
  lane* L = &e->lanes[0];
  if (p.flags & IBFT_FLAG_KEY_CACHE) {
    CU(cudaMalloc(&e->d_learn_counts, (size_t)p.max_table_slots * 4));
    CU(cudaMemset(e->d_learn_counts, 0, (size_t)p.max_table_slots * 4));
    CU(cudaHostAlloc(&e->h_learn_counts, (size_t)p.max_table_slots * 4, cudaHostAllocDefault));
  }
  CU(cudaMalloc(&e->d_slots, (size_t)p.max_table_slots * sizeof(slot_dev)));
  CU(cudaMemset(e->d_slots, 0, (size_t)p.max_table_slots * sizeof(slot_dev)));
  e->slots.resize(p.max_table_slots);
  e->slots_shadow.assign(p.max_table_slots, slot_dev{});
  CU(cudaMemcpyToSymbol(g_gtable, IBFT_GTABLE, sizeof(uint32_t) * IBFT_GTAB_ENTRY_WORDS * IBFT_GTAB_ENTRIES));
  CU(cudaFuncSetAttribute(k_recover<IBFT_BLOCK>, cudaFuncAttributeMaxDynamicSharedMemorySize, IBFT_BLOCK * IBFT_RTAB_WORDS * 4));
  CU(cudaFuncSetAttribute(k_recover<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * IBFT_RTAB_WORDS * 4));
#if IBFT_WC > 0
  CU(cudaFuncSetAttribute(k_recover_split, cudaFuncAttributeMaxDynamicSharedMemorySize, IBFT_SPLIT_SMEM));
  CU(cudaFuncSetAttribute(k_verify_split, cudaFuncAttributeMaxDynamicSharedMemorySize, IBFT_VSPLIT_SMEM));
#endif
  CU(cudaFuncGetAttributes(&e->recover_attr, k_recover<IBFT_BLOCK>));
  {
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, p.device));
    e->sm_count = prop.multiProcessorCount;
  }
#if IBFT_WC > 0
  {
    // position 0 is the combined table of the interleaved window loop; positions 1.. are the comb tables of the split
    // latency kernel's helper warps (36 MB in all, L2-resident while a round is being verified)
    size_t entries = (size_t)IBFT_CTAB_ENTRIES;
    CU(cudaMalloc(&e->d_ctable, (size_t)IBFT_CTAB_POSITIONS * entries * IBFT_GTAB_ENTRY_WORDS * 4));
    k_build_ctable<<<dim3((unsigned)((entries + 63) / 64), IBFT_CTAB_POSITIONS), 64, 0, L->stream>>>(e->d_ctable);
    e->launches++;
    CU(cudaGetLastError());
  }
#endif
  CU(cudaDeviceSynchronize());
  return IBFT_OK;
}

// test hook: copy `count` entries of the generator comb starting at entry `first` (64 bytes each, x then y as 8 little-endian
// words).  The positions lie back to back on the device (load_comb_pos): entry index = position * IBFT_CTAB_ENTRIES + in-position
// index, for every one of the IBFT_CTAB_POSITIONS positions.  Returns IBFT_ERR_INVALID_ARG when the library was built without a
// combined table
extern "C" int ibft_debug_ctable(ibft_engine* e, uint32_t first, uint32_t count, uint8_t* out, int* wc, uint32_t* entries) {
  if (!e) { set_err("null engine"); return IBFT_ERR_INVALID_ARG; }
  if (wc) *wc = IBFT_WC;
#if IBFT_WC > 0
  if (entries) *entries = (uint32_t)IBFT_CTAB_ENTRIES;
  if (count == 0) return IBFT_OK;
  if (!out || (size_t)first + count > (size_t)IBFT_CTAB_POSITIONS * IBFT_CTAB_ENTRIES) { set_err("range"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  CU(cudaMemcpy(out, e->d_ctable + (size_t)first * IBFT_GTAB_ENTRY_WORDS, (size_t)count * 64, cudaMemcpyDeviceToHost));
  return IBFT_OK;
#else
  if (entries) *entries = 0;
  (void)first; (void)out;
  return count == 0 ? IBFT_OK : IBFT_ERR_INVALID_ARG;
#endif
}

// test hook: copy `count` entries of validator `validator`'s key table in `slot` (entry index = position * IBFT_KEYTAB_ENTRIES +
// m - 1 holds m * 2^(8 position) * Q; same 64-byte format as ibft_debug_ctable) and its registry state
extern "C" int ibft_debug_keytab(ibft_engine* e, uint32_t slot, uint32_t validator, uint32_t first, uint32_t count, uint8_t* out,
                                 uint32_t* state_out) {
  if (!e) { set_err("null engine"); return IBFT_ERR_INVALID_ARG; }
  all_lanes_lock lk(e);
  if (slot >= e->p.max_table_slots || !e->slots[slot].valid) { set_err("slot %u not set", slot); return IBFT_ERR_NO_TABLE; }
  const slot_host& s = e->slots[slot];
  if (!s.d_key_state || validator >= s.n) { set_err("no key registry entry %u in slot %u", validator, slot); return IBFT_ERR_INVALID_ARG; }
#if IBFT_WC > 0
  if (count && (!out || (size_t)first + count > (size_t)IBFT_KEYTAB_WORDS / IBFT_GTAB_ENTRY_WORDS)) { set_err("range"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  CU(cudaDeviceSynchronize());
  if (state_out) CU(cudaMemcpy(state_out, s.d_key_state + validator, 4, cudaMemcpyDeviceToHost));
  if (count)
    CU(cudaMemcpy(out, s.d_key_tab + (size_t)validator * IBFT_KEYTAB_WORDS + (size_t)first * IBFT_GTAB_ENTRY_WORDS, (size_t)count * 64,
                  cudaMemcpyDeviceToHost));
#else
  (void)first; (void)count; (void)out; (void)state_out;
#endif
  return IBFT_OK;
}

extern "C" int ibft_engine_create(const ibft_engine_params* params, ibft_engine** out) {
  if (!params || !out) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  *out = nullptr;
  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess || count <= 0) {
    set_err("no CUDA device available (%s): this engine has no CPU fallback", ce != cudaSuccess ? cudaGetErrorString(ce) : "device count 0");
    return IBFT_ERR_NO_DEVICE;
  }
  if (params->device < 0 || params->device >= count || params->max_items == 0 || params->max_groups == 0 ||
      params->max_groups > 65535 || params->max_table_slots == 0 || params->max_table_slots > 65535) {
    set_err("invalid engine parameters");
    return IBFT_ERR_INVALID_ARG;
  }
  ibft_engine* e = new ibft_engine();
  e->p = *params;
  e->p.max_items = (e->p.max_items + 31u) & ~31u;
  int rc = engine_alloc(e);
  if (rc != IBFT_OK) { engine_free(e); return rc; }
  *out = e;
  return IBFT_OK;
}

extern "C" void ibft_engine_destroy(ibft_engine* e) { engine_free(e); }

extern "C" int ibft_engine_device_info(ibft_engine* e, ibft_device_info* out) {
  if (!e || !out) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, e->p.device));
  memset(out, 0, sizeof *out);
  snprintf(out->name, sizeof out->name, "%.63s", prop.name);
  out->sm_count = prop.multiProcessorCount;
  out->cc_major = prop.major;
  out->cc_minor = prop.minor;
  int khz = 0;
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, e->p.device);
  out->clock_khz = khz;
  out->total_mem = prop.totalGlobalMem;
  out->abi_version = IBFT_ABI_VERSION;
  out->kernel_regs = e->recover_attr.numRegs;
  out->kernel_smem_bytes = (int32_t)e->recover_attr.sharedSizeBytes + IBFT_BLOCK * IBFT_RTAB_WORDS * 4;
  out->block_threads = IBFT_BLOCK;
  return IBFT_OK;
}

// 256-bit big-endian -> 4 little-endian u64 limbs
static void be32_to_limbs(const uint8_t* b, uint64_t l[4]) {
  for (int i = 0; i < 4; i++) {
    uint64_t w = 0;
    for (int j = 0; j < 8; j++) w = (w << 8) | b[(3 - i) * 8 + j];
    l[i] = w;
  }
}

extern "C" int ibft_set_validators(ibft_engine* e, uint32_t table_slot, uint64_t height, const uint8_t* addrs,
                                   const uint8_t* powers_be, uint32_t n) {
  if (!e || (!addrs && n)) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (table_slot >= e->p.max_table_slots) { set_err("table slot %u out of range", table_slot); return IBFT_ERR_INVALID_ARG; }
  if (n > e->p.max_validators) { set_err("validator table of %u exceeds capacity %u", n, e->p.max_validators); return IBFT_ERR_CAPACITY; }
  // total voting power and quorum = floor(2*total/3) + 1 in 320-bit arithmetic (validator_manager.go:130-135)
  std::vector<uint64_t> powers((size_t)n * 4);
  uint64_t total[5] = {0, 0, 0, 0, 0};
  for (uint32_t i = 0; i < n; i++) {
    uint64_t l[4] = {1, 0, 0, 0};
    if (powers_be) be32_to_limbs(powers_be + 32 * (size_t)i, l);
    memcpy(&powers[4 * (size_t)i], l, sizeof l);
    unsigned __int128 c = 0;
    for (int k = 0; k < 5; k++) {
      c += (unsigned __int128)total[k] + (k < 4 ? l[k] : 0);
      total[k] = (uint64_t)c;
      c >>= 64;
    }
  }
  if ((total[0] | total[1] | total[2] | total[3] | total[4]) == 0) {
    set_err("total voting power is zero or less");
    return IBFT_ERR_VOTING_POWER;
  }
  uint64_t twice[6] = {0, 0, 0, 0, 0, 0};
  {
    uint64_t c = 0;
    for (int k = 0; k < 5; k++) { twice[k] = (total[k] << 1) | c; c = total[k] >> 63; }
    twice[5] = c;
  }
  uint64_t q[6];
  {
    unsigned __int128 rem = 0;
    for (int k = 5; k >= 0; k--) {
      unsigned __int128 cur = (rem << 64) | twice[k];
      q[k] = (uint64_t)(cur / 3);
      rem = cur % 3;
    }
    unsigned __int128 c = 1;
    for (int k = 0; k < 6; k++) { c += q[k]; q[k] = (uint64_t)c; c >>= 64; }
  }
  // sorted key table: 5 big-endian words + validator index
  std::vector<uint32_t> order(n);
  for (uint32_t i = 0; i < n; i++) order[i] = i;
  std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
    int c = memcmp(addrs + 20 * (size_t)a, addrs + 20 * (size_t)b, 20);
    return c != 0 ? c < 0 : a < b;
  });
  std::vector<uint32_t> keys((size_t)n * 6);
  for (uint32_t r = 0; r < n; r++) {
    const uint8_t* a = addrs + 20 * (size_t)order[r];
    for (int w = 0; w < 5; w++)
      keys[6 * (size_t)r + w] = ((uint32_t)a[4 * w] << 24) | ((uint32_t)a[4 * w + 1] << 16) | ((uint32_t)a[4 * w + 2] << 8) | a[4 * w + 3];
    keys[6 * (size_t)r + 5] = order[r];
  }
  // replacing a table frees device memory the kernels of ANY lane may be reading: take every lane and drain the device
  all_lanes_lock lk(e);
  for (auto& L : e->lanes)
    if (L.pending.active) { set_err("a submitted call is still pending; wait for it first"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  slot_host& s = e->slots[table_slot];
  CU(cudaDeviceSynchronize());
  // the slot's previous content stays alive until its key registry has been carried over
  slot_host old = s;
  slot_dev old_dev = e->slots_shadow[table_slot];
  s = slot_host{};
  int rc_alloc = IBFT_OK;
  do {
    cudaError_t ce = cudaMalloc(&s.d_keys, std::max<size_t>(keys.size(), 6) * 4);
    if (ce == cudaSuccess) ce = cudaMalloc(&s.d_powers, std::max<size_t>(powers.size(), 4) * 8);
    if (ce == cudaSuccess && n) ce = cudaMemcpy(s.d_keys, keys.data(), keys.size() * 4, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess && n) ce = cudaMemcpy(s.d_powers, powers.data(), powers.size() * 8, cudaMemcpyHostToDevice);
#if IBFT_WC > 0
    if (ce == cudaSuccess && (e->p.flags & IBFT_FLAG_KEY_CACHE) && n) {
      ce = cudaMalloc(&s.d_key_state, (size_t)n * 4);
      if (ce == cudaSuccess) ce = cudaMalloc(&s.d_key_xy, (size_t)n * 64);
      if (ce == cudaSuccess) ce = cudaMalloc(&s.d_key_tab, (size_t)n * IBFT_KEYTAB_WORDS * 4);  // 136 KiB per validator (comb)
      if (ce == cudaSuccess) ce = cudaMemset(s.d_key_state, 0, (size_t)n * 4);
      s.d_learn_count = e->d_learn_counts + table_slot;
    }
#endif
    if (ce != cudaSuccess) {
      set_err("validator table of %u validators%s: %s", n, (e->p.flags & IBFT_FLAG_KEY_CACHE) ? " with its key registry (136 KiB per validator)" : "",
              cudaGetErrorString(ce));
      rc_alloc = ce == cudaErrorMemoryAllocation ? IBFT_ERR_CAPACITY : IBFT_ERR_CUDA;
      (void)cudaGetLastError();
    }
  } while (0);
  if (rc_alloc != IBFT_OK) {  // the slot keeps its previous table
    cudaFree(s.d_keys); cudaFree(s.d_powers); cudaFree(s.d_key_state); cudaFree(s.d_key_xy); cudaFree(s.d_key_tab);
    s = old;
    return rc_alloc;
  }
  if (s.d_learn_count) CU(cudaMemset(s.d_learn_count, 0, 4));  // a new validator set starts with an empty registry (then the carry-over)
  s.n = n;
  s.height = height;
  memcpy(s.quorum, q, sizeof s.quorum);
  s.valid = true;
  slot_dev sd{};
  sd.keys = s.d_keys;
  sd.powers = s.d_powers;
  sd.key_state = s.d_key_state;
  sd.key_xy = s.d_key_xy;
  sd.key_tab = s.d_key_tab;
  sd.learn_count = s.d_learn_count;
  memcpy(sd.quorum, q, sizeof sd.quorum);
  sd.n = n;
  sd.valid = 1;
#if IBFT_WC > 0
  if (s.d_key_state) {
    // carry the keys over from the donor table: the resident table of the greatest height that has a registry (the previous
    // block, normally) -- this slot's previous content included
    const slot_dev* donor = nullptr;
    uint64_t best_h = 0;
    if (old.valid && old.d_key_state && old.n) { donor = &old_dev; best_h = old.height; }
    for (uint32_t k = 0; k < e->p.max_table_slots; k++) {
      const slot_host& o = e->slots[k];
      if (k == table_slot || !o.valid || !o.d_key_state || !o.n) continue;
      if (donor == nullptr || o.height > best_h) { donor = &e->slots_shadow[k]; best_h = o.height; }
    }
    if (donor != nullptr) {
      k_carry_keys<<<n, 256>>>(sd, *donor);
      e->launches++;
      CU(cudaGetLastError());
      CU(cudaDeviceSynchronize());
      CU(cudaMemcpy(&s.built_count, s.d_learn_count, 4, cudaMemcpyDeviceToHost));  // carried keys come with finished tables
    }
  }
#endif
  if (old.d_keys) cudaFree(old.d_keys);
  if (old.d_powers) cudaFree(old.d_powers);
  cudaFree(old.d_key_state); cudaFree(old.d_key_xy); cudaFree(old.d_key_tab);
  e->slots_shadow[table_slot] = sd;
  CU(cudaMemcpy(e->d_slots + table_slot, &sd, sizeof sd, cudaMemcpyHostToDevice));
  return IBFT_OK;
}

// Key registry upkeep: for every resident validator table, build the tables of multiples of the keys learned since the last
// call.  Cheap when nothing is new (one 4-byte read per slot).  ibft_verify_batch / ibft_verify_wait call it on their way out;
// callers of the device-resident entry points call it between rounds.
static int refresh_key_tables_locked(ibft_engine* e, lane* L, uint32_t* n_ready_out) {
  uint32_t total = 0;
#if IBFT_WC > 0
  if ((e->p.flags & IBFT_FLAG_KEY_CACHE) && e->d_learn_counts) {
    std::lock_guard<std::mutex> kl(e->keys_mu);
    CU(cudaSetDevice(e->p.device));
    CU(cudaMemcpyAsync(e->h_learn_counts, e->d_learn_counts, (size_t)e->p.max_table_slots * 4, cudaMemcpyDeviceToHost, L->stream));
    CU(cudaStreamSynchronize(L->stream));
    bool built = false;
    for (uint32_t slot = 0; slot < e->p.max_table_slots; slot++) {
      slot_host& s = e->slots[slot];
      if (!s.valid || !s.d_learn_count) continue;
      uint32_t learned = e->h_learn_counts[slot];
      if (learned > s.built_count) {
        k_keytabs_step<<<(s.n + 255) / 256, 256, 0, L->stream>>>(e->d_slots, slot, IBFT_KEY_LEARNED, IBFT_KEY_BUILDING);
        k_build_keytabs<<<(uint32_t)(((size_t)s.n * IBFT_KEYTAB_POSITIONS + 63) / 64), 64, 0, L->stream>>>(e->d_slots, slot);
        k_keytabs_step<<<(s.n + 255) / 256, 256, 0, L->stream>>>(e->d_slots, slot, IBFT_KEY_BUILDING, IBFT_KEY_READY);
        e->launches += 3;
        CU(cudaGetLastError());
        s.built_count = learned;
        built = true;
      }
      total += learned;
    }
    // the tables are complete before anybody can launch the next round on another stream
    if (built) CU(cudaStreamSynchronize(L->stream));
  }
#endif
  if (n_ready_out) *n_ready_out = total;
  return IBFT_OK;
}
extern "C" int ibft_refresh_key_tables(ibft_engine* e, uint32_t* n_keys_out) {
  if (!e) { set_err("null engine"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  if (L->pending.active) { set_err("a submitted call is still pending"); return IBFT_ERR_INVALID_ARG; }
  return refresh_key_tables_locked(e, L, n_keys_out);
}

extern "C" int ibft_get_quorum(ibft_engine* e, uint32_t table_slot, uint64_t quorum_out[5], uint64_t* height_out,
                               uint32_t* n_out) {
  if (!e || table_slot >= e->p.max_table_slots) { set_err("bad slot"); return IBFT_ERR_INVALID_ARG; }
  std::lock_guard<std::mutex> lk(e->lanes[0].mu);
  const slot_host& s = e->slots[table_slot];
  if (!s.valid) { set_err("slot %u not set", table_slot); return IBFT_ERR_NO_TABLE; }
  if (quorum_out) memcpy(quorum_out, s.quorum, sizeof s.quorum);
  if (height_out) *height_out = s.height;
  if (n_out) *n_out = s.n;
  return IBFT_OK;
}

// lay out the voted sets of the call's groups; validates table slots
static int plan_groups(ibft_engine* e, lane* L, const ibft_group_desc* groups, uint32_t n_groups, group_dev* gdev, size_t* total_words) {
  size_t off = 0;
  for (uint32_t g = 0; g < n_groups; g++) {
    uint32_t slot = groups[g].table_slot;
    uint32_t nw = 0;
    if (slot != IBFT_NO_TABLE) {
      if (slot >= e->p.max_table_slots || !e->slots[slot].valid) {
        set_err("group %u references validator-table slot %u which is not set", g, slot);
        return IBFT_ERR_NO_TABLE;
      }
      // IsValidValidator answers for the validator set AT THE MESSAGE'S HEIGHT (core/backend.go:41-45): a slot that has been
      // recycled for another height must never answer for this one
      if (e->slots[slot].height != groups[g].height) {
        set_err("group %u is for height %llu but validator-table slot %u holds height %llu", g, (unsigned long long)groups[g].height,
                slot, (unsigned long long)e->slots[slot].height);
        return IBFT_ERR_NO_TABLE;
      }
      nw = (e->slots[slot].n + 31) / 32;
    }
    gdev[g].voted_off = (uint32_t)off;
    gdev[g].n_words = nw;
    off += nw;
  }
  if (off > L->voted_words_cap) { set_err("voted sets of the call exceed capacity"); return IBFT_ERR_CAPACITY; }
  *total_words = off;
  return IBFT_OK;
}

static int launch_recover(ibft_engine* e, lane* L, const ibft_sig_item* d_items, uint32_t n, const uint8_t* d_arena, size_t arena_len,
                          uint32_t lo, uint32_t hi, const ibft_group_desc* d_groups, uint32_t n_groups, uint32_t* d_bitmap,
                          uint8_t* d_recovered, cudaStream_t st, uint8_t* d_status = nullptr, int forced_path = IBFT_PATH_AUTO,
                          vote_sink sink = vote_sink{nullptr, nullptr, nullptr}, uint32_t worklist_index = 0) {
  if (hi <= lo) return IBFT_OK;
  uint32_t* const worklist = L->d_worklist ? L->d_worklist + (size_t)worklist_index * ((size_t)L->cap_items + 1) : nullptr;
  // path selection (ibft_set_recover_path).  AUTO picks by how many warps each of the SM's four schedulers would hold
  // (B200, kernel time of one batch: profiles/latency_r01_v9.md):
  //   <= SMs x 24 signatures   four-lane chain warps + helper warp, one CTA (3 + 1 warps) per SM                   0.41 ms
  //   <= SMs x 48              the same, two CTAs per SM (two warps per scheduler)                                  0.51 ms
  //   <= SMs x 96              chain warps + helper warp, one CTA (3 + 1 warps) per SM (a 10k-validator round)      0.68 ms
  //   <= SMs x 192             the same, two CTAs per SM (one-thread kernel: 1.16 ms)                               0.90 ms
  //   beyond                   one thread per signature: one-warp CTAs while one wave covers them, then the 128-thread
  //                            throughput kernel
  const uint32_t cnt = hi - lo;
  int path = forced_path != IBFT_PATH_AUTO ? forced_path : e->recover_path.load();
  // key-registry path possible: the worklist holds max_items indices (a larger device-resident shard takes the plain recover
  // path), recovered addresses are not wanted, groups are bound
  const bool known_ok = (e->p.flags & IBFT_FLAG_KEY_CACHE) && d_recovered == nullptr && d_groups != nullptr && worklist != nullptr &&
                        cnt <= L->cap_items;
  // ... and its latency form: one-warp CTAs spread a round over all SMs, and whatever the verification does not accept is
  // recovered by the four-lane kernel in worklist mode (short payloads only: its helper warp hashes for 24 signatures)
  const bool small_batch = cnt <= (uint32_t)e->sm_count * 32u * 8u;
  if (path == IBFT_PATH_AUTO) {
#if IBFT_WC > 0
    // with learned keys, verifying against the validator's comb table (51 additions, no doubling) beats every recover kernel at
    // every batch size -- also the four-lane one: the known-key pass goes first, the recover kernels take what it leaves over
    if (known_ok) path = IBFT_PATH_THREAD;
    else
    // long payloads (ROUND_CHANGE messages with their certificates: up to 909 KB of signed bytes each): the helper warp of the
    // latency kernels hashes for three (or 24) signatures one after the other, which serialises the sponges that dominate such a
    // batch -- one thread per signature hashes them all in parallel (config 4, 10,000 x 909 KB: 156 ms -> see DESIGN.md §6)
    if (arena_len / cnt > 256) path = IBFT_PATH_THREAD;
    else if (cnt <= (uint32_t)e->sm_count * 2u * IBFT_QSPLIT_SIGS) path = IBFT_PATH_QSPLIT;
    else if (cnt <= (uint32_t)e->sm_count * 2u * IBFT_SPLIT_SIGS) path = IBFT_PATH_SPLIT;
    else path = IBFT_PATH_THREAD;
#else
    path = cnt <= (uint32_t)e->sm_count * IBFT_QUAD_SIGS ? IBFT_PATH_QUAD : IBFT_PATH_THREAD;
#endif
  }
#if IBFT_WC > 0
  if (path == IBFT_PATH_QSPLIT) {
    uint32_t blocks = (cnt + IBFT_QSPLIT_SIGS - 1) / IBFT_QSPLIT_SIGS;
    CU(cudaMemsetAsync(d_bitmap + (lo >> 5), 0, (size_t)((hi + 31) / 32 - (lo >> 5)) * 4, st));  // verdict bits are OR-ed in
    k_recover_qsplit<<<blocks, 128, 0, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots,
                                             e->p.max_table_slots, d_bitmap, d_recovered, d_status, e->d_ctable, sink, nullptr);
  } else if (path == IBFT_PATH_SPLIT && known_ok) {
    // known-key latency path: verify against the learned keys, then recover whatever was not accepted (worklist; the second
    // launch finds it empty -- and returns at once -- when every signature of the round verified)
    uint32_t blocks = (cnt + IBFT_SPLIT_SIGS - 1) / IBFT_SPLIT_SIGS;
    CU(cudaStreamWaitEvent(st, L->wl_ev[worklist_index & 3u], 0));
    CU(cudaMemsetAsync(worklist, 0, 4, st));
    L->wl_used |= 1u << (worklist_index & 3u);
    k_verify_split<<<blocks, 32 * (IBFT_SPLIT_CHAINS + 1), IBFT_VSPLIT_SMEM, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups,
                                                                              e->d_slots, e->p.max_table_slots, d_bitmap, d_status, e->d_ctable,
                                                                              sink, worklist);
    e->launches++;
    CU(cudaGetLastError());
    uint32_t blocks2 = (cnt + IBFT_QSPLIT_SIGS - 1) / IBFT_QSPLIT_SIGS;
    k_recover_qsplit<<<blocks2, 128, 0, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots, e->p.max_table_slots,
                                              d_bitmap, nullptr, nullptr, e->d_ctable, sink, worklist);
    CU(cudaEventRecord(L->wl_ev[worklist_index & 3u], st));
  } else if (path == IBFT_PATH_SPLIT) {
    uint32_t blocks = (cnt + IBFT_SPLIT_SIGS - 1) / IBFT_SPLIT_SIGS;
    k_recover_split<<<blocks, 32 * (IBFT_SPLIT_CHAINS + 1), IBFT_SPLIT_SMEM, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups,
                                                                              e->d_slots, e->p.max_table_slots, d_bitmap, d_recovered,
                                                                              d_status, e->d_ctable, sink);
  } else
#endif
  if (path == IBFT_PATH_QUAD) {
    uint32_t blocks = (cnt + IBFT_QUAD_SIGS - 1) / IBFT_QUAD_SIGS;
    k_recover_quad<<<blocks, 4 * IBFT_QUAD_SIGS, 0, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots,
                                                         e->p.max_table_slots, d_bitmap, d_recovered, d_status, e->d_ctable, sink);
  } else
#if IBFT_WC > 0
  if (known_ok) {
    // key-registry path (one thread per signature, any batch size): verify what can be verified, then recover the rest from
    // the worklist (dense second launch; the threads beyond the worklist's length leave at once)
    // device-resident callers may use different streams: launches sharing a worklist are ordered on the device
    CU(cudaStreamWaitEvent(st, L->wl_ev[worklist_index & 3u], 0));
    CU(cudaMemsetAsync(worklist, 0, 4, st));
    L->wl_used |= 1u << (worklist_index & 3u);
    if (small_batch) {
      k_verify_known<32><<<(cnt + 31) / 32, 32, 0, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots,
                                                        e->p.max_table_slots, d_bitmap, d_status, e->d_ctable, sink, worklist);
    } else {
      k_verify_known<IBFT_BLOCK><<<(cnt + IBFT_BLOCK - 1) / IBFT_BLOCK, IBFT_BLOCK, 0, st>>>(
          d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots, e->p.max_table_slots, d_bitmap, d_status, e->d_ctable, sink,
          worklist);
    }
    e->launches++;
    CU(cudaGetLastError());
    if (small_batch && arena_len / cnt <= 256) {
      k_recover_qsplit<<<(cnt + IBFT_QSPLIT_SIGS - 1) / IBFT_QSPLIT_SIGS, 128, 0, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups,
                                                                                    e->d_slots, e->p.max_table_slots, d_bitmap, nullptr, nullptr,
                                                                                    e->d_ctable, sink, worklist);
    } else {
      k_recover<IBFT_BLOCK><<<(cnt + IBFT_BLOCK - 1) / IBFT_BLOCK, IBFT_BLOCK, IBFT_BLOCK * IBFT_RTAB_WORDS * 4, st>>>(
          d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots, e->p.max_table_slots, d_bitmap, nullptr, nullptr, e->d_ctable,
          sink, worklist);
    }
    CU(cudaEventRecord(L->wl_ev[worklist_index & 3u], st));
  } else
#endif
  if (small_batch) {  // one-warp CTAs
    uint32_t blocks = (cnt + 31) / 32;
    k_recover<32><<<blocks, 32, 32 * IBFT_RTAB_WORDS * 4, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots,
                                         e->p.max_table_slots, d_bitmap, d_recovered, d_status, e->d_ctable, sink, nullptr);
  } else {
    uint32_t blocks = (cnt + IBFT_BLOCK - 1) / IBFT_BLOCK;
    k_recover<IBFT_BLOCK><<<blocks, IBFT_BLOCK, IBFT_BLOCK * IBFT_RTAB_WORDS * 4, st>>>(d_items, n, d_arena, arena_len, lo, hi, d_groups, n_groups, e->d_slots,
                                                         e->p.max_table_slots, d_bitmap, d_recovered, d_status, e->d_ctable, sink, nullptr);
  }
  e->launches++;
  CU(cudaGetLastError());
  return IBFT_OK;
}

static int launch_quorum(ibft_engine* e, lane* L, const ibft_sig_item* d_items, uint32_t n, const uint8_t* d_arena, size_t arena_len, const uint32_t* d_bitmap,
                         const ibft_group_desc* d_groups, const group_dev* d_gdev, uint32_t n_groups, size_t voted_words,
                         ibft_group_result* d_results, cudaStream_t st, bool already_marked = false) {
  if (n_groups == 0) return IBFT_OK;
  if (!already_marked) {
    CU(cudaMemsetAsync(L->d_voted, 0, std::max<size_t>(voted_words, 1) * 4, st));
    CU(cudaMemsetAsync(L->d_nvalid, 0, (size_t)n_groups * 4, st));
  }
  if (n && !already_marked) {
    k_quorum_mark<<<(n + 255) / 256, 256, 0, st>>>(d_items, n, d_arena, arena_len, d_bitmap, d_groups, d_gdev, n_groups, e->d_slots,
                                                    e->p.max_table_slots, L->d_voted, L->d_nvalid, 0u, n);
    e->launches++;
    CU(cudaGetLastError());
  }
  k_quorum_reduce<<<n_groups, IBFT_REDUCE_THREADS, 0, st>>>(d_groups, d_gdev, n_groups, e->d_slots, e->p.max_table_slots, L->d_voted,
                                            L->d_nvalid, d_results);
  e->launches++;
  CU(cudaGetLastError());
  return IBFT_OK;
}

// Staging copy of a chunk of pageable caller memory (a cgo caller's Go heap) into the lane's pinned buffer.  One thread moves
// ~4 GB/s on the GPU boxes' hosts -- 134 MB of tuples would take longer than the kernels that consume them -- so large chunks are
// split over a few short-lived helper threads (the copy of chunk k+1 already overlaps the device work on chunk k).
static void stage_copy(void* dst, const void* src, size_t bytes) {
  const size_t kMin = 2u << 20;
  if (bytes < 2 * kMin) { memcpy(dst, src, bytes); return; }
  const unsigned parts = (unsigned)std::min<size_t>(4, bytes / kMin);
  const size_t per = (bytes / parts + 63) & ~(size_t)63;
  std::thread th[3];
  unsigned started = 0;
  for (unsigned k = 1; k < parts; k++) {
    size_t off = k * per, len = k + 1 == parts ? bytes - off : per;
    th[started++] = std::thread([=]() { memcpy((char*)dst + off, (const char*)src + off, len); });
  }
  memcpy(dst, src, std::min(per, bytes));
  for (unsigned k = 0; k < started; k++) th[k].join();
}

static int submit_locked(ibft_engine* e, lane* L, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                         const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out,
                         ibft_group_result* results_out, uint8_t* recovered_out) {
  if (L->pending.active) { set_err("a submitted call is still pending; wait for it first"); return IBFT_ERR_INVALID_ARG; }
  if ((n && !items) || (n && !bitmap_out) || (arena_len && !arena) || (n_groups && !groups)) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (n > L->cap_items || arena_len > L->cap_arena || n_groups > e->p.max_groups) {
    set_err("batch (%u items, %zu payload bytes, %u groups) exceeds engine capacity (%u, %zu, %u)", n, arena_len, n_groups,
            L->cap_items, L->cap_arena, e->p.max_groups);
    return IBFT_ERR_CAPACITY;
  }
  CU(cudaSetDevice(e->p.device));
  size_t voted_words = 0;
  if (n_groups) {
    int rc = plan_groups(e, L, groups, n_groups, L->h_gdev, &voted_words);
    if (rc != IBFT_OK) return rc;
    memcpy(L->h_groups, groups, (size_t)n_groups * sizeof(ibft_group_desc));
    L->last_gdev.assign(L->h_gdev, L->h_gdev + n_groups);
    L->last_groups.assign(groups, groups + n_groups);
  } else {
    L->last_gdev.clear();
    L->last_groups.clear();
  }
  cudaStream_t st = L->stream;
  L->wl_used = 0;
  if (arena_len) {
    memcpy(L->h_arena, arena, arena_len);
    CU(cudaMemcpyAsync(L->d_arena, L->h_arena, arena_len, cudaMemcpyHostToDevice, st));
  }
  if (n_groups) {
    CU(cudaMemcpyAsync(L->d_groups, L->h_groups, (size_t)n_groups * sizeof(ibft_group_desc), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(L->d_gdev, L->h_gdev, (size_t)n_groups * sizeof(group_dev), cudaMemcpyHostToDevice, st));
  }
  // quorum requested: the recover kernels record the votes themselves (no k_quorum_mark pass over the tuples afterwards)
  vote_sink sink{nullptr, nullptr, nullptr};
  if (n_groups && results_out) {
    CU(cudaMemsetAsync(L->d_voted, 0, std::max<size_t>(voted_words, 1) * 4, st));
    CU(cudaMemsetAsync(L->d_nvalid, 0, (size_t)n_groups * 4, st));
    sink = vote_sink{L->d_voted, L->d_nvalid, L->d_gdev};
  }
  // Tuples go up in chunks: while the recover kernel works on chunk k, the host stages chunk k+1 into pinned memory and the
  // copy engine moves it (two streams + events).  Small batches are a single chunk.
  const uint32_t CHUNK = 1u << 17;
  uint32_t n_chunks = n ? (n + CHUNK - 1) / CHUNK : 0;  // (not const: the latency path below takes the round over)
  while (L->chunk_ev.size() < n_chunks + 1) {
    cudaEvent_t ev;
    CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    L->chunk_ev.push_back(ev);
  }
  if (n_chunks > 1) {  // the copy stream must see the arena / groups uploads of this call
    CU(cudaEventRecord(L->chunk_ev[n_chunks], st));
    CU(cudaStreamWaitEvent(L->copy_stream, L->chunk_ev[n_chunks], 0));
  }
  int rc = IBFT_OK;
#if IBFT_WC > 0
  // One mid-size round (the chain + helper kernel's range, e.g. 10,000 seals = 1.28 MB of tuples): the staging copy and the
  // H2D transfer would sit in front of a kernel that cannot start before its last tuple has arrived.  Cut the round into four
  // pieces, each with its own stream -- stage, copy and launch piece k while piece k+1 is being staged; the four kernels
  // (<= 37 CTAs each) run side by side on different SMs and the main stream joins them before the quorum kernels.
  const bool lat_pieces = e->recover_path.load() == IBFT_PATH_AUTO && n > (uint32_t)e->sm_count * 2u * IBFT_QSPLIT_SIGS &&
                          n <= (uint32_t)e->sm_count * IBFT_SPLIT_SIGS && arena_len / n <= 256;
  if (lat_pieces) {
    bool pinned = false;
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, items) == cudaSuccess) pinned = pa.type == cudaMemoryTypeHost;
    else (void)cudaGetLastError();
    CU(cudaEventRecord(L->lat_ev[4], st));  // arena / groups uploads of this call
    const uint32_t per = ((n + 3) / 4 + IBFT_SPLIT_SIGS - 1) / IBFT_SPLIT_SIGS * IBFT_SPLIT_SIGS;
    // with a key registry the pieces go through the known-key pass (one-warp CTAs) + worklist; without, chain + helper warps
    const int piece_path = ((e->p.flags & IBFT_FLAG_KEY_CACHE) && !recovered_out && n_groups && L->d_worklist) ? IBFT_PATH_THREAD : IBFT_PATH_SPLIT;
    for (uint32_t c = 0; c < 4; c++) {
      uint32_t lo = std::min(n, c * per), hi = std::min(n, lo + per);
      if (hi <= lo) break;
      cudaStream_t ls = L->lat_stream[c];
      const ibft_sig_item* src = items + lo;
      if (!pinned) {
        memcpy(L->h_items + lo, items + lo, (size_t)(hi - lo) * sizeof(ibft_sig_item));
        src = L->h_items + lo;
      }
      CU(cudaStreamWaitEvent(ls, L->lat_ev[4], 0));
      CU(cudaMemcpyAsync(L->d_items + lo, src, (size_t)(hi - lo) * sizeof(ibft_sig_item), cudaMemcpyHostToDevice, ls));
      rc = launch_recover(e, L, L->d_items, n, L->d_arena, arena_len, lo, hi, n_groups ? L->d_groups : nullptr, n_groups, L->d_bitmap,
                          recovered_out ? L->d_recovered : nullptr, ls, L->d_status, piece_path, sink, c);
      if (rc != IBFT_OK) return rc;
      CU(cudaEventRecord(L->lat_ev[c], ls));
      CU(cudaStreamWaitEvent(st, L->lat_ev[c], 0));
    }
    n_chunks = 0;  // the generic chunk loop below has nothing left to do
  }
#endif
  // A caller that already holds the tuples in page-locked memory (cudaHostAlloc / cudaHostRegister, e.g. torch pin_memory)
  // is copied from directly; pageable memory (Go heap through cgo) goes through the engine's pinned staging first.
  bool caller_pinned = false;
  if (n) {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, items) == cudaSuccess) caller_pinned = pa.type == cudaMemoryTypeHost;
    else (void)cudaGetLastError();
  }
  // Several chunks: chunk c's kernels run on one of two alternating streams, so that the tail of one chunk (the last CTAs of a
  // 1,024-CTA launch on 444 resident slots) overlaps the head of the next instead of idling the SMs eight times per batch.
  if (n_chunks > 1) {
    CU(cudaEventRecord(L->lat_ev[4], st));  // arena / groups uploads and the vote-sink memsets of this call
    CU(cudaStreamWaitEvent(L->lat_stream[0], L->lat_ev[4], 0));
    CU(cudaStreamWaitEvent(L->lat_stream[1], L->lat_ev[4], 0));
  }
  for (uint32_t c = 0; c < n_chunks; c++) {
    uint32_t lo = c * CHUNK, hi = std::min(n, lo + CHUNK);
    const ibft_sig_item* src = items + lo;
    if (!caller_pinned) {
      stage_copy(L->h_items + lo, items + lo, (size_t)(hi - lo) * sizeof(ibft_sig_item));
      src = L->h_items + lo;
    }
    cudaStream_t cs = n_chunks > 1 ? L->copy_stream : st;
    cudaStream_t ks = n_chunks > 1 ? L->lat_stream[c & 1u] : st;
    CU(cudaMemcpyAsync(L->d_items + lo, src, (size_t)(hi - lo) * sizeof(ibft_sig_item), cudaMemcpyHostToDevice, cs));
    if (n_chunks > 1) {
      CU(cudaEventRecord(L->chunk_ev[c], cs));
      CU(cudaStreamWaitEvent(ks, L->chunk_ev[c], 0));
    }
    rc = launch_recover(e, L, L->d_items, n, L->d_arena, arena_len, lo, hi, n_groups ? L->d_groups : nullptr, n_groups, L->d_bitmap,
                        recovered_out ? L->d_recovered : nullptr, ks, L->d_status, IBFT_PATH_AUTO, sink, c & 1u);
    if (rc != IBFT_OK) return rc;
  }
  if (n_chunks > 1) {
    for (int k = 0; k < 2; k++) {
      CU(cudaEventRecord(L->lat_ev[k], L->lat_stream[k]));
      CU(cudaStreamWaitEvent(st, L->lat_ev[k], 0));
    }
  }
  if (n_groups && results_out) {
    rc = launch_quorum(e, L, L->d_items, n, L->d_arena, arena_len, L->d_bitmap, L->d_groups, L->d_gdev, n_groups, voted_words, L->d_results, st,
                       /*already_marked=*/true);
    if (rc != IBFT_OK) return rc;
    CU(cudaMemcpyAsync(L->h_results, L->d_results, (size_t)n_groups * sizeof(ibft_group_result), cudaMemcpyDeviceToHost, st));
  }
  if (n) {
    CU(cudaMemcpyAsync(L->h_status, L->d_status, (size_t)n, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(L->h_bitmap, L->d_bitmap, (size_t)((n + 31) / 32) * 4, cudaMemcpyDeviceToHost, st));
    if (recovered_out) CU(cudaMemcpyAsync(L->h_recovered, L->d_recovered, (size_t)n * 20, cudaMemcpyDeviceToHost, st));
  }
  CU(cudaEventRecord(L->done_ev, st));
  L->pending.active = true;
  L->pending.n = n;
  L->pending.n_groups = (n_groups && results_out) ? n_groups : 0;
  L->pending.bitmap_out = bitmap_out;
  L->pending.results_out = results_out;
  L->pending.recovered_out = recovered_out;
  return IBFT_OK;
}

static int wait_locked(ibft_engine* e, lane* L) {
  if (!L->pending.active) { set_err("no submitted call to wait for"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  cudaError_t ce = cudaEventSynchronize(L->done_ev);
  pending_call pc = L->pending;
  L->pending.active = false;
  if (ce != cudaSuccess) {
    // launch/execution failure: NO verdict is produced (outputs untouched) -- never `true` (SURVEY.md §5)
    set_err("device execution failed: %s", cudaGetErrorString(ce));
    return IBFT_ERR_CUDA;
  }
  L->last_status_n = pc.n;
  if (pc.n) {
    size_t words = (pc.n + 31) / 32;
    memcpy(pc.bitmap_out, L->h_bitmap, words * 4);
    if (pc.n & 31) pc.bitmap_out[words - 1] &= (1u << (pc.n & 31)) - 1u;
    if (pc.recovered_out) memcpy(pc.recovered_out, L->h_recovered, (size_t)pc.n * 20);
  }
  if (pc.n_groups) memcpy(pc.results_out, L->h_results, (size_t)pc.n_groups * sizeof(ibft_group_result));
  e->last_lane.store((int)(L - e->lanes));
  if (e->p.flags & IBFT_FLAG_KEY_CACHE) return refresh_key_tables_locked(e, L, nullptr);  // new keys -> tables, for the next call
  return IBFT_OK;
}

// Lane selection for a synchronous host-buffer call: a call that fits the small lane takes whichever lane is free (small lane
// first, so that bulk callers find lane 0 free); a large call always takes lane 0.  Returns with the lane's mutex HELD.
static lane* acquire_lane(ibft_engine* e, uint32_t n, size_t arena_len) {
  lane* big = &e->lanes[0];
  lane* small = &e->lanes[1];
  const bool fits_small = n <= small->cap_items && arena_len <= small->cap_arena;
  if (fits_small) {
    if (small->mu.try_lock()) return small;
    if (big->mu.try_lock()) {
      if (!big->pending.active) return big;
      big->mu.unlock();
    }
    small->mu.lock();
    return small;
  }
  big->mu.lock();
  return big;
}

static int verify_batch_on_lane(ibft_engine* e, lane* L, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                                const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out, ibft_group_result* results_out,
                                uint8_t* recovered_out, uint8_t* status_out, uint32_t* voted_out, uint32_t voted_stride_words) {
  int rc = submit_locked(e, L, items, n, arena, arena_len, groups, n_groups, bitmap_out, results_out, recovered_out);
  if (rc != IBFT_OK) return rc;
  rc = wait_locked(e, L);
  if (rc != IBFT_OK) return rc;
  if (status_out && n) memcpy(status_out, L->h_status, n);
  if (voted_out && n_groups) {
    CU(cudaSetDevice(e->p.device));
    for (uint32_t g = 0; g < n_groups; g++) {
      const group_dev& gd = L->last_gdev[g];
      uint32_t* dst = voted_out + (size_t)g * voted_stride_words;
      uint32_t w = std::min<uint32_t>(gd.n_words, voted_stride_words);
      // without results_out the recover kernels recorded no votes: the sets are all-zero by definition
      if (w && results_out) CU(cudaMemcpyAsync(dst, L->d_voted + gd.voted_off, (size_t)w * 4, cudaMemcpyDeviceToHost, L->stream));
      else w = 0;
      for (uint32_t i = w; i < voted_stride_words; i++) dst[i] = 0;
    }
    CU(cudaStreamSynchronize(L->stream));
  }
  return IBFT_OK;
}

extern "C" int ibft_verify_batch(ibft_engine* e, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                                 const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out,
                                 ibft_group_result* results_out, uint8_t* recovered_out) {
  if (!e) { set_err("null engine"); return IBFT_ERR_INVALID_ARG; }
  lane* L = acquire_lane(e, n, arena_len);
  std::lock_guard<std::mutex> lk(L->mu, std::adopt_lock);
  return verify_batch_on_lane(e, L, items, n, arena, arena_len, groups, n_groups, bitmap_out, results_out, recovered_out, nullptr, nullptr, 0);
}

extern "C" int ibft_verify_batch_ex(ibft_engine* e, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                                    const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out,
                                    ibft_group_result* results_out, uint8_t* recovered_out, uint8_t* status_out, uint32_t* voted_out,
                                    uint32_t voted_stride_words) {
  if (!e) { set_err("null engine"); return IBFT_ERR_INVALID_ARG; }
  if (voted_out && !results_out) { set_err("voted_out needs results_out (votes are recorded only when quorum results are requested)"); return IBFT_ERR_INVALID_ARG; }
  lane* L = acquire_lane(e, n, arena_len);
  std::lock_guard<std::mutex> lk(L->mu, std::adopt_lock);
  return verify_batch_on_lane(e, L, items, n, arena, arena_len, groups, n_groups, bitmap_out, results_out, recovered_out, status_out, voted_out,
                              voted_stride_words);
}

extern "C" int ibft_last_item_status(ibft_engine* e, uint8_t* status_out, uint32_t n) {
  if (!e || (n && !status_out)) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[e->last_lane.load()];
  std::lock_guard<std::mutex> lk(L->mu);
  if (L->pending.active) { set_err("a submitted call is still pending"); return IBFT_ERR_INVALID_ARG; }
  if (n > L->last_status_n) { set_err("last call had %u items", L->last_status_n); return IBFT_ERR_INVALID_ARG; }
  memcpy(status_out, L->h_status, n);
  return IBFT_OK;
}

// test hook: items the known-key pass of the most recent completed host-buffer call left to the recover pass -- the sum of the
// counts of the worklists that call filled.  Exact for calls of at most two chunks (2^18 items): a third chunk re-uses a list.
extern "C" int ibft_debug_last_deferred(ibft_engine* e, uint32_t* count) {
  if (!e || !count) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[e->last_lane.load()];
  std::lock_guard<std::mutex> lk(L->mu);
  if (L->pending.active) { set_err("a submitted call is still pending"); return IBFT_ERR_INVALID_ARG; }
  *count = 0;
  if (!L->d_worklist) return IBFT_OK;
  CU(cudaSetDevice(e->p.device));
  for (uint32_t k = 0; k < 4; k++) {
    if (!((L->wl_used >> k) & 1u)) continue;
    uint32_t c = 0;
    CU(cudaMemcpy(&c, L->d_worklist + (size_t)k * ((size_t)L->cap_items + 1), 4, cudaMemcpyDeviceToHost));
    *count += c;
  }
  return IBFT_OK;
}

// The asynchronous API lives on lane 0 (one call pending at a time, as before); synchronous calls that fit the small lane keep
// working while it is pending.
extern "C" int ibft_verify_submit(ibft_engine* e, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                                  const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out,
                                  ibft_group_result* results_out, uint8_t* recovered_out) {
  if (!e) { set_err("null engine"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  return submit_locked(e, L, items, n, arena, arena_len, groups, n_groups, bitmap_out, results_out, recovered_out);
}

extern "C" int ibft_verify_poll(ibft_engine* e, int* done) {
  if (!e || !done) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  if (!L->pending.active) { *done = 1; return IBFT_OK; }
  CU(cudaSetDevice(e->p.device));
  cudaError_t ce = cudaEventQuery(L->done_ev);
  if (ce == cudaSuccess) { *done = 1; return IBFT_OK; }
  if (ce == cudaErrorNotReady) { *done = 0; return IBFT_OK; }
  set_err("device execution failed: %s", cudaGetErrorString(ce));
  return IBFT_ERR_CUDA;
}

extern "C" int ibft_verify_wait(ibft_engine* e) {
  if (!e) { set_err("null engine"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  return wait_locked(e, L);
}

extern "C" int ibft_verify_batch_device(ibft_engine* e, const void* d_items, uint32_t n, const void* d_arena, size_t arena_len,
                                        uint32_t shard_lo, uint32_t shard_hi, void* d_bitmap, void* d_recovered, void* stream) {
  if (!e || (n && (!d_items || !d_bitmap))) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (shard_hi > n || shard_lo > shard_hi || (shard_lo & 31) || ((shard_hi & 31) && shard_hi != n)) {
    set_err("shard [%u,%u) of %u must be 32-aligned", shard_lo, shard_hi, n);
    return IBFT_ERR_INVALID_ARG;
  }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  CU(cudaSetDevice(e->p.device));
  cudaStream_t st = stream ? (cudaStream_t)stream : L->stream;
  L->dev_arena = (const uint8_t*)d_arena;  // remembered for ibft_quorum_reduce_device (raw-frame items carry their signer in the arena)
  L->dev_arena_len = arena_len;
  // membership is applied by ibft_quorum_reduce_device / the host mirror in this mode when no groups are bound
  return launch_recover(e, L, (const ibft_sig_item*)d_items, n, (const uint8_t*)d_arena, arena_len, shard_lo, shard_hi,
                        L->last_groups.empty() ? nullptr : L->d_groups, (uint32_t)L->last_groups.size(), (uint32_t*)d_bitmap,
                        (uint8_t*)d_recovered, st);
}

// binds the groups used by the device-resident entry points (copied to the engine's device buffers)
extern "C" int ibft_bind_groups(ibft_engine* e, const ibft_group_desc* groups, uint32_t n_groups) {
  if (!e || (n_groups && !groups)) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (n_groups > e->p.max_groups) { set_err("too many groups"); return IBFT_ERR_CAPACITY; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  CU(cudaSetDevice(e->p.device));
  size_t voted_words = 0;
  if (n_groups) {
    int rc = plan_groups(e, L, groups, n_groups, L->h_gdev, &voted_words);
    if (rc != IBFT_OK) return rc;
    memcpy(L->h_groups, groups, (size_t)n_groups * sizeof(ibft_group_desc));
    CU(cudaMemcpy(L->d_groups, L->h_groups, (size_t)n_groups * sizeof(ibft_group_desc), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(L->d_gdev, L->h_gdev, (size_t)n_groups * sizeof(group_dev), cudaMemcpyHostToDevice));
    L->last_gdev.assign(L->h_gdev, L->h_gdev + n_groups);
    L->last_groups.assign(groups, groups + n_groups);
  } else {
    L->last_gdev.clear();
    L->last_groups.clear();
  }
  return IBFT_OK;
}

extern "C" int ibft_quorum_reduce_device(ibft_engine* e, const void* d_items, uint32_t n, const void* d_bitmap,
                                         const void* d_groups, uint32_t n_groups, void* d_results, void* stream) {
  if (!e || !d_results || (n && (!d_items || !d_bitmap))) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  if (n_groups != L->last_groups.size()) { set_err("call ibft_bind_groups with the same groups first"); return IBFT_ERR_INVALID_ARG; }
  (void)d_groups;  // the bound copy is authoritative (its voted-set layout was planned on the host)
  CU(cudaSetDevice(e->p.device));
  cudaStream_t st = stream ? (cudaStream_t)stream : L->stream;
  size_t voted_words = 0;
  for (auto& g : L->last_gdev) voted_words += g.n_words;
  return launch_quorum(e, L, (const ibft_sig_item*)d_items, n, L->dev_arena, L->dev_arena_len, (const uint32_t*)d_bitmap, L->d_groups,
                       L->d_gdev, n_groups, voted_words, (ibft_group_result*)d_results, st);
}

extern "C" int ibft_quorum_partial_words(ibft_engine* e, uint32_t* words_out) {
  if (!e || !words_out) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  size_t voted_words = 0;
  for (auto& g : L->last_gdev) voted_words += g.n_words;
  *words_out = (uint32_t)(voted_words + L->last_groups.size());
  return IBFT_OK;
}

extern "C" int ibft_quorum_mark_device(ibft_engine* e, const void* d_items, uint32_t n, uint32_t shard_lo, uint32_t shard_hi,
                                       const void* d_bitmap, void* d_partial, void* stream) {
  if (!e || !d_partial || (n && (!d_items || !d_bitmap))) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (shard_hi > n || shard_lo > shard_hi) { set_err("bad shard"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  uint32_t n_groups = (uint32_t)L->last_groups.size();
  if (n_groups == 0) { set_err("call ibft_bind_groups first"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  cudaStream_t st = stream ? (cudaStream_t)stream : L->stream;
  size_t voted_words = 0;
  for (auto& g : L->last_gdev) voted_words += g.n_words;
  uint32_t* part = (uint32_t*)d_partial;
  CU(cudaMemsetAsync(part, 0, (voted_words + n_groups) * 4, st));
  if (shard_hi > shard_lo) {
    k_quorum_mark<<<(shard_hi - shard_lo + 255) / 256, 256, 0, st>>>((const ibft_sig_item*)d_items, n, L->dev_arena, L->dev_arena_len,
                                                                     (const uint32_t*)d_bitmap, L->d_groups, L->d_gdev, n_groups, e->d_slots,
                                                                     e->p.max_table_slots, part, part + voted_words, shard_lo, shard_hi);
    e->launches++;
    CU(cudaGetLastError());
  }
  return IBFT_OK;
}

extern "C" int ibft_quorum_merge_device(ibft_engine* e, const void* d_partials, uint32_t n_parts, uint32_t part_stride_words,
                                        void* d_results, void* stream) {
  if (!e || !d_partials || !d_results || n_parts == 0) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  uint32_t n_groups = (uint32_t)L->last_groups.size();
  if (n_groups == 0) { set_err("call ibft_bind_groups first"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  cudaStream_t st = stream ? (cudaStream_t)stream : L->stream;
  size_t voted_words = 0;
  for (auto& g : L->last_gdev) voted_words += g.n_words;
  if (part_stride_words < voted_words + n_groups) { set_err("partial stride too small"); return IBFT_ERR_INVALID_ARG; }
  uint32_t total = (uint32_t)(voted_words + n_groups);
  k_quorum_merge<<<(total + 255) / 256, 256, 0, st>>>((const uint32_t*)d_partials, n_parts, part_stride_words, (uint32_t)voted_words,
                                                      n_groups, L->d_voted, L->d_nvalid);
  e->launches++;
  CU(cudaGetLastError());
  k_quorum_reduce<<<n_groups, IBFT_REDUCE_THREADS, 0, st>>>(L->d_groups, L->d_gdev, n_groups, e->d_slots, e->p.max_table_slots, L->d_voted, L->d_nvalid,
                                            (ibft_group_result*)d_results);
  e->launches++;
  CU(cudaGetLastError());
  return IBFT_OK;
}

// Exchange buffers of the peer-memory path: allocated by the engine (a plain cudaMalloc block, so that its IPC handle names
// exactly this buffer), exported as a 64-byte CUDA IPC handle, and opened by the peers ON THEIR OWN DEVICE with lazy peer access --
// which is what makes the mapping dereferenceable from the peer's kernels over NVLink.
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
extern "C" int ibft_exchange_alloc(ibft_engine* e, uint32_t words, void** d_buf_out, uint8_t handle_out[64]) {
  if (!e || !d_buf_out || !handle_out || words == 0) { set_err("bad argument"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  void* p = nullptr;
  CU(cudaMalloc(&p, (size_t)words * 4));
  CU(cudaMemset(p, 0, (size_t)words * 4));
  cudaIpcMemHandle_t h;
  cudaError_t ce = cudaIpcGetMemHandle(&h, p);
  if (ce != cudaSuccess) { cudaFree(p); set_err("cudaIpcGetMemHandle: %s", cudaGetErrorString(ce)); return IBFT_ERR_CUDA; }
  memcpy(handle_out, &h, 64);
  *d_buf_out = p;
  return IBFT_OK;
}
extern "C" int ibft_exchange_open(ibft_engine* e, const uint8_t handle[64], void** d_peer_out) {
  if (!e || !handle || !d_peer_out) { set_err("bad argument"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  void* p = nullptr;
  CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *d_peer_out = p;
  return IBFT_OK;
}
extern "C" int ibft_exchange_close(ibft_engine* e, void* d_peer) {
  if (!e || !d_peer) { set_err("bad argument"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  CU(cudaIpcCloseMemHandle(d_peer));
  return IBFT_OK;
}
extern "C" int ibft_exchange_free(ibft_engine* e, void* d_buf) {
  if (!e || !d_buf) { set_err("bad argument"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  CU(cudaDeviceSynchronize());
  CU(cudaFree(d_buf));
  return IBFT_OK;
}
extern "C" int ibft_exchange_clear(ibft_engine* e, void* d_buf, uint32_t word_off, uint32_t words, void* stream) {
  if (!e || !d_buf) { set_err("bad argument"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  CU(cudaMemsetAsync((uint32_t*)d_buf + word_off, 0, (size_t)words * 4, stream ? (cudaStream_t)stream : e->lanes[0].stream));
  return IBFT_OK;
}

extern "C" int ibft_quorum_exchange_device(ibft_engine* e, const uint64_t* peer_bufs_in, uint32_t world, uint32_t rank,
                                           uint32_t words_per_rank, uint32_t bitmap_words_per_rank, uint32_t epoch, void* d_bitmap_full,
                                           void* d_results, void* d_timeout_flag, void* stream) {
  if (!e || !peer_bufs_in || !d_bitmap_full || !d_results || !d_timeout_flag || world == 0 || world > 8 || rank >= world || epoch == 0) {
    set_err("bad argument");
    return IBFT_ERR_INVALID_ARG;
  }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  uint32_t n_groups = (uint32_t)L->last_groups.size();
  if (n_groups == 0) { set_err("call ibft_bind_groups first"); return IBFT_ERR_INVALID_ARG; }
  size_t voted_words = 0;
  for (auto& g : L->last_gdev) voted_words += g.n_words;
  if (words_per_rank < bitmap_words_per_rank + voted_words + n_groups) { set_err("exchange buffer too small"); return IBFT_ERR_INVALID_ARG; }
  CU(cudaSetDevice(e->p.device));
  cudaStream_t st = stream ? (cudaStream_t)stream : L->stream;
  peer_bufs pb{};
  for (uint32_t r = 0; r < world; r++) {
    pb.buf[r] = (uint32_t*)(uintptr_t)peer_bufs_in[r];
  }
  const uint32_t total = world * bitmap_words_per_rank + (uint32_t)voted_words + n_groups;
  const uint32_t blocks = std::max(1u, std::min(64u, (total + 255u) / 256u));
  k_quorum_exchange<<<blocks, 256, 0, st>>>(pb, world, rank, words_per_rank, bitmap_words_per_rank, (uint32_t)voted_words, n_groups, epoch,
                                            /*spin_limit=*/400000u, (uint32_t*)d_bitmap_full, L->d_voted, L->d_nvalid,
                                            (uint32_t*)d_timeout_flag);
  e->launches++;
  CU(cudaGetLastError());
  k_quorum_reduce<<<n_groups, IBFT_REDUCE_THREADS, 0, st>>>(L->d_groups, L->d_gdev, n_groups, e->d_slots, e->p.max_table_slots, L->d_voted, L->d_nvalid,
                                            (ibft_group_result*)d_results);
  e->launches++;
  CU(cudaGetLastError());
  return IBFT_OK;
}

extern "C" int ibft_get_voted_bitmap(ibft_engine* e, uint32_t group, uint32_t* words_out, uint32_t n_words) {
  if (!e || !words_out) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[e->last_lane.load()];
  std::lock_guard<std::mutex> lk(L->mu);
  if (group >= L->last_gdev.size()) { set_err("group %u not part of the last call", group); return IBFT_ERR_INVALID_ARG; }
  const group_dev& g = L->last_gdev[group];
  if (n_words < g.n_words) { set_err("need %u words", g.n_words); return IBFT_ERR_CAPACITY; }
  CU(cudaSetDevice(e->p.device));
  CU(cudaStreamSynchronize(L->stream));
  if (g.n_words) CU(cudaMemcpy(words_out, L->d_voted + g.voted_off, (size_t)g.n_words * 4, cudaMemcpyDeviceToHost));
  for (uint32_t i = g.n_words; i < n_words; i++) words_out[i] = 0;
  return IBFT_OK;
}

// Hash scratch is engine-owned and only ever grows (no cudaMalloc / cudaFree on the per-call path).
static int hash_scratch_reserve(ibft_engine* e, size_t arena_len, uint32_t n) {
  if (arena_len > e->hs_arena_cap) {
    size_t cap = std::max<size_t>(arena_len, std::max<size_t>(e->hs_arena_cap * 2, 1 << 16));
    cudaFree(e->hs_arena); e->hs_arena = nullptr; e->hs_arena_cap = 0;
    cudaFreeHost(e->hs_h_arena); e->hs_h_arena = nullptr;
    CU(cudaMalloc(&e->hs_arena, cap));
    CU(cudaHostAlloc(&e->hs_h_arena, cap, cudaHostAllocDefault));
    e->hs_arena_cap = cap;
  }
  if (n > e->hs_n_cap) {
    uint32_t cap = std::max<uint32_t>(n, std::max<uint32_t>(e->hs_n_cap * 2, 256));
    cudaFree(e->hs_meta); e->hs_meta = nullptr; e->hs_n_cap = 0;
    cudaFreeHost(e->hs_h_meta); e->hs_h_meta = nullptr;
    // per message: offset (4) + length (4) + round (8) in, 32 bytes out
    CU(cudaMalloc(&e->hs_meta, (size_t)cap * 48));
    CU(cudaHostAlloc(&e->hs_h_meta, (size_t)cap * 48, cudaHostAllocDefault));
    e->hs_n_cap = cap;
  }
  return IBFT_OK;
}

static int hash_batch_locked(ibft_engine* e, const uint8_t* arena, size_t arena_len, const uint32_t* offsets, const uint32_t* lens,
                             const uint64_t* rounds, uint32_t n, uint8_t* out32) {
  CU(cudaSetDevice(e->p.device));
  int rc = hash_scratch_reserve(e, arena_len, n);
  if (rc != IBFT_OK) return rc;
  // layout of the meta block (host mirror and device): rounds[n] | offsets[n] | lens[n] | out[n][32]
  uint8_t* hm = e->hs_h_meta;
  uint8_t* dm = e->hs_meta;
  const size_t o_off = (size_t)n * 8, o_len = o_off + (size_t)n * 4, o_out = o_len + (size_t)n * 4;
  if (rounds) memcpy(hm, rounds, (size_t)n * 8);
  memcpy(hm + o_off, offsets, (size_t)n * 4);
  memcpy(hm + o_len, lens, (size_t)n * 4);
  cudaStream_t st = e->hash_stream;
  if (arena_len) {
    memcpy(e->hs_h_arena, arena, arena_len);
    CU(cudaMemcpyAsync(e->hs_arena, e->hs_h_arena, arena_len, cudaMemcpyHostToDevice, st));
  }
  CU(cudaMemcpyAsync(dm, hm, o_out, cudaMemcpyHostToDevice, st));
  k_keccak_batch<<<(n + 63) / 64, 64, 0, st>>>(e->hs_arena, arena_len, (const uint32_t*)(dm + o_off), (const uint32_t*)(dm + o_len),
                                               rounds ? (const uint64_t*)dm : nullptr, n, dm + o_out);
  e->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(hm + o_out, dm + o_out, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  memcpy(out32, hm + o_out, (size_t)n * 32);
  return IBFT_OK;
}

extern "C" int ibft_keccak256_batch(ibft_engine* e, const uint8_t* arena, size_t arena_len, const uint32_t* offsets,
                                    const uint32_t* lens, uint32_t n, uint8_t* out32) {
  if (!e || (n && (!offsets || !lens || !out32)) || (arena_len && !arena)) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (n == 0) return IBFT_OK;
  std::lock_guard<std::mutex> lk(e->hash_mu);
  return hash_batch_locked(e, arena, arena_len, offsets, lens, nullptr, n, out32);
}

extern "C" int ibft_proposal_hash_batch(ibft_engine* e, const uint8_t* arena, size_t arena_len, const uint32_t* offsets,
                                        const uint32_t* lens, const uint64_t* rounds, uint32_t n, uint8_t* out32) {
  if (!e || (n && (!offsets || !lens || !rounds || !out32)) || (arena_len && !arena)) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (n == 0) return IBFT_OK;
  std::lock_guard<std::mutex> lk(e->hash_mu);
  return hash_batch_locked(e, arena, arena_len, offsets, lens, rounds, n, out32);
}

extern "C" int ibft_sign_batch(ibft_engine* e, const uint8_t* privkeys, const uint8_t* digests, const uint8_t* nonces, uint32_t n,
                               uint8_t* sigs65_out) {
  if (!e || (n && (!privkeys || !digests || !sigs65_out))) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  if (n == 0) return IBFT_OK;
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  CU(cudaSetDevice(e->p.device));
  uint8_t *d_d = nullptr, *d_z = nullptr, *d_k = nullptr, *d_s = nullptr;
  int rc = IBFT_OK;
  cudaError_t ce;
#define CUK(call) if ((ce = (call)) != cudaSuccess) { set_err("%s failed: %s", #call, cudaGetErrorString(ce)); rc = IBFT_ERR_CUDA; goto done; }
  CUK(cudaMalloc(&d_d, (size_t)n * 32));
  CUK(cudaMalloc(&d_z, (size_t)n * 32));
  CUK(cudaMalloc(&d_s, (size_t)n * 65));
  CUK(cudaMemcpyAsync(d_d, privkeys, (size_t)n * 32, cudaMemcpyHostToDevice, L->stream));
  CUK(cudaMemcpyAsync(d_z, digests, (size_t)n * 32, cudaMemcpyHostToDevice, L->stream));
  if (nonces) {
    CUK(cudaMalloc(&d_k, (size_t)n * 32));
    CUK(cudaMemcpyAsync(d_k, nonces, (size_t)n * 32, cudaMemcpyHostToDevice, L->stream));
  }
  k_sign<<<(n + 63) / 64, 64, 0, L->stream>>>(d_d, d_z, d_k, n, d_s);
  e->launches++;
  CUK(cudaGetLastError());
  CUK(cudaMemcpyAsync(sigs65_out, d_s, (size_t)n * 65, cudaMemcpyDeviceToHost, L->stream));
  CUK(cudaStreamSynchronize(L->stream));
  // private keys do not stay on the device
  cudaMemsetAsync(d_d, 0, (size_t)n * 32, L->stream);
  if (d_k) cudaMemsetAsync(d_k, 0, (size_t)n * 32, L->stream);
  cudaStreamSynchronize(L->stream);
done:
#undef CUK
  cudaFree(d_d); cudaFree(d_z); cudaFree(d_k); cudaFree(d_s);
  return rc;
}

extern "C" int ibft_set_recover_path(ibft_engine* e, int path) {
  if (e == nullptr || path < IBFT_PATH_AUTO || path > IBFT_PATH_QSPLIT) { set_err("bad recover path"); return IBFT_ERR_INVALID_ARG; }
  e->recover_path.store(path);
  return IBFT_OK;
}

extern "C" uint64_t ibft_engine_launch_count(ibft_engine* e) { return e ? e->launches.load() : 0; }

extern "C" int ibft_probe_int_peak(ibft_engine* e, double* imad_per_s, double* wide_mac_per_s) {
  if (!e || !imad_per_s || !wide_mac_per_s) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  CU(cudaSetDevice(e->p.device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, e->p.device));
  int blocks = prop.multiProcessorCount * 8, threads = 256;
  uint32_t* d_out = nullptr;
  CU(cudaMalloc(&d_out, (size_t)blocks * threads * 4));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  double best[2] = {0, 0};
  for (int which = 0; which < 2; which++) {
    for (int rep = 0; rep < 4; rep++) {
      CU(cudaEventRecord(e0, L->stream));
      if (which == 0) k_probe_imad<<<blocks, threads, 0, L->stream>>>(d_out, 3, 5);
      else k_probe_wide<<<blocks, threads, 0, L->stream>>>(d_out, 3, 5);
      CU(cudaEventRecord(e1, L->stream));
      CU(cudaEventSynchronize(e1));
      float ms = 0;
      CU(cudaEventElapsedTime(&ms, e0, e1));
      double instr = (double)PROBE_ITERS * PROBE_UNROLL * (which == 0 ? 8 : 4) * (double)blocks * threads;
      double rate = instr / (ms * 1e-3);
      if (rep > 0 && rate > best[which]) best[which] = rate;
    }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d_out);
  *imad_per_s = best[0];
  *wide_mac_per_s = best[1];
  return IBFT_OK;
}

extern "C" int ibft_debug_op(ibft_engine* e, int op, const uint8_t* a, const uint8_t* b, const uint8_t* c, uint32_t n,
                             uint8_t* out, uint32_t out_stride) {
  if (!e || !a || !out || n == 0) { set_err("null argument"); return IBFT_ERR_INVALID_ARG; }
  lane* L = &e->lanes[0];
  std::lock_guard<std::mutex> lk(L->mu);
  CU(cudaSetDevice(e->p.device));
  uint8_t *d_a = nullptr, *d_b = nullptr, *d_c = nullptr, *d_o = nullptr;
  int rc = IBFT_OK;
  cudaError_t ce;
#define CUK(call) if ((ce = (call)) != cudaSuccess) { set_err("%s failed: %s", #call, cudaGetErrorString(ce)); rc = IBFT_ERR_CUDA; goto done; }
  CUK(cudaMalloc(&d_a, (size_t)n * 32));
  CUK(cudaMemcpy(d_a, a, (size_t)n * 32, cudaMemcpyHostToDevice));
  if (b) { CUK(cudaMalloc(&d_b, (size_t)n * 32)); CUK(cudaMemcpy(d_b, b, (size_t)n * 32, cudaMemcpyHostToDevice)); }
  if (c) { CUK(cudaMalloc(&d_c, (size_t)n * 64)); CUK(cudaMemcpy(d_c, c, (size_t)n * 64, cudaMemcpyHostToDevice)); }
  CUK(cudaMalloc(&d_o, (size_t)n * out_stride));
  CUK(cudaMemset(d_o, 0, (size_t)n * out_stride));
  k_debug_op<<<(n + 63) / 64, 64, 0, L->stream>>>(op, d_a, d_b, d_c, n, d_o, out_stride);
  e->launches++;
  CUK(cudaGetLastError());
  CUK(cudaStreamSynchronize(L->stream));
  CUK(cudaMemcpy(out, d_o, (size_t)n * out_stride, cudaMemcpyDeviceToHost));
done:
#undef CUK
  cudaFree(d_a); cudaFree(d_b); cudaFree(d_c); cudaFree(d_o);
  return rc;
}
