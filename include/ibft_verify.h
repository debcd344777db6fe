/*
 * ibft_verify.h -- C ABI of the B200-native batched message-verification engine for go-ibft.
 *
 * This is the drop-in boundary.  go-ibft has NO FFI of its own: the hot path sits behind the Go
 * interfaces core.Verifier (core/backend.go:37-56) and core.Messages (core/ibft.go:23-46), whose
 * production implementation lives in the embedding node.  The entry points below are what a
 * cgo-backed `gpuBackend` (see INTEGRATION.md) binds; each one cites the reference interface it
 * serves.  Plain C types only (no CUDA / torch types): pointers + sizes, little-endian host,
 * 32-byte scalars big-endian as on the wire.  Every function returns an int status
 * (IBFT_OK == 0) and never aborts; a failed launch yields "no verdict" (status != 0, outputs
 * untouched) -- never a `true` verdict (SURVEY.md §5, §8b error convention).
 *
 * There is NO CPU fallback: if no CUDA device is usable ibft_engine_create fails with
 * IBFT_ERR_NO_DEVICE and nothing else can be called.
 */
#ifndef IBFT_VERIFY_H
#define IBFT_VERIFY_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IBFT_ABI_VERSION 2

/* status codes */
#define IBFT_OK 0
#define IBFT_ERR_INVALID_ARG 1
#define IBFT_ERR_NO_DEVICE 2   /* no usable CUDA device / driver: engine cannot exist (no CPU fallback) */
#define IBFT_ERR_CUDA 3        /* a CUDA call or kernel launch failed; see ibft_last_error() */
#define IBFT_ERR_CAPACITY 4    /* batch exceeds the capacity given at ibft_engine_create */
#define IBFT_ERR_VOTING_POWER 5 /* total voting power is zero: core/validator_manager.go:66-68 errVotingPowerNotCorrect */
#define IBFT_ERR_NO_TABLE 6    /* a group references a validator-table slot that was never set, or that holds ANOTHER height's table */

/* ibft_sig_item.kind */
#define IBFT_KIND_DIGEST 0   /* `digest` is the 32-byte message digest z itself */
#define IBFT_KIND_PAYLOAD 1  /* z = Keccak-256(arena[payload_off .. +payload_len]) -- IsValidValidator: the bytes are
                                IbftMessage.PayloadNoSig() (messages/proto/helper.go:13-27) */
#define IBFT_KIND_SEAL 2     /* `digest` holds proposalHash; z = Keccak-256(proposalHash || 0x02) -- IsValidCommittedSeal
                                (0x02 = MessageType_COMMIT, messages/proto/messages.proto:10) */
#define IBFT_KIND_WIRE 3      /* arena slice = the COMPLETE wire encoding of a PREPARE / COMMIT IbftMessage (a raw gossip frame).  The device
                                finds From, Signature and the signed bytes itself: for a canonically encoded frame PayloadNoSig
                                (messages/proto/helper.go:13-27) is the frame minus its field-3 TLV.  r/s/v/signer/digest of the tuple are
                                ignored.  Frames that are not canonical, or carry a nested payload (PREPREPARE / ROUND_CHANGE), get verdict 0
                                and item status IBFT_ITEM_NEEDS_HOST: the host re-submits those as IBFT_KIND_PAYLOAD. */
#define IBFT_KIND_WIRE_SEAL 4 /* same frame; checks the committed seal instead: commitData.committedSeal over
                                Keccak-256(commitData.proposalHash || 0x02), signer = From (IsValidCommittedSeal on the frame) */
#define IBFT_KIND_PAYLOAD2 5  /* z = Keccak-256(arena[payload_off .. +payload_len] || arena[off2 .. +len2]) with off2 = u64 little-endian in
                                digest[0..8) and len2 = u32 little-endian in digest[8..12): PayloadNoSig given as TWO spans.  A
                                ROUND_CHANGE message's signed bytes end with its whole prepared certificate (909 KB at 10k validators,
                                messages/proto/messages.proto:95-103); the 10,000 ROUND_CHANGE messages of a round mostly embed the SAME
                                certificate, so the caller uploads each distinct certificate once and every message's tuple names
                                (its own head, the shared tail).  Same verdict as IBFT_KIND_PAYLOAD over the concatenation. */
#define IBFT_KIND_INVALID 255 /* structurally invalid on the host side (nil seal, signature length != 65, ...):
                                 verdict is always 0.  Mirrors "malformed input => false" (messages/helpers.go:38-42). */

/* per-item status of the last host-buffer verify call (ibft_last_item_status) */
#define IBFT_ITEM_OK 0          /* the verdict bit is the answer */
#define IBFT_ITEM_NEEDS_HOST 1  /* IBFT_KIND_WIRE*: frame not canonical / not a flat PREPARE or COMMIT; verdict bit is 0, re-submit as KIND_PAYLOAD */

#define IBFT_NO_TABLE 0xFFFFu /* ibft_group_desc.table_slot: skip the validator-set membership test */

/* One signature check = one packed 128-byte tuple: (r, s, v, hash) + the expected signer.
 * Serves both IsValidValidator(msg) (core/backend.go:41-45: signer of msg.Signature over the payload
 * == msg.From and From is a validator at msg.View.Height) and IsValidCommittedSeal(hash, seal)
 * (core/backend.go:53-55; seal = {Signer, Signature}, messages/helpers.go:16-19). */
typedef struct ibft_sig_item {
  uint8_t r[32];        /* signature R, big-endian                                              */
  uint8_t s[32];        /* signature S, big-endian                                              */
  uint8_t digest[32];   /* KIND_DIGEST: z; KIND_SEAL: proposalHash; KIND_PAYLOAD: ignored        */
  uint8_t signer[20];   /* expected signer address: msg.From / seal.Signer                       */
  uint8_t v;            /* recovery id, must be 0 or 1                                           */
  uint8_t kind;         /* IBFT_KIND_*                                                           */
  uint16_t group;       /* index into the groups array of the call                               */
  uint32_t payload_off; /* KIND_PAYLOAD: byte offset into the payload arena                      */
  uint32_t payload_len; /* KIND_PAYLOAD: byte length                                             */
} ibft_sig_item;        /* sizeof == 128 */

/* A group is one quorum domain: all items of one (height, round, message type).  Its validator
 * table supplies set membership and voting power (core/validator_manager.go:77-96 HasQuorum).
 * `height` is the height the group's messages carry (msg.View.Height): IsValidValidator must answer for "one of the validators
 * at the height in message" (core/backend.go:41-45), so a call whose group names a slot that currently holds ANOTHER height's
 * table (e.g. a caller mapping height % slots after the slot was recycled) fails with IBFT_ERR_NO_TABLE -- it is never
 * answered from the wrong validator set. */
typedef struct ibft_group_desc {
  uint16_t table_slot; /* slot given to ibft_set_validators, or IBFT_NO_TABLE */
  uint16_t flags;      /* reserved, 0 */
  uint32_t reserved;   /* 0 */
  uint64_t height;     /* height of the group's messages; must equal the height the slot was set with (ignored for IBFT_NO_TABLE) */
} ibft_group_desc;     /* sizeof == 16 */

/* Per-group result of the on-device quorum reduction.
 * power[] is the little-endian 320-bit sum of votingPower over the DISTINCT validators with >= 1 valid
 * item in the group (HasQuorum sums over an address *set*: validator_manager.go:88-92, :147-155).
 * has_quorum = power >= floor(2*total/3)+1 (validator_manager.go:95, :130-135). */
typedef struct ibft_group_result {
  uint64_t power[5];
  uint32_t n_valid;     /* items of the group with verdict 1 */
  uint32_t n_distinct;  /* distinct validators among them */
  uint32_t has_quorum;  /* 0/1; 0 when the group has no table */
  uint32_t reserved;
} ibft_group_result;

typedef struct ibft_engine_params {
  int32_t device;             /* CUDA device ordinal */
  uint32_t max_items;         /* capacity of one verify call (staging is allocated once, pinned) */
  uint32_t max_payload_bytes; /* capacity of the payload arena of one call */
  uint32_t max_groups;        /* capacity of the groups array of one call */
  uint32_t max_table_slots;   /* number of validator-table slots (heights kept resident) */
  uint32_t max_validators;    /* capacity of one validator table */
  uint32_t flags;             /* IBFT_FLAG_* */
} ibft_engine_params;

/* Engine flag: keep a registry of the validators' public keys.  A key is learned from the first successful recovery of a
 * signature by that validator; once its comb table is built (m * 2^(8j) * Q for 17 positions j and m = 1..128), later signatures
 * by the same validator are VERIFIED against the key -- 51 mixed additions, no doubling, no square root, no per-signature table,
 * no address hash -- instead of recovered.  A signature the verification rejects is re-checked by the recover path, so every
 * verdict is the recover path's verdict.  Costs 136 KiB of device memory per validator and table slot (1.39 GB for a
 * 10,000-validator set; ibft_set_validators fails with IBFT_ERR_CAPACITY when the device cannot hold it, and the slot keeps its
 * previous table).  A key belongs to an address, not to a height: ibft_set_validators carries the finished tables over, by
 * address, from the slot's previous content -- or, when the slot was empty, from the resident table of the greatest height --
 * so a chain that moves to the next height with (mostly) the same validators never recovers their signatures again. */
#define IBFT_FLAG_KEY_CACHE 1u

typedef struct ibft_device_info {
  char name[64];
  int32_t sm_count;
  int32_t cc_major, cc_minor;
  int32_t clock_khz;
  uint64_t total_mem;
  int32_t abi_version;
  int32_t kernel_regs;       /* registers/thread of the recover kernel */
  int32_t kernel_smem_bytes; /* static+dynamic shared memory/CTA of the recover kernel */
  int32_t block_threads;     /* CTA size of the recover kernel */
} ibft_device_info;

typedef struct ibft_engine ibft_engine;

/* lifecycle ------------------------------------------------------------------------------------------ */
int ibft_abi_version(void);
/* Thread-local description of the last failure on the calling thread (never NULL). */
const char* ibft_last_error(void);
int ibft_engine_create(const ibft_engine_params* params, ibft_engine** out);
void ibft_engine_destroy(ibft_engine* e);
int ibft_engine_device_info(ibft_engine* e, ibft_device_info* out);

/* validator tables --------------------------------------------------------------------------------- */
/* Replaces ValidatorManager.Init -> Backend.GetVotingPowers(height) (core/validator_manager.go:50-74,
 * core/backend.go via ValidatorBackend :17-20).  addrs: n x 20 bytes in validator-index order;
 * powers_be: n x 32 bytes big-endian (NULL => unit power).  Computes and stores the quorum threshold
 * floor(2*total/3)+1.  Returns IBFT_ERR_VOTING_POWER when the total is zero. */
int ibft_set_validators(ibft_engine* e, uint32_t table_slot, uint64_t height, const uint8_t* addrs,
                        const uint8_t* powers_be, uint32_t n);
/* Little-endian 320-bit quorum threshold of a slot (for the host-side quorum mirror). */
int ibft_get_quorum(ibft_engine* e, uint32_t table_slot, uint64_t quorum_out[5], uint64_t* height_out,
                    uint32_t* n_out);

/* verification ------------------------------------------------------------------------------------- */
/* Synchronous batched verify with HOST buffers (the call the cgo Backend / the batching store makes from
 * GetValidMessages / GetExtendedRCC flushes: messages/messages.go:169-199, :202-245).
 *   items[n], arena[arena_len] (may be NULL/0), groups[n_groups]
 *   bitmap_out: caller-allocated, (n+31)/32 words; bit (i%32) of word i/32 = verdict of item i
 *   results_out: caller-allocated, n_groups entries, or NULL
 *   recovered_out: NULL, or n x 20 bytes receiving the recovered signer address (zero when recovery failed)
 * The copy host->pinned staging->device, the kernels, and the copies back all happen inside the call. */
int ibft_verify_batch(ibft_engine* e, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                      const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out,
                      ibft_group_result* results_out, uint8_t* recovered_out);

/* The same call with everything a CONCURRENT caller needs returned by the call itself (the two getters below describe "the
 * most recent completed call of the engine", which is only meaningful to a single-threaded caller -- and a goroutine may
 * change OS threads between two cgo calls):
 *   status_out  NULL, or n bytes receiving the per-item status (IBFT_ITEM_*)
 *   voted_out   NULL, or n_groups x voted_stride_words words: row g = the voted set of group g (bit i = validator i of the
 *               group's table has >= 1 valid item), zero-padded -- the bitmap core/validator_manager.go's quorum check reads
 *               (HasQuorumVoted in INTEGRATION.md).  Requires results_out.
 * Concurrency: the engine runs up to two host-buffer calls at a time (a full-capacity lane and a small lane of
 * min(max_items, 16,384) items / 4 MiB of payload); further callers block.  ibft_set_validators waits for both. */
int ibft_verify_batch_ex(ibft_engine* e, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                         const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out,
                         ibft_group_result* results_out, uint8_t* recovered_out, uint8_t* status_out, uint32_t* voted_out,
                         uint32_t voted_stride_words);

/* Per-item status (IBFT_ITEM_*) of the most recent completed ibft_verify_batch / ibft_verify_wait on this engine. */
int ibft_last_item_status(ibft_engine* e, uint8_t* status_out, uint32_t n);

/* Asynchronous variant: same arguments; inputs are copied into engine-owned pinned staging before the call
 * returns (cgo rule: no Go pointer is retained).  ibft_verify_poll returns IBFT_OK with *done = 0/1;
 * ibft_verify_wait blocks and copies the outputs into the buffers given at submit time. */
int ibft_verify_submit(ibft_engine* e, const ibft_sig_item* items, uint32_t n, const uint8_t* arena, size_t arena_len,
                       const ibft_group_desc* groups, uint32_t n_groups, uint32_t* bitmap_out,
                       ibft_group_result* results_out, uint8_t* recovered_out);
int ibft_verify_poll(ibft_engine* e, int* done);
int ibft_verify_wait(ibft_engine* e);

/* Binds the groups (and plans their voted-set layout) used by the two device-resident entry points below. */
int ibft_bind_groups(ibft_engine* e, const ibft_group_desc* groups, uint32_t n_groups);

/* Device-resident variant: every pointer is a DEVICE pointer on the engine's device and `stream` is a
 * cudaStream_t passed as void* (NULL = engine stream).  Enqueues only; the caller synchronises the stream.
 * Sharding: only items [shard_lo, shard_hi) are verified and only their bitmap words are written (both must
 * be multiples of 32 or equal to n) -- the multi-GPU path all-gathers the bitmap words afterwards. */
int ibft_verify_batch_device(ibft_engine* e, const void* d_items, uint32_t n, const void* d_arena, size_t arena_len,
                             uint32_t shard_lo, uint32_t shard_hi, void* d_bitmap, void* d_recovered, void* stream);

/* Device-resident quorum reduction over a complete (all-gathered) bitmap: resolves each item's signer to its
 * validator index, ORs the per-group voted sets and reduces voting power against the threshold.
 * d_groups: ibft_group_desc[n_groups]; d_results: ibft_group_result[n_groups] (device). */
int ibft_quorum_reduce_device(ibft_engine* e, const void* d_items, uint32_t n, const void* d_bitmap,
                              const void* d_groups, uint32_t n_groups, void* d_results, void* stream);

/* Multi-GPU form of the reduction (each rank resolves only ITS shard, so no work is repeated across ranks):
 *   ibft_quorum_partial_words  -> W = words of one rank's partial result (voted sets of all bound groups, then one valid
 *                                 count per group); depends only on the bound groups, identical on every rank
 *   ibft_quorum_mark_device    -> marks items [shard_lo, shard_hi) with a set bitmap bit into d_partial (W words, device)
 *   (all-gather the partials -- they can ride in the same collective as the bitmap words)
 *   ibft_quorum_merge_device   -> ORs / sums n_parts partials (part_stride_words apart) and reduces against the thresholds */
int ibft_quorum_partial_words(ibft_engine* e, uint32_t* words_out);
int ibft_quorum_mark_device(ibft_engine* e, const void* d_items, uint32_t n, uint32_t shard_lo, uint32_t shard_hi,
                            const void* d_bitmap, void* d_partial, void* stream);
int ibft_quorum_merge_device(ibft_engine* e, const void* d_partials, uint32_t n_parts, uint32_t part_stride_words,
                             void* d_results, void* stream);

/* The same exchange WITHOUT a library collective (one node, <= 8 ranks): every rank keeps its (bitmap words | partial) in an
 * exchange buffer that its peers have mapped over NVLink (CUDA IPC / peer access; the caller exchanges the handles once).
 *   buffer layout, uint32 words: [2 parities][words_per_rank], then flags[2]; words_per_rank >= bitmap_words_per_rank + W
 *   (W = ibft_quorum_partial_words).  For round `epoch` (1, 2, 3, ...) a rank verifies its shard with the bitmap pointer rebased
 *   into parity (epoch & 1) of ITS buffer and marks its votes behind the bitmap words of that parity (ibft_quorum_mark_device),
 *   then calls this: ONE kernel publishes the rank's flag, waits (bounded) for the peers' flags, reads their words out of peer
 *   memory -- OR-ing voted sets, summing counts, assembling the complete bitmap in d_bitmap_full (world x bitmap_words_per_rank
 *   words) -- and the weighted reduce follows.  peer_bufs[r] = device address of rank r's buffer as mapped in THIS process.
 *   *d_timeout_flag (device uint32, zeroed by the caller) becomes 1 when a peer did not publish in time: results are then
 *   meaningless and the device is NOT left spinning. */
/* Exchange buffers.  The engine allocates one (zeroed, `words` uint32 words = 2 * words_per_rank + 2 flags, rounded up) and
 * exports its 64-byte CUDA IPC handle; the caller passes the handle to the other ranks (any side channel), and every rank opens
 * its peers' handles ON ITS OWN DEVICE with lazy peer access -- the resulting address goes into peer_bufs[].  A rank's own entry
 * is the address ibft_exchange_alloc returned.  ibft_exchange_clear zeroes a word range on a stream (the parity region, before
 * the shard is verified into it). */
int ibft_exchange_alloc(ibft_engine* e, uint32_t words, void** d_buf_out, uint8_t handle_out[64]);
int ibft_exchange_open(ibft_engine* e, const uint8_t handle[64], void** d_peer_out);
int ibft_exchange_close(ibft_engine* e, void* d_peer);
int ibft_exchange_free(ibft_engine* e, void* d_buf);
int ibft_exchange_clear(ibft_engine* e, void* d_buf, uint32_t word_off, uint32_t words, void* stream);
int ibft_quorum_exchange_device(ibft_engine* e, const uint64_t* peer_bufs, uint32_t world, uint32_t rank, uint32_t words_per_rank,
                                uint32_t bitmap_words_per_rank, uint32_t epoch, void* d_bitmap_full, void* d_results,
                                void* d_timeout_flag, void* stream);

/* Per-group voted set of the most recent reduce: bit i = validator i of the group's table has >= 1 valid item.
 * words_out: caller-allocated, (table_n+31)/32 words.  This is the bitmap core/validator_manager.go's quorum
 * check reads in the Go shim (INTEGRATION.md). */
int ibft_get_voted_bitmap(ibft_engine* e, uint32_t group, uint32_t* words_out, uint32_t n_words);

/* hashing ------------------------------------------------------------------------------------------ */
/* Batched Keccak-256 for IsValidProposalHash (core/backend.go:50-51; callers core/ibft.go:545,649,781,858,938):
 * message i = arena[offsets[i] .. offsets[i]+lens[i]); out32: n x 32 bytes.  HOST buffers. */
int ibft_keccak256_batch(ibft_engine* e, const uint8_t* arena, size_t arena_len, const uint32_t* offsets,
                         const uint32_t* lens, uint32_t n, uint8_t* out32);

/* The proposal hash of this engine's synthetic convention (SURVEY.md §8c; real embedders hash an RLP header), both sponges in
 * ONE launch: out32[i] = Keccak-256(Keccak-256(rawProposal_i) || u64_be(rounds[i])).  IsValidProposalHash(proposal, hash)
 * (core/backend.go:50-51; "hash matches keccak(proposal)", core/ibft.go:648-649, :781-787) compares this with the claimed hash.
 * Same argument layout as ibft_keccak256_batch.  Hash calls have their own lock, stream and grow-only scratch: they neither
 * wait for verify calls nor allocate device memory per call.  HOST buffers. */
int ibft_proposal_hash_batch(ibft_engine* e, const uint8_t* arena, size_t arena_len, const uint32_t* offsets,
                             const uint32_t* lens, const uint64_t* rounds, uint32_t n, uint8_t* out32);

/* signing (the MessageConstructor side) --------------------------------------------------------------- */
/* Batched ECDSA signing for MessageConstructor (core/backend.go:12-34: every Build*Message must be signed by the validator,
 * BuildCommitMessage must create the committed seal).  privkeys, digests: n x 32 bytes big-endian; nonces: n x 32 bytes or
 * NULL (then k = Keccak-256(d || z || ctr) mod-checked, deterministic per (key, digest)); sigs65_out: n x 65 bytes R||S||V,
 * s in the low half.  An unusable nonce yields an all-zero signature.  HOST buffers. */
int ibft_sign_batch(ibft_engine* e, const uint8_t* privkeys, const uint8_t* digests, const uint8_t* nonces, uint32_t n,
                    uint8_t* sigs65_out);

/* measurement / test hooks ------------------------------------------------------------------------- */
/* Kernel selection of the recover step (the verdicts are identical on every path; only latency / throughput differ):
 *   AUTO    by batch size: up to SMs x 48 signatures (7,104 on a B200) QSPLIT, up to SMs x 192 (28,416) SPLIT, beyond
 *           that THREAD (the throughput kernel);
 *   THREAD  always one thread per signature;  QUAD  always four lanes per signature;
 *   SPLIT   chain warps (one lane per signature) + a helper warp per CTA that takes the digest, r^-1, sqrt and u1*G off the
 *           chain (mid-size batches: up to SMs x 96 signatures in one wave, e.g. a 10k-validator COMMIT round);
 *   QSPLIT  both: four-lane chain warps + a helper warp (small rounds: up to SMs x 24 signatures in one wave).
 * (The north star asks for one warp per signature; DESIGN.md §3.1 measures why the throughput path uses one thread per
 * signature and the latency paths four lanes / a chain+helper warp pair instead.)  Returns IBFT_ERR_INVALID_ARG for an unknown path. */
#define IBFT_PATH_AUTO 0
#define IBFT_PATH_THREAD 1
#define IBFT_PATH_QUAD 2
#define IBFT_PATH_SPLIT 3
#define IBFT_PATH_QSPLIT 4
int ibft_set_recover_path(ibft_engine* e, int path);

/* Key registry (IBFT_FLAG_KEY_CACHE): build the tables of the keys learned since the last call; *n_keys_out = keys known
 * over all resident tables.  ibft_verify_batch / ibft_verify_wait do this on their way out; users of the device-resident
 * entry points call it between rounds.  No-op (0 keys) when the flag is off. */
int ibft_refresh_key_tables(ibft_engine* e, uint32_t* n_keys_out);

/* Number of kernel launches issued by this engine since creation (bench.py reports gpu_launches from it). */
uint64_t ibft_engine_launch_count(ibft_engine* e);
/* Dependent-free IMAD issue-rate probe on the engine's device (the integer-roofline denominator of bench.py):
 * returns thread-level mad.lo.u32 instructions per second in *imad_per_s and chained 32x32+64 wide MACs per
 * second (IMAD.WIDE.X carry chains, the instruction the field multiplier is made of) in *wide_mac_per_s. */
int ibft_probe_int_peak(ibft_engine* e, double* imad_per_s, double* wide_mac_per_s);
/* Primitive-level parity hooks (tests only): run one device primitive over n independent operand sets.
 * op: see IBFT_DBG_* ; a, b: n x 32-byte big-endian operands (b may be NULL); out: n x 32 (or n x 64 for points). */
#define IBFT_DBG_FE_MUL 1   /* out = a*b mod p */
#define IBFT_DBG_FE_SQR 2   /* out = a^2 mod p */
#define IBFT_DBG_FE_INV 3   /* out = a^-1 mod p (0 -> 0) */
#define IBFT_DBG_FE_SQRT 4  /* out = sqrt(a) candidate a^((p+1)/4) */
#define IBFT_DBG_SC_MUL 5   /* out = a*b mod n */
#define IBFT_DBG_SC_INV 6   /* out = a^-1 mod n (0 -> 0) */
#define IBFT_DBG_ECMULT 7   /* out(64) = a*G + b*P with P = lift_x(Gx-derived test point); see tests */
#define IBFT_DBG_FE_ADD 8   /* out = a+b mod p */
#define IBFT_DBG_FE_SUB 9   /* out = a-b mod p */
#define IBFT_DBG_GLV 10     /* out(64) = |k1| (16B BE) || |k2| (16B BE) || sign1 || sign2 padded -- see tests */
/* Combined generator table (builds with IBFT_WC > 0): *wc = window (0 when absent), *entries = entries of ONE comb position;
 * copies `count` 64-byte entries (x, y as 8 little-endian words each) starting at `first`.  The comb positions j = 0, 1, ...
 * (17 for wc = 8) follow one another: entry index = j * entries + d1 * (2^wc + 1) + d2 + 2^(wc-1) holds
 * 2^(wc j) * (d1*G + d2*lambda*G); first + count may run up to the end of the last position. */
int ibft_debug_ctable(ibft_engine* e, uint32_t first, uint32_t count, uint8_t* out, int* wc, uint32_t* entries);
/* Key registry (IBFT_FLAG_KEY_CACHE, tests only): copies `count` 64-byte entries (same format) of the comb table of validator
 * `validator` (validator-index order) of table slot `slot`, starting at `first`: entry index = j * 128 + m - 1 holds
 * m * 2^(8 j) * Q for comb position j and m = 1..128.  *state_out (may be NULL): 0 key unknown, 1 learned, 3 table being
 * built, 2 table READY (only a READY table is ever read by the verification). */
int ibft_debug_keytab(ibft_engine* e, uint32_t slot, uint32_t validator, uint32_t first, uint32_t count, uint8_t* out,
                      uint32_t* state_out);
/* Key registry (tests only): *count = number of items that the known-key pass of the most recent completed host-buffer call
 * left to the recover pass (key not ready, or the verification against the key rejected).  0 when that call took no
 * known-key pass.  Exact for calls of at most 2^18 items (two upload chunks; a third chunk re-uses a worklist). */
int ibft_debug_last_deferred(ibft_engine* e, uint32_t* count);
int ibft_debug_op(ibft_engine* e, int op, const uint8_t* a, const uint8_t* b, const uint8_t* c, uint32_t n,
                  uint8_t* out, uint32_t out_stride);

#ifdef __cplusplus
}
#endif
#endif /* IBFT_VERIFY_H */
