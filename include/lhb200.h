/*
 * lhb200.h — C ABI of liblhb200.so: the B200-native (sm_100a) replacement for Lighthouse's two
 * compute-bound hot paths.  Plain pointers and sizes only; no exceptions or panics cross this boundary.
 *
 * Citations are file:line under sigp/lighthouse v5.3.0 (/root/reference).  The Rust-side bindings a
 * Lighthouse maintainer would add are shown in INTEGRATION.md.
 *
 * Conventions
 *   - Every entry point returns an int32 status: LHB200_OK (0) or a negative LHB200_E* code;
 *     lhb200_last_error() gives a thread-local human-readable message.  Results go to out-params.
 *   - "Host" entry points take caller-owned host buffers that are only read during the call (they mirror
 *     the borrowed Cow<'a, ..> data of bls::SignatureSet / &self of TreeHash); nothing is retained.
 *   - "dev_" entry points take device pointers (inputs already resident in HBM) and an optional
 *     cudaStream_t passed as void* (NULL = the library's stream); they return after enqueueing unless
 *     documented otherwise.
 *   - There is NO CPU fallback: without a usable sm_100 device every compute entry point returns
 *     LHB200_ENODEV.
 */
#ifndef LHB200_H
#define LHB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LHB200_API __attribute__((visibility("default")))
#else
#define LHB200_API
#endif

#define LHB200_OK 0
#define LHB200_ENODEV (-1)   /* no CUDA device / init not called / init failed */
#define LHB200_EINVAL (-2)   /* bad argument (null pointer, inconsistent sizes, malformed SSZ offsets) */
#define LHB200_ECUDA (-3)    /* CUDA runtime error (message in lhb200_last_error) */
#define LHB200_ENOMEM (-4)   /* device or pinned allocation failed */
#define LHB200_EDECODE (-5)  /* a serialized point failed to decode (bls::Error::InvalidByteLength/BlstError) */

/* ---- lifecycle -------------------------------------------------------------------------------- */

/* Bind the calling process to CUDA device `device` (one process per GPU), create the library stream and
 * scratch arenas and upload constant tables.  Idempotent for the same device. */
LHB200_API int32_t lhb200_init(int32_t device);
LHB200_API void lhb200_shutdown(void);
LHB200_API const char* lhb200_last_error(void);
/* Pinned host memory for callers that want zero-staging H2D (the e2e bench uses it). */
LHB200_API int32_t lhb200_pinned_alloc(void** out, uint64_t nbytes);
LHB200_API int32_t lhb200_pinned_free(void* p);
/* Number of kernel launches issued by this library since init (bench.py's "gpu_launches"). */
LHB200_API uint64_t lhb200_launch_count(void);

/* ---- tree-hash path --------------------------------------------------------------------------- */

/* ethereum_hashing::hash32_concat over n independent 64-byte inputs (consensus/merkle_proof/src/lib.rs:91,
 * :380-384): out[i] = SHA256(in[64i .. 64i+64]). */
LHB200_API int32_t lhb200_hash_pairs(const uint8_t* in, uint8_t* out, uint64_t n);
LHB200_API int32_t lhb200_dev_hash_pairs(const void* d_in, void* d_out, uint64_t n, void* stream);

/* tree_hash::merkle_root / merkleize with a chunk limit of 2^depth (crypto/bls/src/macros.rs:24,
 * SURVEY Appendix B): zero-pads every level with ZERO_HASHES[level]; n_chunks == 0 gives ZERO_HASHES[depth].
 * n_chunks must be <= 2^depth. */
LHB200_API int32_t lhb200_merkleize(const uint8_t* chunks, uint64_t n_chunks, uint32_t depth, uint8_t out[32]);
/* d_chunks must be 16-byte aligned; d_out32 receives the 32-byte root (device memory). */
LHB200_API int32_t lhb200_dev_merkleize(const void* d_chunks, uint64_t n_chunks, uint32_t depth, void* d_out32, void* stream);

/* tree_hash::mix_in_length(root, len) = SHA256(root || le64(len) || 0^24). */
LHB200_API int32_t lhb200_mix_in_length(const uint8_t root[32], uint64_t len, uint8_t out[32]);

/* ZERO_HASHES[depth] (ethereum_hashing::ZERO_HASHES, merkle_proof/src/lib.rs:166), depth <= 64. */
LHB200_API int32_t lhb200_zero_hash(uint32_t depth, uint8_t out[32]);

/* hash_tree_root(List[Validator, 2^40]) from n 121-byte SSZ validators (consensus/types/src/validator.rs:25-35;
 * beacon_state.rs:363).  lhb200_validator_roots writes the n per-validator roots instead. */
LHB200_API int32_t lhb200_validators_root(const uint8_t* ssz, uint64_t n, uint8_t out[32]);
LHB200_API int32_t lhb200_validator_roots(const uint8_t* ssz, uint64_t n, uint8_t* out_roots);

/* BeaconState::update_tree_hash_cache / tree_hash_root for the Deneb variant, mainnet preset, cold (no cached
 * nodes) — consensus/types/src/beacon_state.rs:2031-2038, fields :343-484.  `ssz` is the SSZ encoding of
 * BeaconStateDeneb.  field_roots (28*32 bytes) is optional (NULL to skip). */
LHB200_API int32_t lhb200_beacon_state_root_deneb(const uint8_t* ssz, uint64_t len, uint8_t out[32], uint8_t* field_roots);
/* The other post-Altair variants of the BeaconState superstruct (consensus/types/src/beacon_state.rs:224-571) through
 * the same kernels; `fork` is one of LHB200_FORK_*.  Altair has 24 fields, Bellatrix 25 (+ a 14-field execution payload
 * header), Capella 28 (15-field header, withdrawal indices, historical_summaries), Deneb 28 (17-field header).
 * field_roots (optional, 28 x 32 B): entries beyond the fork's field count are zero chunks. */
#define LHB200_FORK_ALTAIR 1
#define LHB200_FORK_BELLATRIX 2
#define LHB200_FORK_CAPELLA 3
#define LHB200_FORK_DENEB 4
#define LHB200_FORK_ELECTRA 5   /* 37 fields (19-field header, six u64s, three pending_* lists): field_roots is 37 x 32 B */
LHB200_API int32_t lhb200_beacon_state_root(const uint8_t* ssz, uint64_t len, int32_t fork, uint8_t out[32],
                                            uint8_t* field_roots);
LHB200_API int32_t lhb200_state_stage(const uint8_t* ssz, uint64_t len, int32_t fork, struct lhb200_state** out);

/* Device-resident variant: stage once (H2D into the library's aligned HBM layout, DESIGN.md §3), then hash
 * as often as wanted without touching the host link.  The handle owns device memory until released. */
typedef struct lhb200_state lhb200_state;
LHB200_API int32_t lhb200_state_stage_deneb(const uint8_t* ssz, uint64_t len, lhb200_state** out);
LHB200_API int32_t lhb200_state_root(lhb200_state* st, uint8_t out[32], uint8_t* field_roots);
/* Same-length in-place mutation of a staged state — the resident analogue of apply_pending_mutations
 * (beacon_state.rs:2459-2481): bytes [ssz_offset, ssz_offset+len) of the SSZ encoding are replaced; the next
 * lhb200_state_root re-hashes everything on the device (SURVEY.md §8f-3: warm path = patch + full re-hash). */
LHB200_API int32_t lhb200_state_patch(lhb200_state* st, uint64_t ssz_offset, const uint8_t* data, uint64_t len);
/* n non-overlapping same-length mutations in one call (offsets[i], lens[i], bytes concatenated in `data`): one H2D copy
 * and one scatter kernel instead of n round trips — what a slot's worth of milhouse pending updates looks like. */
LHB200_API int32_t lhb200_state_patch_batch(lhb200_state* st, const uint64_t* offsets, const uint32_t* lens,
                                            const uint8_t* data, uint32_t n);
/* Warm path (SURVEY.md §8f-3; the reference's steady state: BeaconState::update_tree_hash_cache re-hashes only dirty
 * paths, beacon_state.rs:2031-2038,2459-2481).  After this call the handle keeps every level of its big lists
 * (validators, balances, inactivity scores, participation x2, randao mixes, block/state roots, slashings) resident:
 * lhb200_state_patch marks the leaves it touches and lhb200_state_root / _enqueue re-hash only the paths above them
 * plus the tail program.  The first root after enabling is cold (it builds the levels); patches to other lists, or
 * more than 65 536 dirty leaves, fall back to a cold root.  Unsharded handles only.  With lhb200_state_root_enqueue the
 * dirty-leaf table is staged through the library's pinned slab: synchronise the stream before the next lhb200_* call
 * (lhb200_state_root does).
 * lhb200_state_last_root_hashes: hash32_concat units the last root actually computed. */
LHB200_API int32_t lhb200_state_enable_incremental(lhb200_state* st);
LHB200_API uint64_t lhb200_state_last_root_hashes(const lhb200_state* st);
/* Same as lhb200_state_root but only enqueues; the root lands in device memory (returned pointer valid until
 * the next call on this handle).  Used by bench.py to time kernels with CUDA events. */
LHB200_API int32_t lhb200_state_root_enqueue(lhb200_state* st, void* stream, const void** d_root);
/* One state sharded over `world` GPUs (a power of two; SURVEY.md §8e): rank r stages and hashes only its leaf range
 * of the big lists (validators, balances, randao_mixes, participation x2, inactivity_scores) plus the small fields.
 *   1. lhb200_state_stage_deneb_shard(ssz, len, rank, world, &h)       every rank, its own slice
 *   2. lhb200_state_shard_roots(h, roots, &n)                          n x 32-byte subtree roots of this rank
 *   3. all-gather the n*32 bytes over NCCL (rank-major)                 the path's single collective
 *   4. lhb200_state_combine(h, gathered, out)                          every rank: log2(world) levels + ladders + top tree */
LHB200_API int32_t lhb200_state_stage_deneb_shard(const uint8_t* ssz, uint64_t len, uint32_t rank, uint32_t world,
                                                  lhb200_state** out);
LHB200_API int32_t lhb200_state_shard_roots(lhb200_state* st, uint8_t* out, uint32_t* n_lists);
LHB200_API int32_t lhb200_state_combine(lhb200_state* st, const uint8_t* gathered, uint8_t out[32]);
/* Steps 2-4 in one call over the library's communicator (lhb200_comm_init): subtree roots stay on the device, one
 * ncclAllGather, every rank folds the top; only the 32-byte root crosses the host link. */
LHB200_API int32_t lhb200_state_root_sharded(lhb200_state* st, uint8_t out[32]);
LHB200_API int32_t lhb200_state_release(lhb200_state* st);
/* Algorithmic work of the last root computed on this handle: number of hash32_concat units. */
LHB200_API uint64_t lhb200_state_hash_units(const lhb200_state* st);
/* Device time (ms) of the dominant kernel (k_validator_roots) in the last completed root, from CUDA events on the
 * launching stream; < 0 if unavailable. */
LHB200_API float lhb200_state_dominant_kernel_ms(const lhb200_state* st);

/* MerkleTree::create(leaves, depth) + generate_proof(index, depth) (consensus/merkle_proof/src/lib.rs:68-99,
 * :290-324): root and the bottom-up branch (depth * 32 bytes).  n <= 2^depth, depth <= 32. */
LHB200_API int32_t lhb200_merkle_tree_proof(const uint8_t* leaves, uint64_t n, uint32_t depth, uint64_t index, uint8_t root[32],
                                 uint8_t* branch);
/* verify_merkle_proof / merkle_root_from_branch batch (merkle_proof/src/lib.rs:357-389): for each i,
 * ok[i] = (fold(leaf_i, branch_i, depth, index_i) == root_i).  branches: n * depth * 32 bytes. */
LHB200_API int32_t lhb200_verify_merkle_proofs(const uint8_t* leaves, const uint8_t* branches, uint32_t depth,
                                    const uint64_t* indices, const uint8_t* roots, uint64_t n, uint8_t* ok);

/* BeaconBlock::canonical_root for BeaconBlockDeneb SSZ bytes, mainnet preset (consensus/types/src/beacon_block.rs:
 * 56-78,158-160; body beacon_block_body.rs:70-121,145-176; payload execution_payload.rs:54-95; operations
 * proposer_slashing.rs:26, attester_slashing.rs:42, indexed_attestation.rs:53, attestation.rs:74, deposit.rs:27,
 * signed_voluntary_exit.rs:25, sync_aggregate.rs:38, signed_bls_to_execution_change.rs:22, withdrawal.rs:22).
 * `body_root` (32 B, optional) receives hash_tree_root(body) — the BeaconBlockHeader.body_root of the block.
 * The batch form hashes n blocks (SSZ blobs concatenated, offsets[n+1]) in one pass: the 32 blocks of an epoch
 * segment (BlockSignatureVerifier / ConsensusContext::get_current_block_root, consensus_context.rs:115-128).
 * Malformed SSZ (bad offsets, over-limit lists, missing bitlist delimiter) -> LHB200_EINVAL. */
LHB200_API int32_t lhb200_beacon_block_root_deneb(const uint8_t* ssz, uint64_t len, uint8_t out[32], uint8_t* body_root);
LHB200_API int32_t lhb200_beacon_block_roots_deneb(const uint8_t* ssz, const uint64_t* offsets, uint32_t n,
                                                   uint8_t* roots, uint8_t* body_roots);
/* Same for BlindedBeaconBlockDeneb SSZ (BlindedBeaconBlock, consensus/types/src/beacon_block.rs:80; the body carries
 * the ExecutionPayloadHeaderDeneb, execution_payload_header.rs:46-87).  The root equals the full block's root. */
LHB200_API int32_t lhb200_blinded_beacon_block_roots_deneb(const uint8_t* ssz, const uint64_t* offsets, uint32_t n,
                                                           uint8_t* roots, uint8_t* body_roots);
/* The same for the earlier variants of the BeaconBlock superstruct (consensus/types/src/beacon_block.rs:41-90,
 * beacon_block_body.rs:43-110): fork = LHB200_FORK_ALTAIR (9 body fields, no execution payload), _BELLATRIX (14-field
 * payload), _CAPELLA (+ withdrawals, bls_to_execution_changes), _DENEB (+ blob gas fields, blob_kzg_commitments);
 * blinded != 0: BlindedBeaconBlock (the body carries the ExecutionPayloadHeader; Bellatrix and later). */
LHB200_API int32_t lhb200_beacon_block_roots(const uint8_t* ssz, const uint64_t* offsets, uint32_t n, int32_t fork,
                                             int32_t blinded, uint8_t* roots, uint8_t* body_roots);

/* swap_or_not_shuffle::shuffle_list (consensus/swap_or_not_shuffle/src/shuffle_list.rs:79-160; SURVEY.md §8f-4):
 * out = shuffle (forwards != 0) or un-shuffle (forwards == 0, the direction the spec uses for committees) of the n
 * 64-bit values of `input`.  n == 0, n > 2^24 or rounds == 0 -> LHB200_EINVAL (the reference returns None). */
LHB200_API int32_t lhb200_shuffle_list(const uint64_t* input, uint64_t n, uint8_t rounds, const uint8_t seed[32],
                                       int32_t forwards, uint64_t* out);

/* ---- BLS batch verification path ---------------------------------------------------------------- */

/* bls::verify_signature_sets (crypto/bls/src/impls/blst.rs:37-119) over SoA-flattened SignatureSets
 * (crypto/bls/src/generic_signature_set.rs:61-121):
 *   sigs        n x 96 B  compressed G2 (ZCash format; all-zero = Lighthouse's "empty" signature -> false)
 *   msgs        n x 32 B  signing roots
 *   pks         K x 96 B  uncompressed affine G1, x || y big-endian (the validator_pubkey_cache.rs:195-199 format;
 *                         keys are NOT re-validated, matching pks_validate=false at blst.rs:115)
 *   pk_offsets  n+1 u32   CSR: set i owns keys [pk_offsets[i], pk_offsets[i+1])
 *   rands       n x u64   nonzero random scalars (blst.rs:55-67), or NULL to have the library draw them
 * *ok = 1 iff  prod_i e(r_i apk_i, H(m_i)) == e(g1, sum_i r_i sig_i)  and every set passed its checks
 * (non-empty, subgroup-checked signature; >= 1 key; aggregate key not at infinity).  n_sets == 0 -> *ok = 0
 * (blst.rs:42-44).  set_status (optional, n bytes): 0 fine, 1 empty sig, 2 sig decode, 3 sig not in subgroup,
 * 4 no keys, 5 aggregate key at infinity, 6 key decode.  fast_aggregate_verify / Signature::verify
 * (blst.rs:196-200, :250-261) are the n_sets == 1 case. */
LHB200_API int32_t lhb200_verify_signature_sets(const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
                                                const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets,
                                                uint8_t* ok, uint8_t* set_status);

/* Many independent bls::verify_signature_sets calls in one pass.  Inputs as lhb200_verify_signature_sets, plus
 *   group_offsets  n_groups+1 u32, CSR over the sets: group g owns sets [group_offsets[g], group_offsets[g+1])
 * ok[g] (n_groups bytes) is exactly what lhb200_verify_signature_sets would return for group g's sets alone
 * (empty group -> 0, blst.rs:42-44).  set_status (optional, n_sets bytes) as in lhb200_verify_signature_sets.
 * group_offsets[0] != 0, not non-decreasing, or group_offsets[n_groups] != n_sets -> LHB200_EINVAL.
 * Per-set verdicts are group_offsets = 0, 1, ..., n; n_groups == 1 is lhb200_verify_signature_sets itself.  Any status
 * other than LHB200_OK leaves every ok[g] = 0.  Re-entrant like lhb200_verify_signature_sets. */
LHB200_API int32_t lhb200_verify_signature_set_groups(const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
        const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets,
        const uint32_t* group_offsets, uint32_t n_groups, uint8_t* ok, uint8_t* set_status);

/* Staged form of the same call (what bench.py times): create once, upload or point at device-resident inputs,
 * enqueue on a stream, read the verdict. */
typedef struct lhb200_bls_batch lhb200_bls_batch;
LHB200_API int32_t lhb200_bls_batch_create(uint32_t max_sets, uint64_t max_keys, lhb200_bls_batch** out);
LHB200_API int32_t lhb200_bls_batch_destroy(lhb200_bls_batch* b);
LHB200_API int32_t lhb200_bls_batch_upload(lhb200_bls_batch* b, const uint8_t* sigs, const uint8_t* msgs,
                                           const uint8_t* pks, const uint32_t* pk_offsets, const uint64_t* rands,
                                           uint32_t n_sets);
LHB200_API int32_t lhb200_bls_batch_set_device_inputs(lhb200_bls_batch* b, const void* d_sigs, const void* d_msgs,
                                                      const void* d_pks, const void* d_offsets, const void* d_rands,
                                                      uint32_t n_sets);
/* Streamed upload: queues the small arrays on `stream` and binds the host key buffer; the host buffers must stay valid
 * and unchanged until lhb200_bls_batch_result returns.  verify_enqueue copies the keys in chunks of whole sets on
 * high-priority streams and aggregates each chunk as it lands while the signature and hash-to-curve kernels already run,
 * so the 1.2 GB of keys of a 100 k x 128 batch cross the host link behind the ALU-bound kernels (SURVEY.md §8d (ii):
 * "H2D must be double-buffered against compute").  lhb200_verify_signature_sets uses this path. */
LHB200_API int32_t lhb200_bls_batch_upload_async(lhb200_bls_batch* b, const uint8_t* sigs, const uint8_t* msgs,
                                                 const uint8_t* pks, const uint32_t* pk_offsets, const uint64_t* rands,
                                                 uint32_t n_sets, void* stream);
LHB200_API int32_t lhb200_bls_batch_verify_enqueue(lhb200_bls_batch* b, void* stream);
LHB200_API int32_t lhb200_bls_batch_result(lhb200_bls_batch* b, void* stream, uint8_t* ok, uint8_t* set_status);
/* Device-resident validator pubkey table — the mirror of ValidatorPubkeyCache
 * (beacon_node/beacon_chain/src/validator_pubkey_cache.rs:20-25,138-140; same 96-byte key format it persists, :195-199).
 * Keys are decoded to Montgomery form once at import; SignatureSets then carry u32 validator indices
 * (what consensus/state_processing/src/per_block_processing/signature_sets.rs:315-320 gathers) instead of 96-byte keys:
 * 512 B instead of 12 288 B per 128-key set on the host link (SURVEY.md §8f-1). */
typedef struct lhb200_pubkey_table lhb200_pubkey_table;
LHB200_API int32_t lhb200_pubkey_table_create(uint64_t capacity, lhb200_pubkey_table** out);
LHB200_API int32_t lhb200_pubkey_table_destroy(lhb200_pubkey_table* t);
LHB200_API int32_t lhb200_pubkey_table_append(lhb200_pubkey_table* t, const uint8_t* pks96, uint64_t n);
LHB200_API uint64_t lhb200_pubkey_table_len(const lhb200_pubkey_table* t);
LHB200_API int32_t lhb200_bls_batch_upload_indexed(lhb200_bls_batch* b, const lhb200_pubkey_table* table,
                                                   const uint8_t* sigs, const uint8_t* msgs, const uint32_t* key_indices,
                                                   const uint32_t* pk_offsets, const uint64_t* rands, uint32_t n_sets);
/* Test hook: final-exponentiated product of the last verify as 12 x 48-byte big-endian Fp (tower order
 * c0.c0.c0 .. c1.c2.c1).  NOTE: this is the cube of the canonical GT element (3 is coprime to r). */
LHB200_API int32_t lhb200_bls_batch_gt(lhb200_bls_batch* b, uint8_t out576[576]);
LHB200_API uint64_t lhb200_bls_batch_launches(const lhb200_bls_batch* b);
/* Device time (ms) of the dominant kernel (k_miller) in the last completed enqueue, from CUDA events recorded on
 * the launching stream; < 0 if unavailable. */
LHB200_API float lhb200_bls_batch_dominant_kernel_ms(const lhb200_bls_batch* b);

/* TSecretKey::public_key / ::sign (crypto/bls/src/impls/blst.rs:282-298): n big-endian 32-byte scalars (< r). */
LHB200_API int32_t lhb200_sk_to_pk(const uint8_t* sk32, uint32_t n, uint8_t* pk48, uint8_t* pk96);
LHB200_API int32_t lhb200_sign(const uint8_t* sk32, const uint8_t* msg32, uint32_t n, uint8_t* sig96);
/* PublicKey::deserialize + key_validate, batch form (blst.rs:130-140; validator_pubkey_cache.rs:116-118).
 * status[i]: 0 ok, 1 infinity (rejected), 2 bad encoding / not on curve, 3 not in subgroup. */
LHB200_API int32_t lhb200_g1_decompress_validate(const uint8_t* pk48, uint32_t n, uint8_t* pk96, uint8_t* status);
/* Signature::deserialize, batch form (blst.rs:192-194): 192-byte affine out; status 0 ok, 1 infinity, 2 bad. */
LHB200_API int32_t lhb200_g2_decompress(const uint8_t* sig96, uint32_t n, uint8_t* out192, uint8_t* status);

/* ---- multi-GPU: the library's own NCCL communicator (one process per GPU; SURVEY.md §8b/§8e) ----
 * Rank 0 obtains the 128-byte id (ncclGetUniqueId) and ships it to the other ranks by any means; every rank then calls
 * lhb200_comm_init (collective).  NCCL is dlopen'ed on first use (libnccl.so.2); single-GPU users never load it.
 * The collectives below run on DEVICE buffers on the library's streams — no host hop, no torch. */
LHB200_API int32_t lhb200_comm_unique_id(uint8_t id[128]);
LHB200_API int32_t lhb200_comm_init(int32_t rank, int32_t world, const uint8_t id[128]);
LHB200_API int32_t lhb200_comm_destroy(void);
LHB200_API int32_t lhb200_comm_info(int32_t* rank, int32_t* world);
/* bls::verify_signature_sets sharded over the communicator: each rank passes its contiguous shard of the sets (an empty
 * shard is allowed); per-rank batch check + ONE ncclAllReduce(min) of the device verdicts; *ok = verdict of the whole
 * batch on every rank.  Shard with equal key counts (lighthouse_b200/parallel.py::shard_ranges_by_keys). */
LHB200_API int32_t lhb200_verify_signature_sets_collective(const uint8_t* sigs, const uint8_t* msgs, const uint8_t* pks,
                                                           const uint32_t* pk_offsets, const uint64_t* rands,
                                                           uint32_t n_sets, uint8_t* ok);
/* Staged form: ncclAllReduce(min) of a batch's device verdict, enqueued on `stream` behind verify_enqueue. */
LHB200_API int32_t lhb200_bls_batch_allreduce_verdict(lhb200_bls_batch* b, void* stream);

/* ---- aggregation surface of a crypto/bls backend (crypto/bls/src/impls/blst.rs) ----
 * TAggregateSignature::add_assign / add_assign_aggregate (blst.rs:230-237): out = sum of n compressed signatures; no
 * subgroup check (the trait's contract), infinity encodings are the identity, n == 0 -> the infinity signature;
 * LHB200_EDECODE if an encoding is malformed. */
LHB200_API int32_t lhb200_g2_aggregate(const uint8_t* sigs96, uint32_t n, uint8_t out96[96]);
/* TAggregatePublicKey::aggregate (blst.rs:178-184; generic_aggregate_public_key.rs:9-15): sum of n uncompressed keys
 * (already validated, per the trait's contract), compressed and/or uncompressed result (either may be NULL).
 * n == 0 -> LHB200_EINVAL; malformed / off-curve key -> LHB200_EDECODE. */
LHB200_API int32_t lhb200_g1_aggregate(const uint8_t* pks96, uint32_t n, uint8_t* out48, uint8_t* out96);
/* TPublicKey::deserialize_uncompressed (blst.rs:142-150), batch form: flag bits and on-curve check, no subgroup check.
 * status[i]: 0 ok, 1 infinity, 2 bad encoding / not on the curve; pk48 (optional) receives the compressed keys.
 * NOTE: lhb200_verify_signature_sets does not repeat the curve check on its explicit `pks` (blst.rs:115
 * pks_validate = false): keys must come from this call, lhb200_g1_decompress_validate or a pubkey table. */
LHB200_API int32_t lhb200_g1_deserialize_uncompressed(const uint8_t* pks96, uint32_t n, uint8_t* pk48, uint8_t* status);
/* TAggregateSignature::aggregate_verify (blst.rs:263-273): *ok = 1 iff e(g1, sig) == prod_i e(pk_i, H(m_i)) and sig is
 * in G2.  n == 0 -> *ok = 0 (generic_aggregate_signature.rs:214-216). */
LHB200_API int32_t lhb200_aggregate_verify(const uint8_t sig96[96], const uint8_t* msgs, const uint8_t* pks96, uint32_t n,
                                           uint8_t* ok);

/* Test hook (no device needed): n blinding scalars from the generator lhb200_verify_signature_sets uses when
 * `rands == NULL` — a ChaCha20 keystream keyed from getrandom(2), zeros skipped (blst.rs:46-68: rand::thread_rng). */
LHB200_API int32_t lhb200_debug_rand_scalars(uint64_t* out, uint32_t n);

/* Test hook: run one stage of the BLS pipeline on a single device thread so `pytest -m gpu` can compare every
 * stage with the oracle.  op: 0 expand_message_xmd(32->256), 1 hash_to_g2(32->96), 2 SSWU(u 96 -> x|y 192),
 * 3 g2_decompress(96 -> [in_subgroup, 96 recompressed], rc=DecodeStatus), 4 g2_mul(96|u64le -> 96),
 * 5 fp2 op([opcode|a|b] -> 96), 6 pairing+final_exp(g1 96|g2 96 -> 576), 7 g1 sum([n|n*96] -> 96). */
LHB200_API int32_t lhb200_debug_bls(int32_t op, const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len,
                                    int32_t* rc);

#ifdef __cplusplus
}
#endif
#endif /* LHB200_H */
