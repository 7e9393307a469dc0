/* poseidon252_b200 -- C ABI of the B200-native batched Poseidon/Hades engine.
 *
 * Drop-in boundary for the hot path of dusk-poseidon (reference = /root/reference, a pure-Rust,
 * one-state-at-a-time CPU crate with no FFI of its own).  The reference's seam for this path is
 * the trait pair dusk_safe::Safe<BlsScalar,5> (impl: src/hades/permutation/scalar.rs:24-36) +
 * Hades<BlsScalar> (src/hades/permutation.rs:34-124) under the public surface src/lib.rs:13-31.
 * This header is what a Rust `extern "C"` block for the batch entry points
 * (hades::permute_batch, Hash::digest_batch, encrypt_batch, decrypt_batch, merkle4) binds; the
 * binding itself is in bindings/rust/ and INTEGRATION.md.
 *
 * Conventions
 *   - p252_fr is bit-identical to `BlsScalar.0`: 4 x u64 little-endian limbs of x*R mod p
 *     (Montgomery form, R = 2^256 mod p, value < p).  No conversion happens at the boundary.
 *   - All batch buffers are item-major arrays (the layout of `&[BlsScalar]`, src/hash.rs:94).
 *   - The caller owns every buffer; the library owns only the context (reference borrows inputs,
 *     src/hash.rs:94, and returns fresh Vecs, src/hash.rs:128).
 *   - `flags` says where the buffers live: P252_MEM_HOST (library stages H2D/D2H itself) or
 *     P252_MEM_DEVICE (pointers are device pointers of ctx's GPU, 16-byte aligned; add
 *     P252_ASYNC to return right after enqueueing on the context's stream).
 *   - Every function returns a p252_status; nothing unwinds across the boundary.  Positive codes
 *     mirror dusk_poseidon::Error (src/error.rs:11-32); negative codes are engine failures.
 *   - There is NO CPU fallback: without a usable sm_100 device p252_create fails.
 *   - A context is bound to one device and one stream; calls on one context serialise (a mutex
 *     inside the context: concurrent callers block, they do not race); separate contexts are
 *     independent (the reference is stateless: ScalarPermutation is a ZST,
 *     src/hades/permutation/scalar.rs:15).
 *   - HOST calls are synchronous; on ANY exit path (success or failure) the staging streams are
 *     joined, and for encrypt/decrypt the staging arenas (secrets, nonces, plaintext) are zeroed.
 */
#ifndef POSEIDON252_B200_H
#define POSEIDON252_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define P252_WIDTH 5 /* dusk_poseidon::HADES_WIDTH, src/hades.rs:34 */

typedef struct p252_fr {
    uint64_t l[4];
} p252_fr;

typedef struct p252_ctx p252_ctx;

typedef enum p252_status {
    P252_OK = 0,
    /* dusk_poseidon::Error, src/error.rs:11-32 */
    P252_ERR_IO_PATTERN_VIOLATION = 1,
    P252_ERR_INVALID_IO_PATTERN = 2,
    P252_ERR_TOO_FEW_INPUT_ELEMENTS = 3,
    P252_ERR_ENCRYPTION_FAILED = 4,
    P252_ERR_DECRYPTION_FAILED = 5,
    P252_ERR_INVALID_POINT = 6,
    /* engine */
    P252_ERR_INVALID_ARGUMENT = -1,
    P252_ERR_CUDA = -2,
    P252_ERR_NCCL = -3,
    P252_ERR_NO_DEVICE = -4,
    P252_ERR_OUT_OF_MEMORY = -5
} p252_status;

/* u64::from(Domain), src/hash.rs:38-56 */
typedef enum p252_domain {
    P252_DOMAIN_MERKLE4 = 0,
    P252_DOMAIN_MERKLE2 = 1,
    P252_DOMAIN_ENCRYPTION = 2,
    P252_DOMAIN_OTHER = 3
} p252_domain;

enum {
    P252_MEM_HOST = 0,
    P252_MEM_DEVICE = 1,
    P252_ASYNC = 2,
    /* p252_merkle4_build_dist only (measurement aids, see p252_tree_level_timings): */
    P252_TIMING = 4,     /* bracket every level's kernel and all-gather with CUDA events */
    P252_NO_GATHER = 8   /* skip the collectives: compute-only timing run, node values above level 0 are NOT valid */
};

/* ---- library / context ------------------------------------------------------------------- */
const char* p252_version(void);
const char* p252_strerror(int status);
int p252_device_count(int* count);

/* Create a context on CUDA device `device` with its own stream.  Fails with P252_ERR_NO_DEVICE
 * when there is no sm_100 GPU (no CPU fallback). */
int p252_create(int device, p252_ctx** out);
/* Same, but enqueue all work on an existing CUDA stream (cudaStream_t passed as void*), e.g. the
 * caller's torch stream, so that the caller's CUDA events bracket the kernels. */
int p252_create_on_stream(int device, void* cuda_stream, p252_ctx** out);
void p252_destroy(p252_ctx* ctx);
int p252_sync(p252_ctx* ctx);
/* Text of the last CUDA/NCCL failure on this context ("" if none). */
const char* p252_last_error(const p252_ctx* ctx);
/* Number of kernels this context has launched since creation. */
uint64_t p252_launch_count(const p252_ctx* ctx);
/* Pinned host memory for P252_MEM_HOST callers that want full PCIe bandwidth. */
int p252_host_alloc(size_t bytes, void** out);
int p252_host_free(void* p);

/* Static facts about the kernels of this build (what one Hades permutation costs in this formulation; used by
 * benchmarks to state the integer-multiplier roofline next to the HBM one).  Set struct_size before the call. */
typedef struct p252_kernel_info {
    uint32_t struct_size;
    uint32_t wide_mul_per_permutation; /* 32x32->64 multiply instructions (IMAD.WIDE / IMAD.HI) per permutation */
    uint32_t dfma_per_permutation;     /* FP64 FMAs of the small-integer MDS layer per permutation              */
    uint32_t montmul_per_permutation;  /* Montgomery products incl. squarings (365; the reference does 2000)    */
    uint32_t threads_per_block;
    uint32_t min_blocks_per_sm;
} p252_kernel_info;
int p252_get_kernel_info(p252_kernel_info* out);

/* Digest and raw-permutation batches of at most `max_items` items run the lane-split kernels (five threads per sponge state: lower latency,
 * ~3x lower throughput per state) -- the regime of single digests and of the top levels of a Merkle tree.  Default
 * 3552 = one lane-split warp per SM sub-partition, the measured crossover (environment variable P252_COOP_MAX
 * overrides it at context creation); 0 disables the lane-split path.  Both
 * kernels produce bit-identical results. */
int p252_set_small_batch_max(p252_ctx* ctx, size_t max_items);

/* Fault injection / inspection for tests (no effect unless called).  p252_debug_fail_chunk: the k-th staged chunk
 * (0-based) of the NEXT host-buffer call on this context fails as if its kernel launch had failed (one shot).
 * p252_debug_staging_nonzero: number of non-zero bytes currently held by the context's staging arenas. */
int p252_debug_fail_chunk(p252_ctx* ctx, long long k);
int p252_debug_staging_nonzero(p252_ctx* ctx, size_t* nonzero_bytes);

/* ---- host-side sponge bookkeeping (no GPU needed) ----------------------------------------- */
/* u64::from(Domain), src/hash.rs:43-55 */
int p252_domain_separator(int domain, uint64_t* out);
/* dusk-safe tag input: `calls` are the io-pattern, absorb(len) = 0x80000000|len, squeeze(len) = len
 * (as produced by io_pattern, src/hash.rs:62-85); consecutive calls of one kind aggregate.
 * Writes the byte string hashed into the tag; *out_len in = capacity, out = length. */
int p252_tag_input(const uint32_t* calls, size_t ncalls, uint64_t domain_sep, uint8_t* out, size_t* out_len);
/* BlsScalar::hash_to_scalar (src/hades/permutation/scalar.rs:29-31): BLAKE2b-512 -> mod p. */
int p252_hash_to_scalar(const uint8_t* bytes, size_t len, p252_fr* out);
/* Safe::tag of the pattern: hash_to_scalar(tag_input(calls, domain_sep)). */
int p252_tag(const uint32_t* calls, size_t ncalls, uint64_t domain_sep, p252_fr* tag);
/* io_pattern(domain, [in_len], out_len) + tag (src/hash.rs:62-85,131-137): checks the Merkle
 * arities (-> P252_ERR_IO_PATTERN_VIOLATION) and zero lengths (-> P252_ERR_INVALID_IO_PATTERN). */
int p252_hash_tag(int domain, size_t in_len, size_t out_len, p252_fr* tag);
/* tag of dusk_safe::encrypt/decrypt for message length L (src/encryption.rs:67-73). */
int p252_encryption_tag(size_t L, p252_fr* tag);

/* ---- batch entry points (the GPU path) ----------------------------------------------------- */
/* hades::permute_batch: n independent Safe::permute calls (src/hades/permutation/scalar.rs:25-27
 * -> Hades::perm, src/hades/permutation.rs:105-123).  states: n x 5, in place. */
int p252_permute_batch(p252_ctx* ctx, p252_fr* states, size_t n, int flags);
/* The reference's dense formulation executed on the device (cross-check / cost comparison). */
int p252_permute_batch_dense(p252_ctx* ctx, p252_fr* states, size_t n, int flags);

/* Sponge with a caller-supplied tag: start(tag) -> absorb(in_len) -> squeeze(out_len)
 * (Hash::finalize, src/hash.rs:128-155).  in: n x in_len, out: n x out_len. */
int p252_digest_batch(p252_ctx* ctx, const p252_fr* tag, const p252_fr* in, size_t n, size_t in_len,
                      p252_fr* out, size_t out_len, int flags);
/* Hash::digest_batch: n x Hash::digest(domain, in[i]) with Hash::output_len(out_len)
 * (src/hash.rs:111-115,191-195); tag computed on the host once per batch. */
int p252_hash_batch(p252_ctx* ctx, int domain, const p252_fr* in, size_t n, size_t in_len, p252_fr* out,
                    size_t out_len, int flags);

/* Hash::digest_truncated batch (src/hash.rs:164-183,203-210): every output scalar is taken out of Montgomery
 * form and masked to 250 bits; out_raw receives the raw limbs the reference passes to JubJubScalar::from_raw. */
int p252_hash_batch_truncated(p252_ctx* ctx, int domain, const p252_fr* in, size_t n, size_t in_len, p252_fr* out_raw,
                              size_t out_len, int flags);

/* Wire format (BlsScalar::from_bytes / to_bytes as used at src/hades.rs:94-105,131): n canonical 32-byte
 * little-endian integers <-> BlsScalar.0.  from_bytes: ok[i] = 0 and out[i] = 0 when the value is >= p (the
 * reference returns None); ok may be NULL. */
int p252_scalars_from_bytes(p252_ctx* ctx, const uint8_t* bytes, size_t n, p252_fr* out, uint8_t* ok, int flags);
int p252_scalars_to_bytes(p252_ctx* ctx, const p252_fr* in, size_t n, uint8_t* bytes, int flags);

/* encrypt_batch: n x encrypt(msg[i], (u,v)[i], nonce[i]) (src/encryption.rs:62-74).
 * msg: n x L, secret_uv: n x 2 (JubJubAffine::get_u/get_v), nonce: n, cipher: n x (L+1). */
int p252_encrypt_batch(p252_ctx* ctx, const p252_fr* msg, size_t n, size_t L, const p252_fr* secret_uv,
                       const p252_fr* nonce, p252_fr* cipher, int flags);
/* decrypt_batch (src/encryption.rs:83-95).  cipher: n x (L+1), msg: n x L, ok: n bytes; ok[i] = 0
 * <=> the reference returns Error::DecryptionFailed for item i (its msg is zeroed; device callers must look at
 * ok[i] before trusting msg[i]).  Returns P252_OK even when some items fail; *n_failed (optional, a HOST pointer
 * for both memory spaces) receives their count -- for device buffers it is counted on the device and, with
 * P252_ASYNC, written by an asynchronous copy that is complete after p252_sync. */
int p252_decrypt_batch(p252_ctx* ctx, const p252_fr* cipher, size_t n, size_t L, const p252_fr* secret_uv,
                       const p252_fr* nonce, p252_fr* msg, uint8_t* ok, size_t* n_failed, int flags);

/* One level of an arity-4 tree: parents[i] = Hash::digest(Domain::Merkle4, children[4i..4i+4])
 * (src/hash.rs:22-26). */
int p252_merkle4_level(p252_ctx* ctx, const p252_fr* children, size_t n_parents, p252_fr* parents, int flags);
/* Number of nodes above the leaves of a full arity-4 tree: (n_leaves-1)/3; n_leaves must be 4^k. */
int p252_merkle4_tree_nodes(size_t n_leaves, size_t* n_internal, int* n_levels);
/* Whole tree on one GPU.  nodes_out: all internal levels, bottom-up, concatenated
 * (n_leaves/4 + n_leaves/16 + ... + 1 scalars); the root is the last element. */
int p252_merkle4_build(p252_ctx* ctx, const p252_fr* leaves, size_t n_leaves, p252_fr* nodes_out, int flags);

/* The same for arity 2 or 4 (node = Hash::digest(Domain::Merkle2 | Merkle4, children), src/hash.rs:22-31):
 * internal nodes = (n_leaves - 1) / (arity - 1); n_leaves must be a power of the arity. */
int p252_merkle_tree_nodes(int arity, size_t n_leaves, size_t* n_internal, int* n_levels);
int p252_merkle_build(p252_ctx* ctx, int arity, const p252_fr* leaves, size_t n_leaves, p252_fr* nodes_out, int flags);

/* ---- Merkle openings (consumer: poseidon-merkle `Opening`, AGENTS.md:62-66; node hash src/hash.rs:22-31) ------
 * A tree is `leaves` (n_leaves = arity^depth) + `nodes` as written by p252_merkle_build.  The opening of leaf i
 * holds, for every level l = 0..depth-1 (0 = the leaf level), the WHOLE sibling group of the path node: the
 * `arity` items at [g*arity, (g+1)*arity) of level l with g = i / arity^(l+1); the path node sits at offset
 * (i / arity^l) % arity inside its group.  Empty slots of a sparse tree are the zero scalar (src/hash.rs:22-31).
 * paths: n x depth x arity scalars, item-major.  leaf_idx lives in the same memory space as the other buffers.  An index
 * >= n_leaves is P252_ERR_INVALID_ARGUMENT for HOST buffers; for DEVICE buffers (not inspected on the host) its opening
 * is all zero, which no root verifies. */
int p252_merkle_open_batch(p252_ctx* ctx, int arity, const p252_fr* leaves, size_t n_leaves, const p252_fr* nodes,
                           const uint64_t* leaf_idx, size_t n, p252_fr* paths_out, int flags);
/* n x Opening::verify: cur = leaf_items[i]; for every level: paths[i][l][pos] must equal cur, then
 * cur = Hash::digest(Domain::Merkle{arity}, paths[i][l]); finally cur must equal *root.  ok[i] = 1 iff all hold
 * (depth permutations per item, fused with the checks in one kernel).  root is a HOST pointer; *n_failed as in
 * p252_decrypt_batch. */
int p252_merkle_verify_batch(p252_ctx* ctx, int arity, int depth, const p252_fr* leaf_items, const uint64_t* leaf_idx,
                             const p252_fr* paths, const p252_fr* root, size_t n, uint8_t* ok, size_t* n_failed,
                             int flags);

/* Overwrite k leaves of a tree held as leaves + nodes (the p252_merkle_build layout; arity 2 or 4, n_leaves = arity^depth)
 * and recompute exactly the internal nodes on their paths.  Afterwards leaves/nodes equal p252_merkle_build of the
 * updated leaves, bit for bit; no other node is written.  leaf_idx / values: k entries, any order; an index may repeat,
 * the LAST occurrence in the batch wins (as k sequential writes would).  leaf_idx lives in the same memory space as the
 * other buffers.  An index >= n_leaves: HOST -> P252_ERR_INVALID_ARGUMENT before anything is written; DEVICE -> that
 * entry is skipped, the others are applied, and *n_rejected (optional HOST pointer, as n_failed of p252_decrypt_batch)
 * receives the number skipped.  k = 0 is a no-op that launches nothing.
 * HOST buffers: only the groups on the dirty paths cross PCIe, and leaves/nodes are written only after all device work
 * succeeded (a failed call leaves the tree untouched).  DEVICE buffers: the plan (sort, dedupe, dirty lists per level)
 * runs on the device with no host synchronisation; a failed call may leave the tree partially updated. */
int p252_merkle_update_batch(p252_ctx* ctx, int arity, p252_fr* leaves, size_t n_leaves, p252_fr* nodes,
                             const uint64_t* leaf_idx, const p252_fr* values, size_t k, size_t* n_rejected, int flags);

/* ---- multi-GPU tree build: one process per GPU, one NCCL all-gather per level ---------------- */
#define P252_NCCL_UNIQUE_ID_BYTES 128
/* rank 0 creates the id and ships it to the other ranks by any means (torch.distributed / MPI) */
int p252_dist_unique_id(uint8_t id[P252_NCCL_UNIQUE_ID_BYTES]);
int p252_dist_init(p252_ctx* ctx, const uint8_t id[P252_NCCL_UNIQUE_ID_BYTES], int rank, int nranks);
int p252_dist_finalize(p252_ctx* ctx);
/* The partition p252_merkle4_build_dist follows (pure host arithmetic, no GPU needed): for every internal
 * level, bottom-up, where it lives in nodes_out, which slice this rank computes, and whether the level is
 * all-gathered (sharded = 1) or computed redundantly by every rank (levels with fewer nodes than ranks). */
typedef struct p252_level_plan {
    uint64_t level_offset; /* first node of the level inside nodes_out            */
    uint64_t level_size;   /* nodes in the level                                   */
    uint64_t my_offset;    /* first node (within the level) this rank computes     */
    uint64_t my_count;     /* how many it computes                                 */
    int32_t sharded;       /* 1: slices + all-gather; 0: every rank computes all   */
    int32_t reserved;
} p252_level_plan;
int p252_merkle4_shard_plan(size_t n_leaves_total, int nranks, int rank, p252_level_plan* levels, int capacity,
                            int* n_levels);
/* leaves_shard: this rank's contiguous n_leaves_total/nranks leaves (DEVICE or HOST per flags).
 * Every level's output is sharded contiguously across ranks, computed, then all-gathered so that
 * each rank ends with the complete level (levels smaller than nranks are computed redundantly).
 * nodes_out (same space as leaves_shard): all internal levels as in p252_merkle4_build. */
int p252_merkle4_build_dist(p252_ctx* ctx, const p252_fr* leaves_shard, size_t n_leaves_total, p252_fr* nodes_out,
                            int flags);
/* Per-level device times of the last p252_merkle4_build_dist(... | P252_TIMING) on this context (synchronises
 * the context first): kernel_ms on the compute stream, gather_ms / gather_bytes of that level's all-gather on the
 * communication stream (0 for levels computed redundantly), and total_ms from the first kernel to the last event. */
typedef struct p252_level_timing {
    uint64_t nodes;        /* nodes of the level                      */
    uint64_t my_nodes;     /* nodes this rank hashed                  */
    uint64_t gather_bytes; /* bytes this rank received + kept (level) */
    float kernel_ms;
    float gather_ms;
} p252_level_timing;
int p252_tree_level_timings(p252_ctx* ctx, p252_level_timing* levels, int capacity, int* n_levels, float* total_ms);

#ifdef __cplusplus
}
#endif
#endif /* POSEIDON252_B200_H */
