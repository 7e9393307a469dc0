// Host-callable launchers of the sm_100a kernels (kernels.cu).  Internal to the library; the public
// boundary is include/poseidon252_b200.h.  All pointers are DEVICE pointers, 16-byte aligned;
// scalars are BlsScalar.0 (4 x u64 LE limbs, Montgomery form, < p).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace p252 {

cudaError_t launch_permute(void* states, size_t n, bool dense, size_t coop_max, cudaStream_t st);
// coop_max: batches of at most this many items run the lane-split (5 threads per state) kernel
cudaError_t launch_digest(const uint64_t tag[4], const void* in, size_t n, uint32_t in_len, void* out,
                          uint32_t out_len, bool truncate, size_t coop_max, cudaStream_t st);
cudaError_t launch_convert(const void* in, size_t n, void* out, uint8_t* ok, bool from_bytes, cudaStream_t st);
cudaError_t launch_encrypt(const uint64_t tag[4], const void* msg, size_t n, uint32_t L, const void* secret_uv,
                           const void* nonce, void* cipher, cudaStream_t st);
// n_failed (device pointer, may be null): incremented by the number of items whose authentication failed
cudaError_t launch_decrypt(const uint64_t tag[4], const void* cipher, size_t n, uint32_t L, const void* secret_uv,
                           const void* nonce, void* msg, uint8_t* ok, unsigned long long* n_failed, cudaStream_t st);
// Merkle openings over the leaves + bottom-up internal-level layout of p252_merkle_build (arity 2 or 4)
cudaError_t launch_merkle_open(const void* leaves, const void* nodes, const uint64_t* leaf_idx, size_t n, int arity,
                               uint32_t depth, uint64_t n_leaves, void* paths, cudaStream_t st);
cudaError_t launch_merkle_verify(const uint64_t tag[4], const uint64_t root[4], const void* leaf_items,
                                 const uint64_t* leaf_idx, const void* paths, size_t n, int arity, uint32_t depth,
                                 uint8_t* ok, unsigned long long* n_failed, cudaStream_t st);

// ---- incremental Merkle updates ----
// Work list of one level: read the `arity` children of group read_idx[j] (null: j) at below + g*arity*32, write the
// digest at out + write_idx[j]*32, for j < min(*d_count, bound) (d_count null: bound); groups >= n_groups are skipped.
// bound <= coop_max takes the lane-split form; both forms are bit-identical.
cudaError_t launch_merkle_update(const uint64_t tag[4], int arity, const void* below, const uint64_t* read_idx,
                                 const uint64_t* write_idx, void* out, size_t bound, const int64_t* d_count,
                                 uint64_t n_groups, size_t coop_max, cudaStream_t st);

// Marks the end of a dirty list; no level has this many nodes.
constexpr uint64_t kUpdateSentinel = ~0ull;
constexpr int kMaxDepth = 64;

// Device scratch of one update batch of k leaves: the (index, batch position) pairs before and after the stable radix
// sort, and for every level l = 0..depth-1 the sorted dirty parent list of level l+1 (lists[l], at most list_cap[l]
// entries, padded with kUpdateSentinel; counts[l] = entries written by the unique, sentinel included) + CUB temp storage.
struct MerkleUpdatePlan {
    uint64_t* keys_in;
    uint64_t* keys_out;
    uint32_t* pos_in;
    uint32_t* pos_out;
    int64_t* counts;
    uint64_t* lists[kMaxDepth];
    size_t list_cap[kMaxDepth];
    size_t lists_bytes;
    void* temp;
    size_t temp_bytes;
    int end_bit;
    size_t total_bytes;
};
// Carves the plan out of `scratch` (null: pointers stay null, only the sizes are computed; total_bytes = what to allocate).
MerkleUpdatePlan merkle_update_layout(void* scratch, size_t k, int log2_arity, uint32_t depth, uint64_t n_leaves);
// Enqueues the whole plan: keys (indices >= n_leaves -> counted into *n_rejected, may be null, and dropped), stable
// sort, last-write-wins store of the new values into `leaves`, and the dirty list of every level.  No host sync.
cudaError_t launch_merkle_update_plan(const MerkleUpdatePlan& p, const uint64_t* leaf_idx, const void* values, size_t k,
                                      int log2_arity, uint32_t depth, uint64_t n_leaves, void* leaves,
                                      unsigned long long* n_rejected, cudaStream_t st);

void kernel_launch_shape(int* threads_per_block, int* min_blocks_per_sm);
size_t coop_max_items();   // default small-batch threshold (P252_COOP_MAX or the built-in value)
// 32x32->64-bit multiply instructions (IMAD.WIDE / IMAD.HI class) and DFMA per Hades permutation, counted from
// the generated PTX (fr_ptx.cuh) and the round structure of hades_permute()
uint32_t wide_mul_per_permutation();
uint32_t dfma_per_permutation();

}  // namespace p252
