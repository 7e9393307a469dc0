// Batch kernels of the B200 Poseidon/Hades engine (sm_100a).  One sponge state per thread, state in
// registers; global memory is touched only by 128-bit accesses: warp-cooperative, fully coalesced
// tiles staged through shared memory for the hash/permute kernels (each LDG.128/STG.128 of a warp
// covers whole 128-byte item chunks), per-thread 2 x 128-bit per scalar for encrypt/decrypt.
//
// Sponge schedule = dusk-safe 0.3 `Sponge` as driven by the reference:
//   Hash::finalize   /root/reference/src/hash.rs:128-155      -> k_sponge_digest
//   encrypt/decrypt  /root/reference/src/encryption.rs:62-95  -> k_encrypt / k_decrypt
//   Safe::permute    /root/reference/src/hades/permutation/scalar.rs:25-27 -> k_permute
// capacity = state[0] = tag, rate = state[1..5]; absorb adds into state[pos+1] and permutes when
// pos == 4; any absorb forces a permutation before the next squeeze.
#include "kernels.h"

#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "hades_device.cuh"

namespace p252 {

#ifndef P252_MINBLOCKS
#define P252_MINBLOCKS 5      // resident 128-thread blocks per SM the register allocation is held to (<= 102 regs)
#endif
#ifndef P252_THREADS
#define P252_THREADS 128
#endif
constexpr int kThreads = P252_THREADS;
constexpr int kMinBlocks = P252_MINBLOCKS;
constexpr int kWarps = kThreads / 32;

#if P252_CONST_SMEM
#define P252_STAGE_TABLES                                             \
    __shared__ __align__(128) uint32_t s_round_tab[P252_TAB_WORDS];   \
    __shared__ __align__(8) uint64_t s_tab_bar;                       \
    const uint32_t* tab = stage_round_tables(s_round_tab, &s_tab_bar);
#else
#define P252_STAGE_TABLES
#endif

struct FrArg {
    uint32_t l[8];
};

__device__ __forceinline__ uint4 ldg128(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

// ---- warp-cooperative 128-byte-chunk gather / scatter -------------------------------------------
// 32 items, one per lane; item k's chunk lives at base + k*stride (stride multiple of 32 B).
// Global side: lane l moves 16 B; 8 consecutive lanes cover one item's 128-byte chunk, so every
// LDG.128 / STG.128 of the warp touches 4 complete 128-byte segments.  Shared side: XOR swizzle on
// the 16-byte column keeps both the row-wise (global side) and the item-per-lane (register side)
// accesses bank-conflict free.
__device__ __forceinline__ void warp_gather(uint4 (*st)[8], const uint8_t* base, size_t stride, int nitems,
                                            int nscal, int lane, uint32_t (&v)[4][8]) {
    const int part = lane & 7;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int item = r * 4 + (lane >> 3);
        uint4 x = make_uint4(0, 0, 0, 0);
        if (item < nitems && (part >> 1) < nscal) x = ldg128(base + (size_t)item * stride + part * 16);
        st[item][part ^ (item & 7)] = x;
    }
    __syncwarp();
#pragma unroll
    for (int p = 0; p < 8; ++p) {
        const uint4 x = st[lane][p ^ (lane & 7)];
        v[p >> 1][(p & 1) * 4 + 0] = x.x;
        v[p >> 1][(p & 1) * 4 + 1] = x.y;
        v[p >> 1][(p & 1) * 4 + 2] = x.z;
        v[p >> 1][(p & 1) * 4 + 3] = x.w;
    }
    __syncwarp();
}

__device__ __forceinline__ void warp_scatter(uint4 (*st)[8], uint8_t* base, size_t stride, int nitems, int nscal,
                                             int lane, const uint32_t (&v)[4][8]) {
#pragma unroll
    for (int p = 0; p < 8; ++p)
        st[lane][p ^ (lane & 7)] = make_uint4(v[p >> 1][(p & 1) * 4 + 0], v[p >> 1][(p & 1) * 4 + 1],
                                              v[p >> 1][(p & 1) * 4 + 2], v[p >> 1][(p & 1) * 4 + 3]);
    __syncwarp();
    const int part = lane & 7;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int item = r * 4 + (lane >> 3);
        if (item < nitems && (part >> 1) < nscal)
            *reinterpret_cast<uint4*>(base + (size_t)item * stride + part * 16) = st[item][part ^ (item & 7)];
    }
    __syncwarp();
}

// ---- per-thread scalar loads / stores (2 x 128-bit) ---------------------------------------------------
__device__ __forceinline__ void load_fr(uint32_t (&d)[8], const uint8_t* p) {
    const uint4 a = ldg128(p), b = ldg128(p + 16);
    d[0] = a.x, d[1] = a.y, d[2] = a.z, d[3] = a.w;
    d[4] = b.x, d[5] = b.y, d[6] = b.z, d[7] = b.w;
}
__device__ __forceinline__ void load_fr_rw(uint32_t (&d)[8], const uint8_t* p) {   // coherent (own stores)
    const uint4 a = *reinterpret_cast<const uint4*>(p), b = *reinterpret_cast<const uint4*>(p + 16);
    d[0] = a.x, d[1] = a.y, d[2] = a.z, d[3] = a.w;
    d[4] = b.x, d[5] = b.y, d[6] = b.z, d[7] = b.w;
}
__device__ __forceinline__ void store_fr(uint8_t* p, const uint32_t (&d)[8]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(d[0], d[1], d[2], d[3]);
    *reinterpret_cast<uint4*>(p + 16) = make_uint4(d[4], d[5], d[6], d[7]);
}

// ---- Hash::digest-shaped sponge: Absorb(in_len) -> Squeeze(out_len), item-major AoS ------------
// One permutation call site: step s > 0 is always preceded by a permutation; steps [0, nin) absorb
// 4-scalar chunks, steps [nin, nin+nout) squeeze 4-scalar chunks.  Permutations = nin + nout - 1
// = ceil(in_len/4) + ceil(out_len/4) - 1  (Merkle4: exactly 1).
// kTruncate: Hash::finalize_truncated (/root/reference/src/hash.rs:164-183) -- every squeezed scalar is taken
// out of Montgomery form and masked to 250 bits; the 4 x u64 written are the raw limbs the reference hands to
// JubJubScalar::from_raw.
// Launch shape: kT threads per block, register allocation held to kMB resident blocks per SM.  128 x 5 (96 registers,
// 20 warps/SM) is the general shape; 256 x 2 (128 registers, 16 warps/SM) is 0.9 % faster on batches of many waves
// and much slower below one wave (8-warp blocks pile onto half the SMs), so only launch_digest's large-batch path uses it.
template <bool kTruncate, int kT = kThreads, int kMB = kMinBlocks>
__global__ void __launch_bounds__(kT, kMB) k_sponge_digest(FrArg tag, const uint8_t* __restrict__ in, size_t n,
                                                            uint32_t in_len, uint8_t* __restrict__ out,
                                                            uint32_t out_len) {
    constexpr int kW = kT / 32;
    __shared__ uint4 stage[kW][32][8];
    P252_STAGE_TABLES
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const size_t item0 = ((size_t)blockIdx.x * kW + warp) * 32;
    if (item0 >= n) return;
    const int nitems = (n - item0 < 32) ? (int)(n - item0) : 32;
    uint4(*st)[8] = stage[warp];

    uint32_t s[5][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        s[0][k] = tag.l[k];
        s[1][k] = s[2][k] = s[3][k] = s[4][k] = 0;
    }
    const uint32_t nin = (in_len + 3) / 4, nout = (out_len + 3) / 4;
    const uint8_t* in_w = in + item0 * (size_t)in_len * 32;
    uint8_t* out_w = out + item0 * (size_t)out_len * 32;
#pragma unroll 1
    for (uint32_t step = 0; step < nin + nout; ++step) {
        if (step > 0) {
            // the last permutation is read only through the rate lanes of the final squeeze chunk
            uint32_t need = 0x1fu;
            if (step + 1 == nin + nout) {
                const uint32_t left = out_len - 4 * (nout - 1);
                need = ((1u << (left < 4 ? left : 4)) - 1u) << 1;
            }
            hades_permute(s, need P252_TAB_PASS);
        }
        if (step < nin) {
            const uint32_t left = in_len - 4 * step;
            const int nscal = left < 4 ? (int)left : 4;
            uint32_t v[4][8];
            warp_gather(st, in_w + (size_t)step * 128, (size_t)in_len * 32, nitems, nscal, lane, v);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q < nscal) {
                    uint32_t t[8];
                    fr_add_mod(t, s[1 + q], v[q]);
#pragma unroll
                    for (int k = 0; k < 8; ++k) s[1 + q][k] = t[k];
                }
            }
        } else {
            const uint32_t c = step - nin;
            const uint32_t left = out_len - 4 * c;
            const int nscal = left < 4 ? (int)left : 4;
            uint32_t v[4][8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (kTruncate) {
                    fr_to_canonical(v[q], s[1 + q]);
                    v[q][7] &= 0x03ffffffu;               // TRUNCATION_MASK, src/hash.rs:167-172
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[q][k] = s[1 + q][k];
                }
            }
            warp_scatter(st, out_w + (size_t)c * 128, (size_t)out_len * 32, nitems, nscal, lane, v);
        }
    }
}

// ---- the same sponge for SMALL batches: five threads per item (hades_permute_coop) ----------------------------------
// 6 items per warp (lanes 0..29), 24 per 128-thread block.  Thread li of a group owns state lane li: lane 0 is the
// capacity (tag), lanes 1..4 the rate, so rate thread li absorbs input scalar 4*step + li - 1 and squeezes output
// scalar 4*c + li - 1.  Loads/stores are 2 x 128-bit per scalar per thread (tiny batches: coalescing is irrelevant).
constexpr int kCoopItemsPerWarp = 6;
__global__ void __launch_bounds__(kThreads) k_sponge_digest_coop(FrArg tag, const uint8_t* __restrict__ in, size_t n,
                                                                 uint32_t in_len, uint8_t* __restrict__ out, uint32_t out_len) {
    const int lane = threadIdx.x & 31;
    const int grp = lane / 5, li = lane - grp * 5, g0 = grp * 5;
    const size_t warp_global = (size_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    const size_t item = warp_global * kCoopItemsPerWarp + grp;
    if (warp_global * kCoopItemsPerWarp >= n) return;            // whole warp idle
    const bool live = (grp < kCoopItemsPerWarp) && (item < n);   // idle threads still take part in the shuffles
    double crow[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) crow[j] = (double)(HADES_LAMBDA / (uint32_t)(li + j + 5));

    uint32_t s[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = (li == 0) ? tag.l[k] : 0u;
    const uint32_t nin = (in_len + 3) / 4, nout = (out_len + 3) / 4;
    const uint8_t* in_i = in + (live ? item : 0) * (size_t)in_len * 32;
    uint8_t* out_i = out + (live ? item : 0) * (size_t)out_len * 32;
#pragma unroll 1
    for (uint32_t step = 0; step < nin + nout; ++step) {
        if (step > 0) hades_permute_coop(s, li, g0, crow);
        if (step < nin) {
            const uint32_t q = 4 * step + (uint32_t)li - 1;      // li == 0 wraps to a huge value -> no absorb
            if (li >= 1 && q < in_len) {
                uint32_t v[8], t[8];
                load_fr(v, in_i + (size_t)q * 32);
                fr_add_mod(t, s, v);
#pragma unroll
                for (int k = 0; k < 8; ++k) s[k] = t[k];
            }
        } else {
            const uint32_t q = 4 * (step - nin) + (uint32_t)li - 1;
            if (live && li >= 1 && q < out_len) store_fr(out_i + (size_t)q * 32, s);
        }
    }
}

// raw permutation, small batches: thread li of a group loads / stores lane li of its state (32 B)
__global__ void __launch_bounds__(kThreads) k_permute_coop(uint8_t* __restrict__ states, size_t n) {
    const int lane = threadIdx.x & 31;
    const int grp = lane / 5, li = lane - grp * 5, g0 = grp * 5;
    const size_t warp_global = (size_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    const size_t item = warp_global * kCoopItemsPerWarp + grp;
    if (warp_global * kCoopItemsPerWarp >= n) return;
    const bool live = (grp < kCoopItemsPerWarp) && (item < n);
    double crow[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) crow[j] = (double)(HADES_LAMBDA / (uint32_t)(li + j + 5));
    uint8_t* p = states + (live ? item : 0) * 160 + (size_t)li * 32;
    uint32_t s[8];
    load_fr_rw(s, p);
    hades_permute_coop(s, li, g0, crow);
    if (live) store_fr(p, s);
}

// ---- raw permutation of n x 5 states in place (Safe::permute) -----------------------------------
template <bool kDense, int kT = kThreads, int kMB = kMinBlocks>
__global__ void __launch_bounds__(kT, kDense ? 1 : kMB) k_permute(uint8_t* __restrict__ states, size_t n) {
    constexpr int kW = kT / 32;
    __shared__ uint4 stage[kW][32][8];
    P252_STAGE_TABLES
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const size_t item0 = ((size_t)blockIdx.x * kW + warp) * 32;
    if (item0 >= n) return;
    const int nitems = (n - item0 < 32) ? (int)(n - item0) : 32;
    uint4(*st)[8] = stage[warp];
    uint8_t* base = states + item0 * 160;

    uint32_t s[5][8];
    {
        uint32_t v[4][8];
        warp_gather(st, base, 160, nitems, 4, lane, v);
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int k = 0; k < 8; ++k) s[q][k] = v[q][k];
        warp_gather(st, base + 128, 160, nitems, 1, lane, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) s[4][k] = v[0][k];
    }
    if (kDense)
        dense_permute(s);
    else
        hades_permute(s, 0x1fu P252_TAB_PASS);
    {
        uint32_t v[4][8];
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int k = 0; k < 8; ++k) v[q][k] = s[q][k];
        warp_scatter(st, base, 160, nitems, 4, lane, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[0][k] = s[4][k];
        warp_scatter(st, base + 128, 160, nitems, 1, lane, v);
    }
}

// ---- encrypt / decrypt (dusk_safe::encrypt / decrypt with Domain::Encryption) -------------------
// pattern [Absorb(2), Absorb(1), Squeeze(L), Absorb(L), Squeeze(1)]; 2*ceil(L/4) permutations.
template <bool kDecrypt>
__global__ void __launch_bounds__(kThreads, kMinBlocks) k_crypt(FrArg tag, const uint8_t* __restrict__ src, size_t n, uint32_t L,
                                                    const uint8_t* __restrict__ secret_uv,
                                                    const uint8_t* __restrict__ nonce, uint8_t* dst,
                                                    uint8_t* __restrict__ ok, unsigned long long* __restrict__ n_failed) {
    P252_STAGE_TABLES
    const size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    // encrypt: src = message (n x L), dst = cipher (n x (L+1)); decrypt: the other way round
    const size_t src_len = kDecrypt ? (size_t)L + 1 : L, dst_len = kDecrypt ? L : (size_t)L + 1;
    const uint8_t* srci = src + i * src_len * 32;
    uint8_t* dsti = dst + i * dst_len * 32;
    const uint8_t* msgi = kDecrypt ? dsti : srci;        // the plaintext, wherever it lives

    uint32_t s[5][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[0][k] = tag.l[k], s[4][k] = 0;
    load_fr(s[1], secret_uv + i * 64);                   // Absorb(2): u, v added to zero
    load_fr(s[2], secret_uv + i * 64 + 32);
    load_fr(s[3], nonce + i * 32);                       // Absorb(1)
    const uint32_t nk = (L + 3) / 4;
    bool good = true;
#pragma unroll 1
    for (uint32_t step = 0; step < 2 * nk; ++step) {
        hades_permute(s, (step + 1 == 2 * nk) ? 0x2u : 0x1fu P252_TAB_PASS);   // last: only the Squeeze(1) lane is read
        if (step < nk) {
            // Squeeze chunk `step` of the keystream and emit cipher (or recovered message)
            const uint32_t left = L - 4 * step;
            const int nscal = left < 4 ? (int)left : 4;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q < nscal) {
                    uint32_t x[8], y[8];
                    load_fr(x, srci + (size_t)(4 * step + q) * 32);
                    if (kDecrypt)
                        fr_sub_mod(y, x, s[1 + q]);      // Encryption::subtract
                    else
                        fr_add_mod(y, x, s[1 + q]);      // Safe::add
                    store_fr(dsti + (size_t)(4 * step + q) * 32, y);
                }
            }
        }
        if (step + 1 >= nk && step + 1 < 2 * nk) {
            // Absorb(L) chunk c of the plaintext: chunk 0 right after the last squeeze (no
            // permutation in between), chunk c > 0 after one more permutation each
            const uint32_t c = step + 1 - nk;
            const uint32_t left = L - 4 * c;
            const int nscal = left < 4 ? (int)left : 4;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q < nscal) {
                    uint32_t x[8], t[8];
                    if (kDecrypt)
                        load_fr_rw(x, msgi + (size_t)(4 * c + q) * 32);
                    else
                        load_fr(x, msgi + (size_t)(4 * c + q) * 32);
                    fr_add_mod(t, s[1 + q], x);
#pragma unroll
                    for (int k = 0; k < 8; ++k) s[1 + q][k] = t[k];
                }
            }
        }
        if (step + 1 == 2 * nk) {
            // Squeeze(1): authentication element
            if (kDecrypt) {
                uint32_t x[8];
                load_fr(x, srci + (size_t)L * 32);
#pragma unroll
                for (int k = 0; k < 8; ++k) good = good && (x[k] == s[1][k]);   // Encryption::is_equal
            } else {
                store_fr(dsti + (size_t)L * 32, s[1]);
            }
        }
    }
    if (kDecrypt) {
        ok[i] = good ? 1 : 0;
        if (!good) {                                      // Error::DecryptionFailed: release nothing
            const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            for (uint32_t k = 0; k < L; ++k) store_fr(dsti + (size_t)k * 32, zero);
        }
        if (n_failed) {                                   // one atomic per warp that saw a failure
            const unsigned act = __activemask();
            const unsigned bad = __ballot_sync(act, !good);
            if (bad && (threadIdx.x & 31) == (unsigned)(__ffs(act) - 1)) atomicAdd(n_failed, (unsigned long long)__popc(bad));
        }
    }
}

// ---- Merkle openings (consumer: poseidon-merkle `Opening`, /root/reference/AGENTS.md:62-66) -------------------
// A tree over n_leaves = arity^depth leaves is stored as `leaves` + `nodes` (internal levels bottom-up, root last:
// the layout p252_merkle_build writes).  The opening of leaf i holds, for every level l = 0..depth-1 (0 = leaf level),
// the whole sibling group of the path node: the `arity` items at positions [g*arity, (g+1)*arity) of level l, with
// g = i / arity^(l+1); the path node itself sits at offset (i / arity^l) % arity inside its group.
// k_merkle_open: pure gather, one thread per (opening, level).
__global__ void __launch_bounds__(256) k_merkle_open(const uint8_t* __restrict__ leaves, const uint8_t* __restrict__ nodes,
                                                     const uint64_t* __restrict__ leaf_idx, size_t n, uint32_t log2_arity,
                                                     uint32_t depth, uint64_t n_leaves, uint8_t* __restrict__ paths) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * depth) return;
    const size_t item = t / depth;
    const uint32_t level = (uint32_t)(t % depth);
    const uint32_t arity = 1u << log2_arity;
    const uint64_t idx = leaf_idx[item];
    uint8_t* dst = paths + ((size_t)item * depth + level) * arity * 32;
    if (idx >= n_leaves) {                                // HOST buffers are rejected on the host; a device index outside
        for (uint32_t q = 0; q < arity * 2; ++q)          // the tree gets an all-zero opening (it cannot verify)
            reinterpret_cast<uint4*>(dst)[q] = make_uint4(0, 0, 0, 0);
        return;
    }
    const uint64_t group = idx >> (log2_arity * (level + 1));
    const uint8_t* src;
    if (level == 0) {
        src = leaves + group * arity * 32;
    } else {
        // offset of internal level (level-1): sum_{q<level-1} n_leaves / arity^(q+1)
        uint64_t off = 0, m = n_leaves >> log2_arity;
        for (uint32_t q = 0; q + 1 < level; ++q, m >>= log2_arity) off += m;
        src = nodes + (off + group * arity) * 32;
    }
    for (uint32_t q = 0; q < arity * 2; ++q)
        reinterpret_cast<uint4*>(dst)[q] = ldg128(src + q * 16);
}

// k_merkle_verify: one thread per opening, `depth` chained Merkle digests (Hash::digest(Domain::MerkleA, group),
// /root/reference/src/hash.rs:22-31,191-195) with the membership check of every level fused in:
//   cur = leaf;  for l: require group[l][pos_l] == cur;  cur = digest(group[l]);   finally require cur == root.
// The sibling groups are read with the same warp-cooperative 128-bit tile as k_sponge_digest.
template <int kLog2Arity>
__global__ void __launch_bounds__(kThreads, kMinBlocks) k_merkle_verify(FrArg tag, FrArg root, const uint8_t* __restrict__ leaf_items,
                                                                        const uint64_t* __restrict__ leaf_idx,
                                                                        const uint8_t* __restrict__ paths, size_t n, uint32_t depth,
                                                                        uint8_t* __restrict__ ok,
                                                                        unsigned long long* __restrict__ n_failed) {
    constexpr int kArity = 1 << kLog2Arity;
    __shared__ uint4 stage[kWarps][32][8];
    P252_STAGE_TABLES
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const size_t item0 = ((size_t)blockIdx.x * kWarps + warp) * 32;
    if (item0 >= n) return;
    const int nitems = (n - item0 < 32) ? (int)(n - item0) : 32;
    const bool live = lane < nitems;
    uint4(*st)[8] = stage[warp];
    const size_t me = item0 + (live ? lane : 0);

    uint32_t cur[8];
    load_fr(cur, leaf_items + me * 32);
    uint64_t idx = leaf_idx[me];
    bool good = true;
    const size_t stride = (size_t)depth * kArity * 32;
    const uint8_t* base = paths + item0 * stride;
#pragma unroll 1
    for (uint32_t level = 0; level < depth; ++level) {
        uint32_t v[4][8];
        warp_gather(st, base + (size_t)level * kArity * 32, stride, nitems, kArity, lane, v);
        const uint32_t pos = (uint32_t)idx & (kArity - 1);
        idx >>= kLog2Arity;
        uint32_t diff = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            uint32_t sel = v[0][k];
#pragma unroll
            for (int q = 1; q < kArity; ++q) sel = (pos == (uint32_t)q) ? v[q][k] : sel;
            diff |= sel ^ cur[k];
        }
        good = good && (diff == 0);
        uint32_t s[5][8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            s[0][k] = tag.l[k];
#pragma unroll
            for (int q = 0; q < 4; ++q) s[1 + q][k] = (q < kArity) ? v[q][k] : 0u;
        }
        hades_permute(s, 0x2u P252_TAB_PASS);          // a Merkle digest reads lane 1 only
#pragma unroll
        for (int k = 0; k < 8; ++k) cur[k] = s[1][k];
    }
    uint32_t diff = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) diff |= cur[k] ^ root.l[k];
    good = good && (diff == 0) && (idx == 0);             // idx != 0: leaf index beyond arity^depth
    if (live) ok[me] = good ? 1 : 0;
    if (n_failed) {
        const unsigned bad = __ballot_sync(0xffffffffu, live && !good);
        if (bad && lane == 0) atomicAdd(n_failed, (unsigned long long)__popc(bad));
    }
}

// ---- incremental Merkle updates: one launch per dirty level -------------------------------------------------------
// Entry j (< n = min(*d_count, bound), or bound when d_count is null) of a level's work list reads the `arity` children
// of group g = read_idx[j] (read_idx null: g = j) at below + g*arity*32, digests them on the Merkle tag and stores the
// parent at out + write_idx[j]*32.  Entries with g >= n_groups are skipped: the device plan ends every list with one
// out-of-range sentinel.  The device path passes the dirty parent list as both indices (read the children of p, write
// p); the host path reads staged groups in list order and writes each parent into its slot among the next level's
// staged groups.
__device__ __forceinline__ size_t update_count(size_t bound, const int64_t* d_count) {
    if (!d_count) return bound;
    const int64_t c = *d_count;
    return c < 0 ? 0 : ((size_t)c < bound ? (size_t)c : bound);
}

// one state per thread; the children of a group are `arity` consecutive scalars (arity 4: one aligned 128-byte line)
template <int kLog2Arity>
__global__ void __launch_bounds__(kThreads, kMinBlocks) k_merkle_update(FrArg tag, const uint8_t* __restrict__ below,
                                                                        const uint64_t* __restrict__ read_idx,
                                                                        const uint64_t* __restrict__ write_idx,
                                                                        uint8_t* __restrict__ out, size_t bound,
                                                                        const int64_t* __restrict__ d_count, uint64_t n_groups) {
    constexpr int kArity = 1 << kLog2Arity;
    P252_STAGE_TABLES
    const size_t j = (size_t)blockIdx.x * kThreads + threadIdx.x;
    if (j >= update_count(bound, d_count)) return;
    const uint64_t g = read_idx ? read_idx[j] : (uint64_t)j;
    if (g >= n_groups) return;
    const uint8_t* src = below + g * (kArity * 32);
    uint32_t s[5][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[0][k] = tag.l[k];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (q < kArity) {
            load_fr(s[1 + q], src + q * 32);
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) s[1 + q][k] = 0;
        }
    }
    hades_permute(s, 0x2u P252_TAB_PASS);              // a Merkle digest reads lane 1 only
    store_fr(out + write_idx[j] * 32, s[1]);
}

// the same with five threads per state (hades_permute_coop): 6 entries per warp, thread li loads lane li of the state
template <int kLog2Arity>
__global__ void __launch_bounds__(kThreads) k_merkle_update_coop(FrArg tag, const uint8_t* __restrict__ below,
                                                                 const uint64_t* __restrict__ read_idx,
                                                                 const uint64_t* __restrict__ write_idx,
                                                                 uint8_t* __restrict__ out, size_t bound,
                                                                 const int64_t* __restrict__ d_count, uint64_t n_groups) {
    constexpr int kArity = 1 << kLog2Arity;
    const int lane = threadIdx.x & 31;
    const int grp = lane / 5, li = lane - grp * 5, g0 = grp * 5;
    const size_t warp_global = (size_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    const size_t j = warp_global * kCoopItemsPerWarp + grp;
    const size_t n = update_count(bound, d_count);
    if (warp_global * kCoopItemsPerWarp >= n) return;            // whole warp idle (n is warp-uniform)
    const uint64_t g = (grp < kCoopItemsPerWarp && j < n) ? (read_idx ? read_idx[j] : (uint64_t)j) : n_groups;
    const bool live = g < n_groups;                              // idle threads still take part in the shuffles
    double crow[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) crow[q] = (double)(HADES_LAMBDA / (uint32_t)(li + q + 5));
    uint32_t s[8];
    if (li == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) s[k] = tag.l[k];
    } else if (live && li <= kArity) {
        load_fr(s, below + g * (kArity * 32) + (size_t)(li - 1) * 32);
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) s[k] = 0;
    }
    hades_permute_coop(s, li, g0, crow);
    if (live && li == 1) store_fr(out + write_idx[j] * 32, s);
}

// ---- device-side planning of an update batch ------------------------------------------------------------------------
// keys[j] = leaf_idx[j], or n_leaves when it is outside the tree (counted into *n_rejected); pos[j] = j.
__global__ void __launch_bounds__(256) k_update_keys(const uint64_t* __restrict__ leaf_idx, size_t k, uint64_t n_leaves,
                                                     uint64_t* __restrict__ keys, uint32_t* __restrict__ pos,
                                                     unsigned long long* __restrict__ n_rejected) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in = j < k;
    bool bad = false;
    if (in) {
        const uint64_t i = leaf_idx[j];
        bad = i >= n_leaves;
        keys[j] = bad ? n_leaves : i;
        pos[j] = (uint32_t)j;
    }
    if (n_rejected) {                                            // one atomic per warp that saw a rejected index
        const unsigned b = __ballot_sync(0xffffffffu, bad);
        if (b && (threadIdx.x & 31) == 0) atomicAdd(n_rejected, (unsigned long long)__popc(b));
    }
}

// After the stable sort the last entry of every run of equal keys is the batch's last write to that leaf.
__global__ void __launch_bounds__(256) k_update_leaves(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ pos,
                                                       size_t k, uint64_t n_leaves, const uint8_t* __restrict__ values,
                                                       uint8_t* __restrict__ leaves) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const uint64_t key = keys[j];
    if (key >= n_leaves || (j + 1 < k && keys[j + 1] == key)) return;
    uint32_t v[8];
    load_fr(v, values + (size_t)pos[j] * 32);
    store_fr(leaves + key * 32, v);
}

// parent of a sorted list entry; everything at or beyond `limit` (rejected leaves, the sentinel) maps to the sentinel
struct ParentOf {
    uint64_t limit;
    int shift;
    __host__ __device__ uint64_t operator()(uint64_t x) const { return x >= limit ? kUpdateSentinel : x >> shift; }
};

MerkleUpdatePlan merkle_update_layout(void* scratch, size_t k, int log2_arity, uint32_t depth, uint64_t n_leaves) {
    MerkleUpdatePlan p{};
    size_t off = 0;
    auto take = [&](size_t bytes) {
        void* q = scratch ? static_cast<uint8_t*>(scratch) + off : nullptr;
        off += (bytes + 255) / 256 * 256;
        return q;
    };
    p.keys_in = static_cast<uint64_t*>(take(k * 8));
    p.keys_out = static_cast<uint64_t*>(take(k * 8));
    p.pos_in = static_cast<uint32_t*>(take(k * 4));
    p.pos_out = static_cast<uint32_t*>(take(k * 4));
    p.counts = static_cast<int64_t*>(take((size_t)depth * 8));
    // list l (parents at level l + 1) holds at most min(entries of the list below, level size + 1 sentinel) entries
    size_t lists_bytes = 0, cap = k;
    uint64_t m = n_leaves;
    for (uint32_t l = 0; l < depth; ++l) {
        m >>= log2_arity;
        cap = cap < m + 1 ? cap : (size_t)(m + 1);
        p.list_cap[l] = cap;
        lists_bytes += cap * 8;
    }
    p.lists_bytes = lists_bytes;
    uint64_t* lists = static_cast<uint64_t*>(take(lists_bytes));
    for (uint32_t l = 0; l < depth; ++l) {
        p.lists[l] = lists;
        if (lists) lists += p.list_cap[l];
    }
    // CUB temporary storage: the larger of the sort's and the widest unique's (sizes only, no device work)
    int end_bit = 1;
    while (end_bit < 64 && (n_leaves >> end_bit) != 0) ++end_bit;   // keys <= n_leaves
    p.end_bit = end_bit;
    size_t sort_bytes = 0, uniq_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, p.keys_in, p.keys_out, p.pos_in, p.pos_out, k, 0, end_bit);
    auto it = thrust::make_transform_iterator(p.keys_out, ParentOf{n_leaves, log2_arity});
    cub::DeviceSelect::Unique(nullptr, uniq_bytes, it, p.lists[0], p.counts, (int64_t)k);
    p.temp_bytes = sort_bytes > uniq_bytes ? sort_bytes : uniq_bytes;
    p.temp = take(p.temp_bytes);
    p.total_bytes = off;
    return p;
}

cudaError_t launch_merkle_update_plan(const MerkleUpdatePlan& p, const uint64_t* leaf_idx, const void* values, size_t k,
                                      int log2_arity, uint32_t depth, uint64_t n_leaves, void* leaves,
                                      unsigned long long* n_rejected, cudaStream_t st) {
    const unsigned grid = (unsigned)((k + 255) / 256);
    k_update_keys<<<grid, 256, 0, st>>>(leaf_idx, k, n_leaves, p.keys_in, p.pos_in, n_rejected);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    size_t tb = p.temp_bytes;
    e = cub::DeviceRadixSort::SortPairs(p.temp, tb, p.keys_in, p.keys_out, p.pos_in, p.pos_out, k, 0, p.end_bit, st);
    if (e != cudaSuccess) return e;
    k_update_leaves<<<grid, 256, 0, st>>>(p.keys_out, p.pos_out, k, n_leaves, static_cast<const uint8_t*>(values),
                                          static_cast<uint8_t*>(leaves));
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    // Entries past a list's unique count stay at the sentinel, so the next level's unique may read the whole
    // capacity: the sentinels collapse into one trailing entry.
    if ((e = cudaMemsetAsync(p.lists[0], 0xff, p.lists_bytes, st)) != cudaSuccess) return e;
    uint64_t m = n_leaves;
    for (uint32_t l = 0; l < depth; ++l) {
        tb = p.temp_bytes;
        if (l == 0)
            e = cub::DeviceSelect::Unique(p.temp, tb, thrust::make_transform_iterator(p.keys_out, ParentOf{n_leaves, log2_arity}),
                                          p.lists[0], p.counts, (int64_t)k, st);
        else
            e = cub::DeviceSelect::Unique(p.temp, tb, thrust::make_transform_iterator(p.lists[l - 1], ParentOf{m, log2_arity}),
                                          p.lists[l], p.counts + l, (int64_t)p.list_cap[l - 1], st);
        if (e != cudaSuccess) return e;
        m >>= log2_arity;
    }
    return cudaSuccess;
}

// ---- host-callable launchers -------------------------------------------------------------------
static inline FrArg to_arg(const uint64_t tag[4]) {
    FrArg a;
    for (int k = 0; k < 4; ++k) {
        a.l[2 * k] = (uint32_t)tag[k];
        a.l[2 * k + 1] = (uint32_t)(tag[k] >> 32);
    }
    return a;
}

static inline unsigned grid_for(size_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }
// digest batches from this size on (>= 7 waves of 256-thread blocks) take the 256 x 2 launch shape
#ifndef P252_WIDE_SHAPE_MIN
#define P252_WIDE_SHAPE_MIN (1u << 19)
#endif
constexpr size_t kWideShapeMinItems = P252_WIDE_SHAPE_MIN;

// Default for p252_set_small_batch_max: batches up to this many items take the lane-split kernel (latency-bound
// regime); the environment variable P252_COOP_MAX overrides it (0 disables the lane-split path).  Measured crossover:
// profiles/README.md "small batches".
#ifndef P252_COOP_MAX_DEFAULT
#define P252_COOP_MAX_DEFAULT 3552   // 148 SMs x 4 sub-partitions x 6 items per warp: one lane-split warp per sub-partition
#endif
size_t coop_max_items() {
    static const size_t v = [] {
        const char* e = getenv("P252_COOP_MAX");
        return e ? (size_t)strtoull(e, nullptr, 10) : (size_t)P252_COOP_MAX_DEFAULT;
    }();
    return v;
}

cudaError_t launch_permute(void* states, size_t n, bool dense, size_t coop_max, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    if (!dense && n <= coop_max) {
        const size_t warps = (n + kCoopItemsPerWarp - 1) / kCoopItemsPerWarp;
        k_permute_coop<<<(unsigned)((warps + kWarps - 1) / kWarps), kThreads, 0, st>>>(static_cast<uint8_t*>(states), n);
        return cudaGetLastError();
    }
    if (dense)
        k_permute<true><<<grid_for(n), kThreads, 0, st>>>(static_cast<uint8_t*>(states), n);
    else if (n >= kWideShapeMinItems)
        k_permute<false, 256, 2><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(static_cast<uint8_t*>(states), n);
    else
        k_permute<false><<<grid_for(n), kThreads, 0, st>>>(static_cast<uint8_t*>(states), n);
    return cudaGetLastError();
}

cudaError_t launch_digest(const uint64_t tag[4], const void* in, size_t n, uint32_t in_len, void* out,
                          uint32_t out_len, bool truncate, size_t coop_max, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    if (!truncate && n <= coop_max) {
        const size_t warps = (n + kCoopItemsPerWarp - 1) / kCoopItemsPerWarp;
        k_sponge_digest_coop<<<(unsigned)((warps + kWarps - 1) / kWarps), kThreads, 0, st>>>(
            to_arg(tag), static_cast<const uint8_t*>(in), n, in_len, static_cast<uint8_t*>(out), out_len);
        return cudaGetLastError();
    }
    if (truncate)
        k_sponge_digest<true><<<grid_for(n), kThreads, 0, st>>>(to_arg(tag), static_cast<const uint8_t*>(in), n, in_len,
                                                                static_cast<uint8_t*>(out), out_len);
    else if (n >= kWideShapeMinItems)
        k_sponge_digest<false, 256, 2><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
            to_arg(tag), static_cast<const uint8_t*>(in), n, in_len, static_cast<uint8_t*>(out), out_len);
    else
        k_sponge_digest<false><<<grid_for(n), kThreads, 0, st>>>(to_arg(tag), static_cast<const uint8_t*>(in), n, in_len,
                                                                 static_cast<uint8_t*>(out), out_len);
    return cudaGetLastError();
}

// ---- wire format: canonical 32-byte little-endian <-> BlsScalar.0 (Montgomery limbs) ---------------------
// BlsScalar::from_bytes / to_bytes (used at /root/reference/src/hades.rs:94-105,131 and
// src/hades/round_constants.rs:64-68).  Elementwise, 32 B in + 32 B out per scalar: the one HBM-bound kernel.
template <bool kFromBytes>
__global__ void __launch_bounds__(256) k_convert(const uint8_t* __restrict__ in, size_t n, uint8_t* __restrict__ out,
                                                 uint8_t* __restrict__ ok) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t x[8], r[8];
    load_fr(x, in + i * 32);
    if (kFromBytes) {
        const bool valid = fr_is_canonical(x);               // from_bytes rejects values >= p
        fr_from_canonical(r, x);
        if (!valid) {
#pragma unroll
            for (int k = 0; k < 8; ++k) r[k] = 0;
        }
        if (ok) ok[i] = valid ? 1 : 0;
    } else {
        fr_to_canonical(r, x);
    }
    store_fr(out + i * 32, r);
}

cudaError_t launch_convert(const void* in, size_t n, void* out, uint8_t* ok, bool from_bytes, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (from_bytes)
        k_convert<true><<<grid, 256, 0, st>>>(static_cast<const uint8_t*>(in), n, static_cast<uint8_t*>(out), ok);
    else
        k_convert<false><<<grid, 256, 0, st>>>(static_cast<const uint8_t*>(in), n, static_cast<uint8_t*>(out), nullptr);
    return cudaGetLastError();
}

cudaError_t launch_encrypt(const uint64_t tag[4], const void* msg, size_t n, uint32_t L, const void* secret_uv,
                           const void* nonce, void* cipher, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_crypt<false><<<grid_for(n), kThreads, 0, st>>>(to_arg(tag), static_cast<const uint8_t*>(msg), n, L,
                                                     static_cast<const uint8_t*>(secret_uv),
                                                     static_cast<const uint8_t*>(nonce),
                                                     static_cast<uint8_t*>(cipher), nullptr, nullptr);
    return cudaGetLastError();
}

cudaError_t launch_decrypt(const uint64_t tag[4], const void* cipher, size_t n, uint32_t L, const void* secret_uv,
                           const void* nonce, void* msg, uint8_t* ok, unsigned long long* n_failed, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_crypt<true><<<grid_for(n), kThreads, 0, st>>>(to_arg(tag), static_cast<const uint8_t*>(cipher), n, L,
                                                    static_cast<const uint8_t*>(secret_uv),
                                                    static_cast<const uint8_t*>(nonce), static_cast<uint8_t*>(msg),
                                                    ok, n_failed);
    return cudaGetLastError();
}

cudaError_t launch_merkle_open(const void* leaves, const void* nodes, const uint64_t* leaf_idx, size_t n, int arity,
                               uint32_t depth, uint64_t n_leaves, void* paths, cudaStream_t st) {
    if (n == 0 || depth == 0) return cudaSuccess;
    const size_t total = n * depth;
    k_merkle_open<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(static_cast<const uint8_t*>(leaves),
                                                                   static_cast<const uint8_t*>(nodes), leaf_idx, n,
                                                                   arity == 4 ? 2u : 1u, depth, n_leaves,
                                                                   static_cast<uint8_t*>(paths));
    return cudaGetLastError();
}

cudaError_t launch_merkle_verify(const uint64_t tag[4], const uint64_t root[4], const void* leaf_items,
                                 const uint64_t* leaf_idx, const void* paths, size_t n, int arity, uint32_t depth,
                                 uint8_t* ok, unsigned long long* n_failed, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    if (arity == 4)
        k_merkle_verify<2><<<grid_for(n), kThreads, 0, st>>>(to_arg(tag), to_arg(root), static_cast<const uint8_t*>(leaf_items),
                                                             leaf_idx, static_cast<const uint8_t*>(paths), n, depth, ok, n_failed);
    else
        k_merkle_verify<1><<<grid_for(n), kThreads, 0, st>>>(to_arg(tag), to_arg(root), static_cast<const uint8_t*>(leaf_items),
                                                             leaf_idx, static_cast<const uint8_t*>(paths), n, depth, ok, n_failed);
    return cudaGetLastError();
}

cudaError_t launch_merkle_update(const uint64_t tag[4], int arity, const void* below, const uint64_t* read_idx,
                                 const uint64_t* write_idx, void* out, size_t bound, const int64_t* d_count,
                                 uint64_t n_groups, size_t coop_max, cudaStream_t st) {
    if (bound == 0) return cudaSuccess;
    const uint8_t* b = static_cast<const uint8_t*>(below);
    uint8_t* o = static_cast<uint8_t*>(out);
    if (bound <= coop_max) {                     // the same choice as launch_digest
        const size_t warps = (bound + kCoopItemsPerWarp - 1) / kCoopItemsPerWarp;
        const unsigned grid = (unsigned)((warps + kWarps - 1) / kWarps);
        if (arity == 4)
            k_merkle_update_coop<2><<<grid, kThreads, 0, st>>>(to_arg(tag), b, read_idx, write_idx, o, bound, d_count, n_groups);
        else
            k_merkle_update_coop<1><<<grid, kThreads, 0, st>>>(to_arg(tag), b, read_idx, write_idx, o, bound, d_count, n_groups);
    } else if (arity == 4) {
        k_merkle_update<2><<<grid_for(bound), kThreads, 0, st>>>(to_arg(tag), b, read_idx, write_idx, o, bound, d_count, n_groups);
    } else {
        k_merkle_update<1><<<grid_for(bound), kThreads, 0, st>>>(to_arg(tag), b, read_idx, write_idx, o, bound, d_count, n_groups);
    }
    return cudaGetLastError();
}

uint32_t wide_mul_per_permutation() { return (uint32_t)kWideMulPerPerm; }
uint32_t dfma_per_permutation() { return (uint32_t)kDfmaPerPerm; }

void kernel_launch_shape(int* threads_per_block, int* min_blocks_per_sm) {
    *threads_per_block = kThreads;
    *min_blocks_per_sm = kMinBlocks;
}

}  // namespace p252
