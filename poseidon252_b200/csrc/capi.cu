// C ABI of poseidon252_b200 (include/poseidon252_b200.h): context, host-side sponge bookkeeping
// (io-pattern checks, tag derivation), staging for HOST buffers, kernel launches, and the
// multi-GPU arity-4 tree build (one process per GPU, NCCL all-gather per level).
//
// Mirrors, for the batch path, the reference's public surface (/root/reference/src/lib.rs:13-31):
//   Hash / Domain / io_pattern      src/hash.rs:21-155      -> p252_hash_tag, p252_hash_batch
//   encrypt / decrypt               src/encryption.rs:62-95 -> p252_encrypt_batch, p252_decrypt_batch
//   Error                           src/error.rs:11-44      -> p252_status
// No permutation is ever computed on the host: without a CUDA device every batch call fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types only: the NCCL entry points are resolved at run time (see NcclApi below)

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/poseidon252_b200.h"
#include "host_field.h"
#include "kernels.h"

namespace {

constexpr int kSlots = 3;                    // H2D / compute / D2H overlap for HOST buffers
constexpr size_t kChunkItemsDefault = 1 << 17;   // items per staged chunk (upper bound, also capped by kChunkBytesTarget);
                                                // P252_CHUNK_ITEMS overrides.  e2e ms per 2^20-digest step: 2^15 6.67, 2^16 6.43,
                                                // 2^17 6.43 (equal within run-to-run noise), 157k (bytes cap) 6.48
size_t chunk_items_max() {
    static const size_t v = [] {
        const char* e = getenv("P252_CHUNK_ITEMS");
        const size_t x = e ? (size_t)strtoull(e, nullptr, 10) : kChunkItemsDefault;
        return x >= 1024 ? x : kChunkItemsDefault;
    }();
    return v;
}
constexpr size_t kChunkBytesTarget = 24u << 20;

struct Slot {
    cudaStream_t stream = nullptr;
    void* arena = nullptr;
    size_t arena_bytes = 0;
};

}  // namespace

struct p252_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    Slot slots[kSlots];
    cudaEvent_t ev_fork = nullptr;
    cudaEvent_t ev_join[kSlots] = {nullptr, nullptr, nullptr};
    uint64_t launches = 0;
    std::string last_error;
    // calls on one context serialise (recursive: public entry points call each other)
    std::recursive_mutex mu;
    // device-side failure counter (decrypt / opening verification on DEVICE buffers) + its pinned mirror
    unsigned long long* d_counter = nullptr;
    unsigned long long* h_counter = nullptr;
    size_t coop_max = 0;          // small-batch threshold of the lane-split digest kernel
    // test hook: index of the staged chunk that fails in the next host-buffer call (-1 = none)
    long long fail_chunk = -1;
    // multi-GPU
    ncclComm_t comm = nullptr;
    int rank = 0, nranks = 1;
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t ev_level = nullptr, ev_comm = nullptr;
    // per-level timing of the last P252_TIMING tree build
    struct LevelEvents {
        cudaEvent_t k0 = nullptr, k1 = nullptr, g0 = nullptr, g1 = nullptr;
    };
    std::vector<LevelEvents> level_events;
    std::vector<p252_level_timing> level_info;   // static part (nodes, bytes) of the last timed build
    std::vector<char> level_gathered;
    int timed_levels = 0;
    cudaEvent_t ev_tree_end = nullptr;
    // device scratch of p252_merkle_update_batch (plan of DEVICE calls, staged groups of HOST calls); grows on demand
    void* upd_scratch = nullptr;
    size_t upd_scratch_bytes = 0;
};

#define P252_LOCK(ctx) std::lock_guard<std::recursive_mutex> lock__((ctx)->mu)

namespace {

// NCCL is bound lazily with dlopen so that (a) single-GPU users carry no NCCL dependency and (b) inside a
// process that already loaded a libnccl.so.2 (e.g. the one bundled with PyTorch) that same copy is used
// instead of a second, possibly older, system copy.
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

NcclApi& nccl() {
    static NcclApi api;
    if (api.handle) return api;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD);     // a copy this process already has
        if (api.handle) break;
    }
    for (const char* n : names) {
        if (api.handle) break;
        api.handle = dlopen(n, RTLD_NOW | RTLD_LOCAL);
    }
    if (!api.handle) return api;
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(api.handle, "ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(api.handle, "ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(api.handle, "ncclCommDestroy"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(dlsym(api.handle, "ncclAllGather"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(api.handle, "ncclGetErrorString"));
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllGather && api.GetErrorString;
    return api;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        cudaGetDevice(&cur);
        if (prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

int fail_cuda(p252_ctx* ctx, cudaError_t e, const char* where) {
    if (ctx) ctx->last_error = std::string(where) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? P252_ERR_OUT_OF_MEMORY : P252_ERR_CUDA;
}
int fail_nccl(p252_ctx* ctx, ncclResult_t e, const char* where) {
    if (ctx) ctx->last_error = std::string(where) + ": " + (nccl().ok ? nccl().GetErrorString(e) : "NCCL unavailable");
    return P252_ERR_NCCL;
}
#define CU(call)                                              \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return fail_cuda(ctx, e__, #call); \
    } while (0)
#define NC(call)                                              \
    do {                                                      \
        ncclResult_t e__ = (call);                            \
        if (e__ != ncclSuccess) return fail_nccl(ctx, e__, #call); \
    } while (0)

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// One staged buffer of a HOST call.
struct Io {
    const void* h_in;    // copied to the device before the launch (may be null)
    void* h_out;         // copied back after the launch (may be null)
    size_t item_bytes;   // bytes per batch item
};

// wipe = true: the staging arenas held secrets (shared secret, nonce, plaintext); they are cleared before
// returning (the reference's dependencies zeroize sponge state, Cargo.toml:15,17 "zeroize").
// Whatever happens inside the chunk loop, the common exit below runs: slot streams are joined back into the
// context stream, the arenas are wiped if asked, and the call returns only after everything enqueued has
// finished -- so on an error no copy into the caller's buffers is still in flight and no secret is left staged.
template <typename Launch>
int run_host_pipeline(p252_ctx* ctx, std::vector<Io>& ios, size_t n, Launch launch, bool wipe = false) {
    if (n == 0) return P252_OK;
    size_t per_item = 0;
    for (auto& io : ios) per_item += (io.item_bytes + 15) / 16 * 16;
    size_t chunk = std::max<size_t>(1024, std::min(chunk_items_max(), kChunkBytesTarget / std::max<size_t>(per_item, 1)));
    chunk = (chunk + 127) / 128 * 128;
    if (chunk > n) chunk = n;
    const long long fail_at = ctx->fail_chunk;
    ctx->fail_chunk = -1;                                  // one shot

    auto body = [&]() -> int {
        // fork: slots wait for everything already enqueued on the context stream
        CU(cudaEventRecord(ctx->ev_fork, ctx->stream));
        for (int s = 0; s < kSlots; ++s) CU(cudaStreamWaitEvent(ctx->slots[s].stream, ctx->ev_fork, 0));
        // Ramp-up (batches of several chunks only): the first chunks are small (chunk/8, /4, /2) so that the first
        // kernel starts after a ~1 MiB copy instead of a full chunk's; from the fourth chunk on every chunk has the
        // full size.  A batch that fits one chunk is one launch.
        size_t k = 0, cur = (n > 2 * chunk) ? std::max<size_t>(1024, chunk / 8 / 128 * 128) : chunk;
        for (size_t off = 0, cnt = 0; off < n; off += cnt, ++k, cur = std::min(chunk, cur * 2)) {
            cnt = std::min(cur, n - off);
            Slot& sl = ctx->slots[k % kSlots];
            // arena layout: one 256-byte aligned region per buffer
            size_t need = 0;
            for (auto& io : ios) need += (chunk * io.item_bytes + 255) / 256 * 256;
            if (sl.arena_bytes < need) {
                CU(cudaStreamSynchronize(sl.stream));
                if (sl.arena) {
                    if (wipe) CU(cudaMemset(sl.arena, 0, sl.arena_bytes));
                    CU(cudaFree(sl.arena));
                }
                sl.arena = nullptr;
                sl.arena_bytes = 0;
                CU(cudaMalloc(&sl.arena, need));
                sl.arena_bytes = need;
            }
            std::vector<void*> d(ios.size());
            size_t pos = 0;
            for (size_t b = 0; b < ios.size(); ++b) {
                d[b] = static_cast<uint8_t*>(sl.arena) + pos;
                pos += (chunk * ios[b].item_bytes + 255) / 256 * 256;
                if (ios[b].h_in)
                    CU(cudaMemcpyAsync(d[b], static_cast<const uint8_t*>(ios[b].h_in) + off * ios[b].item_bytes,
                                       cnt * ios[b].item_bytes, cudaMemcpyHostToDevice, sl.stream));
            }
            cudaError_t le = ((long long)k == fail_at) ? cudaErrorLaunchFailure : launch(d.data(), cnt, sl.stream);
            if (le != cudaSuccess) return fail_cuda(ctx, le, (long long)k == fail_at ? "kernel launch (injected fault)" : "kernel launch");
            ctx->launches++;
            for (size_t b = 0; b < ios.size(); ++b)
                if (ios[b].h_out)
                    CU(cudaMemcpyAsync(static_cast<uint8_t*>(ios[b].h_out) + off * ios[b].item_bytes, d[b],
                                       cnt * ios[b].item_bytes, cudaMemcpyDeviceToHost, sl.stream));
        }
        return P252_OK;
    };
    int rc = body();

    // ---- common exit (success and failure): wipe, join, drain --------------------------------------------------
    const std::string first_error = ctx->last_error;
    cudaError_t ce = cudaSuccess;
    auto keep = [&](cudaError_t e) {
        if (e != cudaSuccess && ce == cudaSuccess) ce = e;
    };
    for (int s = 0; s < kSlots; ++s) {
        Slot& sl = ctx->slots[s];
        if (wipe && sl.arena) keep(cudaMemsetAsync(sl.arena, 0, sl.arena_bytes, sl.stream));
        keep(cudaEventRecord(ctx->ev_join[s], sl.stream));
        keep(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[s], 0));
    }
    keep(cudaStreamSynchronize(ctx->stream));   // HOST calls are synchronous on return, like the reference
    if (rc != P252_OK) {
        // make sure nothing is in flight even if the join itself could not be enqueued
        for (int s = 0; s < kSlots; ++s) cudaStreamSynchronize(ctx->slots[s].stream);
        cudaGetLastError();
        ctx->last_error = first_error;
        return rc;
    }
    if (ce != cudaSuccess) return fail_cuda(ctx, ce, "host pipeline join");
    return P252_OK;
}

// Counts n enqueued kernels, or turns a failed launch into a status.
int count_launch(p252_ctx* ctx, cudaError_t le, const char* what = "kernel launch", int n = 1) {
    if (le != cudaSuccess) return fail_cuda(ctx, le, what);
    ctx->launches += n;
    return P252_OK;
}

void CUDART_CB publish_counter(void* arg) {
    auto* pr = static_cast<std::pair<const unsigned long long*, size_t*>*>(arg);
    *pr->second = (size_t)*pr->first;
    delete pr;
}

// Every DEVICE-buffer call: launch(counter) enqueues the work on the context stream, counts its launches
// (count_launch) and returns a status.  With n_failed, counter is the context's device counter, zeroed before the
// launch and afterwards copied to the pinned mirror and from there to *n_failed by a host function on the stream, so
// that P252_ASYNC callers see it after p252_sync; without, counter is null.  Synchronises unless P252_ASYNC.
template <typename Launch>
int device_call(p252_ctx* ctx, int flags, size_t* n_failed, Launch launch) {
    if (n_failed) CU(cudaMemsetAsync(ctx->d_counter, 0, sizeof(unsigned long long), ctx->stream));
    const int rc = launch(n_failed ? ctx->d_counter : nullptr);
    if (rc != P252_OK) return rc;
    if (n_failed) {
        CU(cudaMemcpyAsync(ctx->h_counter, ctx->d_counter, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        auto* pr = new std::pair<const unsigned long long*, size_t*>(ctx->h_counter, n_failed);
        cudaError_t e = cudaLaunchHostFunc(ctx->stream, publish_counter, pr);
        if (e != cudaSuccess) {
            delete pr;
            return fail_cuda(ctx, e, "cudaLaunchHostFunc");
        }
    }
    if (!(flags & P252_ASYNC)) CU(cudaStreamSynchronize(ctx->stream));
    return P252_OK;
}

// HOST calls that write one ok byte per item: once the call succeeded, *n_failed (optional) = the zero bytes.
int count_failed(int rc, const uint8_t* ok, size_t n, size_t* n_failed) {
    if (rc == P252_OK && n_failed) *n_failed = (size_t)std::count(ok, ok + n, 0);
    return rc;
}

uint64_t domain_sep(int domain, bool* ok) {
    *ok = true;
    switch (domain) {
        case P252_DOMAIN_MERKLE4: return 0x000000000000000fULL;      // src/hash.rs:47
        case P252_DOMAIN_MERKLE2: return 0x0000000000000003ULL;      // src/hash.rs:49
        case P252_DOMAIN_ENCRYPTION: return 0x0000000100000000ULL;   // src/hash.rs:51
        case P252_DOMAIN_OTHER: return 0;                            // src/hash.rs:53
    }
    *ok = false;
    return 0;
}

const uint64_t* limbs(const p252_fr* f) { return f->l; }

// Tag of one Merkle node: Hash::digest(Domain::Merkle2 | Merkle4, `arity` children), src/hash.rs:22-31.
int merkle_tag(int arity, p252_fr* tag) {
    if (arity != 2 && arity != 4) return P252_ERR_INVALID_ARGUMENT;
    return p252_hash_tag(arity == 4 ? P252_DOMAIN_MERKLE4 : P252_DOMAIN_MERKLE2, (size_t)arity, 1, tag);
}

// A full Merkle tree in the layout p252_merkle_build writes: height 0 is the n_leaves = arity^depth leaves (the
// caller's `leaves`), heights 1..depth are the internal levels, bottom-up and concatenated in `nodes`; the root
// (height depth) is the last node.
struct Tree {
    int arity, log2_arity, depth;
    size_t n_leaves, n_internal;
    p252_fr tag;
    size_t off[p252::kMaxDepth + 1];   // offset(h), precomputed: the HOST gathers look it up per item and level
    size_t size(int h) const { return n_leaves >> (log2_arity * h); }
    // first node of height h inside its buffer: 0 for the leaves, n_internal - 1 for the root
    size_t offset(int h) const { return off[h]; }
    template <typename T>
    T* level(T* leaves, T* nodes, int h) const { return (h == 0 ? leaves : nodes) + offset(h); }
    // the `arity` children of group g at height h
    template <typename T>
    T* group(T* leaves, T* nodes, int h, uint64_t g) const { return level(leaves, nodes, h) + g * (uint64_t)arity; }
};
static_assert(p252::kMaxDepth >= 63, "a tree with at most 2^64 - 1 leaves has at most 63 levels");

// P252_ERR_INVALID_ARGUMENT for an arity other than 2 or 4 or fewer than 2 leaves, P252_ERR_IO_PATTERN_VIOLATION when a
// level is not a multiple of the arity.
int make_tree(int arity, size_t n_leaves, Tree* t) {
    int rc = merkle_tag(arity, &t->tag);
    if (rc != P252_OK) return rc;
    if (n_leaves < 2) return P252_ERR_INVALID_ARGUMENT;
    t->arity = arity;
    t->log2_arity = arity == 4 ? 2 : 1;
    t->depth = 0;
    for (size_t m = n_leaves; m > 1; m /= (size_t)arity, ++t->depth)
        if (m % (size_t)arity) return P252_ERR_IO_PATTERN_VIOLATION;
    t->n_leaves = n_leaves;
    t->n_internal = (n_leaves - 1) / (size_t)(arity - 1);
    t->off[0] = t->off[1] = 0;
    for (int h = 2; h <= t->depth; ++h) t->off[h] = t->off[h - 1] + t->size(h - 1);
    return P252_OK;
}

}  // namespace

extern "C" {

const char* p252_version(void) { return "poseidon252_b200 0.1.0 (sm_100a)"; }

const char* p252_strerror(int status) {
    switch (status) {
        case P252_OK: return "ok";
        case P252_ERR_IO_PATTERN_VIOLATION: return "IOPatternViolation";
        case P252_ERR_INVALID_IO_PATTERN: return "InvalidIOPattern";
        case P252_ERR_TOO_FEW_INPUT_ELEMENTS: return "TooFewInputElements";
        case P252_ERR_ENCRYPTION_FAILED: return "EncryptionFailed";
        case P252_ERR_DECRYPTION_FAILED: return "DecryptionFailed";
        case P252_ERR_INVALID_POINT: return "InvalidPoint";
        case P252_ERR_INVALID_ARGUMENT: return "invalid argument";
        case P252_ERR_CUDA: return "CUDA error";
        case P252_ERR_NCCL: return "NCCL error";
        case P252_ERR_NO_DEVICE: return "no usable sm_100 CUDA device (there is no CPU fallback)";
        case P252_ERR_OUT_OF_MEMORY: return "out of device memory";
    }
    return "unknown status";
}

int p252_device_count(int* count) {
    if (!count) return P252_ERR_INVALID_ARGUMENT;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    *count = n;
    return P252_OK;
}

int p252_create_on_stream(int device, void* cuda_stream, p252_ctx** out) {
    if (!out) return P252_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return P252_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) return P252_ERR_INVALID_ARGUMENT;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return P252_ERR_NO_DEVICE;
    if (prop.major != 10) return P252_ERR_NO_DEVICE;   // kernels are sm_100a SASS only
    p252_ctx* ctx = new p252_ctx();
    ctx->device = device;
    ctx->coop_max = p252::coop_max_items();
    DeviceGuard g(device);
    auto bail = [&](cudaError_t e, const char* w) {
        int rc = fail_cuda(nullptr, e, w);
        p252_destroy(ctx);
        return rc;
    };
    cudaError_t e;
    if (cuda_stream) {
        ctx->stream = static_cast<cudaStream_t>(cuda_stream);
        ctx->own_stream = false;
    } else {
        if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess)
            return bail(e, "cudaStreamCreate");
        ctx->own_stream = true;
    }
    for (int s = 0; s < kSlots; ++s) {
        if ((e = cudaStreamCreateWithFlags(&ctx->slots[s].stream, cudaStreamNonBlocking)) != cudaSuccess)
            return bail(e, "cudaStreamCreate");
        if ((e = cudaEventCreateWithFlags(&ctx->ev_join[s], cudaEventDisableTiming)) != cudaSuccess)
            return bail(e, "cudaEventCreate");
    }
    if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess)
        return bail(e, "cudaEventCreate");
    if ((e = cudaEventCreateWithFlags(&ctx->ev_level, cudaEventDisableTiming)) != cudaSuccess)
        return bail(e, "cudaEventCreate");
    if ((e = cudaEventCreateWithFlags(&ctx->ev_comm, cudaEventDisableTiming)) != cudaSuccess)
        return bail(e, "cudaEventCreate");
    if ((e = cudaEventCreate(&ctx->ev_tree_end)) != cudaSuccess) return bail(e, "cudaEventCreate");
    if ((e = cudaMalloc(reinterpret_cast<void**>(&ctx->d_counter), sizeof(unsigned long long))) != cudaSuccess)
        return bail(e, "cudaMalloc");
    if ((e = cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_counter), sizeof(unsigned long long), cudaHostAllocPortable)) != cudaSuccess)
        return bail(e, "cudaHostAlloc");
    *ctx->h_counter = 0;
    *out = ctx;
    return P252_OK;
}

int p252_create(int device, p252_ctx** out) { return p252_create_on_stream(device, nullptr, out); }

void p252_destroy(p252_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard g(ctx->device);
    if (ctx->comm && nccl().ok) nccl().CommDestroy(ctx->comm);
    if (ctx->comm_stream) cudaStreamDestroy(ctx->comm_stream);
    for (int s = 0; s < kSlots; ++s) {
        if (ctx->slots[s].stream) {
            cudaStreamSynchronize(ctx->slots[s].stream);
            cudaStreamDestroy(ctx->slots[s].stream);
        }
        if (ctx->slots[s].arena) cudaFree(ctx->slots[s].arena);
        if (ctx->ev_join[s]) cudaEventDestroy(ctx->ev_join[s]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_level) cudaEventDestroy(ctx->ev_level);
    if (ctx->ev_comm) cudaEventDestroy(ctx->ev_comm);
    if (ctx->ev_tree_end) cudaEventDestroy(ctx->ev_tree_end);
    for (auto& le : ctx->level_events)
        for (cudaEvent_t ev : {le.k0, le.k1, le.g0, le.g1})
            if (ev) cudaEventDestroy(ev);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);   // pending host functions reference h_counter
    if (ctx->upd_scratch) cudaFree(ctx->upd_scratch);
    if (ctx->d_counter) cudaFree(ctx->d_counter);
    if (ctx->h_counter) cudaFreeHost(ctx->h_counter);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int p252_sync(p252_ctx* ctx) {
    if (!ctx) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    CU(cudaStreamSynchronize(ctx->stream));
    return P252_OK;
}

int p252_get_kernel_info(p252_kernel_info* out) {
    if (!out || out->struct_size < sizeof(p252_kernel_info)) return P252_ERR_INVALID_ARGUMENT;
    int t = 0, b = 0;
    p252::kernel_launch_shape(&t, &b);
    out->struct_size = (uint32_t)sizeof(p252_kernel_info);
    out->wide_mul_per_permutation = p252::wide_mul_per_permutation();
    out->dfma_per_permutation = p252::dfma_per_permutation();
    out->montmul_per_permutation = 365;
    out->threads_per_block = (uint32_t)t;
    out->min_blocks_per_sm = (uint32_t)b;
    return P252_OK;
}

int p252_set_small_batch_max(p252_ctx* ctx, size_t max_items) {
    if (!ctx) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    ctx->coop_max = max_items;
    return P252_OK;
}

int p252_debug_fail_chunk(p252_ctx* ctx, long long k) {
    if (!ctx) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    ctx->fail_chunk = k;
    return P252_OK;
}

int p252_debug_staging_nonzero(p252_ctx* ctx, size_t* nonzero_bytes) {
    if (!ctx || !nonzero_bytes) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    size_t bad = 0;
    for (int s = 0; s < kSlots; ++s) {
        Slot& sl = ctx->slots[s];
        if (!sl.arena) continue;
        CU(cudaStreamSynchronize(sl.stream));
        std::vector<uint8_t> h(sl.arena_bytes);
        CU(cudaMemcpy(h.data(), sl.arena, sl.arena_bytes, cudaMemcpyDeviceToHost));
        for (uint8_t v : h) bad += v ? 1 : 0;
    }
    *nonzero_bytes = bad;
    return P252_OK;
}

const char* p252_last_error(const p252_ctx* ctx) { return ctx ? ctx->last_error.c_str() : ""; }
uint64_t p252_launch_count(const p252_ctx* ctx) { return ctx ? ctx->launches : 0; }

int p252_host_alloc(size_t bytes, void** out) {
    if (!out) return P252_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    p252_ctx* ctx = nullptr;
    CU(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
    return P252_OK;
}
int p252_host_free(void* p) {
    p252_ctx* ctx = nullptr;
    if (p) CU(cudaFreeHost(p));
    return P252_OK;
}

// ---- host-side sponge bookkeeping ---------------------------------------------------------------
int p252_domain_separator(int domain, uint64_t* out) {
    bool ok;
    uint64_t v = domain_sep(domain, &ok);
    if (!ok || !out) return P252_ERR_INVALID_ARGUMENT;
    *out = v;
    return P252_OK;
}

int p252_tag_input(const uint32_t* calls, size_t ncalls, uint64_t dsep, uint8_t* out, size_t* out_len) {
    if (!calls || !out_len) return P252_ERR_INVALID_ARGUMENT;
    // a valid io-pattern starts with an absorb, ends with a squeeze and has no zero-length call
    if (ncalls == 0 || !(calls[0] & 0x80000000u) || (calls[ncalls - 1] & 0x80000000u)) return P252_ERR_INVALID_IO_PATTERN;
    std::vector<uint32_t> words;
    for (size_t i = 0; i < ncalls; ++i) {
        if ((calls[i] & 0x7fffffffu) == 0) return P252_ERR_INVALID_IO_PATTERN;
        if (!words.empty() && ((words.back() ^ calls[i]) & 0x80000000u) == 0)
            words.back() += calls[i] & 0x7fffffffu;   // aggregate consecutive calls of one kind
        else
            words.push_back(calls[i]);
    }
    const size_t need = words.size() * 4 + 8;
    if (!out || *out_len < need) {
        *out_len = need;
        return out ? P252_ERR_INVALID_ARGUMENT : P252_OK;
    }
    size_t p = 0;
    for (uint32_t w : words)
        for (int s = 24; s >= 0; s -= 8) out[p++] = (uint8_t)(w >> s);
    for (int s = 56; s >= 0; s -= 8) out[p++] = (uint8_t)(dsep >> s);
    *out_len = need;
    return P252_OK;
}

int p252_hash_to_scalar(const uint8_t* bytes, size_t len, p252_fr* out) {
    if (!out || (!bytes && len)) return P252_ERR_INVALID_ARGUMENT;
    uint8_t digest[64];
    p252::host::blake2b512(bytes, len, digest);
    p252::host::from_bytes_wide(out->l, digest);
    return P252_OK;
}

int p252_tag(const uint32_t* calls, size_t ncalls, uint64_t dsep, p252_fr* tag) {
    if (!tag) return P252_ERR_INVALID_ARGUMENT;
    std::vector<uint8_t> buf(ncalls * 4 + 8 + 8);
    size_t len = buf.size();
    int rc = p252_tag_input(calls, ncalls, dsep, buf.data(), &len);
    if (rc != P252_OK) return rc;
    return p252_hash_to_scalar(buf.data(), len, tag);
}

int p252_hash_tag(int domain, size_t in_len, size_t out_len, p252_fr* tag) {
    bool ok;
    const uint64_t dsep = domain_sep(domain, &ok);
    if (!ok || !tag) return P252_ERR_INVALID_ARGUMENT;
    // io_pattern, src/hash.rs:62-85
    if (domain == P252_DOMAIN_MERKLE2 && (in_len != 2 || out_len != 1)) return P252_ERR_IO_PATTERN_VIOLATION;
    if (domain == P252_DOMAIN_MERKLE4 && (in_len != 4 || out_len != 1)) return P252_ERR_IO_PATTERN_VIOLATION;
    if (in_len == 0 || out_len == 0) return P252_ERR_INVALID_IO_PATTERN;
    if (in_len >= 0x80000000ull || out_len >= 0x80000000ull) return P252_ERR_INVALID_ARGUMENT;
    const uint32_t calls[2] = {0x80000000u | (uint32_t)in_len, (uint32_t)out_len};
    return p252_tag(calls, 2, dsep, tag);
}

int p252_encryption_tag(size_t L, p252_fr* tag) {
    if (!tag) return P252_ERR_INVALID_ARGUMENT;
    if (L == 0) return P252_ERR_INVALID_IO_PATTERN;
    if (L >= 0x7ffffff0ull) return P252_ERR_INVALID_ARGUMENT;
    // [Absorb(2), Absorb(1), Squeeze(L), Absorb(L), Squeeze(1)], src/encryption.rs:67-73
    const uint32_t calls[5] = {0x80000002u, 0x80000001u, (uint32_t)L, 0x80000000u | (uint32_t)L, 1u};
    bool ok;
    return p252_tag(calls, 5, domain_sep(P252_DOMAIN_ENCRYPTION, &ok), tag);
}

// ---- batch entry points ---------------------------------------------------------------------------
static int permute_impl(p252_ctx* ctx, p252_fr* states, size_t n, int flags, bool dense) {
    if (!ctx || (!states && n)) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(states)) return P252_ERR_INVALID_ARGUMENT;
        if (n == 0) return P252_OK;
        return device_call(ctx, flags, nullptr, [&](auto) {
            return count_launch(ctx, p252::launch_permute(states, n, dense, ctx->coop_max, ctx->stream));
        });
    }
    std::vector<Io> ios = {{states, states, 160}};
    return run_host_pipeline(ctx, ios, n, [&](void** d, size_t cnt, cudaStream_t st) {
        return p252::launch_permute(d[0], cnt, dense, ctx->coop_max, st);
    });
}

int p252_permute_batch(p252_ctx* ctx, p252_fr* states, size_t n, int flags) {
    return permute_impl(ctx, states, n, flags, false);
}
int p252_permute_batch_dense(p252_ctx* ctx, p252_fr* states, size_t n, int flags) {
    return permute_impl(ctx, states, n, flags, true);
}

static int digest_impl(p252_ctx* ctx, const p252_fr* tag, const p252_fr* in, size_t n, size_t in_len, p252_fr* out,
                       size_t out_len, int flags, bool truncate) {
    if (!ctx || !tag || ((!in || !out) && n)) return P252_ERR_INVALID_ARGUMENT;
    if (in_len == 0 || out_len == 0) return P252_ERR_INVALID_IO_PATTERN;
    if (in_len > 0x7fffffffull / 32 || out_len > 0x7fffffffull / 32) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    const uint32_t il = (uint32_t)in_len, ol = (uint32_t)out_len;
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(in) || !aligned16(out)) return P252_ERR_INVALID_ARGUMENT;
        if (n == 0) return P252_OK;
        return device_call(ctx, flags, nullptr, [&](auto) {
            return count_launch(ctx, p252::launch_digest(limbs(tag), in, n, il, out, ol, truncate, ctx->coop_max, ctx->stream));
        });
    }
    std::vector<Io> ios = {{in, nullptr, in_len * 32}, {nullptr, out, out_len * 32}};
    return run_host_pipeline(ctx, ios, n, [&](void** d, size_t cnt, cudaStream_t st) {
        return p252::launch_digest(limbs(tag), d[0], cnt, il, d[1], ol, truncate, ctx->coop_max, st);
    });
}

int p252_digest_batch(p252_ctx* ctx, const p252_fr* tag, const p252_fr* in, size_t n, size_t in_len, p252_fr* out,
                      size_t out_len, int flags) {
    return digest_impl(ctx, tag, in, n, in_len, out, out_len, flags, false);
}

int p252_hash_batch(p252_ctx* ctx, int domain, const p252_fr* in, size_t n, size_t in_len, p252_fr* out,
                    size_t out_len, int flags) {
    p252_fr tag;
    int rc = p252_hash_tag(domain, in_len, out_len, &tag);
    if (rc != P252_OK) return rc;
    return digest_impl(ctx, &tag, in, n, in_len, out, out_len, flags, false);
}

int p252_hash_batch_truncated(p252_ctx* ctx, int domain, const p252_fr* in, size_t n, size_t in_len, p252_fr* out_raw,
                              size_t out_len, int flags) {
    p252_fr tag;
    int rc = p252_hash_tag(domain, in_len, out_len, &tag);
    if (rc != P252_OK) return rc;
    return digest_impl(ctx, &tag, in, n, in_len, out_raw, out_len, flags, true);
}

static int convert_impl(p252_ctx* ctx, const void* in, size_t n, void* out, uint8_t* ok, int flags, bool from_bytes) {
    if (!ctx || ((!in || !out) && n)) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(in) || !aligned16(out)) return P252_ERR_INVALID_ARGUMENT;
        if (n == 0) return P252_OK;
        return device_call(ctx, flags, nullptr, [&](auto) {
            return count_launch(ctx, p252::launch_convert(in, n, out, ok, from_bytes, ctx->stream));
        });
    }
    std::vector<Io> ios = {{in, nullptr, 32}, {nullptr, out, 32}};
    if (from_bytes && ok) ios.push_back({nullptr, ok, 1});
    return run_host_pipeline(ctx, ios, n, [&](void** d, size_t cnt, cudaStream_t st) {
        return p252::launch_convert(d[0], cnt, d[1], (from_bytes && ok) ? static_cast<uint8_t*>(d[2]) : nullptr, from_bytes, st);
    });
}

int p252_scalars_from_bytes(p252_ctx* ctx, const uint8_t* bytes, size_t n, p252_fr* out, uint8_t* ok, int flags) {
    return convert_impl(ctx, bytes, n, out, ok, flags, true);
}

int p252_scalars_to_bytes(p252_ctx* ctx, const p252_fr* in, size_t n, uint8_t* bytes, int flags) {
    return convert_impl(ctx, in, n, bytes, nullptr, flags, false);
}

int p252_encrypt_batch(p252_ctx* ctx, const p252_fr* msg, size_t n, size_t L, const p252_fr* secret_uv,
                       const p252_fr* nonce, p252_fr* cipher, int flags) {
    if (!ctx || ((!msg || !secret_uv || !nonce || !cipher) && n)) return P252_ERR_INVALID_ARGUMENT;
    p252_fr tag;
    int rc = p252_encryption_tag(L, &tag);
    if (rc != P252_OK) return rc;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    const uint32_t l32 = (uint32_t)L;
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(msg) || !aligned16(secret_uv) || !aligned16(nonce) || !aligned16(cipher))
            return P252_ERR_INVALID_ARGUMENT;
        if (n == 0) return P252_OK;
        return device_call(ctx, flags, nullptr, [&](auto) {
            return count_launch(ctx, p252::launch_encrypt(limbs(&tag), msg, n, l32, secret_uv, nonce, cipher, ctx->stream));
        });
    }
    std::vector<Io> ios = {{msg, nullptr, L * 32}, {secret_uv, nullptr, 64}, {nonce, nullptr, 32},
                           {nullptr, cipher, (L + 1) * 32}};
    return run_host_pipeline(ctx, ios, n, [&](void** d, size_t cnt, cudaStream_t st) {
        return p252::launch_encrypt(limbs(&tag), d[0], cnt, l32, d[1], d[2], d[3], st);
    }, /*wipe=*/true);
}

int p252_decrypt_batch(p252_ctx* ctx, const p252_fr* cipher, size_t n, size_t L, const p252_fr* secret_uv,
                       const p252_fr* nonce, p252_fr* msg, uint8_t* ok, size_t* n_failed, int flags) {
    if (!ctx || ((!cipher || !secret_uv || !nonce || !msg || !ok) && n)) return P252_ERR_INVALID_ARGUMENT;
    p252_fr tag;
    int rc = p252_encryption_tag(L, &tag);
    if (rc != P252_OK) return rc;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    const uint32_t l32 = (uint32_t)L;
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(cipher) || !aligned16(secret_uv) || !aligned16(nonce) || !aligned16(msg))
            return P252_ERR_INVALID_ARGUMENT;
        if (n_failed) *n_failed = 0;
        if (n == 0) return P252_OK;
        return device_call(ctx, flags, n_failed, [&](unsigned long long* failed) {
            return count_launch(ctx, p252::launch_decrypt(limbs(&tag), cipher, n, l32, secret_uv, nonce, msg, ok, failed,
                                                          ctx->stream));
        });
    }
    std::vector<Io> ios = {{cipher, nullptr, (L + 1) * 32}, {secret_uv, nullptr, 64}, {nonce, nullptr, 32},
                           {nullptr, msg, L * 32}, {nullptr, ok, 1}};
    rc = run_host_pipeline(ctx, ios, n, [&](void** d, size_t cnt, cudaStream_t st) {
        return p252::launch_decrypt(limbs(&tag), d[0], cnt, l32, d[1], d[2], d[3], static_cast<uint8_t*>(d[4]), nullptr, st);
    }, /*wipe=*/true);
    return count_failed(rc, ok, n, n_failed);
}

// ---- arity-4 Merkle tree ------------------------------------------------------------------------------
int p252_merkle4_level(p252_ctx* ctx, const p252_fr* children, size_t n_parents, p252_fr* parents, int flags) {
    return p252_hash_batch(ctx, P252_DOMAIN_MERKLE4, children, n_parents, 4, parents, 1, flags);
}

int p252_merkle_tree_nodes(int arity, size_t n_leaves, size_t* n_internal, int* n_levels) {
    Tree t;
    int rc = make_tree(arity, n_leaves, &t);
    if (rc != P252_OK) return rc;
    if (n_internal) *n_internal = t.n_internal;
    if (n_levels) *n_levels = t.depth;
    return P252_OK;
}

int p252_merkle4_tree_nodes(size_t n_leaves, size_t* n_internal, int* n_levels) {
    return p252_merkle_tree_nodes(4, n_leaves, n_internal, n_levels);
}

// Heights from+1 .. depth, one launch each, reading height `from` where t.level(leaves, nodes, from) points.
static int merkle_build_levels(p252_ctx* ctx, const Tree& t, const p252_fr* leaves, p252_fr* nodes, int from) {
    for (int h = from + 1; h <= t.depth; ++h) {
        int rc = count_launch(ctx, p252::launch_digest(limbs(&t.tag), t.level<const p252_fr>(leaves, nodes, h - 1), t.size(h),
                                                       (uint32_t)t.arity, nodes + t.offset(h), 1, false, ctx->coop_max,
                                                       ctx->stream));
        if (rc != P252_OK) return rc;
    }
    return P252_OK;
}

int p252_merkle_build(p252_ctx* ctx, int arity, const p252_fr* leaves, size_t n_leaves, p252_fr* nodes_out, int flags) {
    if (!ctx || !leaves || !nodes_out) return P252_ERR_INVALID_ARGUMENT;
    Tree t;
    int rc = make_tree(arity, n_leaves, &t);
    if (rc != P252_OK) return rc;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(leaves) || !aligned16(nodes_out)) return P252_ERR_INVALID_ARGUMENT;
        return device_call(ctx, flags, nullptr, [&](auto) { return merkle_build_levels(ctx, t, leaves, nodes_out, 0); });
    }
    // HOST: height 1 (the largest level) streams through the chunked pipeline straight from the host leaves; the
    // heights above run on the device-resident internal nodes.
    const size_t first = t.size(1);
    p252_fr* d_nodes = nullptr;
    CU(cudaMalloc(reinterpret_cast<void**>(&d_nodes), t.n_internal * sizeof(p252_fr)));
    {
        std::vector<Io> ios = {{leaves, nullptr, (size_t)arity * 32}, {nullptr, nodes_out, 32}};
        size_t done = 0;   // the pipeline hands chunks in order; mirror each chunk into d_nodes as well
        rc = run_host_pipeline(ctx, ios, first, [&](void** d, size_t cnt, cudaStream_t st) {
            cudaError_t e = p252::launch_digest(limbs(&t.tag), d[0], cnt, (uint32_t)arity, d[1], 1, false, ctx->coop_max, st);
            if (e != cudaSuccess) return e;
            e = cudaMemcpyAsync(d_nodes + done, d[1], cnt * sizeof(p252_fr), cudaMemcpyDeviceToDevice, st);
            done += cnt;
            return e;
        });
    }
    if (rc == P252_OK && t.depth > 1) {
        rc = merkle_build_levels(ctx, t, nullptr, d_nodes, 1);
        if (rc == P252_OK) {
            cudaError_t e = cudaMemcpyAsync(nodes_out + first, d_nodes + first, (t.n_internal - first) * sizeof(p252_fr),
                                            cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = fail_cuda(ctx, e, "merkle D2H");
        }
    }
    cudaFree(d_nodes);
    return rc;
}

int p252_merkle4_build(p252_ctx* ctx, const p252_fr* leaves, size_t n_leaves, p252_fr* nodes_out, int flags) {
    return p252_merkle_build(ctx, 4, leaves, n_leaves, nodes_out, flags);
}

// ---- Merkle openings ----------------------------------------------------------------------------------------
int p252_merkle_open_batch(p252_ctx* ctx, int arity, const p252_fr* leaves, size_t n_leaves, const p252_fr* nodes,
                           const uint64_t* leaf_idx, size_t n, p252_fr* paths_out, int flags) {
    if (!ctx || !leaves || !nodes || ((!leaf_idx || !paths_out) && n)) return P252_ERR_INVALID_ARGUMENT;
    Tree t;
    int rc = make_tree(arity, n_leaves, &t);
    if (rc != P252_OK) return rc;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(leaves) || !aligned16(nodes) || !aligned16(paths_out) || (reinterpret_cast<uintptr_t>(leaf_idx) & 7))
            return P252_ERR_INVALID_ARGUMENT;
        if (n == 0) return P252_OK;
        return device_call(ctx, flags, nullptr, [&](auto) {
            return count_launch(ctx, p252::launch_merkle_open(leaves, nodes, leaf_idx, n, arity, (uint32_t)t.depth, n_leaves,
                                                              paths_out, ctx->stream));
        });
    }
    // HOST tree: an opening is a pure gather of 32-byte items the caller already holds in host memory -- shipping
    // the whole tree to the GPU to copy depth*arity scalars back would only add PCIe traffic.  No hashing happens here.
    for (size_t i = 0; i < n; ++i)
        if (leaf_idx[i] >= n_leaves) return P252_ERR_INVALID_ARGUMENT;
    const size_t A = (size_t)arity;
    for (size_t i = 0; i < n; ++i) {
        uint64_t grp = leaf_idx[i];
        for (int h = 0; h < t.depth; ++h) {
            grp >>= t.log2_arity;   // the group of the path node at height h
            memcpy(paths_out + (i * (size_t)t.depth + (size_t)h) * A, t.group(leaves, nodes, h, grp), A * sizeof(p252_fr));
        }
    }
    return P252_OK;
}

int p252_merkle_verify_batch(p252_ctx* ctx, int arity, int depth, const p252_fr* leaf_items, const uint64_t* leaf_idx,
                             const p252_fr* paths, const p252_fr* root, size_t n, uint8_t* ok, size_t* n_failed,
                             int flags) {
    if (!ctx || !root || ((!leaf_items || !leaf_idx || !paths || !ok) && n)) return P252_ERR_INVALID_ARGUMENT;
    if (depth < 1 || depth > p252::kMaxDepth) return P252_ERR_INVALID_ARGUMENT;
    p252_fr tag;
    int rc = merkle_tag(arity, &tag);
    if (rc != P252_OK) return rc;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    if (n_failed) *n_failed = 0;
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(leaf_items) || !aligned16(paths) || (reinterpret_cast<uintptr_t>(leaf_idx) & 7))
            return P252_ERR_INVALID_ARGUMENT;
        if (n == 0) return P252_OK;
        return device_call(ctx, flags, n_failed, [&](unsigned long long* failed) {
            return count_launch(ctx, p252::launch_merkle_verify(limbs(&tag), limbs(root), leaf_items, leaf_idx, paths, n, arity,
                                                                (uint32_t)depth, ok, failed, ctx->stream));
        });
    }
    const size_t path_bytes = (size_t)depth * (size_t)arity * 32;
    std::vector<Io> ios = {{leaf_items, nullptr, 32}, {leaf_idx, nullptr, 8}, {paths, nullptr, path_bytes}, {nullptr, ok, 1}};
    rc = run_host_pipeline(ctx, ios, n, [&](void** d, size_t cnt, cudaStream_t st) {
        return p252::launch_merkle_verify(limbs(&tag), limbs(root), d[0], static_cast<const uint64_t*>(d[1]), d[2], cnt, arity,
                                          (uint32_t)depth, static_cast<uint8_t*>(d[3]), nullptr, st);
    });
    return count_failed(rc, ok, n, n_failed);
}

// ---- incremental Merkle updates ---------------------------------------------------------------------------------
// The context's update scratch grows on demand and is never shrunk, so a repeat call with the same or a smaller batch
// allocates nothing (and a P252_ASYNC call stays asynchronous).
static int update_scratch(p252_ctx* ctx, size_t bytes, void** out) {
    if (ctx->upd_scratch_bytes < bytes) {
        if (ctx->upd_scratch) {
            CU(cudaStreamSynchronize(ctx->stream));      // earlier calls may still use it
            CU(cudaFree(ctx->upd_scratch));
            ctx->upd_scratch = nullptr;
            ctx->upd_scratch_bytes = 0;
        }
        CU(cudaMalloc(&ctx->upd_scratch, bytes));
        ctx->upd_scratch_bytes = bytes;
    }
    *out = ctx->upd_scratch;
    return P252_OK;
}

// DEVICE: everything is enqueued on the context stream -- planning (p252::launch_merkle_update_plan) and then one
// hash launch per level, sized by min(k, level size); each kernel reads its level's real list length on the device.
static int merkle_update_device(p252_ctx* ctx, const Tree& t, p252_fr* leaves, p252_fr* nodes, const uint64_t* leaf_idx,
                                const p252_fr* values, size_t k, size_t* n_rejected, int flags) {
    const uint32_t depth = (uint32_t)t.depth;
    p252::MerkleUpdatePlan plan = p252::merkle_update_layout(nullptr, k, t.log2_arity, depth, t.n_leaves);
    void* scratch = nullptr;
    int rc = update_scratch(ctx, plan.total_bytes, &scratch);
    if (rc != P252_OK) return rc;
    plan = p252::merkle_update_layout(scratch, k, t.log2_arity, depth, t.n_leaves);
    return device_call(ctx, flags, n_rejected, [&](unsigned long long* rejected) {
        int st = count_launch(ctx, p252::launch_merkle_update_plan(plan, leaf_idx, values, k, t.log2_arity, depth, t.n_leaves,
                                                                   leaves, rejected, ctx->stream),
                              "merkle update plan", 2);
        for (int h = 1; h <= t.depth && st == P252_OK; ++h)   // plan.lists[h - 1]: the dirty nodes of height h
            st = count_launch(ctx, p252::launch_merkle_update(limbs(&t.tag), t.arity, t.level(leaves, nodes, h - 1),
                                                              plan.lists[h - 1], plan.lists[h - 1], t.level(leaves, nodes, h),
                                                              std::min(k, t.size(h)), plan.counts + h - 1, t.size(h),
                                                              ctx->coop_max, ctx->stream));
        return st;
    });
}

// HOST: only the dirty paths travel.  The children groups of every dirty parent are staged with one H2D (level 1:
// leaves with the new values applied; above: the current nodes, whose dirty entries the level below overwrites on the
// device), every level's kernel writes its parents into their slots among the next level's staged groups (the top
// level into a one-slot buffer), one D2H brings the groups back, and only then are the caller's arrays written.
static int merkle_update_host(p252_ctx* ctx, const Tree& t, p252_fr* leaves, p252_fr* nodes, const uint64_t* leaf_idx,
                              const p252_fr* values, size_t k) {
    const int depth = t.depth, s = t.log2_arity;
    const size_t A = (size_t)t.arity;
    // dedupe: stable order by index, the last occurrence of an index wins
    std::vector<uint32_t> ord(k);
    for (size_t i = 0; i < k; ++i) ord[i] = (uint32_t)i;
    std::stable_sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return leaf_idx[a] < leaf_idx[b]; });
    std::vector<uint32_t> upd;   // batch positions of the surviving writes, by increasing leaf index
    for (size_t j = 0; j < k; ++j)
        if (j + 1 == k || leaf_idx[ord[j + 1]] != leaf_idx[ord[j]]) upd.push_back(ord[j]);
    // dirty parents per level: list[l] = unique(list[l-1] >> log2(arity)), list[0] = the updated leaves
    std::vector<std::vector<uint64_t>> list((size_t)depth + 1);
    for (uint32_t u : upd) list[0].push_back(leaf_idx[u]);
    for (int l = 1; l <= depth; ++l)
        for (uint64_t c : list[(size_t)l - 1])
            if (list[(size_t)l].empty() || list[(size_t)l].back() != (c >> s)) list[(size_t)l].push_back(c >> s);
    // staging layout (scalars): region[l] = |list[l]| groups of `arity` children for l = 1..depth, then the root slot;
    // then the write-slot indices of every level (u64)
    std::vector<size_t> region((size_t)depth + 2, 0), widx_off((size_t)depth + 2, 0);
    for (int l = 1; l <= depth; ++l) {
        region[(size_t)l + 1] = region[(size_t)l] + list[(size_t)l].size() * A;
        widx_off[(size_t)l + 1] = widx_off[(size_t)l] + list[(size_t)l].size();
    }
    const size_t n_stage = region[(size_t)depth + 1] + 1, n_widx = widx_off[(size_t)depth + 1];
    const size_t stage_bytes = n_stage * sizeof(p252_fr);
    std::vector<p252_fr> stage(n_stage);
    std::vector<uint64_t> widx(n_widx);
    for (int l = 1; l <= depth; ++l) {
        const std::vector<uint64_t>& L = list[(size_t)l];
        for (size_t j = 0; j < L.size(); ++j)
            memcpy(&stage[region[(size_t)l] + j * A], t.group(leaves, nodes, l - 1, L[j]), A * sizeof(p252_fr));
        if (l == depth) {
            widx[widx_off[(size_t)l]] = 0;
            continue;
        }
        const std::vector<uint64_t>& up = list[(size_t)l + 1];
        for (size_t j = 0, r = 0; j < L.size(); ++j) {
            while (up[r] != (L[j] >> s)) ++r;
            widx[widx_off[(size_t)l] + j] = r * A + (L[j] & (A - 1));
        }
    }
    for (size_t j = 0, r = 0; j < upd.size(); ++j) {   // the new leaf values
        const uint64_t i = leaf_idx[upd[j]];
        while (list[1][r] != (i >> s)) ++r;
        stage[region[1] + r * A + (i & (A - 1))] = values[upd[j]];
    }
    std::vector<uint8_t> h(stage_bytes + n_widx * 8);
    memcpy(h.data(), stage.data(), stage_bytes);
    memcpy(h.data() + stage_bytes, widx.data(), n_widx * 8);
    void* scratch = nullptr;
    int rc = update_scratch(ctx, h.size(), &scratch);
    if (rc != P252_OK) return rc;
    p252_fr* d_stage = static_cast<p252_fr*>(scratch);
    const uint64_t* d_widx = reinterpret_cast<const uint64_t*>(static_cast<uint8_t*>(scratch) + stage_bytes);
    auto body = [&]() -> int {
        CU(cudaMemcpyAsync(scratch, h.data(), h.size(), cudaMemcpyHostToDevice, ctx->stream));
        for (int l = 1; l <= depth; ++l) {
            const size_t n = list[(size_t)l].size();
            p252_fr* out = d_stage + region[(size_t)l + 1];   // the next level's groups, or the root slot
            int st = count_launch(ctx, p252::launch_merkle_update(limbs(&t.tag), t.arity, d_stage + region[(size_t)l], nullptr,
                                                                  d_widx + widx_off[(size_t)l], out, n, nullptr, n,
                                                                  ctx->coop_max, ctx->stream));
            if (st != P252_OK) return st;
        }
        CU(cudaMemcpyAsync(stage.data() + region[2], d_stage + region[2], (n_stage - region[2]) * sizeof(p252_fr),
                           cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        return P252_OK;
    };
    rc = body();
    if (rc != P252_OK) {
        cudaStreamSynchronize(ctx->stream);   // nothing may still read or write the staging vectors
        cudaGetLastError();
        return rc;
    }
    // all device work succeeded: write the caller's tree
    for (int l = 1; l < depth; ++l) {
        const std::vector<uint64_t>& L = list[(size_t)l];
        for (size_t j = 0; j < L.size(); ++j)
            t.level(leaves, nodes, l)[L[j]] = stage[region[(size_t)l + 1] + widx[widx_off[(size_t)l] + j]];
    }
    *t.level(leaves, nodes, depth) = stage[region[(size_t)depth + 1]];
    for (uint32_t u : upd) leaves[leaf_idx[u]] = values[u];
    return P252_OK;
}

int p252_merkle_update_batch(p252_ctx* ctx, int arity, p252_fr* leaves, size_t n_leaves, p252_fr* nodes,
                             const uint64_t* leaf_idx, const p252_fr* values, size_t k, size_t* n_rejected, int flags) {
    if (!ctx || !leaves || !nodes || ((!leaf_idx || !values) && k)) return P252_ERR_INVALID_ARGUMENT;
    Tree t;
    int rc = make_tree(arity, n_leaves, &t);
    if (rc != P252_OK) return rc;
    if (k > 0xffffffffull) return P252_ERR_INVALID_ARGUMENT;   // batch positions are 32-bit
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    if (n_rejected) *n_rejected = 0;
    if (flags & P252_MEM_DEVICE) {
        if (!aligned16(leaves) || !aligned16(nodes) || !aligned16(values) || (reinterpret_cast<uintptr_t>(leaf_idx) & 7))
            return P252_ERR_INVALID_ARGUMENT;
        if (k == 0) return P252_OK;
        return merkle_update_device(ctx, t, leaves, nodes, leaf_idx, values, k, n_rejected, flags);
    }
    for (size_t i = 0; i < k; ++i)
        if (leaf_idx[i] >= n_leaves) return P252_ERR_INVALID_ARGUMENT;   // before anything is written
    if (k == 0) return P252_OK;
    return merkle_update_host(ctx, t, leaves, nodes, leaf_idx, values, k);
}

// ---- multi-GPU ------------------------------------------------------------------------------------------
int p252_dist_unique_id(uint8_t id[P252_NCCL_UNIQUE_ID_BYTES]) {
    static_assert(sizeof(ncclUniqueId) <= P252_NCCL_UNIQUE_ID_BYTES, "unique id size");
    p252_ctx* ctx = nullptr;
    if (!id) return P252_ERR_INVALID_ARGUMENT;
    if (!nccl().ok) return fail_nccl(ctx, ncclSystemError, "dlopen(libnccl.so.2)");
    ncclUniqueId u;
    NC(nccl().GetUniqueId(&u));
    memset(id, 0, P252_NCCL_UNIQUE_ID_BYTES);
    memcpy(id, &u, sizeof u);
    return P252_OK;
}

int p252_dist_init(p252_ctx* ctx, const uint8_t id[P252_NCCL_UNIQUE_ID_BYTES], int rank, int nranks) {
    if (!ctx || !id || nranks < 1 || rank < 0 || rank >= nranks) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    if (ctx->comm) return P252_ERR_INVALID_ARGUMENT;
    DeviceGuard g(ctx->device);
    if (!nccl().ok) return fail_nccl(ctx, ncclSystemError, "dlopen(libnccl.so.2)");
    ncclUniqueId u;
    memcpy(&u, id, sizeof u);
    NC(nccl().CommInitRank(&ctx->comm, nranks, u, rank));
    ctx->rank = rank;
    ctx->nranks = nranks;
    CU(cudaStreamCreateWithFlags(&ctx->comm_stream, cudaStreamNonBlocking));
    return P252_OK;
}

int p252_dist_finalize(p252_ctx* ctx) {
    if (!ctx) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    if (ctx->comm) {
        CU(cudaStreamSynchronize(ctx->comm_stream));
        NC(nccl().CommDestroy(ctx->comm));
        ctx->comm = nullptr;
    }
    if (ctx->comm_stream) {
        cudaStreamDestroy(ctx->comm_stream);
        ctx->comm_stream = nullptr;
    }
    ctx->rank = 0;
    ctx->nranks = 1;
    return P252_OK;
}

// Contiguous sharding: rank r owns nodes [r*M/G, (r+1)*M/G) of every level with M % G == 0 nodes, whose
// children are exactly rank r's slice of the level below -- so the compute stream climbs its own
// subtree without waiting, while the all-gather of each finished level (the level's replication to
// all GPUs over NVLink) runs on a second stream.  Smaller levels are computed redundantly by every
// rank from the gathered level below.
int p252_merkle4_shard_plan(size_t n_leaves_total, int nranks, int rank, p252_level_plan* levels, int capacity,
                            int* n_levels) {
    if (nranks < 1 || rank < 0 || rank >= nranks) return P252_ERR_INVALID_ARGUMENT;
    Tree t;
    int rc = make_tree(4, n_leaves_total, &t);
    if (rc != P252_OK) return rc;
    if (n_leaves_total % (size_t)nranks || (n_leaves_total / nranks) % 4) return P252_ERR_INVALID_ARGUMENT;
    if (n_levels) *n_levels = t.depth;
    if (!levels) return P252_OK;
    if (capacity < t.depth) return P252_ERR_INVALID_ARGUMENT;
    for (int h = 1; h <= t.depth; ++h) {
        p252_level_plan& p = levels[h - 1];
        p.level_offset = t.offset(h);
        p.level_size = t.size(h);
        p.sharded = (p.level_size % (uint64_t)nranks == 0) ? 1 : 0;
        p.my_count = p.sharded ? p.level_size / nranks : p.level_size;
        p.my_offset = p.sharded ? (uint64_t)rank * p.my_count : 0;
        p.reserved = 0;
    }
    return P252_OK;
}

int p252_merkle4_build_dist(p252_ctx* ctx, const p252_fr* leaves_shard, size_t n_leaves_total, p252_fr* nodes_out,
                            int flags) {
    if (!ctx || !leaves_shard || !nodes_out) return P252_ERR_INVALID_ARGUMENT;
    if (!(flags & P252_MEM_DEVICE)) return P252_ERR_INVALID_ARGUMENT;   // shards live on the GPU
    if (!aligned16(leaves_shard) || !aligned16(nodes_out)) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    const int G = ctx->nranks, r = ctx->rank;
    if (G > 1 && !ctx->comm) return P252_ERR_INVALID_ARGUMENT;
    p252_level_plan plan[p252::kMaxDepth];
    int lv = 0;
    int rc = p252_merkle4_shard_plan(n_leaves_total, G, r, plan, p252::kMaxDepth, &lv);
    if (rc != P252_OK) return rc;
    p252_fr tag;
    if ((rc = merkle_tag(4, &tag)) != P252_OK) return rc;
    DeviceGuard g(ctx->device);

    const bool timing = (flags & P252_TIMING) != 0;
    const bool no_gather = (flags & P252_NO_GATHER) != 0;
    if (timing) {
        // events with timing enabled, created once per context and reused
        while ((int)ctx->level_events.size() < lv) {
            p252_ctx::LevelEvents le;
            for (cudaEvent_t* ev : {&le.k0, &le.k1, &le.g0, &le.g1}) CU(cudaEventCreate(ev));
            ctx->level_events.push_back(le);
        }
        ctx->level_info.assign((size_t)lv, p252_level_timing{});
        ctx->level_gathered.assign((size_t)lv, 0);
    }
    ctx->timed_levels = timing ? lv : 0;

    const p252_fr* below_full = nullptr;        // complete level below (valid once gathered)
    const p252_fr* below_mine = leaves_shard;   // this rank's slice of the level below
    bool gather_in_flight = false;
    CU(cudaEventRecord(ctx->ev_comm, ctx->stream));
    for (int l = 0; l < lv; ++l) {
        const p252_level_plan& p = plan[l];
        p252_fr* level = nodes_out + p.level_offset;
        if (timing) {
            ctx->level_info[(size_t)l].nodes = p.level_size;
            ctx->level_info[(size_t)l].my_nodes = p.my_count;
        }
        if (p.sharded) {
            // the first level is always sharded (n_leaves_total / G is a multiple of 4)
            if (timing) CU(cudaEventRecord(ctx->level_events[(size_t)l].k0, ctx->stream));
            rc = count_launch(ctx, p252::launch_digest(limbs(&tag), below_mine, p.my_count, 4, level + p.my_offset, 1, false,
                                                       ctx->coop_max, ctx->stream));
            if (rc != P252_OK) return rc;
            if (timing) CU(cudaEventRecord(ctx->level_events[(size_t)l].k1, ctx->stream));
            if (G > 1 && !no_gather) {
                CU(cudaEventRecord(ctx->ev_level, ctx->stream));
                CU(cudaStreamWaitEvent(ctx->comm_stream, ctx->ev_level, 0));
                if (timing) CU(cudaEventRecord(ctx->level_events[(size_t)l].g0, ctx->comm_stream));
                NC(nccl().AllGather(level + p.my_offset, level, p.my_count * 4, ncclUint64, ctx->comm, ctx->comm_stream));
                if (timing) {
                    CU(cudaEventRecord(ctx->level_events[(size_t)l].g1, ctx->comm_stream));
                    ctx->level_gathered[(size_t)l] = 1;
                    ctx->level_info[(size_t)l].gather_bytes = p.level_size * sizeof(p252_fr);
                }
                CU(cudaEventRecord(ctx->ev_comm, ctx->comm_stream));
                gather_in_flight = true;
            }
            below_mine = level + p.my_offset;
        } else {
            if (gather_in_flight) {   // needs the complete level below on this rank
                CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_comm, 0));
                gather_in_flight = false;
            }
            if (timing) CU(cudaEventRecord(ctx->level_events[(size_t)l].k0, ctx->stream));
            rc = count_launch(ctx, p252::launch_digest(limbs(&tag), below_full, p.level_size, 4, level, 1, false, ctx->coop_max,
                                                       ctx->stream));
            if (rc != P252_OK) return rc;
            if (timing) CU(cudaEventRecord(ctx->level_events[(size_t)l].k1, ctx->stream));
        }
        below_full = level;
    }
    // every level must be complete on every rank before the call is considered done
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_comm, 0));
    if (timing) CU(cudaEventRecord(ctx->ev_tree_end, ctx->stream));
    if (!(flags & P252_ASYNC)) CU(cudaStreamSynchronize(ctx->stream));
    return P252_OK;
}

int p252_tree_level_timings(p252_ctx* ctx, p252_level_timing* levels, int capacity, int* n_levels, float* total_ms) {
    if (!ctx) return P252_ERR_INVALID_ARGUMENT;
    P252_LOCK(ctx);
    DeviceGuard g(ctx->device);
    const int lv = ctx->timed_levels;
    if (n_levels) *n_levels = lv;
    if (lv == 0) return P252_ERR_INVALID_ARGUMENT;   // no P252_TIMING build on this context yet
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->comm_stream) CU(cudaStreamSynchronize(ctx->comm_stream));
    if (total_ms) CU(cudaEventElapsedTime(total_ms, ctx->level_events[0].k0, ctx->ev_tree_end));
    if (!levels) return P252_OK;
    if (capacity < lv) return P252_ERR_INVALID_ARGUMENT;
    for (int l = 0; l < lv; ++l) {
        p252_level_timing t = ctx->level_info[(size_t)l];
        CU(cudaEventElapsedTime(&t.kernel_ms, ctx->level_events[(size_t)l].k0, ctx->level_events[(size_t)l].k1));
        t.gather_ms = 0.f;
        if (ctx->level_gathered[(size_t)l])
            CU(cudaEventElapsedTime(&t.gather_ms, ctx->level_events[(size_t)l].g0, ctx->level_events[(size_t)l].g1));
        levels[l] = t;
    }
    return P252_OK;
}

}  // extern "C"
