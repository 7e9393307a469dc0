// poseidon252_b200.hpp -- header-only C++17 host mirror of the dusk_poseidon public surface
// (/root/reference/src/lib.rs:13-31) above the C ABI of poseidon252_b200.h.  The reference is compiled
// (Rust) code and no Rust toolchain exists in this image, so the compiled host side is C++; the Rust
// binding a maintainer would add is shown in INTEGRATION.md / bindings/rust/.
//
//   dusk_poseidon::Domain                    -> p252::Domain
//   dusk_poseidon::Hash{new,output_len,update,finalize,digest}   (src/hash.rs:92-195)  -> p252::Hash
//   dusk_poseidon::{encrypt, decrypt}        (src/encryption.rs:62-95) -> p252::encrypt / p252::decrypt
//   dusk_poseidon::Error                     (src/error.rs:11-32)      -> p252::Error (exception)
//   NEW batch entries: Hash::digest_batch, hades::permute_batch, encrypt_batch, decrypt_batch,
//   merkle4_build.
// Scalars are p252_fr == BlsScalar.0 (Montgomery limbs); every digest runs on the GPU (batch of 1 for the
// single-item calls).  No CPU fallback: Engine's constructor throws without an sm_100 device.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "poseidon252_b200.h"

namespace p252 {

using Scalar = p252_fr;

enum class Domain : int {   // src/hash.rs:21-36
    Merkle4 = P252_DOMAIN_MERKLE4,
    Merkle2 = P252_DOMAIN_MERKLE2,
    Encryption = P252_DOMAIN_ENCRYPTION,
    Other = P252_DOMAIN_OTHER,
};

// src/error.rs:11-32 -- `code` is the p252_status (positive = dusk_poseidon::Error variant)
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
    bool is_io_pattern_violation() const { return code == P252_ERR_IO_PATTERN_VIOLATION; }
    bool is_decryption_failed() const { return code == P252_ERR_DECRYPTION_FAILED; }
};

inline void check(int rc, const p252_ctx* ctx = nullptr) {
    if (rc == P252_OK) return;
    std::string msg = p252_strerror(rc);
    if (ctx && *p252_last_error(ctx)) msg += std::string(" (") + p252_last_error(ctx) + ")";
    throw Error(rc, msg);
}

// u64::from(Domain), src/hash.rs:38-56
inline uint64_t domain_separator(Domain d) {
    uint64_t v = 0;
    check(p252_domain_separator(static_cast<int>(d), &v));
    return v;
}

class Engine {
public:
    explicit Engine(int device = 0, void* cuda_stream = nullptr) {
        check(cuda_stream ? p252_create_on_stream(device, cuda_stream, &ctx_) : p252_create(device, &ctx_));
    }
    ~Engine() { p252_destroy(ctx_); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    p252_ctx* get() const { return ctx_; }
    void sync() { check(p252_sync(ctx_), ctx_); }
    uint64_t launch_count() const { return p252_launch_count(ctx_); }

    static Engine& default_engine() {
        static Engine e(0);
        return e;
    }

private:
    p252_ctx* ctx_ = nullptr;
};

namespace hades {
constexpr int WIDTH = P252_WIDTH;   // src/hades.rs:34

// n independent Safe::permute calls (src/hades/permutation/scalar.rs:25-27); states: n x 5, in place
inline void permute_batch(std::vector<Scalar>& states, Engine& e = Engine::default_engine()) {
    if (states.size() % WIDTH) throw Error(P252_ERR_INVALID_ARGUMENT, "states must hold n x 5 scalars");
    check(p252_permute_batch(e.get(), states.data(), states.size() / WIDTH, P252_MEM_HOST), e.get());
}
}  // namespace hades

class Hash {   // src/hash.rs:92-96
public:
    explicit Hash(Domain domain, Engine* e = nullptr) : domain_(domain), engine_(e) {}

    // src/hash.rs:111-115
    void output_len(size_t n) {
        if (domain_ == Domain::Other && n > 0) output_len_ = n;
    }
    // src/hash.rs:118-120 (the reference borrows the slice; this mirror borrows pointer + length)
    void update(const Scalar* input, size_t len) { chunks_.push_back({input, len}); }
    void update(const std::vector<Scalar>& input) { update(input.data(), input.size()); }

    // src/hash.rs:128-155.  Throws Error where the reference panics on an invalid io-pattern.
    std::vector<Scalar> finalize() const {
        // io_pattern, src/hash.rs:62-85: one Absorb per chunk + Squeeze(output_len)
        std::vector<uint32_t> calls;
        std::vector<Scalar> all;
        size_t total = 0;
        for (auto& c : chunks_) {
            calls.push_back(0x80000000u | static_cast<uint32_t>(c.len));
            all.insert(all.end(), c.ptr, c.ptr + c.len);
            total += c.len;
        }
        calls.push_back(static_cast<uint32_t>(output_len_));
        if ((domain_ == Domain::Merkle2 && (total != 2 || output_len_ != 1)) ||
            (domain_ == Domain::Merkle4 && (total != 4 || output_len_ != 1)))
            throw Error(P252_ERR_IO_PATTERN_VIOLATION, p252_strerror(P252_ERR_IO_PATTERN_VIOLATION));
        Scalar tag;
        check(p252_tag(calls.data(), calls.size(), domain_separator(domain_), &tag));
        std::vector<Scalar> out(output_len_);
        Engine& e = engine_ ? *engine_ : Engine::default_engine();
        check(p252_digest_batch(e.get(), &tag, all.data(), 1, total, out.data(), output_len_, P252_MEM_HOST), e.get());
        return out;
    }

    // src/hash.rs:191-195
    static std::vector<Scalar> digest(Domain domain, const std::vector<Scalar>& input, Engine* e = nullptr) {
        Hash h(domain, e);
        h.update(input);
        return h.finalize();
    }

    // NEW: n independent Hash::digest(domain, in[i*in_len .. (i+1)*in_len]) -> n x out_len
    static std::vector<Scalar> digest_batch(Domain domain, const Scalar* in, size_t n, size_t in_len,
                                            size_t output_len = 1, Engine* e = nullptr) {
        const size_t ol = (domain == Domain::Other && output_len > 0) ? output_len : 1;
        std::vector<Scalar> out(n * ol);
        Engine& eng = e ? *e : Engine::default_engine();
        check(p252_hash_batch(eng.get(), static_cast<int>(domain), in, n, in_len, out.data(), ol, P252_MEM_HOST),
              eng.get());
        return out;
    }

private:
    struct Chunk {
        const Scalar* ptr;
        size_t len;
    };
    Domain domain_;
    Engine* engine_;
    std::vector<Chunk> chunks_;
    size_t output_len_ = 1;
};

// src/encryption.rs:62-74; shared_secret = (u, v) of the JubJubAffine point (src/encryption.rs:71)
inline std::vector<Scalar> encrypt(const std::vector<Scalar>& message, const Scalar (&shared_secret_uv)[2],
                                   const Scalar& nonce, Engine& e = Engine::default_engine()) {
    std::vector<Scalar> cipher(message.size() + 1);
    int rc = p252_encrypt_batch(e.get(), message.data(), 1, message.size(), shared_secret_uv, &nonce, cipher.data(),
                                P252_MEM_HOST);
    if (rc > 0) rc = P252_ERR_ENCRYPTION_FAILED;   // dusk-safe maps pattern errors of encrypt
    check(rc, e.get());
    return cipher;
}

// src/encryption.rs:83-95; throws Error{P252_ERR_DECRYPTION_FAILED} like Err(Error::DecryptionFailed)
inline std::vector<Scalar> decrypt(const std::vector<Scalar>& cipher, const Scalar (&shared_secret_uv)[2],
                                   const Scalar& nonce, Engine& e = Engine::default_engine()) {
    if (cipher.size() < 2) throw Error(P252_ERR_DECRYPTION_FAILED, p252_strerror(P252_ERR_DECRYPTION_FAILED));
    std::vector<Scalar> msg(cipher.size() - 1);
    uint8_t ok = 0;
    size_t failed = 0;
    check(p252_decrypt_batch(e.get(), cipher.data(), 1, msg.size(), shared_secret_uv, &nonce, msg.data(), &ok, &failed,
                             P252_MEM_HOST),
          e.get());
    if (!ok) throw Error(P252_ERR_DECRYPTION_FAILED, p252_strerror(P252_ERR_DECRYPTION_FAILED));
    return msg;
}

// NEW batch forms (item-major): msg n x L, secrets n x 2, nonces n  ->  cipher n x (L+1)
inline std::vector<Scalar> encrypt_batch(const Scalar* msg, size_t n, size_t L, const Scalar* secrets_uv,
                                         const Scalar* nonces, Engine& e = Engine::default_engine()) {
    std::vector<Scalar> cipher(n * (L + 1));
    check(p252_encrypt_batch(e.get(), msg, n, L, secrets_uv, nonces, cipher.data(), P252_MEM_HOST), e.get());
    return cipher;
}
// returns the messages; ok[i] == 0 marks items for which the reference returns DecryptionFailed
inline std::vector<Scalar> decrypt_batch(const Scalar* cipher, size_t n, size_t L, const Scalar* secrets_uv,
                                         const Scalar* nonces, std::vector<uint8_t>& ok,
                                         Engine& e = Engine::default_engine()) {
    std::vector<Scalar> msg(n * L);
    ok.assign(n, 0);
    check(p252_decrypt_batch(e.get(), cipher, n, L, secrets_uv, nonces, msg.data(), ok.data(), nullptr, P252_MEM_HOST),
          e.get());
    return msg;
}

// arity-4 tree of Domain::Merkle4 digests; returns the internal levels bottom-up (root last)
inline std::vector<Scalar> merkle4_build(const std::vector<Scalar>& leaves, Engine& e = Engine::default_engine()) {
    size_t n_internal = 0;
    check(p252_merkle4_tree_nodes(leaves.size(), &n_internal, nullptr));
    std::vector<Scalar> nodes(n_internal);
    check(p252_merkle4_build(e.get(), leaves.data(), leaves.size(), nodes.data(), P252_MEM_HOST), e.get());
    return nodes;
}

// Tree of Domain::Merkle2 / Merkle4 digests for arity 2 / 4 (src/hash.rs:22-31), internal levels bottom-up
inline std::vector<Scalar> merkle_build(int arity, const std::vector<Scalar>& leaves, Engine& e = Engine::default_engine()) {
    size_t n_internal = 0;
    check(p252_merkle_tree_nodes(arity, leaves.size(), &n_internal, nullptr));
    std::vector<Scalar> nodes(n_internal);
    check(p252_merkle_build(e.get(), arity, leaves.data(), leaves.size(), nodes.data(), P252_MEM_HOST), e.get());
    return nodes;
}

// Mirror of poseidon-merkle's `Opening<T, H, A>` (consumer crate, AGENTS.md:62-66): the root, for every level
// (0 = leaf level) the whole sibling group of the path node, and the node's offset inside the group.
struct Opening {
    int arity = 4;
    Scalar root{};
    std::vector<Scalar> branch;       // depth x arity
    std::vector<size_t> positions;    // depth
    uint64_t leaf_index = 0;
    size_t depth() const { return positions.size(); }
    // Opening::verify(item): depth chained Merkle digests + membership checks, on the device
    bool verify(const Scalar& item, Engine& e = Engine::default_engine()) const {
        uint8_t ok = 0;
        check(p252_merkle_verify_batch(e.get(), arity, static_cast<int>(depth()), &item, &leaf_index, branch.data(), &root,
                                       1, &ok, nullptr, P252_MEM_HOST),
              e.get());
        return ok != 0;
    }
};

// Openings of the leaves `leaf_idx` of a tree held as leaves + nodes (merkle_build layout)
inline std::vector<Opening> merkle_open_batch(int arity, const std::vector<Scalar>& leaves, const std::vector<Scalar>& nodes,
                                              const std::vector<uint64_t>& leaf_idx, Engine& e = Engine::default_engine()) {
    int depth = 0;
    size_t n_internal = 0;
    check(p252_merkle_tree_nodes(arity, leaves.size(), &n_internal, &depth));
    if (nodes.size() != n_internal) throw Error(P252_ERR_INVALID_ARGUMENT, "node array does not match the leaf count");
    std::vector<Scalar> paths(leaf_idx.size() * depth * arity);
    check(p252_merkle_open_batch(e.get(), arity, leaves.data(), leaves.size(), nodes.data(), leaf_idx.data(), leaf_idx.size(),
                                 paths.data(), P252_MEM_HOST),
          e.get());
    std::vector<Opening> out(leaf_idx.size());
    for (size_t i = 0; i < out.size(); ++i) {
        Opening& o = out[i];
        o.arity = arity;
        o.root = nodes.back();
        o.leaf_index = leaf_idx[i];
        o.branch.assign(paths.begin() + i * depth * arity, paths.begin() + (i + 1) * depth * arity);
        uint64_t idx = leaf_idx[i];
        for (int l = 0; l < depth; ++l, idx /= static_cast<uint64_t>(arity)) o.positions.push_back(idx % arity);
    }
    return out;
}

// Write values[j] to leaf leaf_idx[j] (the last occurrence of a repeated index wins) and rehash only the dirty paths,
// in place: afterwards leaves / nodes equal merkle_build(arity, leaves).  An index outside the tree throws
// Error{P252_ERR_INVALID_ARGUMENT} and leaves the tree untouched.
inline void merkle_update_batch(int arity, std::vector<Scalar>& leaves, std::vector<Scalar>& nodes,
                                const std::vector<uint64_t>& leaf_idx, const std::vector<Scalar>& values,
                                Engine& e = Engine::default_engine()) {
    size_t n_internal = 0;
    check(p252_merkle_tree_nodes(arity, leaves.size(), &n_internal, nullptr));
    if (nodes.size() != n_internal) throw Error(P252_ERR_INVALID_ARGUMENT, "node array does not match the leaf count");
    if (leaf_idx.size() != values.size()) throw Error(P252_ERR_INVALID_ARGUMENT, "leaf_idx and values differ in length");
    check(p252_merkle_update_batch(e.get(), arity, leaves.data(), leaves.size(), nodes.data(), leaf_idx.data(),
                                   values.data(), values.size(), nullptr, P252_MEM_HOST),
          e.get());
}

// n x Opening::verify with all openings in one launch: ok[i] != 0 iff paths[i] proves items[i] under root
inline std::vector<uint8_t> merkle_verify_batch(int arity, int depth, const Scalar* items, const uint64_t* leaf_idx,
                                                const Scalar* paths, const Scalar& root, size_t n,
                                                Engine& e = Engine::default_engine()) {
    std::vector<uint8_t> ok(n);
    check(p252_merkle_verify_batch(e.get(), arity, depth, items, leaf_idx, paths, &root, n, ok.data(), nullptr, P252_MEM_HOST),
          e.get());
    return ok;
}

}  // namespace p252
