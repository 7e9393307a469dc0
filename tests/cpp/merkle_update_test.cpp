// C++ mirror of p252_merkle_update_batch (include/poseidon252_b200.hpp): the statuses that need no device, and with a
// GPU, updates (repeated indices, last write wins) checked against a rebuild.  Built and run by
// tests/test_merkle_update_cpu.py and tests/test_gpu_merkle_update.py.
#include <cstdio>
#include <cstring>

#include "poseidon252_b200.hpp"

using p252::Scalar;

static bool same(const std::vector<Scalar>& a, const std::vector<Scalar>& b) {
    return a.size() == b.size() && memcmp(a.data(), b.data(), a.size() * sizeof(Scalar)) == 0;
}

int main() {
    std::vector<Scalar> leaves(16), nodes(5);
    for (size_t i = 0; i < leaves.size(); ++i) leaves[i] = Scalar{{i + 1, 0, 0, 0}};
    const uint64_t idx[1] = {3};
    const Scalar val[1] = {Scalar{{7, 0, 0, 0}}};
    size_t rejected = 99;
    // no context
    if (p252_merkle_update_batch(nullptr, 4, leaves.data(), 16, nodes.data(), idx, val, 1, &rejected, P252_MEM_HOST) !=
        P252_ERR_INVALID_ARGUMENT)
        return 1;
    // arities other than 2 and 4, with and without a context
    for (int arity : {0, 1, 3, 8}) {
        if (p252_merkle_update_batch(nullptr, arity, leaves.data(), 16, nodes.data(), idx, val, 1, nullptr, P252_MEM_HOST) !=
            P252_ERR_INVALID_ARGUMENT)
            return 2;
        size_t ni = 0;
        if (p252_merkle_tree_nodes(arity, 16, &ni, nullptr) != P252_ERR_INVALID_ARGUMENT) return 3;
    }
    if (leaves[3].l[0] != 4) return 4;   // nothing was written
    int ndev = 0;
    p252_device_count(&ndev);
    if (ndev == 0) {
        try {
            p252::merkle_update_batch(4, leaves, nodes, {3}, {val[0]});
            return 5;   // no CPU fallback
        } catch (const p252::Error& e) {
            if (e.code != P252_ERR_NO_DEVICE) return 6;
        }
        std::puts("merkle update ok (no GPU: statuses only)");
        return 0;
    }
    p252::Engine& eng = p252::Engine::default_engine();
    for (int arity : {4, 2}) {
        const size_t n = arity == 4 ? 1024 : 256;
        std::vector<Scalar> lv(n);
        for (size_t i = 0; i < n; ++i) lv[i] = Scalar{{1000 + i, i * 7, 0, 0}};
        auto nd = p252::merkle_build(arity, lv);
        if (p252_merkle_update_batch(eng.get(), 3, lv.data(), n, nd.data(), idx, val, 1, nullptr, P252_MEM_HOST) !=
            P252_ERR_INVALID_ARGUMENT)
            return 7;
        // repeated indices: the last write wins
        std::vector<uint64_t> ui = {0, n - 1, 5, 5, 17, n / 2, 5, 0};
        std::vector<Scalar> uv(ui.size());
        for (size_t j = 0; j < ui.size(); ++j) uv[j] = Scalar{{50 + j, 3, 0, 0}};
        p252::merkle_update_batch(arity, lv, nd, ui, uv, eng);
        std::vector<Scalar> want = lv;
        for (size_t j = 0; j < ui.size(); ++j) want[ui[j]] = uv[j];
        if (!same(lv, want)) return 8;
        if (!same(nd, p252::merkle_build(arity, want))) return 9;
        // an index outside the tree: Error, the tree is untouched
        const std::vector<Scalar> l0 = lv, n0 = nd;
        try {
            p252::merkle_update_batch(arity, lv, nd, {1, n}, {uv[0], uv[1]}, eng);
            return 10;
        } catch (const p252::Error& e) {
            if (e.code != P252_ERR_INVALID_ARGUMENT) return 11;
        }
        if (!same(lv, l0) || !same(nd, n0)) return 12;
    }
    std::puts("merkle update ok (GPU)");
    return 0;
}
