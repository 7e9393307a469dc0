"""CPU: the tree shape the C ABI derives for Merkle trees -- p252_merkle_tree_nodes / p252_merkle4_tree_nodes, the level
partition of p252_merkle4_shard_plan -- against a small Python model, for every status, plus the null-context status of
every Merkle batch entry point.  None of these calls needs a device."""
import ctypes

import numpy as np
import pytest

from poseidon252_b200 import _native

OK, IO_PATTERN_VIOLATION, INVALID_ARGUMENT = 0, 1, -1
ARITIES = (0, 1, 2, 3, 4, 8)
N_LEAVES = (0, 1, 2, 3, 4, 8, 12, 16, 48, 64, 2 ** 40, 4 ** 31, 2 ** 63, 2 ** 64 - 1)


def model_shape(arity, n_leaves):
    """(status, n_internal, depth): a full tree has n_leaves = arity^depth leaves with depth >= 1, arity 2 or 4."""
    if arity not in (2, 4) or n_leaves < 2:
        return INVALID_ARGUMENT, None, None
    depth, m = 0, n_leaves
    while m % arity == 0:
        m //= arity
        depth += 1
    if m != 1:
        return IO_PATTERN_VIOLATION, None, None        # some level is not a multiple of the arity
    return OK, (n_leaves - 1) // (arity - 1), depth


def model_plan(n_leaves, nranks, rank):
    """(status, depth, [(level_offset, level_size, my_offset, my_count, sharded) per internal level, bottom-up])."""
    if nranks < 1 or not 0 <= rank < nranks:
        return INVALID_ARGUMENT, None, None
    st, _, depth = model_shape(4, n_leaves)
    if st != OK:
        return st, None, None
    if n_leaves % nranks or (n_leaves // nranks) % 4:
        return INVALID_ARGUMENT, None, None
    levels, off = [], 0
    for h in range(1, depth + 1):
        size = n_leaves // 4 ** h
        sharded = size % nranks == 0
        mine = size // nranks if sharded else size
        levels.append((off, size, rank * mine if sharded else 0, mine, int(sharded)))
        off += size
    return OK, depth, levels


@pytest.mark.parametrize("arity", ARITIES)
def test_tree_nodes_against_model(arity):
    lib = _native.lib()
    for n in N_LEAVES:
        st, n_internal, depth = model_shape(arity, n)
        ni, nl = ctypes.c_size_t(7), ctypes.c_int(-7)
        assert lib.p252_merkle_tree_nodes(arity, n, ctypes.byref(ni), ctypes.byref(nl)) == st, (arity, n)
        assert lib.p252_merkle_tree_nodes(arity, n, None, None) == st, (arity, n)
        if st == OK:
            assert (ni.value, nl.value) == (n_internal, depth), (arity, n)
        else:
            assert (ni.value, nl.value) == (7, -7), (arity, n)          # outputs untouched on failure
        if arity == 4:
            ni4, nl4 = ctypes.c_size_t(7), ctypes.c_int(-7)
            assert lib.p252_merkle4_tree_nodes(n, ctypes.byref(ni4), ctypes.byref(nl4)) == st, n
            assert (ni4.value, nl4.value) == (ni.value, nl.value), n


PLAN_CASES = ([(4 ** k, g, r) for k in (1, 2, 3, 5, 8, 14) for g in (1, 2, 3, 4, 8, 16, 64) for r in {0, 1 % g, g - 1}]
              + [(4 ** 31, 2 ** 20, 12345), (2 ** 62, 3, 2)]
              + [(64, 0, 0), (64, -1, 0), (64, 2, -1), (64, 2, 2), (64, 3, 1), (16, 8, 0), (4, 2, 0),
                 (0, 1, 0), (1, 1, 0), (2, 1, 0), (8, 2, 1), (48, 4, 0), (48, 1, 0), (2 ** 63, 2, 0)])


def test_shard_plan_against_model():
    lib = _native.lib()
    for n, g, r in PLAN_CASES:
        st, depth, levels = model_plan(n, g, r)
        nl = ctypes.c_int(-7)
        assert lib.p252_merkle4_shard_plan(n, g, r, None, 0, ctypes.byref(nl)) == st, (n, g, r)
        assert nl.value == (depth if st == OK else -7), (n, g, r)
        if st != OK:
            continue
        arr = (_native.LevelPlan * (depth + 2))()
        for p in arr:
            p.level_offset, p.reserved = 99, 99
        nl.value = -7
        assert lib.p252_merkle4_shard_plan(n, g, r, arr, depth + 2, ctypes.byref(nl)) == OK
        assert nl.value == depth
        got = [(p.level_offset, p.level_size, p.my_offset, p.my_count, p.sharded) for p in arr[:depth]]
        assert got == levels, (n, g, r)
        assert all(p.reserved == 0 for p in arr[:depth])
        assert all((p.level_offset, p.reserved) == (99, 99) for p in arr[depth:])   # nothing past the last level
        assert levels[0][4] == 1                                                     # the first level is always sharded
        # capacity exactly the level count is enough; one less is refused, after *n_levels was written
        assert lib.p252_merkle4_shard_plan(n, g, r, arr, depth, None) == OK
        nl.value = -7
        assert lib.p252_merkle4_shard_plan(n, g, r, arr, depth - 1, ctypes.byref(nl)) == INVALID_ARGUMENT
        assert nl.value == depth


def test_merkle_entry_points_refuse_null_context():
    lib = _native.lib()
    leaves = np.arange(64 * 4, dtype=np.uint64).reshape(64, 4)
    nodes = np.zeros((21, 4), dtype=np.uint64)
    idx = np.array([5, 17], dtype=np.uint64)
    items = leaves[[5, 17]].copy()
    paths = np.zeros((2, 3, 4, 4), dtype=np.uint64)
    ok = np.full(2, 7, dtype=np.uint8)
    root = np.ones(4, dtype=np.uint64)
    before = leaves.copy()
    failed = ctypes.c_size_t(7)
    p = lambda a: a.ctypes.data                                                       # noqa: E731
    for flags in (_native.MEM_HOST, _native.MEM_DEVICE, _native.MEM_DEVICE | _native.ASYNC):
        calls = {
            "merkle4_level": lib.p252_merkle4_level(None, p(leaves), 16, p(nodes), flags),
            "merkle4_build": lib.p252_merkle4_build(None, p(leaves), 64, p(nodes), flags),
            "merkle_build/4": lib.p252_merkle_build(None, 4, p(leaves), 64, p(nodes), flags),
            "merkle_build/2": lib.p252_merkle_build(None, 2, p(leaves), 64, p(nodes), flags),
            "open": lib.p252_merkle_open_batch(None, 4, p(leaves), 64, p(nodes), p(idx), 2, p(paths), flags),
            "verify": lib.p252_merkle_verify_batch(None, 4, 3, p(items), p(idx), p(paths), p(root), 2, p(ok),
                                                   ctypes.byref(failed), flags),
            "update": lib.p252_merkle_update_batch(None, 4, p(leaves), 64, p(nodes), p(idx), p(items), 2,
                                                   ctypes.byref(failed), flags),
            "build_dist": lib.p252_merkle4_build_dist(None, p(leaves), 64, p(nodes), flags),
            "level_timings": lib.p252_tree_level_timings(None, None, 0, None, None),
        }
        assert calls == {k: INVALID_ARGUMENT for k in calls}, flags
    assert np.array_equal(leaves, before) and not nodes.any() and not paths.any()
    assert (ok == 7).all() and failed.value == 7
