"""GPU (-m gpu): incremental Merkle updates (p252_merkle_update_batch).  After an update, leaves and nodes must equal
merkle_build of the expected leaves (the writes applied in order, the last one wins) and a C-oracle tree of them; only
the nodes on dirty paths and their sibling groups may be touched.  Every case runs on both kernel forms (the `engine`
fixture's lane-split and throughput-only arms)."""
import numpy as np
import pytest

import poseidon252_b200 as pb
from conftest import mont
from poseidon252_b200 import merkle
from poseidon252_b200.scalar import random_limbs_fast, random_scalars

pytestmark = pytest.mark.gpu

SENTINEL = np.uint64(0xFFFFFFFFFFFFFFFF)
_ORACLE_CACHE = {}


def oracle_tree(coracle, oracle, leaves, arity):
    """levels[0] = leaves, levels[-1] = [root], every digest by the C oracle"""
    dom = oracle.Domain.Merkle4 if arity == 4 else oracle.Domain.Merkle2
    tag = mont(oracle.hash_to_scalar(oracle.tag_input([oracle.Absorb(arity), oracle.Squeeze(1)], dom)))
    levels, cur = [leaves], leaves
    while cur.shape[0] > 1:
        cur = coracle.digest(tag, cur.reshape(-1, arity, 4), arity, 1).reshape(-1, 4)
        levels.append(cur)
    return levels


def apply_writes(leaves, idx, vals):
    """The leaves after writing vals[j] to idx[j] for j = 0..k-1 in order."""
    out = leaves.copy()
    idx = np.asarray(idx, dtype=np.uint64)
    if len(idx):
        _, first_rev = np.unique(idx[::-1], return_index=True)
        last = len(idx) - 1 - first_rev                       # position of the last occurrence of every index
        out[idx[last].astype(np.int64)] = vals[last]
    return out


def make_batch(rng, n_leaves, k, order):
    """k indices incl. 0 and n_leaves-1 and repeated indices (with different values), sorted or shuffled."""
    idx = rng.integers(0, n_leaves, size=k, dtype=np.uint64)
    if k >= 2:
        idx[0], idx[1] = 0, n_leaves - 1
    if k >= 7:
        idx[k // 2] = idx[2]                                   # repeats: later writes to the same leaf
        idx[k - 1] = idx[2]
        idx[3] = 0
    if order == "sorted":
        idx = np.sort(idx, kind="stable")
    vals = random_limbs_fast(rng, (k,)) if k > 4096 else random_scalars(rng, k)
    return idx, vals.reshape(k, 4)


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def to_host(t):
    return t.cpu().numpy().view(np.uint64)


def run_update(engine, space, leaves, nodes, idx, vals, arity, async_=False):
    """-> (leaves, nodes) after the update, as host arrays"""
    if space == "host":
        l, n = leaves.copy(), nodes.copy()
        engine.merkle_update_batch(l, n, idx, vals, arity=arity, async_=async_)
        return l, n
    dl, dn, di, dv = to_dev(leaves), to_dev(nodes), to_dev(idx), to_dev(vals)   # alive until the engine is done
    engine.merkle_update_batch(dl, dn, di, dv, arity=arity, async_=async_)
    if async_:
        engine.sync()
    return to_host(dl), to_host(dn)


def base_tree(engine, arity, logn, seed):
    rng = np.random.default_rng(seed)
    n = arity ** logn
    leaves = random_limbs_fast(rng, (n,)).reshape(n, 4)
    return rng, leaves, engine.merkle_build(leaves, arity=arity)


K_VALUES = [1, 2, 7, 100, 3552, 3553, 5000, "n"]


@pytest.mark.parametrize("space", ["host", "device"])
@pytest.mark.parametrize("k", K_VALUES)
@pytest.mark.parametrize("arity,logn", [(4, 6), (4, 8), (2, 10), (2, 12)])
def test_update_parity(engine, coracle, oracle, arity, logn, k, space):
    seed = arity * 1000 + logn
    rng, leaves, nodes = base_tree(engine, arity, logn, seed)
    n = arity ** logn
    kk = n if k == "n" else k
    order = "sorted" if k in (2, 100, 3553, "n") else "shuffled"
    idx, vals = make_batch(np.random.default_rng(seed + kk), n, kk, order)
    want_leaves = apply_writes(leaves, idx, vals)
    got_leaves, got_nodes = run_update(engine, space, leaves, nodes, idx, vals, arity)
    assert np.array_equal(got_leaves, want_leaves)
    assert np.array_equal(got_nodes, engine.merkle_build(want_leaves, arity=arity))
    key = (arity, logn, kk)
    if key not in _ORACLE_CACHE:
        _ORACLE_CACHE[key] = np.concatenate(oracle_tree(coracle, oracle, want_leaves, arity)[1:], axis=0)
    assert np.array_equal(got_nodes, _ORACLE_CACHE[key])


def touched(n_leaves, idx, arity):
    """Masks of the leaves and nodes an update of `idx` reads or writes: the sibling groups of every dirty node
    (which contain the dirty nodes themselves) and the root."""
    s = 1 if arity == 2 else 2
    depth = int(round(np.log2(n_leaves))) // s
    idx = np.unique(np.asarray(idx, dtype=np.uint64))
    masks, size = [], n_leaves
    for l in range(depth + 1):
        m = np.zeros(size, dtype=bool)
        if l == depth:
            m[0] = True
        else:
            groups = np.unique(idx >> np.uint64(s * (l + 1))).astype(np.int64)
            for q in range(arity):
                m[groups * arity + q] = True
        masks.append(m)
        size //= arity
    return masks[0], np.concatenate(masks[1:])


@pytest.mark.parametrize("space", ["host", "device"])
@pytest.mark.parametrize("arity,logn,k", [(4, 6, 9), (4, 8, 300), (2, 10, 5), (2, 12, 700)])
def test_only_dirty_paths_written(engine, arity, logn, k, space):
    rng, leaves, nodes = base_tree(engine, arity, logn, 7 + logn)
    n = arity ** logn
    idx, vals = make_batch(rng, n, k, "shuffled")
    lmask, nmask = touched(n, idx, arity)
    assert not lmask.all() and not nmask.all()
    s_leaves, s_nodes = leaves.copy(), nodes.copy()
    s_leaves[~lmask] = SENTINEL
    s_nodes[~nmask] = SENTINEL
    got_leaves, got_nodes = run_update(engine, space, s_leaves, s_nodes, idx, vals, arity)
    want_leaves = apply_writes(leaves, idx, vals)
    want_nodes = engine.merkle_build(want_leaves, arity=arity)
    assert (got_leaves[~lmask] == SENTINEL).all() and (got_nodes[~nmask] == SENTINEL).all()
    assert np.array_equal(got_leaves[lmask], want_leaves[lmask])
    assert np.array_equal(got_nodes[nmask], want_nodes[nmask])


@pytest.mark.parametrize("space", ["host", "device"])
@pytest.mark.parametrize("arity,logn", [(4, 7), (2, 11)])
def test_chain_of_updates(engine, arity, logn, space):
    rng, leaves, nodes = base_tree(engine, arity, logn, 99 + arity)
    n = arity ** logn
    want, inputs = leaves.copy(), []
    if space == "host":
        cur_l, cur_n = leaves.copy(), nodes.copy()
    else:
        cur_l, cur_n = to_dev(leaves), to_dev(nodes)
    for b in range(20):
        k = int(rng.integers(1, 600))
        idx, vals = make_batch(rng, n, k, "shuffled" if b % 2 else "sorted")
        want = apply_writes(want, idx, vals)
        if space == "host":
            engine.merkle_update_batch(cur_l, cur_n, idx, vals, arity=arity)
        else:
            inputs.append((to_dev(idx), to_dev(vals)))          # alive until the engine's stream is done with them
            engine.merkle_update_batch(cur_l, cur_n, *inputs[-1], arity=arity, async_=True)
    if space == "device":
        engine.sync()
        cur_l, cur_n = to_host(cur_l), to_host(cur_n)
    assert np.array_equal(cur_l, want)
    assert np.array_equal(cur_n, engine.merkle_build(want, arity=arity))


@pytest.mark.parametrize("arity,logn", [(4, 5), (2, 9)])
def test_out_of_range_indices(engine, arity, logn):
    rng, leaves, nodes = base_tree(engine, arity, logn, 5)
    n = arity ** logn
    idx, vals = make_batch(rng, n, 50, "shuffled")
    bad = idx.copy()
    bad[[4, 17, 30]] = np.array([n, n + 12345, 2 ** 64 - 1], dtype=np.uint64)
    # HOST: rejected before anything is written
    l, nd = leaves.copy(), nodes.copy()
    with pytest.raises(pb.EngineError) as ei:
        engine.merkle_update_batch(l, nd, bad, vals, arity=arity)
    assert ei.value.code == -1
    assert l.tobytes() == leaves.tobytes() and nd.tobytes() == nodes.tobytes()
    # DEVICE: the out-of-range entries are skipped and counted, the others applied
    keep = np.ones(50, dtype=bool)
    keep[[4, 17, 30]] = False
    want = apply_writes(leaves, bad[keep], vals[keep])
    for async_ in (False, True):
        got_l, got_n = run_update(engine, "device", leaves, nodes, bad, vals, arity, async_=async_)
        assert engine.last_update_rejected() == 3
        assert np.array_equal(got_l, want)
        assert np.array_equal(got_n, engine.merkle_build(want, arity=arity))
    # all entries out of range: nothing changes
    got_l, got_n = run_update(engine, "device", leaves, nodes, np.full(10, n, dtype=np.uint64), vals[:10], arity)
    assert engine.last_update_rejected() == 10
    assert np.array_equal(got_l, leaves) and np.array_equal(got_n, nodes)


def test_edges(engine):
    import torch
    rng, leaves, nodes = base_tree(engine, 4, 4, 3)
    # k = 0 launches nothing, for both memory spaces
    before = engine.launch_count
    l, nd = leaves.copy(), nodes.copy()
    engine.merkle_update_batch(l, nd, np.zeros(0, dtype=np.uint64), np.zeros((0, 4), dtype=np.uint64))
    dl, dn = to_dev(leaves), to_dev(nodes)
    engine.merkle_update_batch(dl, dn, torch.zeros(0, dtype=torch.int64, device="cuda"),
                               torch.zeros((0, 4), dtype=torch.int64, device="cuda"))
    assert engine.launch_count == before
    assert np.array_equal(l, leaves) and np.array_equal(to_host(dn), nodes)
    # depth 1: n_leaves = arity
    for arity in (2, 4):
        lv = random_scalars(rng, arity)
        nd1 = engine.merkle_build(lv, arity=arity)
        v = random_scalars(rng, 1)
        for space in ("host", "device"):
            got_l, got_n = run_update(engine, space, lv, nd1, np.array([arity - 1], dtype=np.uint64), v, arity)
            want = apply_writes(lv, [arity - 1], v)
            assert np.array_equal(got_l, want) and np.array_equal(got_n, engine.merkle_build(want, arity=arity))
    # the wrapper refuses buffers it would have to copy, and mixed memory spaces
    idx, vals = np.array([1, 2], dtype=np.uint64), random_scalars(rng, 2)
    ro = leaves.copy()
    ro.setflags(write=False)
    bad_cases = [
        (ro, nodes.copy(), idx, vals),                                       # not writable
        (np.asfortranarray(leaves), nodes.copy(), idx, vals),                # not C-contiguous
        (leaves.astype(np.float64), nodes.copy(), idx, vals),                # wrong dtype
        (leaves.astype(np.uint32), nodes.copy(), idx, vals),
        (leaves.copy(), nodes[:-1].copy(), idx, vals),                       # wrong shape
        (leaves.copy(), nodes.copy(), idx, vals[:1]),                        # lengths differ
        (leaves.copy(), nodes.copy(), to_dev(idx), vals),                    # mixed memory spaces
        (leaves.copy(), to_dev(nodes), idx, vals),
        (to_dev(leaves), to_dev(nodes), idx, to_dev(vals)),
        (to_dev(leaves), to_dev(nodes), to_dev(idx), vals),
        (to_dev(leaves).t().contiguous().t(), to_dev(nodes), to_dev(idx), to_dev(vals)),   # non-contiguous tensor
        (to_dev(leaves).to(torch.int32), to_dev(nodes), to_dev(idx), to_dev(vals)),
    ]
    for case in bad_cases:
        with pytest.raises(pb.EngineError):
            engine.merkle_update_batch(*case, arity=4)
    assert np.array_equal(ro, leaves)


def test_openings_after_update(engine):
    rng, leaves, nodes = base_tree(engine, 4, 6, 11)
    n = 4 ** 6
    probe = np.array([0, 5, 777, n - 1], dtype=np.uint64)
    old_paths = engine.merkle_open_batch(leaves, nodes, probe)
    idx, vals = make_batch(rng, n, 64, "shuffled")
    idx[:4] = probe                                             # change every probed leaf
    l, nd = leaves.copy(), nodes.copy()
    merkle.update_batch(l, nd, idx, vals, engine=engine)
    assert not np.array_equal(nd[-1], nodes[-1])
    check = np.concatenate([probe, rng.integers(0, n, size=200, dtype=np.uint64)])
    paths = engine.merkle_open_batch(l, nd, check)
    assert engine.merkle_verify_batch(l[check.astype(np.int64)], check, paths, nd[-1]).all()
    stale = engine.merkle_verify_batch(l[probe.astype(np.int64)], probe, old_paths, nd[-1])
    assert not stale.any()                                     # openings taken before the update no longer verify


def test_large_async_on_torch_stream():
    """4^11 leaves, 2^16 random updates, device tensors on a torch side stream, async_=True."""
    import torch
    stream = torch.cuda.Stream()
    eng = pb.Engine(0, stream=stream.cuda_stream)
    try:
        rng = np.random.default_rng(2024)
        n = 4 ** 11
        leaves = random_limbs_fast(rng, (n,)).reshape(n, 4)
        idx = rng.integers(0, n, size=1 << 16, dtype=np.uint64)
        vals = random_limbs_fast(rng, (1 << 16,)).reshape(-1, 4)
        with torch.cuda.stream(stream):
            dl = to_dev(leaves)
            dn = eng.merkle_build(dl, arity=4, async_=True)
            eng.merkle_update_batch(dl, dn, to_dev(idx), to_dev(vals), arity=4, async_=True)
            want = eng.merkle_build(dl, arity=4, async_=True)
        stream.synchronize()
        assert np.array_equal(to_host(dl), apply_writes(leaves, idx, vals))
        assert torch.equal(dn, want)
    finally:
        eng.close()


def test_cpp_merkle_update_gpu():
    from test_merkle_update_cpu import build_and_run_cpp
    res = build_and_run_cpp()
    assert res.returncode == 0, (res.returncode, res.stdout, res.stderr)
    assert "merkle update ok (GPU)" in res.stdout
