"""Arity-4 Merkle trees of Domain::Merkle4 digests (node = Hash::digest(Domain::Merkle4, 4 children),
/root/reference/src/hash.rs:22-26).  Tree logic itself left the reference crate in 0.29.0
(CHANGELOG.md:164-168); only the node hash is defined there."""
from .engine import default_engine


def merkle4_level(children, engine=None, out=None, async_=False):
    eng = engine or default_engine(children.device.index if hasattr(children, "is_cuda") else 0)
    return eng.merkle4_level(children, out=out, async_=async_)


def merkle4_build(leaves, engine=None, out=None, async_=False):
    """leaves (4^k, 4) -> internal nodes bottom-up, root last."""
    eng = engine or default_engine(leaves.device.index if hasattr(leaves, "is_cuda") else 0)
    return eng.merkle4_build(leaves, out=out, async_=async_)


def merkle2_build(leaves, engine=None, out=None, async_=False):
    """Binary tree of Domain::Merkle2 digests (src/hash.rs:27-31): leaves (2^k, 4) -> internal nodes, root last."""
    eng = engine or default_engine(leaves.device.index if hasattr(leaves, "is_cuda") else 0)
    return eng.merkle_build(leaves, arity=2, out=out, async_=async_)


def open_batch(leaves, nodes, leaf_idx, arity=4, engine=None, out=None, async_=False):
    """Openings of the leaves `leaf_idx`: (n, depth, arity, 4) -- per level the whole sibling group of the path
    node, level 0 = the leaf's own group (the `branch` of a poseidon-merkle `Opening`, AGENTS.md:62-66)."""
    eng = engine or default_engine(leaves.device.index if hasattr(leaves, "is_cuda") else 0)
    return eng.merkle_open_batch(leaves, nodes, leaf_idx, arity=arity, out=out, async_=async_)


def verify_batch(leaf_items, leaf_idx, paths, root, arity=4, engine=None, async_=False):
    """n x Opening::verify on the device (depth chained Merkle digests per item) -> ok (n,) uint8."""
    eng = engine or default_engine(paths.device.index if hasattr(paths, "is_cuda") else 0)
    return eng.merkle_verify_batch(leaf_items, leaf_idx, paths, root, arity=arity, async_=async_)


def update_batch(leaves, nodes, leaf_idx, values, arity=4, engine=None, async_=False):
    """Overwrite the leaves `leaf_idx` with `values` (last occurrence wins) and rehash only their paths, in place:
    afterwards (leaves, nodes) equal a rebuild.  Returns (leaves, nodes)."""
    eng = engine or default_engine(leaves.device.index if hasattr(leaves, "is_cuda") else 0)
    return eng.merkle_update_batch(leaves, nodes, leaf_idx, values, arity=arity, async_=async_)


def positions(leaf_idx, depth, arity=4):
    """Offset of the path node inside its sibling group at every level (the `positions` of an Opening)."""
    out, i = [], int(leaf_idx)
    for _ in range(depth):
        out.append(i % arity)
        i //= arity
    return out


class Opening:
    """Host-side mirror of poseidon-merkle's `Opening<T, H, A>`: `root`, `branch[level][slot]`, `positions[level]`
    (level 0 = leaf level here).  `verify(item)` runs the batch verifier on a batch of one."""

    def __init__(self, root, branch, leaf_idx, arity=4):
        import numpy as np
        self.root = np.ascontiguousarray(root, dtype=np.uint64).reshape(4)
        self.branch = np.ascontiguousarray(branch, dtype=np.uint64)
        if self.branch.ndim != 3 or self.branch.shape[1:] != (arity, 4):
            raise ValueError("branch must have shape (depth, arity, 4)")
        self.arity = int(arity)
        self.leaf_idx = int(leaf_idx)
        self.positions = positions(leaf_idx, self.branch.shape[0], arity)

    def verify(self, item, engine=None):
        import numpy as np
        ok = verify_batch(np.ascontiguousarray(item, dtype=np.uint64).reshape(1, 4),
                          np.array([self.leaf_idx], dtype=np.uint64), self.branch[None], self.root, arity=self.arity,
                          engine=engine)
        return bool(ok[0])


def level_offsets(n_leaves, arity=4):
    """[(offset, size)] of each internal level inside the node array, bottom-up."""
    out, off, m = [], 0, n_leaves // arity
    while m >= 1:
        out.append((off, m))
        off += m
        if m == 1:
            break
        m //= arity
    return out


def shard_plan(n_leaves_total, nranks, rank):
    """The per-level partition of the multi-GPU build (p252_merkle4_shard_plan): list of dicts with
    level_offset, level_size, my_offset, my_count, sharded -- bottom-up."""
    import ctypes

    from . import _native
    from .errors import raise_for_status
    lib = _native.lib()
    n = ctypes.c_int(0)
    raise_for_status(lib.p252_merkle4_shard_plan(int(n_leaves_total), int(nranks), int(rank), None, 0, ctypes.byref(n)), lib)
    arr = (_native.LevelPlan * n.value)()
    raise_for_status(lib.p252_merkle4_shard_plan(int(n_leaves_total), int(nranks), int(rank), arr, n.value, ctypes.byref(n)), lib)
    return [{f: int(getattr(a, f)) for f in ("level_offset", "level_size", "my_offset", "my_count", "sharded")} for a in arr]
