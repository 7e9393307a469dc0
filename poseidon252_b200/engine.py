"""Engine: one CUDA device + stream behind the C ABI (include/poseidon252_b200.h).

Buffers are either numpy uint64 arrays (HOST: the library stages H2D/D2H in overlapped chunks) or
torch CUDA tensors of dtype int64/uint64 (DEVICE: zero-copy, enqueued on the engine's stream).
There is no CPU fallback: constructing an Engine without a B200-class GPU raises EngineError."""
import ctypes

import numpy as np

from . import _native
from .errors import EngineError, raise_for_status

_DEFAULT = {}


def _is_torch(x):
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda")


class Engine:
    def __init__(self, device=0, stream=None):
        """stream: None -> the engine creates its own non-blocking stream; an int -> an existing
        cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream; 0 means the legacy
        default stream)."""
        self._lib = _native.lib()
        self._ctx = ctypes.c_void_p()
        self.device = int(device)
        if stream is None:
            rc = self._lib.p252_create(self.device, ctypes.byref(self._ctx))
        else:
            handle = int(stream) or 1          # 0 -> cudaStreamLegacy
            rc = self._lib.p252_create_on_stream(self.device, ctypes.c_void_p(handle), ctypes.byref(self._ctx))
        if rc != 0:
            self._ctx = ctypes.c_void_p()
            raise EngineError(rc, self._lib.p252_strerror(rc).decode())
        self._dist = False
        self._stream_handle = None if stream is None else int(stream)

    def _fence_torch(self):
        """Device tensors are produced on torch's current stream; unless the engine was bound to that
        very stream, wait for it before enqueueing on ours (cross-stream ordering)."""
        import torch
        cur = torch.cuda.current_stream(self.device)
        if self._stream_handle is None or int(cur.cuda_stream) != self._stream_handle:
            cur.synchronize()

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.p252_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def sync(self):
        self._check(self._lib.p252_sync(self._ctx))

    @property
    def launch_count(self):
        return int(self._lib.p252_launch_count(self._ctx))

    def _check(self, rc):
        raise_for_status(rc, self._lib, self._ctx)

    # -- buffer plumbing --------------------------------------------------------------------------
    def _in(self, x, shape_tail):
        """-> (pointer, leading-shape, flags, keepalive)"""
        if _is_torch(x):
            if not x.is_cuda or x.device.index != self.device:
                raise EngineError(-1, "tensor is not on cuda:%d" % self.device)
            if str(x.dtype) not in ("torch.int64", "torch.uint64") or not x.is_contiguous():
                raise EngineError(-1, "device buffers must be contiguous int64/uint64 tensors")
            if tuple(x.shape[-len(shape_tail):]) != tuple(shape_tail):
                raise EngineError(-1, "expected trailing shape %s, got %s" % (shape_tail, tuple(x.shape)))
            self._fence_torch()
            return x.data_ptr(), tuple(x.shape[:-len(shape_tail)]), _native.MEM_DEVICE, x
        a = np.ascontiguousarray(x, dtype=np.uint64)
        if tuple(a.shape[-len(shape_tail):]) != tuple(shape_tail):
            raise EngineError(-1, "expected trailing shape %s, got %s" % (shape_tail, a.shape))
        return a.ctypes.data, tuple(a.shape[:-len(shape_tail)]), _native.MEM_HOST, a

    def _check_out(self, out, shape, like, itemsize=8):
        """A caller-supplied result buffer goes to native code as a raw pointer: refuse anything whose shape,
        element type, contiguity or memory space differs from what the call will write."""
        shape = tuple(int(v) for v in shape)
        if _is_torch(like):
            if not _is_torch(out) or not out.is_cuda or out.device != like.device:
                raise EngineError(-1, "out must be a CUDA tensor on %s" % like.device)
            ok_dtype = str(out.dtype) in (("torch.int64", "torch.uint64") if itemsize == 8 else ("torch.uint8",))
            if tuple(out.shape) != shape or not ok_dtype or not out.is_contiguous():
                raise EngineError(-1, "out must be a contiguous %d-byte integer tensor of shape %s" % (itemsize, shape))
        else:
            want = np.uint64 if itemsize == 8 else np.uint8
            if not isinstance(out, np.ndarray) or out.dtype != want or tuple(out.shape) != shape or \
                    not out.flags.c_contiguous or not out.flags.writeable:
                raise EngineError(-1, "out must be a writable C-contiguous %s array of shape %s" % (np.dtype(want).name, shape))
        return out

    @staticmethod
    def _same_lead(name, lead, n):
        if tuple(lead) != (n,):
            raise EngineError(-1, "%s must have %d rows, got leading shape %s" % (name, n, tuple(lead)))

    def _out_like(self, ref, shape, dtype=None):
        if _is_torch(ref):
            import torch
            return torch.empty(shape, dtype=ref.dtype if dtype is None else dtype, device=ref.device)
        return np.empty(shape, dtype=np.uint64 if dtype is None else dtype)

    @staticmethod
    def _ptr(x):
        return x.data_ptr() if _is_torch(x) else x.ctypes.data

    # -- hades::permute_batch ---------------------------------------------------------------------
    def permute_batch(self, states, dense=False, out=None, async_=False):
        """n x Safe::permute (src/hades/permutation/scalar.rs:25-27).  states: (n, 5, 4)."""
        ptr, lead, flags, keep = self._in(states, (5, 4))
        n = int(np.prod(lead)) if lead else 1
        if _is_torch(keep):
            if out is None:
                res = keep.clone()
            else:
                res = self._check_out(out, keep.shape, keep)
                if out is not keep:
                    out.copy_(keep)
            self._fence_torch()
        elif out is not None:
            res = self._check_out(out, keep.shape, keep)
            if res is not states:
                np.copyto(res, keep)              # the caller's `states` stays untouched
        else:
            res = keep.copy() if keep is states else keep   # `keep` is already a private copy otherwise
        fn = self._lib.p252_permute_batch_dense if dense else self._lib.p252_permute_batch
        self._check(fn(self._ctx, self._ptr(res), n, flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def permute_batch_inplace(self, states, async_=False):
        ptr, lead, flags, keep = self._in(states, (5, 4))
        n = int(np.prod(lead)) if lead else 1
        if not _is_torch(keep) and keep is not states:
            raise EngineError(-1, "in-place permute needs a contiguous uint64 array")
        self._check(self._lib.p252_permute_batch(self._ctx, ptr, n,
                                                 flags | (_native.ASYNC if async_ and flags else 0)))
        return states

    # -- sponges ------------------------------------------------------------------------------------
    def digest_batch_with_tag(self, tag, inputs, out_len=1, out=None, async_=False):
        """start(tag) -> absorb(in_len) -> squeeze(out_len) for every item.  inputs: (n, in_len, 4)."""
        tag = np.ascontiguousarray(tag, dtype=np.uint64).reshape(4)
        if inputs.ndim != 3:
            raise EngineError(-1, "inputs must have shape (n, in_len, 4)")
        in_len = int(inputs.shape[1])
        ptr, lead, flags, keep = self._in(inputs, (in_len, 4))
        n = lead[0]
        res = self._out_like(keep, (n, int(out_len), 4)) if out is None else self._check_out(out, (n, int(out_len), 4), keep)
        self._check(self._lib.p252_digest_batch(self._ctx, tag.ctypes.data, ptr, n, in_len, self._ptr(res),
                                                int(out_len), flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def hash_batch(self, domain, inputs, out_len=1, out=None, async_=False):
        """n x Hash::digest(domain, inputs[i]) with output_len(out_len)."""
        if inputs.ndim != 3:
            raise EngineError(-1, "inputs must have shape (n, in_len, 4)")
        in_len = int(inputs.shape[1])
        ptr, lead, flags, keep = self._in(inputs, (in_len, 4))
        n = lead[0]
        res = self._out_like(keep, (n, int(out_len), 4)) if out is None else self._check_out(out, (n, int(out_len), 4), keep)
        self._check(self._lib.p252_hash_batch(self._ctx, int(domain), ptr, n, in_len, self._ptr(res), int(out_len),
                                              flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def hash_batch_truncated(self, domain, inputs, out_len=1, out=None, async_=False):
        """n x Hash::digest_truncated: raw (canonical, 250-bit masked) limbs for JubJubScalar::from_raw."""
        if inputs.ndim != 3:
            raise EngineError(-1, "inputs must have shape (n, in_len, 4)")
        in_len = int(inputs.shape[1])
        ptr, lead, flags, keep = self._in(inputs, (in_len, 4))
        n = lead[0]
        res = self._out_like(keep, (n, int(out_len), 4)) if out is None else self._check_out(out, (n, int(out_len), 4), keep)
        self._check(self._lib.p252_hash_batch_truncated(self._ctx, int(domain), ptr, n, in_len, self._ptr(res),
                                                        int(out_len), flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def scalars_from_bytes(self, data, async_=False):
        """(n, 32) uint8 canonical little-endian (host) or (n, 4) 64-bit device tensor of the same bytes
        -> (scalars (n, 4), ok (n,) uint8); ok == 0 where the value is >= p."""
        if _is_torch(data):
            import torch
            ptr, lead, flags, keep = self._in(data, (4,))
            n = lead[0]
            out = torch.empty((n, 4), dtype=keep.dtype, device=keep.device)
            ok = torch.empty((n,), dtype=torch.uint8, device=keep.device)
        else:
            keep = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1, 32)
            ptr, n, flags = keep.ctypes.data, keep.shape[0], _native.MEM_HOST
            out = np.empty((n, 4), dtype=np.uint64)
            ok = np.empty((n,), dtype=np.uint8)
        self._check(self._lib.p252_scalars_from_bytes(self._ctx, ptr, n, self._ptr(out), self._ptr(ok),
                                                      flags | (_native.ASYNC if async_ and flags else 0)))
        return out, ok

    def scalars_to_bytes(self, scalars, async_=False):
        """(n, 4) scalars -> canonical little-endian bytes: (n, 32) uint8 (host) or (n, 4) device tensor."""
        ptr, lead, flags, keep = self._in(scalars, (4,))
        n = lead[0]
        if _is_torch(keep):
            import torch
            out = torch.empty((n, 4), dtype=keep.dtype, device=keep.device)
        else:
            out = np.empty((n, 32), dtype=np.uint8)
        self._check(self._lib.p252_scalars_to_bytes(self._ctx, ptr, n, self._ptr(out),
                                                    flags | (_native.ASYNC if async_ and flags else 0)))
        return out

    def encrypt_batch(self, messages, secrets_uv, nonces, out=None, async_=False):
        """messages (n, L, 4), secrets_uv (n, 2, 4), nonces (n, 4) -> ciphers (n, L+1, 4)."""
        L = int(messages.shape[1])
        mp, lead, flags, mk = self._in(messages, (L, 4))
        n = lead[0]
        sp, l2, f2, sk = self._in(secrets_uv, (2, 4))
        np_, l3, f3, nk = self._in(nonces, (4,))
        if not (flags == f2 == f3):
            raise EngineError(-1, "all buffers must live in the same memory space")
        self._same_lead("secrets_uv", l2, n)
        self._same_lead("nonces", l3, n)
        res = self._out_like(mk, (n, L + 1, 4)) if out is None else self._check_out(out, (n, L + 1, 4), mk)
        self._check(self._lib.p252_encrypt_batch(self._ctx, mp, n, L, sp, np_, self._ptr(res),
                                                 flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def decrypt_batch(self, ciphers, secrets_uv, nonces, async_=False):
        """ciphers (n, L+1, 4) -> (messages (n, L, 4), ok (n,) uint8)."""
        L = int(ciphers.shape[1]) - 1
        cp, lead, flags, ck = self._in(ciphers, (L + 1, 4))
        n = lead[0]
        sp, l2, f2, sk = self._in(secrets_uv, (2, 4))
        np_, l3, f3, nk = self._in(nonces, (4,))
        if not (flags == f2 == f3):
            raise EngineError(-1, "all buffers must live in the same memory space")
        self._same_lead("secrets_uv", l2, n)
        self._same_lead("nonces", l3, n)
        if L < 1:
            raise EngineError(-1, "ciphers must hold at least one message scalar plus the authentication scalar")
        if _is_torch(ck):
            import torch
            msg = torch.empty((n, max(L, 0), 4), dtype=ck.dtype, device=ck.device)
            ok = torch.empty((n,), dtype=torch.uint8, device=ck.device)
        else:
            msg = np.empty((n, max(L, 0), 4), dtype=np.uint64)
            ok = np.empty((n,), dtype=np.uint8)
        # the failure count is written through this pointer after the stream reaches it (immediately for
        # synchronous calls): keep it alive on the engine, read it with last_decrypt_failures()
        self._nfail = ctypes.c_size_t(0)
        self._check(self._lib.p252_decrypt_batch(self._ctx, cp, n, max(L, 0), sp, np_, self._ptr(msg), self._ptr(ok),
                                                 ctypes.byref(self._nfail), flags | (_native.ASYNC if async_ and flags else 0)))
        return msg, ok

    def last_decrypt_failures(self):
        """Items of the last decrypt_batch whose authentication failed (counted on the device for device buffers;
        after an async_ call, sync() first)."""
        return int(getattr(self, "_nfail", ctypes.c_size_t(0)).value)

    # -- arity-4 Merkle tree ----------------------------------------------------------------------
    def merkle4_level(self, children, out=None, async_=False):
        """children (4*m, 4) -> parents (m, 4)."""
        cp, lead, flags, ck = self._in(children, (4,))
        m = lead[0] // 4
        if lead[0] % 4:
            from .errors import IOPatternViolation
            raise IOPatternViolation()
        res = self._out_like(ck, (m, 4)) if out is None else self._check_out(out, (m, 4), ck)
        self._check(self._lib.p252_merkle4_level(self._ctx, cp, m, self._ptr(res),
                                                 flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def tree_nodes(self, n_leaves):
        ni, nl = ctypes.c_size_t(0), ctypes.c_int(0)
        self._check(self._lib.p252_merkle4_tree_nodes(int(n_leaves), ctypes.byref(ni), ctypes.byref(nl)))
        return int(ni.value), int(nl.value)

    def merkle4_build(self, leaves, out=None, async_=False):
        """leaves (4^k, 4) -> all internal nodes bottom-up ((4^k-1)/3, 4); root = last row."""
        lp, lead, flags, lk = self._in(leaves, (4,))
        n_internal, _ = self.tree_nodes(lead[0])
        res = self._out_like(lk, (n_internal, 4)) if out is None else self._check_out(out, (n_internal, 4), lk)
        self._check(self._lib.p252_merkle4_build(self._ctx, lp, lead[0], self._ptr(res),
                                                 flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def merkle_build(self, leaves, arity=4, out=None, async_=False):
        """leaves (arity^k, 4) -> all internal nodes bottom-up, root last; arity 2 (Domain::Merkle2) or 4."""
        lp, lead, flags, lk = self._in(leaves, (4,))
        ni = ctypes.c_size_t(0)
        self._check(self._lib.p252_merkle_tree_nodes(int(arity), lead[0], ctypes.byref(ni), None))
        res = self._out_like(lk, (int(ni.value), 4)) if out is None else self._check_out(out, (int(ni.value), 4), lk)
        self._check(self._lib.p252_merkle_build(self._ctx, int(arity), lp, lead[0], self._ptr(res),
                                                flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    # -- Merkle openings --------------------------------------------------------------------------
    def _idx(self, leaf_idx, like):
        if _is_torch(like):
            if not _is_torch(leaf_idx) or not leaf_idx.is_cuda or leaf_idx.device != like.device or \
                    str(leaf_idx.dtype) not in ("torch.int64", "torch.uint64") or not leaf_idx.is_contiguous() or leaf_idx.dim() != 1:
                raise EngineError(-1, "leaf_idx must be a contiguous 1-D int64/uint64 tensor on %s" % like.device)
            return leaf_idx.data_ptr(), int(leaf_idx.shape[0]), leaf_idx
        a = np.ascontiguousarray(leaf_idx, dtype=np.uint64).reshape(-1)
        return a.ctypes.data, int(a.shape[0]), a

    def merkle_open_batch(self, leaves, nodes, leaf_idx, arity=4, out=None, async_=False):
        """Openings of the leaves `leaf_idx` of the tree (leaves (arity^d, 4), nodes as returned by merkle_build):
        (n, d, arity, 4) -- for every level the whole sibling group of the path node (poseidon-merkle `Opening`)."""
        lp, lead, flags, lk = self._in(leaves, (4,))
        np_, nlead, f2, nk = self._in(nodes, (4,))
        if flags != f2:
            raise EngineError(-1, "all buffers must live in the same memory space")
        ni, nl = ctypes.c_size_t(0), ctypes.c_int(0)
        self._check(self._lib.p252_merkle_tree_nodes(int(arity), lead[0], ctypes.byref(ni), ctypes.byref(nl)))
        self._same_lead("nodes", nlead, int(ni.value))
        ip, n, ik = self._idx(leaf_idx, lk)
        depth = int(nl.value)
        shape = (n, depth, int(arity), 4)
        res = self._out_like(lk, shape) if out is None else self._check_out(out, shape, lk)
        self._check(self._lib.p252_merkle_open_batch(self._ctx, int(arity), lp, lead[0], np_, ip, n, self._ptr(res),
                                                     flags | (_native.ASYNC if async_ and flags else 0)))
        return res

    def merkle_verify_batch(self, leaf_items, leaf_idx, paths, root, arity=4, async_=False):
        """n x Opening::verify.  leaf_items (n, 4), leaf_idx (n,), paths (n, d, arity, 4), root (4,) host array
        -> ok (n,) uint8.  The failure count is available from last_verify_failures()."""
        if paths.ndim != 4 or int(paths.shape[2]) != int(arity):
            raise EngineError(-1, "paths must have shape (n, depth, arity, 4)")
        depth = int(paths.shape[1])
        pp, plead, flags, pk = self._in(paths, (depth, int(arity), 4))
        n = plead[0]
        lp, llead, f2, lk = self._in(leaf_items, (4,))
        if flags != f2:
            raise EngineError(-1, "all buffers must live in the same memory space")
        self._same_lead("leaf_items", llead, n)
        ip, ni, ik = self._idx(leaf_idx, pk)
        if ni != n:
            raise EngineError(-1, "leaf_idx must have %d entries" % n)
        if _is_torch(root):
            root = root.detach().cpu().numpy()
        root = np.ascontiguousarray(root)
        root = (root.view(np.uint64) if root.dtype == np.int64 else root.astype(np.uint64)).reshape(4)
        if _is_torch(pk):
            import torch
            ok = torch.empty((n,), dtype=torch.uint8, device=pk.device)
        else:
            ok = np.empty((n,), dtype=np.uint8)
        self._vfail = ctypes.c_size_t(0)
        self._check(self._lib.p252_merkle_verify_batch(self._ctx, int(arity), depth, lp, ip, pp, root.ctypes.data, n,
                                                       self._ptr(ok), ctypes.byref(self._vfail),
                                                       flags | (_native.ASYNC if async_ and flags else 0)))
        return ok

    def last_verify_failures(self):
        return int(getattr(self, "_vfail", ctypes.c_size_t(0)).value)

    # -- incremental Merkle updates ---------------------------------------------------------------
    def _inplace(self, name, x, rows):
        """A buffer the call writes in place: it must already be exactly what native code writes through (a copy would
        silently lose the update)."""
        if _is_torch(x):
            if not x.is_cuda or x.device.index != self.device:
                raise EngineError(-1, "%s is not on cuda:%d" % (name, self.device))
            ok = str(x.dtype) in ("torch.int64", "torch.uint64") and x.is_contiguous()
        else:
            ok = isinstance(x, np.ndarray) and x.dtype in (np.uint64, np.int64) and x.flags.c_contiguous and \
                x.flags.writeable
        if not ok:
            raise EngineError(-1, "%s must be a writable C-contiguous uint64/int64 array or tensor (updated in place)" % name)
        if tuple(x.shape) != (rows, 4):
            raise EngineError(-1, "%s must have shape (%d, 4), got %s" % (name, rows, tuple(x.shape)))
        return self._ptr(x), (_native.MEM_DEVICE if _is_torch(x) else _native.MEM_HOST)

    def merkle_update_batch(self, leaves, nodes, leaf_idx, values, arity=4, async_=False):
        """Write values[j] to leaf leaf_idx[j] (the last occurrence of a repeated index wins) and rehash only the
        dirty paths, in place: afterwards leaves / nodes equal merkle_build of the updated leaves.  Returns
        (leaves, nodes).  Host arrays: an index outside the tree raises before anything is written.  Device tensors:
        such entries are skipped and counted (last_update_rejected(); after an async_ call, sync() first)."""
        n_leaves = int(leaves.shape[0]) if getattr(leaves, "ndim", 0) == 2 else -1
        ni = ctypes.c_size_t(0)
        if n_leaves < 0:
            raise EngineError(-1, "leaves must have shape (n_leaves, 4)")
        self._check(self._lib.p252_merkle_tree_nodes(int(arity), n_leaves, ctypes.byref(ni), None))
        lp, flags = self._inplace("leaves", leaves, n_leaves)
        np_, f2 = self._inplace("nodes", nodes, int(ni.value))
        if getattr(values, "ndim", 0) != 2:
            raise EngineError(-1, "values must have shape (k, 4)")
        vp, vlead, f3, vk = self._in(values, (4,))
        if not (flags == f2 == f3) or _is_torch(leaf_idx) != _is_torch(leaves):
            raise EngineError(-1, "all buffers must live in the same memory space")
        ip, k, ik = self._idx(leaf_idx, leaves)
        if k != vlead[0]:
            raise EngineError(-1, "leaf_idx has %d entries but values has %d rows" % (k, vlead[0]))
        if flags == _native.MEM_DEVICE:
            self._fence_torch()
        # written after the stream reaches it for device calls: keep it alive on the engine
        self._ufail = ctypes.c_size_t(0)
        self._check(self._lib.p252_merkle_update_batch(self._ctx, int(arity), lp, n_leaves, np_, ip, vp, k,
                                                       ctypes.byref(self._ufail),
                                                       flags | (_native.ASYNC if async_ and flags else 0)))
        return leaves, nodes

    def last_update_rejected(self):
        """Entries of the last merkle_update_batch on device tensors whose leaf index was outside the tree."""
        return int(getattr(self, "_ufail", ctypes.c_size_t(0)).value)

    def set_small_batch_max(self, max_items):
        """Digest batches up to `max_items` items use the lane-split (5 threads per state) kernel; 0 disables it."""
        self._check(self._lib.p252_set_small_batch_max(self._ctx, int(max_items)))

    # -- introspection ----------------------------------------------------------------------------
    def kernel_info(self):
        """p252_get_kernel_info as a dict (multiplier / DFMA instructions per permutation, launch shape)."""
        info = _native.KernelInfo()
        info.struct_size = ctypes.sizeof(info)
        self._check(self._lib.p252_get_kernel_info(ctypes.byref(info)))
        return {k: int(getattr(info, k)) for k, _ in info._fields_ if k != "struct_size"}

    def tree_level_timings(self):
        """Per-level device times of the last merkle4_build_dist(timing=True): (list of dicts, total_ms)."""
        arr = (_native.LevelTiming * 64)()
        n, total = ctypes.c_int(0), ctypes.c_float(0)
        self._check(self._lib.p252_tree_level_timings(self._ctx, arr, 64, ctypes.byref(n), ctypes.byref(total)))
        return [{k: (float(getattr(arr[i], k)) if k.endswith("_ms") else int(getattr(arr[i], k))) for k, _ in arr[i]._fields_}
                for i in range(n.value)], float(total.value)

    # -- multi-GPU (one process per GPU) ----------------------------------------------------------
    def dist_unique_id(self):
        buf = (ctypes.c_uint8 * _native.NCCL_UNIQUE_ID_BYTES)()
        self._check(self._lib.p252_dist_unique_id(buf))
        return bytes(buf)

    def dist_init(self, unique_id, rank, nranks):
        buf = (ctypes.c_uint8 * _native.NCCL_UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self._lib.p252_dist_init(self._ctx, buf, int(rank), int(nranks)))
        self._dist = True

    def dist_finalize(self):
        if self._dist:
            self._check(self._lib.p252_dist_finalize(self._ctx))
            self._dist = False

    def merkle4_build_dist(self, leaves_shard, n_leaves_total, out=None, async_=False, timing=False, no_gather=False):
        """This rank's contiguous shard of the leaves (device tensor) -> complete internal levels
        on every rank (one NCCL all-gather per level)."""
        lp, lead, flags, lk = self._in(leaves_shard, (4,))
        if flags != _native.MEM_DEVICE:
            raise EngineError(-1, "merkle4_build_dist takes device tensors")
        n_internal, _ = self.tree_nodes(n_leaves_total)
        res = self._out_like(lk, (n_internal, 4)) if out is None else self._check_out(out, (n_internal, 4), lk)
        self._check(self._lib.p252_merkle4_build_dist(self._ctx, lp, int(n_leaves_total), self._ptr(res),
                                                      flags | (_native.ASYNC if async_ else 0) |
                                                      (_native.TIMING if timing else 0) | (_native.NO_GATHER if no_gather else 0)))
        return res


def default_engine(device=0):
    """Process-wide engine per device (created on first use)."""
    if device not in _DEFAULT:
        _DEFAULT[device] = Engine(device)
    return _DEFAULT[device]
