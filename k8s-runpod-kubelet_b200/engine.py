"""``Engine`` -- thin Python host wrapper over the C-ABI (``include/rpk.h``).

It adds nothing to the computation: numpy columns in (host entry points) or torch CUDA tensors in (device
entry points), the C library does the rest on the GPU.  Method names follow the reference's vocabulary:
``upload_offers`` replaces the per-pod GraphQL decode of ``gpuTypes`` (runpod_client.go:447-455), ``select``
replaces the body of ``GetGPUTypes`` (:465-509) for a whole batch of pods, ``status_diff`` replaces the diff
predicate of ``updateAllPodStatuses`` (kubelet.go:857-880).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _ffi


def _np_ptr(a, dtype, n=None, name="array"):
    if a is None:
        return None
    if not isinstance(a, np.ndarray) or a.dtype != dtype or not a.flags.c_contiguous:
        raise TypeError(f"{name}: expected a C-contiguous numpy array of {np.dtype(dtype).name}")
    if n is not None and a.size != n:
        raise ValueError(f"{name}: expected {n} elements, got {a.size}")
    return C.c_void_p(a.ctypes.data)


def _dev_ptr(t, dtype_name, n=None, name="tensor"):
    """torch CUDA tensor -> raw device pointer (torch is only the allocator here)."""
    if t is None:
        return None
    import torch

    want = getattr(torch, dtype_name)
    if not t.is_cuda or t.dtype != want or not t.is_contiguous():
        raise TypeError(f"{name}: expected a contiguous CUDA tensor of {dtype_name}")
    if n is not None and t.numel() != n:
        raise ValueError(f"{name}: expected {n} elements, got {t.numel()}")
    return C.c_void_p(t.data_ptr())


def pack_offer_sets(members) -> np.ndarray:
    """bool ``(n_sets, G)`` -> uint32 ``(n_sets, ceil(G/32))`` membership words of rpk_offer_sets_upload: offer g of set
    s is bit ``g & 31`` of word ``g // 32`` (little-endian bit and byte order)."""
    m = np.asarray(members, dtype=bool)
    if m.ndim != 2:
        raise ValueError("members: expected a (n_sets, G) bool array")
    n_sets, G = m.shape
    W = (G + 31) // 32
    b = np.packbits(m, axis=1, bitorder="little")
    out = np.zeros((n_sets, W * 4), np.uint8)
    out[:, : b.shape[1]] = b
    return np.ascontiguousarray(out.view("<u4").astype(np.uint32, copy=False))


class Engine:
    """One ``rpk_ctx``.  ``n_gpus > 1`` = one process driving several GPUs (the Go kubelet's shape)."""

    def __init__(self, n_gpus: int = 1, device_ids=None):
        self._lib = _ffi.load()
        self._ctx = C.c_void_p()
        ids = None
        if device_ids is not None:
            ids = (C.c_int * len(device_ids))(*device_ids)
            n_gpus = len(device_ids)
        rc = self._lib.rpk_create(n_gpus, ids, C.byref(self._ctx))
        if rc != 0:
            msg = self._lib.rpk_last_error(None)
            self._ctx = C.c_void_p()
            raise _ffi.RpkError(rc, (msg or b"").decode())
        self.n_gpus = n_gpus
        self.G = 0

    # -- plumbing ------------------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise _ffi.RpkError(rc, (self._lib.rpk_last_error(self._ctx) or b"").decode())

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.rpk_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def stats(self) -> dict:
        s = _ffi.RpkStats()
        self._check(self._lib.rpk_stats_get(self._ctx, C.byref(s)))
        return {k: getattr(s, k) for k, _ in s._fields_}

    def launch_count(self) -> int:
        return int(self._lib.rpk_launch_count(self._ctx))

    # -- offers --------------------------------------------------------------------------------------
    def upload_offers(self, offers: dict):
        G = int(offers["mem_gb"].shape[0])
        self._check(self._lib.rpk_offers_upload(
            self._ctx, G, _np_ptr(offers["mem_gb"], np.int32, G, "mem_gb"), _np_ptr(offers.get("vcpu"), np.int32, G, "vcpu"),
            _np_ptr(offers.get("ram_gb"), np.int32, G, "ram_gb"), _np_ptr(offers["secure_price"], np.float64, G, "secure_price"),
            _np_ptr(offers["community_price"], np.float64, G, "community_price"), _np_ptr(offers["flags"], np.uint8, G, "flags")))
        self.G = G

    # -- selection -----------------------------------------------------------------------------------
    def select(self, pods: dict, want_top5: bool = False, out_best=None, out_top5=None):
        """Host columns in, ``(best[P], top5[P,5] | None)`` out (numpy)."""
        P = int(pods["req_mem_gb"].shape[0])
        best = out_best if out_best is not None else np.empty(P, np.int32)
        top5 = (out_top5 if out_top5 is not None else np.empty((P, 5), np.int32)) if want_top5 else None
        self._check(self._lib.rpk_select(
            self._ctx, P, _np_ptr(pods["req_mem_gb"], np.int32, P, "req_mem_gb"), _np_ptr(pods.get("req_vcpu"), np.int32, P, "req_vcpu"),
            _np_ptr(pods.get("req_ram_gb"), np.int32, P, "req_ram_gb"), _np_ptr(pods.get("max_price"), np.float64, P, "max_price"),
            _np_ptr(pods.get("cloud"), np.uint8, P, "cloud"), _np_ptr(best, np.int32, P, "best"),
            _np_ptr(top5, np.int32, P * 5, "top5") if top5 is not None else None))
        return best, top5

    def select_device(self, pods: dict, d_best, d_top5=None, shard: int = 0, stream=None):
        """torch CUDA columns in, result enqueued on ``stream`` (default: torch's current stream)."""
        import torch

        P = int(pods["req_mem_gb"].numel())
        st = stream if stream is not None else (torch.cuda.current_stream().cuda_stream or 1)  # 0 -> cudaStreamLegacy
        self._check(self._lib.rpk_select_device(
            self._ctx, shard, P, _dev_ptr(pods["req_mem_gb"], "int32", P), _dev_ptr(pods.get("req_vcpu"), "int32", P),
            _dev_ptr(pods.get("req_ram_gb"), "int32", P), _dev_ptr(pods.get("max_price"), "float64", P),
            _dev_ptr(pods.get("cloud"), "uint8", P), _dev_ptr(d_best, "int32", P), _dev_ptr(d_top5, "int32", P * 5),
            C.c_void_p(st)))

    def select_device_gather(self, pods: dict, full_ptrs, row0: int, d_top5=None, shard: int = 0, stream=None):
        """Shard + fused all-gather: results land at [row0, row0+P) of every vector in ``full_ptrs`` (raw
        device pointers: own vector first or anywhere, peers' via IPC / peer access)."""
        import torch

        P = int(pods["req_mem_gb"].numel())
        st = stream if stream is not None else (torch.cuda.current_stream().cuda_stream or 1)  # 0 -> cudaStreamLegacy
        arr = (C.c_void_p * len(full_ptrs))(*[C.c_void_p(int(p)) for p in full_ptrs])
        self._check(self._lib.rpk_select_device_gather(
            self._ctx, shard, P, _dev_ptr(pods["req_mem_gb"], "int32", P), _dev_ptr(pods.get("req_vcpu"), "int32", P),
            _dev_ptr(pods.get("req_ram_gb"), "int32", P), _dev_ptr(pods.get("max_price"), "float64", P),
            _dev_ptr(pods.get("cloud"), "uint8", P), len(full_ptrs), arr, row0, _dev_ptr(d_top5, "int32", P * 5),
            C.c_void_p(st)))

    # -- offer sets ----------------------------------------------------------------------------------------
    def upload_offer_sets(self, members):
        """``members``: bool ``(n_sets, G)`` -- row s marks the offers of set s (``G`` = the resident table's).
        Replaces every previous set; ``n_sets = 0`` clears them (rpk_offer_sets_upload)."""
        words = pack_offer_sets(members)
        n_sets, G = np.asarray(members).shape
        self._check(self._lib.rpk_offer_sets_upload(self._ctx, n_sets, G, C.c_void_p(words.ctypes.data) if words.size else None))

    def select_sets(self, pods: dict, set_id, want_top5: bool = False):
        """``select`` with every row restricted to offer set ``set_id[p]`` (uint16; ``RPK_SET_ALL`` = the whole table,
        ``None`` = every row unrestricted).  -> ``(best[P], top5[P,5] | None)``"""
        P = int(pods["req_mem_gb"].shape[0])
        best = np.empty(P, np.int32)
        top5 = np.empty((P, 5), np.int32) if want_top5 else None
        self._check(self._lib.rpk_select_sets(
            self._ctx, P, _np_ptr(pods["req_mem_gb"], np.int32, P, "req_mem_gb"), _np_ptr(pods.get("req_vcpu"), np.int32, P, "req_vcpu"),
            _np_ptr(pods.get("req_ram_gb"), np.int32, P, "req_ram_gb"), _np_ptr(pods.get("max_price"), np.float64, P, "max_price"),
            _np_ptr(pods.get("cloud"), np.uint8, P, "cloud"), _np_ptr(set_id, np.uint16, P, "set_id"), _np_ptr(best, np.int32, P, "best"),
            _np_ptr(top5, np.int32, P * 5, "top5") if top5 is not None else None))
        return best, top5

    def select_sets_device(self, pods: dict, d_set_id, d_best, d_top5=None, shard: int = 0, stream=None):
        """torch CUDA columns in (``d_set_id`` int16 holding the uint16 ids, or None), results enqueued on ``stream``;
        the call synchronises the stream once to read the per-set row counts."""
        import torch

        P = int(pods["req_mem_gb"].numel())
        st = stream if stream is not None else (torch.cuda.current_stream().cuda_stream or 1)  # 0 -> cudaStreamLegacy
        if d_set_id is not None and (not d_set_id.is_cuda or d_set_id.element_size() != 2 or not d_set_id.is_contiguous()
                                     or d_set_id.numel() != P):
            raise TypeError("d_set_id: expected a contiguous CUDA tensor of P 16-bit ids (torch.int16 / torch.uint16)")
        self._check(self._lib.rpk_select_sets_device(
            self._ctx, shard, P, _dev_ptr(pods["req_mem_gb"], "int32", P), _dev_ptr(pods.get("req_vcpu"), "int32", P),
            _dev_ptr(pods.get("req_ram_gb"), "int32", P), _dev_ptr(pods.get("max_price"), "float64", P),
            _dev_ptr(pods.get("cloud"), "uint8", P), C.c_void_p(d_set_id.data_ptr()) if d_set_id is not None else None,
            _dev_ptr(d_best, "int32", P), _dev_ptr(d_top5, "int32", P * 5), C.c_void_p(st)))

    # -- cross-process peer vectors (CUDA IPC) ------------------------------------------------------------
    def ipc_alloc(self, nbytes: int, shard: int = 0):
        """-> (device pointer, 64-byte handle) of a fresh cudaMalloc buffer other processes can map."""
        ptr = C.c_void_p()
        handle = C.create_string_buffer(64)
        self._check(self._lib.rpk_ipc_alloc(self._ctx, shard, nbytes, C.byref(ptr), handle))
        return int(ptr.value), handle.raw

    def ipc_open(self, handle: bytes, shard: int = 0) -> int:
        ptr = C.c_void_p()
        self._check(self._lib.rpk_ipc_open(self._ctx, shard, handle, C.byref(ptr)))
        return int(ptr.value)

    def peer_fence(self, flag_ptrs, my_rank: int, epoch: int, shard: int = 0, stream=None):
        """Signal every peer and wait for every peer on ``stream`` (one tiny kernel; see rpk_peer_fence)."""
        import torch

        st = stream if stream is not None else (torch.cuda.current_stream().cuda_stream or 1)
        arr = (C.c_void_p * len(flag_ptrs))(*[C.c_void_p(int(p)) for p in flag_ptrs])
        self._check(self._lib.rpk_peer_fence(self._ctx, shard, len(flag_ptrs), arr, my_rank, epoch & 0xFFFFFFFF, C.c_void_p(st)))

    def peer_bind(self, flag_ptrs, my_rank: int, shard: int = 0):
        """Bind the peer group's flag arrays: gathers on this shard signal by themselves from now on (rpk_peer_bind)."""
        n = len(flag_ptrs) if flag_ptrs else 0
        arr = (C.c_void_p * max(n, 1))(*[C.c_void_p(int(p)) for p in (flag_ptrs or [])])
        self._check(self._lib.rpk_peer_bind(self._ctx, shard, n, arr, my_rank))

    def peer_inline_wait(self, on: bool = True, shard: int = 0):
        """Bound gathers also wait for every peer's signal before they complete (no rpk_peer_wait launch needed)."""
        self._check(self._lib.rpk_peer_inline_wait(self._ctx, shard, 1 if on else 0))

    def peer_wait(self, what: int = 1, shard: int = 0, stream=None):
        """The wait half of the fence (bit 0: select gather, bit 1: status gather)."""
        import torch

        st = stream if stream is not None else (torch.cuda.current_stream().cuda_stream or 1)
        self._check(self._lib.rpk_peer_wait(self._ctx, shard, what, C.c_void_p(st)))

    def best_device_ptr(self, shard: int = 0) -> int:
        return int(self._lib.rpk_best_device_ptr(self._ctx, shard) or 0)

    # -- status sweep --------------------------------------------------------------------------------
    def status_reset(self, N: int):
        self._check(self._lib.rpk_status_reset(self._ctx, N))

    def status_seed(self, records: np.ndarray):
        N, stride = records.shape
        self._check(self._lib.rpk_status_seed(self._ctx, N, _np_ptr(records, np.uint8, N * stride, "records"), stride))

    def status_diff(self, records: np.ndarray, want_hashes: bool = False, want_codes: bool = False):
        """-> (changed_idx ascending, hashes | None) or, with ``want_codes``, (changed_idx, codes, hashes | None)"""
        N, stride = records.shape
        idx = np.empty(max(N, 1), np.uint32)
        codes = np.empty(max(N, 1), np.uint16) if want_codes else None
        n = C.c_uint32(0)
        hashes = np.empty(N, np.uint64) if want_hashes else None
        self._check(self._lib.rpk_status_diff_codes(
            self._ctx, N, _np_ptr(records, np.uint8, N * stride, "records"), stride, C.c_void_p(idx.ctypes.data),
            C.c_void_p(codes.ctypes.data) if want_codes else None, C.cast(C.byref(n), C.c_void_p),
            _np_ptr(hashes, np.uint64, N, "hashes") if want_hashes else None))
        if want_codes:
            return idx[: n.value].copy(), codes[: n.value].copy(), hashes
        return idx[: n.value].copy(), hashes

    def status_seed_slots(self, slots: np.ndarray, records: np.ndarray):
        """Previous state of individual slots (records[i] -> slot slots[i]); nothing is reported."""
        n, stride = records.shape
        slots = np.ascontiguousarray(slots, np.uint32)  # keep the converted array alive across the call
        self._check(self._lib.rpk_status_seed_slots(self._ctx, n, _np_ptr(slots, np.uint32, n, "slots"),
                                                    _np_ptr(records, np.uint8, n * stride, "records"), stride))

    def tick(self, pods: dict | None, records: np.ndarray, want_top5: bool = False, want_codes: bool = True, out_best=None):
        """One kubelet tick: selection over ``pods`` (None: none pending) and the status sweep over ``records`` enqueued
        together (rpk_tick).  -> (best | None, top5 | None, changed_idx, codes | None)"""
        N, stride = records.shape
        P = int(pods["req_mem_gb"].shape[0]) if pods else 0
        best = (out_best if out_best is not None else np.empty(P, np.int32)) if P else None
        top5 = np.empty((P, 5), np.int32) if (want_top5 and P) else None
        idx = np.empty(max(N, 1), np.uint32)
        codes = np.empty(max(N, 1), np.uint16) if want_codes else None
        n = C.c_uint32(0)
        g = (lambda k, dt: _np_ptr(pods.get(k), dt, P, k)) if P else (lambda k, dt: None)
        self._check(self._lib.rpk_tick(
            self._ctx, P, g("req_mem_gb", np.int32), g("req_vcpu", np.int32), g("req_ram_gb", np.int32), g("max_price", np.float64),
            g("cloud", np.uint8), _np_ptr(best, np.int32, P, "best") if P else None, _np_ptr(top5, np.int32, P * 5, "top5") if top5 is not None else None,
            N, _np_ptr(records, np.uint8, N * stride, "records"), stride, C.c_void_p(idx.ctypes.data),
            C.c_void_p(codes.ctypes.data) if want_codes else None, C.cast(C.byref(n), C.c_void_p)))
        return best, top5, idx[: n.value].copy(), (codes[: n.value].copy() if want_codes else None)

    def status_diff_device(self, d_records, stride: int, d_hash_prev, d_changed_idx, d_n_changed, shard: int = 0, stream=None,
                           d_changed_code=None):
        import torch

        N = int(d_hash_prev.numel())
        st = stream if stream is not None else (torch.cuda.current_stream().cuda_stream or 1)  # 0 -> cudaStreamLegacy
        self._check(self._lib.rpk_status_diff_device_codes(
            self._ctx, shard, N, _dev_ptr(d_records, "uint8", N * stride), stride, C.c_void_p(d_hash_prev.data_ptr()),
            C.c_void_p(d_changed_idx.data_ptr()), C.c_void_p(d_changed_code.data_ptr()) if d_changed_code is not None else None,
            C.c_void_p(d_n_changed.data_ptr()), C.c_void_p(st)))

    def xchg_bytes(self, n_ranks: int, cap: int) -> int:
        return int(self._lib.rpk_xchg_bytes(n_ranks, cap))

    def status_diff_device_gather(self, d_records, stride: int, d_hash_prev, idx_base: int, xchg_ptrs, cap: int, my_rank: int,
                                  d_n_changed, shard: int = 0, stream=None):
        """Sharded sweep: this rank's changed list (count, global ids, codes) lands in region ``my_rank`` of every
        rank's exchange buffer (rpk_status_diff_device_gather)."""
        import torch

        N = int(d_hash_prev.numel())
        st = stream if stream is not None else (torch.cuda.current_stream().cuda_stream or 1)
        arr = (C.c_void_p * len(xchg_ptrs))(*[C.c_void_p(int(p)) for p in xchg_ptrs])
        self._check(self._lib.rpk_status_diff_device_gather(
            self._ctx, shard, N, _dev_ptr(d_records, "uint8", N * stride), stride, C.c_void_p(d_hash_prev.data_ptr()), idx_base,
            len(xchg_ptrs), arr, cap, my_rank, C.c_void_p(d_n_changed.data_ptr()), C.c_void_p(st)))
