"""ctypes binding of the C ABI (include/ibft_verify.h) -- the same entry points the cgo Backend binds.

PyTorch is used by callers only for device memory / streams / torch.distributed; this module passes raw pointers.
There is no CPU fallback: constructing an Engine without a CUDA device raises EngineError.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_size_t, c_uint8, c_uint16, c_uint32, c_uint64, c_void_p

import numpy as np

from . import build as _build

IBFT_OK, ERR_INVALID_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_CAPACITY, ERR_VOTING_POWER, ERR_NO_TABLE = range(7)
KIND_DIGEST, KIND_PAYLOAD, KIND_SEAL, KIND_WIRE, KIND_WIRE_SEAL, KIND_PAYLOAD2, KIND_INVALID = 0, 1, 2, 3, 4, 5, 255
ITEM_OK, ITEM_NEEDS_HOST = 0, 1
NO_TABLE = 0xFFFF
DBG = dict(FE_MUL=1, FE_SQR=2, FE_INV=3, FE_SQRT=4, SC_MUL=5, SC_INV=6, ECMULT=7, FE_ADD=8, FE_SUB=9, GLV=10)

# numpy mirrors of the ABI structs
ITEM_DTYPE = np.dtype([
    ("r", "u1", 32), ("s", "u1", 32), ("digest", "u1", 32), ("signer", "u1", 20),
    ("v", "u1"), ("kind", "u1"), ("group", "<u2"), ("payload_off", "<u4"), ("payload_len", "<u4"),
])
GROUP_DTYPE = np.dtype([("table_slot", "<u2"), ("flags", "<u2"), ("reserved", "<u4"), ("height", "<u8")])
RESULT_DTYPE = np.dtype([("power", "<u8", 5), ("n_valid", "<u4"), ("n_distinct", "<u4"), ("has_quorum", "<u4"), ("reserved", "<u4")])
assert ITEM_DTYPE.itemsize == 128 and GROUP_DTYPE.itemsize == 16 and RESULT_DTYPE.itemsize == 56

EXPORTS = [
    "ibft_abi_version", "ibft_last_error", "ibft_engine_create", "ibft_engine_destroy", "ibft_engine_device_info",
    "ibft_set_validators", "ibft_get_quorum", "ibft_verify_batch", "ibft_verify_batch_ex", "ibft_last_item_status", "ibft_verify_submit", "ibft_verify_poll",
    "ibft_verify_wait", "ibft_bind_groups", "ibft_verify_batch_device", "ibft_quorum_reduce_device", "ibft_quorum_partial_words", "ibft_quorum_mark_device", "ibft_quorum_merge_device", "ibft_quorum_exchange_device",
    "ibft_exchange_alloc", "ibft_exchange_open", "ibft_exchange_close", "ibft_exchange_free", "ibft_exchange_clear",
    "ibft_get_voted_bitmap", "ibft_keccak256_batch", "ibft_proposal_hash_batch", "ibft_sign_batch", "ibft_engine_launch_count", "ibft_set_recover_path", "ibft_refresh_key_tables", "ibft_probe_int_peak", "ibft_debug_op", "ibft_debug_ctable",
    "ibft_debug_keytab", "ibft_debug_last_deferred",
]


class EngineParams(ctypes.Structure):
    _fields_ = [("device", c_int32), ("max_items", c_uint32), ("max_payload_bytes", c_uint32), ("max_groups", c_uint32),
                ("max_table_slots", c_uint32), ("max_validators", c_uint32), ("flags", c_uint32)]


class DeviceInfo(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char * 64), ("sm_count", c_int32), ("cc_major", c_int32), ("cc_minor", c_int32),
                ("clock_khz", c_int32), ("total_mem", c_uint64), ("abi_version", c_int32), ("kernel_regs", c_int32),
                ("kernel_smem_bytes", c_int32), ("block_threads", c_int32)]


class EngineError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"ibft engine error {code}: {msg}")
        self.code = code


_LIB = None


def load_library(path: str | None = None) -> ctypes.CDLL:
    """Load (building if needed) libibftverify.so and declare the prototypes."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    so = path or os.environ.get("IBFT_LIB") or _build.build()  # IBFT_LIB: kernel-variant experiments (tools/quick_bench.py)
    lib = ctypes.CDLL(so)
    lib.ibft_last_error.restype = c_char_p
    lib.ibft_refresh_key_tables.restype = c_int
    lib.ibft_refresh_key_tables.argtypes = [c_void_p, POINTER(c_uint32)]
    lib.ibft_set_recover_path.restype = c_int
    lib.ibft_set_recover_path.argtypes = [c_void_p, c_int]
    lib.ibft_engine_launch_count.restype = c_uint64
    lib.ibft_engine_launch_count.argtypes = [c_void_p]
    lib.ibft_engine_create.argtypes = [POINTER(EngineParams), POINTER(c_void_p)]
    lib.ibft_engine_destroy.argtypes = [c_void_p]
    lib.ibft_engine_destroy.restype = None
    lib.ibft_engine_device_info.argtypes = [c_void_p, POINTER(DeviceInfo)]
    lib.ibft_set_validators.argtypes = [c_void_p, c_uint32, c_uint64, c_void_p, c_void_p, c_uint32]
    lib.ibft_get_quorum.argtypes = [c_void_p, c_uint32, POINTER(c_uint64), POINTER(c_uint64), POINTER(c_uint32)]
    for name in ("ibft_verify_batch", "ibft_verify_submit"):
        getattr(lib, name).argtypes = [c_void_p, c_void_p, c_uint32, c_void_p, c_size_t, c_void_p, c_uint32, c_void_p, c_void_p, c_void_p]
    lib.ibft_verify_batch_ex.argtypes = [c_void_p, c_void_p, c_uint32, c_void_p, c_size_t, c_void_p, c_uint32, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_uint32]
    lib.ibft_last_item_status.argtypes = [c_void_p, c_void_p, c_uint32]
    lib.ibft_verify_poll.argtypes = [c_void_p, POINTER(c_int)]
    lib.ibft_verify_wait.argtypes = [c_void_p]
    lib.ibft_bind_groups.argtypes = [c_void_p, c_void_p, c_uint32]
    lib.ibft_verify_batch_device.argtypes = [c_void_p, c_void_p, c_uint32, c_void_p, c_size_t, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p]
    lib.ibft_quorum_reduce_device.argtypes = [c_void_p, c_void_p, c_uint32, c_void_p, c_void_p, c_uint32, c_void_p, c_void_p]
    lib.ibft_quorum_partial_words.argtypes = [c_void_p, POINTER(c_uint32)]
    lib.ibft_quorum_mark_device.argtypes = [c_void_p, c_void_p, c_uint32, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p]
    lib.ibft_quorum_merge_device.argtypes = [c_void_p, c_void_p, c_uint32, c_uint32, c_void_p, c_void_p]
    lib.ibft_quorum_exchange_device.argtypes = [c_void_p, c_void_p, c_uint32, c_uint32, c_uint32, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.ibft_exchange_alloc.argtypes = [c_void_p, c_uint32, POINTER(c_void_p), c_void_p]
    lib.ibft_exchange_open.argtypes = [c_void_p, c_void_p, POINTER(c_void_p)]
    lib.ibft_exchange_close.argtypes = [c_void_p, c_void_p]
    lib.ibft_exchange_free.argtypes = [c_void_p, c_void_p]
    lib.ibft_exchange_clear.argtypes = [c_void_p, c_void_p, c_uint32, c_uint32, c_void_p]
    lib.ibft_get_voted_bitmap.argtypes = [c_void_p, c_uint32, c_void_p, c_uint32]
    lib.ibft_keccak256_batch.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_uint32, c_void_p]
    lib.ibft_proposal_hash_batch.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_uint32, c_void_p]
    lib.ibft_sign_batch.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_uint32, c_void_p]
    lib.ibft_probe_int_peak.argtypes = [c_void_p, POINTER(c_double), POINTER(c_double)]
    lib.ibft_debug_ctable.argtypes = [c_void_p, c_uint32, c_uint32, c_void_p, POINTER(c_int), POINTER(c_uint32)]
    lib.ibft_debug_op.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_uint32, c_void_p, c_uint32]
    lib.ibft_debug_keytab.argtypes = [c_void_p, c_uint32, c_uint32, c_uint32, c_uint32, c_void_p, POINTER(c_uint32)]
    lib.ibft_debug_last_deferred.argtypes = [c_void_p, POINTER(c_uint32)]
    if path is None:
        _LIB = lib
    return lib


def _ptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(c_void_p)


class Engine:
    """One engine per process per GPU (one process per GPU is the deployment model)."""

    def __init__(self, device: int = 0, max_items: int = 1 << 16, max_payload_bytes: int = 1 << 24, max_groups: int = 64,
                 max_table_slots: int = 16, max_validators: int = 16384, key_cache: bool = False):
        """key_cache: IBFT_FLAG_KEY_CACHE -- verify (instead of recover) signatures of validators whose key is already known."""
        self.lib = load_library()
        self.params = EngineParams(device, max_items, max_payload_bytes, max_groups, max_table_slots, max_validators, 1 if key_cache else 0)
        self.handle = c_void_p()
        self.slot_height: dict[int, int] = {}  # slot -> height of the resident validator table (mirrors the engine's own record)
        rc = self.lib.ibft_engine_create(ctypes.byref(self.params), ctypes.byref(self.handle))
        if rc != IBFT_OK:
            self.handle = None
            raise EngineError(rc, self.lib.ibft_last_error().decode())

    def close(self):
        if getattr(self, "handle", None):
            self.lib.ibft_engine_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != IBFT_OK:
            raise EngineError(rc, self.lib.ibft_last_error().decode())

    # ---- info / probes
    def device_info(self) -> dict:
        di = DeviceInfo()
        self._check(self.lib.ibft_engine_device_info(self.handle, ctypes.byref(di)))
        return {f: (getattr(di, f).decode() if f == "name" else getattr(di, f)) for f, _ in DeviceInfo._fields_}

    PATH_AUTO, PATH_THREAD, PATH_QUAD, PATH_SPLIT, PATH_QSPLIT = 0, 1, 2, 3, 4

    def set_recover_path(self, path: int) -> None:
        """Kernel selection of the recover step (include/ibft_verify.h IBFT_PATH_*): verdicts are identical on every path."""
        self._check(self.lib.ibft_set_recover_path(self.handle, int(path)))

    def refresh_key_tables(self) -> int:
        """Key registry upkeep (engine flag key_cache): returns the number of validator keys known so far."""
        n = c_uint32(0)
        self._check(self.lib.ibft_refresh_key_tables(self.handle, ctypes.byref(n)))
        return int(n.value)

    def launch_count(self) -> int:
        return int(self.lib.ibft_engine_launch_count(self.handle))

    def probe_int_peak(self):
        a, b = c_double(), c_double()
        self._check(self.lib.ibft_probe_int_peak(self.handle, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    # ---- validator tables (ValidatorManager.Init / Backend.GetVotingPowers)
    def set_validators(self, slot: int, height: int, addrs: np.ndarray, powers_be: np.ndarray | None = None):
        addrs = np.ascontiguousarray(addrs, dtype=np.uint8).reshape(-1, 20)
        if powers_be is not None:
            powers_be = np.ascontiguousarray(powers_be, dtype=np.uint8).reshape(-1, 32)
            assert len(powers_be) == len(addrs)
        self._check(self.lib.ibft_set_validators(self.handle, slot, height, _ptr(addrs) if len(addrs) else None,
                                                 _ptr(powers_be), len(addrs)))
        self.slot_height[slot] = height

    def groups(self, n_groups: int, slot=0) -> np.ndarray:
        """n group descriptors; `slot` is one slot for all groups or a sequence of slots.  Each group carries the height of the
        table resident in its slot (ibft_group_desc.height: a group for another height is refused with ERR_NO_TABLE)."""
        g = np.zeros(n_groups, dtype=GROUP_DTYPE)
        slots = [slot] * n_groups if np.isscalar(slot) else list(slot)
        for i, sl in enumerate(slots):
            g[i]["table_slot"] = sl
            g[i]["height"] = self.slot_height.get(int(sl), 0) if sl != NO_TABLE else 0
        return g

    def get_quorum(self, slot: int):
        q = (c_uint64 * 5)()
        h, n = c_uint64(), c_uint32()
        self._check(self.lib.ibft_get_quorum(self.handle, slot, q, ctypes.byref(h), ctypes.byref(n)))
        return sum(int(q[i]) << (64 * i) for i in range(5)), int(h.value), int(n.value)

    # ---- host-buffer verify (the e2e call)
    def verify_batch_ex(self, items: np.ndarray, arena: bytes | np.ndarray = b"", groups: np.ndarray | None = None,
                        voted_stride_words: int = 0):
        """ibft_verify_batch_ex: returns (bitmap, results, status, voted) -- everything from the call itself (concurrent callers)."""
        items = np.ascontiguousarray(items)
        assert items.dtype == ITEM_DTYPE
        n = len(items)
        arena_np = np.frombuffer(arena, dtype=np.uint8) if isinstance(arena, (bytes, bytearray)) else np.ascontiguousarray(arena, dtype=np.uint8)
        bitmap = np.zeros(max(1, (n + 31) // 32), dtype=np.uint32)
        ng = 0 if groups is None else len(groups)
        if groups is not None:
            groups = np.ascontiguousarray(groups)
            assert groups.dtype == GROUP_DTYPE
        results = np.zeros(ng, dtype=RESULT_DTYPE) if ng else None
        status = np.zeros(max(1, n), dtype=np.uint8)
        voted = np.zeros((ng, voted_stride_words), dtype=np.uint32) if (ng and voted_stride_words) else None
        self._check(self.lib.ibft_verify_batch_ex(self.handle, _ptr(items) if n else None, n,
                                                  _ptr(arena_np) if len(arena_np) else None, len(arena_np),
                                                  _ptr(groups) if ng else None, ng, _ptr(bitmap), _ptr(results), None,
                                                  _ptr(status), _ptr(voted), voted_stride_words))
        return bitmap[: (n + 31) // 32], results, status[:n], voted

    def verify_batch(self, items: np.ndarray, arena: bytes | np.ndarray = b"", groups: np.ndarray | None = None,
                     want_results: bool = True, want_recovered: bool = False):
        items = np.ascontiguousarray(items)
        assert items.dtype == ITEM_DTYPE
        n = len(items)
        arena_np = np.frombuffer(arena, dtype=np.uint8) if isinstance(arena, (bytes, bytearray)) else np.ascontiguousarray(arena, dtype=np.uint8)
        bitmap = np.zeros(max(1, (n + 31) // 32), dtype=np.uint32)
        ng = 0 if groups is None else len(groups)
        if groups is not None:
            groups = np.ascontiguousarray(groups)
            assert groups.dtype == GROUP_DTYPE
        results = np.zeros(ng, dtype=RESULT_DTYPE) if (ng and want_results) else None
        recovered = np.zeros((n, 20), dtype=np.uint8) if want_recovered else None
        self._check(self.lib.ibft_verify_batch(self.handle, _ptr(items) if n else None, n,
                                               _ptr(arena_np) if len(arena_np) else None, len(arena_np),
                                               _ptr(groups) if ng else None, ng, _ptr(bitmap), _ptr(results), _ptr(recovered)))
        return bitmap[: (n + 31) // 32], results, recovered

    def last_item_status(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=np.uint8)
        self._check(self.lib.ibft_last_item_status(self.handle, _ptr(out) if n else None, n))
        return out

    def verify_submit(self, items, arena, groups, bitmap, results, recovered=None):
        """Async variant; caller owns (and keeps alive) the output arrays until wait()."""
        n, ng = len(items), 0 if groups is None else len(groups)
        arena_np = np.frombuffer(arena, dtype=np.uint8) if isinstance(arena, (bytes, bytearray)) else arena
        self._check(self.lib.ibft_verify_submit(self.handle, _ptr(items) if n else None, n,
                                                _ptr(arena_np) if len(arena_np) else None, len(arena_np),
                                                _ptr(groups) if ng else None, ng, _ptr(bitmap), _ptr(results), _ptr(recovered)))

    def poll(self) -> bool:
        d = c_int()
        self._check(self.lib.ibft_verify_poll(self.handle, ctypes.byref(d)))
        return bool(d.value)

    def wait(self):
        self._check(self.lib.ibft_verify_wait(self.handle))

    # ---- device-resident path (pointers are ints: torch tensor.data_ptr(); stream: torch stream .cuda_stream)
    def bind_groups(self, groups: np.ndarray | None):
        ng = 0 if groups is None else len(groups)
        if ng:
            groups = np.ascontiguousarray(groups)
        self._check(self.lib.ibft_bind_groups(self.handle, _ptr(groups) if ng else None, ng))

    def verify_device(self, d_items: int, n: int, d_arena: int, arena_len: int, lo: int, hi: int, d_bitmap: int,
                      d_recovered: int = 0, stream: int = 0):
        self._check(self.lib.ibft_verify_batch_device(self.handle, d_items, n, d_arena or None, arena_len, lo, hi, d_bitmap,
                                                      d_recovered or None, stream or None))

    def quorum_reduce_device(self, d_items: int, n: int, d_bitmap: int, n_groups: int, d_results: int, stream: int = 0):
        self._check(self.lib.ibft_quorum_reduce_device(self.handle, d_items, n, d_bitmap, None, n_groups, d_results, stream or None))

    def quorum_partial_words(self) -> int:
        w = c_uint32()
        self._check(self.lib.ibft_quorum_partial_words(self.handle, ctypes.byref(w)))
        return int(w.value)

    def quorum_mark_device(self, d_items: int, n: int, lo: int, hi: int, d_bitmap: int, d_partial: int, stream: int = 0):
        self._check(self.lib.ibft_quorum_mark_device(self.handle, d_items, n, lo, hi, d_bitmap, d_partial, stream or None))

    def quorum_merge_device(self, d_partials: int, n_parts: int, stride_words: int, d_results: int, stream: int = 0):
        self._check(self.lib.ibft_quorum_merge_device(self.handle, d_partials, n_parts, stride_words, d_results, stream or None))

    def quorum_exchange_device(self, peer_ptrs, rank: int, words_per_rank: int, bitmap_words_per_rank: int, epoch: int, d_bitmap_full: int,
                               d_results: int, d_timeout_flag: int, stream: int = 0):
        """all-gather + merge + reduce over NVLink peer memory in one exchange kernel (ibft_quorum_exchange_device)"""
        arr = (c_uint64 * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        self._check(self.lib.ibft_quorum_exchange_device(self.handle, arr, len(peer_ptrs), rank, words_per_rank, bitmap_words_per_rank, epoch,
                                                         d_bitmap_full, d_results, d_timeout_flag, stream or None))

    def exchange_alloc(self, words: int) -> tuple[int, bytes]:
        """(device address, 64-byte CUDA IPC handle) of a fresh zeroed exchange buffer"""
        p, h = c_void_p(), (ctypes.c_uint8 * 64)()
        self._check(self.lib.ibft_exchange_alloc(self.handle, words, ctypes.byref(p), h))
        return int(p.value), bytes(h)

    def exchange_open(self, handle: bytes) -> int:
        p, h = c_void_p(), (ctypes.c_uint8 * 64).from_buffer_copy(handle)
        self._check(self.lib.ibft_exchange_open(self.handle, h, ctypes.byref(p)))
        return int(p.value)

    def exchange_close(self, d_peer: int):
        self._check(self.lib.ibft_exchange_close(self.handle, c_void_p(d_peer)))

    def exchange_free(self, d_buf: int):
        self._check(self.lib.ibft_exchange_free(self.handle, c_void_p(d_buf)))

    def exchange_clear(self, d_buf: int, word_off: int, words: int, stream: int = 0):
        self._check(self.lib.ibft_exchange_clear(self.handle, c_void_p(d_buf), word_off, words, stream or None))

    def voted_bitmap(self, group: int, n_validators: int) -> np.ndarray:
        words = np.zeros((n_validators + 31) // 32, dtype=np.uint32)
        self._check(self.lib.ibft_get_voted_bitmap(self.handle, group, _ptr(words), len(words)))
        return words

    # ---- hashing (IsValidProposalHash)
    def keccak256_batch(self, messages: list[bytes]) -> list[bytes]:
        n = len(messages)
        if n == 0:
            return []
        offs = np.zeros(n, dtype=np.uint32)
        lens = np.array([len(m) for m in messages], dtype=np.uint32)
        offs[1:] = np.cumsum(lens)[:-1]
        arena = np.frombuffer(b"".join(messages), dtype=np.uint8) if int(lens.sum()) else np.zeros(0, dtype=np.uint8)
        out = np.zeros((n, 32), dtype=np.uint8)
        self._check(self.lib.ibft_keccak256_batch(self.handle, _ptr(arena) if len(arena) else None, len(arena), _ptr(offs), _ptr(lens), n, _ptr(out)))
        return [bytes(out[i]) for i in range(n)]

    def proposal_hash_batch(self, proposals: list[bytes], rounds: list[int]) -> list[bytes]:
        """Keccak-256(Keccak-256(raw) || u64_be(round)) for each proposal, both sponges in one launch (IsValidProposalHash)."""
        n = len(proposals)
        if n == 0:
            return []
        offs = np.zeros(n, dtype=np.uint32)
        lens = np.array([len(m) for m in proposals], dtype=np.uint32)
        offs[1:] = np.cumsum(lens)[:-1]
        arena = np.frombuffer(b"".join(proposals), dtype=np.uint8) if int(lens.sum()) else np.zeros(0, dtype=np.uint8)
        rd = np.array(rounds, dtype=np.uint64)
        out = np.zeros((n, 32), dtype=np.uint8)
        self._check(self.lib.ibft_proposal_hash_batch(self.handle, _ptr(arena) if len(arena) else None, len(arena), _ptr(offs), _ptr(lens),
                                                      _ptr(rd), n, _ptr(out)))
        return [bytes(out[i]) for i in range(n)]

    # ---- signing (MessageConstructor side)
    def sign_batch(self, privkeys: list[int], digests: list[bytes], nonces: list[int] | None = None) -> list[bytes]:
        n = len(privkeys)
        if n == 0:
            return []
        D = np.frombuffer(b"".join(x.to_bytes(32, "big") for x in privkeys), dtype=np.uint8)
        Z = np.frombuffer(b"".join(digests), dtype=np.uint8)
        K = np.frombuffer(b"".join(x.to_bytes(32, "big") for x in nonces), dtype=np.uint8) if nonces is not None else None
        out = np.zeros((n, 65), dtype=np.uint8)
        self._check(self.lib.ibft_sign_batch(self.handle, _ptr(D), _ptr(Z), _ptr(K), n, _ptr(out)))
        return [bytes(out[i]) for i in range(n)]

    def combined_table_info(self):
        wc, n = c_int(), c_uint32()
        self._check(self.lib.ibft_debug_ctable(self.handle, 0, 0, None, ctypes.byref(wc), ctypes.byref(n)))
        return int(wc.value), int(n.value)

    def combined_table_entries(self, first: int, count: int) -> np.ndarray:
        """entries [first, first + count) of the generator comb, all positions back to back (x, y as 8 little-endian words)"""
        out = np.zeros((count, 16), dtype=np.uint32)
        self._check(self.lib.ibft_debug_ctable(self.handle, first, count, _ptr(out), None, None))
        return out

    def key_table_entries(self, slot: int, validator: int, first: int = 0, count: int = 0):
        """(registry state, entries [first, first + count) of a validator's key comb): entry j * 128 + m - 1 = m * 2^(8j) * Q"""
        out = np.zeros((count, 16), dtype=np.uint32)
        st = c_uint32()
        self._check(self.lib.ibft_debug_keytab(self.handle, slot, validator, first, count, _ptr(out) if count else None, ctypes.byref(st)))
        return int(st.value), out

    def last_deferred(self) -> int:
        """items the known-key pass of the last completed host-buffer call left to the recover pass"""
        c = c_uint32()
        self._check(self.lib.ibft_debug_last_deferred(self.handle, ctypes.byref(c)))
        return int(c.value)

    # ---- primitive parity hooks (tests)
    def debug_op(self, op: str, a: list[int], b: list[int] | None = None, c: list[bytes] | None = None, out_stride: int = 32):
        n = len(a)
        A = np.frombuffer(b"".join(x.to_bytes(32, "big") for x in a), dtype=np.uint8)
        Bm = np.frombuffer(b"".join(x.to_bytes(32, "big") for x in b), dtype=np.uint8) if b is not None else None
        C = np.frombuffer(b"".join(c), dtype=np.uint8) if c is not None else None
        out = np.zeros((n, out_stride), dtype=np.uint8)
        self._check(self.lib.ibft_debug_op(self.handle, DBG[op], _ptr(A), _ptr(Bm), _ptr(C), n, _ptr(out), out_stride))
        return [bytes(out[i]) for i in range(n)]
