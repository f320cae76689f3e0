"""Host-side binding of the engine's C ABI (include/ipcfp.h) for tests, bench and Python callers.

Mirrors the reference's API surface for the hot path — `EventProofSpec`, `StorageProofSpec`,
`generate_event_proof`, `read_storage_slot`, `generate_storage_proof`, `generate_proof_bundle`
(reference src/proofs/generator.rs:12-95, events/generator.rs:60-68, storage/decode.rs:36-40,
storage/generator.rs:29-35) — over the CUDA library. There is NO CPU implementation behind these
calls: if libipcfp.so is missing or no CUDA device is present they raise.
"""
import ctypes as C
import os
import subprocess
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _abi as A

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "libipcfp.so")


def build_lib(force=False, jobs=8):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    if force or not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", _ROOT, "-j%d" % jobs, os.path.relpath(LIB_PATH, _ROOT)])
    else:
        subprocess.check_call(["make", "-C", _ROOT, "-j%d" % jobs, "-s", os.path.relpath(LIB_PATH, _ROOT)])
    return LIB_PATH


_lib = None

EXPORTS = [
    "ipcfp_last_error", "ipcfp_last_error_index", "ipcfp_version", "ipcfp_kernel_launch_count", "ipcfp_host_alloc", "ipcfp_host_free",
    "ipcfp_store_create", "ipcfp_store_destroy", "ipcfp_store_n_blocks", "ipcfp_store_get", "ipcfp_store_has",
    "ipcfp_store_first_bad_block", "ipcfp_blake2b256_batch", "ipcfp_keccak256_batch", "ipcfp_sha256_batch",
    "ipcfp_compute_mapping_slots", "ipcfp_generate_event_proof", "ipcfp_event_result_free", "ipcfp_read_storage_slots",
    "ipcfp_slot_result_free", "ipcfp_generate_storage_proofs", "ipcfp_storage_result_free", "ipcfp_generate_proof_bundle",
    "ipcfp_bundle_free", "ipcfp_generate_event_proof_shard", "ipcfp_witness_cids_to_device", "ipcfp_merge_witness_cids",
    "ipcfp_tipset_upload", "ipcfp_tipset_free", "ipcfp_generate_event_proof_resident", "ipcfp_generate_event_proof_shard_resident",
    "ipcfp_store_stream", "ipcfp_exec_bucketize", "ipcfp_exec_dedup", "ipcfp_exec_fetch",
    "ipcfp_comm_unique_id", "ipcfp_comm_init", "ipcfp_comm_destroy", "ipcfp_generate_event_proof_sharded",
    "ipcfp_verify_event_proofs", "ipcfp_verify_storage_proofs", "ipcfp_bundle_to_json", "ipcfp_event_result_to_json", "ipcfp_json_free",
    "ipcfp_bundle_from_json", "ipcfp_parsed_bundle_free", "ipcfp_generate_event_proof_multi", "ipcfp_generate_event_proof_multi_resident",
]


def lib():
    """Loads libipcfp.so. Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `make` (or __graft_entry__.build()). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.ipcfp_last_error.restype = C.c_char_p
        L.ipcfp_last_error_index.restype = C.c_uint64
        L.ipcfp_version.restype = C.c_char_p
        L.ipcfp_kernel_launch_count.restype = C.c_uint64
        L.ipcfp_host_alloc.restype = C.c_int32
        L.ipcfp_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
        L.ipcfp_host_free.argtypes = [C.c_void_p]
        L.ipcfp_store_create.restype = C.c_int32
        L.ipcfp_store_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_uint32,
                                         C.POINTER(C.c_void_p)]
        L.ipcfp_store_destroy.argtypes = [C.c_void_p]
        L.ipcfp_store_n_blocks.restype = C.c_uint64
        L.ipcfp_store_n_blocks.argtypes = [C.c_void_p]
        L.ipcfp_store_first_bad_block.restype = C.c_uint64
        L.ipcfp_store_first_bad_block.argtypes = [C.c_void_p]
        L.ipcfp_store_get.restype = C.c_int32
        L.ipcfp_store_get.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
        L.ipcfp_store_has.restype = C.c_int32
        L.ipcfp_store_has.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
        for name in ("ipcfp_blake2b256_batch", "ipcfp_keccak256_batch", "ipcfp_sha256_batch"):
            f = getattr(L, name)
            f.restype = C.c_int32
            f.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]
        L.ipcfp_compute_mapping_slots.restype = C.c_int32
        L.ipcfp_compute_mapping_slots.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p]
        L.ipcfp_generate_event_proof.restype = C.c_int32
        L.ipcfp_generate_event_proof.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.POINTER(A.EventSpec), C.c_uint32,
                                                 C.POINTER(C.POINTER(A.EventResultC))]
        L.ipcfp_generate_event_proof_shard.restype = C.c_int32
        L.ipcfp_generate_event_proof_shard.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.POINTER(A.EventSpec), C.c_uint64, C.c_uint64,
                                                       C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.POINTER(A.EventResultC))]
        L.ipcfp_event_result_free.argtypes = [C.POINTER(A.EventResultC)]
        L.ipcfp_generate_event_proof_multi.restype = C.c_int32
        L.ipcfp_generate_event_proof_multi.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.POINTER(A.EventSpec), C.c_uint32, C.c_uint32,
                                                       C.c_void_p, C.c_void_p, C.POINTER(C.POINTER(A.EventResultC))]
        L.ipcfp_generate_event_proof_multi_resident.restype = C.c_int32
        L.ipcfp_generate_event_proof_multi_resident.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(A.EventSpec), C.c_uint32, C.c_uint32,
                                                                C.c_void_p, C.c_void_p, C.POINTER(C.POINTER(A.EventResultC))]
        L.ipcfp_read_storage_slots.restype = C.c_int32
        L.ipcfp_read_storage_slots.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.POINTER(A.SlotResultC))]
        L.ipcfp_slot_result_free.argtypes = [C.POINTER(A.SlotResultC)]
        L.ipcfp_generate_storage_proofs.restype = C.c_int32
        L.ipcfp_generate_storage_proofs.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.c_void_p, C.c_uint64,
                                                    C.POINTER(C.POINTER(A.StorageResultC))]
        L.ipcfp_storage_result_free.argtypes = [C.POINTER(A.StorageResultC)]
        L.ipcfp_generate_proof_bundle.restype = C.c_int32
        L.ipcfp_generate_proof_bundle.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                                  C.POINTER(C.POINTER(A.BundleC))]
        L.ipcfp_bundle_free.argtypes = [C.POINTER(A.BundleC)]
        L.ipcfp_tipset_upload.restype = C.c_int32
        L.ipcfp_tipset_upload.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.POINTER(C.c_void_p)]
        L.ipcfp_tipset_free.argtypes = [C.c_void_p]
        L.ipcfp_generate_event_proof_resident.restype = C.c_int32
        L.ipcfp_generate_event_proof_resident.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(A.EventSpec), C.c_uint32,
                                                          C.POINTER(C.POINTER(A.EventResultC))]
        L.ipcfp_generate_event_proof_shard_resident.restype = C.c_int32
        L.ipcfp_generate_event_proof_shard_resident.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(A.EventSpec), C.c_uint64, C.c_uint64,
                                                                C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.POINTER(A.EventResultC))]
        L.ipcfp_store_stream.restype = C.c_void_p
        L.ipcfp_store_stream.argtypes = [C.c_void_p]
        L.ipcfp_exec_bucketize.restype = C.c_int32
        L.ipcfp_exec_bucketize.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]
        L.ipcfp_exec_dedup.restype = C.c_int32
        L.ipcfp_exec_dedup.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.ipcfp_exec_fetch.restype = C.c_int32
        L.ipcfp_exec_fetch.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]
        L.ipcfp_witness_cids_to_device.restype = C.c_int32
        L.ipcfp_witness_cids_to_device.argtypes = [C.POINTER(A.EventResultC), C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.ipcfp_merge_witness_cids.restype = C.c_int32
        L.ipcfp_merge_witness_cids.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64,
                                               C.POINTER(C.c_uint64)]
        L.ipcfp_comm_unique_id.restype = C.c_int32
        L.ipcfp_comm_unique_id.argtypes = [C.c_void_p]
        L.ipcfp_comm_init.restype = C.c_int32
        L.ipcfp_comm_init.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.ipcfp_comm_destroy.argtypes = [C.c_void_p]
        L.ipcfp_generate_event_proof_sharded.restype = C.c_int32
        L.ipcfp_generate_event_proof_sharded.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(A.EventSpec), C.c_void_p, C.c_uint32,
                                                         C.POINTER(C.POINTER(A.EventResultC))]
        L.ipcfp_verify_event_proofs.restype = C.c_int32
        L.ipcfp_verify_event_proofs.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.ipcfp_verify_storage_proofs.restype = C.c_int32
        L.ipcfp_verify_storage_proofs.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.c_void_p, C.c_uint64, C.c_void_p]
        for name in ("ipcfp_bundle_to_json", "ipcfp_event_result_to_json"):
            f = getattr(L, name)
            f.restype = C.c_int32
            f.argtypes = [C.c_void_p, C.POINTER(A.TipsetDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        L.ipcfp_json_free.argtypes = [C.c_void_p]
        L.ipcfp_bundle_from_json.restype = C.c_int32
        L.ipcfp_bundle_from_json.argtypes = [C.c_char_p, C.c_uint64, C.POINTER(C.POINTER(A.ParsedBundleC))]
        L.ipcfp_parsed_bundle_free.argtypes = [C.POINTER(A.ParsedBundleC)]
        _lib = L
    return _lib


def _u8(x):
    if isinstance(x, (bytes, bytearray, memoryview)):
        return np.frombuffer(bytes(x), dtype=np.uint8).copy()
    return np.ascontiguousarray(x, dtype=np.uint8)


def _check(st):
    if st != A.OK:
        L = lib()
        raise A.IpcfpError(st, L.ipcfp_last_error().decode(errors="replace"), L.ipcfp_last_error_index())


def kernel_launch_count():
    return int(lib().ipcfp_kernel_launch_count())


@dataclass
class EventProofSpec:  # reference src/proofs/generator.rs:18-22
    event_signature: str
    topic_1: str
    actor_id_filter: Optional[int] = None

    def as_c(self):
        return A.make_event_spec(self.event_signature, self.topic_1, self.actor_id_filter)


@dataclass
class StorageProofSpec:  # reference src/proofs/generator.rs:12-15
    actor_id: int
    slot: bytes


@dataclass
class MultiEventResult:
    """Result of BlockStore.generate_event_proof_multi: one EventResultPy for all specs (witness = the union of the specs'
    witnesses), with spec k's matching receipts at match_offsets[k]:match_offsets[k+1] and its proofs at
    proof_offsets[k]:proof_offsets[k+1]."""
    result: A.EventResultPy
    match_offsets: np.ndarray
    proof_offsets: np.ndarray

    def spec(self, k):
        """(matching receipt indices, proofs) of spec k."""
        m, p = self.match_offsets, self.proof_offsets
        return self.result.matching[int(m[k]):int(m[k + 1])], self.result.proofs[int(p[k]):int(p[k + 1])]


class PinnedArray:
    """Pinned host memory (ipcfp_host_alloc) exposed as a numpy array."""

    def __init__(self, nbytes):
        p = C.c_void_p()
        _check(lib().ipcfp_host_alloc(max(int(nbytes), 1), C.byref(p)))
        self._p = p
        self.array = np.frombuffer((C.c_uint8 * max(int(nbytes), 1)).from_address(p.value), dtype=np.uint8)[:int(nbytes)]

    def free(self):
        if self._p:
            self.array = None
            lib().ipcfp_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class BlockStore:
    """Device-resident block store (replaces the reference's Blockstore implementations)."""

    def __init__(self, cids, offsets, lengths, blob, device=0, verify_cids=False):
        cids = np.ascontiguousarray(cids, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        lengths = np.ascontiguousarray(lengths, dtype=np.uint32)
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self.n_blocks = len(lengths)
        self.device = device
        h = C.c_void_p()
        st = lib().ipcfp_store_create(cids.ctypes.data if cids.size else None, offsets.ctypes.data if offsets.size else None,
                                      lengths.ctypes.data if lengths.size else None, blob.ctypes.data if blob.size else None, blob.size,
                                      self.n_blocks, device, A.STORE_VERIFY_CIDS if verify_cids else 0, C.byref(h))
        self._h = h
        if st != A.OK:
            bad = lib().ipcfp_store_first_bad_block(h) if h else None
            msg, idx = lib().ipcfp_last_error().decode(errors="replace"), lib().ipcfp_last_error_index()
            if h:
                lib().ipcfp_store_destroy(h)
                self._h = None
            e = A.IpcfpError(st, msg, idx)
            e.first_bad_block = bad
            raise e

    @classmethod
    def from_tipset(cls, ts, device=0, verify_cids=False):
        return cls(ts.cids, ts.offsets, ts.lengths, ts.blob, device, verify_cids)

    def get(self, cid):
        cid = _u8(cid)
        ln = C.c_uint32()
        found = C.c_int()
        _check(lib().ipcfp_store_get(self._h, cid.ctypes.data, None, 0, C.byref(ln), C.byref(found)))
        if not found.value:
            return None
        buf = np.zeros(max(ln.value, 1), dtype=np.uint8)
        _check(lib().ipcfp_store_get(self._h, cid.ctypes.data, buf.ctypes.data, ln.value, C.byref(ln), C.byref(found)))
        return bytes(buf[:ln.value])

    def has(self, cid):
        cid = _u8(cid)
        found = C.c_int()
        _check(lib().ipcfp_store_has(self._h, cid.ctypes.data, C.byref(found)))
        return bool(found.value)

    # --- generate_event_proof (events/generator.rs:60-107)
    def generate_event_proof(self, ts, spec, flags=0):
        d, keep = A.make_tipset_desc(ts)
        cs = spec.as_c() if isinstance(spec, EventProofSpec) else spec
        out = C.POINTER(A.EventResultC)()
        _check(lib().ipcfp_generate_event_proof(self._h, C.byref(d), C.byref(cs), flags, C.byref(out)))
        try:
            return A.event_result_from_c(out.contents)
        finally:
            lib().ipcfp_event_result_free(out)

    # --- the event specs of generate_proof_bundle (proofs/generator.rs:57-78) in one scan of the tipset
    def generate_event_proof_multi(self, ts, specs, flags=0):
        d, keep = A.make_tipset_desc(ts)
        return self._multi(lambda *a: lib().ipcfp_generate_event_proof_multi(self._h, C.byref(d), *a), specs, flags)

    def generate_event_proof_multi_resident(self, tipset, specs, flags=0):
        """The same against a ResidentTipset of this store."""
        return self._multi(lambda *a: lib().ipcfp_generate_event_proof_multi_resident(self._h, tipset._h, *a), specs, flags)

    def upload_tipset(self, ts):
        return ResidentTipset(self, ts)

    @staticmethod
    def _multi(call, specs, flags):
        cs = [s.as_c() if isinstance(s, EventProofSpec) else s for s in specs]
        arr = (A.EventSpec * max(len(cs), 1))(*cs)
        mo, po = np.zeros(len(cs) + 1, dtype=np.uint64), np.zeros(len(cs) + 1, dtype=np.uint64)
        out = C.POINTER(A.EventResultC)()
        _check(call(arr, len(cs), flags, mo.ctypes.data, po.ctypes.data, C.byref(out)))
        try:
            return MultiEventResult(A.event_result_from_c(out.contents), mo, po)
        finally:
            lib().ipcfp_event_result_free(out)

    def generate_event_proof_shard(self, ts, spec, lo, hi, world, rank, flags=0):
        d, keep = A.make_tipset_desc(ts)
        cs = spec.as_c() if isinstance(spec, EventProofSpec) else spec
        out = C.POINTER(A.EventResultC)()
        _check(lib().ipcfp_generate_event_proof_shard(self._h, C.byref(d), C.byref(cs), lo, hi, world, rank, flags, C.byref(out)))
        try:
            return A.event_result_from_c(out.contents)
        finally:
            lib().ipcfp_event_result_free(out)

    # --- read_storage_slot (storage/decode.rs:36-97), batched
    def read_storage_slots(self, root, slots):
        root = _u8(root)
        slots = _u8(slots).reshape(-1, 32)
        out = C.POINTER(A.SlotResultC)()
        _check(lib().ipcfp_read_storage_slots(self._h, root.ctypes.data, slots.ctypes.data if slots.size else None, len(slots), C.byref(out)))
        try:
            return A.slot_result_from_c(out.contents)
        finally:
            lib().ipcfp_slot_result_free(out)

    # --- generate_storage_proof (storage/generator.rs:29-67), batched
    def generate_storage_proofs(self, ts, specs):
        specs = [(s.actor_id, s.slot) if isinstance(s, StorageProofSpec) else s for s in specs]
        d, keep = A.make_tipset_desc(ts)
        arr = A.make_storage_specs(specs)
        out = C.POINTER(A.StorageResultC)()
        _check(lib().ipcfp_generate_storage_proofs(self._h, C.byref(d), arr, len(specs), C.byref(out)))
        try:
            return A.storage_result_from_c(out.contents)
        finally:
            lib().ipcfp_storage_result_free(out)

    # --- generate_proof_bundle (proofs/generator.rs:25-95)
    def generate_proof_bundle(self, ts, storage_specs, event_specs):
        sspecs = [(s.actor_id, s.slot) if isinstance(s, StorageProofSpec) else s for s in storage_specs]
        especs = [s.as_c() if isinstance(s, EventProofSpec) else s for s in event_specs]
        d, keep = A.make_tipset_desc(ts)
        sarr = A.make_storage_specs(sspecs)
        earr = (A.EventSpec * len(especs))(*especs)
        out = C.POINTER(A.BundleC)()
        _check(lib().ipcfp_generate_proof_bundle(self._h, C.byref(d), sarr, len(sspecs), earr, len(especs), C.byref(out)))
        try:
            return A.bundle_from_c(out.contents)
        finally:
            lib().ipcfp_bundle_free(out)

    def close(self):
        if self._h:
            lib().ipcfp_store_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ResidentTipset:
    """A tipset descriptor uploaded to the device once (ipcfp_tipset_upload) for many calls against one BlockStore."""

    def __init__(self, store, ts):
        d, keep = A.make_tipset_desc(ts)
        self._h = C.c_void_p()
        _check(lib().ipcfp_tipset_upload(store._h, C.byref(d), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().ipcfp_tipset_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _to_json(fn, obj_ptr, ts):
    d, keep = A.make_tipset_desc(ts)
    out, n = C.c_void_p(), C.c_uint64()
    _check(getattr(lib(), fn)(obj_ptr, C.byref(d), C.byref(out), C.byref(n)))
    try:
        return C.string_at(out.value, n.value).decode()
    finally:
        lib().ipcfp_json_free(out)


def bundle_to_json(bundle_c_ptr, ts):
    """`serde_json::to_string(&UnifiedProofBundle)` of an ipcfp_bundle (POINTER(BundleC) or its address)."""
    return _to_json("ipcfp_bundle_to_json", C.cast(bundle_c_ptr, C.c_void_p), ts)


def event_result_to_json(result_c_ptr, ts):
    """`serde_json::to_string(&EventProofBundle)` of an ipcfp_event_result."""
    return _to_json("ipcfp_event_result_to_json", C.cast(result_c_ptr, C.c_void_p), ts)


class ParsedBundle:
    """`serde_json::from_str::<UnifiedProofBundle | EventProofBundle>` through the C ABI (ipcfp_bundle_from_json): PODs ready for the
    batched verifiers + the witness block arrays. Owns the C object; `.c` is the ipcfp_parsed_bundle."""

    def __init__(self, text):
        raw = text.encode() if isinstance(text, str) else bytes(text)
        self._p = C.POINTER(A.ParsedBundleC)()
        st = lib().ipcfp_bundle_from_json(raw, len(raw), C.byref(self._p))
        if st != A.OK:
            raise A.IpcfpError(st, "ipcfp_bundle_from_json", 0)
        self.c = self._p.contents

    @property
    def witness(self):
        return A.witness_from_c(self.c.witness)

    @property
    def event_proofs_raw(self):
        n = int(self.c.n_event_proofs)
        return A._arr(self.c.event_proofs, n * C.sizeof(A.EventProofC), np.uint8), A._arr(self.c.data_blob, int(self.c.data_blob_size), np.uint8)

    @property
    def storage_proofs_raw(self):
        return A._arr(self.c.storage_proofs, int(self.c.n_storage_proofs) * C.sizeof(A.StorageProofC), np.uint8)

    def tipset_fields(self):
        t = self.c.tipset
        P = int(t.n_parents)
        return dict(parent_epoch=int(t.parent_epoch), child_epoch=int(t.child_epoch),
                    parent_cids=A._arr(t.parent_cids, P * A.CID_LEN, np.uint8).tobytes(),
                    child_cid=A._arr(t.child_cid, A.CID_LEN if t.child_cid else 0, np.uint8).tobytes(),
                    parent_state_root=A._arr(t.child_parent_state_root, A.CID_LEN if t.child_parent_state_root else 0, np.uint8).tobytes())

    def close(self):
        if self._p:
            lib().ipcfp_parsed_bundle_free(self._p)
            self._p = C.POINTER(A.ParsedBundleC)()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def verify_event_proofs(witness, ts, result, filter_spec=None, device=0):
    """verify_event_proof (events/verifier.rs:51-74) batched on the GPU: the witness (WitnessPy) becomes a store with every block
    Blake2b-checked against its CID, then every proof of `result` (EventResultPy) is replayed. → list of bools."""
    store = BlockStore(witness.cids, witness.offsets, witness.lengths, witness.blob, device, verify_cids=True)
    try:
        d, keep = A.make_tipset_desc(ts)
        n = len(result.proofs)
        res = np.zeros(max(n, 1), dtype=np.uint8)
        raw = np.ascontiguousarray(result.raw_proofs)
        blob = np.ascontiguousarray(result.data_blob)
        fs = filter_spec.as_c() if isinstance(filter_spec, EventProofSpec) else filter_spec
        _check(lib().ipcfp_verify_event_proofs(store._h, C.byref(d), raw.ctypes.data if n else None, n, blob.ctypes.data if blob.size else None, blob.size,
                                               C.addressof(fs) if fs is not None else None, res.ctypes.data))
        return [bool(x) for x in res[:n]]
    finally:
        store.close()


def verify_storage_proofs(witness, ts, result, device=0):
    """verify_storage_proof (storage/verifier.rs:24-63) batched on the GPU over a CID-checked witness store."""
    store = BlockStore(witness.cids, witness.offsets, witness.lengths, witness.blob, device, verify_cids=True)
    try:
        d, keep = A.make_tipset_desc(ts)
        n = len(result.proofs)
        res = np.zeros(max(n, 1), dtype=np.uint8)
        raw = np.ascontiguousarray(result.raw_proofs)
        _check(lib().ipcfp_verify_storage_proofs(store._h, C.byref(d), raw.ctypes.data if n else None, n, res.ctypes.data))
        return [bool(x) for x in res[:n]]
    finally:
        store.close()


def _hash_batch(fn, messages, device=0):
    n = len(messages)
    lengths = np.array([len(m) for m in messages], dtype=np.uint32)
    offsets = np.zeros(n, dtype=np.uint64)
    if n:
        offsets[1:] = np.cumsum(lengths[:-1], dtype=np.uint64)
    blob = np.frombuffer(b"".join(bytes(m) for m in messages), dtype=np.uint8) if n else np.zeros(0, dtype=np.uint8)
    out = np.zeros((n, 32), dtype=np.uint8)
    _check(getattr(lib(), fn)(blob.ctypes.data if blob.size else None, blob.size, offsets.ctypes.data if n else None,
                              lengths.ctypes.data if n else None, n, device, out.ctypes.data if n else None))
    return [bytes(r) for r in out]


def blake2b256_batch(messages, device=0):
    return _hash_batch("ipcfp_blake2b256_batch", messages, device)


def keccak256_batch(messages, device=0):
    return _hash_batch("ipcfp_keccak256_batch", messages, device)


def sha256_batch(messages, device=0):
    return _hash_batch("ipcfp_sha256_batch", messages, device)


def compute_mapping_slots(keys32, slot_indices, device=0):
    """compute_mapping_slot (storage/utils.rs:5-12) batched on the GPU."""
    keys = np.ascontiguousarray(np.frombuffer(b"".join(bytes(k) for k in keys32), dtype=np.uint8))
    idx = np.ascontiguousarray(slot_indices, dtype=np.uint64)
    n = len(idx)
    out = np.zeros((n, 32), dtype=np.uint8)
    _check(lib().ipcfp_compute_mapping_slots(keys.ctypes.data if n else None, idx.ctypes.data if n else None, n, device,
                                             out.ctypes.data if n else None))
    return [bytes(r) for r in out]


def calculate_storage_slot(subnet_ascii, subnets_slot_index, device=0):
    """calculate_storage_slot (storage/utils.rs:16-19)."""
    b = subnet_ascii.encode()[:32]
    return compute_mapping_slots([b + bytes(32 - len(b))], [subnets_slot_index], device)[0]
