"""Thin object layer over the C ABI (include/csvb200.h): Context and StructureIndex.

Everything here forwards to libcsvb200.so; nothing is computed in Python.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .errors import raise_for

BUILD_DEFAULT = 0
BUILD_KEEP_BYTES = 1
BUILD_STRICT_MIN64 = 2
BUILD_VALIDATE = 4
FIELD_RAW = 0
FIELD_UNQUOTE = 1
FIELD_TRIM = 2

NONE = np.uint64(0xFFFFFFFFFFFFFFFF)


class host_registered:
    """Pins a NumPy array the caller owns for the duration of a `with` block (csvb200_host_register / _unregister), so the
    end-to-end calls DMA it in place: `with host_registered(out): ctx.index_build_to_host(...)`."""

    def __init__(self, array: np.ndarray, read_only: bool = False):
        self._ptr, self._bytes, self._ro = array.ctypes.data, array.nbytes, read_only
        self._array = array           # keeps the memory alive while it is registered

    def __enter__(self):
        rc = _lib.load().csvb200_host_register(C.c_void_p(self._ptr), self._bytes, int(self._ro))
        if rc:
            raise_for(rc, "csvb200_host_register")
        return self._array

    def __exit__(self, *exc):
        _lib.load().csvb200_host_unregister(C.c_void_p(self._ptr))
        return False


def _as_u8(data) -> np.ndarray:
    if isinstance(data, np.ndarray):
        a = data
        if a.dtype != np.uint8:
            a = a.view(np.uint8)
        return np.ascontiguousarray(a)
    return np.frombuffer(data, dtype=np.uint8)


class Context:
    """csvb200_ctx: one per GPU (process-per-GPU model)."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.csvb200_ctx_create(int(device), C.byref(h))
        raise_for(rc, f"csvb200_ctx_create(device={device}) failed: no usable CUDA device (no CPU fallback)")
        self._h = h
        self.device = int(device)

    # -- plumbing -------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc:
            raise_for(rc, self._lib.csvb200_last_error(self._h).decode("utf-8", "replace"))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.csvb200_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_stream(self, cuda_stream: int | None):
        """Bind the context to an external cudaStream_t handle.  None restores the private stream;
        0 (what torch reports for its default stream) is mapped to cudaStreamLegacy (0x1), because a
        NULL handle means "restore the private stream" in the C ABI."""
        if cuda_stream is None:
            handle = 0
        else:
            handle = 1 if int(cuda_stream) == 0 else int(cuda_stream)
        self._check(self._lib.csvb200_ctx_set_stream(self._h, C.c_void_p(handle)))

    def set_reserve(self, num: int, den: int):
        self._check(self._lib.csvb200_ctx_set_reserve(self._h, num, den))

    def last_build_ms(self) -> float:
        ms = C.c_float()
        self._check(self._lib.csvb200_ctx_last_build_ms(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return int(self._lib.csvb200_ctx_launch_count(self._h))

    # -- csv -> index ---------------------------------------------------------------------
    def index_build(self, data, flags: int = BUILD_DEFAULT) -> "StructureIndex":
        """reader::read (src/reader.rs:150-306) for host bytes."""
        a = _as_u8(data)
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_build(self._h, a.ctypes.data, a.size, flags, C.byref(h)))
        return StructureIndex(self, h)

    def index_build_ptr(self, host_ptr: int, n: int, flags: int = BUILD_DEFAULT) -> "StructureIndex":
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_build(self._h, C.c_void_p(host_ptr), n, flags, C.byref(h)))
        return StructureIndex(self, h)

    def index_build_device(self, dev_ptr: int, n: int, flags: int = BUILD_DEFAULT) -> "StructureIndex":
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_build_device(self._h, C.c_void_p(dev_ptr), n, flags, C.byref(h)))
        return StructureIndex(self, h)

    def index_build_to_host(self, host_ptr: int, n: int, dst_ptr: int, dst_cap: int) -> int:
        ln = C.c_size_t()
        self._check(self._lib.csvb200_index_build_to_host(self._h, C.c_void_p(host_ptr), n, C.c_void_p(dst_ptr),
                                                          dst_cap, C.byref(ln)))
        return ln.value

    # -- streaming ingest -------------------------------------------------------------------
    def index_build_stream(self, read, sink, chunk_bytes: int = 0) -> dict:
        """csvb200_index_build_stream: read(cap) -> bytes-like (b"" = end of input); sink(entries: np.ndarray
        of u64 (a view, copy it to keep it), first_slot: int).  Returns the stream stats."""
        err = []

        def _read(_user, dst, cap):
            try:
                b = read(cap)
                k = len(b)
                if k > cap:   # checked BEFORE the copy: dst is a pinned ring slot of exactly `cap` bytes
                    raise ValueError(f"read({cap}) returned {k} bytes")
                if k:
                    C.memmove(dst, bytes(b) if not isinstance(b, (bytes, bytearray)) else b, k)
                return k
            except BaseException as e:  # never unwind through the C frames
                err.append(e)
                return 0

        def _sink(_user, entries, count, first):
            try:
                sink(np.ctypeslib.as_array(entries, shape=(count,)), int(first))
                return 0
            except BaseException as e:
                err.append(e)
                return 1

        st = _lib.StreamStats()
        rc = self._lib.csvb200_index_build_stream(self._h, _lib.READ_FN(_read), None, _lib.SINK_FN(_sink), None,
                                                  chunk_bytes, C.byref(st))
        if err:
            raise err[0]
        self._check(rc)
        return {k: getattr(st, k) for k, _ in _lib.StreamStats._fields_}

    def index_build_file(self, path: str, out: np.ndarray | None = None):
        """csvb200_index_build_file: file -> host index (u64 array).  Returns (index, stats)."""
        import os
        st = _lib.StreamStats()
        ln = C.c_size_t()
        if out is None:
            size = os.path.getsize(path) if os.path.exists(path) else 0
            out = np.empty(size // 3 + 4096, dtype=np.uint64)
        rc = self._lib.csvb200_index_build_file(self._h, os.fsencode(path), out.ctypes.data, out.size, C.byref(ln),
                                                C.byref(st))
        if rc == 9 and ln.value > out.size:   # denser than the reserve: the count is known now
            out = np.empty(ln.value, dtype=np.uint64)
            rc = self._lib.csvb200_index_build_file(self._h, os.fsencode(path), out.ctypes.data, out.size,
                                                    C.byref(ln), C.byref(st))
        self._check(rc)
        return out[:ln.value], {k: getattr(st, k) for k, _ in _lib.StreamStats._fields_}

    def index_build_file_ptr(self, path: str, dst_ptr: int, dst_cap: int):
        import os
        st = _lib.StreamStats()
        ln = C.c_size_t()
        self._check(self._lib.csvb200_index_build_file(self._h, os.fsencode(path), C.c_void_p(dst_ptr), dst_cap,
                                                       C.byref(ln), C.byref(st)))
        return ln.value, {k: getattr(st, k) for k, _ in _lib.StreamStats._fields_}

    def shard_quote_parity(self, dev_ptr: int, n: int) -> int:
        p = C.c_uint32()
        self._check(self._lib.csvb200_shard_quote_parity(self._h, C.c_void_p(dev_ptr), n, C.byref(p)))
        return p.value

    def index_build_shard_device(self, dev_ptr: int, n: int, carry_parity: int, global_offset: int,
                                 emit_sentinel: bool) -> "StructureIndex":
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_build_shard_device(self._h, C.c_void_p(dev_ptr), n, carry_parity,
                                                               global_offset, int(emit_sentinel), C.byref(h)))
        return StructureIndex(self, h)

    def shard_quote_parity_device(self, dev_ptr: int, n: int, d_parity_out: int):
        self._check(self._lib.csvb200_shard_quote_parity_device(self._h, C.c_void_p(dev_ptr), n,
                                                                C.c_void_p(d_parity_out)))

    def index_build_shard_device_ex(self, dev_ptr: int, n: int, d_shard_parities: int, shard_rank: int,
                                    global_offset: int, emit_sentinel: bool, d_result_out: int = 0
                                    ) -> "StructureIndex":
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_build_shard_device_ex(
            self._h, C.c_void_p(dev_ptr), n, C.c_void_p(d_shard_parities), shard_rank, global_offset,
            int(emit_sentinel), C.c_void_p(d_result_out or 0), C.byref(h)))
        return StructureIndex(self, h)

    def index_build_shard_speculative(self, dev_ptr: int, n: int, shard_rank: int, global_offset: int,
                                      emit_sentinel: bool, d_result_out: int, predict_window: int = 0
                                      ) -> "StructureIndex":
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_build_shard_speculative(
            self._h, C.c_void_p(dev_ptr), n, shard_rank, global_offset, int(emit_sentinel), predict_window,
            C.c_void_p(d_result_out), C.byref(h)))
        return StructureIndex(self, h)

    def shard_build_to_host(self, host_ptr: int, n: int, shard_rank: int, global_offset: int, emit_sentinel: bool,
                            dst_ptr: int, dst_cap: int, d_result_out: int):
        """csvb200_shard_build_to_host -> (entries written to dst, job handle for shard_job_verify)."""
        ln, job = C.c_size_t(), C.c_void_p()
        self._check(self._lib.csvb200_shard_build_to_host(self._h, C.c_void_p(host_ptr), n, shard_rank, global_offset,
                                                          int(emit_sentinel), C.c_void_p(dst_ptr), dst_cap, C.byref(ln),
                                                          C.c_void_p(d_result_out), C.byref(job)))
        return ln.value, job

    def shard_job_verify(self, job, d_gathered: int, world: int, d_final_out: int = 0):
        """-> (final entry count in dst, whether the shard had to be re-indexed); frees the job."""
        ln, redone = C.c_size_t(), C.c_int()
        rc = self._lib.csvb200_shard_job_verify(job, C.c_void_p(d_gathered), world, C.c_void_p(d_final_out or 0),
                                                C.byref(ln), C.byref(redone))
        self._lib.csvb200_shard_job_free(job)
        self._check(rc)
        return ln.value, bool(redone.value)

    # -- the exchange: peer-mapped mailboxes instead of a collective (include/csvb200.h) ---------------------
    def exchange(self, rank: int, world: int) -> "Exchange":
        return Exchange(self, rank, world)

    def index_build_shard_exchange(self, ex: "Exchange", dev_ptr: int, n: int, global_offset: int,
                                   predict_window: int = 0) -> "StructureIndex":
        """Prediction, build, in-kernel exchange and conditional re-index of this rank's shard: one call, nothing
        waits on the host.  COLLECTIVE: every rank calls it in the same order."""
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_build_shard_exchange(self._h, ex._h, C.c_void_p(dev_ptr), n, global_offset,
                                                                 predict_window, C.byref(h)))
        idx = StructureIndex(self, h)
        idx._exchange = ex
        return idx

    def shard_build_to_host_exchange(self, ex: "Exchange", host_ptr: int, n: int, global_offset: int, dst_ptr: int,
                                     dst_cap: int, want_counts: bool = False):
        """End-to-end form -> (entries in dst, info dict, counts per rank or None)."""
        ln = C.c_size_t()
        info = _lib.ShardInfo()
        counts = (C.c_uint64 * ex.world)() if want_counts else None
        self._check(self._lib.csvb200_shard_build_to_host_exchange(self._h, ex._h, C.c_void_p(host_ptr), n, global_offset,
                                                                   C.c_void_p(dst_ptr), dst_cap, C.byref(ln), C.byref(info),
                                                                   counts, None))
        return ln.value, {k: int(getattr(info, k)) for k, _ in _lib.ShardInfo._fields_}, (list(counts) if counts else None)

    def index_wrap_device(self, d_entries: int, length: int, input_bytes: int, d_bytes: int = 0) -> "StructureIndex":
        """csvb200_index_wrap_device: an index object over caller-owned device entries (not freed with it)."""
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_wrap_device(self._h, C.c_void_p(d_entries), length, input_bytes,
                                                        C.c_void_p(d_bytes or 0), C.byref(h)))
        return StructureIndex(self, h)

    # -- input validation / on-disk index ------------------------------------------------------
    def validate_utf8(self, data):
        """(valid_up_to or None when well-formed UTF-8, is_ascii) -- csvb200_validate_utf8."""
        a = _as_u8(data)
        v, asc = C.c_uint64(), C.c_int()
        self._check(self._lib.csvb200_validate_utf8(self._h, a.ctypes.data, a.size, C.byref(v), C.byref(asc)))
        if a.size == 0:
            return None, True
        return (None if v.value == 0xFFFFFFFFFFFFFFFF else v.value), bool(asc.value)

    def validate_utf8_device(self, dev_ptr: int, n: int, d_result: int):
        self._check(self._lib.csvb200_validate_utf8_device(self._h, C.c_void_p(dev_ptr), n, C.c_void_p(d_result)))

    def index_load(self, path: str) -> "StructureIndex":
        import os
        h = C.c_void_p()
        self._check(self._lib.csvb200_index_load(self._h, os.fsencode(path), C.byref(h)))
        return StructureIndex(self, h)

    # -- K1 known-answer exports ------------------------------------------------------------
    def block_masks(self, data):
        a = _as_u8(data)
        nb = (a.size + 63) // 64
        q = np.zeros(nb, dtype=np.uint64)
        s = np.zeros(nb, dtype=np.uint64)
        self._check(self._lib.csvb200_block_masks(self._h, a.ctypes.data, a.size, q.ctypes.data, s.ctypes.data))
        return q, s

    def class_bytes(self, data) -> np.ndarray:
        a = _as_u8(data)
        out = np.zeros(a.size, dtype=np.uint8)
        self._check(self._lib.csvb200_class_bytes(self._h, a.ctypes.data, a.size, out.ctypes.data))
        return out


class Exchange:
    """csvb200_exchange: this rank's endpoint of the mailbox exchange.  handle() -> 64 bytes to give to every peer;
    connect(handles) maps the peers' mailboxes (CUDA IPC between processes of one node)."""

    def __init__(self, ctx: Context, rank: int, world: int):
        self.ctx, self.rank, self.world = ctx, int(rank), int(world)
        self._lib = ctx._lib
        h = C.c_void_p()
        ctx._check(self._lib.csvb200_exchange_create(ctx._h, self.rank, self.world, C.byref(h)))
        self._h = h

    def handle(self) -> bytes:
        buf = (C.c_uint8 * 64)()
        self.ctx._check(self._lib.csvb200_exchange_handle(self._h, buf))
        return bytes(buf)

    def connect(self, handles):
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * self.world
        self.ctx._check(self._lib.csvb200_exchange_connect(self._h, blob))

    @staticmethod
    def connect_local(exchanges):
        arr = (C.c_void_p * len(exchanges))(*[e._h for e in exchanges])
        rc = exchanges[0]._lib.csvb200_exchange_connect_local(arr, len(exchanges))
        for e in exchanges:
            if rc:
                e.ctx._check(rc)

    def counts(self, idx: "StructureIndex"):
        """Host-side wait for every rank's row of that build -> (entries per rank, carry-in per rank)."""
        counts = (C.c_uint64 * self.world)()
        carries = (C.c_uint32 * self.world)()
        self.ctx._check(self._lib.csvb200_exchange_counts(self._h, idx._h, counts, carries))
        return list(counts), list(carries)

    def close(self):
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            self._lib.csvb200_exchange_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Multi:
    """csvb200_multi: every listed GPU of THIS process behind one call (one host thread per device inside the
    library): host bytes in, ONE contiguous host index out -- reader::read (src/reader.rs:150) at N GPUs."""

    def __init__(self, devices):
        self._lib = _lib.load()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        h = C.c_void_p()
        rc = self._lib.csvb200_multi_create(devs, len(devices), C.byref(h))
        raise_for(rc, f"csvb200_multi_create({list(devices)}) failed")
        self._h = h
        self.devices = list(devices)

    def index_build_to_host(self, host_ptr: int, n: int, dst_ptr: int, dst_cap: int, cuts=None) -> int:
        ln = C.c_size_t()
        c = (C.c_size_t * len(cuts))(*cuts) if cuts is not None else None
        rc = self._lib.csvb200_multi_index_build_to_host(self._h, C.c_void_p(host_ptr), n, c, C.c_void_p(dst_ptr),
                                                         dst_cap, C.byref(ln))
        if rc:
            raise_for(rc, self._lib.csvb200_multi_last_error(self._h).decode("utf-8", "replace"))
        return ln.value

    def index_build(self, data, cuts=None) -> np.ndarray:
        a = _as_u8(data)
        out = np.empty(a.size // 2 + 4096, dtype=np.uint64)
        try:
            ln = self.index_build_to_host(a.ctypes.data, a.size, out.ctypes.data, out.size, cuts)
        except BufferError:
            out = np.empty(a.size + 2, dtype=np.uint64)
            ln = self.index_build_to_host(a.ctypes.data, a.size, out.ctypes.data, out.size, cuts)
        return out[:ln]

    def index_build_distributed(self, data, cuts=None) -> "MultiIndex":
        """csvb200_multi_index_build: the index stays distributed over the devices, for lookups."""
        a = _as_u8(data)
        c = (C.c_size_t * len(cuts))(*cuts) if cuts is not None else None
        h = C.c_void_p()
        rc = self._lib.csvb200_multi_index_build(self._h, a.ctypes.data, a.size, c, C.byref(h))
        if rc:
            raise_for(rc, self._lib.csvb200_multi_last_error(self._h).decode("utf-8", "replace"))
        return MultiIndex(self, h)

    def stream(self, k: int) -> int:
        return int(self._lib.csvb200_multi_stream(self._h, k) or 0)

    def stats(self) -> dict:
        st = _lib.MultiStats()
        self._lib.csvb200_multi_last_stats(self._h, C.byref(st))
        return {k: getattr(st, k) for k, _ in _lib.MultiStats._fields_}

    def close(self):
        if getattr(self, "_h", None):
            self._lib.csvb200_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiIndex:
    """csvb200_multi_index: segment k of the index in device k's HBM; lookups read remote segments over NVLink."""

    def __init__(self, multi: Multi, handle):
        self.multi, self._h, self._lib = multi, handle, multi._lib

    def _check(self, rc):
        if rc:
            raise_for(rc, self._lib.csvb200_multi_last_error(self.multi._h).decode("utf-8", "replace"))

    def __len__(self):
        return int(self._lib.csvb200_multi_index_len(self._h))

    def segments(self):
        out = []
        for k in range(len(self.multi.devices)):
            b, e, d = C.c_uint64(), C.c_uint64(), C.c_int()
            self._check(self._lib.csvb200_multi_index_segment(self._h, k, C.byref(b), C.byref(e), C.byref(d)))
            out.append({"base": b.value, "entries": e.value, "device": d.value})
        return out

    def to_host(self) -> np.ndarray:
        out = np.empty(len(self), dtype=np.uint64)
        self._check(self._lib.csvb200_multi_index_copy_out(self._h, out.ctypes.data, out.size))
        return out

    def tape_init(self, field_cnt: int, crlf: bool):
        rc_, j = C.c_uint32(), C.c_uint64()
        self._check(self._lib.csvb200_multi_tape_init(self._h, field_cnt, int(crlf), C.byref(rc_), C.byref(j)))
        return rc_.value, j.value

    def seek_fields(self, rec: np.ndarray, fld: np.ndarray) -> np.ndarray:
        rec = np.ascontiguousarray(rec, dtype=np.uint32)
        fld = np.ascontiguousarray(fld, dtype=np.uint32)
        out = np.empty((rec.size, 2), dtype=np.uint64)
        self._check(self._lib.csvb200_multi_seek_fields(self._h, rec.ctypes.data, fld.ctypes.data, rec.size, out.ctypes.data))
        return out

    def seek_records(self, rec: np.ndarray) -> np.ndarray:
        rec = np.ascontiguousarray(rec, dtype=np.uint32)
        out = np.empty((rec.size, 2), dtype=np.uint64)
        self._check(self._lib.csvb200_multi_seek_records(self._h, rec.ctypes.data, rec.size, out.ctypes.data))
        return out

    def materialize_columns(self, fields, first_record: int, nrec: int, flags: int = FIELD_RAW):
        """csvb200_multi_materialize_columns: as StructureIndex.materialize_columns, each device materialising the records
        it holds -> [(offsets, values)] per requested field."""
        f = np.ascontiguousarray(fields, dtype=np.uint32)
        k = int(f.size)
        offs = [np.zeros(nrec + 1, dtype=np.uint64) for _ in range(k)]
        p_off = (C.c_void_p * k)(*[o.ctypes.data for o in offs])
        lens = (C.c_size_t * k)()
        caps = (C.c_size_t * k)()
        rc = self._lib.csvb200_multi_materialize_columns(self._h, f.ctypes.data, k, first_record, nrec, flags, p_off, None,
                                                         caps, lens)
        if rc not in (0, 9):      # CSVB200_ERR_CAPACITY sizes the outputs
            self._check(rc)
        vals = [np.empty(int(lens[c]), dtype=np.uint8) for c in range(k)]
        if any(v.size for v in vals):
            p_out = (C.c_void_p * k)(*[v.ctypes.data if v.size else None for v in vals])
            caps = (C.c_size_t * k)(*[v.size for v in vals])
            self._check(self._lib.csvb200_multi_materialize_columns(self._h, f.ctypes.data, k, first_record, nrec, flags,
                                                                    p_off, p_out, caps, lens))
        return list(zip(offs, vals))

    def seek_fields_device(self, k: int, d_rec: int, d_fld: int, nq: int, d_out: int):
        self._check(self._lib.csvb200_multi_seek_fields_device(self._h, k, C.c_void_p(d_rec), C.c_void_p(d_fld), nq,
                                                               C.c_void_p(d_out)))

    def free(self):
        if getattr(self, "_h", None) and getattr(self.multi, "_h", None):
            self._lib.csvb200_multi_index_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class StructureIndex:
    """csvb200_index: the device-resident StructureIndex(Vec<CodeUnitPos>) (src/stage1.rs:61)."""

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self._lib = ctx._lib
        self._h = handle
        self._host = None

    def free(self):
        if getattr(self, "_h", None):
            self._lib.csvb200_index_free(self._h)
            self._h = None

    def __del__(self):
        try:
            if self.ctx._h:
                self.free()
        except Exception:
            pass

    def sync(self):
        self.ctx._check(self._lib.csvb200_index_sync(self._h))

    def __len__(self) -> int:
        self.sync()
        return int(self._lib.csvb200_index_len(self._h))

    @property
    def end_parity(self) -> int:
        self.sync()
        return int(self._lib.csvb200_index_end_parity(self._h))

    @property
    def device_ptr(self) -> int:
        return int(self._lib.csvb200_index_device_ptr(self._h) or 0)

    def to_host(self, out: np.ndarray | None = None) -> np.ndarray:
        """csvb200_index_copy_out: the index as a host u64 array (what Rust receives as Vec<usize>)."""
        n = len(self)
        if out is None:
            out = np.empty(n, dtype=np.uint64)
        self.ctx._check(self._lib.csvb200_index_copy_out(self._h, out.ctypes.data, out.size))
        return out[:n]

    def host(self) -> np.ndarray:
        if self._host is None:
            self._host = self.to_host()
        return self._host

    def shard_verify(self, d_gathered: int, world: int, d_final_out: int = 0):
        self.ctx._check(self._lib.csvb200_index_shard_verify(self._h, C.c_void_p(d_gathered), world,
                                                             C.c_void_p(d_final_out or 0)))

    def validation(self):
        """BUILD_VALIDATE by-products of the build launch -> (is_ascii, CR / LF bytes outside quotes)."""
        a, nl = C.c_int(), C.c_uint64()
        self.ctx._check(self._lib.csvb200_index_validation(self._h, C.byref(a), C.byref(nl)))
        return bool(a.value), int(nl.value)

    def validate_utf8(self):
        """from_utf8's valid_up_to (None = well-formed), reading only the tiles the build flagged as non-ASCII."""
        v = C.c_uint64()
        self.ctx._check(self._lib.csvb200_index_validate_utf8(self._h, C.byref(v)))
        return None if v.value == 0xFFFFFFFFFFFFFFFF else int(v.value)

    def shard_info(self) -> dict:
        """csvb200_index_shard_info (exchange builds): base slot, entries, true carry-in, whether it was re-indexed."""
        info = _lib.ShardInfo()
        self.ctx._check(self._lib.csvb200_index_shard_info(self._h, C.byref(info)))
        return {k: int(getattr(info, k)) for k, _ in _lib.ShardInfo._fields_}

    def shard_redone(self):
        """(misprediction rebuild ran?, true carry-in parity) of a speculative shard build."""
        r, c = C.c_int(), C.c_int()
        self.ctx._check(self._lib.csvb200_index_shard_redone(self._h, C.byref(r), C.byref(c)))
        return bool(r.value), c.value

    def save(self, path: str):
        import os
        self.ctx._check(self._lib.csvb200_index_save(self._h, os.fsencode(path)))

    def copy_out_ptr(self, dst_ptr: int, dst_cap: int):
        self.ctx._check(self._lib.csvb200_index_copy_out(self._h, C.c_void_p(dst_ptr), dst_cap))

    # -- Tape metadata / lookups ------------------------------------------------------------
    def tape_init(self, field_cnt: int, crlf: bool):
        rc_, j = C.c_uint32(), C.c_uint64()
        rc = self._lib.csvb200_tape_init(self._h, field_cnt, int(crlf), C.byref(rc_), C.byref(j))
        self.ctx._check(rc)
        return rc_.value, j.value

    def tape_validate(self, field_cnt: int, crlf: bool) -> dict:
        """csvb200_tape_validate: first slot whose separator class does not fit its place in the row."""
        rep = _lib.TapeReport()
        self.ctx._check(self._lib.csvb200_tape_validate(self._h, field_cnt, int(crlf), C.byref(rep)))
        return {k: int(getattr(rep, k)) for k, _ in _lib.TapeReport._fields_}

    def tape_chunks(self, num: int):
        """csvb200_tape_chunks: Tape::chunks(num) (src/tape.rs:95-140) + the byte range of every chunk."""
        arr = (_lib.Chunk * 256)()
        n = C.c_size_t()
        self.ctx._check(self._lib.csvb200_tape_chunks(self._h, num & 0xFF, arr, 256, C.byref(n)))
        return [{k: int(getattr(arr[i], k)) for k, _ in _lib.Chunk._fields_} for i in range(n.value)]

    def seek_record(self, r: int):
        rg, f = _lib.Range(), C.c_int()
        self.ctx._check(self._lib.csvb200_seek_record(self._h, r & 0xFFFFFFFF, C.byref(rg), C.byref(f)))
        return (rg.start, rg.end) if f.value else None

    def seek_field(self, r: int, fld: int):
        rg, f = _lib.Range(), C.c_int()
        self.ctx._check(self._lib.csvb200_seek_field(self._h, r & 0xFFFFFFFF, fld & 0xFFFFFFFF, C.byref(rg),
                                                     C.byref(f)))
        return (rg.start, rg.end) if f.value else None

    def seek_fields(self, rec: np.ndarray, fld: np.ndarray) -> np.ndarray:
        rec = np.ascontiguousarray(rec, dtype=np.uint32)
        fld = np.ascontiguousarray(fld, dtype=np.uint32)
        assert rec.size == fld.size
        out = np.empty((rec.size, 2), dtype=np.uint64)
        self.ctx._check(self._lib.csvb200_seek_fields(self._h, rec.ctypes.data, fld.ctypes.data, rec.size,
                                                      out.ctypes.data))
        return out

    def seek_records(self, rec: np.ndarray) -> np.ndarray:
        rec = np.ascontiguousarray(rec, dtype=np.uint32)
        out = np.empty((rec.size, 2), dtype=np.uint64)
        self.ctx._check(self._lib.csvb200_seek_records(self._h, rec.ctypes.data, rec.size, out.ctypes.data))
        return out

    def seek_fields_device(self, d_rec: int, d_fld: int, nq: int, d_out: int):
        self.ctx._check(self._lib.csvb200_seek_fields_device(self._h, C.c_void_p(d_rec), C.c_void_p(d_fld), nq,
                                                             C.c_void_p(d_out)))

    def seek_records_device(self, d_rec: int, nq: int, d_out: int):
        self.ctx._check(self._lib.csvb200_seek_records_device(self._h, C.c_void_p(d_rec), nq, C.c_void_p(d_out)))

    def materialize_column(self, field_idx: int, first_record: int, nrec: int, flags: int = FIELD_RAW):
        """csvb200_materialize_column: (offsets[nrec + 1], packed values) of one column."""
        offs = np.zeros(nrec + 1, dtype=np.uint64)
        ln = C.c_size_t()
        # first call sizes the output (CSVB200_ERR_CAPACITY is expected), second call fills it
        rc = self._lib.csvb200_materialize_column(self._h, field_idx, first_record, nrec, flags, offs.ctypes.data,
                                                  None, 0, C.byref(ln))
        if rc not in (0, 9):
            self.ctx._check(rc)
        out = np.empty(ln.value, dtype=np.uint8)
        if out.size:
            self.ctx._check(self._lib.csvb200_materialize_column(self._h, field_idx, first_record, nrec, flags,
                                                                 offs.ctypes.data, out.ctypes.data, out.size,
                                                                 C.byref(ln)))
        return offs, out

    def materialize_columns(self, fields, first_record: int, nrec: int, flags: int = FIELD_RAW):
        """csvb200_materialize_columns: several columns in one sweep -> [(offsets, values)] per requested field."""
        f = np.ascontiguousarray(fields, dtype=np.uint32)
        k = int(f.size)
        offs = [np.zeros(nrec + 1, dtype=np.uint64) for _ in range(k)]
        p_off = (C.c_void_p * k)(*[o.ctypes.data for o in offs])
        lens = (C.c_size_t * k)()
        caps = (C.c_size_t * k)()
        rc = self._lib.csvb200_materialize_columns(self._h, f.ctypes.data, k, first_record, nrec, flags, p_off, None, caps, lens)
        if rc not in (0, 9):      # CSVB200_ERR_CAPACITY sizes the outputs
            self.ctx._check(rc)
        vals = [np.empty(int(lens[c]), dtype=np.uint8) for c in range(k)]
        if any(v.size for v in vals):
            p_out = (C.c_void_p * k)(*[v.ctypes.data if v.size else None for v in vals])
            caps = (C.c_size_t * k)(*[v.size for v in vals])
            self.ctx._check(self._lib.csvb200_materialize_columns(self._h, f.ctypes.data, k, first_record, nrec, flags, p_off,
                                                                  p_out, caps, lens))
        return list(zip(offs, vals))

    def materialize_columns_device(self, fields, first_record: int, nrec: int, flags: int, d_offsets, d_outs=None, out_caps=None):
        f = np.ascontiguousarray(fields, dtype=np.uint32)
        k = int(f.size)
        p_off = (C.c_void_p * k)(*d_offsets)
        p_out = (C.c_void_p * k)(*d_outs) if d_outs is not None else None
        caps = (C.c_size_t * k)(*out_caps) if out_caps is not None else None
        self.ctx._check(self._lib.csvb200_materialize_columns_device(self._h, f.ctypes.data, k, first_record, nrec, flags, p_off,
                                                                     p_out, caps))

    def materialize_column_device(self, field_idx: int, first_record: int, nrec: int, flags: int, d_offsets: int,
                                  d_out: int, out_cap: int):
        self.ctx._check(self._lib.csvb200_materialize_column_device(self._h, field_idx, first_record, nrec, flags,
                                                                    C.c_void_p(d_offsets), C.c_void_p(d_out or 0),
                                                                    out_cap))

    def gather_fields(self, rec: np.ndarray, fld: np.ndarray):
        rec = np.ascontiguousarray(rec, dtype=np.uint32)
        fld = np.ascontiguousarray(fld, dtype=np.uint32)
        offs = np.zeros(rec.size + 1, dtype=np.uint64)
        # first call sizes the output (CSVB200_ERR_CAPACITY is expected), second call fills it
        rc = self._lib.csvb200_gather_fields(self._h, rec.ctypes.data, fld.ctypes.data, rec.size, offs.ctypes.data,
                                             None, 0)
        if rc not in (0, 9):
            self.ctx._check(rc)
        out = np.empty(int(offs[-1]), dtype=np.uint8)
        if out.size:
            self.ctx._check(self._lib.csvb200_gather_fields(self._h, rec.ctypes.data, fld.ctypes.data, rec.size,
                                                            offs.ctypes.data, out.ctypes.data, out.size))
        return offs, out
