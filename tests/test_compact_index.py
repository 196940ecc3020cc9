"""Compact (4-byte entry) storage of the device-resident index: a context made with CSVB200_INDEX_ENTRY_BYTES=8 keeps
8-byte entries and is the reference; a default context stores the index of csvb200_index_build / _build_device over at
most 4 GiB as u32 positions.  Every consumer must give the same answers on both, for both build kernels, before and
after csvb200_index_device_ptr has widened the index in place; the entries themselves are checked against the oracle."""
import os
import tempfile

import numpy as np
import pytest

import csv_simd_b200 as cs
from oracle import oracle as O
from tools import gen

pytestmark = pytest.mark.gpu


def _make_ctx(kernel=None, entry_bytes=None):
    saved = {k: os.environ.get(k) for k in ("CSVB200_KERNEL", "CSVB200_INDEX_ENTRY_BYTES")}
    try:
        for k, v in (("CSVB200_KERNEL", kernel), ("CSVB200_INDEX_ENTRY_BYTES", entry_bytes)):
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        return cs.Context(0)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module", params=["simple", "tma"])
def pair(request):
    """(compact context, 8-byte context) forced onto one build kernel."""
    c4, c8 = _make_ctx(request.param), _make_ctx(request.param, "8")
    yield c4, c8
    c4.close()
    c8.close()


def _random_bytes(n, seed):
    alphabet = np.frombuffer(b'ab,,\n"\r x', dtype=np.uint8)
    return alphabet[np.random.default_rng(seed).integers(0, alphabet.size, n)].tobytes()


def _inputs():
    return {
        "cfg2_64mib": gen.unquoted(64 << 20, seed=61)[0].tobytes(),
        "cfg3_64mib": gen.quoted(64 << 20, seed=62)[0].tobytes(),
        "random_odd_a": _random_bytes(1_000_003, 63),
        "random_odd_b": _random_bytes(3_333_331, 64),
        "short": b'a,"b\n",c\n1,2,3\n',
        "one_byte": b",",
        "empty": b"",
    }


@pytest.fixture(scope="module")
def inputs():
    return _inputs()


def _pinned_copy_out(idx):
    import torch
    out = torch.empty(max(len(idx), 1), dtype=torch.int64).pin_memory()
    idx.copy_out_ptr(out.data_ptr(), out.numel())
    return out.numpy()[:len(idx)].view(np.uint64).copy()


def _outcome(fn):
    """The value of fn(), or the exception type it raised: both contexts must agree on either."""
    try:
        return fn()
    except (cs.errors.StructureError, MemoryError, ValueError) as e:
        return type(e).__name__


def _consumers(idx, nfields, seed=5):
    """Everything the single-GPU consumers answer about one index (host values only, comparable with ==)."""
    import torch
    res = {"len": len(idx), "end_parity": idx.end_parity}
    res["to_host"] = idx.to_host().tobytes()
    res["to_host_pinned"] = _pinned_copy_out(idx).tobytes()
    res["tape_validate"] = _outcome(lambda: idx.tape_validate(nfields, False))
    res["tape_validate_3"] = _outcome(lambda: idx.tape_validate(3, False))     # fails early on most inputs
    res["tape_init"] = _outcome(lambda: idx.tape_init(nfields, False))
    if not isinstance(res["tape_init"], tuple):
        return res
    rc, _ = res["tape_init"]
    res["chunks"] = _outcome(lambda: idx.tape_chunks(4))
    rng = np.random.default_rng(seed)
    nq = 4096
    rec = rng.integers(0, rc + 2, nq).astype(np.uint32)
    fld = rng.integers(0, nfields + 1, nq).astype(np.uint32)
    res["seek_fields"] = idx.seek_fields(rec, fld).tobytes()
    res["seek_records"] = idx.seek_records(rec).tobytes()
    dev = torch.device("cuda", 0)
    d_rec = torch.from_numpy(rec.view(np.int32)).to(dev)
    d_fld = torch.from_numpy(fld.view(np.int32)).to(dev)
    d_out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    idx.seek_fields_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, d_out.data_ptr())
    torch.cuda.synchronize()
    res["seek_fields_device"] = d_out.cpu().numpy().tobytes()
    idx.seek_records_device(d_rec.data_ptr(), nq, d_out.data_ptr())
    torch.cuda.synchronize()
    res["seek_records_device"] = d_out.cpu().numpy().tobytes()
    res["gather"] = _outcome(lambda: tuple(a.tobytes() for a in idx.gather_fields(rec[:512], fld[:512])))
    nrec = max(min(rc - 1, 20000), 0)
    for ncols in (1, 4, 32):
        fields = [(3 * c) % nfields for c in range(ncols)]
        for flags in range(4):
            cols = idx.materialize_columns(fields, 0, nrec, flags)
            res[f"mat_{ncols}_{flags}"] = [(o.tobytes(), v.tobytes()) for o, v in cols]
            d_offs = [torch.empty(nrec + 1, dtype=torch.int64, device=dev) for _ in fields]
            d_vals = [torch.empty(max(v.size, 1), dtype=torch.uint8, device=dev) for _, v in cols]
            idx.materialize_columns_device(fields, 0, nrec, flags, [t.data_ptr() for t in d_offs],
                                           [t.data_ptr() for t in d_vals], [v.size for _, v in cols])
            torch.cuda.synchronize()
            res[f"mat_dev_{ncols}_{flags}"] = [(o.cpu().numpy().tobytes(), t.cpu().numpy()[:v.size].tobytes())
                                               for o, t, (_, v) in zip(d_offs, d_vals, cols)]
    return res


def _nfields(name):
    return 16 if name.startswith("cfg") else 3


@pytest.mark.parametrize("name", list(_inputs().keys()))
def test_compact_matches_8_byte_and_oracle(pair, inputs, name):
    import torch
    raw = inputs[name]
    c4, c8 = pair
    want = O.read_sse(raw) if len(raw) >= 64 else None
    flags = cs.BUILD_KEEP_BYTES | cs.BUILD_VALIDATE
    i4, i8 = c4.index_build(raw, flags), c8.index_build(raw, flags)
    host = i4.to_host()
    if want is not None:
        assert host.shape == want.shape and (host == want).all()
    assert i4.validation() == i8.validation()
    assert i4.validate_utf8() == i8.validate_utf8()
    r8 = _consumers(i8, _nfields(name))
    assert _consumers(i4, _nfields(name)) == r8
    with tempfile.TemporaryDirectory() as td:
        p4, p8 = os.path.join(td, "a.idx"), os.path.join(td, "b.idx")
        i4.save(p4)
        i8.save(p8)
        assert open(p4, "rb").read() == open(p8, "rb").read()
        loaded = c4.index_load(p4)
        assert (loaded.to_host() == host).all()
        loaded.free()
    # csvb200_index_device_ptr widens the compact index in place, once: u64 values, then every consumer again
    ptr = i4.device_ptr
    assert ptr != 0 and i4.device_ptr == ptr
    E = len(i4)

    class _Raw:
        __cuda_array_interface__ = {"shape": (E,), "typestr": "<u8", "data": (ptr, False), "version": 2}
    if E:
        got = torch.as_tensor(_Raw(), device=torch.device("cuda", 0)).view(torch.int64).cpu().numpy().view(np.uint64)
        assert (got == host).all()
    assert _consumers(i4, _nfields(name)) == r8
    i4.free()
    i8.free()


def test_capacity_overflow_rebuild_compact(pair):
    c4, c8 = pair
    raw = b",\n" * (3 << 19) + b'"a,b",\n' * 1000       # one separator per byte: far above the 1/64 reserve
    for c in (c4, c8):
        c.set_reserve(1, 64)
    try:
        a, b = c4.index_build(raw), c8.index_build(raw)
        assert (a.to_host() == O.read_sse(raw)).all() and (b.to_host() == a.to_host()).all()
        a.free()
        b.free()
    finally:
        for c in (c4, c8):
            c.set_reserve(1, 3)


def test_unsynchronised_compact_and_shard_builds_alternate():
    """Compact builds and 8-byte shard builds of the same sizes on one context, none synchronised before the last."""
    import torch
    c = _make_ctx()
    dev = torch.device("cuda", 0)
    data = gen.unquoted(8 << 20, seed=65)[0]
    n = data.size
    d = torch.empty(n + 64, dtype=torch.uint8, device=dev)
    d[:n].copy_(torch.from_numpy(data))
    torch.cuda.synchronize()
    want = O.read_sse(data.tobytes())
    idxs = [c.index_build_device(d.data_ptr(), n) if k % 2 == 0 else c.index_build_shard_device(d.data_ptr(), n, 0, 0, True)
            for k in range(5)]
    for i in idxs:
        assert (i.to_host() == want).all()
        i.free()
    c.close()


@pytest.mark.parametrize("extra", [0, 1])
def test_4gib_edge(extra):
    """n = 2^32 with a separator in the last byte is compact and its last entry is 0xFFFFFFFF; n = 2^32 + 1 with a
    separator in the last byte has an entry of 2^32, which only 8-byte storage holds."""
    import torch
    dev = torch.device("cuda", 0)
    n = (1 << 32) + extra
    free, _ = torch.cuda.mem_get_info(dev)
    if free < n + (4 << 30):
        pytest.skip("needs ~8 GB of free device memory")
    step = 4096
    d = torch.full((n + 64,), 0x61, dtype=torch.uint8, device=dev)
    d[step - 1::step] = 0x2C
    d[n - 1] = 0x0A
    d[n:] = 0
    torch.cuda.synchronize()
    c = _make_ctx()
    c.set_reserve(1, 2048)
    try:
        idx = c.index_build_device(d.data_ptr(), n)
        want = np.concatenate([[0], np.arange(step - 1, n, step, dtype=np.uint64)]).astype(np.uint64)
        if extra:
            want = np.append(want, np.uint64(n - 1))
        assert len(idx) == want.size
        host = idx.to_host()
        assert int(host[-1]) == n - 1 and (host[-4096:] == want[-4096:]).all() and (host == want).all()
        ptr = idx.device_ptr
        E = len(idx)

        class _Raw:
            __cuda_array_interface__ = {"shape": (E,), "typestr": "<u8", "data": (ptr, False), "version": 2}
        entries = torch.as_tensor(_Raw(), device=dev).view(torch.int64)
        probe = torch.randint(0, E, (1 << 16,), device=dev, generator=torch.Generator(device=dev).manual_seed(3))
        got = entries[probe].cpu().numpy().view(np.uint64)
        assert (got == want[probe.cpu().numpy()]).all()
        idx.free()
    finally:
        c.close()
        del d
        torch.cuda.empty_cache()
