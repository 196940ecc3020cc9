"""csvb200_seek_values and its device and distributed forms: the values behind a batch of lookups.  The reference is
always built from the existing calls and the oracle: the ranges of seek_fields / seek_records, the input bytes sliced
with them, and the oracle's field_value applied to every slice.  The distributed index must give the one-GPU results
byte for byte and bit for bit, with the cuts where values, records and shards meet."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

import csv_simd_b200 as cs
from csv_simd_b200.errors import InvalidState, ReferencePanic
from oracle import oracle as O
from tests.test_multi_materialize import _boundary_records, _cut_sets, _text
from tools import gen

pytestmark = pytest.mark.gpu

U64MAX = 0xFFFFFFFFFFFFFFFF
FLAGS = [0, 1, 2, 3]


def _want(idx, raw, rec, fld, flags):
    """(offsets, values, found) from the ranges of seek_fields / seek_records and the oracle's field_value"""
    rg = idx.seek_records(rec) if fld is None else idx.seek_fields(rec, fld)
    found = rg[:, 0] != U64MAX
    vals = []
    for i in range(rec.size):
        if not found[i]:
            vals.append(b"")
            continue
        s = raw[int(rg[i, 0]):int(rg[i, 1])]
        vals.append(s if fld is None else O.field_value(s, flags))
    offs = np.zeros(rec.size + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(v) for v in vals], dtype=np.uint64)
    return offs, b"".join(vals), found


def _same(got, want, what):
    g_off, g_val, g_found = got
    w_off, w_val, w_found = want
    assert (g_off == w_off).all(), what
    assert g_val.tobytes() == bytes(w_val), what
    assert (g_found == w_found).all(), what


def _queries(rc, field_cnt, seed, n=3000):
    """every (record, field) of the first and last rows, None probes past both ends and at r = 0xFFFFFFFF, duplicates
    and random queries"""
    rng = np.random.default_rng(seed)
    rows = list(range(0, 12)) + list(range(rc - 6, rc + 2))
    rec = [r for r in rows for _ in range(field_cnt + 2)]
    fld = [f for _ in rows for f in range(field_cnt + 2)]
    rec += [0xFFFFFFFF] * 4 + [rc - 1, rc, rc + 7]
    fld += [0, 1, field_cnt, 0xFFFFFFFF, 0, 1, 2]
    rec += list(rng.integers(0, rc + 2, n))
    fld += list(rng.integers(0, field_cnt + 1, n))
    rec += rec[:50]
    fld += fld[:50]
    return np.array(rec, dtype=np.uint32), np.array(fld, dtype=np.uint32)


@pytest.fixture(params=[4, 8], ids=["compact", "u64"])
def any_ctx(request, ctx, monkeypatch):
    if request.param == 4:
        yield ctx
        return
    monkeypatch.setenv("CSVB200_INDEX_ENTRY_BYTES", "8")
    c = cs.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("crlf", [False, True], ids=["lf", "crlf"])
def test_parity_with_ranges_and_oracle(any_ctx, crlf):
    raw = _text()
    if crlf:
        raw = raw.replace(b"\n", b"\r\n")
    idx = any_ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, _ = idx.tape_init(3, crlf)
    rec, fld = _queries(rc, 3, seed=3)
    for flags in FLAGS:
        for nq in (0, 1, 63, 64, 65, rec.size):
            r, f = rec[-nq:] if nq else rec[:0], fld[-nq:] if nq else fld[:0]
            _same(idx.seek_values(r, f, flags), _want(idx, raw, r, f, flags), (crlf, flags, nq))
    # records: the raw seek_records slices
    for nq in (0, 1, 65, rec.size):
        r = rec[:nq]
        _same(idx.seek_values(r), _want(idx, raw, r, None, 0), ("records", nq))
    for flags in (1, 2, 3):
        with pytest.raises(ValueError):
            idx.seek_values(rec[:5], None, flags)
    with pytest.raises(ValueError):
        idx.seek_values(rec[:5], fld[:5], 4)
    # gather_fields is the raw form
    g_off, g_val = idx.gather_fields(rec[:500], fld[:500])
    w_off, w_val, _ = _want(idx, raw, rec[:500], fld[:500], 0)
    assert (g_off == w_off).all() and g_val.tobytes() == w_val
    idx.free()


def _c_call(idx, rec, fld, flags, out_cap, out=None):
    offs = np.full(rec.size + 1, 7, dtype=np.uint64)
    words = np.zeros((rec.size + 63) // 64 + 1, dtype=np.uint64)
    ln = C.c_size_t(12345)
    code = idx._lib.csvb200_seek_values(idx._h, rec.ctypes.data, fld.ctypes.data if fld is not None else None, rec.size,
                                        flags, offs.ctypes.data, out.ctypes.data if out is not None else None, out_cap,
                                        C.byref(ln), words.ctypes.data)
    return code, offs, ln.value


def test_status_codes(ctx):
    raw = _text()
    rec = np.array([0, 3, 7], dtype=np.uint32)
    fld = np.array([1, 2, 0], dtype=np.uint32)
    # InvalidState: before tape_init, without the input bytes, and an index read from disk
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    with pytest.raises(InvalidState):
        idx.seek_values(rec, fld)
    rc, _ = idx.tape_init(3, False)
    bare = ctx.index_build(raw)
    bare.tape_init(3, False)
    with pytest.raises(InvalidState):
        bare.seek_values(rec, fld)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "t.idx")
        bare.save(path)
        loaded = ctx.index_load(path)
        with pytest.raises(InvalidState):
            loaded.seek_values(rec, fld)
        loaded.free()
    bare.free()
    # CAPACITY: offsets and out_len valid, out not written
    w_off, w_val, _ = _want(idx, raw, rec, fld, 3)
    out = np.full(len(w_val), 0xEE, dtype=np.uint8)
    code, offs, ln = _c_call(idx, rec, fld, 3, len(w_val) - 1, out)
    assert code == 9 and ln == len(w_val) and (offs == w_off).all() and (out == 0xEE).all()
    code, offs, ln = _c_call(idx, rec, fld, 3, len(w_val), out)
    assert code == 0 and out.tobytes() == w_val
    with pytest.raises(BufferError):
        cs.errors.raise_for(_c_call(idx, rec, fld, 3, 0)[0])
    # INVALID_ARG: null arrays
    assert idx._lib.csvb200_seek_values(idx._h, None, None, 3, 0, offs.ctypes.data, None, 0, C.byref(C.c_size_t()), None) == 1
    assert idx._lib.csvb200_seek_values(idx._h, rec.ctypes.data, None, 3, 0, None, None, 0, C.byref(C.c_size_t()), None) == 1
    idx.free()


def test_outside_bytes_wins_over_capacity(ctx):
    """An index object that holds fewer bytes than its positions refer to: OUT_OF_BOUNDS, before the capacity check;
    its device form gives an empty value there and writes nothing."""
    import torch
    data, _ = gen.unquoted(1 << 20, seed=7)
    raw = data.tobytes()
    full = O.closed_form_numpy(raw)
    cut = int(full[16 * 1000]) + 1
    shard = np.frombuffer(raw[cut:], dtype=np.uint8)
    dev = torch.device("cuda", ctx.device)
    d = torch.zeros(shard.size + 64 + 16, dtype=torch.uint8, device=dev)
    off = (-d.data_ptr()) % 16
    d[off:off + shard.size].copy_(torch.from_numpy(shard.copy()))
    torch.cuda.synchronize()
    idx = ctx.index_build_shard_device(d.data_ptr() + off, shard.size, 0, cut, True)
    rc, _ = idx.tape_init(16, False)
    rec = np.array([0, 5, 17, rc - 2], dtype=np.uint32)
    fld = np.array([1, 0, 15, 7], dtype=np.uint32)
    offs, vals, found = idx.seek_values(rec, fld)
    rg = idx.seek_fields(rec, fld)
    assert found.all()
    for i in range(rec.size):
        assert vals[int(offs[i]):int(offs[i + 1])].tobytes() == raw[int(rg[i, 0]):int(rg[i, 1])]
    wrapped = ctx.index_wrap_device(idx.device_ptr, len(idx), 100, d.data_ptr() + off)
    wrapped.tape_init(16, False)
    with pytest.raises(ReferencePanic):
        wrapped.seek_values(rec[:1], fld[:1])
    code, _, _ = _c_call(wrapped, rec, fld, 0, 0)
    assert code == 10   # CSVB200_ERR_OUT_OF_BOUNDS, not CSVB200_ERR_CAPACITY
    d_rec = torch.from_numpy(rec.view(np.int32)).to(dev)
    d_fld = torch.from_numpy(fld.view(np.int32)).to(dev)
    d_off = torch.full((rec.size + 1,), 7, dtype=torch.int64, device=dev)
    d_out = torch.full((64,), 0xEE, dtype=torch.uint8, device=dev)
    wrapped.seek_values_device(d_rec.data_ptr(), d_fld.data_ptr(), rec.size, 0, d_off.data_ptr(), d_out.data_ptr(), 64)
    torch.cuda.synchronize()
    assert (d_off.cpu().numpy() == 0).all() and (d_out.cpu().numpy() == 0xEE).all()
    wrapped.free()
    idx.free()


def _device_call(idx, rec, fld, flags, out_cap=None, values=True, k=None):
    import torch
    dev = torch.device("cuda", idx.ctx.device if k is None else idx.multi.devices[k])
    nq = rec.size
    d_rec = torch.from_numpy(rec.view(np.int32).copy()).to(dev)
    d_fld = torch.from_numpy(fld.view(np.int32).copy()).to(dev) if fld is not None else None
    d_off = torch.full((nq + 1,), -1, dtype=torch.int64, device=dev)
    d_found = torch.full(((nq + 63) // 64 + 1,), -1, dtype=torch.int64, device=dev)
    cap = out_cap if out_cap is not None else 1 << 16
    d_out = torch.full((cap + 64,), 0xEE, dtype=torch.uint8, device=dev)
    args = (d_rec.data_ptr(), d_fld.data_ptr() if d_fld is not None else None, nq, flags, d_off.data_ptr(),
            d_out.data_ptr() if values else None, cap, d_found.data_ptr())
    if k is None:
        idx.seek_values_device(*args)
    else:
        idx.seek_values_device(k, *args)
    torch.cuda.synchronize(dev)
    offs = d_off.cpu().numpy().view(np.uint64)
    words = d_found.cpu().numpy().view(np.uint64)[:(nq + 63) // 64]
    found = np.unpackbits(words.view(np.uint8), bitorder="little")[:nq].astype(bool)
    return offs, d_out.cpu().numpy(), found


def test_device_form(ctx):
    raw = _text()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, _ = idx.tape_init(3, False)
    rec, fld = _queries(rc, 3, seed=4, n=700)
    for flags in FLAGS:
        w_off, w_val, w_found = idx.seek_values(rec, fld, flags)
        offs, out, found = _device_call(idx, rec, fld, flags)
        assert (offs == w_off).all() and (found == w_found).all()
        assert out[:w_val.size].tobytes() == w_val.tobytes() and (out[w_val.size:] == 0xEE).all()
        # offsets only
        offs, out, found = _device_call(idx, rec, fld, flags, values=False)
        assert (offs == w_off).all() and (found == w_found).all() and (out == 0xEE).all()
        # a small out_cap: whole values up to it, nothing past it
        cap = int(w_val.size // 3)
        offs, out, _ = _device_call(idx, rec, fld, flags, out_cap=cap)
        for q in range(rec.size):
            a, b = int(w_off[q]), int(w_off[q + 1])
            if b <= cap:
                assert out[a:b].tobytes() == w_val[a:b].tobytes()
        assert (out[cap:] == 0xEE).all()
    w_off, w_val, w_found = idx.seek_values(rec)
    offs, out, found = _device_call(idx, rec, None, 0)
    assert (offs == w_off).all() and (found == w_found).all() and out[:w_val.size].tobytes() == w_val.tobytes()
    idx.free()


def test_chunked_host_form(ctx):
    """More queries than one chunk of the host form (2^20): offsets, bytes and found bits against ranges + numpy."""
    data, _ = gen.unquoted(48 << 20, seed=9)
    raw = data.tobytes()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, _ = idx.tape_init(16, False)
    rec, fld = gen.queries(2_600_000, rc, 16, seed=10)
    rec[::1001] = rc - 1 + np.arange(rec[::1001].size, dtype=np.uint32) % 3
    fld[7::997] = 16 + np.arange(fld[7::997].size, dtype=np.uint32) % 2
    offs, vals, found = idx.seek_values(rec, fld)
    rg = idx.seek_fields(rec, fld)
    w_found = rg[:, 0] != U64MAX
    a = np.where(w_found, rg[:, 0], 0).astype(np.int64)
    lens = np.where(w_found, rg[:, 1].astype(np.int64) - a, 0)
    assert (found == w_found).all() and (~w_found).sum() > 1000
    assert offs[0] == 0 and (np.diff(offs.astype(np.int64)) == lens).all()
    pos = np.arange(int(lens.sum()), dtype=np.int64) - np.repeat(offs[:-1].astype(np.int64), lens) + np.repeat(a, lens)
    assert (vals == data[pos]).all()
    idx.free()


def _multi_check(mi, idx, raw, rec, fld, what, device=True):
    for flags in (FLAGS if fld is not None else [0]):
        want = idx.seek_values(rec, fld, flags)
        got = mi.seek_values(rec, fld, flags)
        _same(got, (want[0], want[1].tobytes(), want[2]), (what, flags))
        if not device:
            continue
        for k in range(len(mi.multi.devices)):
            offs, out, found = _device_call(mi, rec, fld, flags, out_cap=max(int(want[1].size), 1), k=k)
            assert (offs == want[0]).all() and (found == want[2]).all(), (what, flags, k)
            assert out[:want[1].size].tobytes() == want[1].tobytes(), (what, flags, k)


def _cut_queries(mi, host, jump, rc, cuts):
    """every field whose range contains a cut and every record whose slots span segments"""
    rec, fld = [], []
    for r in range(rc - 1):
        for f in range(3):
            s = (r + 1) * jump + f
            a, b = int(host[s]) + 1, int(host[s + 1])
            if any(a <= c < b for c in cuts[1:-1]):
                rec.append(r)
                fld.append(f)
    recs = _boundary_records(mi, jump, rc)
    return np.array(rec, dtype=np.uint32), np.array(fld, dtype=np.uint32), np.array(recs, dtype=np.uint32)


def _run_cut_sets(ctx, devices_for):
    raw = _text()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, jump = idx.tape_init(3, False)
    host = idx.to_host()
    for name, cuts in _cut_sets(raw, host).items():
        g = len(cuts) - 1
        m = cs.Multi(devices_for(g))
        mi = m.index_build_distributed(raw, cuts)
        mi.tape_init(3, False)
        rec, fld, recs = _cut_queries(mi, host, jump, rc, cuts)
        assert rec.size and recs.size, name
        _multi_check(mi, idx, raw, rec, fld, name)
        _multi_check(mi, idx, raw, recs, None, name)
        for nq in (1, 63, 64 * g - 1, 64 * g + 5, 1500):
            r, f = _queries(rc, 3, seed=nq, n=nq)
            r, f = r[-nq:], f[-nq:]
            _multi_check(mi, idx, raw, r, f, (name, nq), device=nq == 1500)
            _multi_check(mi, idx, raw, r, None, (name, nq, "records"), device=False)
        _multi_check(mi, idx, raw, rec[:0], fld[:0], (name, 0), device=False)
        with pytest.raises(ValueError):
            mi.seek_values(rec[:3], None, 1)
        mi.free()
        m.close()
    idx.free()


def test_distributed_cut_placements_on_one_gpu(ctx):
    _run_cut_sets(ctx, lambda g: [ctx.device] * g)


def test_distributed_cut_placements_across_gpus(ctx):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs at least 2 GPUs")
    _run_cut_sets(ctx, lambda g: [k % ndev for k in range(g)])


def test_distributed_status_codes(ctx):
    raw = _text()
    m = cs.Multi([ctx.device] * 3)
    mi = m.index_build_distributed(raw)
    rec = np.array([0, 1], dtype=np.uint32)
    with pytest.raises(InvalidState):
        mi.seek_values(rec, rec)
    mi.tape_init(3, False)
    with pytest.raises(ValueError):
        mi.seek_values(rec, rec, 4)
    offs = np.zeros(3, dtype=np.uint64)
    ln = C.c_size_t()
    code = mi._lib.csvb200_multi_seek_values(mi._h, rec.ctypes.data, rec.ctypes.data, 2, 0, offs.ctypes.data, None, 0,
                                             C.byref(ln), None)
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    idx.tape_init(3, False)
    w_off, w_val, _ = idx.seek_values(rec, rec)
    assert code == 9 and ln.value == w_val.size and (offs == w_off).all()
    idx.free()
    mi.free()
    m.close()
