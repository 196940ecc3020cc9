"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the
same inputs (bit-exact: the index is integer data), the committed golden vectors, and -- at
BASELINE.json's full sizes -- size-independent properties."""
import os
import tempfile

import numpy as np
import pytest

import csv_simd_b200 as cs
from oracle import oracle as O
from tests import cases
from tests.conftest import golden_bytes
from tools import gen

pytestmark = pytest.mark.gpu

U64MAX = 0xFFFFFFFFFFFFFFFF


def build(ctx, data, flags=0):
    idx = ctx.index_build(data, flags)
    out = idx.to_host().copy()
    par = idx.end_parity
    idx.free()
    return out, par


# ---- golden vectors (config 1: res/sample.csv -> stage1 -> tape index) -------------------------
@pytest.mark.parametrize("name", ["reader_test01.csv", "sample.csv", "sample_rx.csv"])
def test_golden_index(ctx, golden, name):
    data = golden_bytes(name)
    got, _ = build(ctx, data)
    assert got.tolist() == golden[name]["index"]


def test_reference_mk_index_pin(ctx):
    got, _ = build(ctx, golden_bytes("reader_test01.csv"))  # src/reader.rs:318-327
    assert got[1] == 4 and got[-1] == 95


@pytest.mark.parametrize("name", ["sample.csv", "sample_rx.csv"])
def test_golden_tape_and_seeks(ctx, golden, name):
    g = golden[name]
    with tempfile.NamedTemporaryFile(suffix=".csv", delete=False) as f:
        f.write(golden_bytes(name))
        path = f.name
    try:
        tape = cs.create(path, ctx)  # the reference's factory: open -> mmap -> Header -> read -> Tape
        assert tape.header() == g["header"]
        assert tape.record_cnt() == g["record_cnt"] and tape.record_jump_size() == g["jump"]
        assert tape.index().to_host().tolist() == g["index"]
        data = golden_bytes(name)
        for r, want in g["seek_record"].items():
            assert tape.seek_record(int(r)) == want
            rg = tape.index().seek_record(int(r))  # device scalar path
            assert (None if rg is None else data[rg[0]:rg[1]].decode()) == want
        for key, want in g["seek_field"].items():
            r, f = map(int, key.split(","))
            assert tape.seek_field(r, f) == want
            rg = tape.index().seek_field(r, f)
            assert (None if rg is None else data[rg[0]:rg[1]].decode()) == want
        # Display of WithRecordSource prints first / last record: last = record_cnt - 2
        assert tape.seek_record(g["record_cnt"] - 2) is not None
        assert tape.seek_record(g["record_cnt"] - 1) is None
    finally:
        os.unlink(path)


def test_invalid_csv_format(ctx):
    with tempfile.NamedTemporaryFile(suffix=".csv", delete=False) as f:
        f.write(golden_bytes("reader_test01.csv"))  # ragged last row: (E-1) % jump != 0
        path = f.name
    try:
        with pytest.raises(cs.InvalidCsvFormat):
            cs.create(path, ctx)
    finally:
        os.unlink(path)


def test_seek_before_init_is_invalid_state(ctx):
    data = golden_bytes("sample.csv")
    mm = cs.Mmap(data=data)
    core = cs.TapeCore.create(mm, cs.reader.read(mm, ctx), cs.Header.new(mm))
    with pytest.raises(cs.InvalidState):   # record_cnt() is None before init (record_source.rs:77-79)
        core.seek_record(0)
    with pytest.raises(cs.InvalidState):
        core.index().seek_field(0, 0)      # C ABI: csvb200_tape_init not called yet
    core.init()
    assert core.seek_record(0) == 'Edm nd,3, "o"'


# ---- edge semantics ---------------------------------------------------------------------------
@pytest.mark.parametrize("name,data", cases.edge_cases(), ids=[c[0] for c in cases.edge_cases()])
def test_edge_cases_vs_sse_oracle(ctx, name, data):
    want = O.read_sse(data)  # literal restatement of the reference
    got, par = build(ctx, data)
    assert got.shape == want.shape and (got == want).all()
    assert par == (data.count(b'"') & 1)


@pytest.mark.parametrize("name,data", cases.small_cases(), ids=[c[0] for c in cases.small_cases()])
def test_small_inputs(ctx, name, data):
    # n < 64: the reference panics; the C ABI returns the closed form, or mirrors the panic on request
    want, _ = O.read_closed_form(data)
    got, _ = build(ctx, data)
    assert (got == want).all()
    with pytest.raises(cs.ReferencePanic):
        ctx.index_build(data, cs.BUILD_STRICT_MIN64)
    with pytest.raises(cs.ReferencePanic):
        cs.reader.read(data, ctx)


def test_fuzz_vs_oracle(ctx):
    for seed in range(120):
        n = 64 + (seed * 7919) % 70000
        data = cases.full_random(n, seed) if seed % 4 == 0 else cases.rand_bytes(n, seed)
        want = O.read_sse(data)
        got, _ = build(ctx, data)
        assert got.shape == want.shape and (got == want).all(), (seed, n)


def test_capacity_overflow_rebuild(ctx):
    # denser than the reserve heuristic (one entry per byte): transparently rebuilt with the exact size
    data = b"," * (1 << 20)
    ctx.set_reserve(1, 64)
    try:
        got, _ = build(ctx, data)
    finally:
        ctx.set_reserve(1, 3)
    assert got.size == (1 << 20) + 1 and (got[1:] == np.arange(1 << 20, dtype=np.uint64)).all()


# ---- K1 known-answer exports --------------------------------------------------------------------
def test_block_masks_vs_closed_form(ctx):
    data = np.frombuffer(cases.rand_bytes(100003, 5), dtype=np.uint8)
    q, s = ctx.block_masks(data)
    pad = np.zeros(q.size * 64, dtype=np.uint8)
    pad[:data.size] = data
    wq = np.packbits((pad == 0x22).reshape(-1, 64), axis=1, bitorder="little").view(np.uint64).ravel()
    ws = np.packbits(((pad == 0x2C) | (pad == 0x0D) | (pad == 0x0A)).reshape(-1, 64), axis=1,
                     bitorder="little").view(np.uint64).ravel()
    assert (q == wq).all() and (s == ws).all()


def test_class_bytes_vs_structure_run(ctx):
    data = bytes(range(256)) * 3 + cases.rand_bytes(16 * 50, 3)
    got = ctx.class_bytes(data)
    want = np.concatenate([O.structure_run(data, at) for at in range(0, len(data), 16)])
    assert (got == want).all()


# ---- sharded build: arbitrary cuts, forced inside quotes / between "" / between CR and LF -------
def _shard_chain(ctx, data, cuts):
    import torch
    dev = torch.device("cuda", ctx.device)
    segs, par, ps = [], 0, []
    for k in range(len(cuts) - 1):
        lo, hi = cuts[k], cuts[k + 1]
        t = torch.from_numpy(np.frombuffer(data, dtype=np.uint8)[lo:hi].copy()).to(dev)
        p = ctx.shard_quote_parity(t.data_ptr(), hi - lo)
        idx = ctx.index_build_shard_device(t.data_ptr(), hi - lo, par, lo, emit_sentinel=(k == 0))
        segs.append(idx.to_host().copy())
        assert idx.end_parity == par ^ p
        idx.free()
        ps.append(p)
        par ^= p
    return np.concatenate(segs), ps


def test_sharded_equals_single(ctx):
    data, _ = gen.quoted(3 << 20, seed=44)
    data = data.tobytes()
    want = O.closed_form_numpy(data)
    n = len(data)
    for G in (2, 4, 8):
        cuts = [0] + [(k * n) // G + 37 * k + 13 for k in range(1, G)] + [n]
        got, _ = _shard_chain(ctx, data, cuts)
        assert got.shape == want.shape and (got == want).all(), G


def test_sharded_forced_boundaries(ctx):
    body = b'id,"text, with ""escapes"" and\r\nnewlines",tail\r\n' * 4000
    data = b"h1,h2,h3\r\n" + body
    want = O.closed_form_numpy(data)
    inside = data.index(b"text")            # (a) inside a quoted field
    esc = data.index(b'""') + 1             # (b) between the two quotes of ""
    crlf = data.index(b"\r\n", 50) + 1      # (c) between CR and LF
    for cut in (inside, esc, crlf, inside + 48 * 1000, esc + 48 * 2001, crlf + 48 * 3999):
        got, ps = _shard_chain(ctx, data, [0, cut, len(data)])
        assert (got == want).all(), cut
    got, _ = _shard_chain(ctx, data, [0, inside, esc, crlf, len(data) // 2 + 5, len(data)])
    assert (got == want).all()


# ---- batched lookups (config 5 in miniature) ------------------------------------------------------
def test_batched_seeks_vs_oracle(ctx):
    data, rows = gen.unquoted(2 << 20, seed=45, nfields=256, modulus=10 ** 15)
    raw = data.tobytes()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    host = idx.to_host()
    want_idx = O.closed_form_numpy(raw)
    assert (host == want_idx).all()
    rc, jump = idx.tape_init(256, False)
    assert (jump, rc) == O.tape_init(host.size, 256, False) and rc == rows + 1
    rec, fld = gen.queries(20000, rc, 256, seed=46)
    # 1 % tail of out-of-range probes must come back as None
    rec[-200:-100] = rc - 1 + np.arange(100, dtype=np.uint32)
    fld[-100:] = 256 + np.arange(100, dtype=np.uint32)
    got = idx.seek_fields(rec, fld)
    for i in list(range(0, 20000, 97)) + list(range(19800, 20000)):
        w = O.seek_field(want_idx, len(raw), rc, 256, False, int(rec[i]), int(fld[i]))
        if w is None:
            assert got[i, 0] == U64MAX and got[i, 1] == U64MAX
        else:
            assert (int(got[i, 0]), int(got[i, 1])) == w
    # vectorised check of everything in range
    live = (rec + 1 < rc) & (fld < 256)
    s = (rec[live].astype(np.int64) + 1) * 256 + fld[live]
    assert (got[live, 0] == want_idx[s] + 1).all() and (got[live, 1] == want_idx[s + 1]).all()
    assert (got[~live] == U64MAX).all()
    gr = idx.seek_records(rec[:500])
    for i in range(0, 500, 7):
        w = O.seek_record(want_idx, len(raw), rc, jump, 256, int(rec[i]))
        assert (int(gr[i, 0]), int(gr[i, 1])) == w
    offs, blob = idx.gather_fields(rec[:300], fld[:300])
    for i in range(300):
        a, b = int(got[i, 0]), int(got[i, 1])
        assert blob[int(offs[i]):int(offs[i + 1])].tobytes() == raw[a:b]
    # past the first sweep of the gather kernel (lookup.cu: SMs x 16 blocks of 32 ranges, ~75 K ranges on a B200),
    # None probes scattered through every sweep: every byte against the oracle's slices
    rec, fld = gen.queries(260_000, rc, 256, seed=47)
    rec[::997] = rc - 1 + np.arange(rec[::997].size, dtype=np.uint32) % 3
    fld[5::1009] = 256 + np.arange(fld[5::1009].size, dtype=np.uint32) % 5
    offs, blob = idx.gather_fields(rec, fld)
    live = (rec + 1 < rc) & (fld < 256)
    s = np.where(live, (rec.astype(np.int64) + 1) * 256 + fld, 0)
    a = np.where(live, want_idx[s] + 1, 0).astype(np.int64)
    lens = np.where(live, want_idx[s + 1].astype(np.int64) - a, 0)
    assert (~live).sum() > 400 and offs[0] == 0 and (np.diff(offs.astype(np.int64)) == lens).all()
    src = np.repeat(a, lens) + np.arange(int(lens.sum())) - np.repeat(offs[:-1].astype(np.int64), lens)
    assert blob.size == src.size and (blob == np.frombuffer(raw, dtype=np.uint8)[src]).all()
    idx.free()


def test_crlf_seeks_vs_oracle(ctx):
    data, rows = gen.quoted(1 << 20, seed=43)
    raw = data.tobytes()
    idx = ctx.index_build(raw)
    host = idx.to_host()
    # quoted fields contain bare LF / CRLF, so rows are NOT fixed width: InvalidCsvFormat is expected
    want = O.closed_form_numpy(raw)
    assert (host == want).all()
    if (host.size - 1) % 17:
        with pytest.raises(cs.InvalidCsvFormat):
            idx.tape_init(16, True)
    idx.free()
    body = b"a,\"x,y\",c\r\n" * 5000
    idx = ctx.index_build(b"h1,h2,h3\r\n" + body)
    rc, jump = idx.tape_init(3, True)
    assert (rc, jump) == (5001, 4)
    host = idx.to_host()
    raw = b"h1,h2,h3\r\n" + body
    for r, f in ((0, 0), (0, 1), (0, 2), (4999, 1), (4999, 2), (5000, 0), (17, 3)):
        w = O.seek_field(host, len(raw), rc, 3, True, r, f)
        assert idx.seek_field(r, f) == w
    assert raw[slice(*idx.seek_field(4999, 1))] == b'"x,y"'
    idx.free()


# ---- full-size properties (BASELINE configs 2 and 3) ------------------------------------------------
@pytest.mark.parametrize("kind", ["cfg2_unquoted", "cfg3_quoted"])
def test_full_size_properties(ctx, kind):
    import torch
    target = 1 << 30
    if kind == "cfg2_unquoted":
        data, rows = gen.unquoted(target, seed=42)
        nf, crlf = 16, False
    else:
        data, rows = gen.quoted(target, seed=43)
        nf, crlf = 16, True
    n = data.size
    dev = torch.device("cuda", ctx.device)
    d = torch.from_numpy(data).to(dev)
    idx = ctx.index_build_device(d.data_ptr(), n)
    E = len(idx)
    # oracle (literal SSE restatement) over the full input: length + checksum (sum of entries mod 2^64)
    cnt, checksum = O.read_sse_timed(O.aligned_copy(data))
    assert E == cnt
    host = idx.to_host()
    assert int(host.sum(dtype=np.uint64)) == checksum
    # element-wise, once per run: the whole 0.5-1.25 GB index against the oracle's index of the same bytes
    want, _ = O.read_closed_form(data, 0, 0, with_sentinel=True)
    assert want.size == E and np.array_equal(host, want)
    del want
    assert host[0] == 0 and (np.diff(host[1:].astype(np.int64)) > 0).all()             # strictly sorted
    assert np.isin(data[host[1:]], np.array([0x2C, 0x0D, 0x0A], dtype=np.uint8)).all()  # entries are separators
    if kind == "cfg2_unquoted":
        rc, jump = idx.tape_init(nf, crlf)
        assert rc == rows + 1 and jump == 16 and E == 1 + 16 * (rows + 1)
        assert host[-1] == n - 1
    # idempotence: a second build of the same bytes gives the same index
    idx2 = ctx.index_build_device(d.data_ptr(), n)
    assert len(idx2) == E and (idx2.to_host() == host).all()
    # sharded at arbitrary offsets == single build (checksum of checksums)
    G = 4
    cuts = [0] + [(k * n) // G + 37 * k + 13 for k in range(1, G)] + [n]
    par, total, csum = 0, 0, 0
    for k in range(G):
        lo, hi = cuts[k], cuts[k + 1]
        lo16 = lo & ~15                      # device pointers handed to the ABI are 16-byte aligned
        sh = d[lo16:hi]
        if lo16 != lo:                       # re-materialise the shard at an aligned address
            sh = d[lo:hi].clone()
            torch.cuda.synchronize()
        p = ctx.shard_quote_parity(sh.data_ptr(), hi - lo)
        si = ctx.index_build_shard_device(sh.data_ptr(), hi - lo, par, lo, emit_sentinel=(k == 0))
        hs = si.to_host()
        total += hs.size
        csum = (csum + int(hs.sum(dtype=np.uint64))) & 0xFFFFFFFFFFFFFFFF
        par ^= p
        si.free()
    assert total == E and csum == checksum
    idx.free()
    idx2.free()


# ---- the two CUDA kernels (one-tile-per-CTA and the persistent TMA pipeline) against each other and the oracle ----
@pytest.fixture(scope="module")
def forced_ctxs():
    out = {}
    for k in ("simple", "tma"):
        os.environ["CSVB200_KERNEL"] = k
        out[k] = cs.Context(0)
    os.environ.pop("CSVB200_KERNEL", None)
    yield out
    for c in out.values():
        c.close()


@pytest.mark.parametrize("name,data", [c for c in cases.edge_cases() if len(c[1]) >= 128],
                         ids=[c[0] for c in cases.edge_cases() if len(c[1]) >= 128])
def test_both_kernels_edge_cases(forced_ctxs, name, data):
    want = O.read_sse(data)
    for k, c in forced_ctxs.items():
        got, par = build(c, data)
        assert got.shape == want.shape and (got == want).all(), k
        assert par == (data.count(b'"') & 1), k


def test_both_kernels_fuzz_multi_tile(forced_ctxs):
    for seed in range(40):
        n = 128 + (seed * 104729) % (40 * cases.TILE)
        data = cases.rand_bytes(n, 1000 + seed) if seed % 5 else cases.full_random(n, seed)
        want = O.read_sse(data)
        for k, c in forced_ctxs.items():
            got, _ = build(c, data)
            assert got.shape == want.shape and (got == want).all(), (k, seed, n)


def test_tma_kernel_dense_rounds_and_shards(forced_ctxs):
    c = forced_ctxs["tma"]
    # one entry per byte: every tile needs 4 staging rounds
    data = b"," * (5 * cases.TILE + 77)
    got, _ = build(c, data)
    assert got.size == len(data) + 1 and (got[1:] == np.arange(len(data), dtype=np.uint64)).all()
    data = (b'",' * (3 * cases.TILE))[: 5 * cases.TILE + 1]
    want = O.read_sse(data)
    got, _ = build(c, data)
    assert (got == want).all()
    # shard chain (carry-in parity, global offsets, odd output bases) through the TMA kernel
    q, _ = gen.quoted(2 << 20, seed=44)
    raw = q.tobytes()
    want = O.closed_form_numpy(raw)
    n = len(raw)
    cuts = [0] + [(k * n) // 3 + 37 * k + 13 for k in range(1, 3)] + [n]
    got, _ = _shard_chain(c, raw, cuts)
    assert (got == want).all()


def test_stream_ordered_shard_api_on_torch_stream(ctx):
    """csvb200_shard_quote_parity_device + csvb200_index_build_shard_device_ex: the carry-in parity is
    derived on the device from the gathered parity array; everything runs on torch's current stream
    (handle 0 = legacy default stream must NOT fall back to the context's private stream)."""
    import torch
    dev = torch.device("cuda", ctx.device)
    q, _ = gen.quoted(6 << 20, seed=44)
    raw = q.tobytes()
    want = O.closed_form_numpy(raw)
    n = len(raw)
    G = 5
    cuts = [0] + [(k * n) // G + 37 * k + 13 for k in range(1, G)] + [n]
    # make at least one cut land inside a quoted field
    inside = raw.index(b'"', cuts[2]) + 1
    cuts[2] = inside
    for stream in (torch.cuda.current_stream(dev), torch.cuda.Stream(dev)):
        with torch.cuda.stream(stream):
            ctx.set_stream(stream.cuda_stream)
            try:
                shards = [torch.from_numpy(np.frombuffer(raw, dtype=np.uint8)[cuts[k]:cuts[k + 1]].copy()).to(dev)
                          for k in range(G)]
                pars = torch.full((G,), 7, dtype=torch.int32, device=dev)   # garbage: pass A must overwrite it
                for k in range(G):
                    ctx.shard_quote_parity_device(shards[k].data_ptr(), shards[k].numel(), pars[k:].data_ptr())
                res = torch.zeros((G, 2), dtype=torch.int64, device=dev)
                torch.cuda.synchronize()
                idxs = [ctx.index_build_shard_device_ex(shards[k].data_ptr(), shards[k].numel(), pars.data_ptr(), k,
                                                        cuts[k], k == 0, res[k].data_ptr()) for k in range(G)]
                got = np.concatenate([i.to_host() for i in idxs])
                assert got.shape == want.shape and (got == want).all()
                ps = pars.cpu().tolist()
                assert ps == [O.shard_summary(raw[cuts[k]:cuts[k + 1]])[0] for k in range(G)] and 1 in ps
                counts = res[:, 0].cpu().tolist()
                assert counts == [len(i) - (1 if k == 0 else 0) for k, i in enumerate(idxs)]
                assert res[-1, 1].item() == (raw.count(b'"') & 1)
                for i in idxs:
                    i.free()
            finally:
                ctx.set_stream(None)


def _speculative_chain(c, raw, cuts, dev, window=0):
    """All shards of `raw` built speculatively on one GPU; res (G x 4) plays the all-gathered array."""
    import torch
    G = len(cuts) - 1
    shards = [torch.from_numpy(np.frombuffer(raw, dtype=np.uint8)[cuts[k]:cuts[k + 1]].copy()).to(dev) for k in range(G)]
    res = torch.full((G, 4), 99, dtype=torch.int64, device=dev)   # garbage: the build must overwrite it
    final = torch.zeros((G, 2), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()   # torch's stream is not ordered against the context's non-blocking stream
    idxs = [c.index_build_shard_speculative(shards[k].data_ptr(), shards[k].numel(), k, cuts[k], k == 0,
                                            res[k].data_ptr(), window) for k in range(G)]
    for i in idxs:
        i.shard_verify(res.data_ptr(), G, final.data_ptr())
    got = np.concatenate([i.to_host() for i in idxs])
    redone = [i.shard_redone() for i in idxs]
    fin = final.cpu().tolist()
    lens = [len(i) for i in idxs]
    for i in idxs:
        i.free()
    return got, redone, fin, lens


def test_speculative_shard_build(forced_ctxs):
    """csvb200_index_build_shard_speculative + csvb200_index_shard_verify: exact for any input; no rebuild
    on RFC-4180-shaped data even when a cut lands inside a quoted field; a misleading quote triggers the
    rebuild of that shard only; true counts of ALL shards are derived without a second exchange."""
    import torch
    for kname in ("tma", "simple"):
        c = forced_ctxs[kname]
        dev = torch.device("cuda", c.device)
        q, _ = gen.quoted(6 << 20, seed=44)
        raw = q.tobytes()
        want = O.closed_form_numpy(raw)
        n = len(raw)
        G = 5
        cuts = [0] + [(k * n) // G + 37 * k + 13 for k in range(1, G)] + [n]
        cuts[2] = raw.index(b'"', cuts[2]) + 1            # inside (or at the edge of) a quoted field
        got, redone, fin, lens = _speculative_chain(c, raw, cuts, dev)
        assert got.shape == want.shape and (got == want).all()
        true_carry = [O.shard_summary(raw[:cuts[k]])[0] for k in range(G)]
        assert [r[1] for r in redone] == true_carry and 1 in true_carry
        assert not any(r[0] for r in redone), "well-formed CSV must not need a rebuild"
        assert [f[1] for f in fin] == true_carry
        assert [f[0] + (k == 0) for k, f in enumerate(fin)] == lens
        # misleading data: an unescaped quote after a letter and before a newline looks like a closing quote
        raw2 = (b'aa,bb"\n,cc,dd\n' * 40000) + b'x,y\n'
        want2 = O.closed_form_numpy(raw2)
        cuts2 = [0, 14 * 10000 + 3, 14 * 20001 + 5, 14 * 30001 + 3, len(raw2)]   # 14-byte rows, one quote each
        got, redone, fin, lens = _speculative_chain(c, raw2, cuts2, dev)
        assert got.shape == want2.shape and (got == want2).all()
        assert any(r[0] for r in redone) and not redone[0][0]
        assert [r[1] for r in redone] == [O.shard_summary(raw2[:k])[0] for k in cuts2[:-1]]
        assert [f[0] + (k == 0) for k, f in enumerate(fin)] == lens
        # SURVEY 8d forced boundaries: inside a quoted field, between the two quotes of "", between CR and LF
        body = b'id,"text, with ""escapes"" and\r\nnewlines",tail\r\n' * 4000
        raw4 = b"h1,h2,h3\r\n" + body
        want4 = O.closed_form_numpy(raw4)
        inside = raw4.index(b"text")
        esc = raw4.index(b'""') + 1
        crlf = raw4.index(b"\r\n", 50) + 1
        for cut in (inside, esc, crlf, inside + 48 * 1000, esc + 48 * 2001, crlf + 48 * 3999):
            got, redone, fin, lens = _speculative_chain(c, raw4, [0, cut, len(raw4)], dev)
            assert got.shape == want4.shape and (got == want4).all(), cut
            assert redone[1][1] == O.shard_summary(raw4[:cut])[0]
        got, redone, fin, lens = _speculative_chain(c, raw4, [0, inside, esc, crlf, len(raw4) // 2 + 5, len(raw4)], dev)
        assert (got == want4).all()
        # no quote at all inside the window / empty shard / tiny shards
        raw3 = b"1,2,3\n" * 30000
        got, redone, fin, lens = _speculative_chain(c, raw3, [0, 7, 7, 100, 100000, len(raw3)], dev, window=4096)
        assert (got == O.closed_form_numpy(raw3)).all() and not any(r[0] for r in redone)


def test_build_to_host_pipeline_multi_chunk(ctx):
    """csvb200_index_build_to_host: chunked H2D / chained launches / overlapped D2H (3 chunks of 64 MiB),
    quote regions and odd output bases crossing the chunk boundaries; pageable and pinned buffers."""
    import torch
    data, _ = gen.quoted(150 << 20, seed=43)
    n = data.size
    want = O.read_sse(data)
    out = np.zeros(want.size + 16, dtype=np.uint64)
    ln = ctx.index_build_to_host(data.ctypes.data, n, out.ctypes.data, out.size)      # pageable in / out
    assert ln == want.size and (out[:ln] == want).all()
    h_in = torch.from_numpy(data).pin_memory()
    h_out = torch.zeros(want.size + 16, dtype=torch.int64).pin_memory()
    ln = ctx.index_build_to_host(h_in.data_ptr(), n, h_out.data_ptr(), h_out.numel())  # pinned in / out
    assert ln == want.size and (h_out.numpy()[:ln].view(np.uint64) == want).all()
    with pytest.raises(BufferError):
        ctx.index_build_to_host(h_in.data_ptr(), n, h_out.data_ptr(), 1000)
    # dense input overflows the reserve heuristic: transparent fallback to the exact-size path
    dense = np.full(130 << 20, 0x2C, dtype=np.uint8)
    out = np.zeros(dense.size + 2, dtype=np.uint64)
    ln = ctx.index_build_to_host(dense.ctypes.data, dense.size, out.ctypes.data, out.size)
    assert ln == dense.size + 1 and out[1] == 0 and out[ln - 1] == dense.size - 1
    assert (np.diff(out[1:ln].astype(np.int64)) == 1).all()


# ---- SURVEY 8f "next" rows: device-side tape validation, chunks with byte ranges, column materialisation ----
def _ragged(kind):
    rows = [b"c0,c1,c2"] + [b"%d,%d,%d" % (i, i * 7, i * 13) for i in range(5000)]
    nl = b"\r\n" if kind == "crlf" else b"\n"
    return rows, nl


@pytest.mark.parametrize("kind", ["lf", "crlf"])
def test_tape_validate_vs_oracle(ctx, kind):
    rows, nl = _ragged(kind)
    crlf = kind == "crlf"
    good = nl.join(rows) + nl
    idx = ctx.index_build(good, cs.BUILD_KEEP_BYTES)
    rep = idx.tape_validate(3, crlf)
    assert rep["ok"] == 1 and rep["first_bad_slot"] == U64MAX and rep["problem"] == 0
    assert rep["record_cnt"] == len(rows) and rep["jump"] == (4 if crlf else 3)
    assert O.tape_first_bad_slot(good, idx.to_host(), 3, crlf) == U64MAX
    idx.free()
    # ragged rows whose separator counts cancel: the reference's (len-1) % jump test passes, the seeks go wrong
    bad_rows = list(rows)
    bad_rows[1234] = b"1,2"            # one field short ...
    bad_rows[4000] = b"1,2,3,4"        # ... one field long
    for data in (nl.join(bad_rows) + nl, nl.join(rows[:777] + [b"x"] + rows[777:]) + nl,
                 nl.join(rows) + nl + b"7,8", good.replace(b"10,70,130" + nl, b"10,70,130" + (b"\n" if crlf else b"\r\n"), 1)):
        idx = ctx.index_build(data, cs.BUILD_KEEP_BYTES)
        host = idx.to_host()
        rep = idx.tape_validate(3, crlf)
        want = O.tape_first_bad_slot(data, host, 3, crlf)
        assert rep["first_bad_slot"] == want
        jump = 4 if crlf else 3
        assert rep["problem"] == (host.size - 1) % jump and rep["record_cnt"] == (host.size - 1) // jump
        if want != U64MAX:
            assert rep["ok"] == 0 and rep["first_bad_record"] == (want - 1) // jump and rep["first_bad_pos"] == host[want]
        else:
            assert rep["ok"] == (1 if rep["problem"] == 0 else 0)
        idx.free()
    # without the bytes the call must refuse, not guess
    idx = ctx.index_build(good)
    with pytest.raises(cs.InvalidState):
        idx.tape_validate(3, crlf)
    idx.free()


def test_tape_validate_large_random(ctx):
    data, rows = gen.unquoted(8 << 20, seed=9)
    raw = bytearray(data.tobytes())
    idx = ctx.index_build(bytes(raw), cs.BUILD_KEEP_BYTES)
    assert idx.tape_validate(16, False)["ok"] == 1
    host = idx.to_host()
    idx.free()
    rng = np.random.default_rng(3)
    for _ in range(4):
        s = int(rng.integers(1, host.size))
        pos = int(host[s])
        old = raw[pos]
        raw[pos] = 0x0A if old == 0x2C else 0x2C       # swap the class of one separator
        idx = ctx.index_build(bytes(raw), cs.BUILD_KEEP_BYTES)
        rep = idx.tape_validate(16, False)
        assert rep["first_bad_slot"] == s == O.tape_first_bad_slot(bytes(raw), idx.to_host(), 16, False)
        idx.free()
        raw[pos] = old


def test_tape_chunks_vs_oracle(ctx):
    for name, fc, crlf in (("sample.csv", 3, False), ("sample_rx.csv", 8, True)):
        raw = golden_bytes(name)
        idx = ctx.index_build(raw)
        with pytest.raises(cs.InvalidState):
            idx.tape_chunks(3)                       # before tape_init
        rc, jump = idx.tape_init(fc, crlf)
        host = idx.to_host()
        for num in (1, 2, 3, 5, 12, 200):
            got = idx.tape_chunks(num)
            want = O.chunks(rc, jump, num)
            assert [(c["id"], c["start"], c["end"], c["record_cnt"]) for c in got] == \
                   [(c["id"], c["start"], c["end"], c["record_cnt"]) for c in want]
            for c in got:
                assert c["byte_start"] == int(host[c["start"]]) + 1 and c["byte_end"] == int(host[c["end"]]) + 1
                if c["record_cnt"]:
                    seg = raw[c["byte_start"]:c["byte_end"]]
                    assert seg.endswith(b"\n") and seg.count(b"\n") >= c["record_cnt"]
            assert got[-1]["byte_end"] == len(raw)
        with pytest.raises(cs.InvalidState):
            idx.tape_chunks(0)
        idx.free()


@pytest.mark.parametrize("flags", [0, 1, 2, 3])
def test_materialize_columns_vs_oracle(ctx, flags):
    """csvb200_materialize_columns: several columns of the same records in one sweep per pass; every column equals what
    the oracle's scalar definition and the single-column call give.  Cases: every escape shape of _column_cases, alone
    and behind a 40 KB quoted field, one column, a column listed more than once, an out-of-range field, empty ranges, a
    range that runs past the last record, 17 columns = more columns than warps, clipping by out_cap in the device form,
    CRLF rows and a wide quoted file."""
    import torch
    dev = torch.device("cuda", ctx.device)
    big = b'"' + b'ab""cd, \n' * 4000 + b'"'
    head, rest = _column_cases().split(b"\n", 1)
    for raw in (_column_cases(), head + b"\n" + b"77, " + big + b" ,tail\n" + b"78,x,y\n" * 40 + rest):
        idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
        rc, jump = idx.tape_init(3, False)
        host = idx.to_host()
        for fields, first, nrec in (([0, 1, 2], 0, rc - 1), ([2, 0], 17, 1000), ([1], 3, 700), ([1, 1, 1, 1], 0, 60),
                                    ([1, 7, 2, 2], rc - 5, 20), ([0, 1], 5, 0), ([2, 1, 0] * 5 + [1, 2], 1024, 1100)):
            got = idx.materialize_columns(fields, first, nrec, flags)
            for f, (offs, out) in zip(fields, got):
                w_offs, w_out = O.materialize_column(raw, host, rc, 3, False, f, first, nrec, flags)
                assert (offs == w_offs).all(), (fields, f, first, nrec)
                assert out.tobytes() == w_out, (fields, f, first, nrec)
        # device form, destination too small for the last values: whole values are clipped, nothing past out_cap is written
        fields, nrec = [1, 2], rc - 1
        want = [O.materialize_column(raw, host, rc, 3, False, f, 0, nrec, flags) for f in fields]
        caps = [len(w[1]) // 2 + 3 for w in want]
        d_off = [torch.zeros(nrec + 1, dtype=torch.int64, device=dev) for _ in fields]
        d_out = [torch.full((len(w[1]) + 64,), 0xEE, dtype=torch.uint8, device=dev) for w in want]
        torch.cuda.synchronize()
        idx.materialize_columns_device(fields, 0, nrec, flags, [t.data_ptr() for t in d_off], [t.data_ptr() for t in d_out], caps)
        idx.sync()
        torch.cuda.synchronize()
        for (w_offs, w_out), cap, o, v in zip(want, caps, d_off, d_out):
            assert (o.cpu().numpy().view(np.uint64) == w_offs).all()
            keep = int(w_offs[w_offs <= cap].max())
            got = v.cpu().numpy()
            assert got[:keep].tobytes() == w_out[:keep]
            assert (got[keep:] == 0xEE).all()
        idx.free()
    # CRLF rows (row_size = field_cnt + 1) and a wide quoted file against the single-column kernels
    raw = golden_bytes("sample_rx.csv")
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, jump = idx.tape_init(8, True)
    host = idx.to_host()
    got = idx.materialize_columns([7, 0, 3, 2], 0, rc - 1, flags)
    for f, (offs, out) in zip([7, 0, 3, 2], got):
        w_offs, w_out = O.materialize_column(raw, host, rc, 8, True, f, 0, rc - 1, flags)
        assert (offs == w_offs).all() and out.tobytes() == w_out
    idx.free()
    q, _ = gen.quoted(3 << 20, seed=43)
    idx = ctx.index_build(q, cs.BUILD_KEEP_BYTES)
    rc, _ = idx.tape_init(16, True)
    got = idx.materialize_columns(list(range(16)), 0, rc - 1, flags)
    for f in (0, 1, 7, 15):
        offs, out = idx.materialize_column(f, 0, rc - 1, flags)
        assert (got[f][0] == offs).all() and got[f][1].tobytes() == out.tobytes()
    idx.free()


def test_materialize_device_forms_reject_null_destinations(ctx):
    """Both device forms check every column's destinations before they launch anything: a null offsets array, or a
    capacity above 0 with no value buffer, is CSVB200_ERR_INVALID_ARG (ValueError).  The index stays usable."""
    import torch
    raw = _column_cases()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, _ = idx.tape_init(3, False)
    host = idx.to_host()
    fields, nrec, flags = [1, 2], rc - 1, cs.FIELD_UNQUOTE | cs.FIELD_TRIM
    want = [O.materialize_column(raw, host, rc, 3, False, f, 0, nrec, flags) for f in fields]
    dev = torch.device("cuda", ctx.device)
    d_off = [torch.zeros(nrec + 1, dtype=torch.int64, device=dev) for _ in fields]
    d_out = [torch.zeros(len(w[1]), dtype=torch.uint8, device=dev) for w in want]
    p_off, p_out, caps = [t.data_ptr() for t in d_off], [t.data_ptr() for t in d_out], [len(w[1]) for w in want]
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        idx.materialize_columns_device(fields, 0, nrec, flags, [p_off[0], 0])
    with pytest.raises(ValueError):
        idx.materialize_columns_device(fields, 0, nrec, flags, p_off, [p_out[0], 0], caps)
    with pytest.raises(ValueError):
        idx.materialize_columns_device(fields, 0, nrec, flags, p_off, None, caps)
    with pytest.raises(ValueError):
        idx.materialize_column_device(fields[0], 0, nrec, flags, 0, p_out[0], caps[0])
    with pytest.raises(ValueError):
        idx.materialize_column_device(fields[0], 0, nrec, flags, p_off[0], 0, caps[0])
    idx.materialize_columns_device(fields, 0, nrec, flags, p_off, p_out, caps)
    torch.cuda.synchronize()
    for (w_offs, w_out), o, v in zip(want, d_off, d_out):
        assert (o.cpu().numpy().view(np.uint64) == w_offs).all()
        assert v.cpu().numpy().tobytes() == w_out
    idx.free()


def test_build_to_host_small_inputs_zero_copy(ctx):
    """csvb200_index_build_to_host at <= 256 KiB: the kernel reads and writes pinned host memory directly (one launch, one
    synchronisation).  Every edge case of tests/cases.py plus sizes around the 32 KiB tile and the 256 KiB limit, into
    pageable and pinned destinations, a destination that is too small, and a dense input (one entry per byte)."""
    import torch
    rng = np.random.default_rng(11)
    inputs = [raw for _, raw in cases.edge_cases() + cases.small_cases() if 0 < len(raw) <= (256 << 10)]
    q, _ = gen.quoted(300 << 10, seed=52)
    for size in (1, 63, 64, 65, 32767, 32768, 32769, 65536 + 5, (256 << 10) - 1, 256 << 10):
        inputs.append(q[:size].tobytes())
    inputs.append(b"," * 70000)                                   # one entry per byte
    inputs.append(bytes(rng.choice(np.frombuffer(b'a,"\n\r ', dtype=np.uint8), size=100000)))
    h_out = torch.zeros((256 << 10) + 64, dtype=torch.int64).pin_memory()
    for raw in inputs:
        a = np.frombuffer(raw, dtype=np.uint8)
        want = O.read_sse(a) if a.size >= 64 else O.read_closed_form(a, 0, 0, with_sentinel=True)[0]
        out = np.zeros(want.size + 8, dtype=np.uint64)
        ln = ctx.index_build_to_host(a.ctypes.data, a.size, out.ctypes.data, out.size)              # pageable destination
        assert ln == want.size and (out[:ln] == want).all(), len(raw)
        h_out.zero_()
        ln = ctx.index_build_to_host(a.ctypes.data, a.size, h_out.data_ptr(), h_out.numel())        # pinned: written in place
        assert ln == want.size and (h_out.numpy()[:ln].view(np.uint64) == want).all(), len(raw)
        assert (h_out.numpy()[ln:ln + 8] == 0).all()
        if want.size > 3:
            h_out.zero_()
            with pytest.raises(BufferError):                      # CSVB200_ERR_CAPACITY
                ctx.index_build_to_host(a.ctypes.data, a.size, h_out.data_ptr(), want.size - 2)
            assert (h_out.numpy()[want.size - 2:want.size + 8] == 0).all()   # nothing past the capacity is written


def test_host_register_pins_caller_memory(ctx):
    """csvb200_host_register: an ordinary array becomes DMA-able in place (the end-to-end call takes its pinned branch),
    the result equals the oracle's, a second registration of the same range is refused, unregister restores it."""
    q, _ = gen.quoted(96 << 20, seed=51)
    want = O.read_sse(q)
    out = np.zeros(want.size + 64, dtype=np.uint64)
    lib = cs._lib.load()
    with cs.host_registered(out), cs.host_registered(q, read_only=False):
        assert lib.csvb200_host_register(out.ctypes.data, out.nbytes, 0) == 1      # CSVB200_ERR_INVALID_ARG
        ln = ctx.index_build_to_host(q.ctypes.data, q.size, out.ctypes.data, out.size)
        assert ln == want.size and (out[:ln] == want).all()
    assert lib.csvb200_host_unregister(out.ctypes.data) == 1                        # no longer registered
    out[:] = 0
    ln = ctx.index_build_to_host(q.ctypes.data, q.size, out.ctypes.data, out.size)   # pageable again: staged copies
    assert ln == want.size and (out[:ln] == want).all()


def _column_cases():
    rows = [b'id,name,note']
    vals = [b'plain', b'"quoted"', b'  padded\t', b'"with ""escapes"" inside"', b'""', b'"', b'', b' "q, and\nnewline" ',
            b'"a""', b'""""', b'x"y', b'"tail""', b'\t\t', b'" "']
    for i in range(3000):
        rows.append(b"%d,%s,%s" % (i, vals[i % len(vals)], vals[(i * 5 + 3) % len(vals)]))
    return b"\n".join(rows) + b"\n"


@pytest.mark.parametrize("flags", [0, 1, 2, 3])
def test_materialize_column_vs_oracle(ctx, flags):
    raw = _column_cases()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, jump = idx.tape_init(3, False)
    host = idx.to_host()
    for fld, first, nrec in ((1, 0, rc - 1), (2, 0, rc - 1), (0, 17, 1000), (1, rc - 5, 20), (2, 5, 0), (7, 0, 10), (1, 1024, 1024)):
        offs, out = idx.materialize_column(fld, first, nrec, flags)
        w_offs, w_out = O.materialize_column(raw, host, rc, 3, False, fld, first, nrec, flags)
        assert (offs == w_offs).all(), (fld, first, nrec)
        assert out.tobytes() == w_out, (fld, first, nrec)
    idx.free()


def test_materialize_column_crlf_and_device_form(ctx):
    import torch
    raw = golden_bytes("sample_rx.csv")
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, jump = idx.tape_init(8, True)
    host = idx.to_host()
    dev = torch.device("cuda", ctx.device)
    for fld in range(8):
        offs, out = idx.materialize_column(fld, 0, rc - 1, cs.FIELD_UNQUOTE | cs.FIELD_TRIM)
        w_offs, w_out = O.materialize_column(raw, host, rc, 8, True, fld, 0, rc - 1, 3)
        assert (offs == w_offs).all() and out.tobytes() == w_out
        d_off = torch.zeros(rc, dtype=torch.int64, device=dev)
        d_out = torch.zeros(max(len(w_out), 1), dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        idx.materialize_column_device(fld, 0, rc - 1, 3, d_off.data_ptr(), d_out.data_ptr(), len(w_out))
        torch.cuda.synchronize()
        assert (d_off.cpu().numpy().view(np.uint64) == w_offs).all()
        assert d_out.cpu().numpy()[:len(w_out)].tobytes() == w_out
    assert idx.materialize_column(2, 1, 1, 3)[1].tobytes() == b"INTERNAL MED, CARD. ELECTROPHYSIOLOGY"
    idx.free()


# ---- streaming ingest (SURVEY 8f rank 3) ---------------------------------------------------------
def test_stream_build_vs_oracle(ctx):
    """csvb200_index_build_stream: many small chunks (quote regions, CRLF pairs and "" escapes cut by the
    chunk boundaries), short reads from the reader, segments delivered in order."""
    q, _ = gen.quoted(3 << 20, seed=47)
    raw = q.tobytes()
    want = O.read_sse(raw)
    for chunk, read_max in ((64 << 10, 1 << 30), (64 << 10, 5000), (1 << 20, 777777), (0, 1 << 30)):
        pos = [0]
        parts, firsts = [], []

        def read(cap):
            k = min(cap, read_max, len(raw) - pos[0])
            b = raw[pos[0]:pos[0] + k]
            pos[0] += k
            return b

        def sink(entries, first):
            parts.append(entries.copy())
            firsts.append(first)

        st = ctx.index_build_stream(read, sink, chunk)
        got = np.concatenate(parts)
        assert got.shape == want.shape and (got == want).all(), (chunk, read_max)
        assert firsts == list(np.cumsum([0] + [p.size for p in parts[:-1]]))
        assert st["bytes"] == len(raw) and st["entries"] == want.size and st["end_parity"] == (raw.count(b'"') & 1)
        assert st["chunks"] == -(-len(raw) // (chunk or (16 << 20)))
    # empty input: the sentinel alone
    parts = []
    st = ctx.index_build_stream(lambda cap: b"", lambda e, f: parts.append(e.copy()), 0)
    assert st["entries"] == 1 and len(parts) == 1 and parts[0].tolist() == [0]
    # a failing sink aborts with Io
    with pytest.raises(ZeroDivisionError):
        pos = [0]
        ctx.index_build_stream(lambda cap: raw[:1000] if not pos[0] and not pos.__setitem__(0, 1) else b"", lambda e, f: 1 / 0, 0)
    # dense chunk: more entries than a pinned output slot holds (drained in pieces)
    dense = b"," * (300 << 10)
    parts = []
    pos = [0]

    def read2(cap):
        k = min(cap, len(dense) - pos[0])
        pos[0] += k
        return dense[:k]

    ctx.index_build_stream(read2, lambda e, f: parts.append(e.copy()), 128 << 10)
    got = np.concatenate(parts)
    assert got.size == len(dense) + 1 and (got[1:] == np.arange(len(dense), dtype=np.uint64)).all()


def test_index_build_file_vs_oracle(ctx):
    import torch
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "big.csv")
        q, _ = gen.quoted(40 << 20, seed=48)     # 3 chunks of 16 MiB
        q.tofile(path)
        want = O.read_sse(q)
        got, st = ctx.index_build_file(path)      # pageable destination: copied out of the pinned ring
        assert got.shape == want.shape and (got == want).all()
        assert st["bytes"] == q.size and st["chunks"] == 3
        h = torch.zeros(want.size + 8, dtype=torch.int64).pin_memory()   # pinned destination: DMA in place
        ln, st = ctx.index_build_file_ptr(path, h.data_ptr(), h.numel())
        assert ln == want.size and (h.numpy()[:ln].view(np.uint64) == want).all()
        with pytest.raises(BufferError):
            ctx.index_build_file_ptr(path, h.data_ptr(), 100)
        small = np.empty(10, dtype=np.uint64)
        got, _ = ctx.index_build_file(path, small)           # too small: retried with the reported size
        assert (got == want).all()
        for name in ("sample.csv", "sample_rx.csv", "reader_test01.csv"):
            p2 = os.path.join(d, name)
            open(p2, "wb").write(golden_bytes(name))
            got, _ = ctx.index_build_file(p2)
            assert (got == O.read_sse(golden_bytes(name))).all()
        open(os.path.join(d, "empty.csv"), "wb").close()
        got, _ = ctx.index_build_file(os.path.join(d, "empty.csv"))
        assert got.tolist() == [0]
    with pytest.raises(cs.Io):
        ctx.index_build_file("/nonexistent/definitely_missing.csv")


# ---- SURVEY 8f rank 4: input validation and the on-disk index ---------------------------------------
def test_validate_utf8_vs_python_decoder(ctx):
    good = "id,name\n1,héllo\n2,wörld – ✓\n3,🙂🙂\n".encode() * 3000
    assert ctx.validate_utf8(good) == (None, False)
    assert ctx.validate_utf8(b"a,b\n1,2\n" * 50000) == (None, True)
    assert ctx.validate_utf8(b"") == (None, True)
    crafted = [b"ab\xe2\x82", b"ab\xc0\xaf", b"\xed\xa0\x80", b"a\x80", b"\xf4\x90\x80\x80", b"\xf0\x8f\xbf\xbf",
               b"\xe0\x9f\xbf", b"\xc2", b"x\xf0\x9f\x99", b"\xf5\x80\x80\x80", b"\xff", b"\xc2\x80\x80",
               b"\xe1\x80\xc2\x80", b"ok\xe2\x82\xac\xe2\x82\xac\x80", b"\xf0\x9f\x99\x82" * 5 + b"\xbf"]
    for c in crafted:
        for pad in (0, 1, 13, 14, 15, 16, 17, 31, 4093):     # every position relative to the 16-byte chunks
            for tail in (b"", b"tail,more\n"):
                data = b"x" * pad + c + tail
                want = O.utf8_valid_up_to(data)
                got, asc = ctx.validate_utf8(data)
                assert got == want, (c, pad, tail, got, want)
                assert asc == O.is_ascii(data) == False  # noqa: E712
    rng = np.random.default_rng(5)
    alphabet = np.array([0x41, 0x2C, 0x0A, 0x80, 0xBF, 0xC2, 0xC1, 0xE0, 0xA0, 0x9F, 0xED, 0xEF, 0xF0, 0x90, 0x8F, 0xF4,
                         0xF5, 0xE2, 0x82, 0xAC], dtype=np.uint8)
    for seed in range(60):
        n = int(rng.integers(1, 3000))
        # mostly ASCII with bursts of bytes from the tricky alphabet
        data = np.full(n, 0x61, dtype=np.uint8)
        k = int(rng.integers(0, 12))
        pos = rng.integers(0, n, size=k)
        for p_ in pos:
            seg = alphabet[rng.integers(0, alphabet.size, size=int(rng.integers(1, 6)))]
            data[p_:p_ + seg.size] = seg[:max(0, min(seg.size, n - p_))]
        raw = data.tobytes()
        got, asc = ctx.validate_utf8(raw)
        assert got == O.utf8_valid_up_to(raw), (seed, raw)
        assert asc == O.is_ascii(raw)
    # valid multi-byte text stays valid wherever the chunk boundaries fall
    txt = "αβγ,δεζ\nκόσμε,🙂\n".encode()
    for pad in range(0, 40):
        assert ctx.validate_utf8(b"y" * pad + txt * 100)[0] is None
    # past the first sweep of the grid-stride kernel (validate.cu: SMs x 8 blocks of 256 threads, each judging groups
    # g and g + half of every sweep of 2 x half 32-byte groups; ~19 MB per sweep on a B200)
    import torch
    half = torch.cuda.get_device_properties(ctx.device).multi_processor_count * 8 * 256
    sweep = 64 * half
    n = max(64 << 20, 3 * sweep + sweep // 2)
    base = np.resize(np.frombuffer(b"id,x\n1,ab\n", dtype=np.uint8), n)
    smile = np.frombuffer("🙂".encode(), dtype=np.uint8)
    e_acute = np.frombuffer("é".encode(), dtype=np.uint8)
    t = 1000                                                      # one thread of the first block
    inputs = []
    v = base.copy()                                               # errors in the second and third sweeps only
    v[100:102] = e_acute
    v[sweep + 4321] = 0x80
    v[2 * sweep + 77] = 0xC0
    inputs.append(v)
    v = base.copy()                                               # two errors one thread meets in iterations 1 and 2
    v[32 * (t + 3 * half) + 5] = 0xFF
    v[32 * (t + 4 * half) + 9] = 0x80
    inputs.append(v)
    v = base.copy()                                               # the reverse: only the later iteration's error
    v[32 * (t + 4 * half) + 9] = 0x80
    inputs.append(v)
    v = base.copy()                                               # valid 4-byte sequences across sweep / group edges
    for at in (half * 32 - 1, sweep - 2, 2 * sweep - 3, 3 * sweep - 1):
        v[at:at + 4] = smile
    inputs.append(v)
    for v in inputs:
        got, asc = ctx.validate_utf8(v)
        assert got == O.utf8_valid_up_to(v.tobytes()) and asc == O.is_ascii(v)
    assert got is None and asc is False


def test_index_save_load_roundtrip(ctx):
    raw = golden_bytes("sample_rx.csv")
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, jump = idx.tape_init(8, True)
    want = idx.to_host().copy()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "rx.idx")
        idx.save(path)
        assert os.path.getsize(path) == 64 + 8 * want.size
        blob = open(path, "rb").read()
        assert blob[:8] == b"CSVB2IDX" and np.frombuffer(blob[64:], dtype="<u8").tolist() == want.tolist()
        got = ctx.index_load(path)
        assert (got.to_host() == want).all() and got.end_parity == idx.end_parity
        assert got.seek_field(1, 2) == idx.seek_field(1, 2) and got.seek_record(6) == idx.seek_record(6)
        assert got.seek_field(6, 8) is None
        with pytest.raises(cs.InvalidState):
            got.tape_validate(8, True)           # needs the input bytes, which a loaded index does not have
        got.free()
        # an index saved before tape_init loads without Tape metadata
        idx2 = ctx.index_build(raw)
        idx2.save(path)
        got = ctx.index_load(path)
        with pytest.raises(cs.InvalidState):
            got.seek_record(0)
        got.free()
        idx2.free()
        # corruption is detected
        bad = bytearray(blob)
        bad[70] ^= 1
        open(path, "wb").write(bytes(bad))
        with pytest.raises(cs.InvalidCsvFormat):
            ctx.index_load(path)
        open(path, "wb").write(blob[:-8])
        with pytest.raises(cs.InvalidCsvFormat):
            ctx.index_load(path)
        open(path, "wb").write(b"NOTANIDX" + blob[8:])
        with pytest.raises(cs.InvalidCsvFormat):
            ctx.index_load(path)
        with pytest.raises(cs.Io):
            ctx.index_load(os.path.join(d, "missing.idx"))
    idx.free()


def test_shard_build_to_host_pipeline(ctx):
    """csvb200_shard_build_to_host + csvb200_shard_job_verify: all ranks of a sharded file emulated on one GPU,
    multi-chunk shards (64 MiB chunks), a cut inside a quoted field, a mispredicted shard that is redone."""
    import torch
    dev = torch.device("cuda", ctx.device)
    q, _ = gen.quoted(200 << 20, seed=49)
    raw = q
    want = O.read_sse(raw)
    n = raw.size
    blob = raw.tobytes()
    cut1 = blob.index(b'"', n // 3) + 1                       # inside / at the edge of a quoted field
    cuts = [0, cut1, (2 * n) // 3 + 7, n]
    G = 3
    res = torch.zeros((G, 4), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    outs, jobs, lens = [], [], []
    for k in range(G):
        shard = torch.from_numpy(raw[cuts[k]:cuts[k + 1]].copy()).pin_memory()
        out = torch.zeros(shard.numel() // 3 + 8192, dtype=torch.int64).pin_memory()
        ln, job = ctx.shard_build_to_host(shard.data_ptr(), shard.numel(), k, cuts[k], k == 0, out.data_ptr(), out.numel(),
                                          res[k].data_ptr())
        outs.append((shard, out))
        jobs.append(job)
        lens.append(ln)
    final = torch.zeros((G, 2), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    got, redone = [], []
    for k in range(G):
        ln, rd = ctx.shard_job_verify(jobs[k], res.data_ptr(), G, final.data_ptr())
        got.append(outs[k][1].numpy()[:ln].view(np.uint64).copy())
        redone.append(rd)
    full = np.concatenate(got)
    assert full.shape == want.shape and (full == want).all()
    assert not any(redone)
    fin = final.cpu().tolist()
    assert [f[0] + (k == 0) for k, f in enumerate(fin)] == [g.size for g in got]
    # misleading data: the guess of shard 1 is wrong, the job re-indexes it from the device copy
    raw2 = np.frombuffer((b'aa,bb"\n,cc,dd\n' * (6 << 20)) + b'x,y\n', dtype=np.uint8)
    want2 = O.closed_form_numpy(raw2)
    cuts2 = [0, 14 * (3 << 20) + 3, raw2.size]
    res = torch.zeros((2, 4), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    outs, jobs = [], []
    for k in range(2):
        shard = torch.from_numpy(raw2[cuts2[k]:cuts2[k + 1]].copy()).pin_memory()
        out = torch.zeros(shard.numel() // 3 + 8192, dtype=torch.int64).pin_memory()
        ln, job = ctx.shard_build_to_host(shard.data_ptr(), shard.numel(), k, cuts2[k], k == 0, out.data_ptr(), out.numel(),
                                          res[k].data_ptr())
        outs.append((shard, out))
        jobs.append(job)
    got, redone = [], []
    for k in range(2):
        ln, rd = ctx.shard_job_verify(jobs[k], res.data_ptr(), 2, 0)
        got.append(outs[k][1].numpy()[:ln].view(np.uint64).copy())
        redone.append(rd)
    full = np.concatenate(got)
    assert redone == [False, True]
    assert full.shape == want2.shape and (full == want2).all()


def test_beyond_4gib_positions(ctx):
    """Maximum-size edge: an input just past 2^32 bytes in ONE launch (positions need more than 32 bits, the
    reference's u32 arithmetic in seek_* would wrap: SURVEY 8c quirk vi).  Count, wrapping sum and the entries
    around the 2^32 boundary against the oracle; K5 over the whole tape."""
    import torch
    target = (1 << 32) + (64 << 20)
    data, rows = gen.unquoted(target, seed=51, nfields=256, modulus=10 ** 15)   # wide rows keep E < 2^32
    n = data.size
    dev = torch.device("cuda", ctx.device)
    d = torch.empty(n + 64, dtype=torch.uint8, device=dev)
    d[:n].copy_(torch.from_numpy(data))
    idx = ctx.index_build_device(d.data_ptr(), n)
    E = len(idx)
    cnt, checksum = O.read_sse_timed(O.aligned_copy(data))
    assert E == cnt == 1 + 256 * (rows + 1)
    host = idx.to_host()
    assert int(host.sum(dtype=np.uint64)) == checksum
    assert int(host[-1]) == n - 1 and int(host[-1]) > (1 << 32)
    assert (np.diff(host[1:].view(np.int64)) > 0).all()
    k = int(np.searchsorted(host, np.uint64(1 << 32)))
    lo = max(k - 2000, 1)
    win = data[int(host[lo]):int(host[k + 2000]) + 1]
    want = O.closed_form_numpy(win, 0, int(host[lo]), with_sentinel=False)
    assert (host[lo:k + 2001] == want).all()
    assert idx.tape_validate(256, False)["ok"] == 1
    # BASELINE config 5 at full size on the same file: 10 M random (record, field) lookups + a 1 % tail of
    # out-of-range probes, hit count and checksum of every (start, end) pair against the oracle's seek_field
    rc, jump = idx.tape_init(256, False)
    assert rc == rows + 1 and jump == 256
    nq = 10_000_000
    rec, fld = gen.queries(nq, rc, 256, seed=46)
    tail = nq // 100
    rec[-tail:-tail // 2] = rc - 1 + np.arange(tail - tail // 2, dtype=np.uint32)   # rec >= record_cnt - 1 -> None
    fld[-tail // 2:] = 256 + np.arange(tail // 2, dtype=np.uint32) % 7               # fld >= field_cnt   -> None
    d_rec = torch.from_numpy(rec.view(np.int32)).to(dev)
    d_fld = torch.from_numpy(fld.view(np.int32)).to(dev)
    d_out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    idx.seek_fields_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, d_out.data_ptr())
    torch.cuda.synchronize()
    got = d_out.cpu().numpy().view(np.uint64)
    cs_cpu, hits = O.seek_fields_timed(host, n, rc, 256, False, rec, fld)
    live = got[:, 0] != np.uint64(U64MAX)
    cs_gpu = int((got[live, 0] ^ (got[live, 1] << np.uint64(1))).sum(dtype=np.uint64))
    assert hits == int(live.sum()) == nq - tail and cs_cpu == cs_gpu
    assert not live[-tail:].any()
    for i in range(0, nq - tail, nq // 64):   # and the bytes the ranges delimit
        a, b = int(got[i, 0]), int(got[i, 1])
        assert bytes(data[a:b]).isdigit() and data[a - 1] in (0x2C, 0x0A) and data[b] in (0x2C, 0x0A)
    idx.free()


def test_index_wrap_device(ctx):
    """csvb200_index_wrap_device: caller-owned device entries behave like a built index (Tape, seeks, K5, K6)."""
    import torch
    raw = golden_bytes("sample_rx.csv")
    dev = torch.device("cuda", ctx.device)
    built = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    host = built.to_host()
    entries = torch.from_numpy(host.view(np.int64).copy()).to(dev)
    d_bytes = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).to(dev)
    w = ctx.index_wrap_device(entries.data_ptr(), entries.numel(), len(raw), d_bytes.data_ptr())
    assert len(w) == host.size and (w.to_host() == host).all()
    assert w.tape_init(8, True) == built.tape_init(8, True)
    for r, f in ((1, 2), (6, 3), (6, 8), (10, 1), (0, 0)):
        assert w.seek_field(r, f) == built.seek_field(r, f)
    assert w.seek_record(6) == built.seek_record(6)
    assert w.tape_validate(8, True) == built.tape_validate(8, True)
    a, b = w.materialize_column(2, 0, 7, 3), built.materialize_column(2, 0, 7, 3)
    assert (a[0] == b[0]).all() and a[1].tobytes() == b[1].tobytes()
    w.free()                                   # must not free the caller's tensor
    assert (entries.cpu().numpy().view(np.uint64) == host).all()
    w2 = ctx.index_wrap_device(entries.data_ptr(), entries.numel(), len(raw))     # without the bytes
    w2.tape_init(8, True)
    with pytest.raises(cs.InvalidState):
        w2.tape_validate(8, True)
    w2.free()
    built.free()


def test_more_than_2_pow_32_entries(ctx):
    """Maximum-size edge (SURVEY 8c quirk ii): the reference's `array_idx: u32` wraps once the index holds 2^32
    entries; here the count travels as 61 bits through the look-back chain.  4.3 G separators in one launch: the
    entry count and sampled entries on both sides of slot 2^32 are checked on the device (index = 34 GB)."""
    import torch
    dev = torch.device("cuda", ctx.device)
    free, _ = torch.cuda.mem_get_info(dev)
    n = (1 << 32) + (3 << 20) + 77
    if free < 9 * n + (8 << 30):
        pytest.skip("needs ~45 GB of free device memory")
    d = torch.full((n + 64,), 0x2C, dtype=torch.uint8, device=dev)
    d[n - 1] = 0x0A
    torch.cuda.synchronize()
    ctx.set_reserve(1, 1)                      # one entry per byte is the worst case: no overflow rebuild
    try:
        idx = ctx.index_build_device(d.data_ptr(), n)
        E = len(idx)
        assert E == n + 1 and E > (1 << 32)
        class _Raw:
            __cuda_array_interface__ = {"shape": (E,), "typestr": "<i8", "data": (idx.device_ptr, False), "version": 2}
        entries = torch.as_tensor(_Raw(), device=dev)
        probe = torch.cat([torch.arange(0, 4096, device=dev), torch.arange((1 << 32) - 4096, (1 << 32) + 4096, device=dev),
                           torch.arange(E - 4096, E, device=dev),
                           torch.randint(1, E, (1 << 20,), device=dev, generator=torch.Generator(device=dev).manual_seed(1))])
        got = entries[probe]
        want = torch.clamp(probe - 1, min=0)     # entry k (k >= 1) is byte k - 1; the sentinel is 0
        assert bool((got == want).all())
        # sortedness of the whole index without bringing it to the host: every difference is exactly 1 after the sentinel
        step = 1 << 28
        for lo in range(1, E - 1, step):
            hi = min(lo + step, E - 1)
            assert bool((entries[lo + 1:hi + 1] - entries[lo:hi] == 1).all())
        idx.free()
    finally:
        ctx.set_reserve(1, 3)
        del d
        torch.cuda.empty_cache()


# ---- round 2: ownership of the result cells, shard-local gathers, a second device ------------------------------
def test_result_cells_are_owned_until_free(ctx):
    """More unsynced index objects than the context has result cells (4095): the build that cannot get a cell fails
    loudly instead of aliasing a live one, every index still reports ITS length, and freeing makes room again."""
    raw = [(b"a,b\n" + b"1,2\n" * (k % 7 + 1)) for k in range(16)]
    raw = [r + b"x" * (64 - len(r) % 64) for r in raw]     # >= 64 bytes each
    want = [O.closed_form_numpy(r).size for r in raw]
    live = []
    with pytest.raises(MemoryError) as ei:
        for k in range(5000):
            live.append((k % 16, ctx.index_build(raw[k % 16])))
    assert "result cell" in str(ei.value) or "live index" in str(ei.value)
    assert len(live) >= 4000
    for j, idx in live[::97]:
        assert len(idx) == want[j]
    for _, idx in live:
        idx.free()
    again = ctx.index_build(raw[3])
    assert len(again) == want[3]
    again.free()


def test_gather_fields_on_a_shard_with_global_offset(ctx):
    """ADVICE r1: gather_fields must rebase the global (start, end) ranges by the shard's offset.  A shard that starts
    at a row boundary is a CSV in its own right: its fields come back as bytes, identical to the oracle's slices."""
    import torch
    data, rows = gen.unquoted(1 << 20, seed=7)
    raw = data.tobytes()
    full = O.closed_form_numpy(raw)
    cut = int(full[16 * 1000]) + 1              # first byte of row 1000 (16 separators per row)
    assert cut % 16 != 0 or True
    shard = np.frombuffer(raw[cut:], dtype=np.uint8)
    dev = torch.device("cuda", ctx.device)
    d = torch.zeros(shard.size + 64 + 16, dtype=torch.uint8, device=dev)
    off = (-d.data_ptr()) % 16
    d[off:off + shard.size].copy_(torch.from_numpy(shard.copy()))
    torch.cuda.synchronize()
    # emit_sentinel so that the shard's own index starts with a sentinel entry; positions are GLOBAL (>= cut)
    idx = ctx.index_build_shard_device(d.data_ptr() + off, shard.size, 0, cut, True)
    host = idx.to_host()
    assert host[0] == 0 and int(host[1]) > cut
    rc, _ = idx.tape_init(16, False)
    rec = np.array([0, 5, 17, rc - 2], dtype=np.uint32)
    fld = np.array([1, 0, 15, 7], dtype=np.uint32)
    offs, vals = idx.gather_fields(rec, fld)
    rg = idx.seek_fields(rec, fld)
    for i in range(rec.size):
        a, b = int(rg[i, 0]), int(rg[i, 1])
        assert a >= cut and bytes(vals[int(offs[i]):int(offs[i + 1])]) == raw[a:b] and raw[a:b].isdigit()
    # an index object that holds FEWER bytes than its positions refer to must refuse, never read out of bounds
    wrapped = ctx.index_wrap_device(idx.device_ptr, len(idx), 100, d.data_ptr() + off)
    wrapped.tape_init(16, False)
    with pytest.raises(cs.errors.ReferencePanic):   # CSVB200_ERR_OUT_OF_BOUNDS
        wrapped.gather_fields(np.array([0], dtype=np.uint32), np.array([1], dtype=np.uint32))
    wrapped.free()
    idx.free()


def test_second_device_in_the_same_process():
    """ADVICE r1: kernel attributes (> 48 KiB dynamic shared memory opt-in, occupancy) are per device.  A context on
    device 1 of the same process must build the same index (both kernels)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    data, _ = gen.quoted(3 << 20, seed=9)
    want = O.read_sse(data.tobytes())
    for dev in (0, 1, 0):
        c = cs.Context(dev)
        for sl in (data, data[:100_000]):
            idx = c.index_build(sl)
            assert np.array_equal(idx.to_host(), O.read_sse(sl.tobytes()) if sl is not data else want)
            idx.free()
        c.close()


def test_stream_read_callback_overrun_is_rejected(ctx):
    """ADVICE r1: a read() that returns more than `cap` bytes is refused before anything is copied."""
    def read(cap):
        return b"x" * (cap + 1)
    with pytest.raises(ValueError):
        ctx.index_build_stream(read, lambda e, f: None, chunk_bytes=1 << 20)


# ---- round 2: the exchange (peer-mapped mailboxes instead of a collective) and the single-process multi-GPU front end ----
def _exchange_chain(ctxs, exs, raw, cuts, dev_of, window=0):
    """Shards of `raw` through csvb200_index_build_shard_exchange, one rank after another IN RANK ORDER (a rank only
    ever waits for lower ranks, so ranks that share one GPU may run sequentially).  Returns the concatenated index,
    the shard infos and the per-rank counts / carries every rank's host view derives."""
    import torch
    G = len(cuts) - 1
    keep, idxs, infos = [], [], []
    for k in range(G):
        lo, hi = cuts[k], cuts[k + 1]
        buf = torch.zeros(max(hi - lo, 1) + 64, dtype=torch.uint8, device=dev_of(k))
        if hi > lo:
            buf[:hi - lo].copy_(torch.from_numpy(np.frombuffer(raw[lo:hi], dtype=np.uint8).copy()))
        torch.cuda.synchronize(dev_of(k))
        keep.append(buf)
        idx = ctxs[k].index_build_shard_exchange(exs[k], buf.data_ptr(), hi - lo, lo, window)
        infos.append(idx.shard_info())     # synchronises: rank k has posted before rank k + 1 starts
        idxs.append(idx)
    views = [exs[k].counts(idxs[k]) for k in range(G)]
    got = np.concatenate([i.to_host() for i in idxs])
    for i in idxs:
        i.free()
    return got, infos, views


def _check_exchange_result(raw, cuts, got, infos, views):
    want = O.closed_form_numpy(raw)
    assert got.shape == want.shape and (got == want).all()
    G = len(cuts) - 1
    true_carry = [O.shard_summary(raw[:cuts[k]])[0] for k in range(G)]
    seg = [O.closed_form_numpy(raw[cuts[k]:cuts[k + 1]], true_carry[k], cuts[k], with_sentinel=(k == 0)).size for k in range(G)]
    assert [i["carry_in"] for i in infos] == true_carry
    assert [i["entries"] for i in infos] == seg
    assert [i["base"] for i in infos] == [sum(seg[:k]) for k in range(G)]
    for counts, carries in views:          # every rank's host view of the whole exchange agrees with the oracle
        assert counts == seg and carries == true_carry


def test_exchange_emulated_ranks_on_one_gpu():
    """The mailbox protocol with G ranks emulated by G contexts on ONE device (rank order): posts, waits on the lower
    ranks, carry chain, bases, the misprediction re-index, the epochs of repeated builds; both kernels."""
    import torch
    dev = torch.device("cuda", 0)
    for kname in ("tma", "simple"):
        os.environ["CSVB200_KERNEL"] = kname
        try:
            G = 5
            ctxs = [cs.Context(0) for _ in range(G)]
            exs = [c.exchange(k, G) for k, c in enumerate(ctxs)]
            cs.Exchange.connect_local(exs)
            q, _ = gen.quoted(6 << 20, seed=44)
            raw = q.tobytes()
            n = len(raw)
            cuts = [0] + [(k * n) // G + 37 * k + 13 for k in range(1, G)] + [n]
            cuts[2] = raw.index(b'"', cuts[2]) + 1            # inside (or at the edge of) a quoted field
            got, infos, views = _exchange_chain(ctxs, exs, raw, cuts, lambda k: dev)
            _check_exchange_result(raw, cuts, got, infos, views)
            assert 1 in [i["carry_in"] for i in infos] and not any(i["redone"] for i in infos)
            # misleading data (an unescaped quote that looks like a closing one): that shard alone is re-indexed
            raw2 = (b'aa,bb"\n,cc,dd\n' * 40000) + b'x,y\n'
            cuts2 = [0, 14 * 10000 + 3, 14 * 20001 + 5, 14 * 30001 + 3, 14 * 35000, len(raw2)]
            got, infos, views = _exchange_chain(ctxs, exs, raw2, cuts2, lambda k: dev)
            _check_exchange_result(raw2, cuts2, got, infos, views)
            assert any(i["redone"] for i in infos) and not infos[0]["redone"]
            # forced boundaries (SURVEY 8d), empty and tiny shards, a third and fourth epoch on the same endpoints
            body = b'id,"text, with ""escapes"" and\r\nnewlines",tail\r\n' * 4000
            raw4 = b"h1,h2,h3\r\n" + body
            inside, esc, crlf = raw4.index(b"text"), raw4.index(b'""') + 1, raw4.index(b"\r\n", 50) + 1
            cuts4 = [0, inside, esc, crlf, len(raw4) // 2 + 5, len(raw4)]
            got, infos, views = _exchange_chain(ctxs, exs, raw4, cuts4, lambda k: dev)
            _check_exchange_result(raw4, cuts4, got, infos, views)
            raw3 = b"1,2,3\n" * 30000
            cuts3 = [0, 7, 7, 100, 100000, len(raw3)]
            got, infos, views = _exchange_chain(ctxs, exs, raw3, cuts3, lambda k: dev, window=4096)
            _check_exchange_result(raw3, cuts3, got, infos, views)
            assert [i["epoch"] for i in infos] == [4] * G
            for e in exs:
                e.close()
            for c in ctxs:
                c.close()
        finally:
            os.environ.pop("CSVB200_KERNEL", None)


def test_exchange_missing_rank_times_out_not_hangs():
    """A rank whose lower rank never posts gets CSVB200_ERR_EXCHANGE after the timeout: the wait is bounded."""
    import torch
    os.environ["CSVB200_EXCHANGE_TIMEOUT_MS"] = "50"
    try:
        ctxs = [cs.Context(0) for _ in range(2)]
        exs = [c.exchange(k, 2) for k, c in enumerate(ctxs)]
        cs.Exchange.connect_local(exs)
        raw = b"a,b,c\n" * 50000
        buf = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).to("cuda:0")
        idx = ctxs[1].index_build_shard_exchange(exs[1], buf.data_ptr(), len(raw), 12345)   # rank 0 never builds
        with pytest.raises(cs.GpuError) as ei:
            idx.sync()
        assert "exchange" in str(ei.value)
        idx.free()
        for e in exs:
            e.close()
        for c in ctxs:
            c.close()
    finally:
        os.environ.pop("CSVB200_EXCHANGE_TIMEOUT_MS", None)


def _multi_cases():
    q, _ = gen.quoted(40 << 20, seed=44)
    raw2 = (b'aa,bb"\n,cc,dd\n' * 300000) + b'x,y\n'
    return [("quoted40M", q.tobytes()), ("misleading", raw2), ("tiny", b"a,b\n1,2\n" * 20)]


@pytest.mark.parametrize("pinned", [False, True])
def test_multi_one_gpu_listed_several_times(pinned):
    """csvb200_multi_*: ONE byte slice in, ONE contiguous index out, the file cut at unaligned offsets across the
    listed devices.  Listing device 0 four times runs the whole protocol (uploads, exchange, bases, the
    misprediction re-index, placement of every segment in the caller's array) on a single GPU."""
    import torch
    m = cs.Multi([0, 0, 0, 0])
    for name, raw in _multi_cases():
        want = O.closed_form_numpy(raw)
        a = np.frombuffer(raw, dtype=np.uint8)
        if pinned:
            h_in = torch.from_numpy(a.copy()).pin_memory()
            h_out = torch.zeros(want.size + 8, dtype=torch.int64).pin_memory()
            ln = m.index_build_to_host(h_in.data_ptr(), a.size, h_out.data_ptr(), h_out.numel())
            got = h_out.numpy()[:ln].view(np.uint64)
        else:
            got = m.index_build(a)
        assert got.size == want.size and (got == want).all(), name
        st = m.stats()
        assert st["entries"] == want.size
        if name == "misleading":
            assert st["redone_mask"] != 0
    # explicit cuts: inside a quoted field, between the quotes of an escape, between CR and LF
    body = b'id,"text, with ""escapes"" and\r\nnewlines",tail\r\n' * 4000
    raw4 = b"h1,h2,h3\r\n" + body
    cuts = [0, raw4.index(b"text"), raw4.index(b'""') + 1, raw4.index(b"\r\n", 50) + 1, len(raw4)]
    got = m.index_build(np.frombuffer(raw4, dtype=np.uint8), cuts=cuts)
    assert (got == O.closed_form_numpy(raw4)).all()
    with pytest.raises(BufferError):
        out = np.zeros(10, dtype=np.uint64)
        m.index_build_to_host(np.frombuffer(raw4, dtype=np.uint8).ctypes.data, len(raw4), out.ctypes.data, out.size)
    m.close()


def test_multi_and_exchange_on_two_gpus():
    """Real peer memory: two devices of one process, host threads running concurrently, rows crossing NVLink."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    G = min(torch.cuda.device_count(), 8)
    m = cs.Multi(list(range(G)))
    for name, raw in _multi_cases():
        got = m.index_build(np.frombuffer(raw, dtype=np.uint8))
        assert (got == O.closed_form_numpy(raw)).all(), name
    m.close()


def test_c_caller_of_the_multi_gpu_abi():
    """VERDICT r1 J1: a C program with no Python / torch in the process indexes one buffer across the GPUs of the box
    through libcsvb200.so alone and equals the oracle (with one visible GPU the device is listed twice)."""
    import json
    import subprocess
    import torch
    from csv_simd_b200 import build as cbuild
    so = cbuild.build()
    oso = O.build()
    ndev = max(2, min(torch.cuda.device_count(), 8))
    devs = list(range(ndev)) if torch.cuda.device_count() >= 2 else [0] * ndev
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "test_multi")
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        subprocess.check_call(["gcc", "-O2", "-std=gnu99", "-Wall", "-I", os.path.join(root, "include"), "-I",
                               os.path.join(root, "oracle"), os.path.join(root, "tests", "c", "test_multi.c"), "-o", exe,
                               "-L", os.path.dirname(so), "-lcsvb200", "-L", os.path.dirname(oso), "-lcsv_oracle",
                               "-Wl,-rpath," + os.path.dirname(so), "-Wl,-rpath," + os.path.dirname(oso)])
        env = dict(os.environ, CSVB200_TEST_DEVICES=",".join(str(x) for x in devs))
        out = subprocess.run([exe, str(ndev), str(48 << 20)], capture_output=True, text=True, env=env, timeout=300)
        assert out.returncode == 0, out.stdout + out.stderr
        rep = json.loads(out.stdout.strip().splitlines()[-1])
        assert rep["equal_oracle"] is True and rep["ndev"] == ndev


def test_build_validate_byproducts(forced_ctxs):
    """CSVB200_BUILD_VALIDATE: is_ascii, the CR / LF count outside quotes and the per-tile non-ASCII map come out of
    the build launch itself; validate_utf8 on the index then reads only flagged tiles.  Against the oracle's
    is_ascii, the index itself (entries that are CR / LF) and CPython's decoder; both kernels; the index stays exact."""
    import torch
    rng = np.random.default_rng(11)
    for kname in ("tma", "simple"):
        c = forced_ctxs[kname]
        dev = torch.device("cuda", c.device)
        q, _ = gen.quoted(5 << 20, seed=45)
        cases_ = [("ascii quoted", q.tobytes())]
        u = bytearray(q.tobytes())
        good = "é,ü – ✓,🙂".encode()
        for pos in (0, 65500, 65536 - 2, 3 * 65536 - 1, 1 << 20, len(u) - len(good)):   # incl. sequences that straddle 64 KiB tiles
            u[pos:pos + len(good)] = good
        cases_.append(("valid utf8", bytes(u)))
        for bad_pos in (5, 65535, 2 * 65536, 4 * 65536 + 17, len(u) - 1):
            v = bytearray(u)
            v[bad_pos] = 0xFF
            cases_.append((f"invalid at {bad_pos}", bytes(v)))
        v = bytearray(q.tobytes())
        v[65534:65536] = b"\xe2\x82"          # truncated 3-byte sequence: its last byte would sit in the next tile
        cases_.append(("truncated at a tile edge", bytes(v)))
        for _ in range(3):
            v = bytearray(q.tobytes())
            for pos in rng.integers(0, len(v) - 8, size=40):
                v[pos] = int(rng.integers(0x80, 0x100))
            cases_.append(("random high bytes", bytes(v)))
        cases_.append(("small", ("a,b\n1,\"x\ny\"\r\n" * 20).encode() + "ö".encode()))
        for name, raw in cases_:
            a = np.frombuffer(raw, dtype=np.uint8)
            d = torch.empty(a.size + 64, dtype=torch.uint8, device=dev)
            d[:a.size].copy_(torch.from_numpy(a.copy()))
            idx = c.index_build_device(d.data_ptr(), a.size, cs.BUILD_VALIDATE)
            host = idx.to_host()
            want = O.closed_form_numpy(raw)
            assert host.size == want.size and (host == want).all(), (kname, name)
            is_ascii, newlines = idx.validation()
            assert is_ascii == O.is_ascii(raw), (kname, name)
            assert newlines == int(np.isin(a[host[1:].astype(np.int64)], np.array([0x0D, 0x0A], dtype=np.uint8)).sum()), (kname, name)
            assert idx.validate_utf8() == O.utf8_valid_up_to(raw), (kname, name)
            idx.free()
        # host form + KEEP_BYTES
        raw = cases_[1][1]
        idx = c.index_build(raw, cs.BUILD_VALIDATE | cs.BUILD_KEEP_BYTES)
        assert idx.validation()[0] is False and idx.validate_utf8() is None
        idx.free()
        idx = c.index_build(raw)
        with pytest.raises(cs.InvalidState):
            idx.validation()
        idx.free()


def _check_multi_lookups(m, nfields=64, size=6 << 20):
    data, rows = gen.unquoted(size, seed=45, nfields=nfields, modulus=10 ** 9)
    raw = data.tobytes()
    want_idx = O.closed_form_numpy(raw)
    mi = m.index_build_distributed(data)
    assert len(mi) == want_idx.size and (mi.to_host() == want_idx).all()
    segs = mi.segments()
    assert segs[0]["base"] == 0 and sum(s_["entries"] for s_ in segs) == want_idx.size
    assert all(segs[k]["base"] + segs[k]["entries"] == segs[k + 1]["base"] for k in range(len(segs) - 1))
    rc, jump = mi.tape_init(nfields, False)
    assert (jump, rc) == O.tape_init(want_idx.size, nfields, False) and rc == rows + 1
    nq = 200_000
    rec, fld = gen.queries(nq, rc, nfields, seed=46)
    rec[-2000:-1000] = rc - 1 + np.arange(1000, dtype=np.uint32)     # out of range -> None
    fld[-1000:] = nfields + np.arange(1000, dtype=np.uint32) % 5
    got = mi.seek_fields(rec, fld)
    live = (rec + 1 < rc) & (fld < nfields)
    s = (rec[live].astype(np.int64) + 1) * nfields + fld[live]
    assert (got[live, 0] == want_idx[s] + 1).all() and (got[live, 1] == want_idx[s + 1]).all()
    assert (got[~live] == U64MAX).all()
    for i in range(0, nq, 4001):
        w = O.seek_field(want_idx, len(raw), rc, nfields, False, int(rec[i]), int(fld[i]))
        assert (w is None and got[i, 0] == U64MAX) or (int(got[i, 0]), int(got[i, 1])) == w
    gr = mi.seek_records(rec[:5000])
    for i in range(0, 5000, 53):
        w = O.seek_record(want_idx, len(raw), rc, jump, nfields, int(rec[i]))
        assert (int(gr[i, 0]), int(gr[i, 1])) == w
    # a ragged file is reported exactly as TapeCore::init reports it (src/tape.rs:327,342-344)
    mi2 = m.index_build_distributed(np.frombuffer(raw + b"1,2\n", dtype=np.uint8))
    with pytest.raises(cs.InvalidCsvFormat):
        mi2.tape_init(nfields, False)
    with pytest.raises(cs.InvalidState):
        m.index_build_distributed(data).seek_fields(rec[:10], fld[:10])
    mi2.free()
    mi.free()


def test_multi_distributed_index_lookups_one_gpu():
    """csvb200_multi_index_*: the index stays distributed (segment k on device k), a batch of lookups is split over the
    devices and every kernel reads the slots it needs from whichever segment owns them.  Device 0 listed three times:
    the segment table, the slot routing and the batch split are exercised on one GPU."""
    m = cs.Multi([0, 0, 0])
    _check_multi_lookups(m)
    m.close()


def test_multi_distributed_index_lookups_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    m = cs.Multi(list(range(min(torch.cuda.device_count(), 8))))
    _check_multi_lookups(m, nfields=256, size=64 << 20)
    m.close()


def test_bench_dump_outputs_vs_oracle():
    """bench.py --dump-outputs: the index of the last timed step, as float64 .npy files within 64 MB, equal to the
    oracle's index of the same seeded bytes (length, end parity, both ends, the seeded sample, every block sum)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    size = 8 << 20
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "7", "--warmup", "1",
                              "--size", str(size), "--no-also", "--no-cpu-baseline", "--dump-outputs", d],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 7
        files = sorted(os.listdir(d))
        assert sum(os.path.getsize(os.path.join(d, f)) for f in files) <= 64 << 20
        got = {f[:-4]: np.load(os.path.join(d, f)) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    data, _ = gen.unquoted(size, seed=42)
    want, par = O.read_closed_form(data)
    pos = got["index_sample_pos"].astype(np.int64)
    assert got["index_len"].tolist() == [want.size] and got["end_parity"].tolist() == [par]
    assert (got["index_head"] == want[:got["index_head"].size]).all()
    assert (got["index_tail"] == want[want.size - got["index_tail"].size:]).all()
    assert pos.size > 0 and (got["index_sample"] == want[pos]).all()
    sums = got["index_block_sums"].astype(np.uint64)
    block = 1 << 16
    assert sums.size == -(-want.size // block)
    for k in range(sums.size):
        assert int(sums[k]) == int(want[k * block:(k + 1) * block].sum(dtype=np.uint64)), k
