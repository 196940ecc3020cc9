"""csvb200_seek_values on BASELINE config 5: the index of a 4 GiB wide-row (256-field) CSV, 10 M random (record, field)
queries (the input and queries of tools/bench_lookup.py, seeds 45 / 46).  One JSON line per case:

  values_device   seek_values_device, flags 0 (raw) and 3 (trim + unquote), CUDA events over --steps steps, with
                  seek_fields_device timed in the same process for reference
  records_device  seek_values_device in record mode (fld = NULL), --record-queries queries of ~4 KiB each
  values_host     the host form with pinned arrays (queries up, offsets / found bits / values down)
  gather_fields   csvb200_gather_fields with the same queries and pinned arrays
  multi_*         (--devices 0,1,...) the distributed index of the same bytes: host form, and the device form on every
                  device at once, each device a 1/G share of the queries
  cpu             one core: scalar seek_field plus the copy of the raw value (tools/values_cpu.c)

Every line carries the card name and its power limit read in the same run, the algorithmic bytes per query with their
formula, and a checksum of the values and found bits (equal to the CPU baseline's for the raw cases).

    python tools/bench_values.py [--size BYTES] [--queries N] [--steps K] [--devices 0,1] [--cases a,b]
    python tools/bench_values.py --cases gather_fields --package-root OTHER_CHECKOUT   # A/B against another tree
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools import gen  # noqa: E402

CASES = ["values_device", "records_device", "values_host", "gather_fields", "multi", "cpu"]


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"gpu": name, "power_limit": power}


def hbm_peak():
    """bytes/s: MEASURED_PEAKS.json next to the repository when present, else the data-sheet 7.7 TB/s"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        for k in ("hbm_bytes_per_s", "hbm_GBps", "hbm_gbps"):
            if k in d:
                return float(d[k]) * (1e9 if "GB" in k or "gb" in k else 1.0), "MEASURED_PEAKS.json"
    return 7.7e12, "data sheet (not measured)"


def checksum(offs, vals, found_words, nq):
    n_found = int(np.unpackbits(found_words.view(np.uint8), bitorder="little")[:nq].sum())
    total = int(offs[nq])
    return (int(vals[:total].astype(np.uint64).sum()) + 31 * total + 7 * n_found) & 0xFFFFFFFFFFFFFFFF


def cpu_lib():
    d = tempfile.mkdtemp(prefix="bench_values_")
    so = os.path.join(d, "values_cpu.so")
    subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tools", "values_cpu.c")])
    lib = C.CDLL(so)
    lib.values_cpu.restype = C.c_uint64
    lib.values_cpu.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                               C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=4 << 30)
    ap.add_argument("--queries", type=int, default=10_000_000)
    ap.add_argument("--record-queries", type=int, default=250_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--devices", default="")
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--package-root", default="", help="import csv_simd_b200 from this checkout instead")
    a = ap.parse_args()
    cases = set(a.cases.split(","))
    if a.package_root:
        sys.path.insert(0, os.path.abspath(a.package_root))
    import torch
    import csv_simd_b200 as cs
    info = card()
    peak, peak_src = hbm_peak()
    dev = torch.device("cuda", 0)
    data, rows = gen.unquoted(a.size, seed=45, nfields=256, modulus=10 ** 15)
    n = data.size
    d = torch.empty(n + 64, dtype=torch.uint8, device=dev)
    d[:n].copy_(torch.from_numpy(data))
    ctx = cs.Context(0)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)
    idx = ctx.index_build_device(d.data_ptr(), n)
    rc, jump = idx.tape_init(256, False)
    assert rc == rows + 1 and jump == 256
    nq = a.queries
    rec, fld = gen.queries(nq, rc, 256, seed=46)
    d_rec, d_fld = torch.from_numpy(rec.view(np.int32)).to(dev), torch.from_numpy(fld.view(np.int32)).to(dev)
    entry = 4 if n <= (1 << 32) else 8
    base = {"config": 5, "bytes": n, "queries": nq, "entry_bytes": entry, **info, "hbm_peak_Bps": peak, "peak_source": peak_src,
            "package_root": a.package_root or "."}

    def emit(d_):
        print(json.dumps({**base, **d_}), flush=True)

    def timed(fn, steps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    d_ranges = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    seek_ms = None
    if cases & {"values_device", "gather_fields"}:
        seek_ms = timed(lambda: idx.seek_fields_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, d_ranges.data_ptr()), a.steps)
    want_raw = None
    if "values_device" in cases:
        d_off = torch.empty(nq + 1, dtype=torch.int64, device=dev)
        d_found = torch.empty((nq + 63) // 64, dtype=torch.int64, device=dev)
        for flags in (0, 3):
            idx.seek_values_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, flags, d_off.data_ptr(), None, 0, d_found.data_ptr())
            torch.cuda.synchronize()
            total = int(d_off[nq].item())
            d_out = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)
            ms = timed(lambda: idx.seek_values_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, flags, d_off.data_ptr(),
                                                      d_out.data_ptr(), total, d_found.data_ptr()), a.steps)
            offs = d_off.cpu().numpy().view(np.uint64)
            vals = d_out.cpu().numpy()
            words = d_found.cpu().numpy().view(np.uint64)
            if flags == 0:
                want_raw = (offs, vals, words)
            vb = total / nq
            # offsets pass: queries in, 2 entries, the value's bytes, offsets + found bits out; write pass: queries and 2
            # entries again, the offsets, the value's bytes read and written
            alg = 2 * (8 + 2 * entry) + 8 + 16 + 1 / 8 + 3 * vb
            emit({"case": "values_device", "flags": flags, "ms": ms, "Mvalues_per_s": nq / ms / 1e3,
                  "value_bytes": total, "alg_bytes_per_query": alg,
                  "alg_formula": "2*(8 + 2*entry_bytes) + 8 + 16 + 1/8 + 3*mean_value_bytes",
                  "alg_GBps": alg * nq / ms / 1e6, "share_of_hbm_peak": alg * nq / ms * 1e3 / peak,
                  "seek_fields_device_ms": seek_ms, "checksum": checksum(offs, vals, words, nq)})
            del d_out
    if "records_device" in cases:
        nr = a.record_queries
        r_rec, _ = gen.queries(nr, rc, 256, seed=47)
        dr = torch.from_numpy(r_rec.view(np.int32)).to(dev)
        d_off = torch.empty(nr + 1, dtype=torch.int64, device=dev)
        d_found = torch.empty((nr + 63) // 64, dtype=torch.int64, device=dev)
        idx.seek_values_device(dr.data_ptr(), None, nr, 0, d_off.data_ptr(), None, 0, d_found.data_ptr())
        torch.cuda.synchronize()
        total = int(d_off[nr].item())
        d_out = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)
        d_rr = torch.empty((nr, 2), dtype=torch.int64, device=dev)
        rec_seek_ms = timed(lambda: idx.seek_records_device(dr.data_ptr(), nr, d_rr.data_ptr()), a.steps)
        ms = timed(lambda: idx.seek_values_device(dr.data_ptr(), None, nr, 0, d_off.data_ptr(), d_out.data_ptr(), total,
                                                  d_found.data_ptr()), a.steps)
        vb = total / nr
        alg = 2 * (4 + 2 * entry) + 8 + 8 + 1 / 8 + 2 * vb
        emit({"case": "records_device", "queries": nr, "ms": ms, "Mvalues_per_s": nr / ms / 1e3, "value_bytes": total,
              "alg_bytes_per_query": alg, "alg_formula": "2*(4 + 2*entry_bytes) + 8 + 8 + 1/8 + 2*mean_record_bytes",
              "alg_GBps": alg * nr / ms / 1e6, "share_of_hbm_peak": alg * nr / ms * 1e3 / peak,
              "seek_records_device_ms": rec_seek_ms,
              "checksum": checksum(d_off.cpu().numpy().view(np.uint64), d_out.cpu().numpy(),
                                   d_found.cpu().numpy().view(np.uint64), nr)})
        del d_out
    h_rec = torch.from_numpy(rec.view(np.int32)).pin_memory()
    h_fld = torch.from_numpy(fld.view(np.int32)).pin_memory()
    h_off = torch.empty(nq + 1, dtype=torch.int64).pin_memory()
    L = idx._lib
    if cases & {"values_host", "gather_fields"}:
        ln = C.c_size_t()
        assert L.csvb200_gather_fields(idx._h, C.c_void_p(h_rec.data_ptr()), C.c_void_p(h_fld.data_ptr()), nq,
                                       C.c_void_p(h_off.data_ptr()), None, 0) in (0, 9)
        total = int(h_off[nq].item())
        h_out = torch.empty(max(total, 1), dtype=torch.uint8).pin_memory()
        h_found = torch.empty((nq + 63) // 64, dtype=torch.int64).pin_memory()

        def best_of(fn, reps=5):
            best = 1e9
            for _ in range(reps):
                torch.cuda.synchronize()
                t = time.perf_counter()
                assert fn() == 0
                best = min(best, time.perf_counter() - t)
            return best

        if "values_host" in cases:
            s = best_of(lambda: L.csvb200_seek_values(idx._h, C.c_void_p(h_rec.data_ptr()), C.c_void_p(h_fld.data_ptr()), nq, 0,
                                                      C.c_void_p(h_off.data_ptr()), C.c_void_p(h_out.data_ptr()), total,
                                                      C.byref(ln), C.c_void_p(h_found.data_ptr())))
            emit({"case": "values_host", "flags": 0, "pinned": True, "s": s, "Mvalues_per_s": nq / s / 1e6,
                  "checksum": checksum(h_off.numpy().view(np.uint64), h_out.numpy(), h_found.numpy().view(np.uint64), nq)})
        if "gather_fields" in cases:
            times = []
            for _ in range(5):
                times.append(best_of(lambda: L.csvb200_gather_fields(idx._h, C.c_void_p(h_rec.data_ptr()),
                                                                     C.c_void_p(h_fld.data_ptr()), nq,
                                                                     C.c_void_p(h_off.data_ptr()),
                                                                     C.c_void_p(h_out.data_ptr()), total), reps=1))
            offs = h_off.numpy().view(np.uint64)
            vals = h_out.numpy()
            emit({"case": "gather_fields", "pinned": True, "s": min(times), "s_median": float(np.median(times)),
                  "Mvalues_per_s": nq / min(times) / 1e6, "value_bytes": total,
                  "byte_sum": int(vals[:total].astype(np.uint64).sum()), "offsets_sum": int(offs.sum())})
        del h_out
    if "cpu" in cases:
        host = idx.to_host()
        lib = cpu_lib()
        offs = np.empty(nq + 1, dtype=np.uint64)
        words = np.zeros((nq + 63) // 64, dtype=np.uint64)
        out = np.empty(int(want_raw[0][nq]) if want_raw is not None else nq * 32, dtype=np.uint8)
        t = time.perf_counter()
        cs_cpu = lib.values_cpu(host.ctypes.data, host.size, data.ctypes.data, rc, 256, 256, rec.ctypes.data, fld.ctypes.data,
                                nq, offs.ctypes.data, out.ctypes.data, words.ctypes.data)
        s = time.perf_counter() - t
        line = {"case": "cpu", "threads": 1, "s": s, "Mvalues_per_s": nq / s / 1e6, "checksum": int(cs_cpu)}
        if want_raw is not None:
            line["parity_with_values_device_flags0"] = (int(cs_cpu) == checksum(*want_raw, nq)
                                                        and bool((offs == want_raw[0]).all()))
        emit(line)
    if a.devices and "multi" in cases:
        devs = [int(x) for x in a.devices.split(",")]
        m = cs.Multi(devs)
        mi = m.index_build_distributed(data)
        mi.tape_init(256, False)
        G = len(devs)
        ln = C.c_size_t()
        assert mi._lib.csvb200_multi_seek_values(mi._h, C.c_void_p(h_rec.data_ptr()), C.c_void_p(h_fld.data_ptr()), nq, 0,
                                                 C.c_void_p(h_off.data_ptr()), None, 0, C.byref(ln), None) in (0, 9)
        total = ln.value
        h_out = torch.empty(max(total, 1), dtype=torch.uint8).pin_memory()
        h_found = torch.empty((nq + 63) // 64, dtype=torch.int64).pin_memory()
        best = 1e9
        for _ in range(3):
            t = time.perf_counter()
            assert mi._lib.csvb200_multi_seek_values(mi._h, C.c_void_p(h_rec.data_ptr()), C.c_void_p(h_fld.data_ptr()), nq, 0,
                                                     C.c_void_p(h_off.data_ptr()), C.c_void_p(h_out.data_ptr()), total,
                                                     C.byref(ln), C.c_void_p(h_found.data_ptr())) == 0
            best = min(best, time.perf_counter() - t)
        line = {"case": "multi_values_host", "devices": devs, "s": best, "Mvalues_per_s": nq / best / 1e6,
                "checksum": checksum(h_off.numpy().view(np.uint64), h_out.numpy(), h_found.numpy().view(np.uint64), nq)}
        if want_raw is not None:
            line["parity_with_one_gpu"] = line["checksum"] == checksum(*want_raw, nq)
        emit(line)
        del h_out
        # device form: device k resolves its 1/G share of the queries, all devices at once
        shares = []
        for k, dv in enumerate(devs):
            q0, q1 = nq * k // G, nq * (k + 1) // G
            tdev = torch.device("cuda", dv)
            sr = torch.from_numpy(rec[q0:q1].view(np.int32).copy()).to(tdev)
            sf = torch.from_numpy(fld[q0:q1].view(np.int32).copy()).to(tdev)
            so = torch.empty(q1 - q0 + 1, dtype=torch.int64, device=tdev)
            mi.seek_values_device(k, sr.data_ptr(), sf.data_ptr(), q1 - q0, 0, so.data_ptr())
            torch.cuda.synchronize(tdev)
            tot = int(so[q1 - q0].item())
            sv = torch.empty(max(tot, 1), dtype=torch.uint8, device=tdev)
            shares.append((k, tdev, sr, sf, so, sv, tot, q1 - q0))

        def all_devices():
            for k, tdev, sr, sf, so, sv, tot, cnt in shares:
                mi.seek_values_device(k, sr.data_ptr(), sf.data_ptr(), cnt, 0, so.data_ptr(), sv.data_ptr(), tot)
            for s_ in shares:
                torch.cuda.synchronize(s_[1])

        all_devices()
        t = time.perf_counter()
        for _ in range(a.steps):
            all_devices()
        s = (time.perf_counter() - t) / a.steps
        emit({"case": "multi_values_device", "devices": devs, "ms": s * 1e3, "Mvalues_per_s": nq / s / 1e6,
              "timing": "host clock around all devices' launches, ending in a synchronise of every device"})
        mi.free()
        m.close()
    idx.free()
    ctx.close()


if __name__ == "__main__":
    main()
