"""Column materialisation over a distributed index (csvb200_multi_materialize_columns), config 4: G GiB of quote-heavy
CSV, 1 GiB per GPU, at G = 1, 2 and 8, for 1, 8 and 16 columns with UNQUOTE | TRIM.  One JSON line per (G, columns):

  - wall time of the host call that fills the caller's (pageable, numpy) arrays: both passes on every device, the
    boundary rows, and the device-to-host copies of offsets and values;
  - device time per pass, from torch.profiler in a separate run: per device the summed duration of the offsets kernels
    (the sizing pass and the rebased re-run before the copy) and of the write kernels, then the max over devices;
  - the same columns from csvb200_materialize_columns on one GPU's 1 GiB share (the first part), as the reference point;
  - parity: the first share's records of the distributed result equal the one-GPU result byte for byte.

The name and power limit of the cards are read with nvidia-smi in the same run.  With fewer GPUs than G, device 0 is
listed G times; its shards then run one after another and the line says so ("emulated").

    python tools/bench_multi_mat.py [--gpus 1,2,8] [--cols 1,8,16] [--steps 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import csv_simd_b200 as cs  # noqa: E402
from tools import gen  # noqa: E402

GiB = 1 << 30
FLAGS = cs.FIELD_UNQUOTE | cs.FIELD_TRIM


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout
    return [line.strip() for line in out.splitlines() if line.strip()]


def make_data(G):
    parts = [None] * G
    ts = [threading.Thread(target=lambda j=j: parts.__setitem__(j, gen.quoted(GiB, seed=44, first_row=j << 32,
                                                                              with_header=(j == 0))[0].copy()))
          for j in range(G)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return np.concatenate(parts), int(parts[0].size)


class Filler:
    """one csvb200_*materialize_columns fill call into preallocated numpy arrays (sizes from a first call)"""

    def __init__(self, fn, handle, fields, nrec, lens):
        k = len(fields)
        self.fn, self.h, self.nrec = fn, handle, nrec
        self.f = np.ascontiguousarray(fields, dtype=np.uint32)
        self.offs = [np.zeros(nrec + 1, dtype=np.uint64) for _ in range(k)]
        self.vals = [np.empty(int(n), dtype=np.uint8) for n in lens]
        for a in self.offs + self.vals:
            a.fill(0)   # fault the pages in before the timed calls
        self.p_off = (C.c_void_p * k)(*[o.ctypes.data for o in self.offs])
        self.p_out = (C.c_void_p * k)(*[v.ctypes.data if v.size else None for v in self.vals])
        self.caps = (C.c_size_t * k)(*[v.size for v in self.vals])
        self.lens = (C.c_size_t * k)()

    def __call__(self):
        rc = self.fn(self.h, self.f.ctypes.data, self.f.size, 0, self.nrec, FLAGS, self.p_off, self.p_out, self.caps, self.lens)
        assert rc == 0, rc

    def d2h_bytes(self):
        return sum(v.size for v in self.vals) + 8 * sum(o.size for o in self.offs)


def timed(fill, steps):
    fill()
    best = 1e9
    for _ in range(steps):
        t = time.perf_counter()
        fill()
        best = min(best, time.perf_counter() - t)
    return best


def kernel_ms(fill):
    """per device: summed ms of the offsets kernels and of the write kernels of one call (torch.profiler, CUPTI)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fill()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA or "materialize" not in e.name:
            continue
        kind = "offsets" if "offsets" in e.name else "write" if "write" in e.name else None
        if kind:
            d = per.setdefault(e.device_index, {"offsets": 0.0, "write": 0.0})
            d[kind] += e.time_range.elapsed_us() / 1e3
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--cols", default="1,8,16")
    ap.add_argument("--steps", type=int, default=3)
    a = ap.parse_args()
    cards = gpu_info()
    ndev = torch.cuda.device_count()
    lib = cs._lib.load()
    for G in [int(x) for x in a.gpus.split(",")]:
        devs = list(range(G)) if ndev >= G else [0] * G
        data, share = make_data(G)
        # reference: the first 1 GiB part on one GPU
        ctx = cs.Context(0)
        idx = ctx.index_build(data[:share], cs.BUILD_KEEP_BYTES)
        rc1, _ = idx.tape_init(16, True)
        m = cs.Multi(devs)
        mi = m.index_build_distributed(data)
        rc, _ = mi.tape_init(16, True)
        for ncols in [int(x) for x in a.cols.split(",")]:
            fields = list(range(ncols))
            ref = idx.materialize_columns(fields, 0, rc1 - 1, FLAGS)
            ref_fill = Filler(lib.csvb200_materialize_columns, idx._h, fields, rc1 - 1, [v.size for _, v in ref])
            got = mi.materialize_columns(fields, 0, rc - 1, FLAGS)
            ok = all((g_off[:rc1] == w_off).all() and g_val[:w_val.size].tobytes() == w_val.tobytes()
                     for (g_off, g_val), (w_off, w_val) in zip(got, ref))
            fill = Filler(lib.csvb200_multi_materialize_columns, mi._h, fields, rc - 1, [v.size for _, v in got])
            del got, ref
            wall = timed(fill, a.steps)
            ref_wall = timed(ref_fill, a.steps)
            per = kernel_ms(fill)
            ref_per = kernel_ms(ref_fill)
            d2h = fill.d2h_bytes()
            print(json.dumps({
                "bench": "multi_materialize_columns", "gpus": G, "devices": devs, "emulated": ndev < G, "cards": cards,
                "workload": "cfg4 grammar, 1 GiB per GPU, default cuts, UNQUOTE | TRIM", "bytes": int(data.size),
                "records": rc - 1, "columns": ncols,
                "wall_s": wall, "d2h_bytes": d2h, "d2h_gbs": d2h / wall / 1e9,
                "offsets_kernels_ms_max_over_devices": max(d["offsets"] for d in per.values()),
                "write_kernels_ms_max_over_devices": max(d["write"] for d in per.values()),
                "per_device_ms": {str(k): v for k, v in sorted(per.items())},
                "one_gpu_reference": {"bytes": share, "records": rc1 - 1, "wall_s": ref_wall, "d2h_bytes": ref_fill.d2h_bytes(),
                                      "offsets_kernels_ms": sum(d["offsets"] for d in ref_per.values()),
                                      "write_kernels_ms": sum(d["write"] for d in ref_per.values())},
                "parity": {"checked": True, "ok": bool(ok), "what": "first share's records == csvb200_materialize_columns"},
            }), flush=True)
            assert ok
            del fill, ref_fill
        mi.free()
        m.close()
        idx.free()
        ctx.close()
        del data


if __name__ == "__main__":
    main()
