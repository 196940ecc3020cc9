"""A/B of CSVB200_TUNE values in ONE process on the same box and the same bytes.

    python tools/kvariants.py "0 1024" [builds] [bytes] [workloads]

Round 2 ran every kernel shape and experiment knob through it (profiles/r02_kvariants.md, decoded by
tools/kvariants_table.py); the losers are deleted, and the one value left is 1024 (bit 0x400): the no-chain timing
experiment, where each build reuses the look-back descriptors of the build before it.

For every workload (cfg2_unquoted, cfg3_quoted) and every tune value: a fresh context with CSVB200_TUNE set,
3 warm-up builds, `builds` timed device-resident builds (CUDA events around each launch), and an element-wise
compare of the index with the one the FIRST tune value produced (which the -m gpu suite pins to the oracle).
The variants are interleaved round-robin so that clock / thermal drift hits all of them alike.
Prints one JSON line per (workload, tune)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import csv_simd_b200 as cs  # noqa: E402
from tools import gen  # noqa: E402


def index_tensor(idx, dev):
    n = len(idx)

    class _Raw:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (idx.device_ptr, False), "version": 2}
    return torch.as_tensor(_Raw(), device=dev)


def main():
    tunes = [int(t) for t in (sys.argv[1] if len(sys.argv) > 1 else "0").split()]
    builds = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    size = int(sys.argv[3]) if len(sys.argv) > 3 else (1 << 30)
    wls = sys.argv[4].split(",") if len(sys.argv) > 4 else ["cfg2_unquoted", "cfg3_quoted"]
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    dev = torch.device("cuda", 0)
    for wl in wls:
        data, _ = (gen.unquoted(size, seed=42) if wl == "cfg2_unquoted" else gen.quoted(size, seed=43))
        n = int(data.size)
        d = torch.empty(n + 64, dtype=torch.uint8, device=dev)
        d[:n].copy_(torch.from_numpy(data))
        ctxs = {}
        for t in tunes:
            os.environ["CSVB200_TUNE"] = str(t)
            ctxs[t] = cs.Context(0)
        ref = None
        ms = {t: [] for t in tunes}
        ok = {}
        E = 0
        for t in tunes:   # warm-up + parity
            for _ in range(3):
                idx = ctxs[t].index_build_device(d.data_ptr(), n)
                idx.sync()
                cur = index_tensor(idx, dev)
                if ref is None:
                    ref = cur.clone()
                    E = len(idx)
                ok[t] = bool(len(idx) == ref.numel() and torch.equal(cur, ref))
                idx.free()
        for _ in range(builds):
            for t in tunes:
                idx = ctxs[t].index_build_device(d.data_ptr(), n)
                idx.sync()
                ms[t].append(ctxs[t].last_build_ms())
                idx.free()
        for t in tunes:
            m = sorted(ms[t])
            med = m[len(m) // 2]
            avg = sum(m) / len(m)
            print(json.dumps({"workload": wl, "tune": t, "n": n, "entries": E, "parity_vs_first": ok[t],
                              "kernel_ms_avg": round(avg, 5), "kernel_ms_med": round(med, 5), "kernel_ms_min": round(m[0], 5),
                              "frac_of_measured_hbm": round((n + 8 * E) / (avg * 1e-3) / 1e9 / peak, 4),
                              "csv_gbs": round(n / (avg * 1e-3) / 1e9, 1)}), flush=True)
            ctxs[t].close()
        del d, ref
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
