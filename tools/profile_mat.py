"""K6 multi-column materialisation on a mid-sized input, for timing and ncu:
    python tools/profile_mat.py [cfg2_unquoted|cfg3_quoted] [ncols] [bytes]
Prints the time of the offsets pass alone and of offsets + write (CUDA events on the context's stream)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import csv_simd_b200 as cs  # noqa: E402
from tools import gen  # noqa: E402


def main():
    wl = sys.argv[1] if len(sys.argv) > 1 else "cfg2_unquoted"
    ncols = int(sys.argv[2]) if len(sys.argv) > 2 else 8
    size = int(sys.argv[3]) if len(sys.argv) > 3 else (256 << 20)
    dev = torch.device("cuda", 0)
    ctx = cs.Context(0)
    data, rows = gen.unquoted(size, seed=42) if wl == "cfg2_unquoted" else gen.quoted(size, seed=43)
    n = data.size
    d = torch.empty(n + 64, dtype=torch.uint8, device=dev)
    d[:n].copy_(torch.from_numpy(data))
    torch.cuda.synchronize()
    idx = ctx.index_build_device(d.data_ptr(), n)
    rc, jump = idx.tape_init(16, wl != "cfg2_unquoted")
    nrec = rc - 1
    cols = list(range(1, 16, 2))[:ncols] if ncols <= 8 else list(range(ncols))
    stream = torch.cuda.Stream(dev)
    ctx.set_stream(stream.cuda_stream)
    d_offs = [torch.empty(nrec + 1, dtype=torch.int64, device=dev) for _ in cols]
    p_offs = [t.data_ptr() for t in d_offs]
    torch.cuda.synchronize()
    idx.materialize_columns_device(cols, 0, nrec, 3, p_offs)
    torch.cuda.synchronize()     # (index.sync() waits for the BUILD only)
    totals = [int(t[-1].item()) for t in d_offs]
    d_outs = [torch.empty(max(t, 1), dtype=torch.uint8, device=dev) for t in totals]
    p_outs = [t.data_ptr() for t in d_outs]
    torch.cuda.synchronize()

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / reps
    ms_off = timed(lambda: idx.materialize_columns_device(cols, 0, nrec, 3, p_offs))
    ms_both = timed(lambda: idx.materialize_columns_device(cols, 0, nrec, 3, p_offs, p_outs, totals))
    print(json.dumps({"workload": wl, "bytes": n, "records": nrec, "columns": cols, "ms_offsets": ms_off, "ms_offsets_plus_write": ms_both, "value_bytes": sum(totals)}))
    idx.free()
    ctx.close()


if __name__ == "__main__":
    main()
