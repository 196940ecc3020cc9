"""The interior / boundary split of csvb200_multi_materialize_columns (csrc/record_split.h), compiled with g++ alone and
checked against a brute-force statement record by record: over random segment tables with empty segments and segments
shorter than a row, every requested record is assigned exactly once, in record order, to the right kind of piece."""
import os
import subprocess
import tempfile

SRC = r'''
#include "record_split.h"
#include <cstdio>
#include <cstdint>
#include <vector>
using namespace csvb200;

static uint64_t rng = 88172645463325252ull;
static uint64_t next() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return rng; }

int main()
{
    long bad = 0, cases = 0, boundary = 0, interior = 0, dead = 0, wide = 0;
    for (int t = 0; t < 20000; ++t) {
        const uint32_t nseg = 1 + next() % 16;
        const uint64_t jump = 1 + next() % 9;
        std::vector<uint64_t> base(nseg + 1, 0);
        for (uint32_t k = 1; k <= nseg; ++k) {
            const uint64_t kind = next() % 4;   // empty, shorter than a row, about a row, long
            const uint64_t len = kind == 0 ? 0 : kind == 1 ? next() % jump : kind == 2 ? jump + next() % 3 : next() % 200;
            base[k] = base[k - 1] + len;
        }
        base[nseg] += 1 + next() % 3;
        const uint64_t len = base[nseg];
        const uint32_t record_cnt = (uint32_t)((len - 1) / jump);
        uint32_t first = (uint32_t)(next() % (record_cnt + 4));
        if (t % 7 == 0) first = 0xFFFFFFFFu - (uint32_t)(next() % 4);   // the window wraps past record 0xFFFFFFFF
        const uint32_t nrec = (uint32_t)(next() % (record_cnt + 6));
        const std::vector<RecordPiece> pieces = split_records(base.data(), nseg, jump, record_cnt, first, nrec);
        ++cases;
        uint64_t pos = 0;
        for (size_t i = 0; i < pieces.size(); ++i) {
            const RecordPiece& p = pieces[i];
            if (p.count == 0 || p.first != (uint32_t)(first + pos)) { ++bad; break; }
            if (i > 0 && p.interior() && pieces[i - 1].interior() && p.seg_lo == pieces[i - 1].seg_lo) ++bad;   // not maximal
            if (!p.interior() && p.count != 1) ++bad;
            for (uint32_t j = 0; j < p.count; ++j, ++pos) {
                const uint32_t rp1 = (uint32_t)(first + pos) + 1u;
                if (rp1 >= record_cnt) {
                    if (p.seg_lo != nseg || p.seg_hi != nseg) ++bad;
                    ++dead;
                    continue;
                }
                // brute force: the segment of every slot the record reads
                std::vector<uint32_t> segs;
                for (uint64_t s = (uint64_t)rp1 * jump; s <= (uint64_t)(rp1 + 1) * jump; ++s) {
                    uint32_t k = 0;
                    while (!(base[k] <= s && s < base[k + 1])) ++k;
                    segs.push_back(k);
                }
                const bool one = segs.front() == segs.back();
                if (one != p.interior() || p.seg_lo != segs.front() || p.seg_hi != segs.back()) ++bad;
                if (one) ++interior; else ++boundary;
                if (segs.back() > segs.front() + 1) ++wide;
            }
        }
        if (pos != nrec) ++bad;
    }
    std::printf("bad=%ld cases=%ld interior=%ld boundary=%ld dead=%ld three_segments=%ld\n", bad, cases, interior, boundary,
                dead, wide);
    return bad != 0 || boundary == 0 || wide == 0 || dead == 0;
}
'''


def test_split_assigns_every_record_once_in_order():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "t.cpp")
        exe = os.path.join(td, "t")
        open(src, "w").write(SRC)
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-I", os.path.join(root, "csv_simd_b200", "csrc"), src, "-o", exe],
                       check=True)
        out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        assert "bad=0" in out.stdout
