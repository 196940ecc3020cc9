"""The halo of csvb200_multi_validate_utf8 (csrc/utf8_halo.h), compiled with g++ alone and checked against a brute-force
statement over random cut tables with empty shards and shards of 1-3 bytes: built from the first and last 3 bytes of
every shard only, the halo of shard k holds exactly the 3 bytes of the whole input before cuts[k] (0 before the first
byte) and the bytes after cuts[k + 1] up to 3 or the end of the input."""
import os
import subprocess
import tempfile

SRC = r'''
#include "utf8_halo.h"
#include <cstdio>
#include <cstdint>
#include <vector>
using namespace csvb200;

static uint64_t rng = 88172645463325252ull;
static uint64_t next() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return rng; }

int main()
{
    long bad = 0, cases = 0, multi = 0, short_after = 0;
    for (int t = 0; t < 50000; ++t) {
        const uint32_t nshard = 1 + next() % 10;
        std::vector<uint64_t> cuts(nshard + 1, 0);
        for (uint32_t k = 1; k <= nshard; ++k) {
            const uint64_t kind = next() % 4;   // empty, 1-3 bytes, a few bytes, longer
            const uint64_t len = kind == 0 ? 0 : kind == 1 ? 1 + next() % 3 : kind == 2 ? 4 + next() % 3 : next() % 40;
            cuts[k] = cuts[k - 1] + len;
        }
        const uint64_t n = cuts[nshard];
        std::vector<uint8_t> bytes(n);
        for (uint64_t i = 0; i < n; ++i) bytes[i] = (uint8_t)(1 + next() % 255);   // never 0: a 0 would hide a missing byte
        std::vector<uint8_t> first3(3 * nshard, 0), last3(3 * nshard, 0);
        for (uint32_t j = 0; j < nshard; ++j) {
            const uint64_t len = cuts[j + 1] - cuts[j];
            for (uint64_t i = 0; i < 3 && i < len; ++i) {
                first3[3 * j + i] = bytes[cuts[j] + i];
                last3[3 * j + i] = bytes[cuts[j + 1] - 1 - i];
            }
        }
        for (uint32_t k = 0; k < nshard; ++k) {
            const Utf8Halo h = utf8_halo(cuts.data(), nshard, k, reinterpret_cast<const uint8_t(*)[3]>(first3.data()),
                                         reinterpret_cast<const uint8_t(*)[3]>(last3.data()));
            ++cases;
            uint32_t before = 0, after = 0, after_len = 0;
            for (uint64_t d = 0; d < 3; ++d) {
                if (cuts[k] >= d + 1) before |= (uint32_t)bytes[cuts[k] - 1 - d] << (8 * d);
                if (cuts[k + 1] + d < n) {
                    after |= (uint32_t)bytes[cuts[k + 1] + d] << (8 * d);
                    after_len = (uint32_t)d + 1;
                }
            }
            if (h.before != before || h.after != after || h.after_len != after_len) {
                if (bad < 5) std::printf("t=%d k=%u: %06x/%06x/%u want %06x/%06x/%u\n", t, k, h.before, h.after, h.after_len,
                                         before, after, after_len);
                ++bad;
            }
            // the halo reaches over at least one more cut than its own (a neighbour shorter than 3 bytes, or empty)
            bool spans = false;
            for (uint32_t j = 0; j <= nshard; ++j)
                if (j != k && j != k + 1 && ((cuts[j] < cuts[k] && cuts[j] + 3 > cuts[k]) ||
                                             (cuts[j] > cuts[k + 1] && cuts[j] < cuts[k + 1] + 3 && cuts[j] < n)))
                    spans = true;
            if (spans) ++multi;
            if (after_len > 0 && after_len < 3) ++short_after;
        }
    }
    std::printf("bad=%ld cases=%ld across_cuts=%ld short_after=%ld\n", bad, cases, multi, short_after);
    return bad != 0 || multi == 0 || short_after == 0;
}
'''


def test_halo_is_the_bytes_around_the_shard():
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
