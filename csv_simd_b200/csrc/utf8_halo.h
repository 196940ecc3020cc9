// utf8_halo.h -- the bytes around one byte shard of a distributed input that K7 needs to judge that shard alone
// (csvb200_multi_validate_utf8).  Pure host code with no CUDA dependency, so a CPU test can compile it with g++ alone.
//
// Every UTF-8 rule is local to 4 bytes (validate.cu), so shard k = global bytes [cuts[k], cuts[k + 1]) can be judged on
// its own device once it sees up to 3 bytes before cuts[k] (continuation bytes owed by a sequence led earlier) and up
// to 3 bytes after cuts[k + 1] (look-ahead of the leads near its end).  Shards may be empty or shorter than 3 bytes, so
// a halo byte can come from any shard on either side; the host knows the first and last (up to) 3 bytes of every shard
// and assembles the halo from those.  At the ends of the input the halo is absent, as the one-GPU kernel reads it there:
// 0 before the first byte, nothing after the last.
#pragma once
#include <cstdint>

namespace csvb200 {

struct Utf8Halo {
    uint32_t before;      // byte d (bits 8d .. 8d + 7) = global byte cuts[k] - 1 - d, or 0 where the input has none
    uint32_t after;       // byte d = global byte cuts[k + 1] + d, for d < after_len (the other bytes are 0)
    uint32_t after_len;   // 0 .. 3: fewer than 3 where the input ends sooner
};

// cuts[0 .. nshard] non-decreasing, cuts[0] = 0, cuts[nshard] = n.  first3[j][i] = global byte cuts[j] + i and
// last3[j][i] = global byte cuts[j + 1] - 1 - i, both for i < min(3, cuts[j + 1] - cuts[j]).
inline Utf8Halo utf8_halo(const uint64_t* cuts, uint32_t nshard, uint32_t k, const uint8_t (*first3)[3],
                          const uint8_t (*last3)[3])
{
    Utf8Halo h{0u, 0u, 0u};
    for (uint64_t d = 0; d < 3; ++d) {
        if (cuts[k] >= d + 1) {
            // the shard j < k that holds byte g: the last one starting at or below it (the shards between are empty)
            const uint64_t g = cuts[k] - 1 - d;
            uint32_t j = k;
            while (cuts[j] > g) --j;
            h.before |= (uint32_t)last3[j][cuts[j + 1] - 1 - g] << (8 * d);
        }
        const uint64_t g = cuts[k + 1] + d;
        if (g < cuts[nshard]) {
            uint32_t j = k + 1;
            while (cuts[j + 1] <= g) ++j;
            h.after |= (uint32_t)first3[j][g - cuts[j]] << (8 * d);
            h.after_len = (uint32_t)d + 1;
        }
    }
    return h;
}

}  // namespace csvb200
