// internal.h -- declarations shared by the CUDA translation units of libcsvb200.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace csvb200 {

// ---- tile geometry of the fused index-build kernel --------------------------
constexpr int kThreads = 256;                              // threads per CTA
constexpr int kBytesPerThread = 128;                       // four 32-byte bit-slice groups = one 128 B swizzle row
constexpr int kTileBytes = kThreads * kBytesPerThread;     // 32 KiB of CSV per tile
constexpr int kWarps = kThreads / 32;

// ---- look-back descriptor (one u64 per tile, written/read as a single word) --
//   [63:62] status   0 = not ready, 1 = tile aggregate, 2 = inclusive prefix
//   [61]    parity   aggregate: quote parity of the tile; prefix: absolute parity at tile end
//   [60:41] tag      of the launch that wrote the word (BuildParams::desc_tag, 1 .. 2^20 - 1): a descriptor whose tag is
//                    not the reader's own launch reads as "not ready", so the scratch is NOT zeroed between launches
//                    (round 1 memset 2 MiB per GiB of input in front of every launch); the ticket and the counters in
//                    the head of the scratch are put back to zero by the last CTA that touches them
//   aggregate: [19:0] c0 = unquoted separators if the tile is entered outside quotes
//              [39:20] c1 = same if entered inside quotes
//   prefix:    [40:0] absolute number of index entries emitted up to the tile end (2.2e12: an 8 TB index)
// Each descriptor sits alone in a 128-byte line: every resident CTA polls the descriptors of the
// same few hundred predecessor tiles, and packed (8-byte stride) descriptors put all of that
// traffic on a handful of L2 slices (measured: 5x slower with a 320-tile window).  One line per
// descriptor spreads the polls over all slices through the address hash.
constexpr uint64_t kDescStride = 16;  // in u64 words
constexpr uint64_t kStatusAgg = 1ull << 62;
constexpr uint64_t kStatusPrefix = 2ull << 62;
constexpr uint64_t kParityBit = 1ull << 61;
constexpr int kTagShift = 41;
constexpr uint64_t kTagMask = 0xfffffull;
constexpr uint64_t kCountMask = (1ull << kTagShift) - 1;

// ---- cross-GPU exchange over peer-mapped mailboxes (NVLink P2P stores; no collective library) ----------------
// Every rank owns a mailbox in its own HBM: kExRing slots (one per build, epoch % kExRing) of kExMaxWorld rows of
// 8 words {entries under the carry used, end parity, carry used, total separators, epoch, -, -, -}.  A rank POSTS its
// row into the same (slot, row = its rank) of EVERY rank's mailbox (remote stores, then the epoch word after a
// system-scope fence) and WAITS, on its own mailbox only, for the rows of the LOWER ranks: the true carry of shard k is
// the XOR of the lower shards' parities and its base the sum of their true counts, so nothing above k is needed
// before k can go on -- which also means ranks emulated one after another on one GPU never wait on a later launch.
constexpr uint32_t kExRing = 1024;
constexpr uint32_t kExMaxWorld = 16;
constexpr uint32_t kExRowWords = 8;
constexpr size_t kExMailboxBytes = (size_t)kExRing * kExMaxWorld * kExRowWords * sizeof(uint64_t);   // 1 MiB

struct ExchangeArgs {
    uint64_t* const* peers;  // device array [world]: every rank's mailbox as mapped into THIS device; null = no exchange
    uint32_t rank, world;
    uint64_t epoch;          // >= 1, the same on every rank for the same build
    uint64_t timeout_ns;     // bound on the wait for the lower ranks' rows (a rank that never posts is an error, not a hang)
    // out: {0, true carry-in parity, entries of the lower ranks | error << 63, redo flag} -- the carry cell the
    // conditional redo launch reads -- and its pinned host mirror
    uint64_t* out;
    uint64_t* out_host;
};

struct BuildParams {
    const uint8_t* in;       // 16-byte aligned device pointer to the shard's bytes
    uint64_t n;              // bytes
    uint64_t* index;         // output entries (u64, == Rust usize); 16-byte aligned
    uint64_t cap;            // number of u64 slots available at `index`
    uint64_t out_base;       // slot of the first entry produced by the virtual predecessor (1 after the sentinel)
    uint64_t pos_bias;       // added to every emitted byte position (global offset of the shard)
    const uint64_t* carry;   // optional device cell {entries so far, parity}; overrides the two below
    uint32_t carry_parity_only;  // with `carry`: take only the parity from the cell, count = carry_count (streaming ingest:
                                 // every chunk writes its own segment buffer from slot 0)
    uint64_t carry_count;    // entries emitted by earlier launches of the same build
    uint32_t carry_parity;   // quote parity entering byte 0 of `in`
    uint32_t num_tiles;
    uint64_t* desc;          // [num_tiles] look-back descriptors (tagged, never zeroed between launches)
    uint32_t desc_tag;       // this launch's tag
    uint32_t scratch_totals; // total_out / nl_out / hi_out live in the scratch head: the last CTA resets them after use
    uint32_t* ticket;        // dynamic tile counter; zero at launch, reset by the CTA that takes the last ticket
    uint64_t* result;        // {entries emitted through the end of this launch, end parity}
    uint64_t* result_host;   // optional pinned (UVA-mapped) host mirror of `result`: written straight over PCIe, no D2H copy node
    uint32_t write_sentinel; // the CTA of tile 0 writes index[0] = 0 (src/reader.rs:216) instead of a separate memset
    uint64_t* result2;       // optional second copy of `result` in caller-owned device memory
    uint32_t result2_words;  // 2, or 4: {entries, end parity, carry parity used, (total separators via total_out)}
    // optional: every CTA adds the separator count (inside + outside quotes) of its tiles; zeroed by the
    // caller.  With it the entry count under the OTHER carry parity is total - entries (c0 + c1 = total).
    unsigned long long* total_out;
    // multi-GPU: quote parities of all shards as all-gathered on the device; the carry-in parity of
    // this shard is the XOR of shard_par[0 .. shard_rank) (overrides carry_parity when non-null)
    const uint32_t* shard_par;
    uint32_t shard_rank;
    uint64_t* dbg;           // debug timeline (CSVB200_DBG_TIMELINE): 8 words per super-tile, see tools/timeline.py; null normally
    // speculative multi-GPU build: when non-null the launch is a conditional redo and exits at once
    // unless *run_flag != 0 (the carry prediction turned out wrong)
    const uint32_t* run_flag;
    // exchange inside the launch (multi-GPU, see ExchangeArgs): the last CTA to finish its look-back role posts this
    // shard's row to every peer's mailbox and resolves the carry chain of the lower ranks
    ExchangeArgs ex;
    uint32_t* ex_done;       // CTAs whose look-back role is over; zeroed before launch (scratch); needed by ex / validate
    // by-products of the classification (CSVB200_BUILD_VALIDATE): newlines (CR or LF) outside quotes and "any byte
    // >= 0x80", accumulated per CTA into the zeroed scratch words nl_out / hi_out and copied by the last CTA into
    // result[3] / result[2]; nonascii_bitmap has one bit per look-back tile (flag_tile_bytes of input each)
    // the launch was made with programmatic stream serialization right behind predict_carry_kernel: the threads that
    // read the carry cell (the look-back of the first tiles, the epilogue) execute griddepcontrol.wait first, every
    // other thread starts classifying while the predictor still runs
    uint32_t pdl_wait;
    uint32_t validate;
    unsigned long long* nl_out;
    uint32_t* hi_out;
    uint32_t* nonascii_bitmap;
};

// one tile per CTA, plain loads: small inputs and cross-check of the TMA kernel
cudaError_t launch_index_build(const BuildParams& p, cudaStream_t stream);
// persistent warp-specialised TMA pipeline (index_build_tma.cu): the production path for large inputs
cudaError_t launch_index_build_tma(const BuildParams& p, cudaStream_t stream);
bool tma_path_usable(uint64_t n);

// quote parity of a byte range (pass A of the multi-GPU protocol); *out ^= parity
cudaError_t launch_quote_parity(const uint8_t* in, uint64_t n, uint32_t* out, cudaStream_t stream);

// speculative carry (multi-GPU): predict the quote parity entering a shard from the first unambiguous
// quote in its first `window` bytes; cell = {0, predicted parity, 1 if a decisive quote was found}
cudaError_t launch_predict_carry(const uint8_t* in, uint64_t n, uint64_t window, uint64_t* cell, cudaStream_t stream);
// gathered[world][4] = {entries, end parity, carry parity used, total separators} per rank; writes
// cell = {0, true carry of `rank`, -, redo flag (true carry != the one used)} and, when non-null,
// final_out[world][2] = {true entry count, true carry} of every rank
cudaError_t launch_verify_carry(const uint64_t* gathered, uint32_t world, uint32_t rank, uint64_t* cell,
                                uint64_t* final_out, cudaStream_t stream);
// the exchange as a launch of its own (end-to-end pipelines, whose last chunk is not known in advance): posts
// row4 = {entries, end parity, carry used, total separators} (device words) and resolves like the in-kernel form
cudaError_t launch_exchange(const ExchangeArgs& ex, const uint64_t* row4, cudaStream_t stream);

// debug / known-answer exports (K1): per 64-byte block quote and separator words, class bytes
cudaError_t launch_block_masks(const uint8_t* in, uint64_t n, uint64_t* quote_words, uint64_t* sep_words,
                               cudaStream_t stream);
cudaError_t launch_class_bytes(const uint8_t* in, uint64_t n, uint8_t* out, cudaStream_t stream);

// K4 batched lookups. ranges[2*i] = start, ranges[2*i+1] = end; (UINT64_MAX, UINT64_MAX) = None.
struct LookupParams {
    const uint64_t* index;
    uint64_t index_len;
    uint32_t record_cnt;
    uint32_t field_cnt;
    uint32_t row_size;       // jump: field_cnt (+1 for CRLF)
    const uint32_t* rec;
    const uint32_t* fld;     // nullptr => seek_record
    uint64_t nq;
    uint64_t* ranges;
    uint32_t* oob;           // incremented for queries whose index slot is out of bounds (reference would panic)
};
cudaError_t launch_seek(const LookupParams& p, cudaStream_t stream);
// the same over an index that is distributed over several GPUs of one process: segment k holds the global slots
// [base[k], base[k + 1]) and lives in device k's HBM, mapped into the launching device (peer access over NVLink).
// p.index is ignored; p.index_len is the total length.
struct SegmentTable {
    const uint64_t* ptr[kExMaxWorld];
    uint64_t base[kExMaxWorld + 1];
    uint32_t nseg;
};
cudaError_t launch_seek_sharded(const LookupParams& p, const SegmentTable& seg, cudaStream_t stream);

// gather the bytes of resolved ranges into a packed buffer: out[out_off[i] .. out_off[i+1]) = the input bytes
// [start, end); ranges are GLOBAL positions, bytes[0] is global byte pos_bias and n bytes are addressable
cudaError_t launch_gather_bytes(const uint8_t* bytes, uint64_t n, uint64_t pos_bias, const uint64_t* ranges,
                                const uint64_t* out_off, uint64_t nq, uint8_t* out, cudaStream_t stream);
cudaError_t launch_range_lengths(const uint64_t* ranges, uint64_t nq, uint64_t* lens, cudaStream_t stream);

// K5 tape validation (tape.cu): first index slot whose separator class does not fit its place in the record
struct TapeValidateParams {
    const uint64_t* index;
    uint64_t index_len;
    const uint8_t* bytes;    // the shard the index positions refer to
    uint64_t n;
    uint64_t pos_bias;       // global offset of bytes[0] (index positions are global)
    uint64_t jump;
    int crlf;
    uint64_t* first_bad_slot;   // device word, preset to UINT64_MAX; atomicMin
};
cudaError_t launch_tape_validate(const TapeValidateParams& p, cudaStream_t stream);
// out[i] = index[slots[i]] (UINT64_MAX when the slot is past the end)
cudaError_t launch_gather_slots(const uint64_t* index, uint64_t index_len, const uint64_t* slots, uint64_t n,
                                uint64_t* out, cudaStream_t stream);

// K7 ASCII / UTF-8 validation (validate.cu): result[0] (preset UINT64_MAX) <- start of the first ill-formed
// sequence, result[1] (preset 0) <- 1 when any byte is >= 0x80
cudaError_t launch_utf8_validate(const uint8_t* in, uint64_t n, uint64_t* result, cudaStream_t stream);
// the same over the tiles (tile_bytes each) whose bit is set in `bitmap` only: the build kernel flags the tiles that
// hold a byte >= 0x80, every other tile is ASCII and leads (and owes) no multi-byte sequence
cudaError_t launch_utf8_validate_flagged(const uint8_t* in, uint64_t n, const uint32_t* bitmap, uint64_t tile_bytes,
                                         uint64_t* result, cudaStream_t stream);
// bytes per bit of the non-ASCII bitmap for an input of n bytes (depends on the kernel the build picks)
uint64_t build_flag_tile_bytes(bool use_tma);

// K6 column materialisation (materialize.cu)
struct MaterializeParams {
    const uint64_t* index;
    uint64_t index_len;
    const uint8_t* bytes;
    uint64_t n;
    uint64_t pos_bias;
    uint32_t record_cnt, field_cnt, row_size;
    uint32_t field_idx, first_record, nrec;
    uint32_t flags;          // 1 = unquote, 2 = trim
    uint64_t* offsets;       // [nrec + 1] exclusive prefix sums of the value lengths
    uint8_t* out;
    uint64_t out_cap;
    uint64_t* tile_desc;     // look-back descriptors (zeroed), materialize_scratch_bytes(nrec) - 128 bytes
    uint32_t* ticket;        // zeroed
    uint64_t offset_base;    // added to every offset the offsets pass writes (0: offsets start at 0)
};
size_t materialize_scratch_bytes(uint32_t nrec);   // [128 B ticket cell][descriptors]

// Several columns of the same records in ONE sweep: a thread owns a row and walks the requested fields of that row
// (adjacent index slots, adjacent bytes: the sectors one column drags in serve its neighbours), so the input and the
// index cross DRAM once per pass instead of once per column and pass.
constexpr uint32_t kMatMaxCols = 32;
constexpr int kMultiThreads = 256;   // threads per CTA of the multi-column kernels = records per tile
struct MaterializeMultiParams {
    const uint64_t* index;
    uint64_t index_len;
    const uint8_t* bytes;
    uint64_t n;
    uint64_t pos_bias;
    uint32_t record_cnt, field_cnt, row_size;
    uint32_t first_record, nrec;
    uint32_t flags;
    uint32_t ncols;
    uint32_t field_idx[kMatMaxCols];
    uint64_t* offsets[kMatMaxCols];   // per column [nrec + 1]
    uint8_t* out[kMatMaxCols];        // per column packed values (write pass)
    uint64_t out_cap[kMatMaxCols];
    uint64_t* tile_desc;              // [ncols][tiles] look-back descriptors (zeroed)
    uint32_t* ticket;                 // zeroed
    uint32_t tiles;
    uint64_t offset_base[kMatMaxCols];   // per column, added to every offset the offsets pass writes
};
size_t materialize_multi_scratch_bytes(uint32_t nrec, uint32_t ncols);
cudaError_t launch_materialize_multi_offsets(const MaterializeMultiParams& p, cudaStream_t stream);
cudaError_t launch_materialize_multi_write(const MaterializeMultiParams& p, cudaStream_t stream);
cudaError_t launch_materialize_offsets(const MaterializeParams& p, cudaStream_t stream);
cudaError_t launch_materialize_write(const MaterializeParams& p, cudaStream_t stream);

}  // namespace csvb200
