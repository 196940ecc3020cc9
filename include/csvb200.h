/*
 * csvb200.h -- C ABI of libcsvb200: the B200 (sm_100a) drop-in for csv-simd's hot path
 *
 *     csv bytes -> in-memory structural index -> (record #) -> record -> (record, field #) -> field
 *
 * The reference (EdmundsEcho/csv-simd, a Rust crate) has no FFI; the boundary is its
 * public Rust API.  Every entry point below names the reference item it replaces
 * (file:line under the reference tree).  INTEGRATION.md shows the `extern "C"` block
 * and the replacement bodies of reader.rs / record_source.rs that bind these symbols.
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns a csvb200_status (0 = OK)
 *     and never unwinds across the ABI; csvb200_last_error(ctx) gives the detail string.
 *   - one csvb200_ctx per GPU and per host thread at a time (process-per-GPU model);
 *     built indexes are immutable and may be queried concurrently.
 *   - the index is an array of native-endian u64 byte offsets, ABI-identical to the
 *     reference's StructureIndex(Vec<CodeUnitPos>) (src/stage1.rs:61,67):
 *       index[0] = 0 (sentinel, src/reader.rs:216), then every ',', CR or LF byte that
 *       lies outside double-quoted regions, in file order; CR and LF are separate entries.
 *   - there is NO CPU fallback: every compute entry point needs a CUDA device.
 */
#ifndef CSVB200_H
#define CSVB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSVB200_VERSION 100 /* 0.1.0 */

typedef enum csvb200_status {
    CSVB200_OK = 0,
    CSVB200_ERR_INVALID_ARG = 1,
    CSVB200_ERR_INVALID_STATE = 2,      /* StructureError::InvalidState      (src/error.rs:17-18) */
    CSVB200_ERR_INVALID_CSV_FORMAT = 3, /* StructureError::InvalidCsvFormat  (src/error.rs:19-20) */
    CSVB200_ERR_MISSING_VALUE = 4,      /* StructureError::MissingValue      (src/error.rs:15-16) */
    CSVB200_ERR_IO = 5,                 /* StructureError::Io                (src/error.rs:11-12) */
    CSVB200_ERR_CUDA = 6,
    CSVB200_ERR_OOM = 7,
    CSVB200_ERR_INPUT_TOO_SMALL = 8,    /* n < 64: the reference panics (src/reader.rs:220-229, src/avx/stage1.rs:45-48) */
    CSVB200_ERR_CAPACITY = 9,
    CSVB200_ERR_OUT_OF_BOUNDS = 10,     /* a lookup slot past the index end: the reference panics on the Vec bounds check */
    CSVB200_ERR_EXCHANGE = 11           /* a peer GPU never posted its row (timeout) or lapped the mailbox ring */
} csvb200_status;

typedef struct csvb200_ctx csvb200_ctx;
typedef struct csvb200_index csvb200_index;

/* (start, end) byte range of a record or field in the input; both UINT64_MAX = None. */
typedef struct csvb200_range {
    uint64_t start;
    uint64_t end;
} csvb200_range;

/* build flags */
#define CSVB200_BUILD_DEFAULT 0u
#define CSVB200_BUILD_KEEP_BYTES 1u   /* keep the device copy of the input for csvb200_gather_fields */
#define CSVB200_BUILD_STRICT_MIN64 2u /* mirror the reference's n < 64 panic as CSVB200_ERR_INPUT_TOO_SMALL */
#define CSVB200_BUILD_VALIDATE 4u     /* by-products of the same launch: is_ascii, newlines outside quotes, non-ASCII tile map */

int csvb200_version(void);
const char* csvb200_status_string(int status);

/* ---- context ----------------------------------------------------------------------------- */
/* Creates the per-GPU context: stream, look-back scratch, pinned result cells.  `device` is a
 * CUDA ordinal.  Fails with CSVB200_ERR_CUDA when no usable device exists (no CPU fallback). */
int csvb200_ctx_create(int device, csvb200_ctx** out);
void csvb200_ctx_destroy(csvb200_ctx* ctx);
const char* csvb200_last_error(const csvb200_ctx* ctx);
/* Run all work of this context on an externally owned cudaStream_t (e.g. the caller's current
 * stream, so the caller's CUDA events bracket the kernels).  NULL restores the private stream;
 * pass cudaStreamLegacy ((cudaStream_t)0x1) to run on the legacy default stream.
 * The private stream is NON-BLOCKING: it is not ordered against the legacy default stream or any
 * other stream of the caller.  Device buffers handed to a *_device entry point must be complete
 * (and output buffers free of pending writes) before the call: synchronise the producing stream,
 * or make it this context's stream with this function. */
int csvb200_ctx_set_stream(csvb200_ctx* ctx, void* cuda_stream);
/* Initial index capacity = n / ratio_den * ratio_num + 4096 entries (default 1/3); an index that
 * overflows it is transparently rebuilt with the exact size. */
int csvb200_ctx_set_reserve(csvb200_ctx* ctx, uint32_t ratio_num, uint32_t ratio_den);
/* Device time (ms, CUDA events on the context's stream) of the kernels of the last build call. */
int csvb200_ctx_last_build_ms(csvb200_ctx* ctx, float* ms);
/* Number of kernel launches issued by this context so far. */
uint64_t csvb200_ctx_launch_count(const csvb200_ctx* ctx);

/* pinned host memory for staging (cudaHostAlloc / cudaFreeHost) */
int csvb200_host_alloc(size_t bytes, void** out);
int csvb200_host_free(void* p);
/* Pin memory the caller already owns (a Vec<usize> it reuses, an Mmap) so that the end-to-end calls DMA it in
 * place instead of staging it through host copies (cudaHostRegister; read_only != 0 for a PROT_READ mapping).
 * Costs ~25-30 ms per GiB, so it pays for buffers used more than once.  The range must stay mapped until
 * csvb200_host_unregister(p) (same pointer).  CSVB200_ERR_INVALID_ARG: already registered / not registrable. */
int csvb200_host_register(void* p, size_t bytes, int read_only);
int csvb200_host_unregister(void* p);

/* ---- csv -> index : replaces reader::read (src/reader.rs:150-306) -------------------------- */
/* Host bytes -> device-resident index.  Copies the input to the GPU in chunks
 * (cudaMemcpyAsync from pinned memory; pageable input is staged through a pinned ring),
 * runs the fused classify / quote-scan / compaction kernel, leaves the index in HBM. */
int csvb200_index_build(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint32_t flags,
                        csvb200_index** out);
/* Same, input already in device memory (16-byte aligned).  Asynchronous: returns after
 * enqueueing; csvb200_index_len / copy_out / sync wait for completion. */
int csvb200_index_build_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t flags,
                               csvb200_index** out);
/* Host bytes -> host index in one call, H2D and D2H overlapped chunk by chunk (the end-to-end
 * path the reference's callers see: &[u8] in, Vec<usize> out).  dst_cap in entries; *len_out
 * receives the entry count; CSVB200_ERR_CAPACITY (with *len_out set) if dst is too small. */
int csvb200_index_build_to_host(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* dst,
                                size_t dst_cap, size_t* len_out);

/* ---- streaming ingest (reference README.md:23 "Decisions" 3; src/lib.rs:64-65 maps the whole file) -- */
/* csv of any size -> index in bounded device and pinned memory: the input is pulled in chunks into a
 * pinned ring, uploaded, indexed by launches chained through a device-resident quote-parity cell, and
 * every finished index segment is handed to the sink in order while later chunks are still going up.
 *   read : fill dst (pinned) with up to cap of the NEXT input bytes, return the count; 0 = end of input
 *   sink : consume `count` consecutive index entries starting at global slot first_slot (entries are
 *          global byte offsets; the sentinel index[0] = 0 arrives first); the pointer is only valid
 *          during the call; a non-zero return aborts the build with CSVB200_ERR_IO
 * chunk_bytes = 0 selects the default (16 MiB). */
typedef size_t (*csvb200_read_fn)(void* user, uint8_t* dst, size_t cap);
typedef int (*csvb200_sink_fn)(void* user, const uint64_t* entries, size_t count, uint64_t first_slot);
typedef struct csvb200_stream_stats {
    uint64_t bytes;    /* input bytes consumed */
    uint64_t entries;  /* index entries produced, sentinel included */
    double seconds;    /* wall time of the call */
    uint32_t chunks;
    int end_parity;    /* quote parity after the last byte */
} csvb200_stream_stats;
int csvb200_index_build_stream(csvb200_ctx* ctx, csvb200_read_fn read, void* read_user, csvb200_sink_fn sink,
                               void* sink_user, size_t chunk_bytes, csvb200_stream_stats* stats);
/* csv_simd::create's data path for a file (src/lib.rs:61-74: File::open -> Mmap::map -> reader::read):
 * a pool of threads pread()s the file straight into the pinned ring; the index lands in dst (DMA'd in
 * place when dst is pinned, else copied out of the pinned ring by the same pool).  *len_out receives
 * the entry count even when dst_cap is too small (CSVB200_ERR_CAPACITY); a file that cannot be opened
 * or read is CSVB200_ERR_IO (StructureError::Io). */
int csvb200_index_build_file(csvb200_ctx* ctx, const char* path, uint64_t* dst, size_t dst_cap, size_t* len_out,
                             csvb200_stream_stats* stats);

/* ---- sharded build (multi-GPU, SURVEY 8e / README.md:24 "splitting work without first knowing
 * record breaks") --------------------------------------------------------------------------- */
/* Pass A: quote parity (0/1) of a device-resident shard -- the only thing that must cross GPUs
 * before a shard can be indexed. */
int csvb200_shard_quote_parity(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t* parity_out);
/* Pass B: index a shard that is entered with quote parity `carry_parity` and starts at global
 * byte offset `global_offset`; the sentinel entry is emitted only when emit_sentinel != 0
 * (rank 0).  Positions are global. */
int csvb200_index_build_shard_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t carry_parity,
                                     uint64_t global_offset, int emit_sentinel, csvb200_index** out);

/* Stream-ordered forms of the two passes: no host synchronisation between pass A, the collective and
 * pass B.  Pass A writes the parity to a device cell; after the caller has all-gathered the cells
 * into d_shard_parities[world] (NCCL, same stream order), pass B derives its carry-in parity on the
 * device as XOR of d_shard_parities[0 .. shard_rank).  d_result_out (optional, 2 x u64 device words)
 * receives {entries emitted by this shard excluding the sentinel, end parity} for a device-side
 * all-gather of the counts. */
int csvb200_shard_quote_parity_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t* d_parity_out);
int csvb200_index_build_shard_device_ex(csvb200_ctx* ctx, const void* dev_bytes, size_t n,
                                        const uint32_t* d_shard_parities, uint32_t shard_rank, uint64_t global_offset,
                                        int emit_sentinel, uint64_t* d_result_out, csvb200_index** out);

/* Speculative form: no pass A in the common case, ONE all-gather per build.  The carry-in parity of
 * the shard is PREDICTED from the first unambiguous quote in its first predict_window bytes (0 = 64 KiB;
 * rank 0 is known to start outside quotes), the shard is indexed at once with that guess, and
 * d_result_out (4 x u64 device words) receives {entries emitted excluding the sentinel, end parity,
 * carry parity used, total separator count of the shard}.  After the caller has all-gathered those
 * 32 bytes per rank into d_gathered[world][4] (NCCL, same stream order), csvb200_index_shard_verify
 * derives the true carry of every shard on the device and re-indexes this shard only if its guess was
 * wrong (the conditional launch exits immediately otherwise), so the result is exact for ANY input.
 * Because flipping a shard's carry swaps its inside / outside separators, every rank also derives every
 * shard's true entry count without a second exchange: d_final_out (optional, world x 2 u64 device
 * words) receives {entry count excluding the sentinel, carry-in parity} per rank.  Nothing here
 * synchronises with the host. */
int csvb200_index_build_shard_speculative(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t shard_rank,
                                          uint64_t global_offset, int emit_sentinel, uint64_t predict_window,
                                          uint64_t* d_result_out, csvb200_index** out);
int csvb200_index_shard_verify(csvb200_index* idx, const uint64_t* d_gathered, uint32_t world, uint64_t* d_final_out);
/* diagnostics (synchronises): whether the misprediction rebuild ran, and the true carry-in parity */
int csvb200_index_shard_redone(csvb200_index* idx, int* redone, int* carry_parity);

/* End-to-end form of the speculative protocol: this rank's shard in HOST memory -> this rank's segment
 * of the index in HOST memory, uploads / launches / downloads overlapped chunk by chunk exactly like
 * csvb200_index_build_to_host.  The segment is produced under the predicted carry and d_result_out
 * (4 x u64 device words, as above) is ready for the all-gather when the call returns; after the
 * all-gather csvb200_shard_job_verify derives the true carries and counts (d_final_out, optional,
 * world x 2 u64 device words) and, only if this shard's guess was wrong, re-indexes it from the device
 * copy it kept and overwrites dst (*len_out updated, *redone = 1). */
typedef struct csvb200_shard_job csvb200_shard_job;
int csvb200_shard_build_to_host(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint32_t shard_rank,
                                uint64_t global_offset, int emit_sentinel, uint64_t* dst, size_t dst_cap, size_t* len_out,
                                uint64_t* d_result_out, csvb200_shard_job** job_out);
int csvb200_shard_job_verify(csvb200_shard_job* job, const uint64_t* d_gathered, uint32_t world, uint64_t* d_final_out,
                             size_t* len_out, int* redone);
void csvb200_shard_job_free(csvb200_shard_job* job);

/* ---- the same protocol without a collective library: peer-mapped mailboxes over NVLink -----------------------
 * (north_star: "one tiny allgather over NVLink exchanges those parity bits and counts"; README.md:24.)  Every rank
 * owns a 1 MiB mailbox in its own HBM.  A build posts its 32-byte row {entries, end parity, carry used, separator
 * total} into the same slot of EVERY rank's mailbox with plain remote stores from inside the index-build launch (the
 * last CTA to finish does it, while others still compact), then waits -- on its own memory -- for the rows of the LOWER
 * ranks only, derives its true carry-in, the entries before its segment and whether its guess was wrong, and leaves
 * them where the conditional redo launch and the host find them.  No NCCL, no host round trip, no extra launch; a
 * rank that never posts is reported as CSVB200_ERR_EXCHANGE after a timeout (CSVB200_EXCHANGE_TIMEOUT_MS, default
 * 5000) instead of hanging the GPU.  Builds through an exchange are COLLECTIVE: every rank issues them in the same
 * order.  At most 16 ranks; at most 1024 builds may be in flight ahead of the slowest rank (detected, not silent).
 *
 * Wiring: create one endpoint per context, hand every rank's 64-byte handle to every other rank by any means (the
 * Python layer uses torch.distributed, a Rust caller its own channel) and connect.  Processes on one node map each
 * other's mailboxes through CUDA IPC; contexts of ONE process (one per device) connect directly with peer access. */
typedef struct csvb200_exchange csvb200_exchange;
#define CSVB200_EXCHANGE_HANDLE_BYTES 64
#define CSVB200_EXCHANGE_MAX_WORLD 16
int csvb200_exchange_create(csvb200_ctx* ctx, uint32_t rank, uint32_t world, csvb200_exchange** out);
int csvb200_exchange_handle(csvb200_exchange* ex, uint8_t out[CSVB200_EXCHANGE_HANDLE_BYTES]);
/* handles = world x 64 bytes in rank order (this rank's own slot is ignored) */
int csvb200_exchange_connect(csvb200_exchange* ex, const uint8_t* handles);
/* all = the endpoints of every rank of this process, in rank order; connects every one of them */
int csvb200_exchange_connect_local(csvb200_exchange* const* all, uint32_t world);
void csvb200_exchange_destroy(csvb200_exchange* ex);

/* Index this rank's device-resident shard [global_offset, global_offset + n): prediction, build, exchange and the
 * conditional re-index are all enqueued on the context's stream; nothing waits on the host.  Rank 0 emits the
 * sentinel.  predict_window as above. */
int csvb200_index_build_shard_exchange(csvb200_ctx* ctx, csvb200_exchange* ex, const void* dev_bytes, size_t n,
                                       uint64_t global_offset, uint64_t predict_window, csvb200_index** out);
typedef struct csvb200_shard_info {
    uint64_t base;      /* global slot of this rank's first entry (rank 0: 0, the sentinel) */
    uint64_t entries;   /* entries in this rank's segment (rank 0 incl. the sentinel) */
    uint64_t epoch;
    uint32_t carry_in;  /* true quote parity entering the shard */
    uint32_t redone;    /* the guess was wrong and the shard was re-indexed */
    uint32_t rank, world;
} csvb200_shard_info;
/* synchronises with the build */
int csvb200_index_shard_info(csvb200_index* idx, csvb200_shard_info* out);
/* Waits (host side, bounded) until EVERY rank's row of that build has arrived and derives every rank's true entry
 * count (rank 0 incl. the sentinel) and carry-in: counts[world], carries[world] (either may be NULL). */
int csvb200_exchange_counts(csvb200_exchange* ex, csvb200_index* idx, uint64_t* counts, uint32_t* carries);

/* End-to-end form: this rank's shard in HOST memory -> this rank's index segment in HOST memory (chunked uploads,
 * chained launches, overlapped downloads under the predicted carry, exchange, re-index from the device copy only if
 * the guess was wrong).  Synchronous.  counts / carries as above (optional: they make the call wait for all ranks). */
int csvb200_shard_build_to_host_exchange(csvb200_ctx* ctx, csvb200_exchange* ex, const uint8_t* host_bytes, size_t n,
                                         uint64_t global_offset, uint64_t* dst, size_t dst_cap, size_t* len_out,
                                         csvb200_shard_info* info, uint64_t* counts, uint32_t* carries);

/* ---- all GPUs of one process behind one call (what makes reader::read, src/reader.rs:150, drop-in at 8 GPUs:
 * the caller of src/lib.rs:61-74 hands over ONE byte slice and gets ONE Vec<usize> back) ------------------------ */
typedef struct csvb200_multi csvb200_multi;
/* one context + exchange endpoint per listed device (a device may be listed twice: its shards then run one after
 * another, which is how the protocol is exercised on a single GPU) */
int csvb200_multi_create(const int* devices, int ndev, csvb200_multi** out);
void csvb200_multi_destroy(csvb200_multi* m);
const char* csvb200_multi_last_error(const csvb200_multi* m);
int csvb200_multi_device_count(const csvb200_multi* m);
/* Cuts host_bytes into ndev contiguous shards at arbitrary (unaligned) offsets -- cuts[ndev+1] if given, else
 * k * n / ndev + 37 k + 13 -- uploads and indexes them concurrently (one host thread per device), exchanges carries
 * and bases over peer memory, and writes ONE contiguous index into dst: exactly reader::read's output. */
int csvb200_multi_index_build_to_host(csvb200_multi* m, const uint8_t* host_bytes, size_t n, const size_t* cuts,
                                      uint64_t* dst, size_t dst_cap, size_t* len_out);
/* The same build, leaving the index DISTRIBUTED over the devices (segment k in device k's HBM, global byte positions)
 * for lookups: SURVEY 8e "the index stays distributed; lookups route the slot to the owning rank".  Here the routing
 * is done by the memory system: every device has every segment mapped (peer access), a batch of (record, field)
 * queries is split evenly over the devices and each lookup kernel reads index[s], index[s + 1] from whichever GPU owns
 * them -- 16 bytes over NVLink per remote query, nothing is gathered or replicated.  RecordSource semantics as
 * csvb200_seek_fields (src/record_source.rs:104-140). */
typedef struct csvb200_multi_index csvb200_multi_index;
int csvb200_multi_index_build(csvb200_multi* m, const uint8_t* host_bytes, size_t n, const size_t* cuts,
                              csvb200_multi_index** out);
void csvb200_multi_index_free(csvb200_multi_index* mi);
size_t csvb200_multi_index_len(const csvb200_multi_index* mi);
int csvb200_multi_index_segment(const csvb200_multi_index* mi, int k, uint64_t* base, uint64_t* entries, int* device);
int csvb200_multi_index_copy_out(csvb200_multi_index* mi, uint64_t* dst, size_t dst_cap);
int csvb200_multi_tape_init(csvb200_multi_index* mi, uint32_t field_cnt, int crlf, uint32_t* record_cnt, uint64_t* jump);
int csvb200_multi_seek_fields(csvb200_multi_index* mi, const uint32_t* rec, const uint32_t* fld, size_t nq, csvb200_range* out);
int csvb200_multi_seek_records(csvb200_multi_index* mi, const uint32_t* rec, size_t nq, csvb200_range* out);
/* device arrays on device number k of the list; asynchronous on that device's stream (csvb200_multi_stream) */
int csvb200_multi_seek_fields_device(csvb200_multi_index* mi, int k, const uint32_t* d_rec, const uint32_t* d_fld, size_t nq,
                                     csvb200_range* d_out);
void* csvb200_multi_stream(csvb200_multi* m, int k);
/* csvb200_materialize_columns over the distributed index, with the same results byte for byte and the same status
 * codes, into host arrays; before csvb200_multi_tape_init it is CSVB200_ERR_INVALID_STATE.  Every device materialises
 * the records whose index slots all lie in its segment, from its own shard of the bytes.  A record whose slots run
 * over a cut (at most one per cut) has its slots and bytes copied to one device and goes through the same kernels
 * there.  Offsets and values go straight from every device to their place in the caller's arrays.  An index of more
 * than 2^32 entries is CSVB200_ERR_INVALID_ARG: the kernels address slots in u32, as the reference does. */
int csvb200_multi_materialize_columns(csvb200_multi_index* mi, const uint32_t* fields, uint32_t ncols,
                                      uint32_t first_record, uint32_t nrec, uint32_t flags,
                                      uint64_t* const* out_offsets, uint8_t* const* outs,
                                      const size_t* out_caps, size_t* out_lens);

typedef struct csvb200_multi_stats {
    double seconds, upload_seconds, download_seconds;
    uint64_t entries;
    uint32_t redone_mask;     /* bit k: shard k was re-indexed */
    uint32_t carry_mask;      /* bit k: shard k starts inside a quoted field */
} csvb200_multi_stats;
int csvb200_multi_last_stats(const csvb200_multi* m, csvb200_multi_stats* out);

/* ---- index object: StructureIndex (src/stage1.rs:61) --------------------------------------- */
/* Wrap `len` entries that already sit in device memory (e.g. the segments of a sharded build gathered
 * into one array) as an index object, so the Tape / seek / validate / materialise calls run on them.
 * The memory stays the caller's (never freed by csvb200_index_free) and must outlive the object;
 * d_bytes (optional) is the device copy of the input the positions refer to. */
int csvb200_index_wrap_device(csvb200_ctx* ctx, const uint64_t* d_entries, size_t len, size_t input_bytes,
                              const void* d_bytes, csvb200_index** out);
int csvb200_index_sync(csvb200_index* idx);
size_t csvb200_index_len(csvb200_index* idx);          /* entries incl. the sentinel if emitted */
int csvb200_index_end_parity(csvb200_index* idx);      /* quote parity after the last byte */
const uint64_t* csvb200_index_device_ptr(csvb200_index* idx);
int csvb200_index_copy_out(csvb200_index* idx, uint64_t* dst, size_t dst_cap); /* fills a caller Vec<usize> */
void csvb200_index_free(csvb200_index* idx);

/* ---- Tape metadata: TapeCore::init (src/tape.rs:315-347) ----------------------------------- */
/* jump = field_cnt (+1 for CRLF); record_cnt = (len-1)/jump; (len-1)%jump != 0 ->
 * CSVB200_ERR_INVALID_CSV_FORMAT.  Must precede the seek calls (else CSVB200_ERR_INVALID_STATE,
 * as TapeCore::record_jump_size, src/tape.rs:200-201). */
int csvb200_tape_init(csvb200_index* idx, uint32_t field_cnt, int crlf, uint32_t* record_cnt, uint64_t* jump);

/* Device-side validation of what the seeks assume (beyond the reference, which only tests
 * (len-1) % jump): entry s >= 1 is the k-th separator of its record, k = (s-1) % jump, and must be
 * ',' for the field separators and the line end (CR or LF; CR then the adjacent LF for CRLF files) in
 * the last slot(s).  Reports the first slot that is not, i.e. the first ragged / malformed record.
 * Needs the input bytes (CSVB200_BUILD_KEEP_BYTES, or a device-built index whose input is still alive). */
typedef struct csvb200_tape_report {
    uint64_t index_len;
    uint64_t jump;
    uint64_t problem;          /* (len-1) % jump, src/tape.rs:327 */
    uint64_t first_bad_slot;   /* UINT64_MAX: every entry has the class its slot requires */
    uint64_t first_bad_record; /* row (0 = header) containing it; the trailing partial row when only problem != 0 */
    uint64_t first_bad_pos;    /* byte offset of the offending separator */
    uint32_t record_cnt;       /* (len-1) / jump, src/tape.rs:323-325 */
    uint32_t ok;               /* first_bad_slot == UINT64_MAX && problem == 0 */
} csvb200_tape_report;
int csvb200_tape_validate(csvb200_index* idx, uint32_t field_cnt, int crlf, csvb200_tape_report* out);

/* Tape::chunks(num) (src/tape.rs:95-140) over boundaries(record_cnt, num) (src/tape.rs:385-428): slot
 * ranges of `num` near-equal runs of rows (chunk 0 skips the header row), plus the byte range each run
 * occupies in the input ([byte_start, byte_end), through its last line end) for downstream consumers.
 * record_cnt == 0 or num == 0 -> CSVB200_ERR_INVALID_STATE; fewer rows than chunks -> one chunk. */
typedef struct csvb200_chunk {
    uint64_t start;      /* KeyToPos of the chunk's first row (slot of the separator that precedes it) */
    uint64_t end;        /* KeyToPos one row past its last row */
    uint64_t byte_start; /* index[start] + 1 */
    uint64_t byte_end;   /* index[end] + 1 */
    uint32_t record_cnt;
    uint8_t id;
} csvb200_chunk;
int csvb200_tape_chunks(csvb200_index* idx, uint8_t num, csvb200_chunk* out, size_t out_cap, size_t* n_out);

/* ---- lookups: RecordSource (src/record_source.rs:70-140) ----------------------------------- */
/* scalar: *found = 0 means Ok(None) */
int csvb200_seek_record(csvb200_index* idx, uint32_t record_idx, csvb200_range* out, int* found);
int csvb200_seek_field(csvb200_index* idx, uint32_t record_idx, uint32_t field_idx, csvb200_range* out, int* found);
/* batched (K4), host arrays in / out */
int csvb200_seek_records(csvb200_index* idx, const uint32_t* rec, size_t nq, csvb200_range* out);
int csvb200_seek_fields(csvb200_index* idx, const uint32_t* rec, const uint32_t* fld, size_t nq, csvb200_range* out);
/* batched, device arrays in / out, asynchronous on the context's stream */
int csvb200_seek_fields_device(csvb200_index* idx, const uint32_t* d_rec, const uint32_t* d_fld, size_t nq,
                               csvb200_range* d_out);
int csvb200_seek_records_device(csvb200_index* idx, const uint32_t* d_rec, size_t nq, csvb200_range* d_out);
/* materialise the field bytes of a batch (needs CSVB200_BUILD_KEEP_BYTES): out_offsets[nq+1] are
 * exclusive prefix sums of the lengths, out receives the packed bytes (out_cap bytes). */
int csvb200_gather_fields(csvb200_index* idx, const uint32_t* rec, const uint32_t* fld, size_t nq,
                          uint64_t* out_offsets, uint8_t* out, size_t out_cap);

/* ---- column materialisation (beyond the reference: seek_field returns the RAW slice incl. quotes and
 * padding, src/record_source.rs:135-139) ----------------------------------------------------------- */
/* The values of field `field_idx` of records [first_record, first_record + nrec) (numbered as in
 * seek_field: 0 = first row after the header), packed back to back; out_offsets[nrec + 1] are the
 * exclusive prefix sums of their lengths.  A record seek_field reports as None contributes an empty
 * value.  flags: TRIM strips ASCII space / tab at both ends, then UNQUOTE strips the outer quotes when
 * both are present and turns every "" into ".  Needs the input bytes (CSVB200_BUILD_KEEP_BYTES).
 * Host form: *out_len receives the total; CSVB200_ERR_CAPACITY (offsets and *out_len valid) when
 * out_cap is too small.  Device form: asynchronous on the context's stream, d_out may be NULL to get
 * the offsets only; values that would end past out_cap are skipped. */
#define CSVB200_FIELD_RAW 0u
#define CSVB200_FIELD_UNQUOTE 1u
#define CSVB200_FIELD_TRIM 2u
int csvb200_materialize_column(csvb200_index* idx, uint32_t field_idx, uint32_t first_record, uint32_t nrec,
                               uint32_t flags, uint64_t* out_offsets, uint8_t* out, size_t out_cap, size_t* out_len);
int csvb200_materialize_column_device(csvb200_index* idx, uint32_t field_idx, uint32_t first_record, uint32_t nrec,
                                      uint32_t flags, uint64_t* d_offsets, uint8_t* d_out, size_t out_cap);

/* Several columns of the same records in ONE sweep per pass (ncols <= 32): a device thread owns a row and walks its
 * requested fields, whose index slots and bytes sit next to each other, so the input and the index cross DRAM once
 * per pass instead of once per column and pass (a single column of a row-major file touches one 32-byte sector of
 * every row: ~14 x more traffic than the bytes it returns).  Arrays of ncols pointers / capacities; semantics per
 * column exactly as csvb200_materialize_column. */
int csvb200_materialize_columns(csvb200_index* idx, const uint32_t* fields, uint32_t ncols, uint32_t first_record,
                                uint32_t nrec, uint32_t flags, uint64_t* const* out_offsets, uint8_t* const* outs,
                                const size_t* out_caps, size_t* out_lens);
int csvb200_materialize_columns_device(csvb200_index* idx, const uint32_t* fields, uint32_t ncols, uint32_t first_record,
                                       uint32_t nrec, uint32_t flags, uint64_t* const* d_offsets, uint8_t* const* d_outs,
                                       const size_t* out_caps);

/* ---- input validation (the reference's is_ascii, src/reader.rs:26-132, and its dead UTF-8 checker,
 * src/avx/utf8check.rs; seek_record builds &str unchecked, src/record_source.rs:97-101) ----------- */
/* One pass over the bytes: *is_ascii = no byte >= 0x80 (is_ascii's answer); *valid_up_to = what
 * core::str::from_utf8 reports, the start of the first ill-formed UTF-8 sequence, UINT64_MAX when the
 * input is well-formed.  Device form: asynchronous, d_result = {valid_up_to, 1 if any byte >= 0x80}. */
int csvb200_validate_utf8(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* valid_up_to, int* is_ascii);
int csvb200_validate_utf8_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint64_t* d_result);

/* Fused form (CSVB200_BUILD_VALIDATE on csvb200_index_build / _device): the classification already holds bit 7 of every
 * byte and the CR / LF class, so the build launch itself reports is_ascii (src/reader.rs:26-132) and the number of
 * CR / LF bytes outside quotes (= record terminators; rows for LF files, 2 x rows for CRLF files), and marks the
 * 64 KiB tiles that hold a byte >= 0x80.  csvb200_index_validate_utf8 then reads ONLY the marked tiles (nothing at all
 * for ASCII input) and returns what core::str::from_utf8 would: needs the input bytes (KEEP_BYTES / device build). */
int csvb200_index_validation(csvb200_index* idx, int* is_ascii, uint64_t* newlines_outside_quotes);
int csvb200_index_validate_utf8(csvb200_index* idx, uint64_t* valid_up_to);

/* ---- on-disk index: 64-byte little-endian header {"CSVB2IDX", version 1, flags, input bytes, entries,
 * field_cnt, record_cnt, jump, end parity, wrapping sum of the entries} + the u64 entries ------------ */
int csvb200_index_save(csvb200_index* idx, const char* path);
/* The loaded index supports the Tape / seek calls (metadata restored when it was saved after
 * csvb200_tape_init); calls that need the input bytes report CSVB200_ERR_INVALID_STATE.  A file with a
 * bad magic, size or checksum is CSVB200_ERR_INVALID_CSV_FORMAT; an unreadable one CSVB200_ERR_IO. */
int csvb200_index_load(csvb200_ctx* ctx, const char* path, csvb200_index** out);

/* ---- K1 known-answer exports (debug) -------------------------------------------------------- */
/* per 64-byte block: quote_bits / all_struct as get_struct_positions(16 | 3) (src/avx/stage1.rs:392,394) */
int csvb200_block_masks(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* quote_words,
                        uint64_t* sep_words);
/* class byte per input byte: structure::run (src/structure.rs:10-58) */
int csvb200_class_bytes(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif /* CSVB200_H */
