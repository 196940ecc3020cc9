// csv_simd.hpp -- C++17 host-side mirror of the csv-simd crate's public API for the hot path,
// sitting on the C ABI of libcsvb200 (include/csvb200.h).  Same names, argument meaning and error
// behaviour as the Rust items it stands in for (there is no Rust toolchain in the build image):
//
//   csv_simd::create(filename) -> Tape                 src/lib.rs:61-74
//   reader::read(mmap) -> StructureIndex               src/reader.rs:150-306   (GPU: csvb200_index_build)
//   Header::make(mmap)            [Header::new]        src/tape.rs:226-273
//   TapeCore::create / init, Tape::from_core           src/tape.rs:303-347, 83-94
//   Tape::chunks(num), boundaries(task, jobs)          src/tape.rs:95-140, 385-428
//   RecordSource::seek_record / seek_field             src/record_source.rs:70-140
//   StructureError {Io, MissingValue, InvalidState, InvalidCsvFormat}   src/error.rs:9-21
//
// Only O(first line) / O(1) metadata work happens on the host; the index build and the batched
// lookups run on the GPU.  There is no CPU implementation of the index build here.
#pragma once
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cerrno>
#include <cstdint>
#include <cstring>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <string_view>
#include <utility>
#include <vector>

#include "../../../include/csvb200.h"

namespace csv_simd {

// ---- src/error.rs:9-21 ---------------------------------------------------------------------
enum class ErrorKind { Io, MissingValue, InvalidState, InvalidCsvFormat, ReferencePanic, Gpu };

struct StructureError : std::runtime_error {
    ErrorKind kind;
    StructureError(ErrorKind k, const std::string& what) : std::runtime_error(what), kind(k) {}
    static StructureError invalid_state() { return {ErrorKind::InvalidState, "Invalid state"}; }
    static StructureError missing_value() { return {ErrorKind::MissingValue, "Missing a value"}; }
    static StructureError invalid_csv_format()
    {
        return {ErrorKind::InvalidCsvFormat, "Unsupported csv structure: likely variable number of fields"};
    }
};

inline void check(int rc, csvb200_ctx* ctx)
{
    if (rc == CSVB200_OK) return;
    const std::string detail = ctx ? csvb200_last_error(ctx) : csvb200_status_string(rc);
    switch (rc) {
    case CSVB200_ERR_INVALID_STATE: throw StructureError::invalid_state();
    case CSVB200_ERR_INVALID_CSV_FORMAT: throw StructureError::invalid_csv_format();
    case CSVB200_ERR_MISSING_VALUE: throw StructureError::missing_value();
    case CSVB200_ERR_IO: throw StructureError(ErrorKind::Io, detail);
    case CSVB200_ERR_INPUT_TOO_SMALL:
    case CSVB200_ERR_OUT_OF_BOUNDS: throw StructureError(ErrorKind::ReferencePanic, detail);
    default: throw StructureError(ErrorKind::Gpu, detail);
    }
}

// ---- memmap::Mmap (src/lib.rs:64-65) ----------------------------------------------------------
class Mmap {
public:
    static Mmap map(const std::string& path)
    {
        const int fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) throw StructureError(ErrorKind::Io, path + ": " + std::strerror(errno));  // File::open(..)?
        struct stat st {};
        if (::fstat(fd, &st) != 0) {
            const int e = errno;
            ::close(fd);
            throw StructureError(ErrorKind::Io, path + ": " + std::strerror(e));
        }
        Mmap m;
        m.len_ = static_cast<size_t>(st.st_size);
        if (m.len_ > 0) {
            void* p = ::mmap(nullptr, m.len_, PROT_READ, MAP_PRIVATE, fd, 0);
            if (p == MAP_FAILED) {
                const int e = errno;
                ::close(fd);
                throw StructureError(ErrorKind::Io, path + ": " + std::strerror(e));  // Mmap::map(..)?
            }
            m.data_ = static_cast<const uint8_t*>(p);
            m.mapped_ = true;
        }
        ::close(fd);
        return m;
    }
    static Mmap borrow(const uint8_t* data, size_t len)
    {
        Mmap m;
        m.data_ = data;
        m.len_ = len;
        return m;
    }
    Mmap() = default;
    Mmap(Mmap&& o) noexcept { *this = std::move(o); }
    Mmap& operator=(Mmap&& o) noexcept
    {
        if (this != &o) {
            release();
            data_ = o.data_;
            len_ = o.len_;
            mapped_ = o.mapped_;
            o.data_ = nullptr;
            o.len_ = 0;
            o.mapped_ = false;
        }
        return *this;
    }
    Mmap(const Mmap&) = delete;
    Mmap& operator=(const Mmap&) = delete;
    ~Mmap() { release(); }
    const uint8_t* data() const { return data_; }
    size_t len() const { return len_; }
    uint8_t operator[](size_t i) const { return data_[i]; }

private:
    void release()
    {
        if (mapped_ && data_) ::munmap(const_cast<uint8_t*>(data_), len_);
        mapped_ = false;
    }
    const uint8_t* data_ = nullptr;
    size_t len_ = 0;
    bool mapped_ = false;
};

// ---- one csvb200_ctx per process / GPU -----------------------------------------------------------
class Gpu {
public:
    explicit Gpu(int device = 0)
    {
        const int rc = csvb200_ctx_create(device, &ctx_);
        if (rc != CSVB200_OK) throw StructureError(ErrorKind::Gpu, "csvb200_ctx_create failed: no usable CUDA device");
    }
    ~Gpu() { csvb200_ctx_destroy(ctx_); }
    Gpu(const Gpu&) = delete;
    Gpu& operator=(const Gpu&) = delete;
    csvb200_ctx* raw() const { return ctx_; }
    static Gpu& instance()
    {
        static Gpu g(0);
        return g;
    }

private:
    csvb200_ctx* ctx_ = nullptr;
};

// ---- StructureIndex(Vec<CodeUnitPos>) (src/stage1.rs:61) ------------------------------------------
class StructureIndex {
public:
    StructureIndex() = default;
    StructureIndex(csvb200_ctx* ctx, csvb200_index* h) : ctx_(ctx), h_(h) {}
    StructureIndex(StructureIndex&& o) noexcept { *this = std::move(o); }
    StructureIndex& operator=(StructureIndex&& o) noexcept
    {
        if (this != &o) {
            if (h_) csvb200_index_free(h_);
            ctx_ = o.ctx_;
            h_ = o.h_;
            host_ = std::move(o.host_);
            o.h_ = nullptr;
        }
        return *this;
    }
    StructureIndex(const StructureIndex&) = delete;
    StructureIndex& operator=(const StructureIndex&) = delete;
    ~StructureIndex()
    {
        if (h_) csvb200_index_free(h_);
    }
    size_t len() const { return h_ ? csvb200_index_len(h_) : 0; }
    csvb200_index* raw() const { return h_; }
    csvb200_ctx* ctx() const { return ctx_; }
    // the host copy (what Rust holds as Vec<usize>); fetched once, on first use
    const std::vector<uint64_t>& host() const
    {
        if (host_.empty() && h_) {
            host_.resize(len());
            check(csvb200_index_copy_out(h_, host_.data(), host_.size()), ctx_);
        }
        return host_;
    }
    uint64_t operator[](size_t i) const { return host().at(i); }  // Vec bounds check = reference panic

private:
    csvb200_ctx* ctx_ = nullptr;
    csvb200_index* h_ = nullptr;
    mutable std::vector<uint64_t> host_;
};

// ---- src/stage1.rs:472-480 -------------------------------------------------------------------------
enum class NewLine { CRLF, LF };

// ---- src/tape.rs:217-277 ----------------------------------------------------------------------------
struct Header {
    std::vector<std::string> header;
    NewLine new_line = NewLine::LF;
    uint32_t field_cnt = 0;
    uint8_t delimiter = 0x2C;
    uint32_t record_offset = 0;

    // Header::new (src/tape.rs:226-273)
    static Header make(const Mmap& memmap)
    {
        const size_t n = memmap.len();
        size_t end = 0;  // :228-232
        while (end < n && memmap[end] != 0x0D && memmap[end] != 0x0A) ++end;
        if (end + 1 >= n)  // memmap[header_end_idx + 1] :236
            throw StructureError(ErrorKind::ReferencePanic, "Header::new indexes past the end of the input");
        Header h;
        h.new_line = memmap[end + 1] == 0x0A ? NewLine::CRLF : NewLine::LF;  // :235-238
        size_t start = 0;                                                   // :241-249
        while (start < n && (memmap[start] == 0xEF || memmap[start] == 0xBB || memmap[start] == 0xBF)) ++start;
        if (start > end) throw StructureError(ErrorKind::ReferencePanic, "Header::new slices start > end");
        auto is_ws = [](uint8_t c) { return c == 0x20 || (c >= 0x09 && c <= 0x0D); };
        size_t s = start;
        for (size_t p = start; p <= end; ++p) {  // split(",").map(trim) :259-262 (not quote aware)
            if (p == end || memmap[p] == 0x2C) {
                size_t a = s, b = p;
                while (a < b && is_ws(memmap[a])) ++a;
                while (b > a && is_ws(memmap[b - 1])) --b;
                h.header.emplace_back(reinterpret_cast<const char*>(memmap.data() + a), b - a);
                s = p + 1;
            }
        }
        h.field_cnt = static_cast<uint32_t>(h.header.size());  // :264
        h.record_offset = static_cast<uint32_t>(end);          // :271
        return h;
    }
};

// ---- src/reader.rs -----------------------------------------------------------------------------------
namespace reader {
// reader::read (src/reader.rs:150-306); n < 64 mirrors the reference's panic as ReferencePanic
inline StructureIndex read(const Mmap& memmap, Gpu& gpu = Gpu::instance())
{
    csvb200_index* h = nullptr;
    check(csvb200_index_build(gpu.raw(), memmap.data(), memmap.len(), CSVB200_BUILD_KEEP_BYTES | CSVB200_BUILD_STRICT_MIN64,
                              &h),
          gpu.raw());
    return StructureIndex(gpu.raw(), h);
}

// The same over several GPUs of this process: ONE byte slice in, ONE Vec<usize>-shaped index out
// (csvb200_multi_index_build_to_host: the slice is cut "without first knowing record breaks", README.md:24, the
// 32-byte rows cross NVLink from inside the build launches).  What `create` (src/lib.rs:61-74) would call at 8 GPUs.
inline std::vector<uint64_t> read_multi(const Mmap& memmap, const std::vector<int>& devices)
{
    if (memmap.len() < 64) throw StructureError(ErrorKind::ReferencePanic, "n < 64: the reference panics on this input");
    csvb200_multi* m = nullptr;
    if (csvb200_multi_create(devices.data(), static_cast<int>(devices.size()), &m) != CSVB200_OK)
        throw StructureError(ErrorKind::Gpu, "csvb200_multi_create failed");
    std::vector<uint64_t> out(memmap.len() / 3 + 4096);
    size_t len = 0;
    int rc = csvb200_multi_index_build_to_host(m, memmap.data(), memmap.len(), nullptr, out.data(), out.size(), &len);
    if (rc == CSVB200_ERR_CAPACITY && len > out.size()) {   // denser than the first guess: the exact size is reported
        out.resize(len);
        rc = csvb200_multi_index_build_to_host(m, memmap.data(), memmap.len(), nullptr, out.data(), out.size(), &len);
    }
    const std::string why = rc ? csvb200_multi_last_error(m) : "";
    csvb200_multi_destroy(m);
    if (rc != CSVB200_OK) throw StructureError(ErrorKind::Gpu, why);
    out.resize(len);
    return out;
}
}  // namespace reader

// ---- src/tape.rs:281-284, 385-428 -------------------------------------------------------------------
struct Boundary {
    size_t start;
    size_t len;
    bool operator==(const Boundary& o) const { return start == o.start && len == o.len; }
};

inline std::optional<std::vector<Boundary>> boundaries(uint32_t task_size, uint8_t job_count)
{
    if (task_size == 0 || job_count == 0) return std::nullopt;  // :387-389
    if (task_size < static_cast<uint32_t>(job_count)) return std::vector<Boundary>{{0, task_size}};
    const uint32_t job_size = task_size / job_count, remainder = task_size % job_count;
    std::vector<Boundary> out;
    out.reserve(job_count);
    uint32_t acc_end = 0, share = 1;
    for (uint8_t i = 0; i < job_count; ++i) {  // :412-421
        if (share == 1 && i >= static_cast<uint8_t>(remainder)) share = 0;
        out.push_back({acc_end, job_size + share});
        acc_end += job_size + share;
    }
    return out;
}

// ---- src/tape.rs:13-19 --------------------------------------------------------------------------------
struct Chunk {
    uint8_t id;
    size_t start;  // KeyToPos
    size_t end;    // KeyToPos
    uint32_t record_cnt;
    const StructureIndex* index;
};

// ---- trait RecordSource (src/record_source.rs:68-147) --------------------------------------------------
class RecordSource {
public:
    virtual ~RecordSource() = default;
    virtual std::optional<uint32_t> record_cnt() const = 0;
    virtual const StructureIndex& index() const = 0;
    virtual size_t record_jump_size() const = 0;  // throws InvalidState before init
    virtual uint32_t field_cnt() const = 0;
    virtual NewLine new_line_tag() const = 0;
    virtual std::string_view data_bytes() const = 0;

    // src/record_source.rs:70-102
    std::optional<std::string_view> seek_record(uint32_t record_idx) const
    {
        const auto rc = record_cnt();
        if (!rc) throw StructureError::invalid_state();
        if (record_idx + 1u >= *rc) return std::nullopt;
        const uint32_t fc = field_cnt();
        const uint32_t idx_start = (record_idx + 1u) * static_cast<uint32_t>(record_jump_size());
        const uint64_t mem_start = index()[idx_start];
        const uint64_t mem_end = index()[static_cast<size_t>(idx_start) + fc];
        return slice(mem_start + 1, mem_end);
    }
    // src/record_source.rs:104-140 (the unconditional println! are not reproduced)
    std::optional<std::string_view> seek_field(uint32_t record_idx, uint32_t field_idx) const
    {
        const auto rc = record_cnt();
        if (!rc) throw StructureError::invalid_state();
        if (record_idx + 1u >= *rc) return std::nullopt;
        const uint32_t fc = field_cnt();
        if (field_idx >= fc) return std::nullopt;
        const uint32_t row_size = new_line_tag() == NewLine::CRLF ? fc + 1u : fc;
        const uint32_t idx_start = (record_idx + 1u) * row_size + field_idx;
        const uint64_t mem_start = index()[idx_start];
        const uint64_t mem_end = index()[static_cast<size_t>(idx_start) + 1];
        return slice(mem_start + 1, mem_end);
    }
    // batched forms on the GPU (K4 gather kernel): (UINT64_MAX, UINT64_MAX) = None
    std::vector<csvb200_range> seek_fields(const std::vector<uint32_t>& rec, const std::vector<uint32_t>& fld) const
    {
        if (!record_cnt()) throw StructureError::invalid_state();
        if (rec.size() != fld.size()) throw std::invalid_argument("rec / fld size mismatch");
        std::vector<csvb200_range> out(rec.size());
        check(csvb200_seek_fields(index().raw(), rec.data(), fld.data(), rec.size(), out.data()), index().ctx());
        return out;
    }

private:
    std::string_view slice(uint64_t s, uint64_t e) const
    {
        const std::string_view d = data_bytes();
        if (s > e || e > d.size()) throw std::out_of_range("slice index out of range");  // Rust slice panic
        return d.substr(s, e - s);
    }
};

// ---- TapeCore (src/tape.rs:185-212, 301-352) -----------------------------------------------------------
class TapeCore : public RecordSource {
public:
    static TapeCore create(Mmap memmap, StructureIndex index, Header header)  // :303-312
    {
        TapeCore t;
        t.header_ = std::move(header);
        t.index_ = std::move(index);
        t.memmap_ = std::move(memmap);
        return t;
    }
    void init()  // :315-347, through csvb200_tape_init
    {
        uint32_t rc = 0;
        uint64_t jump = 0;
        const int st = csvb200_tape_init(index_.raw(), header_.field_cnt, header_.new_line == NewLine::CRLF, &rc, &jump);
        if (st == CSVB200_OK || st == CSVB200_ERR_INVALID_CSV_FORMAT) {  // both fields are set before the error (:318-325)
            record_jump_size_ = static_cast<size_t>(jump);
            record_cnt_ = rc;
        }
        check(st, index_.ctx());
    }
    const std::vector<std::string>& header() const { return header_.header; }
    std::optional<uint32_t> record_cnt() const override { return record_cnt_; }
    const StructureIndex& index() const override { return index_; }
    size_t record_jump_size() const override
    {
        if (!record_jump_size_) throw StructureError::invalid_state();  // :200-201
        return *record_jump_size_;
    }
    uint32_t field_cnt() const override { return header_.field_cnt; }
    NewLine new_line_tag() const override { return header_.new_line; }
    std::string_view data_bytes() const override
    {
        return {reinterpret_cast<const char*>(memmap_.data()), memmap_.len()};
    }

private:
    friend class Tape;
    Header header_;
    StructureIndex index_;
    Mmap memmap_;
    std::optional<uint32_t> record_cnt_;
    std::optional<size_t> record_jump_size_;
};

// ---- Tape (src/tape.rs:74-174) ----------------------------------------------------------------------------
class Tape : public RecordSource {
public:
    Header header_info;
    uint32_t record_cnt_value = 0;
    size_t record_jump = 0;

    static Tape from_core(TapeCore core)  // :83-94
    {
        core.init();
        Tape t;
        t.header_info = std::move(core.header_);
        t.bytes_ = std::move(core.memmap_);
        t.record_cnt_value = *core.record_cnt_;
        t.record_jump = *core.record_jump_size_;
        t.index_ = std::move(core.index_);
        return t;
    }
    std::vector<Chunk> chunks(uint8_t num) const  // :95-140
    {
        const auto bs = boundaries(record_cnt_value, num);
        if (!bs) throw StructureError::invalid_state();
        std::vector<Chunk> out;
        uint8_t id = 0;
        for (const Boundary& b : *bs)
            out.push_back({id++, b.start * record_jump, (b.start + b.len) * record_jump, static_cast<uint32_t>(b.len), &index_});
        out[0] = Chunk{out[0].id, record_jump, out[0].end, out[0].record_cnt - 1, out[0].index};  // :117-123
        return out;
    }
    // ---- beyond the crate (SURVEY 8f), same device-resident tape ----
    // which row breaks the fixed-width assumption TapeCore::init only counts on (:327)
    csvb200_tape_report validate() const
    {
        csvb200_tape_report rep{};
        check(csvb200_tape_validate(index_.raw(), header_info.field_cnt, header_info.new_line == NewLine::CRLF, &rep), index_.ctx());
        return rep;
    }
    // a whole column of seek_field values (record 0 = first row after the header), trimmed / unquoted
    struct Column {
        std::vector<uint64_t> offsets;   // nrec + 1
        std::string bytes;
        std::string_view operator[](size_t i) const { return std::string_view(bytes).substr(offsets[i], offsets[i + 1] - offsets[i]); }
        size_t size() const { return offsets.empty() ? 0 : offsets.size() - 1; }
    };
    Column column(uint32_t field_idx, uint32_t first_record, uint32_t nrec, uint32_t flags = CSVB200_FIELD_UNQUOTE | CSVB200_FIELD_TRIM) const
    {
        Column c;
        c.offsets.assign(static_cast<size_t>(nrec) + 1, 0);
        size_t total = 0;
        int rc = csvb200_materialize_column(index_.raw(), field_idx, first_record, nrec, flags, c.offsets.data(), nullptr, 0, &total);
        if (rc != CSVB200_ERR_CAPACITY) check(rc, index_.ctx());
        c.bytes.resize(total);
        if (total)
            check(csvb200_materialize_column(index_.raw(), field_idx, first_record, nrec, flags, c.offsets.data(),
                                             reinterpret_cast<uint8_t*>(&c.bytes[0]), total, &total), index_.ctx());
        return c;
    }
    // the values behind a batch of lookups: fld non-empty = field fld[q] of record rec[q] (trimmed / unquoted by flags,
    // as column()), fld empty = the text of record rec[q]; get(q) is nullopt exactly where seek_field / seek_record is
    struct Values {
        std::vector<uint64_t> offsets;   // nq + 1
        std::string bytes;
        std::vector<uint64_t> found;     // bit q % 64 of word q / 64
        std::optional<std::string_view> get(size_t q) const
        {
            if (!(found[q / 64] >> (q % 64) & 1u)) return std::nullopt;
            return std::string_view(bytes).substr(offsets[q], offsets[q + 1] - offsets[q]);
        }
        size_t size() const { return offsets.empty() ? 0 : offsets.size() - 1; }
    };
    Values seek_values(const std::vector<uint32_t>& rec, const std::vector<uint32_t>& fld, uint32_t flags = CSVB200_FIELD_RAW) const
    {
        if (!fld.empty() && rec.size() != fld.size()) throw std::invalid_argument("rec / fld size mismatch");
        Values v;
        v.offsets.assign(rec.size() + 1, 0);
        v.found.assign((rec.size() + 63) / 64 + 1, 0);
        const uint32_t* f = fld.empty() ? nullptr : fld.data();
        size_t total = 0;
        int rc = csvb200_seek_values(index_.raw(), rec.data(), f, rec.size(), flags, v.offsets.data(), nullptr, 0, &total,
                                     v.found.data());
        if (rc != CSVB200_ERR_CAPACITY) check(rc, index_.ctx());
        v.bytes.resize(total);
        if (total)
            check(csvb200_seek_values(index_.raw(), rec.data(), f, rec.size(), flags, v.offsets.data(),
                                      reinterpret_cast<uint8_t*>(&v.bytes[0]), total, &total, v.found.data()), index_.ctx());
        return v;
    }
    // core::str::from_utf8 over the whole file: nullopt = well-formed (seek_record hands out &str unchecked, record_source.rs:97-101)
    std::optional<uint64_t> utf8_valid_up_to() const
    {
        uint64_t v = 0;
        int ascii = 0;
        check(csvb200_validate_utf8(index_.ctx(), bytes_.data(), bytes_.len(), &v, &ascii), index_.ctx());
        return bytes_.len() == 0 || v == UINT64_MAX ? std::nullopt : std::optional<uint64_t>(v);
    }
    const StructureIndex& index() const override { return index_; }
    const Mmap& bytes() const { return bytes_; }
    const std::vector<std::string>& header() const { return header_info.header; }
    std::optional<uint32_t> record_cnt() const override { return record_cnt_value; }
    size_t record_jump_size() const override { return record_jump; }
    uint32_t field_cnt() const override { return header_info.field_cnt; }
    NewLine new_line_tag() const override { return header_info.new_line; }
    std::string_view data_bytes() const override { return {reinterpret_cast<const char*>(bytes_.data()), bytes_.len()}; }

private:
    Mmap bytes_;
    StructureIndex index_;
};

// ---- csv_simd::create (src/lib.rs:61-74) ---------------------------------------------------------------------
inline Tape create(const std::string& filename, Gpu* gpu = nullptr)
{
    Mmap memmap = Mmap::map(filename);        // I/O errors first, exactly as File::open(..)? / Mmap::map(..)?
    Header header = Header::make(memmap);
    StructureIndex index = reader::read(memmap, gpu ? *gpu : Gpu::instance());
    TapeCore core = TapeCore::create(std::move(memmap), std::move(index), std::move(header));
    return Tape::from_core(std::move(core));
}

}  // namespace csv_simd
