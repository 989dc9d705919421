// scrubby_host.cpp -- see scrubby_host.hpp for the reference items each function mirrors.
#include "scrubby_host.hpp"

#include <sys/stat.h>
#include <zlib.h>

#include <atomic>
#include <chrono>
#include <thread>
#include <fcntl.h>
#include <sys/wait.h>
#include <unistd.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <functional>
#include <future>
#include <mutex>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <fstream>
#include <sstream>
#include <thread>

namespace scrubby {

// ------------------------------------------------------------------------------------------ errors
ScrubbyError ScrubbyError::from_status(int st, uint64_t index, const std::string &what) {
    std::string msg = what + ": " + sgpu_strerror(st);
    switch (st) {
    case SGPU_ERR_IO: return {IoError, msg, index};
    case SGPU_ERR_FASTQ_INVALID_START:
    case SGPU_ERR_FASTQ_INVALID_SEPARATOR:
    case SGPU_ERR_FASTQ_UNEQUAL_LENGTHS:
    case SGPU_ERR_FASTQ_UNEXPECTED_END:
    case SGPU_ERR_FASTQ_UNKNOWN_FORMAT: return {NeedletailParseError, msg, index};
    case SGPU_ERR_RECORD_NAME_UTF8: return {RecordNameUtf8Error, msg, index};
    case SGPU_ERR_FASTQ_HEADER: return {NeedletailFastqHeader, msg, index};
    case SGPU_ERR_PAF_INTEGER: return {PafRecordIntegerError, msg, index};
    case SGPU_ERR_WOULD_PANIC: return {WouldPanic, msg, index};
    case SGPU_ERR_FASTA_UNSUPPORTED: return {Unsupported, msg, index};
    default: return {Gpu, msg + " (" + sgpu_last_cuda_error() + ")", index};
    }
}

static void check(int st, uint64_t index, const char *what) {
    if (st != SGPU_OK) throw ScrubbyError::from_status(st, index, what);
}

// ------------------------------------------------------------------------------------------ enums
const char *serde_name(Aligner a) {
    switch (a) {
    case Aligner::Bowtie2: return "bowtie2";
    case Aligner::Minimap2: return "minimap2";
    case Aligner::Minigraph: return "minigraph";
    default: return "strobealign";
    }
}
const char *serde_name(Classifier c) { return c == Classifier::Kraken2 ? "kraken2" : "metabuli"; }
const char *serde_name(Preset p) {
    static const char *n[] = {"LrHq", "Splice", "SpliceHq", "Asm", "Asm5", "Asm10", "Asm20",
                              "Sr", "Lr", "MapPb", "MapHifi", "MapOnt", "AvaPb", "AvaOnt"};
    return n[(int)p];
}
const char *display_name(Preset p) {  // scrubby.rs:136-155
    static const char *n[] = {"lr:hq", "splice", "splice:hq", "asm", "asm5", "asm10", "asm20",
                              "sr", "lr", "map-pb", "map-hifi", "map-ont", "ava-pb", "ava-ont"};
    return n[(int)p];
}
std::optional<Aligner> parse_aligner(const std::string &s) {
    if (s == "bowtie2") return Aligner::Bowtie2;
    if (s == "minimap2") return Aligner::Minimap2;
    if (s == "minigraph") return Aligner::Minigraph;
    if (s == "strobealign") return Aligner::Strobealign;
    return std::nullopt;  // "minimap2-rs" exists only with the reference's `mm2` feature
}
std::optional<Preset> parse_preset(const std::string &s) {
    static const char *n[] = {"lr-hq", "splice", "splice-hq", "asm", "asm5", "asm10", "asm20",
                              "sr", "lr", "map-pb", "map-hifi", "map-ont", "ava-pb", "ava-ont"};
    for (int i = 0; i < 14; i++)
        if (s == n[i]) return (Preset)i;
    return std::nullopt;
}
std::optional<Classifier> parse_classifier(const std::string &s) {
    if (s == "kraken2") return Classifier::Kraken2;
    if (s == "metabuli") return Classifier::Metabuli;
    return std::nullopt;
}
std::optional<AlignmentFormat> parse_alignment_format(const std::string &s) {
    static const std::pair<const char *, AlignmentFormat> t[] = {
        {"sam", AlignmentFormat::Sam}, {"bam", AlignmentFormat::Bam}, {"cram", AlignmentFormat::Cram},
        {"paf", AlignmentFormat::Paf}, {"txt", AlignmentFormat::Txt}, {"gaf", AlignmentFormat::Gaf}};
    for (auto &p : t)
        if (s == p.first) return p.second;
    return std::nullopt;
}

// ------------------------------------------------------------------------------------------ handles
GpuContext::GpuContext(int device) { check(sgpu_ctx_create(device, &ctx_), 0, "sgpu_ctx_create"); }
GpuContext::~GpuContext() { sgpu_ctx_destroy(ctx_); }

std::vector<std::string> ReadIdSet::sorted(const GpuContext &g) const {
    uint8_t *buf = nullptr;
    size_t n = 0;
    check(sgpu_idset_dump(g.get(), h_, &buf, &n), 0, "sgpu_idset_dump");
    std::vector<std::string> out;
    size_t pos = 0;
    while (pos < n) {
        const uint8_t *e = (const uint8_t *)memchr(buf + pos, '\n', n - pos);
        out.emplace_back((const char *)buf + pos, (size_t)(e - (buf + pos)));
        pos = (size_t)(e - buf) + 1;
    }
    sgpu_free(buf);
    return out;
}

// ------------------------------------------------------------------------------------------ host I/O stage
static std::string extension(const std::string &path) {  // std::path::Path::extension
    size_t slash = path.find_last_of('/');
    std::string name = slash == std::string::npos ? path : path.substr(slash + 1);
    size_t dot = name.find_last_of('.');
    if (dot == std::string::npos || dot == 0) return "";
    return name.substr(dot + 1);
}

Compression compression_from_path(const std::string &path) {
    std::string e = extension(path);
    if (e == "gz") return Compression::Gzip;
    if (e == "bz" || e == "bz2") return Compression::Bzip;
    if (e == "lzma" || e == "xz") return Compression::Lzma;
    return Compression::No;
}

static std::vector<uint8_t> slurp(const std::string &path) {
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) throw ScrubbyError(ScrubbyError::IoError, "No such file or directory: " + path);
    std::vector<uint8_t> data;
    struct stat stt;
    if (fstat(fileno(f), &stt) == 0 && stt.st_size > 0) data.reserve((size_t)stt.st_size);
    uint8_t chunk[1 << 16];
    size_t r;
    while ((r = fread(chunk, 1, sizeof(chunk), f)) > 0) data.insert(data.end(), chunk, chunk + r);
    fclose(f);
    return data;
}

// niffler::get_reader: sniff the magic bytes (needs 5 bytes), then decode.  gz via zlib (multi-member);
// bz2 / xz need libraries this image does not have and are reported as NifflerError.
// BGZF (bgzip, BAM): every gzip member carries its compressed size in a "BC" extra field and its inflated size in the
// trailer, so the members are located without inflating and inflated on all host threads, each into its own slice
// of the output.  Returns false (nothing done) when some member is not a BGZF block: the serial path takes over.
static bool inflate_bgzf_parallel(const std::vector<uint8_t> &raw, std::vector<uint8_t> &out) {
    struct Blk {
        size_t src, clen, dst;
        uint32_t isize, crc;
    };
    std::vector<Blk> blks;
    size_t p = 0, total = 0;
    while (p < raw.size()) {
        if (raw.size() - p < 18 || raw[p] != 0x1f || raw[p + 1] != 0x8b || raw[p + 2] != 8 || !(raw[p + 3] & 4)) return false;
        const size_t xlen = raw[p + 10] | (raw[p + 11] << 8);
        if (raw.size() - p < 12 + xlen + 8) return false;
        size_t bsize = 0;
        for (size_t q = p + 12; q + 4 <= p + 12 + xlen;) {
            const size_t sl = raw[q + 2] | (raw[q + 3] << 8);
            if (raw[q] == 'B' && raw[q + 1] == 'C' && sl == 2 && q + 6 <= p + 12 + xlen) bsize = (raw[q + 4] | (raw[q + 5] << 8)) + 1;
            q += 4 + sl;
        }
        if (bsize < 12 + xlen + 8 || bsize > raw.size() - p) return false;
        const uint8_t *t = raw.data() + p + bsize - 4;
        const uint32_t isize = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16) | ((uint32_t)t[3] << 24);
        const uint32_t crc = (uint32_t)t[-4] | ((uint32_t)t[-3] << 8) | ((uint32_t)t[-2] << 16) | ((uint32_t)t[-1] << 24);
        // the BGZF specification caps a block's payload at 64 KiB: a member that claims more is not BGZF (and must not
        // size the output: 28-byte members claiming 4 GiB each would ask for terabytes) -- the serial path decides
        if (isize > 65536) return false;
        blks.push_back(Blk{p + 12 + xlen, bsize - 12 - xlen - 8, total, isize, crc});
        total += isize;
        p += bsize;
    }
    const auto t0 = std::chrono::steady_clock::now();
    try {
        out.resize(total);
    } catch (const std::bad_alloc &) {
        return false;
    }
    const auto t1 = std::chrono::steady_clock::now();
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const unsigned nt = (unsigned)std::min<size_t>(hw, std::max<size_t>(1, blks.size() / 16));
    std::atomic<size_t> next{0};
    std::atomic<bool> bad{false};
    auto work = [&] {
        z_stream zs;
        memset(&zs, 0, sizeof(zs));
        if (inflateInit2(&zs, -15) != Z_OK) {
            bad = true;
            return;
        }
        for (size_t i; (i = next.fetch_add(1)) < blks.size() && !bad;) {
            const Blk &b = blks[i];
            inflateReset(&zs);
            zs.next_in = const_cast<uint8_t *>(raw.data() + b.src);
            zs.avail_in = (uInt)b.clen;
            zs.next_out = out.data() + b.dst;
            zs.avail_out = b.isize;
            const int rc = inflate(&zs, Z_FINISH);
            if (rc != Z_STREAM_END || zs.avail_out != 0 || zs.avail_in != 0 ||
                (uint32_t)crc32(crc32(0L, Z_NULL, 0), out.data() + b.dst, b.isize) != b.crc)
                bad = true;  // (the serial path then reports the corrupt member)
        }
        inflateEnd(&zs);
    };
    std::vector<std::thread> th;
    for (unsigned k = 1; k < nt; k++) th.emplace_back(work);
    work();
    for (auto &t : th) t.join();
    if (getenv("SCRUBBY_DEBUG")) {
        const auto t2 = std::chrono::steady_clock::now();
        fprintf(stderr, "[scrubby] BGZF: %zu blocks, %zu -> %zu bytes, %u threads: output allocated in %.1f ms, inflated in %.1f ms\n",
                blks.size(), raw.size(), total, nt, std::chrono::duration<double, std::milli>(t1 - t0).count(),
                std::chrono::duration<double, std::milli>(t2 - t1).count());
    }
    return !bad;
}

// is_file_empty (utils.rs:359-375): niffler's FileTooShort rule applies to the RAW file (fewer than 5 bytes), after that
// only "one decompressed byte can be read" counts -- a .gz whose content is "r1\n" is NOT empty
std::vector<uint8_t> read_file(const std::string &path, bool *empty) {
    size_t raw_size = 0;
    std::vector<uint8_t> v = read_file(path, &raw_size);
    *empty = raw_size < 5 || v.empty();
    return v;
}

std::vector<uint8_t> read_file(const std::string &path, size_t *raw_size) {
    std::vector<uint8_t> raw = slurp(path);
    if (raw_size) *raw_size = raw.size();
    if (raw.size() < 5) return raw;  // FileTooShort => callers treat it as empty (utils.rs:365)
    if (raw[0] == 0x1f && raw[1] == 0x8b) {
        std::vector<uint8_t> out;
        if ((raw[3] & 4) && inflate_bgzf_parallel(raw, out)) return out;
        out.clear();
        z_stream zs;
        memset(&zs, 0, sizeof(zs));
        if (inflateInit2(&zs, 15 + 32) != Z_OK) throw ScrubbyError(ScrubbyError::NifflerError, "zlib init failed");
        zs.next_in = raw.data();
        zs.avail_in = (uInt)std::min<size_t>(raw.size(), 0x7fffffff);
        size_t consumed_base = 0;
        std::vector<uint8_t> chunk(1 << 20);
        while (true) {
            zs.next_out = chunk.data();
            zs.avail_out = (uInt)chunk.size();
            int rc = inflate(&zs, Z_NO_FLUSH);
            out.insert(out.end(), chunk.data(), chunk.data() + (chunk.size() - zs.avail_out));
            if (rc == Z_STREAM_END) {
                size_t used = consumed_base + (size_t)(zs.next_in - (raw.data() + consumed_base));
                if (used >= raw.size()) break;
                consumed_base = used;  // next gzip member
                inflateReset(&zs);
                zs.next_in = raw.data() + used;
                zs.avail_in = (uInt)std::min<size_t>(raw.size() - used, 0x7fffffff);
            } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
                inflateEnd(&zs);
                throw ScrubbyError(ScrubbyError::IoError, "corrupt gzip stream: " + path);
            } else if (zs.avail_in == 0 && zs.avail_out != 0) {
                size_t used = (size_t)(zs.next_in - raw.data());
                if (used >= raw.size()) break;
                zs.avail_in = (uInt)std::min<size_t>(raw.size() - used, 0x7fffffff);
            }
        }
        inflateEnd(&zs);
        return out;
    }
    if (raw[0] == 'B' && raw[1] == 'Z' && raw[2] == 'h')
        throw ScrubbyError(ScrubbyError::NifflerError, "bzip2 input: feature disabled in this build: " + path);
    if (raw[0] == 0xfd && raw[1] == '7' && raw[2] == 'z' && raw[3] == 'X' && raw[4] == 'Z')
        throw ScrubbyError(ScrubbyError::NifflerError, "xz input: feature disabled in this build: " + path);
    return raw;
}

// Host stage (SURVEY 8f row 2): output bytes are deflated in independent 4 MiB blocks on all host threads, each block a
// complete gzip member (as pigz -i / bgzip do).  The concatenation is a valid gzip file whose DEcompressed bytes equal
// the reference's output; the compressed bytes differ (they depend on flate2's backend in the reference and are not
// part of the parity contract).  n == 0 writes one empty member.
static void deflate_members(FILE *f, const uint8_t *data, size_t n, int gz_level, const std::string &path) {
    const size_t BLOCK = (size_t)4 << 20;
    const size_t nb = n ? (n + BLOCK - 1) / BLOCK : 1;
    std::vector<std::vector<uint8_t>> parts(nb);
    std::atomic<size_t> next{0};
    std::atomic<bool> failed{false};
    auto work = [&]() {
        for (size_t b = next.fetch_add(1); b < nb && !failed; b = next.fetch_add(1)) {
            const size_t a = b * BLOCK, len = std::min(BLOCK, n - a);
            z_stream zs;
            memset(&zs, 0, sizeof(zs));
            if (deflateInit2(&zs, gz_level, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) {
                failed = true;
                return;
            }
            std::vector<uint8_t> &o = parts[b];
            o.resize(deflateBound(&zs, (uLong)len) + 64);
            zs.next_in = const_cast<Bytef *>(data + a);
            zs.avail_in = (uInt)len;
            zs.next_out = o.data();
            zs.avail_out = (uInt)o.size();
            const int rc = deflate(&zs, Z_FINISH);
            if (rc != Z_STREAM_END) failed = true;
            o.resize(o.size() - zs.avail_out);
            deflateEnd(&zs);
        }
    };
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const size_t nt = std::min<size_t>(std::min<size_t>(hw, 32), nb);
    std::vector<std::thread> th;
    for (size_t i = 1; i < nt; i++) th.emplace_back(work);
    work();
    for (auto &t : th) t.join();
    if (failed) throw ScrubbyError(ScrubbyError::NifflerError, "deflate failed: " + path);
    for (auto &o : parts) {
        if (!o.empty() && fwrite(o.data(), 1, o.size(), f) != o.size())
            throw ScrubbyError(ScrubbyError::IoError, "write failed: " + path);
    }
}

void write_file(const std::string &path, const uint8_t *data, size_t n, int gz_level) {
    OutSink sink(path, gz_level);
    sink.append(data, n);
    sink.close();
}

// get_fastx_writer (utils.rs:38-74) as a sink that takes the output piece by piece: the file is created by the first
// append (or by close), gz output gets its members appended as they are produced
OutSink::OutSink(const std::string &path, int gz_level) : path_(path), level_(gz_level) {
    Compression c = compression_from_path(path);
    if (c == Compression::Bzip || c == Compression::Lzma)
        throw ScrubbyError(ScrubbyError::NifflerError, "bzip2/xz output: feature disabled in this build: " + path);
    gz_ = c == Compression::Gzip;
}

OutSink::~OutSink() {
    if (f_) fclose((FILE *)f_);
}

void OutSink::open() {
    if (f_) return;
    f_ = fopen(path_.c_str(), "wb");
    if (!f_) throw ScrubbyError(ScrubbyError::IoError, "cannot create " + path_);
}

void OutSink::append(const uint8_t *data, size_t n) {
    open();
    if (!n) return;
    if (gz_)
        deflate_members((FILE *)f_, data, n, level_, path_);
    else if (fwrite(data, 1, n, (FILE *)f_) != n)
        throw ScrubbyError(ScrubbyError::IoError, "write failed: " + path_);
    total_ += n;
}

void OutSink::close() {
    open();
    if (gz_ && total_ == 0) deflate_members((FILE *)f_, nullptr, 0, level_, path_);  // an empty gzip member, as the writer leaves
    const int rc = fclose((FILE *)f_);
    f_ = nullptr;
    if (rc != 0) throw ScrubbyError(ScrubbyError::IoError, "write failed: " + path_);
}

// ------------------------------------------------------------------------------------------ gzip input as a stream
// SURVEY 8f row 2: a plain (non-BGZF) gzip FASTQ is inflated by ONE thread at a few hundred MB/s -- the slowest stage of
// the whole tool.  Instead of inflating the file, then filtering it, then deflating the output, the three stages run
// concurrently: a producer thread inflates into a bounded queue of blocks, the calling thread feeds the filter chunk by
// chunk through the shard entry point of the C ABI (own range + halo, running newline count, the first chunk's CRLF
// decision), and the previous chunk's output is deflated / written behind it.  Host memory: a few chunks instead of the
// whole file and its output.
namespace {

struct ByteSource {  // decompressed bytes of a file, block by block
    virtual ~ByteSource() {}
    virtual bool next(std::vector<uint8_t> &block) = 0;  // false (and an empty block) at the end of the stream
};

class GzSource : public ByteSource {  // serial inflate of a (multi-member) gzip file, pulled piece by piece
  public:
    GzSource(const std::string &path, size_t block) : path_(path), block_(block), in_(1 << 20) {
        f_ = fopen(path.c_str(), "rb");
        if (!f_) throw ScrubbyError(ScrubbyError::IoError, "No such file or directory: " + path);
        init();
    }
    // continues a file another reader has opened: `pending` are the raw bytes it had read but not consumed
    GzSource(const std::string &path, size_t block, FILE *f, const uint8_t *pending, size_t n_pending)
        : path_(path), block_(block), f_(f), in_(std::max<size_t>(1 << 20, n_pending)) {
        init();
        if (n_pending) memcpy(in_.data(), pending, n_pending);
        zs_.next_in = in_.data();
        zs_.avail_in = (uInt)n_pending;
    }
    ~GzSource() override {
        inflateEnd(&zs_);
        fclose(f_);
    }
    GzSource(const GzSource &) = delete;
    GzSource &operator=(const GzSource &) = delete;
    bool next(std::vector<uint8_t> &block) override {
        block.resize(block_);
        block.resize(read(block.data(), block_));
        return !block.empty();
    }
    // up to `cap` decompressed bytes into dst; fewer than cap only at the end of the stream (a truncated last member
    // ends the stream quietly, bytes that are not a gzip member after one are an error: as read_file has it)
    size_t read(uint8_t *dst, size_t cap) {
        size_t got = 0;
        while (got < cap && !done_) {
            if (zs_.avail_in == 0) {
                const size_t r = fread(in_.data(), 1, in_.size(), f_);
                if (r == 0) {
                    done_ = true;
                    break;
                }
                zs_.next_in = in_.data();
                zs_.avail_in = (uInt)r;
                if (member_done_) {  // a further member starts here
                    inflateReset(&zs_);
                    member_done_ = false;
                }
            }
            zs_.next_out = dst + got;
            zs_.avail_out = (uInt)std::min<size_t>(cap - got, 0x40000000);
            const int rc = inflate(&zs_, Z_NO_FLUSH);
            got = (size_t)(zs_.next_out - dst);
            if (rc == Z_STREAM_END) {
                member_done_ = true;
                if (zs_.avail_in) {
                    inflateReset(&zs_);
                    member_done_ = false;
                }
            } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
                throw ScrubbyError(ScrubbyError::IoError, "corrupt gzip stream: " + path_);
            }
        }
        return got;
    }

  private:
    void init() {
        memset(&zs_, 0, sizeof(zs_));
        if (inflateInit2(&zs_, 15 + 32) != Z_OK) {
            fclose(f_);
            throw ScrubbyError(ScrubbyError::NifflerError, "zlib init failed");
        }
    }
    std::string path_;
    size_t block_;
    FILE *f_ = nullptr;
    z_stream zs_;
    std::vector<uint8_t> in_;
    bool done_ = false, member_done_ = false;
};

// BGZF (bgzip): every member names its compressed size (BSIZE in the "BC" extra field) and its inflated size (ISIZE), so
// a batch of members is cut out of the raw bytes without inflating and inflated on all host threads, each member into
// its own slice of the block.  The first member that is not a BGZF block (a plain gzip member appended to the file, a
// truncated tail) hands the rest of the file to the serial reader.
class BgzfSource : public ByteSource {
  public:
    BgzfSource(const std::string &path, size_t block) : path_(path), block_(std::max<size_t>(block, 1 << 16)) {
        const char *pc = getenv("SCRUBBY_BGZF_PIECE");  // (tests: raw bytes read per refill)
        if (pc && *pc) piece_ = std::max<size_t>((size_t)strtoull(pc, nullptr, 10), 1 << 10);
        f_ = fopen(path.c_str(), "rb");
        if (!f_) throw ScrubbyError(ScrubbyError::IoError, "No such file or directory: " + path);
    }
    ~BgzfSource() override {
        if (f_) fclose(f_);
    }
    BgzfSource(const BgzfSource &) = delete;
    BgzfSource &operator=(const BgzfSource &) = delete;
    bool next(std::vector<uint8_t> &block) override {
        block.clear();
        while (block.empty()) {
            if (serial_) return serial_->next(block);
            if (!batch(block)) return false;
        }
        return true;
    }

  private:
    struct Blk {
        size_t src, clen, dst;
        uint32_t isize, crc;
    };
    // 1: a complete BGZF member at p (b filled, *size = its length); 0: more raw bytes needed; -1: not a BGZF member
    static int member(const uint8_t *p, size_t avail, Blk &b, size_t *size) {
        if (avail < 18) return 0;
        if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return -1;
        const size_t xlen = p[10] | (p[11] << 8);
        if (avail < 12 + xlen) return 0;
        size_t bsize = 0;
        for (size_t q = 12; q + 4 <= 12 + xlen;) {
            const size_t sl = p[q + 2] | (p[q + 3] << 8);
            if (p[q] == 'B' && p[q + 1] == 'C' && sl == 2 && q + 6 <= 12 + xlen) bsize = (p[q + 4] | (p[q + 5] << 8)) + 1;
            q += 4 + sl;
        }
        if (bsize < 12 + xlen + 8) return -1;
        if (avail < bsize) return 0;
        const uint8_t *t = p + bsize - 4;
        b.isize = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16) | ((uint32_t)t[3] << 24);
        b.crc = (uint32_t)t[-4] | ((uint32_t)t[-3] << 8) | ((uint32_t)t[-2] << 16) | ((uint32_t)t[-1] << 24);
        if (b.isize > 65536) return -1;  // the specification's cap: a member that claims more is not BGZF
        b.src = 12 + xlen;
        b.clen = bsize - 12 - xlen - 8;
        *size = bsize;
        return 1;
    }
    // one batch: the complete members at hand, up to about block_ bytes of output; false at the end of the file
    bool batch(std::vector<uint8_t> &out) {
        std::vector<Blk> blks;
        size_t total = 0, p = pos_;
        bool not_bgzf = false;
        while (total < block_) {
            Blk b;
            size_t size = 0;
            const int rc = member(raw_.data() + p, raw_.size() - p, b, &size);
            if (rc == 0) {  // the member at p is not complete yet
                if (!blks.empty()) break;  // inflate what is at hand first; the next call reads on
                const bool more = refill();  // (drops the consumed bytes: offsets restart at 0)
                p = pos_;
                if (!more) {  // end of the file: leftover bytes are a truncated member (the serial reader's case)
                    not_bgzf = raw_.size() > pos_;
                    break;
                }
                continue;
            }
            if (rc < 0) {
                not_bgzf = true;
                break;
            }
            b.src += p;
            b.dst = total;
            total += b.isize;
            blks.push_back(b);
            p += size;
        }
        if (!blks.empty()) inflate_all(blks, total, out);
        pos_ = p;
        if (not_bgzf) {  // the serial reader takes the file from here
            serial_.reset(new GzSource(path_, block_, f_, raw_.data() + pos_, raw_.size() - pos_));
            f_ = nullptr;
            raw_.clear();
            pos_ = 0;
            return true;
        }
        return !blks.empty();
    }
    // drops the consumed raw bytes and appends the next piece of the file; false at the end of the file
    bool refill() {
        raw_.erase(raw_.begin(), raw_.begin() + (ptrdiff_t)pos_);
        pos_ = 0;
        const size_t old = raw_.size();
        raw_.resize(old + piece_);
        const size_t r = fread(raw_.data() + old, 1, piece_, f_);
        raw_.resize(old + r);
        return r > 0;
    }
    void inflate_all(const std::vector<Blk> &blks, size_t total, std::vector<uint8_t> &out) {
        out.resize(std::max<size_t>(total, 1));  // (a batch of empty members -- the EOF marker -- still needs a valid pointer)
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const unsigned nt = (unsigned)std::min<size_t>(hw, std::max<size_t>(1, blks.size() / 8));
        std::atomic<size_t> next{0};
        std::atomic<bool> bad{false};
        const uint8_t *raw = raw_.data();
        auto work = [&] {
            z_stream zs;
            memset(&zs, 0, sizeof(zs));
            if (inflateInit2(&zs, -15) != Z_OK) {
                bad = true;
                return;
            }
            for (size_t i; (i = next.fetch_add(1)) < blks.size() && !bad;) {
                const Blk &b = blks[i];
                inflateReset(&zs);
                zs.next_in = const_cast<uint8_t *>(raw + b.src);
                zs.avail_in = (uInt)b.clen;
                zs.next_out = out.data() + b.dst;
                zs.avail_out = b.isize;
                const int rc = inflate(&zs, Z_FINISH);
                if (rc != Z_STREAM_END || zs.avail_out != 0 || zs.avail_in != 0 ||
                    (uint32_t)crc32(crc32(0L, Z_NULL, 0), out.data() + b.dst, b.isize) != b.crc)
                    bad = true;
            }
            inflateEnd(&zs);
        };
        std::vector<std::thread> th;
        for (unsigned k = 1; k < nt; k++) th.emplace_back(work);
        work();
        for (auto &t : th) t.join();
        if (bad) throw ScrubbyError(ScrubbyError::IoError, "corrupt gzip stream: " + path_);
        out.resize(total);
    }
    std::string path_;
    size_t block_;
    FILE *f_ = nullptr;
    std::vector<uint8_t> raw_;
    size_t pos_ = 0, piece_ = (size_t)8 << 20;
    std::unique_ptr<GzSource> serial_;
};

class BlockQueue {  // producer: the inflating thread; consumer: the thread that owns the GPU context
  public:
    BlockQueue(std::function<std::unique_ptr<ByteSource>()> make, size_t max_blocks) : max_(max_blocks) {
        th_ = std::thread([this, make] { produce(make); });
    }
    ~BlockQueue() {
        {
            std::lock_guard<std::mutex> l(m_);
            cancel_ = true;
        }
        cv_.notify_all();
        th_.join();
    }
    // the next block (empty at the end of the stream); rethrows the producer's error
    std::vector<uint8_t> pop() {
        std::unique_lock<std::mutex> l(m_);
        cv_.wait(l, [this] { return !q_.empty() || finished_; });
        if (q_.empty()) {
            if (err_) std::rethrow_exception(err_);
            return {};
        }
        std::vector<uint8_t> b = std::move(q_.front());
        q_.pop_front();
        l.unlock();
        cv_.notify_all();
        return b;
    }

  private:
    void produce(const std::function<std::unique_ptr<ByteSource>()> &make) {
        try {
            std::unique_ptr<ByteSource> src = make();
            while (true) {
                std::vector<uint8_t> b;
                if (!src->next(b)) break;
                std::unique_lock<std::mutex> l(m_);
                cv_.wait(l, [this] { return q_.size() < max_ || cancel_; });
                if (cancel_) break;
                q_.push_back(std::move(b));
                l.unlock();
                cv_.notify_all();
            }
        } catch (...) {
            std::lock_guard<std::mutex> l(m_);
            err_ = std::current_exception();
        }
        {
            std::lock_guard<std::mutex> l(m_);
            finished_ = true;
        }
        cv_.notify_all();
    }
    size_t max_;
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<std::vector<uint8_t>> q_;
    bool finished_ = false, cancel_ = false;
    std::exception_ptr err_;
    std::thread th_;
};

size_t env_size(const char *name, size_t dflt) {
    const char *v = getenv(name);
    return (v && *v) ? (size_t)strtoull(v, nullptr, 10) : dflt;
}

}  // namespace

namespace {

// one chunk of a stream through a format's shard entry point: (window, n, own_len, is_first, is_last, out, cap, &n_out,
// &counts) -> status.  `next` is told about every chunk that produced its records and is not the last one: the state
// the following chunk starts from (FASTQ: running newline count, line ending; FASTA: line-ending decision)
using ChunkFn = std::function<int(const uint8_t *, size_t, size_t, int, int, uint8_t *, size_t, size_t *, sgpu_counts *)>;
using NextFn = std::function<void(const uint8_t *own_bytes, size_t own, const sgpu_counts &)>;

// the inflate thread -> chunked shard calls -> deflate / write behind them pipeline shared by the formats.  false: not
// gzip, or the decoded input does not start with `lead` (or is shorter than `min_len`): nothing was done
bool gz_stream(const std::string &input, const std::string &output, uint8_t lead, size_t min_len, size_t chunk, size_t halo,
               const ChunkFn &run, const NextFn &next) {
    bool bgzf = false;
    {   // gzip only (by magic bytes, as niffler sniffs): plain members are inflated serially, BGZF members in parallel
        FILE *f = fopen(input.c_str(), "rb");
        if (!f) throw ScrubbyError(ScrubbyError::IoError, "No such file or directory: " + input);
        uint8_t h[18];
        const size_t r = fread(h, 1, sizeof(h), f);
        fclose(f);
        if (r < 5 || h[0] != 0x1f || h[1] != 0x8b) return false;
        bgzf = r >= 16 && h[2] == 8 && (h[3] & 4) && h[12] == 'B' && h[13] == 'C';
        if (bgzf && getenv("SCRUBBY_NO_BGZF_STREAM")) return false;
    }
    chunk = std::max<size_t>(chunk, 16);
    halo = std::max<size_t>(halo, 1);
    const size_t BLOCK = std::min<size_t>((size_t)4 << 20, std::max<size_t>(chunk / 4, 64));
    BlockQueue q([&input, bgzf, BLOCK]() -> std::unique_ptr<ByteSource> {
        if (bgzf) return std::unique_ptr<ByteSource>(new BgzfSource(input, 4 * BLOCK));
        return std::unique_ptr<ByteSource>(new GzSource(input, BLOCK));
    }, bgzf ? 8 : 24);
    std::vector<uint8_t> win;
    bool src_end = false;
    auto fill = [&](size_t want) {
        while (!src_end && win.size() < want) {
            std::vector<uint8_t> b = q.pop();
            if (b.empty())
                src_end = true;
            else
                win.insert(win.end(), b.begin(), b.end());
        }
    };
    fill(chunk + halo);
    // nothing inside, another format, or not a sequence file: the whole-file path reports those exactly as before
    if (win.empty() || win[0] != lead || (src_end && win.size() < min_len)) return false;

    OutSink sink(output, 6);  // niffler::compression::Level::Six
    std::vector<uint8_t> out[2];
    std::future<void> writing;
    auto settle = [&] {
        if (writing.valid()) writing.get();
    };
    uint64_t reads_before = 0;
    bool first = true;
    for (unsigned turn = 0;; turn ^= 1) {
        fill(chunk + halo);
        const bool last = src_end;  // the buffer reaches EOF: this chunk owns the rest and applies the end-of-file rules
        const size_t own = last ? win.size() : chunk;
        std::vector<uint8_t> &o = out[turn];
        size_t cap = win.size() + win.size() / 16 + 4096;
        size_t n_out = 0;
        sgpu_counts counts;
        int st;
        while (true) {
            if (o.size() < cap) o.resize(cap);
            memset(&counts, 0, sizeof(counts));
            st = run(win.data(), win.size(), own, first ? 1 : 0, last ? 1 : 0, o.data(), o.size(), &n_out, &counts);
            if (st != SGPU_ERR_CAPACITY || cap >= 2 * win.size() + 64) break;
            cap = 2 * win.size() + 64;
        }
        if (st == SGPU_ERR_HALO && !last) {  // a record longer than the halo: look further ahead and run the chunk again
            halo *= 2;
            turn ^= 1;
            continue;
        }
        const bool parse_error = st >= SGPU_ERR_FASTQ_INVALID_START && st <= SGPU_ERR_FASTQ_HEADER;
        if (st == SGPU_OK || parse_error) {  // (on a parse error the reference has written the records before it)
            settle();
            const uint8_t *data = o.data();
            writing = std::async(std::launch::async, [&sink, data, n_out] { sink.append(data, n_out); });
        }
        if (st != SGPU_OK) {
            settle();
            if (parse_error) sink.close();
            check(st, reads_before + counts.error_record, "clean_reads");
        }
        first = false;
        if (last) break;
        next(win.data(), own, counts);
        reads_before += counts.reads_in;
        win.erase(win.begin(), win.begin() + (ptrdiff_t)own);
    }
    settle();
    sink.close();
    return true;
}

}  // namespace

bool clean_fastq_gz_stream(const std::string &input, const std::string &output, const ShardFn &shard, size_t chunk, size_t halo) {
    uint64_t nlb = 0;  // running newline count: the line phase of the next chunk
    int crlf = -1;     // the first chunk decides the line ending
    return gz_stream(
        input, output, '@', 0, chunk, halo,
        [&](const uint8_t *in, size_t n, size_t own, int is_first, int is_last, uint8_t *out, size_t cap, size_t *n_out,
            sgpu_counts *counts) { return shard(in, n, own, nlb, is_first, is_last, crlf, out, cap, n_out, counts); },
        [&](const uint8_t *own_bytes, size_t own, const sgpu_counts &counts) {
            if (crlf < 0) crlf = counts.crlf ? 1 : 0;
            nlb += (uint64_t)std::count(own_bytes, own_bytes + own, (uint8_t)'\n');
        });
}

bool clean_fasta_gz_stream(const std::string &input, const std::string &output, const FastaShardFn &shard, size_t chunk,
                           size_t halo) {
    int le = -1, le_chunk = -1;  // the next chunk's le_before: this chunk's, once decided, else its own decision
    return gz_stream(
        input, output, '>', 5, chunk, halo,
        [&](const uint8_t *in, size_t n, size_t own, int is_first, int is_last, uint8_t *out, size_t cap, size_t *n_out,
            sgpu_counts *counts) {
            le_chunk = -1;
            return shard(in, n, own, is_first, is_last, le, out, cap, n_out, counts, &le_chunk);
        },
        [&](const uint8_t *, size_t, const sgpu_counts &) {
            if (le < 0) le = le_chunk;
        });
}

static bool file_exists(const std::string &p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0 && S_ISREG(st.st_mode);
}

// ------------------------------------------------------------------------------------------ alignment.rs
ReadAlignment ReadAlignment::from(const GpuContext &g, const std::string &path, uint64_t min_len, double min_cov,
                                  uint8_t min_mapq, std::optional<AlignmentFormat> fmt) {
    if (fmt) {  // alignment.rs:40-47
        switch (*fmt) {
        case AlignmentFormat::Paf:
        case AlignmentFormat::Gaf: return from_paf(g, path, min_len, min_cov, min_mapq);
        case AlignmentFormat::Txt: return from_txt(g, path);
        case AlignmentFormat::Sam:
        case AlignmentFormat::Bam:
        case AlignmentFormat::Cram:  // alignment.rs:45 (`htslib`): one reader, it sniffs the CONTENT
            return from_sam(g, path, min_len, min_cov, min_mapq);
        }
    }
    // alignment.rs:48-56: only the LAST extension is seen, so "x.paf.gz" is not recognised
    std::string e = extension(path);
    if (e == "paf" || e == "gaf") return from_paf(g, path, min_len, min_cov, min_mapq);
    if (e == "txt") return from_txt(g, path);
    if (e == "sam" || e == "bam" || e == "cram") return from_sam(g, path, min_len, min_cov, min_mapq);  // alignment.rs:54 (`htslib`)
    throw ScrubbyError(ScrubbyError::AlignmentInputFormatNotRecognized,
                       "Unable to recognize alignment input format from extension.");
}

ReadAlignment ReadAlignment::from_paf(const GpuContext &g, const std::string &path, uint64_t min_len, double min_cov,
                                      uint8_t min_mapq) {
    bool empty = false;
    std::vector<uint8_t> buf = read_file(path, &empty);
    ReadAlignment r;
    uint64_t err = 0;
    if (empty) buf.clear();  // is_file_empty => empty set (alignment.rs:93)
    check(sgpu_idset_from_paf(g.get(), buf.data(), buf.size(), min_len, min_cov, min_mapq, r.aligned_reads.out(), &err),
          err, "from_paf");
    return r;
}

// alignment.rs:117-146 (rust-htslib reads "-" as stdin and has no is_file_empty test here).  Like htslib's reader this
// looks at the content, not at --format or the extension: BGZF / gzip is inflated by read_file (BGZF blocks are gzip
// members), a stream that starts with "BAM\1" is binary BAM, "CRAM" is refused (reference-based decoder: not built),
// anything else is SAM text
ReadAlignment ReadAlignment::from_sam(const GpuContext &g, const std::string &path, uint64_t min_len, double min_cov,
                                      uint8_t min_mapq) {
    std::vector<uint8_t> buf = read_file(path);
    ReadAlignment r;
    uint64_t err = 0;
    if (buf.size() >= 4 && memcmp(buf.data(), "BAM\1", 4) == 0) {
        check(sgpu_idset_from_bam(g.get(), buf.data(), buf.size(), min_len, min_cov, min_mapq, r.aligned_reads.out(), &err),
              err, "from_bam");
        return r;
    }
    if (buf.size() >= 4 && memcmp(buf.data(), "CRAM", 4) == 0)
        throw ScrubbyError(ScrubbyError::AlignmentInputFormatInvalid,
                           "CRAM input needs a reference-based decoder, which this build does not have: " + path);
    check(sgpu_idset_from_sam(g.get(), buf.data(), buf.size(), min_len, min_cov, min_mapq, r.aligned_reads.out(), &err),
          err, "from_sam");
    return r;
}

ReadAlignment ReadAlignment::from_txt(const GpuContext &g, const std::string &path) {
    bool empty = false;
    std::vector<uint8_t> buf = read_file(path, &empty);
    ReadAlignment r;
    uint64_t err = 0;
    if (empty) buf.clear();
    check(sgpu_idset_from_txt(g.get(), buf.data(), buf.size(), r.aligned_reads.out(), &err), err, "from_txt");
    return r;
}

// ------------------------------------------------------------------------------------------ classifier.rs (host)
namespace {

bool utf8_valid(const uint8_t *s, size_t n) {
    size_t i = 0;
    while (i < n) {
        uint8_t c = s[i];
        if (c < 0x80) { i++; continue; }
        size_t need;
        uint8_t lo = 0x80, hi = 0xBF;
        if (c >= 0xC2 && c <= 0xDF) need = 1;
        else if (c >= 0xE0 && c <= 0xEF) { need = 2; if (c == 0xE0) lo = 0xA0; if (c == 0xED) hi = 0x9F; }
        else if (c >= 0xF0 && c <= 0xF4) { need = 3; if (c == 0xF0) lo = 0x90; if (c == 0xF4) hi = 0x8F; }
        else return false;
        if (i + need >= n) return false;
        if (s[i + 1] < lo || s[i + 1] > hi) return false;
        for (size_t k = 2; k <= need; k++)
            if ((s[i + k] & 0xC0) != 0x80) return false;
        i += need + 1;
    }
    return true;
}

bool is_ws(uint32_t cp) {
    return (cp >= 9 && cp <= 13) || cp == 0x20 || cp == 0x85 || cp == 0xA0 || cp == 0x1680 || (cp >= 0x2000 && cp <= 0x200A) ||
           cp == 0x2028 || cp == 0x2029 || cp == 0x202F || cp == 0x205F || cp == 0x3000;
}

// str::trim over valid UTF-8
std::string trim(const std::string &s) {
    auto decode = [&](size_t i, uint32_t *cp) -> size_t {
        uint8_t c = (uint8_t)s[i];
        if (c < 0x80) { *cp = c; return 1; }
        if (c < 0xE0) { *cp = ((c & 0x1Fu) << 6) | ((uint8_t)s[i + 1] & 0x3F); return 2; }
        if (c < 0xF0) { *cp = ((c & 0x0Fu) << 12) | (((uint8_t)s[i + 1] & 0x3Fu) << 6) | ((uint8_t)s[i + 2] & 0x3F); return 3; }
        *cp = ((c & 0x07u) << 18) | (((uint8_t)s[i + 1] & 0x3Fu) << 12) | (((uint8_t)s[i + 2] & 0x3Fu) << 6) | ((uint8_t)s[i + 3] & 0x3F);
        return 4;
    };
    size_t i = 0, j = s.size();
    while (i < j) {
        uint32_t cp;
        size_t l = decode(i, &cp);
        if (!is_ws(cp)) break;
        i += l;
    }
    while (j > i) {
        size_t k = j - 1;
        while (k > i && ((uint8_t)s[k] & 0xC0) == 0x80) k--;
        uint32_t cp;
        decode(k, &cp);
        if (!is_ws(cp)) break;
        j = k;
    }
    return s.substr(i, j - i);
}

bool parse_u64(const std::string &f) {  // <u64 as FromStr>
    if (f.empty()) return false;
    size_t i = 0;
    if (f[0] == '+' || f[0] == '-') {
        if (f.size() == 1 || f[0] == '-') return false;
        i = 1;
    }
    unsigned __int128 v = 0;
    for (; i < f.size(); i++) {
        if (f[i] < '0' || f[i] > '9') return false;
        v = v * 10 + (unsigned)(f[i] - '0');
        if (v > (unsigned __int128)UINT64_MAX) return false;
    }
    return true;
}
uint64_t value_u64(const std::string &f) {
    uint64_t v = 0;
    for (char c : f)
        if (c >= '0' && c <= '9') v = v * 10 + (uint64_t)(c - '0');
    return v;
}

enum Level { None, Unclassified, NoRank, Root, Domain, Kingdom, Phylum, Class, Order, Family, Genus, Species, Unspecified };

bool starts(const std::string &s, const char *p) { return s.compare(0, strlen(p), p) == 0; }

Level get_tax_level(const std::string &r) {  // classifier.rs:345-373
    if (starts(r, "U")) return Unclassified;
    if (starts(r, "no rank")) return NoRank;
    if (starts(r, "R")) return Root;
    if (starts(r, "D") || starts(r, "superkingdom")) return Domain;
    if (starts(r, "K") || starts(r, "kingdom")) return Kingdom;
    if (starts(r, "P") || starts(r, "phylum")) return Phylum;
    if (starts(r, "C") || starts(r, "class")) return Class;
    if (starts(r, "O") || starts(r, "order")) return Order;
    if (starts(r, "F") || starts(r, "family")) return Family;
    if (starts(r, "G") || starts(r, "genus")) return Genus;
    if (starts(r, "S") || starts(r, "species")) return Species;
    return Unspecified;
}

bool contains(const std::vector<std::string> &v, const std::string &x) { return std::find(v.begin(), v.end(), x) != v.end(); }

}  // namespace

std::vector<std::string> get_taxids_from_report_bytes(const uint8_t *buf, size_t n, const std::vector<std::string> &taxa_in,
                                                      const std::vector<std::string> &direct_in) {
    std::vector<std::string> taxa, direct;
    for (auto &t : taxa_in) taxa.push_back(trim(t));       // classifier.rs:132
    for (auto &t : direct_in) direct.push_back(trim(t));   // classifier.rs:133
    std::set<std::string> taxids;
    Level extract_level = None;
    std::string extract_parent;
    size_t pos = 0;
    uint64_t line_no = 0;
    while (pos < n) {  // BufRead::lines
        const uint8_t *nl = (const uint8_t *)memchr(buf + pos, '\n', n - pos);
        size_t raw = nl ? (size_t)(nl - (buf + pos)) + 1 : n - pos;
        if (!utf8_valid(buf + pos, raw)) throw ScrubbyError(ScrubbyError::IoError, "stream did not contain valid UTF-8", line_no);
        size_t len = raw;
        if (len && buf[pos + len - 1] == '\n') {
            len--;
            if (len && buf[pos + len - 1] == '\r') len--;
        }
        std::string line((const char *)buf + pos, len);
        pos += raw;
        // KrakenReportRecord::from_str, classifier.rs:449-466
        std::vector<std::string> f;
        size_t st = 0;
        for (size_t i = 0; i <= line.size(); i++)
            if (i == line.size() || line[i] == '\t') {
                f.push_back(line.substr(st, i - st));
                st = i + 1;
            }
        if (f.size() < 2) throw ScrubbyError(ScrubbyError::WouldPanic, "report line has too few columns", line_no);
        if (!parse_u64(f[1])) throw ScrubbyError(ScrubbyError::KrakenReportReadFieldConversion,
                                                  "failed to convert the read field in the report from `Kraken2`", line_no);
        if (f.size() < 3) throw ScrubbyError(ScrubbyError::WouldPanic, "report line has too few columns", line_no);
        if (!parse_u64(f[2])) throw ScrubbyError(ScrubbyError::KrakenReportDirectReadFieldConversion,
                                                  "failed to convert the direct read field in the report from `Kraken2`", line_no);
        if (f.size() < 6) throw ScrubbyError(ScrubbyError::WouldPanic, "report line has too few columns", line_no);
        uint64_t reads_direct = value_u64(f[2]);
        std::string tax_level = trim(f[3]), tax_id = trim(f[4]), tax_name = trim(f[5]);
        Level level = get_tax_level(tax_level);

        if (contains(direct, tax_name) || contains(direct, tax_id)) taxids.insert(tax_id);  // :145-155
        if (level < Domain) {                                                                 // :157-166
            line_no++;
            continue;
        }
        if (contains(taxa, tax_name) || contains(taxa, tax_id)) {  // :168-187
            extract_level = level;
            extract_parent = tax_name;
            if (reads_direct > 0) taxids.insert(tax_id);
        } else if (extract_level != None) {  // :189-199 skip when no subtree is open
            if (level <= extract_level && tax_level.size() == 1) {
                extract_level = None;  // :200-208
            } else if (reads_direct > 0) {  // :210-223
                taxids.insert(tax_id);
                if (extract_parent.empty())
                    throw ScrubbyError(ScrubbyError::KrakenReportTaxonParent,
                                       "failed to provide a parent taxon while parsing report from `Kraken2`", line_no);
            }
        }
        line_no++;
    }
    return std::vector<std::string>(taxids.begin(), taxids.end());
}

std::vector<std::string> get_taxids_from_report(const std::string &report, const std::vector<std::string> &taxa,
                                                const std::vector<std::string> &direct) {
    std::vector<uint8_t> buf = slurp(report);  // classifier.rs:130 plain File::open, no decompression
    return get_taxids_from_report_bytes(buf.data(), buf.size(), taxa, direct);
}

static ReadIdSet taxid_reads(const GpuContext &g, const std::vector<std::string> &taxids, const std::string &reads, int style) {
    ReadIdSet out;
    std::vector<uint8_t> buf;
    if (file_exists(reads)) buf = slurp(reads);  // classifier.rs:276-278 missing file => empty set
    std::vector<const char *> p;
    std::vector<size_t> l;
    for (auto &t : taxids) {
        p.push_back(t.data());
        l.push_back(t.size());
    }
    uint64_t err = 0;
    check(sgpu_idset_from_reads(g.get(), buf.data(), buf.size(), style, p.data(), l.data(), p.size(), out.out(), &err), err,
          "get_taxid_reads");
    return out;
}
ReadIdSet get_taxid_reads_kraken(const GpuContext &g, const std::vector<std::string> &t, const std::string &r) {
    return taxid_reads(g, t, r, 0);
}
ReadIdSet get_taxid_reads_metabuli(const GpuContext &g, const std::vector<std::string> &t, const std::string &r) {
    return taxid_reads(g, t, r, 1);
}

// ------------------------------------------------------------------------------------------ cleaner.rs
void FastqCleaner::clean_reads(const GpuContext &g, const ReadIdSet &read_ids, bool reverse) const {
    if (!getenv("SCRUBBY_NO_GZ_STREAM")) {  // gzip / BGZF FASTQ or FASTA: inflate, filter and deflate as one pipeline
        ShardFn shard = [&](const uint8_t *in, size_t n_in, size_t own_len, uint64_t newlines_before, int is_first, int is_last,
                            int crlf, uint8_t *out, size_t cap, size_t *n_out, sgpu_counts *counts) {
            return (int)sgpu_clean_fastq_shard(g.get(), read_ids.get(), in, n_in, own_len, newlines_before, is_first, is_last, crlf,
                                               reverse ? 1 : 0, out, cap, n_out, nullptr, 0, nullptr, counts);
        };
        const size_t chunk = env_size("SCRUBBY_STREAM_CHUNK", (size_t)64 << 20), halo = env_size("SCRUBBY_STREAM_HALO", (size_t)8 << 20);
        if (clean_fastq_gz_stream(input, output, shard, chunk, halo)) return;
        FastaShardFn fasta = [&](const uint8_t *in, size_t n_in, size_t own_len, int is_first, int is_last, int le_before,
                                 uint8_t *out, size_t cap, size_t *n_out, sgpu_counts *counts, int *le_own) {
            return (int)sgpu_clean_fasta_shard(g.get(), read_ids.get(), in, n_in, own_len, is_first, is_last, le_before,
                                               reverse ? 1 : 0, out, cap, n_out, nullptr, 0, nullptr, counts, le_own);
        };
        if (clean_fasta_gz_stream(input, output, fasta, chunk, halo)) return;
    }
    bool empty = false;
    std::vector<uint8_t> in = read_file(input, &empty);
    if (empty) {  // parse_fastx_file_with_check => None: warn, create nothing (cleaner.rs:755-757)
        fprintf(stderr, "[WARN] - Input file is empty: %s\n", input.c_str());
        return;
    }
    // write_fastq re-serialises the input: the output only outgrows it when LF records follow a CRLF first record (+4
    // bytes per record); uninitialised storage (a zero-filled vector of twice a 33 GB mate file is seconds of memset)
    size_t cap = in.size() + in.size() / 16 + 4096;
    std::unique_ptr<uint8_t[]> out(new uint8_t[cap]);
    size_t n_out = 0;
    sgpu_counts counts;
    int st = sgpu_clean_fastq(g.get(), read_ids.get(), in.data(), in.size(), reverse ? 1 : 0, out.get(), cap, &n_out, nullptr, 0,
                              nullptr, &counts);
    if (st == SGPU_ERR_CAPACITY) {
        cap = 2 * in.size() + 64;
        out.reset(new uint8_t[cap]);
        st = sgpu_clean_fastq(g.get(), read_ids.get(), in.data(), in.size(), reverse ? 1 : 0, out.get(), cap, &n_out, nullptr, 0,
                              nullptr, &counts);
    }
    // on a parse error the reference has already written the records before it; an input that is neither FASTQ nor
    // FASTA fails before the writer exists (utils.rs:377-383), so nothing is created for it
    if (st == SGPU_OK || (st >= SGPU_ERR_FASTQ_INVALID_START && st <= SGPU_ERR_FASTQ_HEADER && st != SGPU_ERR_FASTQ_UNKNOWN_FORMAT)) {
        write_file(output, out.get(), n_out, 6);  // niffler::compression::Level::Six
    }
    check(st, counts.error_record, "clean_reads");
}

ReadIdSet Cleaner::parse_classifier_output(const GpuContext &g, const std::string &report, const std::string &reads) const {
    std::vector<std::string> taxids = get_taxids_from_report(report, scrubby.config.taxa, scrubby.config.taxa_direct);
    if (!scrubby.config.classifier) throw ScrubbyError(ScrubbyError::MissingClassifier, "No classifier configured.");
    return *scrubby.config.classifier == Classifier::Kraken2 ? get_taxid_reads_kraken(g, taxids, reads)
                                                            : get_taxid_reads_metabuli(g, taxids, reads);
}

// ------------------------------------------------------------------------------------------ cleaner.rs external tools
SamtoolsConfig SamtoolsConfig::from_scrubby(const Scrubby &s) {  // cleaner.rs:46-71
    const unsigned threads = s.config.samtools_threads.value_or(4);
    SamtoolsConfig c;
    const char *flag = s.extract ? (s.config.paired_end ? "-F 12" : "-F 4") : (s.config.paired_end ? "-f 12" : "-f 4");
    c.filter = std::string("samtools view -h ") + flag + " -";
    const std::string t = std::to_string(threads);
    if (s.config.paired_end)
        c.fastq = "samtools fastq --threads " + t + " " + (s.config.unpaired ? "" : "-s /dev/null") + " -c 6 -n -1 '" +
                  s.output[0] + "' -2 '" + s.output[1] + "'";
    else
        c.fastq = "samtools fastq --threads " + t + " -c 6 -n -0 '" + s.output[0] + "'";
    return c;
}

// Command::new("sh").arg("-c").arg(cmd) with stderr (and optionally stdout) discarded: the exit code, or -1
static int sh_status(const std::string &cmd, bool quiet_stdout) {
    const pid_t pid = fork();
    if (pid < 0) return -2;
    if (pid == 0) {
        const int nul = open("/dev/null", O_WRONLY);
        if (nul >= 0) {
            dup2(nul, 2);
            if (quiet_stdout) dup2(nul, 1);
        }
        execl("/bin/sh", "sh", "-c", cmd.c_str(), (char *)nullptr);
        _exit(127);
    }
    int st = 0;
    if (waitpid(pid, &st, 0) < 0) return -2;
    return WIFEXITED(st) ? WEXITSTATUS(st) : -1;
}

Cleaner Cleaner::from_scrubby(const Scrubby &s) {  // cleaner.rs:110-123, 255-291
    Cleaner c{s, SamtoolsConfig::from_scrubby(s)};
    if (s.config.aligner) {
        static const char *ver[] = {"bowtie2 --version", "minimap2 --version", "minigraph --version", "strobealign --version"};
        if (sh_status(ver[(int)*s.config.aligner], true) != 0)
            throw ScrubbyError(ScrubbyError::AlignerDependencyMissing,
                               std::string("Aligner `") + serde_name(*s.config.aligner) + "` cannot be executed - is it installed?");
    } else if (s.config.classifier && !(s.config.reads && s.config.report)) {
        // (the reference also probes the tool when only its OUTPUTS are given -- `scrubby classifier`, SURVEY F11;
        //  there the tool is not needed and is not probed here)
        const char *cmd = *s.config.classifier == Classifier::Kraken2 ? "kraken2 --version" : "metabuli";
        if (sh_status(cmd, true) != 0)
            throw ScrubbyError(ScrubbyError::ClassifierDependencyMissing,
                               std::string("Classifier `") + serde_name(*s.config.classifier) + "` cannot be executed - is it installed?");
    }
    return c;
}

void Cleaner::run_command(const std::string &cmd) const {  // cleaner.rs:626-641 (stdout inherited, stderr discarded)
    const int rc = sh_status(cmd, false);
    if (rc == -2) throw ScrubbyError(ScrubbyError::CommandExecutionFailed, "Failed to execute command '" + cmd + "'");
    if (rc != 0) throw ScrubbyError(ScrubbyError::CommandFailed, "Command '" + cmd + "' failed with exit code " + std::to_string(rc));
}

// cleaner.rs:651-687: the child's stdout is PAF; the reference parses it line by line while the child runs, here the
// whole stream is collected and handed to the PAF kernel (same predicate, same errors; a PAF error wins over the
// child's exit status because the reference returns it from inside the read loop)
ReadIdSet Cleaner::run_command_stdout_paf(const GpuContext &g, const std::string &cmd) const {
    int fds[2];
    if (pipe(fds) != 0) throw ScrubbyError(ScrubbyError::CommandExecutionFailed, "Failed to execute command '" + cmd + "': pipe");
    const pid_t pid = fork();
    if (pid < 0) throw ScrubbyError(ScrubbyError::CommandExecutionFailed, "Failed to execute command '" + cmd + "': fork");
    if (pid == 0) {
        close(fds[0]);
        dup2(fds[1], 1);
        const int nul = open("/dev/null", O_WRONLY);
        if (nul >= 0) dup2(nul, 2);
        execl("/bin/sh", "sh", "-c", cmd.c_str(), (char *)nullptr);
        _exit(127);
    }
    close(fds[1]);
    std::vector<uint8_t> buf;
    std::vector<uint8_t> chunk(1 << 20);
    while (true) {
        const ssize_t n = read(fds[0], chunk.data(), chunk.size());
        if (n < 0 && errno == EINTR) continue;
        if (n <= 0) break;
        buf.insert(buf.end(), chunk.data(), chunk.data() + n);
    }
    close(fds[0]);
    int st = 0;
    waitpid(pid, &st, 0);
    ReadIdSet ids;
    uint64_t err = 0;
    check(sgpu_idset_from_paf(g.get(), buf.data(), buf.size(), scrubby.config.min_query_length, scrubby.config.min_query_coverage,
                              scrubby.config.min_mapq, ids.out(), &err),
          err, "run_command_stdout_paf");
    const int rc = WIFEXITED(st) ? WEXITSTATUS(st) : -1;
    if (rc != 0) throw ScrubbyError(ScrubbyError::CommandFailed, "Command '" + cmd + "' failed with exit code " + std::to_string(rc));
    return ids;
}

static std::string temp_dir_of(const Scrubby &s) {  // workdir, else std::env::temp_dir()
    if (s.workdir) {
        mkdir(s.workdir->c_str(), 0755);
        return *s.workdir;
    }
    const char *t = getenv("TMPDIR");
    return (t && *t) ? t : "/tmp";
}
static std::string join_path(const std::string &dir, const std::string &name) {
    return (!dir.empty() && dir.back() == '/') ? dir + name : dir + "/" + name;
}

std::string Cleaner::kraken_command(const std::string &reads_out, const std::string &report_out) const {  // cleaner.rs:300-322
    const ScrubbyConfig &c = scrubby.config;
    const std::string args = c.classifier_args.value_or("");
    const std::string head = "kraken2 --threads " + std::to_string(scrubby.threads) + " --db " + *c.classifier_index + " " + args;
    if (c.paired_end)
        return head + " --paired " + scrubby.input[0] + " " + scrubby.input[1] + " --output " + reads_out + " --report " + report_out;
    return head + " --single " + scrubby.input[0] + " --output " + reads_out + " --report " + report_out;
}

std::string Cleaner::metabuli_command(const std::string &dir) const {  // cleaner.rs:341-362
    const ScrubbyConfig &c = scrubby.config;
    const std::string args = c.classifier_args.value_or("");
    const std::string t = std::to_string(scrubby.threads);
    if (c.paired_end)
        return "metabuli classify --seq-mode 2 --threads " + t + " " + args + " " + scrubby.input[0] + " " + scrubby.input[1] + " " +
               *c.classifier_index + " " + dir + " metabuli";
    return "metabuli classify --seq-mode 3 --threads " + t + " " + args + " " + scrubby.input[0] + " " + *c.classifier_index + " " +
           dir + " metabuli";
}

void Cleaner::run_classifier() const {  // cleaner.rs:155-161, 293-376
    const ScrubbyConfig &c = scrubby.config;
    if (!c.classifier) throw ScrubbyError(ScrubbyError::MissingClassifier, "No classifier configured.");
    if (!c.classifier_index) throw ScrubbyError(ScrubbyError::MissingClassifierIndex, "Classifier index must be set when classifier is configured.");
    const std::string dir = temp_dir_of(scrubby);
    GpuContext g(scrubby.device);
    if (*c.classifier == Classifier::Kraken2) {
        const std::string reads = join_path(dir, "kraken.reads"), report = join_path(dir, "kraken.report");
        run_command(kraken_command(reads, report));
        clean_reads(parse_classifier_output(g, report, reads));
    } else {
        run_command(metabuli_command(dir));
        clean_reads(parse_classifier_output(g, join_path(dir, "metabuli_report.tsv"), join_path(dir, "metabuli_classifications.tsv")));
    }
}

std::string Cleaner::aligner_command() const {  // cleaner.rs:385-470, 573-624
    const ScrubbyConfig &c = scrubby.config;
    const std::string args = c.aligner_args.value_or(""), t = std::to_string(scrubby.threads);
    const std::string &idx = *c.aligner_index, &r1 = scrubby.input[0];
    const std::string r2 = c.paired_end ? scrubby.input[1] : "";
    auto q = [](const std::string &p) { return "'" + p + "'"; };
    switch (*c.aligner) {
    case Aligner::Minimap2:
        if (!c.preset) throw ScrubbyError(ScrubbyError::MissingMinimap2Preset, "Minimap2 preset must be set.");
        return std::string("minimap2 -ax ") + display_name(*c.preset) + " --secondary=no -t " + t + " " + args + " " + q(idx) + " " + q(r1) +
               (c.paired_end ? " " + q(r2) : "") + " | " + samtools.get_pipeline();
    case Aligner::Minigraph:
        if (!c.preset) throw ScrubbyError(ScrubbyError::MissingMinigraphPreset, "Minigraph preset must be set.");
        return std::string("minigraph -cx ") + display_name(*c.preset) + " -N 0 -t " + t + " " + args + " " + q(idx) + " " + q(r1) +
               (c.paired_end ? " " + q(r2) : "");
    case Aligner::Bowtie2:
        if (c.paired_end)
            return "bowtie2 -x " + q(idx) + " -1 " + q(r1) + " -2 " + q(r2) + " -k 1 --mm -p " + t + " " + args + " | " + samtools.get_pipeline();
        return "bowtie2 -x " + q(idx) + " -U " + q(r1) + " -k 1 --mm -p " + t + " " + args + " | " + samtools.get_pipeline() + " ";
    case Aligner::Strobealign:
        return "strobealign -t " + t + " " + args + " " + q(idx) + " " + q(r1) + (c.paired_end ? " " + q(r2) : "") + " | " +
               samtools.get_pipeline();
    }
    throw ScrubbyError(ScrubbyError::MissingAligner, "No aligner configured.");
}

void Cleaner::run_aligner() const {  // cleaner.rs:137-148
    const ScrubbyConfig &c = scrubby.config;
    if (!c.aligner) throw ScrubbyError(ScrubbyError::MissingAligner, "No aligner configured.");
    if (!c.aligner_index) throw ScrubbyError(ScrubbyError::MissingAlignmentIndex, "Aligner index must be set when aligner is configured.");
    const std::string cmd = aligner_command();
    if (*c.aligner == Aligner::Minigraph) {
        // the one aligner whose output comes back into the in-repo path: PAF on stdout -> id set -> clean_reads
        GpuContext g(scrubby.device);
        clean_reads(run_command_stdout_paf(g, cmd));
    } else {
        run_command(cmd);  // SAM-emitting aligners: samtools does the depletion and writes the outputs
    }
}

void Cleaner::run_classifier_output() const {
    if (!scrubby.config.report)
        throw ScrubbyError(ScrubbyError::MissingClassifierClassificationReport,
                           "Classifier read classification report input must be set when classifier cleaning procedure is configured.");
    if (!scrubby.config.reads)
        throw ScrubbyError(ScrubbyError::MissingClassifierReadClassfications,
                           "Classifier read classification input must be set when classifier cleaning procedure is configured.");
    GpuContext g(scrubby.device);
    ReadIdSet ids = parse_classifier_output(g, *scrubby.config.report, *scrubby.config.reads);
    clean_reads(ids);
}

void Cleaner::run_aligner_output() const {
    if (!scrubby.config.alignment) throw ScrubbyError(ScrubbyError::MissingAlignment, "Alignment output must be set when alignment is configured.");
    GpuContext g(scrubby.device);
    ReadAlignment a = ReadAlignment::from(g, *scrubby.config.alignment, scrubby.config.min_query_length,
                                          scrubby.config.min_query_coverage, scrubby.config.min_mapq, scrubby.config.alignment_format);
    clean_reads(a.aligned_reads);
}

void Cleaner::clean_reads(const ReadIdSet &read_ids) const {
    auto one = [&](size_t i) {
        GpuContext g(scrubby.device);  // one context (stream) per mate file; the set is shared read-only
        FastqCleaner::from(scrubby.input[i], scrubby.output[i]).clean_reads(g, read_ids, scrubby.extract);
    };
    if (scrubby.config.paired_end && scrubby.config.needletail_parallel) {
        std::exception_ptr e0, e1;
        std::thread t0([&] { try { one(0); } catch (...) { e0 = std::current_exception(); } });
        std::thread t1([&] { try { one(1); } catch (...) { e1 = std::current_exception(); } });
        t0.join();
        t1.join();
        if (e0) std::rethrow_exception(e0);
        if (e1) std::rethrow_exception(e1);
    } else {
        for (size_t i = 0; i < (scrubby.config.paired_end ? 2u : 1u); i++) one(i);
    }
}

// ------------------------------------------------------------------------------------------ scrubby.rs
static void validate_base_config(Scrubby &s) {  // scrubby.rs:760-799
    if (s.input.empty() || s.output.empty()) throw ScrubbyError(ScrubbyError::EmptyInputOutput, "Input and output vectors must not be empty.");
    if (s.input.size() != s.output.size())
        throw ScrubbyError(ScrubbyError::MismatchedInputOutputLength, "Input and output must be of the same length.");
    if (s.input.size() > 2) throw ScrubbyError(ScrubbyError::InputOutputLengthExceeded, "Input and output vectors must not contain more than two elements.");
    for (auto &f : s.input)
        if (!file_exists(f)) throw ScrubbyError(ScrubbyError::MissingInputReadFile, "Read input file was not found: " + f);
    if (s.workdir) mkdir(s.workdir->c_str(), 0755);
    s.config.paired_end = s.input.size() == 2;
    if (s.config.index) {  // scrubby.rs:787-796
        if (s.config.aligner) s.config.aligner_index = s.config.index;
        else if (s.config.classifier) s.config.classifier_index = s.config.index;
        else s.config.aligner_index = s.config.index;
    }
}

static bool dir_exists(const std::string &p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}
static bool path_exists(const std::string &p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0;
}
// Path::with_extension: the text after the last '.' of the file name is replaced ("" removes it)
static std::string with_extension(const std::string &path, const std::string &ext) {
    const size_t slash = path.find_last_of('/');
    const size_t name0 = slash == std::string::npos ? 0 : slash + 1;
    const size_t dot = path.find_last_of('.');
    std::string stem = (dot != std::string::npos && dot > name0) ? path.substr(0, dot) : path;
    return ext.empty() ? stem : stem + "." + ext;
}

Scrubby build(Scrubby s) {  // scrubby.rs:813-975
    validate_base_config(s);
    ScrubbyConfig &c = s.config;
    if (!c.aligner && !c.classifier) c.aligner = c.paired_end ? Aligner::Bowtie2 : Aligner::Minimap2;  // (no `mm2` feature)
    if (c.aligner && c.classifier)
        throw ScrubbyError(ScrubbyError::AlignerAndClassifierConfigured, "Unable to specify both aligner and classifier.");
    if (c.aligner_index && c.classifier_index)
        throw ScrubbyError(ScrubbyError::AlignerAndClassifierIndexConfigured, "Unable to specify both aligner and classifier index.");
    if (c.classifier) {
        if (!c.classifier_index) throw ScrubbyError(ScrubbyError::MissingClassifierIndex, "Classifier index must be set when classifier is configured.");
        if (c.taxa.empty() && c.taxa_direct.empty())
            throw ScrubbyError(ScrubbyError::MissingTaxa, "If classifier is set, `taxa` or `taxa_direct` must not be empty.");
    }
    if (c.aligner && !c.aligner_index)
        throw ScrubbyError(ScrubbyError::MissingAlignmentIndex, "Aligner index must be set when aligner is configured.");
    if (c.classifier_index && !dir_exists(*c.classifier_index))
        throw ScrubbyError(ScrubbyError::MissingClassifierIndexDirectory, "Classifier index directory was not found: " + *c.classifier_index);
    if (c.aligner && *c.aligner == Aligner::Strobealign && c.aligner_index) {
        const std::string &f = *c.aligner_index;
        if (f.size() > 4 && f.compare(f.size() - 4, 4, ".sti") == 0) {
            const std::string base = with_extension(with_extension(f, ""), "");
            if (!path_exists(base))
                throw ScrubbyError(ScrubbyError::MissingStrobealignIndexBaseFile, "Strobealign index base file was not found: " + base);
        }
    }
    if (c.aligner && *c.aligner == Aligner::Bowtie2) {
        if (c.aligner_index) {
            static const char *small[] = {"1.bt2", "2.bt2", "3.bt2", "4.bt2", "rev.1.bt2", "rev.2.bt2"};
            static const char *large[] = {"1.bt21", "2.bt21", "3.bt21", "4.bt21", "rev.1.bt21", "rev.2.bt21"};
            for (int i = 0; i < 6; i++)
                if (!file_exists(with_extension(*c.aligner_index, small[i])) && !file_exists(with_extension(*c.aligner_index, large[i])))
                    throw ScrubbyError(ScrubbyError::MissingBowtie2IndexFiles, "Bowtie2 index files were not found: " + *c.aligner_index);
        }
    } else if (c.aligner_index && !file_exists(*c.aligner_index)) {
        throw ScrubbyError(ScrubbyError::MissingAlignmentIndexFile, "Alignment index file was not found: " + *c.aligner_index);
    }
    if (c.aligner && *c.aligner == Aligner::Minimap2) {
        if (!c.preset) c.preset = c.paired_end ? Preset::Sr : Preset::MapOnt;
        else if (*c.preset == Preset::Lr)
            throw ScrubbyError(ScrubbyError::Minimap2PresetNotSupported, std::string("Preset not supported for minimap2: ") + display_name(*c.preset));
    }
    if (c.aligner && *c.aligner == Aligner::Minigraph) {
        if (!c.preset) c.preset = c.paired_end ? Preset::Sr : Preset::Lr;
        else if (*c.preset != Preset::Lr && *c.preset != Preset::Sr && *c.preset != Preset::Asm)
            throw ScrubbyError(ScrubbyError::MinigraphPresetNotSupported, std::string("Preset not supported for minigraph: ") + display_name(*c.preset));
    }
    return s;
}

Scrubby build_classifier(Scrubby s) {  // scrubby.rs:978-1006
    validate_base_config(s);
    if (!s.config.reads) throw ScrubbyError(ScrubbyError::MissingClassifierReadClassfications,
                                            "Classifier read classification input must be set when classifier cleaning procedure is configured.");
    if (!s.config.report) throw ScrubbyError(ScrubbyError::MissingClassifierClassificationReport,
                                             "Classifier read classification report input must be set when classifier cleaning procedure is configured.");
    if (s.config.taxa.empty() && s.config.taxa_direct.empty())
        throw ScrubbyError(ScrubbyError::MissingTaxa, "If classifier is set, `taxa` or `taxa_direct` must not be empty.");
    return s;
}

Scrubby build_alignment(Scrubby s) {  // scrubby.rs:1019-1038
    validate_base_config(s);
    if (!s.config.alignment) throw ScrubbyError(ScrubbyError::MissingAlignment, "Alignment output must be set when alignment is configured.");
    return s;
}

void Scrubby::clean() const {  // scrubby.rs:255-281
    Cleaner cleaner = Cleaner::from_scrubby(*this);
    if (config.aligner) {
        cleaner.run_aligner();
    } else if (config.reads && config.report) {
        // SURVEY F11: the reference's `classifier` subcommand reaches run_kraken and fails; the intended
        // path is run_classifier_output, which is what runs here (before the `classifier` arm for that reason).
        cleaner.run_classifier_output();
    } else if (config.classifier) {
        cleaner.run_classifier();
    } else if (config.alignment) {
        cleaner.run_aligner_output();
    } else {
        throw ScrubbyError(ScrubbyError::NoAlignerOrClassifierConfigured, "Unable to specify both aligner and classifier.");
    }
    if (json || read_ids) ScrubbyReport::create(*this, true);
}

// ------------------------------------------------------------------------------------------ utils.rs diff
ReadDifference ReadDifference::build(const std::vector<std::string> &in, const std::vector<std::string> &out,
                                     std::optional<std::string> json, std::optional<std::string> read_ids) {
    if (in.empty() || out.empty()) throw ScrubbyError(ScrubbyError::EmptyInputOutput, "Input and output vectors must not be empty.");
    if (in.size() != out.size()) throw ScrubbyError(ScrubbyError::MismatchedInputOutputLength, "Input and output must be of the same length.");
    if (in.size() > 2) throw ScrubbyError(ScrubbyError::InputOutputLengthExceeded, "Input and output vectors must not contain more than two elements.");
    for (auto &f : in)
        if (!file_exists(f)) throw ScrubbyError(ScrubbyError::MissingInputReadFile, "Read input file was not found: " + f);
    ReadDifference d;
    d.input_reads = in;
    d.output_reads = out;
    d.json = json;
    d.read_ids = read_ids;
    return d;
}

Difference ReadDifference::get_difference() const {
    GpuContext g(device);
    ReadIdSet diff_ids;
    sgpu_counts c;
    memset(&c, 0, sizeof(c));
    for (size_t i = 0; i < input_reads.size() && i < output_reads.size(); i++) {  // zip, utils.rs:256
        std::vector<uint8_t> out = read_file(output_reads[i]);  // a missing output is an I/O error (utils.rs:259,360)
        bool in_empty = false;
        std::vector<uint8_t> in = read_file(input_reads[i], &in_empty);
        if (in_empty) fprintf(stderr, "[WARN] - Input file is empty: %s\n", input_reads[i].c_str());
        check(sgpu_diff(g.get(), in.data(), in.size(), out.data(), out.size(), &c, diff_ids.out()), c.error_record, "get_difference");
    }
    Difference d;
    d.reads_in = c.reads_in;
    d.reads_out = c.reads_out;
    d.difference = c.difference;
    if (diff_ids.get()) d.read_ids = diff_ids.sorted(g);
    return d;
}

Difference ReadDifference::compute() const {  // utils.rs:238-249
    Difference d = get_difference();
    if (json) d.to_json(*json);
    if (read_ids) d.write_read_ids(*read_ids, true);
    return d;
}

std::string Difference::to_json_string() const {  // serde pretty, read_ids skipped (utils.rs:180-187)
    std::ostringstream o;
    o << "{\n  \"reads_in\": " << reads_in << ",\n  \"reads_out\": " << reads_out << ",\n  \"difference\": " << difference << "\n}";
    return o.str();
}
void Difference::to_json(const std::string &output) const {
    std::string s = to_json_string();
    write_file(output, (const uint8_t *)s.data(), s.size(), 6);
}

std::string csv_field(const std::string &f) {  // csv crate, QuoteStyle::Necessary, delimiter '\t'
    bool q = f.empty();
    for (char c : f)
        if (c == '\t' || c == '"' || c == '\n' || c == '\r') q = true;
    if (!q) return f;
    std::string o = "\"";
    for (char c : f) {
        if (c == '"') o += '"';
        o += c;
    }
    return o + "\"";
}

void Difference::write_read_ids(const std::string &output, bool header) const {  // utils.rs:198-219
    std::string s;
    if (header && !read_ids.empty()) s += "id\n";  // serde headers are emitted with the first record
    for (auto &id : read_ids) s += csv_field(id) + "\n";
    write_file(output, (const uint8_t *)s.data(), s.size(), 9);  // Level::Nine
}

// ------------------------------------------------------------------------------------------ report.rs
std::string json_escape(const std::string &s) {
    std::string o = "\"";
    for (unsigned char c : s) {
        switch (c) {
        case '"': o += "\\\""; break;
        case '\\': o += "\\\\"; break;
        case '\n': o += "\\n"; break;
        case '\r': o += "\\r"; break;
        case '\t': o += "\\t"; break;
        case '\b': o += "\\b"; break;
        case '\f': o += "\\f"; break;
        default:
            if (c < 0x20) {
                char b[8];
                snprintf(b, sizeof(b), "\\u%04x", c);
                o += b;
            } else {
                o += (char)c;
            }
        }
    }
    return o + "\"";
}

std::string format_f64(double v) {  // serde_json -> ryu "pretty" format
    if (!std::isfinite(v)) return "null";
    if (v == 0) return std::signbit(v) ? "-0.0" : "0.0";
    char buf[64];
    int prec = 1;
    for (; prec <= 17; prec++) {
        snprintf(buf, sizeof(buf), "%.*e", prec - 1, v);
        if (strtod(buf, nullptr) == v) break;
    }
    std::string s(buf);  // d.ddddde[+-]xx
    bool neg = s[0] == '-';
    if (neg) s = s.substr(1);
    size_t epos = s.find('e');
    int exp10 = atoi(s.c_str() + epos + 1);
    std::string digits;
    for (size_t i = 0; i < epos; i++)
        if (s[i] != '.') digits += s[i];
    while (digits.size() > 1 && digits.back() == '0') digits.pop_back();
    int len = (int)digits.size();
    int kk = exp10 + 1;  // position of the decimal point relative to the digits
    std::string o;
    if (len <= kk && kk <= 16) {
        o = digits + std::string((size_t)(kk - len), '0') + ".0";
    } else if (0 < kk && kk <= 16) {
        o = digits.substr(0, (size_t)kk) + "." + digits.substr((size_t)kk);
    } else if (-5 < kk && kk <= 0) {
        o = "0." + std::string((size_t)(-kk), '0') + digits;
    } else if (len == 1) {
        o = digits + "e" + std::to_string(kk - 1);
    } else {
        o = digits.substr(0, 1) + "." + digits.substr(1) + "e" + std::to_string(kk - 1);
    }
    return (neg ? "-" : "") + o;
}

static std::string opt_str(const std::optional<std::string> &v) { return v ? json_escape(*v) : "null"; }
static std::string str_array(const std::vector<std::string> &v, const std::string &indent) {
    if (v.empty()) return "[]";
    std::string o = "[\n";
    for (size_t i = 0; i < v.size(); i++) o += indent + "  " + json_escape(v[i]) + (i + 1 < v.size() ? ",\n" : "\n");
    return o + indent + "]";
}

ScrubbyReport ScrubbyReport::create(const Scrubby &s, bool header) {  // report.rs:24-57
    ReadDifference rd;
    rd.input_reads = s.input;
    rd.output_reads = s.output;
    rd.device = s.device;
    Difference diff = rd.compute();
    ScrubbyReport r;
    r.version = CRATE_VERSION;
    time_t now = time(nullptr);
    struct tm tmv;
    gmtime_r(&now, &tmv);
    char date[32];
    strftime(date, sizeof(date), "%Y-%m-%dT%H:%M:%SZ", &tmv);  // to_rfc3339_opts(Secs, true)
    r.date = date;
    r.command = s.config.command ? *s.config.command : "";
    r.input = s.input;
    r.output = s.output;
    r.reads_in = diff.reads_in;
    r.reads_out = diff.reads_out;
    r.reads_removed = s.extract ? 0 : diff.difference;
    r.reads_extracted = s.extract ? diff.difference : 0;
    r.scrubby = &s;
    if (s.read_ids) diff.write_read_ids(*s.read_ids, header);
    if (s.json) {
        std::string js = r.to_json_string();
        write_file(*s.json, (const uint8_t *)js.data(), js.size(), 6);
    }
    return r;
}

std::string ScrubbyReport::to_json_string() const {  // struct order of report.rs:11-22 and :72-88
    const ScrubbyConfig &c = scrubby->config;
    std::ostringstream o;
    o << "{\n";
    o << "  \"version\": " << json_escape(version) << ",\n";
    o << "  \"date\": " << json_escape(date) << ",\n";
    o << "  \"command\": " << json_escape(command) << ",\n";
    o << "  \"input\": " << str_array(input, "  ") << ",\n";
    o << "  \"output\": " << str_array(output, "  ") << ",\n";
    o << "  \"reads_in\": " << reads_in << ",\n";
    o << "  \"reads_out\": " << reads_out << ",\n";
    o << "  \"reads_removed\": " << reads_removed << ",\n";
    o << "  \"reads_extracted\": " << reads_extracted << ",\n";
    o << "  \"settings\": {\n";
    o << "    \"aligner\": " << (c.aligner ? json_escape(serde_name(*c.aligner)) : "null") << ",\n";
    o << "    \"classifier\": " << (c.classifier ? json_escape(serde_name(*c.classifier)) : "null") << ",\n";
    o << "    \"index\": " << opt_str(c.index) << ",\n";
    o << "    \"alignment\": " << opt_str(c.alignment) << ",\n";
    o << "    \"reads\": " << opt_str(c.reads) << ",\n";
    o << "    \"report\": " << opt_str(c.report) << ",\n";
    o << "    \"taxa\": " << str_array(c.taxa, "    ") << ",\n";
    o << "    \"taxa_direct\": " << str_array(c.taxa_direct, "    ") << ",\n";
    o << "    \"classifier_args\": " << opt_str(c.classifier_args) << ",\n";
    o << "    \"aligner_args\": " << opt_str(c.aligner_args) << ",\n";
    o << "    \"preset\": " << (c.preset ? json_escape(serde_name(*c.preset)) : "null") << ",\n";
    o << "    \"min_len\": " << c.min_query_length << ",\n";
    o << "    \"min_cov\": " << format_f64(c.min_query_coverage) << ",\n";
    o << "    \"min_mapq\": " << (unsigned)c.min_mapq << ",\n";
    o << "    \"extract\": " << (scrubby->extract ? "true" : "false") << "\n";
    o << "  }\n}";
    return o.str();
}

}  // namespace scrubby

// ---------------------------------------------------------------------------------------------- test shim
// plain C entry points so that the CPU test-suite can drive the host logic through ctypes
extern "C" {

// taxids joined with '\n' into a malloc'ed buffer; returns 0 or 100 + ScrubbyError::Kind
int scrubby_host_taxids_from_report(const uint8_t *buf, size_t n, const char *const *taxa, size_t n_taxa,
                                    const char *const *direct, size_t n_direct, char **out, size_t *out_n,
                                    uint64_t *err_line) {
    try {
        std::vector<std::string> t(taxa, taxa + n_taxa), d(direct, direct + n_direct);
        std::vector<std::string> ids = scrubby::get_taxids_from_report_bytes(buf, n, t, d);
        std::string s;
        for (auto &i : ids) s += i + "\n";
        *out = (char *)malloc(s.size() + 1);
        memcpy(*out, s.data(), s.size());
        *out_n = s.size();
        return 0;
    } catch (const scrubby::ScrubbyError &e) {
        if (err_line) *err_line = e.index;
        return 100 + (int)e.kind;
    }
}

void scrubby_host_free(void *p) { free(p); }

// niffler::get_reader's role (magic-byte sniffing + inflate; BGZF members on all host threads): the decoded bytes of
// a file in a malloc'ed buffer; returns 0 or 100 + ScrubbyError::Kind
int scrubby_host_read_file(const char *path, uint8_t **out, size_t *out_n) {
    try {
        std::vector<uint8_t> v = scrubby::read_file(path);
        *out = (uint8_t *)malloc(v.size() + 1);
        if (!v.empty()) memcpy(*out, v.data(), v.size());
        *out_n = v.size();
        return 0;
    } catch (const scrubby::ScrubbyError &e) {
        return 100 + (int)e.kind;
    }
}

// FastqCleaner::clean_reads' gzip pipeline (clean_fastq_gz_stream) with the shard call supplied by the caller: the CPU
// tests pass a stand-in built on the oracle, so the chunking, the newline / CRLF bookkeeping, the halo growth, the error
// indices and both writers are exercised without a GPU.  *handled = 0: the input is not a plain-gzip FASTQ.
typedef int (*scrubby_shard_cb)(const uint8_t *in, size_t n_in, size_t own_len, uint64_t newlines_before, int is_first,
                                int is_last, int crlf, uint8_t *out, size_t cap, size_t *n_out, sgpu_counts *counts);
int scrubby_host_stream_clean(const char *input, const char *output, size_t chunk, size_t halo, scrubby_shard_cb cb,
                              int *handled, uint64_t *err_index) {
    try {
        scrubby::ShardFn fn = cb;
        *handled = scrubby::clean_fastq_gz_stream(input, output, fn, chunk, halo) ? 1 : 0;
        return 0;
    } catch (const scrubby::ScrubbyError &e) {
        if (err_index) *err_index = e.index;
        return 100 + (int)e.kind;
    }
}

// the same for FASTA (clean_fasta_gz_stream) with a sgpu_clean_fasta_shard-shaped callback.  *handled = 0: the input is
// not a gzip FASTA
typedef int (*scrubby_fasta_shard_cb)(const uint8_t *in, size_t n_in, size_t own_len, int is_first, int is_last,
                                      int le_before, uint8_t *out, size_t cap, size_t *n_out, sgpu_counts *counts,
                                      int *le_own);
int scrubby_host_stream_clean_fasta(const char *input, const char *output, size_t chunk, size_t halo,
                                    scrubby_fasta_shard_cb cb, int *handled, uint64_t *err_index) {
    try {
        scrubby::FastaShardFn fn = cb;
        *handled = scrubby::clean_fasta_gz_stream(input, output, fn, chunk, halo) ? 1 : 0;
        return 0;
    } catch (const scrubby::ScrubbyError &e) {
        if (err_index) *err_index = e.index;
        return 100 + (int)e.kind;
    }
}

// the two string encoders of the report writers (serde_json string escaping, report.rs:60; csv crate quoting with
// QuoteStyle::Necessary and a tab delimiter, utils.rs:207-216): which = 0 JSON, 1 TSV field.  Returns the length or -1.
int scrubby_host_encode_string(int which, const char *in, size_t n, char *out, size_t cap) {
    const std::string s = which == 0 ? scrubby::json_escape(std::string(in, n)) : scrubby::csv_field(std::string(in, n));
    if (s.size() > cap) return -1;
    memcpy(out, s.data(), s.size());
    return (int)s.size();
}

// report JSON of a classifier / alignment run with the given counts (date passed in): layout test
int scrubby_host_format_f64(double v, char *out, size_t cap) {
    std::string s = scrubby::format_f64(v);
    if (s.size() + 1 > cap) return -1;
    memcpy(out, s.c_str(), s.size() + 1);
    return (int)s.size();
}

}  // extern "C"
