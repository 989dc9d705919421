// scrubby_host.hpp -- C++ host side of the drop-in: mirrors the reference's Rust interface for the
// depletion path (same names, argument meaning and error behaviour) on top of the C ABI in
// include/scrubby_gpu.h.  The reference is Rust; no Rust toolchain exists in this image, so the
// host is written in C++ (see INTEGRATION.md for the Rust-side binding a maintainer would add).
//
//   reference item (file:line under /root/reference/src)          -> here
//   ScrubbyError                     error.rs:7-171               -> scrubby::ScrubbyError
//   CompressionExt / get_fastx_writer utils.rs:14-74              -> scrubby::Compression, write_file
//   is_file_empty / parse_fastx_file_with_check utils.rs:359-383  -> scrubby::read_file (+ C ABI sniffing)
//   ReadAlignment::from              alignment.rs:33-58           -> scrubby::ReadAlignment::from
//   get_taxids_from_report           classifier.rs:124-252        -> scrubby::get_taxids_from_report (host only)
//   get_taxid_reads_kraken/_metabuli classifier.rs:270-328        -> scrubby::get_taxid_reads_*
//   FastqCleaner / Cleaner::clean_reads cleaner.rs:236-254,691-760 -> scrubby::FastqCleaner, Cleaner
//   ReadDifference / Difference      utils.rs:175-357             -> scrubby::ReadDifference, Difference
//   ScrubbyReport / ScrubbySettings  report.rs:11-108             -> scrubby::ScrubbyReport
//   Scrubby / ScrubbyConfig / enums  scrubby.rs:32-309            -> scrubby::Scrubby, Aligner, Classifier, Preset
#pragma once
#include <cstdint>
#include <functional>
#include <memory>
#include <optional>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/scrubby_gpu.h"

namespace scrubby {

constexpr const char *CRATE_VERSION = "1.0.2";  // clap crate_version!() of the reference (Cargo.toml)

// ---------------------------------------------------------------- errors (error.rs)
class ScrubbyError : public std::runtime_error {
   public:
    enum Kind {
        IoError, NifflerError, NeedletailParseError, RecordNameUtf8Error, PafRecordIntegerError,
        NeedletailFastqHeader, NoAlignerOrClassifierConfigured, AlignmentInputFormatNotRecognized,
        AlignmentInputFormatInvalid, MismatchedInputOutputLength, MissingTaxa, MissingClassifierIndex,
        MissingClassifierReadClassfications, MissingClassifierClassificationReport, MissingAlignment,
        EmptyInputOutput, InputOutputLengthExceeded, MissingClassifier, MissingInputReadFile,
        KrakenReportTaxonParent, KrakenReportReadFieldConversion, KrakenReportDirectReadFieldConversion,
        WouldPanic, Gpu, Unsupported,
        // `scrubby reads` (scrubby.rs:813-975 build, cleaner.rs:255-649 external tools)
        AlignerAndClassifierConfigured, AlignerAndClassifierIndexConfigured, MissingAlignmentIndex, MissingAlignmentIndexFile,
        MissingBowtie2IndexFiles, MissingClassifierIndexDirectory, MissingStrobealignIndexBaseFile, Minimap2PresetNotSupported,
        MinigraphPresetNotSupported, MissingMinimap2Preset, MissingMinigraphPreset, MissingAligner, AlignerDependencyMissing,
        ClassifierDependencyMissing, CommandExecutionFailed, CommandFailed
    };
    ScrubbyError(Kind k, const std::string &msg, uint64_t index = 0) : std::runtime_error(msg), kind(k), index(index) {}
    Kind kind;
    uint64_t index;  // record / line index where known
    // maps an sgpu_status onto the ScrubbyError variant the reference would raise
    static ScrubbyError from_status(int status, uint64_t index, const std::string &what);
};

// ---------------------------------------------------------------- enums (scrubby.rs:32-155, alignment.rs:15-23)
enum class Aligner { Bowtie2, Minimap2, Minigraph, Strobealign };
enum class Classifier { Kraken2, Metabuli };
enum class Preset { LrHq, Splice, SpliceHq, Asm, Asm5, Asm10, Asm20, Sr, Lr, MapPb, MapHifi, MapOnt, AvaPb, AvaOnt };
enum class AlignmentFormat { Sam, Bam, Cram, Paf, Txt, Gaf };
const char *serde_name(Aligner);        // "bowtie2" ... (serde rename)
const char *serde_name(Classifier);     // "kraken2", "metabuli"
const char *serde_name(Preset);         // variant names: "Sr", "MapOnt", ... (no rename in the reference)
const char *display_name(Preset);      // fmt::Display: "sr", "map-ont", "lr:hq", ... (what the aligner's -x gets)
std::optional<Classifier> parse_classifier(const std::string &);
std::optional<Aligner> parse_aligner(const std::string &);  // clap ValueEnum names
std::optional<Preset> parse_preset(const std::string &);    // clap ValueEnum names: kebab-case of the variants
std::optional<AlignmentFormat> parse_alignment_format(const std::string &);

// ---------------------------------------------------------------- config (scrubby.rs:159-309)
struct ScrubbyConfig {
    std::optional<Aligner> aligner;
    std::optional<Classifier> classifier;
    std::optional<std::string> index, alignment, reads, report;
    std::optional<std::string> aligner_index, classifier_index;  // set from `index` by validate_base_config (scrubby.rs:787-796)
    bool unpaired = false;                                       // scrubby.rs:381
    std::optional<unsigned> samtools_threads;                    // scrubby.rs:382 (None: 4, cleaner.rs:47)
    std::vector<std::string> taxa, taxa_direct;
    std::optional<std::string> classifier_args, aligner_args;
    std::optional<Preset> preset;
    bool paired_end = false;
    bool needletail_parallel = true;  // scrubby.rs:384
    uint64_t min_query_length = 0;
    double min_query_coverage = 0.0;
    uint8_t min_mapq = 0;
    std::optional<AlignmentFormat> alignment_format;
    std::optional<std::string> command;
};

struct Scrubby {
    std::vector<std::string> input, output;
    std::optional<std::string> json, workdir, read_ids;
    bool extract = false;
    unsigned threads = 4;  // terminal.rs:134-135
    ScrubbyConfig config;
    int device = 0;
    void clean() const;  // scrubby.rs:255-281
};

// validate_base_config (scrubby.rs:760-799) + build_classifier (:978-1006) / build_alignment (:1019-1038)
Scrubby build(Scrubby s);  // ScrubbyBuilder::build, scrubby.rs:813-975 (`scrubby reads`)
Scrubby build_classifier(Scrubby s);
Scrubby build_alignment(Scrubby s);

// ---------------------------------------------------------------- GPU handles (RAII over the C ABI)
class GpuContext {
   public:
    explicit GpuContext(int device = 0);
    ~GpuContext();
    GpuContext(const GpuContext &) = delete;
    sgpu_ctx *get() const { return ctx_; }
   private:
    sgpu_ctx *ctx_ = nullptr;
};

// HashSet<String> of read ids living in HBM
class ReadIdSet {
   public:
    ReadIdSet() = default;
    explicit ReadIdSet(sgpu_idset *h) : h_(h) {}
    ~ReadIdSet() { if (h_) sgpu_idset_free(h_); }
    ReadIdSet(ReadIdSet &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ReadIdSet &operator=(ReadIdSet &&o) noexcept { if (h_) sgpu_idset_free(h_); h_ = o.h_; o.h_ = nullptr; return *this; }
    ReadIdSet(const ReadIdSet &) = delete;
    sgpu_idset *get() const { return h_; }
    sgpu_idset **out() { return &h_; }
    uint64_t len() const { return sgpu_idset_len(h_); }
    std::vector<std::string> sorted(const GpuContext &) const;
   private:
    sgpu_idset *h_ = nullptr;
};

// ---------------------------------------------------------------- host I/O stage (niffler / needletail open)
enum class Compression { No, Gzip, Bzip, Lzma };
Compression compression_from_path(const std::string &path);         // utils.rs:27-36 (by extension, for writing)
std::vector<uint8_t> read_file(const std::string &path, size_t *raw_size = nullptr);  // magic-byte sniffing + inflate (niffler::get_reader)
std::vector<uint8_t> read_file(const std::string &path, bool *empty);  // + is_file_empty (utils.rs:359-375)
void write_file(const std::string &path, const uint8_t *data, size_t n, int gz_level);  // get_fastx_writer
// get_fastx_writer as a sink fed piece by piece (gz output: independent members deflated on all host threads)
class OutSink {
  public:
    OutSink(const std::string &path, int gz_level);
    ~OutSink();
    OutSink(const OutSink &) = delete;
    OutSink &operator=(const OutSink &) = delete;
    void append(const uint8_t *data, size_t n);  // creates the file on first use
    void close();                                // creates it when nothing was appended (an empty gzip member for .gz)
  private:
    void open();
    std::string path_;
    int level_;
    bool gz_ = false;
    void *f_ = nullptr;
    size_t total_ = 0;
};
// SURVEY 8f row 2: a plain-gzip FASTQ as a pipeline inflate -> filter -> deflate.  `shard` has sgpu_clean_fastq_shard's
// contract (minus context, set, mode and the second output).  false: not a plain-gzip FASTQ, nothing was done.
using ShardFn = std::function<int(const uint8_t *in, size_t n_in, size_t own_len, uint64_t newlines_before, int is_first,
                                  int is_last, int crlf, uint8_t *out, size_t cap, size_t *n_out, sgpu_counts *counts)>;
bool clean_fastq_gz_stream(const std::string &input, const std::string &output, const ShardFn &shard, size_t chunk, size_t halo);
// the same pipeline for a gzip / BGZF FASTA: `shard` has sgpu_clean_fasta_shard's contract (same omissions); chunk k+1
// starts from chunk k's line-ending state.  false: not a gzip FASTA (or fewer than 5 decoded bytes), nothing was done.
using FastaShardFn = std::function<int(const uint8_t *in, size_t n_in, size_t own_len, int is_first, int is_last,
                                       int le_before, uint8_t *out, size_t cap, size_t *n_out, sgpu_counts *counts,
                                       int *le_own)>;
bool clean_fasta_gz_stream(const std::string &input, const std::string &output, const FastaShardFn &shard, size_t chunk,
                           size_t halo);

// ---------------------------------------------------------------- alignment.rs
struct ReadAlignment {
    ReadIdSet aligned_reads;
    static ReadAlignment from(const GpuContext &, const std::string &path, uint64_t min_qaln_len, double min_qaln_cov,
                              uint8_t min_mapq, std::optional<AlignmentFormat> fmt);
    static ReadAlignment from_paf(const GpuContext &, const std::string &path, uint64_t, double, uint8_t);
    static ReadAlignment from_sam(const GpuContext &, const std::string &path, uint64_t, double, uint8_t);
    static ReadAlignment from_txt(const GpuContext &, const std::string &path);
};

// ---------------------------------------------------------------- classifier.rs
// host-only state machine: tiny, sequential, order dependent (SURVEY F10)
std::vector<std::string> get_taxids_from_report_bytes(const uint8_t *buf, size_t n, const std::vector<std::string> &taxa,
                                                      const std::vector<std::string> &taxa_direct);
std::vector<std::string> get_taxids_from_report(const std::string &report, const std::vector<std::string> &taxa,
                                                const std::vector<std::string> &taxa_direct);
ReadIdSet get_taxid_reads_kraken(const GpuContext &, const std::vector<std::string> &taxids, const std::string &reads);
ReadIdSet get_taxid_reads_metabuli(const GpuContext &, const std::vector<std::string> &taxids, const std::string &reads);

// ---------------------------------------------------------------- cleaner.rs
struct FastqCleaner {
    std::string input, output;
    static FastqCleaner from(const std::string &input, const std::string &output) { return {input, output}; }
    void clean_reads(const GpuContext &, const ReadIdSet &read_ids, bool reverse) const;  // cleaner.rs:731-760
};

// cleaner.rs:29-87: the samtools stages behind the SAM-emitting aligners (the depletion of those pipelines is done by
// samtools, not by the in-repo path)
struct SamtoolsConfig {
    std::string filter, fastq;
    static SamtoolsConfig from_scrubby(const Scrubby &);
    std::string get_pipeline() const { return filter + " | " + fastq; }
};

struct Cleaner {
    Scrubby scrubby;
    SamtoolsConfig samtools;
    static Cleaner from_scrubby(const Scrubby &s);  // cleaner.rs:110-123 (checks the external tool's presence)
    // external tools through `sh -c` (cleaner.rs:137-161, 255-649): the command strings are the reference's
    void run_aligner() const;
    void run_classifier() const;
    std::string kraken_command(const std::string &reads_out, const std::string &report_out) const;
    std::string metabuli_command(const std::string &dir) const;
    std::string aligner_command() const;
    void run_command(const std::string &cmd) const;                              // cleaner.rs:626-641
    ReadIdSet run_command_stdout_paf(const GpuContext &, const std::string &cmd) const;  // cleaner.rs:651-687
    void run_classifier_output() const;  // cleaner.rs:177-194
    void run_aligner_output() const;     // cleaner.rs:206-219
    void clean_reads(const ReadIdSet &read_ids) const;  // cleaner.rs:236-254 (two mate files on two threads)
    ReadIdSet parse_classifier_output(const GpuContext &, const std::string &report, const std::string &reads) const;
};

// ---------------------------------------------------------------- utils.rs:175-357
struct Difference {
    uint64_t reads_in = 0, reads_out = 0, difference = 0;
    std::vector<std::string> read_ids;  // sorted (the reference's order is HashSet-random)
    std::string to_json_string() const;
    void to_json(const std::string &output) const;
    void write_read_ids(const std::string &output, bool header) const;
};

struct ReadDifference {
    std::vector<std::string> input_reads, output_reads;
    std::optional<std::string> json, read_ids;
    int device = 0;
    static ReadDifference build(const std::vector<std::string> &in, const std::vector<std::string> &out,
                                std::optional<std::string> json, std::optional<std::string> read_ids);
    Difference compute() const;
    Difference get_difference() const;
};

// ---------------------------------------------------------------- report.rs
struct ScrubbyReport {
    std::string version, date, command;
    std::vector<std::string> input, output;
    uint64_t reads_in = 0, reads_out = 0, reads_removed = 0, reads_extracted = 0;
    const Scrubby *scrubby = nullptr;
    static ScrubbyReport create(const Scrubby &, bool header);
    std::string to_json_string() const;  // serde_json::to_string_pretty layout
};

std::string csv_field(const std::string &);  // csv crate, QuoteStyle::Necessary, tab delimiter
std::string json_escape(const std::string &);
std::string format_f64(double);  // serde_json (ryu) formatting of f64

}  // namespace scrubby
