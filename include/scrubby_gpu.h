/*
 * scrubby_gpu.h -- C ABI of libscrubby_gpu.so: the B200 (sm_100a) depletion hot path.
 *
 * The reference (esteinig/scrubby 1.0.2, pure Rust) has no FFI of its own; the seams
 * this library sits behind are the Rust functions cited on each entry point below
 * (file:line under the reference's src/).  INTEGRATION.md shows the `extern "C"`
 * block + build.rs a maintainer would add to call them from cleaner.rs /
 * alignment.rs / classifier.rs / utils.rs.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Every function returns an sgpu_status
 *    (0 = ok); none aborts.  Would-be panics of the reference (fields[] index out of
 *    bounds) are reported as SGPU_ERR_WOULD_PANIC.
 *  - Buffers hold DECOMPRESSED bytes.  gz/bz2/xz sniffing and .gz writing stay in
 *    the host stage (utils.rs:56-74, niffler), outside the timed region.
 *  - `*_dev` variants take device pointers (cudaMalloc / torch tensors) on the
 *    context's device and enqueue on the context's stream; the plain variants take
 *    host pointers and perform the H2D / D2H copies themselves.
 *  - A context belongs to one device (one process per GPU).  An idset is immutable
 *    once built and may be shared by concurrent cleaners (cleaner.rs:238-248 runs
 *    the two mate files on two threads against one &HashSet); calls on ONE context
 *    are serialised by the library, so use one context per host thread for overlap.
 *  - There is no CPU fallback: without a CUDA device sgpu_ctx_create fails with
 *    SGPU_ERR_CUDA.
 */
#ifndef SCRUBBY_GPU_H
#define SCRUBBY_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGPU_ABI_VERSION 2

typedef enum {
    SGPU_OK = 0,
    SGPU_ERR_IO = 1,                    /* ScrubbyError::IoError (error.rs:14): invalid UTF-8 in BufRead::lines */
    SGPU_ERR_NIFFLER = 2,               /* ScrubbyError::NifflerError (error.rs:20); host stage only */
    SGPU_ERR_FASTQ_INVALID_START = 3,   /* NeedletailParseError (error.rs:23): record does not start with '@' */
    SGPU_ERR_FASTQ_INVALID_SEPARATOR = 4, /* ... separator line does not start with '+' */
    SGPU_ERR_FASTQ_UNEQUAL_LENGTHS = 5, /* ... sequence and quality lengths differ */
    SGPU_ERR_FASTQ_UNEXPECTED_END = 6,  /* ... truncated last record */
    SGPU_ERR_FASTQ_UNKNOWN_FORMAT = 7,  /* ... first byte is neither '@' nor '>' */
    SGPU_ERR_RECORD_NAME_UTF8 = 8,      /* ScrubbyError::RecordNameUtf8Error (error.rs:41) from get_id */
    SGPU_ERR_FASTQ_HEADER = 9,          /* ScrubbyError::NeedletailFastqHeader (error.rs:53) */
    SGPU_ERR_PAF_INTEGER = 10,          /* ScrubbyError::PafRecordIntegerError (error.rs:47) */
    SGPU_ERR_WOULD_PANIC = 11,          /* reference indexes a missing column: alignment.rs:248-259, classifier.rs:412-415,508-513 */
    SGPU_ERR_KRAKEN_REPORT_READS = 12,  /* KrakenReportReadFieldConversion (error.rs:142) */
    SGPU_ERR_KRAKEN_REPORT_DIRECT = 13, /* KrakenReportDirectReadFieldConversion (error.rs:144) */
    SGPU_ERR_KRAKEN_REPORT_PARENT = 14, /* KrakenReportTaxonParent (error.rs:140) */
    SGPU_ERR_FASTA_UNSUPPORTED = 15,    /* a shard of '>' input given to sgpu_fastq_ids_shard_dev: FASTA shards go to sgpu_*fasta*_shard* */
    SGPU_ERR_CUDA = 16,                 /* CUDA runtime failure / no device; sgpu_last_cuda_error() has the text */
    SGPU_ERR_NOMEM = 17,
    SGPU_ERR_INVALID_ARG = 18,
    SGPU_ERR_CAPACITY = 19,             /* an output buffer is too small; required sizes are returned */
    SGPU_ERR_KEY_TOO_LONG = 20,         /* a read id of 16 MiB or more */
    SGPU_ERR_HALO = 21,                 /* shard: the last owned record does not end inside the buffer */
    SGPU_ERR_SAM_RECORD = 22,           /* a SAM line htslib's sam_parse1 rejects (rust_htslib error through `result?`, alignment.rs:131) */
    SGPU_ERR_BAM_RECORD = 23,           /* a BAM header / record htslib's bam_hdr_read / bam_read1 rejects (bad magic, truncated or inconsistent) */
    SGPU_ERR_NOT_SHARDABLE = 25,        /* sgpu_idset_assemble_dev: the evidence holds ids of 16 bytes and more, or more keys than the virtual
                                           pages were sized for: replicate the evidence and build the set on every rank instead */
    SGPU_ERR_PHASE_UNKNOWN = 24         /* shard called with SGPU_NEWLINES_UNKNOWN that the single-pass kernel cannot take (not canonical FASTQ,
                                           no "\n+\n" in sight ...): nothing was produced, call again with the exact newlines_before / crlf */
} sgpu_status;

/* `newlines_before` of a shard whose line phase has not been exchanged yet (see sgpu_clean_fastq_shard_dev) */
#define SGPU_NEWLINES_UNKNOWN UINT64_MAX

typedef struct sgpu_ctx sgpu_ctx;     /* device, stream, scratch arena */
typedef struct sgpu_idset sgpu_idset; /* exact read-id set (HashSet<String>) resident in HBM */

typedef struct {
    uint64_t reads_in;      /* records parsed from the input                                   */
    uint64_t reads_out;     /* records written (clean) / records of the output file (diff)     */
    uint64_t difference;    /* diff: input records whose id is absent from the output          */
    uint64_t error_record;  /* 0-based record (FASTQ) or line (evidence) index of the error    */
    uint32_t crlf;          /* 1: first record ends its header with CRLF, output uses CRLF     */
    uint32_t empty_input;   /* 1: fewer than 5 bytes => "empty" (utils.rs:359-375); no output  */
    uint32_t path;          /* 1: fused single-pass kernel produced the result, 2: general path */
    uint32_t speculated;    /* 1: the shard's line phase was speculated (SGPU_NEWLINES_UNKNOWN): verify it  */
    uint64_t own_newlines;  /* speculated shards: '\n' bytes in the owned range [0, own_len)                */
    uint64_t lead_newlines; /* speculated shards: '\n' bytes before the first record the shard produced    */
} sgpu_counts;

/* ---- context ------------------------------------------------------------------- */
sgpu_status sgpu_ctx_create(int device, sgpu_ctx **out);
void sgpu_ctx_destroy(sgpu_ctx *);
/* enqueue on a caller-owned cudaStream_t (e.g. torch's current stream); NULL = own stream.
 * The default stream is named by cudaStreamLegacy ((cudaStream_t)0x1). */
sgpu_status sgpu_ctx_set_stream(sgpu_ctx *, void *cuda_stream);
/* 0: auto (fused kernel when the input is canonical, else general); 1: force the general path */
sgpu_status sgpu_ctx_set_mode(sgpu_ctx *, int mode);
sgpu_status sgpu_ctx_sync(sgpu_ctx *);
const char *sgpu_strerror(int status);
const char *sgpu_last_cuda_error(void);
int sgpu_abi_version(void);
/* number of kernel launches issued by this context so far (bench.py's gpu_launches) */
uint64_t sgpu_ctx_launch_count(const sgpu_ctx *);
/* measurement aid: time every fused-kernel launch with CUDA events on the launching stream.
 * sgpu_ctx_fused_stats synchronises, returns the summed device time, the launch count and the
 * algorithmic bytes (input + every output byte produced) of those launches, and resets them. */
sgpu_status sgpu_ctx_set_profiling(sgpu_ctx *, int on);
sgpu_status sgpu_ctx_fused_stats(sgpu_ctx *, double *ms, uint64_t *launches, uint64_t *alg_bytes);

/* ---- evidence -> read-id set ---------------------------------------------------- */
/* ReadAlignment::from_paf, alignment.rs:84-114 (+ PafRecord::from_str :244-263, predicate :102-104;
 * same loop as cleaner.rs:669-678).  PAF and GAF share it (alignment.rs:41,49-50). */
sgpu_status sgpu_idset_from_paf(sgpu_ctx *, const uint8_t *buf, size_t n, uint64_t min_len,
                                double min_cov, uint8_t min_mapq, sgpu_idset **out,
                                uint64_t *err_line);
sgpu_status sgpu_idset_from_paf_dev(sgpu_ctx *, const uint8_t *d_buf, size_t n, uint64_t min_len,
                                    double min_cov, uint8_t min_mapq, sgpu_idset **out,
                                    uint64_t *err_line);
/* ReadAlignment::from_bam, alignment.rs:117-146 (+ BamRecord::from / qalen_from_cigar / query_coverage
 * :154-211; `htslib` feature) for TEXT SAM: header lines skipped, unmapped records skipped, aligned length =
 * sum of CIGAR M and I, query length = SEQ length, the PAF predicate.  (Binary BAM: sgpu_idset_from_bam below.)  The sam_parse1 behaviour restated here (htslib is an un-vendored
 * dependency of the reference; parity unpinned):
 *   - lines split on '\n', one trailing '\r' dropped; lines starting with '@' are header lines (skipped);
 *   - a record has >= 11 tab-separated fields: QNAME FLAG RNAME POS MAPQ CIGAR RNEXT PNEXT TLEN SEQ QUAL;
 *   - FLAG like strtol(.., 0): decimal, 0x hex or 0 octal, 0..65535; POS / PNEXT / TLEN signed decimal;
 *     MAPQ decimal 0..255; CIGAR "*" or (count op)+ with op in MIDNSHP=XB, count < 2^28;
 *   - SEQ "*" (length 0) or its byte length; with a CIGAR and a SEQ the CIGAR's query length (M I S = X)
 *     must equal it; QUAL "*" or as long as SEQ; any violation -> SGPU_ERR_SAM_RECORD at that line;
 *   - RNAME other than "*" is looked up among the SN: names of the header's @SQ lines (bam_name2id): with no @SQ
 *     line at all that is htslib's parse error "no SQ lines present in the header" -> SGPU_ERR_SAM_RECORD; a name the
 *     header does not declare makes the record unmapped ("unrecognized reference name; treated as unmapped");
 *   - unmapped = FLAG & 4, or RNAME "*" / undeclared, or POS < 1 (htslib sets BAM_FUNMAP for all of them): skipped;
 *   - QNAME must be valid UTF-8 (alignment.rs:187) -> SGPU_ERR_RECORD_NAME_UTF8.
 * Not restated: textual FLAG strings; @SQ lines without LN: (htslib rejects the header). */
sgpu_status sgpu_idset_from_sam(sgpu_ctx *, const uint8_t *buf, size_t n, uint64_t min_len,
                                double min_cov, uint8_t min_mapq, sgpu_idset **out,
                                uint64_t *err_line);
sgpu_status sgpu_idset_from_sam_dev(sgpu_ctx *, const uint8_t *d_buf, size_t n, uint64_t min_len,
                                    double min_cov, uint8_t min_mapq, sgpu_idset **out,
                                    uint64_t *err_line);
/* ReadAlignment::from_bam, alignment.rs:117-146 (+ BamRecord::from :180-197) for BINARY BAM records.  `buf` is the
 * BGZF-DECOMPRESSED BAM stream in host memory (BGZF blocks are concatenated gzip members: inflating them is a host
 * stage like gz for FASTQ; the C++ host's reader does it).  Restated from the BAM specification (SAMv1 4.2) and
 * htslib's bam_hdr_read / bam_read1 / bam_tag2cigar (un-vendored dependency; parity unpinned):
 *   - header: magic "BAM\1", l_text, text, n_ref, (l_name, name, l_ref) per reference; anything else ->
 *     SGPU_ERR_BAM_RECORD with *err_record = 0;
 *   - records: block_size (u32 LE) + block_size bytes; the data may end only at a record boundary; block_size >= 32,
 *     l_read_name >= 1, l_seq >= 0 and 32 + l_read_name + 4 n_cigar_op + (l_seq+1)/2 + l_seq <= block_size, else
 *     SGPU_ERR_BAM_RECORD at that record's index (the first failing record wins);
 *   - FLAG & 4 (unmapped): skipped before anything else is looked at (alignment.rs:132-134);
 *   - qname = the l_read_name - 1 bytes before the terminating NUL (rust_htslib Record::qname; a read_name without
 *     the NUL is taken whole: htslib appends it); must be UTF-8 -> SGPU_ERR_RECORD_NAME_UTF8;
 *   - aligned length = sum of M and I operation lengths (u32, wrapping), query length = l_seq; a record with the
 *     long-CIGAR placeholder (first op soft clip of l_seq, refID >= 0, pos >= 0) and a CG:B,I tag of >= n_cigar_op
 *     and < 2^29 entries takes its CIGAR from the tag (bam_tag2cigar); then the PAF predicate.
 * CRAM needs a reference-based decoder and is not built. */
sgpu_status sgpu_idset_from_bam(sgpu_ctx *, const uint8_t *buf, size_t n, uint64_t min_len,
                                double min_cov, uint8_t min_mapq, sgpu_idset **out,
                                uint64_t *err_record);
/* ReadAlignment::from_txt, alignment.rs:60-82: every line verbatim */
sgpu_status sgpu_idset_from_txt(sgpu_ctx *, const uint8_t *buf, size_t n, sgpu_idset **out,
                                uint64_t *err_line);
sgpu_status sgpu_idset_from_txt_dev(sgpu_ctx *, const uint8_t *d_buf, size_t n, sgpu_idset **out,
                                    uint64_t *err_line);
/* get_taxid_reads_kraken (style 0, classifier.rs:270-290) / get_taxid_reads_metabuli (style 1,
 * :308-328).  `taxids` is the HashSet<String> returned by get_taxids_from_report
 * (classifier.rs:124-252, computed on the host), passed as n_taxids byte strings. */
sgpu_status sgpu_idset_from_reads(sgpu_ctx *, const uint8_t *buf, size_t n, int style,
                                  const char *const *taxids, const size_t *taxid_lens,
                                  size_t n_taxids, sgpu_idset **out, uint64_t *err_line);
sgpu_status sgpu_idset_from_reads_dev(sgpu_ctx *, const uint8_t *d_buf, size_t n, int style,
                                      const char *const *taxids, const size_t *taxid_lens,
                                      size_t n_taxids, sgpu_idset **out, uint64_t *err_line);
/* a caller-built HashSet<String> (the `read_ids: &HashSet<String>` argument of
 * FastqCleaner::clean_reads, cleaner.rs:731): ids[i] has lens[i] bytes */
sgpu_status sgpu_idset_from_ids(sgpu_ctx *, const char *const *ids, const size_t *lens, size_t n,
                                sgpu_idset **out);
sgpu_status sgpu_idset_new(sgpu_ctx *, sgpu_idset **out); /* empty set (diff accumulator) */
uint64_t sgpu_idset_len(const sgpu_idset *);              /* HashSet::len */
sgpu_status sgpu_idset_contains(sgpu_ctx *, const sgpu_idset *, const char *id, size_t len,
                                int *found);
/* sorted (bytewise) ids, each followed by '\n', in a malloc'ed buffer freed with sgpu_free */
sgpu_status sgpu_idset_dump(sgpu_ctx *, const sgpu_idset *, uint8_t **out, size_t *n);
void sgpu_idset_free(sgpu_idset *);
void sgpu_free(void *);

/* ---- FASTQ filter ---------------------------------------------------------------- */
/* FASTA input.  When the first byte is '>' needletail switches to its FASTA reader (utils.rs:377-383) and the same
 * clean_reads / get_difference loops run on those records; sgpu_clean_fastq{,_dev} and sgpu_diff{,_dev} follow on whole
 * files, and sgpu_clean_fasta_shard{,_dev} / sgpu_fasta_ids_shard_dev below on shards (the FASTQ shard entry points do
 * not take '>' input: the caller picks the entry point from byte 0).  needletail 0.5.1 fasta::Reader restated (parity unpinned): a
 * record runs from its '>' to the newline in front of the next "\n>" or to the end of the input; its
 * positions are its newlines, except that a newline on the input's LAST byte is only counted after another one, and
 * that without a trailing newline the end of the input closes the last line; id = trim_cr(start+1 .. first position),
 * raw_seq = trim_cr(first position + 1 .. last position) when there are >= 2 positions, else empty -- the inner line
 * breaks of a multi-line sequence are kept verbatim; a record without a position is SGPU_ERR_FASTQ_UNEXPECTED_END;
 * the line ending E comes from the first record whose bytes before its last position hold a newline (CRLF when that
 * newline follows a CR), records written before it use LF; output '>' id E raw_seq E. */
/* FastqCleaner::clean_reads, cleaner.rs:731-760 (loop :742-754) including needletail's
 * framing and re-serialisation and get_id (utils.rs:91-103).
 *   out_written : the bytes the reference writes to its output file
 *                 (kept records when reverse == 0, matched records when reverse != 0)
 *   out_other   : the complementary partition (may be NULL: not produced)
 * cap_* are the buffer capacities; n_* receive the produced sizes.  On a parse error
 * the records before the failing one are produced (the reference leaves them on disk)
 * and the error class is returned with counts->error_record set. */
sgpu_status sgpu_clean_fastq(sgpu_ctx *, const sgpu_idset *, const uint8_t *in, size_t n_in,
                             int reverse, uint8_t *out_written, size_t cap_written,
                             size_t *n_written, uint8_t *out_other, size_t cap_other,
                             size_t *n_other, sgpu_counts *counts);
sgpu_status sgpu_clean_fastq_dev(sgpu_ctx *, const sgpu_idset *, const uint8_t *d_in, size_t n_in,
                                 int reverse, uint8_t *d_out_written, size_t cap_written,
                                 size_t *n_written, uint8_t *d_out_other, size_t cap_other,
                                 size_t *n_other, sgpu_counts *counts);

/* One shard of a file cut at arbitrary byte offsets (multi-GPU, SURVEY 8e).  The buffer holds
 * the shard's own bytes [0, own_len) followed by a halo; the shard produces exactly the
 * records that START inside [0, own_len).  `newlines_before` is the number of '\n' bytes in
 * the file before this shard (allgathered by the caller), `crlf` the file-level line ending
 * (decided by the first record, i.e. by shard 0), `is_last` marks the shard that holds EOF.
 * Concatenating the shards' outputs in order is byte-identical to the unsharded call.
 * Only the is_last shard applies the end-of-file rules (a last record without a newline, a tail of blank lines); any
 * other shard that finds fewer than four newlines after a record start it owns reports SGPU_ERR_HALO.  A caller must
 * therefore never hand a buffer that reaches EOF to a shard that is not the last one: when own range + halo would reach
 * EOF, that shard owns the rest of the file (own_len = n_in, is_last = 1) and the later ranks own nothing
 * (scrubby_b200/dist.py: plan_shards does exactly that).
 *
 * One pass without a prior newline count (round 2): pass newlines_before = SGPU_NEWLINES_UNKNOWN (and crlf = -1) on
 * every shard but the first.  The shard then SPECULATES its line phase from the first "\n+\n" among its first four
 * newlines, runs the single-pass kernel and returns counts->{speculated = 1, own_newlines, lead_newlines}.  The caller
 * all-gathers own_newlines (a few bytes per shard, AFTER the kernels instead of a pass over the file before them) and
 * accepts shard r iff (sum of own_newlines of the shards before r + lead_newlines_r) % 4 == 0 and shard 0 reported
 * crlf == 0; otherwise -- or when the call returned SGPU_ERR_PHASE_UNKNOWN -- the shard is run again with the exact
 * values.  The first shard may also be called with crlf = -1: it decides the line ending itself (counts->crlf). */
sgpu_status sgpu_clean_fastq_shard_dev(sgpu_ctx *, const sgpu_idset *, const uint8_t *d_in,
                                       size_t n_in, size_t own_len, uint64_t newlines_before,
                                       int is_first, int is_last, int crlf, int reverse,
                                       uint8_t *d_out_written, size_t cap_written,
                                       size_t *n_written, uint8_t *d_out_other, size_t cap_other,
                                       size_t *n_other, sgpu_counts *counts);
/* The same shard contract on HOST buffers (pinned memory for full PCIe rate): the shard goes through the device in
 * chunks, the host->device copy of chunk k+1, the kernels of chunk k and the device->host copy of chunk k-1 overlapped
 * (what sgpu_clean_fastq does for a whole file).  With SGPU_NEWLINES_UNKNOWN the first chunk speculates, the later chunks
 * continue from its phase; counts->{own_newlines, lead_newlines} cover the whole shard. */
sgpu_status sgpu_clean_fastq_shard(sgpu_ctx *, const sgpu_idset *, const uint8_t *in, size_t n_in, size_t own_len,
                                   uint64_t newlines_before, int is_first, int is_last, int crlf, int reverse,
                                   uint8_t *out_written, size_t cap_written, size_t *n_written,
                                   uint8_t *out_other, size_t cap_other, size_t *n_other, sgpu_counts *counts);
/* One shard of a FASTA file cut at arbitrary byte offsets (the rules above, restated per shard).  The buffer holds the
 * shard's own bytes [0, own_len) followed by a halo.
 *   Ownership (as for FASTQ shards: no look-behind byte is needed): a record starts at byte 0 of the file or at any '>'
 *     that follows a '\n'.  The first shard owns the starts in [0, own_len], any other shard the starts p in
 *     [1, own_len] with buf[p-1] == '\n' (a start exactly at own_len belongs to this shard: the next one cannot see
 *     the byte in front of its byte 0).  An owned record ends at the newline in front of the next record start, which
 *     may lie in the halo.
 *   Halo: a shard that is not last and does not hold the start of the record after its last owned one returns
 *     SGPU_ERR_HALO.  Only the is_last shard applies the end-of-file rules (the last-byte newline, an unterminated last
 *     line, UnexpectedEnd); the caller must never hand a buffer that reaches EOF to another shard (see FASTQ shards).
 *   Line ending: the deciding record is the first record whose bytes before its last position hold a newline; it fixes
 *     E, and records before it are written with LF.  le_before = -1: nothing decided before this shard, its own first
 *     deciding record decides (always the case for the first shard); 0 / 1: an earlier shard decided LF / CRLF, and
 *     every record of this shard uses it.  *le_own returns what this shard's own first deciding record (before an
 *     error) says, -1 when it has none, whatever le_before was: shard k+1's le_before is le_before(k) when that was
 *     decided, else le_own(k).  counts->crlf is the E this shard wrote with.
 *   Errors: class and record index (counts->error_record) are local to the shard; the records before the error are
 *     produced.  Records are counted as in the whole-file call.
 *   Arguments: d_in 16-byte aligned; is_first requires le_before == -1 and a first byte '>' (else SGPU_ERR_INVALID_ARG:
 *     the caller chose the wrong entry point); the fewer-than-5-bytes empty-input rule applies only to a shard that is
 *     both first and last.
 * A whole file is the shard (own_len = n_in, is_first = 1, is_last = 1, le_before = -1). */
sgpu_status sgpu_clean_fasta_shard_dev(sgpu_ctx *, const sgpu_idset *, const uint8_t *d_in, size_t n_in, size_t own_len,
                                       int is_first, int is_last, int le_before, int reverse,
                                       uint8_t *d_out_written, size_t cap_written, size_t *n_written,
                                       uint8_t *d_out_other, size_t cap_other, size_t *n_other,
                                       sgpu_counts *counts, int *le_own);
/* The same on HOST buffers: the shard goes through the device in chunks with the three-stream overlap of
 * sgpu_clean_fastq_shard, each chunk starting from the line-ending state of the one before (exact, nothing is
 * speculated).  sgpu_clean_fastq on a host FASTA file takes the same path. */
sgpu_status sgpu_clean_fasta_shard(sgpu_ctx *, const sgpu_idset *, const uint8_t *in, size_t n_in, size_t own_len,
                                   int is_first, int is_last, int le_before, int reverse,
                                   uint8_t *out_written, size_t cap_written, size_t *n_written,
                                   uint8_t *out_other, size_t cap_other, size_t *n_other,
                                   sgpu_counts *counts, int *le_own);
/* '\n' count of a device buffer (the per-shard figure that is allgathered) */
sgpu_status sgpu_count_newlines_dev(sgpu_ctx *, const uint8_t *d_buf, size_t n, uint64_t *count);

/* ---- diff / report counts -------------------------------------------------------- */
/* One shard of either loop of ReadDifference::get_difference (utils.rs:259-267 collects the output file's ids,
 * :269-283 tests the input file's ids) for multi-GPU runs (SURVEY 8e): the ids of the records that START in the
 * owned range of the buffer (same shard convention as sgpu_clean_fastq_shard_dev) and are absent from `probe`
 * (NULL: every record) are inserted into `into` (NULL: count only).  counts->reads_in += records,
 * counts->difference += picked records; both accumulate so that shards and file pairs can share one struct. */
sgpu_status sgpu_fastq_ids_shard_dev(sgpu_ctx *, const sgpu_idset *probe, const uint8_t *d_buf, size_t n_buf,
                                     size_t own_len, uint64_t newlines_before, int is_first, int is_last,
                                     sgpu_idset *into, sgpu_counts *counts);
/* sgpu_fastq_ids_shard_dev for FASTA shards (the ownership and halo rules of sgpu_clean_fasta_shard_dev; the line
 * ending plays no part): ids of the owned records absent from `probe` (NULL: all) go into `into`;
 * counts->reads_in += records, counts->difference += picked records. */
sgpu_status sgpu_fasta_ids_shard_dev(sgpu_ctx *, const sgpu_idset *probe, const uint8_t *d_buf, size_t n_buf,
                                     size_t own_len, int is_first, int is_last, sgpu_idset *into, sgpu_counts *counts);
/* ReadDifference::get_difference, utils.rs:250-285, for ONE (input, output) file pair:
 * counts->{reads_in, reads_out, difference} are incremented (+=) and the ids absent from the
 * output are inserted into *diff_ids (created when *diff_ids == NULL), so calling it once
 * per pair reproduces the loop at utils.rs:256. */
sgpu_status sgpu_diff(sgpu_ctx *, const uint8_t *in, size_t n_in, const uint8_t *out, size_t n_out,
                      sgpu_counts *counts, sgpu_idset **diff_ids);
sgpu_status sgpu_diff_dev(sgpu_ctx *, const uint8_t *d_in, size_t n_in, const uint8_t *d_out,
                          size_t n_out, sgpu_counts *counts, sgpu_idset **diff_ids);

/* ---- multi-GPU plumbing: replicate a set over NCCL ---------------------------------- */
typedef struct {
    void *d_table;        /* device pointer: capacity 16-byte slots, 128-byte aligned */
    uint64_t table_bytes;
    void *d_arena;        /* device pointer: key bytes of ids longer than 15  */
    uint64_t arena_bytes;
    uint64_t capacity;    /* slots (a multiple of 8: 128-byte buckets)        */
    uint64_t count;       /* distinct ids                                     */
    uint64_t has_empty;   /* the empty string is a member (txt blank line)    */
} sgpu_idset_image;
/* Sharded set build (round 2): every rank turns ITS byte range of the evidence into slot images grouped by virtual page
 * (step 1), the ranks pull each other's lists over NVLink (symmetric memory: plain device pointers here), and every
 * rank assembles the whole table from all lists (step 2) -- the parse, the hashing and the partition are done once per
 * key across the box, only the 16-byte images travel, and ReadAlignment::from_txt's result (alignment.rs:60-82) is
 * the same set on every rank (cleaner.rs:236-254: one global set).
 *   d_buf      : the shard's own bytes [0, own_len) followed by a halo (the start of the next shard: a line of this
 *                shard may end there); 16-byte aligned.  starts_line: the byte before the buffer is '\n' (or the buffer
 *                starts the file) -- otherwise the first, partial line belongs to the previous shard.
 *   log2_vpages: virtual pages = 2^log2_vpages, the same on every rank (>= total keys / 410 for load 0.2).
 *   d_recs     : cap_recs x 16 bytes; d_vstart: (2^log2_vpages + 2) x u64 (exclusive starts, count, flags).
 * The call returns when the lists are final (stream synchronised): signal the other ranks then. */
sgpu_status sgpu_idset_partition_txt_dev(sgpu_ctx *, const uint8_t *d_buf, size_t n, size_t own_len, int starts_line,
                                         int is_last, uint32_t log2_vpages, void *d_recs, size_t cap_recs,
                                         uint64_t *d_vstart, uint64_t *n_recs, uint64_t *err_line);
/* step 2: n_parts (<= 8) lists, as device pointers valid on this device.  SGPU_ERR_NOT_SHARDABLE: fall back to the
 * replicated build. */
sgpu_status sgpu_idset_assemble_dev(sgpu_ctx *, int n_parts, const void *const *d_recs, const uint64_t *const *d_vstart,
                                    uint32_t log2_vpages, sgpu_idset **out);

/* the set's keys as an unsorted one-column list ("id\n" per key; a blank line for the empty id) written to a
 * caller-owned DEVICE buffer.  *n = bytes needed / written; SGPU_ERR_CAPACITY (with *n set) when d_out is NULL
 * or cap < *n.  Exchange format of the multi-GPU diff: ReadDifference::get_difference (utils.rs:250-285) keeps
 * one HashSet per output file and one global diff set; across ranks they are united by an all-gather of these
 * lists followed by sgpu_idset_from_txt_dev on the concatenation (exact for FASTQ ids: tokens hold no
 * whitespace and are valid UTF-8, so BufRead::lines returns them verbatim). */
sgpu_status sgpu_idset_keys_dev(sgpu_ctx *, const sgpu_idset *, uint8_t *d_out, size_t cap, size_t *n);
/* the set's device buffers (still owned by the set): broadcast them, then import */
sgpu_status sgpu_idset_export(const sgpu_idset *, sgpu_idset_image *img);
/* builds a set on this context's device by COPYING the image's device buffers */
sgpu_status sgpu_idset_import(sgpu_ctx *, const sgpu_idset_image *img, sgpu_idset **out);

#ifdef __cplusplus
}
#endif
#endif /* SCRUBBY_GPU_H */
