/*
 * bnpk.h -- C-ABI of libbnpk.so, the B200 (sm_100a) k-mer hot path behind BioNumPy's API.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  The reference
 * (bionumpy @ 6773266) is pure Python/NumPy and has no FFI; the seam it offers for this path
 * is `bnp.set_backend(lib)` + `CupyFileReader` (bionumpy/__init__.py:47-94,
 * bionumpy/cupy_compatible/parser.py:10-17) and the `buffer_type=` plug-in protocol
 * (bionumpy/io/files.py:52-68, bionumpy/io/file_buffers.py:80-271).  Each entry point below
 * names the reference function(s) it replaces (paths relative to /root/reference/bionumpy/).
 * INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - all work is stream-ordered and asynchronous; nothing here synchronises unless stated;
 *   - inputs are borrowed and never written; outputs are caller-allocated;
 *   - return value: 0 = ok, >0 = cudaError_t, <0 = BNPK_E_* argument error;
 *     `bnpk_last_error()` gives a thread-local message;
 *   - kernels never trap on bad data: they fill a device-side `bnpk_status` block that the
 *     host reads when it chooses to (the Python layer turns it into the reference's
 *     FormatException(line_number) / EncodingError(offset)).
 */
#ifndef BNPK_H
#define BNPK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNPK_ABI_VERSION 2

/* argument errors */
#define BNPK_E_BADARG   (-1)
#define BNPK_E_K        (-2)   /* k outside 1..31            (sequence/kmers.py:69)        */
#define BNPK_E_WINDOW   (-3)   /* window_size < k            (sequence/minimizers.py:50)   */
#define BNPK_E_WORKSPACE (-4)  /* workspace too small                                      */
#define BNPK_E_BINS     (-5)

/* byte -> 2-bit code modes (encodings/alphabet_encoding.py:19-46,102-107).  Modes 0-2 are
 * closed-form bit tricks; mode 3 uses a caller-supplied 256-byte LUT (any 4-letter alphabet,
 * e.g. RNA "ACUG"; 255 = invalid), which is what AlphabetEncoding._lookup is. */
#define BNPK_ENC_ASCII_ACGT 0  /* DNAEncoding  A/a0 C/c1 G/g2 T/t3                        */
#define BNPK_ENC_ASCII_ACTG 1  /* ACTGEncoding A/a0 C/c1 T/t2 G/g3                        */
#define BNPK_ENC_CODES      2  /* bytes already are codes 0..3 (an encoded EncodedArray)  */
#define BNPK_ENC_LUT        3

/* histogram modes */
#define BNPK_HIST_AUTO   0     /* smem-privatised when bins fit, else global atomics       */
#define BNPK_HIST_SMEM   1
#define BNPK_HIST_GLOBAL 2

/* Device-side status block (int64[16]); zero/sentinel-initialised by bnpk_status_init. */
enum {
    BNPK_ST_N_LINES = 0,       /* newlines seen in the chunk                               */
    BNPK_ST_N_RECORDS = 1,     /* complete entries = n_lines / lines_per_entry             */
    BNPK_ST_N_COMPLETE_BYTES = 2, /* bytes up to and including the last kept newline
                                     (FileBuffer.size, io/one_line_buffer.py:67-69)        */
    BNPK_ST_BAD_HEADER_ENTRY = 3, /* min entry whose first byte != header char (INT64_MAX = none)
                                     -> FormatException(line_number = entry*lines_per_entry),
                                     io/one_line_buffer.py:155-173                         */
    BNPK_ST_BAD_PLUS_ENTRY = 4,   /* min entry whose 3rd line does not start with '+'
                                     -> line_number = 2 + entry*4, io/fastq_buffer.py:38-45 */
    BNPK_ST_BAD_BASE = 5,      /* min (row << 32 | position-in-row) of a byte outside the
                                  alphabet (INT64_MAX = none) -> EncodingError(offset),
                                  encodings/alphabet_encoding.py:34-46                     */
    BNPK_ST_N_BASES = 6,       /* sum of row lengths processed                             */
    BNPK_ST_N_VALUES = 7,      /* k-mers / minimizers produced or counted                  */
    BNPK_ST_N_LONG_ROWS = 8,   /* rows that did not fit a tile halo and took the long path */
    BNPK_ST_CR = 9,            /* 1 if '\r' trimming is active (io/one_line_buffer.py:175-182) */
    BNPK_ST_LAST_ROW_START = 10, /* internal: 1 + start of the last sequence line counted  */
    BNPK_ST_LAST_ROW_INDEX = 11, /* internal: 1 + its entry index                          */
    BNPK_ST_OVERFLOW = 12,     /* != 0: the fused pass met more long/odd rows than its scratch holds,
                                  or (malformed input) the record phase it read from a tile's own
                                  bytes was not the one the line count gives;
                                  the counts are incomplete -- use bnpk_line_split + bnpk_rows_kmer_count */
    BNPK_ST_WORDS = 16
};

int         bnpk_abi_version(void);
const char *bnpk_last_error(void);
/* number of SMs of the current device, for callers that size their own grids */
int         bnpk_sm_count(void);

/* Initialise a status block (device int64[BNPK_ST_WORDS]). */
int bnpk_status_init(int64_t *status, void *stream);

/* ---------------------------------------------------------------------------------------
 * K0  byte census.  Replaces nothing by itself; lets a caller size the outputs of
 *     bnpk_line_split exactly (the reference gets the size from np.flatnonzero's result,
 *     io/one_line_buffer.py:63).  count_out: device int64[1].
 * ------------------------------------------------------------------------------------- */
int bnpk_count_byte(const uint8_t *chunk, size_t n, uint8_t value, int64_t *count_out, void *stream);

/* ---------------------------------------------------------------------------------------
 * K1  line split.  Replaces OneLineBuffer.from_raw_buffer + _validate +
 *     _get_buffer_extractor (io/one_line_buffer.py:44-71,139-173), FastQBuffer._validate
 *     (io/fastq_buffer.py:38-45) and TextBufferExtractor.get_field_by_number
 *     (io/file_buffers.py:315-338) for ONE field of every complete entry.
 *
 *   lines_per_entry  4 (FASTQ) or 2 (two-line FASTA)
 *   field_line       which line of the entry (FASTQ: 0 name, 1 sequence, 3 quality)
 *   start_offset     bytes skipped at the line start (_line_offsets: 1 for the header line)
 *   header_char      '@' or '>';  check_plus: validate the '+' line (FASTQ)
 *   trim_cr          -1 = decide like the reference (first entries' header ends in '\r'),
 *                    0 = never, 1 = always
 *   starts/lens      out, capacity `max_rows` rows (extra rows are counted, not written)
 *   status           device int64[BNPK_ST_WORDS], pre-initialised
 *   workspace        device scratch of bnpk_tile_workspace_bytes(n) bytes (look-back state, deferred
 *                    long-row list and a 64 MiB table of 32-bit counters used by K6 for global
 *                    tables of 2^22..2^24 bins).  The entry points clear what they use on the first
 *                    slice of a chunk; bnpk_tile_workspace_reset zeroes all of it.
 * A single pass over the chunk (decoupled look-back over per-tile newline counts).
 * ------------------------------------------------------------------------------------- */
size_t bnpk_tile_workspace_bytes(size_t n);
int    bnpk_tile_workspace_reset(void *workspace, size_t workspace_bytes, void *stream);
int bnpk_line_split(const uint8_t *chunk, size_t n, int lines_per_entry, int field_line,
                    int start_offset, uint8_t header_char, int check_plus, int trim_cr,
                    int64_t *starts, int32_t *lens, size_t max_rows,
                    int64_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------
 * K6  fused count: raw FASTQ / two-line FASTA chunk bytes -> histogram, never materialising
 *     offsets, codes or hashes.  Replaces, for one chunk, the chain
 *       OneLineBuffer.from_raw_buffer            io/one_line_buffer.py:44-71
 *       change_encoding(..., DNAEncoding)        encoded_array.py:655-695 -> alphabet_encoding.py:34-46
 *       _get_dna_kmers                           sequence/kmers.py:105-126
 *       [get_minimizers]                         sequence/minimizers.py:20-54
 *       count_encoded(axis=None)                 sequence/count_encoded.py:150-188
 *     hist[b] += #{values v : v mod n_bins == b} over all COMPLETE entries of the chunk
 *     (n_bins = 4^k gives the reference's exact np.bincount; other n_bins = the hashed-bucket
 *     extension).  window_size = 0 counts k-mers, otherwise minimizers (window in bases).
 *     hist is int64[n_bins] and is ACCUMULATED into (zero it yourself for a fresh count).
 *     Chunks may be fed in slices: call with the same workspace/status and consecutive
 *     [slice_begin, slice_end) byte ranges of one resident buffer; `final` marks the last.
 * ------------------------------------------------------------------------------------- */
int bnpk_chunk_kmer_count(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end,
                          int final_slice, int lines_per_entry, uint8_t header_char, int check_plus,
                          int trim_cr, int enc_mode, const uint8_t *lut256, int k, int window_size,
                          int64_t n_bins, int hist_mode, int64_t *hist,
                          int64_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------
 * Row-driven kernels: operate on an arbitrary ragged view (base bytes, starts[R], lens[R])
 * -- what EncodedRaggedArray(data, RaggedView2(starts, lens)) is (io/file_buffers.py:335-338).
 * `offsets` are int64[R+1] exclusive prefix sums produced by bnpk_row_offsets.
 * ------------------------------------------------------------------------------------- */

/* offsets[r] = sum_{q<r} max(lens[q] - shrink, 0); offsets[R] = total.  (The ragged shape of
 * out[..., :-shrink], sequence/kmers.py:100, sequence/rollable.py:66.)  workspace as for K1
 * with n := R. */
int bnpk_row_offsets(const int32_t *lens, size_t n_rows, int shrink, int64_t *offsets,
                     void *workspace, size_t workspace_bytes, void *stream);

/* K2  change_encoding / AlphabetEncoding._encode (encoded_array.py:655-695,
 *     alphabet_encoding.py:34-46): gather the rows contiguously and map bytes to codes. */
int bnpk_rows_encode(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                     int enc_mode, const uint8_t *lut256, const int64_t *offsets, uint8_t *codes_out,
                     int64_t *status, void *stream);

/* K3  get_kmers / _get_dna_kmers + the ragged [..., :-k+1] (sequence/kmers.py:36-126):
 *     out[offsets[r] + i] = sum_j code[r][i+j] * 4^j  (int64), offsets from shrink = k-1. */
int bnpk_rows_kmer_hash(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                        int enc_mode, const uint8_t *lut256, int k, const int64_t *offsets,
                        int64_t *hashes_out, int64_t *status, void *stream);

/* K3' the reference's generic path for alphabets whose size is not 4 (KmerEncoder dot product,
 *     sequence/kmers.py:17-27,87): out[offsets[r] + i] = sum_j code[r][i+j] * alphabet_size^j in
 *     int64 (wrapping) arithmetic.  lut256 maps bytes to codes (255 = invalid), NULL = bytes are codes. */
int bnpk_rows_generic_hash(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                           const uint8_t *lut256, int alphabet_size, int k, const int64_t *offsets,
                           int64_t *hashes_out, int64_t *status, void *stream);

/* K4  get_minimizers (sequence/minimizers.py:20-54): out[offsets[r] + j] = min of the
 *     window_size-k+1 k-mer hashes of window j; offsets from shrink = window_size-1. */
int bnpk_rows_minimizers(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                         int enc_mode, const uint8_t *lut256, int k, int window_size,
                         const int64_t *offsets, int64_t *mins_out, int64_t *status, void *stream);

/* K3+K5 / K4+K5 fused on a ragged view: get_kmers|get_minimizers -> count_encoded(axis=None)
 *     without materialising the values (sequence/kmers.py:129-145 count_kmers). */
int bnpk_rows_kmer_count(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                         int enc_mode, const uint8_t *lut256, int k, int window_size,
                         int64_t n_bins, int hist_mode, int64_t *hist, int64_t *status, void *stream);

/* get_reverse_complement (sequence/dna.py:36-65: complement Lookup, then every row reversed):
 *     out[offsets[r] + i] = lut256[base[starts[r] + lens[r] - 1 - i]]; offsets from shrink = 0.  lut256 (device) is
 *     the complement table of the array's encoding (_get_complement_lookup, sequence/dna.py:13-34). */
int bnpk_rows_reverse_complement(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                 size_t n_rows, const uint8_t *lut256, const int64_t *offsets, uint8_t *out, void *stream);

/* EXTENSION (no reference counterpart; what Jellyfish --canonical does, benchmarks/rules/kmer_counting.smk:11):
 *     canonical k-mers = min(h, hash of the reverse complement of the same k-mer).  complement_xor is the
 *     complement as an XOR on a 2-bit code: 3 for "ACGT"-ordered alphabets (DNAEncoding), 2 for "ACTG"-ordered.
 *     Same outputs as bnpk_rows_kmer_hash / bnpk_rows_kmer_count otherwise. */
int bnpk_rows_kmer_hash_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                  size_t n_rows, int enc_mode, const uint8_t *lut256, int k, int complement_xor,
                                  const int64_t *offsets, int64_t *hashes_out, int64_t *status, void *stream);
int bnpk_rows_kmer_count_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                   size_t n_rows, int enc_mode, const uint8_t *lut256, int k, int complement_xor,
                                   int64_t n_bins, int hist_mode, int64_t *hist, int64_t *status, void *stream);
/*     The K6 fused count of canonical k-mers straight from raw chunk bytes: the arguments of bnpk_chunk_kmer_count
 *     with complement_xor in place of window_size (canonical minimizers: bnpk_chunk_minimizer_count_canonical).  Counts
 *     the values bnpk_rows_kmer_count_canonical counts over the sequence lines of the chunk's complete entries; slices,
 *     status and workspace as for bnpk_chunk_kmer_count.  complement_xor outside 1..3 returns BNPK_E_BADARG before any
 *     CUDA call. */
int bnpk_chunk_kmer_count_canonical(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end,
                                    int final_slice, int lines_per_entry, uint8_t header_char, int check_plus,
                                    int trim_cr, int enc_mode, const uint8_t *lut256, int k, int complement_xor,
                                    int64_t n_bins, int hist_mode, int64_t *hist,
                                    int64_t *status, void *workspace, size_t workspace_bytes, void *stream);
/*     Canonical minimizers: out[offsets[r] + j] = min over the window_size-k+1 k-mers i of window j of
 *     min(h_i, hash of the reverse complement of k-mer i), with h_i and complement_xor as above.  A read and its reverse
 *     complement give the same values (window j of one is window L - window_size - j of the other); window_size == k
 *     gives the canonical k-mers.  The three entry points take the arguments of bnpk_rows_minimizers,
 *     bnpk_rows_kmer_count and bnpk_chunk_kmer_count with complement_xor after window_size, and give their outputs.
 *     Before any CUDA call: complement_xor outside 1..3 returns BNPK_E_BADARG, window_size < k or > 1024
 *     BNPK_E_WINDOW, k outside 1..31 BNPK_E_K. */
int bnpk_rows_minimizers_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                   size_t n_rows, int enc_mode, const uint8_t *lut256, int k, int window_size,
                                   int complement_xor, const int64_t *offsets, int64_t *mins_out, int64_t *status,
                                   void *stream);
int bnpk_rows_minimizer_count_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts,
                                        const int32_t *lens, size_t n_rows, int enc_mode, const uint8_t *lut256, int k,
                                        int window_size, int complement_xor, int64_t n_bins, int hist_mode,
                                        int64_t *hist, int64_t *status, void *stream);
int bnpk_chunk_minimizer_count_canonical(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end,
                                         int final_slice, int lines_per_entry, uint8_t header_char, int check_plus,
                                         int trim_cr, int enc_mode, const uint8_t *lut256, int k, int window_size,
                                         int complement_xor, int64_t n_bins, int hist_mode, int64_t *hist,
                                         int64_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* K5  np.bincount(values % n_bins, minlength=n_bins) accumulated into hist
 *     (sequence/count_encoded.py:173-177; EncodedArray.__array_function__ encoded_array.py:459-460).
 *     Values must be non-negative; n_bins = len(alphabet) reproduces count_encoded exactly
 *     (out-of-range values are reported in status[BNPK_ST_BAD_BASE]). */
int bnpk_bincount(const int64_t *values, size_t n, int64_t n_bins, int hist_mode, int64_t *hist,
                  int64_t *status, void *stream);

/* K5' count_encoded(axis=-1) (sequence/count_encoded.py:180-182): per-row bincount,
 *     out[r * n_bins + b]; offsets int64[R+1] delimit the rows of `values`. */
int bnpk_bincount_rows(const int64_t *values, const int64_t *offsets, size_t n_rows, int64_t n_bins,
                       int64_t *out, int64_t *status, void *stream);

/* ---------------------------------------------------------------------------------------
 * Indexed FASTA (io/indexed_fasta.py:101-206, IndexedFasta.__getitem__ / get_interval_sequences): rows of bases out of
 * a device-resident FASTA file image, line ends skipped.  Row r = bases [row_start[r], row_start[r] + row_len[r]) of
 * the contig whose first base is file byte contig_offset[r] (.fai column 3), lenc[r] bases per line of lenb[r] bytes
 * (.fai columns 4, 5).  out[out_offsets[r] + i]; a position outside the file is reported in status[BNPK_ST_BAD_BASE].
 * ------------------------------------------------------------------------------------- */
int bnpk_fasta_gather(const uint8_t *file, size_t file_bytes, size_t n_rows, const int64_t *contig_offset,
                      const int64_t *row_start, const int64_t *row_len, const int32_t *lenc, const int32_t *lenb,
                      const int64_t *out_offsets, uint8_t *out, int64_t *status, void *stream);

/* Multi-line FASTA bookkeeping over the per-line arrays of bnpk_line_split(lines_per_entry = 1)
 * (MultiLineFastaBuffer.from_raw_buffer / get_data, io/multiline_buffer.py:46-62,89-106):
 *   bnpk_multiline_flags    is_header[i] (line starts with '>'), out2[0] = 1 + the last line whose newline is followed by
 *                           '>' (0: no complete entry), out2[1] = 1 if one of the first ten lines ends in '\r'
 *   bnpk_multiline_entries  with hdr_before = bnpk_row_offsets(is_header, 0): header fields (h_starts/h_lens per entry),
 *                           the sequence lines compacted in order (s_starts/s_lens) and entry_lens (zero-initialised by
 *                           the caller) = bases per entry; trim_cr as decided from out2[1]. */
int bnpk_multiline_flags(const uint8_t *chunk, size_t n, const int64_t *line_starts, const int32_t *line_lens, size_t n_lines,
                         int32_t *is_header, int64_t *out2, void *stream);
int bnpk_multiline_entries(const uint8_t *chunk, const int64_t *line_starts, const int32_t *line_lens, const int32_t *is_header,
                           const int64_t *hdr_before, size_t keep, int trim_cr, int64_t *h_starts, int32_t *h_lens,
                           int64_t *s_starts, int32_t *s_lens, int64_t *entry_lens, void *stream);

/* Bloom filter over k-mer hashes (sequence/bloom_filter.py:15-42): hash function i is v ^ offsets[i]; the filter is
 * one byte per position (the reference's bool mask).  insert: mask[(v ^ offsets[i]) % mask_size] = 1 for every value and
 * function; query: out[j] = AND over the functions. */
int bnpk_bloom_insert(const int64_t *values, size_t n, const int64_t *offsets, int n_hash, uint8_t *mask, size_t mask_size,
                      void *stream);
int bnpk_bloom_query(const int64_t *values, size_t n, const int64_t *offsets, int n_hash, const uint8_t *mask, size_t mask_size,
                     uint8_t *out, void *stream);

/* ---------------------------------------------------------------------------------------
 * Host-buffer entry point (end-to-end): the call a reader loop makes with a chunk that is
 * still in host memory.  Copies `chunk_host` (pinned or pageable) to the device in slices on
 * a private copy stream, overlapping each slice's H2D with the fused count of the previous
 * one, accumulates into the DEVICE histogram `hist`, and copies the status block back to
 * `status_host` (int64[BNPK_ST_WORDS]).  Synchronises before returning.
 * Replaces CupyFileReader._get_buffer's cp.asanyarray(chunk) (cupy_compatible/parser.py:11-17)
 * plus the K6 chain above.  `ctx` comes from bnpk_pipeline_create (owns the device staging
 * buffer, workspace, streams, events); capacity = largest chunk it will be given.
 * ------------------------------------------------------------------------------------- */
typedef struct bnpk_pipeline bnpk_pipeline;
int  bnpk_pipeline_create(bnpk_pipeline **ctx, size_t capacity_bytes, size_t slice_bytes);
void bnpk_pipeline_destroy(bnpk_pipeline *ctx);
int  bnpk_pipeline_kmer_count_host(bnpk_pipeline *ctx, const uint8_t *chunk_host, size_t n,
                                   int lines_per_entry, uint8_t header_char, int check_plus, int trim_cr,
                                   int enc_mode, const uint8_t *lut256_host, int k, int window_size,
                                   int64_t n_bins, int hist_mode, int64_t *hist, int64_t *status_host);
/* The same, ordered after the work already queued on `stream` (whatever produced or zeroed `hist`); the entry point
 * above orders itself after the legacy default stream. */
int  bnpk_pipeline_kmer_count_host_on(bnpk_pipeline *ctx, const uint8_t *chunk_host, size_t n,
                                      int lines_per_entry, uint8_t header_char, int check_plus, int trim_cr,
                                      int enc_mode, const uint8_t *lut256_host, int k, int window_size,
                                      int64_t n_bins, int hist_mode, int64_t *hist, int64_t *status_host, void *stream);

/* ---------------------------------------------------------------------------------------
 * Synthetic workload generator (SURVEY 8d record: "@r%010d\n" + 150 bases + "\n+\n" +
 * 150*'I' + "\n" = 317 B), bit-identical to oracle/bnp_oracle.py:synthetic_fastq.
 * Test/bench utility; out must hold n_records*317 bytes.
 * ------------------------------------------------------------------------------------- */
int bnpk_synth_fastq(uint8_t *out, uint64_t first_record, uint64_t n_records, uint64_t seed, void *stream);

/* Measurement hooks: when enabled, every launch of the dominant (tile) kernel is bracketed by
 * CUDA events on the launching stream; bnpk_profile_read waits for them, returns the summed
 * duration and the launch count, and clears the list. */
int bnpk_profile_enable(int on);
int bnpk_profile_read(double *total_ms, uint64_t *n_launches);

/* how many kernels this library has launched in this process (bench's gpu_launches) */
uint64_t bnpk_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* BNPK_H */
