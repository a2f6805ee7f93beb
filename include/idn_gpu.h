/*
 * idn_gpu.h -- C-ABI of libidn_gpu.so: the B200 (sm_100a) implementation of idencomp's rANS hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI today; the seam a
 * maintainer would bind is "one call per batch of blocks" replacing
 *     IdnBlockCompressor::process      idencomp/src/idn/compressor_block.rs:76-120
 *     IdnBlockDecompressor::process    idencomp/src/idn/decompressor_block.rs:77-129
 *     ModelProvider::preprocess_*      idencomp/src/idn/model_provider.rs:154-173
 *     ModelTester::compute_size        idencomp/src/idn/model_chooser.rs:215-243
 * INTEGRATION.md shows the Rust `extern "C"` block + build.rs a maintainer would add.
 *
 * Conventions: every entry point returns an int32 status (0 = IDN_OK); plain pointers and sizes only;
 * the caller owns every buffer it passes; the library owns device memory inside `idn_gpu_ctx`; no pointer
 * escapes a call.  A ctx is single-owner (one per device per host thread); model handles are immutable
 * after upload.  Functions ending in `_dev` take DEVICE pointers and enqueue on `stream` (a cudaStream_t
 * passed as void*; NULL = the legacy default stream) without synchronising; the others take HOST pointers
 * (pinned memory recommended), do the H2D/D2H copies themselves and return when the result is in the
 * caller's buffers.  There is no CPU fallback: every call fails with IDN_E_CUDA when no device is usable.
 */
#ifndef IDN_GPU_H
#define IDN_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IDN_GPU_ABI_VERSION 1

/* Status codes: 1..9 map 1:1 onto the reference's error enums
 * (IdnCompressorError idn/compressor.rs:22-33, IdnDecompressorError idn/decompressor.rs:25-48). */
enum {
    IDN_OK = 0,
    IDN_E_INVALID_STATE = 1,
    IDN_E_IO = 2,
    IDN_E_SERIALIZE = 3,        /* malformed container / slice */
    IDN_E_SEQUENCE_TOO_LONG = 4,
    IDN_E_INVALID_VERSION = 5,
    IDN_E_CHECKSUM = 6,         /* BlockChecksumMismatch */
    IDN_E_INVALID_MODEL_INDEX = 7,
    IDN_E_NO_ACTIVE_MODEL = 8,
    IDN_E_UNKNOWN_MODEL = 9,
    IDN_E_UNSUPPORTED = 10,     /* e.g. an unknown container mode, > 16 candidate models of one type */
    IDN_E_NOSPACE = 11,         /* output capacity too small; required size is reported */
    IDN_E_INVALID_ARG = 12,
    IDN_E_INVALID_SYMBOL = 13,  /* acid > 4 or quality score > 93 in the input */
    IDN_E_CUDA = 100
};

enum { IDN_MODEL_ACID = 0, IDN_MODEL_QSCORE = 1 };   /* ModelType, model.rs:56-61 */
enum { IDN_SPEC_GENERIC = 0, IDN_SPEC_LIGHT = 1 };   /* context_spec.rs:218,421 ("dummy" = generic 0,0,0) */
enum { IDN_MODE_COMPAT = 1, IDN_MODE_NATIVE = 2 };   /* container version byte (idn/data.rs:3-8) */

#define IDN_SCALE_BITS 14   /* idn/model_provider.rs:407 */
#define IDN_ACID_SYMS 5
#define IDN_Q_SYMS 94
#define IDN_MAX_MODELS 255  /* SwitchModel index is a u8 (idn/data.rs:72-76) */

typedef struct idn_gpu_ctx idn_gpu_ctx;
typedef int32_t idn_model_t; /* handle, >= 0 */

/* ---- lifecycle ------------------------------------------------------------------------------------- */
int32_t idn_gpu_abi_version(void);
int32_t idn_gpu_device_count(void);
int32_t idn_gpu_create(int32_t device, idn_gpu_ctx **ctx);
void idn_gpu_destroy(idn_gpu_ctx *ctx);
const char *idn_gpu_last_error(const idn_gpu_ctx *ctx);
/* lane quantum of IDN_MODE_NATIVE compression: a lane holds the reads whose first symbol falls into the same run of
 * `lane_syms` symbols of the block (default 2048); the value travels in the container, decoders need no setting */
int32_t idn_gpu_set_lane_symbols(idn_gpu_ctx *ctx, uint32_t lane_syms);
/* decode side, compat containers: which slice walk indexes the blocks (IdnBlockDecompressor::next_sequence_internal,
 * idn/decompressor_block.rs:115-129).  0 = automatic (the parallel speculative walk for calls of fewer than 512 blocks,
 * the one-warp-per-block walk otherwise and as its fallback), 1 = always the one-warp-per-block walk, 2 = always try the
 * parallel walk first.  Results do not depend on the setting; the environment variable IDN_WALK=serial|fast sets the
 * default of new contexts. */
int32_t idn_gpu_set_walk(idn_gpu_ctx *ctx, int32_t mode);
/* the host-pointer entry points idn_gpu_compress_blocks / idn_gpu_decompress_blocks cut a call into sub-chunks of this many
 * blocks (default 32; environment variable IDN_PIPE_BLOCKS) and overlap the upload of one sub-chunk with the kernels of the
 * one before and the download of the one before that, on three streams of this ctx.  Results do not depend on the setting. */
int32_t idn_gpu_set_pipeline_blocks(idn_gpu_ctx *ctx, uint32_t blocks);
/* number of kernel launches this ctx has issued since creation (bench.py's gpu_launches) */
uint64_t idn_gpu_launch_count(const idn_gpu_ctx *ctx);
/* which codec kernel instantiation a call with exactly this (acid, q-score) model pair launches: the index of the
 * compile-time-specialised spec-type pair (0 .. idn_gpu_kernel_variant_count() - 1, table in idn_gpu.cu), or -1 for the
 * run-time-generic kernels.  Lets the parity tests assert that every specialised instantiation was compared with the
 * oracle; results never depend on the variant. */
int32_t idn_gpu_kernel_variant(const idn_gpu_ctx *ctx, idn_model_t acid_model, idn_model_t q_model);
int32_t idn_gpu_kernel_variant_count(void);

/* page-locked host memory for the buffers a caller passes to the host-pointer entry points (a copy from / to pageable
 * memory is staged by the driver at a fraction of the link's speed); usable from any thread and any device */
int32_t idn_gpu_host_alloc(uint64_t bytes, void **p);
void idn_gpu_host_free(void *p);

/* ---- models: replaces RansEncModel/RansDecModel::from_model (sequence_compressor.rs:21-48,175-201) --
 * `cum`: integer cumulative frequencies, row-major [(n_ctx+1)][nsym+1] u16, row 0 = the uniform dummy
 * context (sequence_compressor.rs:26-29), last column = 1<<14; produced on the host by the bit-exact
 * f32 quantiser (context.rs:346-394).  `spec_keys[i]` -> 0-based context index `spec_ctx[i]`; specs not
 * listed map to the dummy context (sequence_compressor.rs:37-40). */
int32_t idn_gpu_model_upload(idn_gpu_ctx *ctx, int32_t model_type, int32_t spec_kind, int32_t acid_order,
                             int32_t q_order, int32_t pos_bits, int32_t q_max, uint32_t n_ctx,
                             const uint16_t *cum, const uint32_t *spec_keys, const uint32_t *spec_ctx,
                             uint64_t n_specs, idn_model_t *handle);
int32_t idn_gpu_model_release(idn_gpu_ctx *ctx, idn_model_t handle);

/* ---- batches ----------------------------------------------------------------------------------------
 * SoA batch of reads grouped into blocks (block forming stays on the host: idn/compressor.rs:517-559).
 * acids: 0..4 (N,A,C,T,G  sequence.rs:401-413); quals: 0..93.  Block b holds reads
 * [block_first_read[b], block_first_read[b+1]).  `names`/`name_off` are optional (NULL = empty names);
 * when given, the block CRC covers name bytes as the reference's does (sequence.rs:381-394). */
typedef struct {
    uint64_t n_reads;
    uint64_t n_symbols;               /* = read_off[n_reads] */
    uint32_t n_blocks;
    const uint8_t *acids;             /* [n_symbols] */
    const uint8_t *quals;             /* [n_symbols] */
    const uint64_t *read_off;         /* [n_reads+1] */
    const uint32_t *block_first_read; /* [n_blocks+1] */
    const uint8_t *names;             /* optional */
    const uint64_t *name_off;         /* optional [n_reads+1] */
} idn_batch;

typedef struct {
    uint64_t out_bytes;         /* bytes written to `out` */
    uint64_t acid_switches;     /* SwitchModel slices emitted per type */
    uint64_t q_switches;
    uint64_t payload_bytes;     /* sum of rANS payload lengths */
    uint64_t required_bytes;    /* set on IDN_E_NOSPACE */
} idn_compress_stats;

/* a6: ModelTester::compute_size for every (read, model): sizes[r * n_models + m] = byte length of a
 * forward single-state rANS encode of read r under models[m] (+4 flush bytes). */
int32_t idn_gpu_score(idn_gpu_ctx *ctx, const idn_batch *batch, const idn_model_t *models, uint32_t n_models,
                      uint32_t *sizes);
int32_t idn_gpu_score_dev(idn_gpu_ctx *ctx, const idn_batch *batch, const idn_model_t *models,
                          uint32_t n_models, uint32_t *sizes, void *stream);

/* a7+a8+a10: compress a batch of blocks.
 * `models[k]` is the retained provider list in container order (k = SwitchModel index; acid ids first,
 * then q-score ids: compressor_initializer.rs:57-65).  fast != 0 reproduces `--fast`
 * (compressor_block.rs:95-106: exactly 2 models, switches 0 and 1 at the start of each block).
 * prefix_len[b] (optional, NULL = 0) reserves room right after the block header for the identifiers
 * slice, which the host compresses and copies in (names stay on the host as in the reference).
 * Output, for each block b at out[block_off[b] .. block_off[b+1]):
 *     u32be length | u32be crc32 | prefix_len[b] reserved bytes | SwitchModel / Sequence slices
 * i.e. exactly the bytes IdnBlockCompressor::write emits (compressor_block.rs:122-128,
 * writer_block.rs:27-40) once the host has filled the reserved bytes.  block_crc[b] (optional) also
 * receives the CRC.  With IDN_MODE_NATIVE the slices use the multi-lane layout of DESIGN.md. */
int32_t idn_gpu_compress_blocks(idn_gpu_ctx *ctx, const idn_batch *batch, int32_t mode,
                                const idn_model_t *models, uint32_t n_models, int32_t fast,
                                const uint32_t *prefix_len, uint8_t *out, uint64_t out_cap,
                                uint64_t *block_off, uint32_t *block_crc, idn_compress_stats *stats);
int32_t idn_gpu_compress_blocks_dev(idn_gpu_ctx *ctx, const idn_batch *batch, int32_t mode,
                                    const idn_model_t *models, uint32_t n_models, int32_t fast,
                                    const uint32_t *prefix_len, uint8_t *out, uint64_t out_cap,
                                    uint64_t *block_off, uint32_t *block_crc, idn_compress_stats *stats_dev,
                                    void *stream);
/* upper bound of the output size of idn_gpu_compress_blocks for a batch shape */
uint64_t idn_gpu_compress_bound(uint64_t n_reads, uint64_t n_symbols, uint32_t n_blocks, uint64_t prefix_total);

/* a9+a11: decompress a batch of blocks given as container bytes.
 * Block b's payload (the slices, WITHOUT its 8-byte block header) is blocks[block_off[b] .. block_off[b] + len_b) with
 * len_b = block_len ? block_len[b] : block_off[b+1] - block_off[b]; block_off[n_blocks] is the size of the `blocks`
 * region and block_crc[b] the block's header checksum.  With block_len the region may hold other bytes between the
 * payloads, so a chunk of an .idn file can be passed as it lies on disk (block_off[b] = header position + 8); the blocks
 * must not overlap (IDN_E_INVALID_ARG).  The library walks the
 * slices (Identifiers slices are skipped: names stay on the host), tracks the active models per type
 * (decompressor_block.rs:194-214), decodes every Sequence slice and verifies the CRC of the symbols
 * (names, if any, are passed per read through `names`/`name_off` after the host inflated them; NULL =
 * the block has no names).  A Sequence slice (or native lane) whose rANS stream runs out early, or does not end with
 * both states back at their initial value and every payload byte consumed, fails the call with IDN_E_SERIALIZE in both
 * container modes, with or without a CRC to compare against.
 * A failing call reports the first failing block in file order (bad_block / status_dev[1]; -1 only for errors of the
 * whole call such as IDN_E_NOSPACE): the blocks in front of a malformed one are still decoded and checked, so a
 * checksum mismatch or a garbled stream there is reported instead; within one block malformed slices come before a
 * checksum mismatch before a garbled stream.  The report does not depend on idn_gpu_set_walk, on
 * idn_gpu_set_pipeline_blocks or on the entry point.  (A native lane table that does not match its read lengths stops
 * the call where it is found: the blocks in front of it are not checked.)
 * Two-step use: idn_gpu_index_blocks returns the read count / symbol count so the caller can size the
 * outputs, then idn_gpu_decompress_blocks fills them.  The index call leaves the container bytes on the device: a
 * decode call (idn_gpu_decompress_blocks, idn_gpu_decompress_to_fastq) that follows it on the same context with the
 * same table may pass blocks == NULL to decode those bytes instead of uploading them a second time (such a call is not
 * split into pipelined sub-chunks); NULL without a matching index call before it is IDN_E_INVALID_ARG. */
typedef struct {
    uint64_t n_reads;
    uint64_t n_symbols;
} idn_block_index_totals;

int32_t idn_gpu_index_blocks(idn_gpu_ctx *ctx, const uint8_t *blocks, const uint64_t *block_off,
                             const uint32_t *block_len /* optional */, uint32_t n_blocks, int32_t mode, const idn_model_t *models, uint32_t n_models,
                             idn_block_index_totals *totals, uint32_t *block_first_read /*[n_blocks+1], optional*/);
int32_t idn_gpu_decompress_blocks(idn_gpu_ctx *ctx, const uint8_t *blocks, const uint64_t *block_off,
                                  const uint32_t *block_len /* optional */, const uint32_t *block_crc, uint32_t n_blocks, int32_t mode,
                                  const idn_model_t *models, uint32_t n_models, const uint8_t *names,
                                  const uint64_t *name_off, uint8_t *acids_out, uint8_t *quals_out,
                                  uint64_t *read_off_out /*[n_reads+1]*/, uint64_t out_reads_cap,
                                  uint64_t out_symbols_cap, int32_t *bad_block /* first failing block or -1 */);
int32_t idn_gpu_decompress_blocks_dev(idn_gpu_ctx *ctx, const uint8_t *blocks, const uint64_t *block_off,
                                      const uint32_t *block_len /* optional */, const uint32_t *block_crc, uint32_t n_blocks, uint64_t blocks_bytes,
                                      int32_t mode, const idn_model_t *models, uint32_t n_models,
                                      uint8_t *acids_out, uint8_t *quals_out, uint64_t *read_off_out,
                                      uint64_t out_reads_cap, uint64_t out_symbols_cap,
                                      int32_t *status_dev /* [4]: code, bad block, n_reads, n_symbols(lo) */,
                                      void *stream);

/* per-read form (host already holds the slice index): decode read r from payload[pay_off[r] ..
 * pay_off[r]+pay_len[r]) into acids_out/quals_out at out_off[r]; model index per read into models[]. */
typedef struct {
    uint64_t n_reads;
    const uint64_t *pay_off;
    const uint32_t *pay_len;
    const uint32_t *seq_len;
    const uint64_t *out_off;   /* [n_reads+1] exclusive scan of seq_len */
    const uint8_t *acid_model; /* index into models[] */
    const uint8_t *q_model;
} idn_read_index;

int32_t idn_gpu_decompress_reads(idn_gpu_ctx *ctx, const uint8_t *payload, uint64_t payload_bytes,
                                 const idn_read_index *index, const idn_model_t *models, uint32_t n_models,
                                 uint8_t *acids_out, uint8_t *quals_out, uint32_t *read_status /* optional */);

/* IEEE CRC-32 of the per-read stream name|acids|quals for each block (writer_block.rs:64,
 * sequence.rs:381-394), computed on the device. */
int32_t idn_gpu_block_crc(idn_gpu_ctx *ctx, const idn_batch *batch, uint32_t *block_crc);

/* ---- workload generator (bench/test utility; nothing in the reference corresponds to it) -------------
 * Fills acids/quals (DEVICE pointers) with model-driven synthetic reads: each symbol is sampled from the
 * distribution `acid_model` / `q_model` hold for the context the read is in (SURVEY.md 8d), `n_ppm` per
 * million positions become an N call with quality 2.  Deterministic in (seed, first_read_index + r). */
int32_t idn_gpu_synth_reads_dev(idn_gpu_ctx *ctx, idn_model_t acid_model, idn_model_t q_model,
                                const uint64_t *read_off /* device, [n_reads+1] */, uint64_t n_reads,
                                uint64_t first_read_index, uint64_t seed, uint32_t n_ppm, uint8_t *acids,
                                uint8_t *quals, void *stream);

/* ---- FASTQ text <-> symbol arrays on the device ("next" row f1: fastq/reader.rs:166-282, fastq/writer.rs:190-245) ----
 * Same acceptance rules as FastqReader::read_sequence for '\n'-delimited input: blank lines are skipped where a title
 * is expected, the title starts with '@' and is trimmed, acids are ATCGN, the separator line starts with '+', quality
 * scores are '!'..'~', both symbol lines have one length.  A violation fails with IDN_E_SERIALIZE; error_kind names
 * the FastqReaderError variant (1 InvalidFormat, 2 InvalidAcid, 3 InvalidQualityScore, 4 length mismatch, 5 end of
 * input inside a record) and bad_record the record, counted from 0, that the reference stops at: the first error in
 * file order, a record's lines checked in the reference's order. */
typedef struct {
    uint64_t n_reads, n_symbols, n_name_bytes, n_lines;
    int32_t error_kind;
    int32_t reserved;
    uint64_t bad_record;
} idn_fastq_info;
/* parse: the SoA result stays in the ctx until the next parse; fetch copies it to host buffers sized from `info`,
 * batch_dev exposes it as device pointers for the *_dev entry points (block_first_read is the caller's to add) */
int32_t idn_gpu_fastq_parse(idn_gpu_ctx *ctx, const uint8_t *text, uint64_t n, idn_fastq_info *info);
int32_t idn_gpu_fastq_parse_dev(idn_gpu_ctx *ctx, const uint8_t *text /* device */, uint64_t n, idn_fastq_info *info,
                                void *stream);
int32_t idn_gpu_fastq_fetch(idn_gpu_ctx *ctx, uint8_t *acids, uint8_t *quals, uint64_t *read_off, uint8_t *names,
                            uint64_t *name_off);
int32_t idn_gpu_fastq_batch_dev(idn_gpu_ctx *ctx, idn_batch *out);
/* format: "@name\nACGT\n+[name]\n!!!!\n" per read (FastqWriterParams::output_title_with_separator = the flag) */
int32_t idn_gpu_fastq_format(idn_gpu_ctx *ctx, const idn_batch *batch, int32_t title_with_separator, uint8_t *text,
                             uint64_t cap, uint64_t *n_out);
int32_t idn_gpu_fastq_format_dev(idn_gpu_ctx *ctx, const idn_batch *batch /* device pointers */,
                                 int32_t title_with_separator, uint8_t *text, uint64_t cap, uint64_t *n_out_dev,
                                 void *stream);

/* ---- FASTQ text <-> .idn blocks without a symbol round trip over PCIe ---------------------------------------------------
 * What the reference does between FastqReader and IdnCompressor::add_sequence (fastq/reader.rs:166-282 ->
 * idn/compressor.rs:517-585) and between IdnDecompressor::next_sequence and FastqWriter (fastq/writer.rs:190-245), for a
 * whole chunk of text at a time: the text is uploaded once, records are split and blocks are formed on the device with
 * the reference's rule (a read that would push the block past max_block_total_len opens the next one), the block kernels
 * run on the symbol arrays where they lie; only identifiers (for the host's Deflate / Brotli) and container bytes come
 * back.  All pointers are HOST pointers. */
typedef struct {
    uint64_t n_reads, n_symbols, n_name_bytes; /* of the blocks idn_gpu_compress_parsed will code */
    uint32_t n_blocks;
    int32_t error_kind;      /* as idn_fastq_info */
    uint64_t bad_record;
    uint64_t consumed_text;  /* bytes of `text` those blocks cover: the caller's next chunk starts here */
} idn_fastq_chunk;
/* final == 0: `text` is a piece of a longer input and must end on a line boundary; a record cut short at its end and the
 * reads of the last block (which may go on in the next chunk) are NOT consumed.  final != 0: everything is consumed.
 * IDN_E_SEQUENCE_TOO_LONG when a read exceeds max_block_total_len / 2 (idn/compressor.rs:542-544). */
int32_t idn_gpu_fastq_parse_chunk(idn_gpu_ctx *ctx, const uint8_t *text, uint64_t n, int32_t final,
                                  uint32_t max_block_total_len, idn_fastq_chunk *out);
/* identifiers (for the host's identifiers codec), tables and -- for the file-level model selection on the first block --
 * symbols of the blocks of the chunk parsed last; any pointer may be NULL */
int32_t idn_gpu_fastq_chunk_fetch(idn_gpu_ctx *ctx, uint8_t *names, uint64_t *name_off /*[n_reads+1]*/,
                                  uint32_t *block_first_read /*[n_blocks+1]*/, uint64_t *read_off /*[n_reads+1]*/,
                                  uint8_t *acids /*[n_symbols]*/, uint8_t *quals /*[n_symbols]*/);
/* compress the blocks of the chunk parsed last; output as idn_gpu_compress_blocks.  with_names != 0: the block CRCs cover
 * the identifiers as the reference's do (sequence.rs:381-394) */
int32_t idn_gpu_compress_parsed(idn_gpu_ctx *ctx, int32_t mode, const idn_model_t *models, uint32_t n_models, int32_t fast,
                                int32_t with_names, const uint32_t *prefix_len, uint8_t *out, uint64_t out_cap,
                                uint64_t *block_off, uint32_t *block_crc, idn_compress_stats *stats);
/* idn_gpu_compress_parsed with the identifiers Deflated on the device (idn_gpu_deflate_names_dev) and put into the room after
 * each block header there: `out` comes back complete, the names never leave the device, the block CRCs cover them. */
int32_t idn_gpu_compress_parsed_ids(idn_gpu_ctx *ctx, int32_t mode, const idn_model_t *models, uint32_t n_models, int32_t fast,
                                    uint8_t *out, uint64_t out_cap, uint64_t *block_off, uint32_t *block_crc,
                                    idn_compress_stats *stats);
/* idn_gpu_decompress_blocks + FastqWriter: the FASTQ text of the decoded reads into `text` (the symbols stay on the
 * device); names / name_off = the identifiers the caller inflated (optional) */
int32_t idn_gpu_decompress_to_fastq(idn_gpu_ctx *ctx, const uint8_t *blocks, const uint64_t *block_off,
                                    const uint32_t *block_len, const uint32_t *block_crc, uint32_t n_blocks, int32_t mode,
                                    const idn_model_t *models, uint32_t n_models, const uint8_t *names,
                                    const uint64_t *name_off, uint64_t reads_cap, uint64_t symbols_cap,
                                    int32_t title_with_separator, uint8_t *text, uint64_t text_cap, uint64_t *text_len,
                                    uint64_t *n_reads_out, int32_t *bad_block);

/* ---- identifiers slices: raw Deflate (RFC 1951) on the device ----------------------------------------------------------
 * For each block b (reads [block_first_read[b], block_first_read[b+1]), block_first_read[0] = 0, names[name_off[r] ..
 * name_off[r+1]) per read) the bytes write_identifiers emits (compressor_block.rs:146-206) with Deflate:
 *     0x00 | u32be n | 0x01 | n bytes of raw Deflate of the block's names joined by '\n'
 * at out[slice_off[b] .. slice_off[b+1]).  The Deflate bytes are not zlib's: the names are coded in segments of 64 KiB,
 * each one block with its own Huffman code, the segments of a block joined by empty stored blocks; any inflater reads
 * them.  They depend only on the block's names (not on the other blocks of the call, the device or scheduling).
 * IDN_E_INVALID_ARG for a name_off or block_first_read that is not monotone or a block_first_read[0] != 0;
 * IDN_E_NOSPACE when out_cap is too small, slice_off[n_blocks] then holds the size needed.  The _dev form takes DEVICE
 * pointers and synchronises `stream` three times to size its work; the other stages them and returns when done. */
int32_t idn_gpu_deflate_names(idn_gpu_ctx *ctx, const uint8_t *names, const uint64_t *name_off, const uint32_t *block_first_read,
                              uint32_t n_blocks, uint8_t *out, uint64_t out_cap, uint64_t *slice_off /*[n_blocks+1]*/);
int32_t idn_gpu_deflate_names_dev(idn_gpu_ctx *ctx, const uint8_t *names, const uint64_t *name_off, const uint32_t *block_first_read,
                                  uint32_t n_blocks, uint8_t *out, uint64_t out_cap, uint64_t *slice_off /*[n_blocks+1]*/,
                                  void *stream);
/* upper bound of slice_off[n_blocks] for any names of this shape (name_bytes = name_off[R] - name_off[0]) */
uint64_t idn_gpu_deflate_names_bound(uint64_t name_bytes, uint64_t n_reads, uint32_t n_blocks);

/* ---- identifiers slices: raw Inflate (RFC 1951) on the device ----------------------------------------------------------
 * What the host's inflate_names does for a batch of blocks (decompressor_block.rs:146-192), on the device: every block's
 * leading Identifiers slices (0x00 | u32be n | compression | n bytes) are inflated, joined with '\n', and split at '\n'
 * into at most as many names as the block has reads (block b holds reads [block_first_read[b], block_first_read[b+1]));
 * reads without a line get an empty name, text after the last wanted line is dropped.  Acceptance is zlib's raw inflate
 * (windowBits -15), bytes after the final block included.  blocks / block_off / block_len are as idn_gpu_decompress_blocks
 * takes them; blocks == NULL uses the bytes the last idn_gpu_index_blocks call left on the device (same rule as the decode
 * calls) and keeps them there.  The names stay in the ctx: idn_gpu_inflate_names_fetch copies them out (names:
 * n_name_bytes bytes, name_off: n_reads + 1 entries), the _ids decode calls below read them where they are.
 * IDN_E_UNSUPPORTED for a Brotli slice (compression 0; nothing is written), IDN_E_SERIALIZE for a compression byte above 1,
 * a truncated slice or a slice that does not inflate, with bad_block = the first such block. */
typedef struct {
    uint64_t n_streams;     /* Identifiers slices (0: no block has names) */
    uint64_t n_chunks;      /* ranges the slices were cut into (idn_gpu_set_inflate_range) */
    uint64_t n_speculative; /* chunks after a slice's first that found a block start and were decoded from it */
    uint64_t n_joined;      /* of them, chunks whose start the verified decode before them ended on */
    uint64_t serial_bytes;  /* output bytes decoded again from the end of the verified decode (chunks that did not join) */
    uint64_t in_bytes;      /* Deflate bytes of all slices */
} idn_inflate_stats;

int32_t idn_gpu_inflate_names(idn_gpu_ctx *ctx, const uint8_t *blocks, const uint64_t *block_off, const uint32_t *block_len /* optional */,
                              uint32_t n_blocks, const uint32_t *block_first_read /*[n_blocks+1]*/, uint64_t n_reads,
                              uint64_t *n_name_bytes, int32_t *bad_block, idn_inflate_stats *stats /* optional */);
int32_t idn_gpu_inflate_names_fetch(idn_gpu_ctx *ctx, uint8_t *names, uint64_t *name_off);
/* compressed bytes per range of the parallel inflate (default 4096); results do not depend on it */
int32_t idn_gpu_set_inflate_range(idn_gpu_ctx *ctx, uint32_t bytes);
/* idn_gpu_decompress_blocks / idn_gpu_decompress_to_fastq with the names the preceding idn_gpu_inflate_names call on this
 * ctx left on the device, for the block CRC and the title lines (no host round trip; the calls are not pipelined).
 * IDN_E_INVALID_ARG without such a call of the same number of blocks and reads. */
int32_t idn_gpu_decompress_blocks_ids(idn_gpu_ctx *ctx, const uint8_t *blocks, const uint64_t *block_off,
                                      const uint32_t *block_len /* optional */, const uint32_t *block_crc, uint32_t n_blocks, int32_t mode,
                                      const idn_model_t *models, uint32_t n_models, uint8_t *acids_out, uint8_t *quals_out,
                                      uint64_t *read_off_out, uint64_t out_reads_cap, uint64_t out_symbols_cap, int32_t *bad_block);
int32_t idn_gpu_decompress_to_fastq_ids(idn_gpu_ctx *ctx, const uint8_t *blocks, const uint64_t *block_off, const uint32_t *block_len,
                                        const uint32_t *block_crc, uint32_t n_blocks, int32_t mode, const idn_model_t *models,
                                        uint32_t n_models, uint64_t reads_cap, uint64_t symbols_cap, int32_t title_with_separator,
                                        uint8_t *text, uint64_t text_cap, uint64_t *text_len, uint64_t *n_reads_out, int32_t *bad_block);

/* ---- per-kernel timing (CUDA events on the launching stream; what bench.py's roofline line is made of) ----
 * idn_gpu_profile(ctx, 1) starts recording an event after every kernel launch of the *_dev entry points;
 * idn_gpu_profile_read synchronises the device and writes one text line per kernel, "name launches total_ms",
 * then clears the record. */
int32_t idn_gpu_profile(idn_gpu_ctx *ctx, int32_t enable);
int32_t idn_gpu_profile_read(idn_gpu_ctx *ctx, char *buf, uint64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* IDN_GPU_H */
