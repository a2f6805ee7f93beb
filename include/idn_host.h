/*
 * idn_host.h -- flat C view of the host-side mirror of idencomp's API (libidn_host.so).
 *
 * The host mirror itself is C++ (idencomp_b200/csrc/host/, the .hpp files: Model, ModelProvider, IdnCompressor,
 * IdnDecompressor -- same names, arguments and error behaviour as the reference's Rust types) and calls
 * only the C-ABI of include/idn_gpu.h.  This header exists so that the Python test/bench harness (ctypes)
 * and other FFI users can drive those classes; every function cites the reference item it stands for.
 * Status codes are the IDN_* codes of idn_gpu.h.  idn_host_last_error() is per thread.
 */
#ifndef IDN_HOST_H
#define IDN_HOST_H

#include <stddef.h>
#include <stdint.h>

#include "idn_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct idn_host_model idn_host_model;

const char *idn_host_last_error(void);

/* ---- Model (model.rs:176-259, model_serializer.rs:90-114) ---------------------------------------- */
/* SerializableModel::read_model: parses the msgpack file, recomputes the SHA3-256 identifier and fails
 * with IDN_E_SERIALIZE if it differs from the stored one (model_serializer.rs:111-114). */
int32_t idn_host_model_load(const char *path, idn_host_model **out);
int32_t idn_host_model_from_bytes(const uint8_t *data, size_t n, idn_host_model **out);
/* Model::with_model_and_spec_type from raw contexts: probs[n_ctx][nsym] f32, spec lists given as
 * (spec_keys[i] -> context spec_ctx[i]) pairs (used by tests to build the reference's toy models). */
int32_t idn_host_model_new(int32_t model_type, const char *spec_name, uint32_t n_ctx, const float *probs,
                           const uint32_t *spec_keys, const uint32_t *spec_ctx, uint64_t n_specs,
                           idn_host_model **out);
int32_t idn_host_model_empty(int32_t model_type, idn_host_model **out); /* Model::empty, model.rs:251-259 */
void idn_host_model_free(idn_host_model *m);
int32_t idn_host_model_type(const idn_host_model *m);          /* IDN_MODEL_ACID / IDN_MODEL_QSCORE */
uint32_t idn_host_model_len(const idn_host_model *m);          /* number of contexts */
const char *idn_host_model_spec_name(const idn_host_model *m); /* e.g. "light_ao8_qo0_pb0_qm1" */
void idn_host_model_identifier(const idn_host_model *m, uint8_t out[32]);
/* integer tables: cum [(len+1)][nsym+1] u16 (row 0 = dummy context); returns the number of u16 written
 * (call with out == NULL to size) */
uint64_t idn_host_model_cum_table(const idn_host_model *m, uint16_t *out, uint64_t cap);
/* RansEncModel/RansDecModel::from_model (sequence_compressor.rs:21-48,175-201) on the device:
 * quantises every context (context.rs:346-394) and uploads the tables through idn_gpu_model_upload */
int32_t idn_host_model_upload(idn_gpu_ctx *ctx, const idn_host_model *m, idn_model_t *handle);

/* Context::as_integer_cum_freqs (context.rs:346-371) -- exposed for the known-answer tests */
int32_t idn_host_quantise(const float *probs, uint32_t nsym, uint32_t scale_bits, uint32_t *cum_out);

/* ---- IdnCompressor (idn/compressor.rs:443-585) ------------------------------------------------------- */
typedef struct idn_host_compressor idn_host_compressor;
typedef struct {                    /* IdnCompressorParamsBuilder, idn/compressor.rs:164-274 */
    uint32_t max_block_total_len;   /* default 4 Mi */
    uint32_t thread_num;            /* default 0 */
    int32_t include_identifiers;    /* default 1 */
    uint32_t quality;               /* 1..9, default 7 */
    int32_t fast;                   /* default 0; sets quality 1 */
    int32_t device;                 /* CUDA device, default 0 (used when n_devices == 0) */
    int32_t mode;                   /* IDN_MODE_COMPAT (container version 1) or IDN_MODE_NATIVE (version 2) */
    uint32_t batch_blocks;          /* blocks per device call, default 32 */
    uint32_t lane_symbols;          /* native mode lane quantum, default 2048 */
    uint64_t text_chunk_bytes;      /* add_text: bytes of FASTQ text per device call, default 256 Mi */
    uint32_t n_devices;             /* > 0: the GPUs that share the file (batches go round robin, results are committed in block
                                       order; the container does not depend on the device count) */
    int32_t devices[16];
    int32_t identifiers_on_device;  /* default 0; != 0: identifiers slices Deflated on the device (idn_gpu_deflate_names),
                                       IDN_E_UNSUPPORTED with include_identifiers at quality 8-9 (Brotli) */
} idn_host_params;
void idn_host_params_default(idn_host_params *p);
/* IdnCompressor::with_params over an in-memory writer; `models` is the ModelProvider (order = provider order) */
int32_t idn_host_compressor_new(const idn_host_model *const *models, uint32_t n_models, const idn_host_params *params,
                                idn_host_compressor **out);
/* IdnCompressor::add_sequence; IDN_E_SEQUENCE_TOO_LONG when len > max_block_total_len / 2 */
int32_t idn_host_compressor_add(idn_host_compressor *c, const uint8_t *name, uint64_t name_len, const uint8_t *acids,
                                const uint8_t *quals, uint64_t len);
/* add_sequence for every read of an SoA batch (name_off/names may be NULL) */
int32_t idn_host_compressor_add_batch(idn_host_compressor *c, uint64_t n_reads, const uint64_t *read_off,
                                      const uint8_t *acids, const uint8_t *quals, const uint64_t *name_off,
                                      const uint8_t *names);
/* FASTQ text instead of parsed sequences: consecutive pieces of the text, cut anywhere (FastqReader + add_sequence of the
 * reference, done on the device); not to be mixed with the two calls above on one compressor */
int32_t idn_host_compressor_add_text(idn_host_compressor *c, const uint8_t *text, uint64_t n);
int32_t idn_host_compressor_finish(idn_host_compressor *c);     /* IdnCompressor::finish */
/* the container (complete after finish: blocks reach the output from a writer thread, in order, while the add_* calls go
 * on; an error of a block or of the output is reported by the next add_* call or by finish); the pointer stays valid until
 * the next call on `c` */
uint64_t idn_host_compressor_output(const idn_host_compressor *c, const uint8_t **data);
/* identifiers written to the metadata, acid models first; returns their number */
uint32_t idn_host_compressor_retained(const idn_host_compressor *c, uint8_t *ids /* [cap][32] */, uint32_t cap);
/* in_symbols, in_reads, in_identifier_bytes, out_bytes, out_identifier_bytes, out_payload_bytes, blocks,
 * acid_model_switches, q_score_model_switches */
void idn_host_compressor_stats(const idn_host_compressor *c, uint64_t out[9]);
void idn_host_compressor_free(idn_host_compressor *c);

/* ---- IdnDecompressor (idn/decompressor.rs:455-566): next_sequence until None, results as one SoA batch ---- */
typedef struct idn_host_decoded idn_host_decoded;
/* the whole file as FASTQ text (FastqWriter of the reference, formatted on the device); free with idn_host_text_free */
int32_t idn_host_decompress_text(const idn_host_model *const *models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                 uint32_t thread_num, int32_t title_with_separator, const uint8_t *idn, uint64_t idn_len,
                                 uint8_t **text, uint64_t *text_len);
void idn_host_text_free(uint8_t *text);
/* The library keeps device contexts (with their device buffers) and page-locked host buffers of closed compressors /
 * decompressors for the next one; this gives them back. */
void idn_host_release_cached(void);
/* the same into the caller's buffer; IDN_E_NOSPACE when it is too small */
int32_t idn_host_decompress_text_into(const idn_host_model *const *models, uint32_t n_models, int32_t device,
                                      uint32_t batch_blocks, uint32_t thread_num, int32_t title_with_separator,
                                      const uint8_t *idn, uint64_t idn_len, uint8_t *text, uint64_t cap, uint64_t *text_len);
/* streaming form: each call hands out the FASTQ text of the next batch of blocks in the library's page-locked memory, where
 * the device wrote it (valid until the next call on the reader); *len = 0 at the end.  devices as in the compressor
 * parameters (an ordinal may repeat: that many contexts on the device, so that one batch's copies overlap another's
 * kernels) */
typedef struct idn_host_text_reader idn_host_text_reader;
int32_t idn_host_text_reader_new(const idn_host_model *const *models, uint32_t n_models, const int32_t *devices,
                                 uint32_t n_devices, uint32_t batch_blocks, uint32_t thread_num, int32_t title_with_separator,
                                 const uint8_t *idn, uint64_t idn_len, idn_host_text_reader **out);
int32_t idn_host_text_reader_next(idn_host_text_reader *r, const uint8_t **text, uint64_t *len);
void idn_host_text_reader_free(idn_host_text_reader *r);
/* the compressor writes the container into the caller's buffer instead of the library's growing one (before the first add) */
int32_t idn_host_compressor_set_output(idn_host_compressor *c, uint8_t *buf, uint64_t cap);
/* `device` >= 0: that GPU; < 0: the first (-device) GPUs share the file */
int32_t idn_host_decompress(const idn_host_model *const *models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                            const uint8_t *idn, uint64_t idn_len, idn_host_decoded **out);
uint64_t idn_host_decoded_reads(const idn_host_decoded *d);
uint32_t idn_host_decoded_version(const idn_host_decoded *d);
const uint64_t *idn_host_decoded_read_off(const idn_host_decoded *d); /* [reads+1] */
const uint8_t *idn_host_decoded_acids(const idn_host_decoded *d);
const uint8_t *idn_host_decoded_quals(const idn_host_decoded *d);
const uint64_t *idn_host_decoded_name_off(const idn_host_decoded *d); /* [reads+1] */
const uint8_t *idn_host_decoded_names(const idn_host_decoded *d);
void idn_host_decoded_free(idn_host_decoded *d);
/* decompressor parameters the forms above leave at their defaults (IdnDecompressorParams) */
typedef struct {
    int32_t identifiers_on_device; /* inflate the Identifiers slices on the device (idn_gpu_inflate_names); default 0 */
} idn_host_decompress_params;
/* the decompression entry points with parameters (NULL = the defaults, which is what the forms without _ex use) */
int32_t idn_host_decompress_ex(const idn_host_model *const *models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                               const uint8_t *idn, uint64_t idn_len, idn_host_decoded **out, const idn_host_decompress_params *dparams);
int32_t idn_host_decompress_text_ex(const idn_host_model *const *models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                    uint32_t thread_num, int32_t title_with_separator, const uint8_t *idn, uint64_t idn_len,
                                    uint8_t **text, uint64_t *text_len, const idn_host_decompress_params *dparams);
int32_t idn_host_decompress_text_into_ex(const idn_host_model *const *models, uint32_t n_models, int32_t device,
                                         uint32_t batch_blocks, uint32_t thread_num, int32_t title_with_separator,
                                         const uint8_t *idn, uint64_t idn_len, uint8_t *text, uint64_t cap, uint64_t *text_len,
                                         const idn_host_decompress_params *dparams);
int32_t idn_host_text_reader_new_ex(const idn_host_model *const *models, uint32_t n_models, const int32_t *devices,
                                    uint32_t n_devices, uint32_t batch_blocks, uint32_t thread_num, int32_t title_with_separator,
                                    const uint8_t *idn, uint64_t idn_len, idn_host_text_reader **out,
                                    const idn_host_decompress_params *dparams);

/* ---- file-level model subset selection on a cost matrix cost[value][centroid] (exposed for the known-answer tests) ----
 * Clustering::make_clusters (clustering.rs:21-118): centroid index per cluster and the cluster of every value;
 * returns the number of clusters.  `state` = a Clustering object whose random stream runs on from call to call (the
 * reference's ModelChooser holds ONE for the acid models and then the q-score models, model_chooser.rs:14-24); NULL = a
 * fresh Clustering::new().  get_model_ranking (idn/model_chooser.rs:103-138): the best `model_num` columns. */
typedef struct idn_host_clustering idn_host_clustering;
idn_host_clustering *idn_host_clustering_new(void);
void idn_host_clustering_free(idn_host_clustering *c);
uint32_t idn_host_cluster(idn_host_clustering *state, const uint32_t *cost, uint64_t n_values, uint32_t n_centroids,
                          uint32_t num_clusters, uint32_t *centroids_out, uint32_t *value_cluster_out);
/* the restated third-party generators behind Clustering (rand_xoshiro 0.6.0, rand 0.8.5; clustering.hpp), for their
 * published known-answer vectors: SplitMix64 stream; xoshiro256++ from four state words (state4 != NULL) or
 * seed_from_u64(seed); index::sample / gen_range(0..=high) on seed_from_u64(seed) */
void idn_host_splitmix64(uint64_t seed, uint32_t n, uint64_t *out);
void idn_host_xoshiro256pp(const uint64_t *state4, uint64_t seed, uint32_t n, uint64_t *out);
uint32_t idn_host_sample_indices(uint64_t seed, uint32_t length, uint32_t amount, uint32_t *out);
uint32_t idn_host_gen_range(uint64_t seed, uint32_t high, uint32_t n, uint32_t *out);
uint32_t idn_host_rank(const uint32_t *cost, uint64_t n_values, uint32_t n_models, uint32_t model_num, uint32_t *models_out);

#ifdef __cplusplus
}
#endif
#endif /* IDN_HOST_H */
