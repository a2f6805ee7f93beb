// idn.hpp -- host-side mirror of idencomp's compressor / decompressor API (the drop-in surface above the C-ABI).
//
//   FastqSequence                 fastq/mod.rs (identifier, acids, quality scores)
//   IdnCompressorParams(Builder)  idn/compressor.rs:164-274   model_provider, max_block_total_len, thread_num,
//                                                             include_identifiers, quality, fast  (+ device, mode, batch_blocks)
//   IdnCompressor                 idn/compressor.rs:443-585   with_params, add_sequence, finish
//   IdnDecompressorParams         idn/decompressor.rs:167-229
//   IdnDecompressor               idn/decompressor.rs:455-566 with_params, next_sequence
//   IdnError                      idn/compressor.rs:22-33, idn/decompressor.rs:25-48 (same variants, same conditions)
//
// Everything below add_sequence / next_sequence that touches symbols runs on the GPU through include/idn_gpu.h; the
// host keeps what the reference keeps on the host: block forming, container framing, name Deflate, ordered writes.
// The reference hands one block to one thread-pool job; here `batch_blocks` blocks go to the device in one call.
#pragma once
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <functional>
#include <future>
#include <memory>
#include <mutex>
#include <optional>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/idn_gpu.h"
#include "model.hpp"

namespace idencomp {

struct FastqSequence {
    std::string identifier;
    std::vector<uint8_t> acids;           // Acid as u8: N=0 A=1 C=2 T=3 G=4 (sequence.rs:401-413)
    std::vector<uint8_t> quality_scores;  // 0..93
    size_t len() const { return acids.size(); }
};

// IdnCompressorError / IdnDecompressorError: `code` is the IDN_* status of include/idn_gpu.h
struct IdnError : std::runtime_error {
    int32_t code;
    IdnError(int32_t c, const std::string& what) : std::runtime_error(what), code(c) {}
};

struct CompressionStats {  // idn/compressor.rs:596-737 (the counters that exist on this path)
    uint64_t in_symbols = 0, in_reads = 0, in_identifier_bytes = 0;
    uint64_t out_bytes = 0, out_identifier_bytes = 0, out_payload_bytes = 0;
    uint64_t blocks = 0, acid_model_switches = 0, q_score_model_switches = 0;
};

struct IdnCompressorParams {
    ModelProvider model_provider;
    uint32_t max_block_total_len = 4 * 1024 * 1024;  // idn/compressor.rs:187
    uint32_t thread_num = 0;                          // host threads for the name codec (0 = caller thread)
    bool include_identifiers = true;
    uint8_t quality = 7;                              // 1..9
    bool fast = false;
    // additions of this implementation (defaults keep the reference's behaviour)
    // GPUs that share the file: batches of `batch_blocks` blocks go round robin to the devices (blocks are independent,
    // compressor_block.rs:61-62), every device holds the retained models, the file-level model selection runs on
    // devices[0], and the results are committed in block order -- the container does not depend on the device count
    std::vector<int32_t> devices{0};
    int32_t mode = IDN_MODE_COMPAT;  // IDN_MODE_NATIVE writes container version 2
    uint32_t batch_blocks = 32;      // blocks per device call
    uint32_t lane_symbols = 2048;    // native mode lane quantum
    uint64_t text_chunk_bytes = 256ull << 20;  // add_fastq_text: bytes of FASTQ text per device call
    // identifiers slices Deflated on the device (idn_gpu_deflate_names) instead of by the host's zlib: other Deflate bytes,
    // somewhat larger, the same names after inflation.  Not available for the Brotli slices of quality 8-9.
    bool identifiers_on_device = false;
};

class IdnCompressorParamsBuilder {
public:
    IdnCompressorParamsBuilder& model_provider(ModelProvider p) { p_.model_provider = std::move(p); return *this; }
    IdnCompressorParamsBuilder& max_block_total_len(uint32_t v) { p_.max_block_total_len = v; return *this; }
    IdnCompressorParamsBuilder& thread_num(uint32_t v) { p_.thread_num = v; return *this; }
    IdnCompressorParamsBuilder& include_identifiers(bool v) { p_.include_identifiers = v; return *this; }
    IdnCompressorParamsBuilder& quality(uint8_t v);  // throws std::invalid_argument outside 1..9 (CompressionQuality::new)
    IdnCompressorParamsBuilder& fast(bool v) { p_.fast = v; return *this; }
    IdnCompressorParamsBuilder& device(int32_t v) { p_.devices.assign(1, v); return *this; }
    IdnCompressorParamsBuilder& devices(std::vector<int32_t> v) { if (!v.empty()) p_.devices = std::move(v); return *this; }
    IdnCompressorParamsBuilder& mode(int32_t v) { p_.mode = v; return *this; }
    IdnCompressorParamsBuilder& batch_blocks(uint32_t v) { p_.batch_blocks = v ? v : 1; return *this; }
    IdnCompressorParamsBuilder& lane_symbols(uint32_t v) { p_.lane_symbols = v; return *this; }
    IdnCompressorParamsBuilder& text_chunk_bytes(uint64_t v) { p_.text_chunk_bytes = v ? v : 1; return *this; }
    IdnCompressorParamsBuilder& identifiers_on_device(bool v) { p_.identifiers_on_device = v; return *this; }
    IdnCompressorParams build() const { return p_; }

private:
    IdnCompressorParams p_;
};

// page-locked host buffers, reused: what the device copies into (container bytes, FASTQ text) before the sink / the caller
// gets it.  Fresh pageable memory per batch costs a page fault per 4 KB and a staged copy; these cost neither.
struct PinnedBuf {
    uint8_t* p = nullptr;
    size_t cap = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf&) = delete;
    PinnedBuf& operator=(const PinnedBuf&) = delete;
    ~PinnedBuf() { idn_gpu_host_free(p); }
    void ensure(size_t n);                 // contents are not kept
    void ensure_keep(size_t n, size_t used);  // the first `used` bytes are
};
// One pool per process: page-locking memory costs about as much per byte as the page faults it avoids, so the buffers
// outlive the compressor / decompressor that asked for them (release_cached_resources() gives them back).
class PinnedPool {
public:
    std::shared_ptr<PinnedBuf> get(size_t n);  // a buffer of at least n bytes; goes back to the pool when the last owner lets go
    static void trim();
private:
    struct State {
        std::mutex mu;
        std::vector<std::unique_ptr<PinnedBuf>> free_;
    };
    static State& state();
};
// frees the page-locked buffers and device contexts the library keeps for the next compressor / decompressor
void release_cached_resources();

// RAII over idn_gpu_ctx + the handles of the uploaded models of one provider
class DeviceModels {
public:
    DeviceModels() = default;
    ~DeviceModels();
    DeviceModels(const DeviceModels&) = delete;
    DeviceModels& operator=(const DeviceModels&) = delete;
    void open(int32_t device);  // a context from the process-wide cache (its device buffers are already sized) or a new one
    // the handles of the provider's models, in its order.  Models stay resident in the context (keyed by their identifier)
    // when the object closes and the context goes back to the cache: the next compressor / decompressor with the same
    // models finds them there instead of paying cudaMalloc / cudaFree (which synchronise the device: 0.03 - 3 s measured).
    void upload(const ModelProvider& provider);
    idn_gpu_ctx* ctx() const { return ctx_; }
    const std::vector<idn_model_t>& handles() const { return handles_; }
    [[noreturn]] void raise(int32_t rc) const;  // IdnError from idn_gpu_last_error
    void mark_broken() const { broken_ = true; }

private:
    idn_gpu_ctx* ctx_ = nullptr;
    int32_t device_ = 0;
    mutable bool broken_ = false;  // a CUDA error was reported on this context: it is destroyed, not kept for the next object
    std::vector<idn_model_t> handles_;
    std::vector<std::pair<ModelIdentifier, idn_model_t>> resident_;  // every model this context holds
};

class IdnCompressor {
public:
    using Sink = std::function<void(const uint8_t*, size_t)>;  // the reference's `W: Write`
    IdnCompressor(Sink sink, IdnCompressorParams params);  // IdnCompressor::with_params
    ~IdnCompressor();
    void add_sequence(FastqSequence seq);  // SequenceTooLong when len > max_block_total_len / 2 (idn/compressor.rs:542-544)
    // the same for many sequences at once, given as one SoA batch (what a FASTQ parser produces); blocks form exactly as
    // if add_sequence had been called per read.  name_off / names may be NULL (empty identifiers).
    void add_batch(uint64_t n_reads, const uint64_t* read_off, const uint8_t* acids, const uint8_t* quals, const uint64_t* name_off,
                   const uint8_t* names);
    // FASTQ text instead of parsed sequences (what FastqReader + add_sequence do in the reference, fastq/reader.rs:166-282):
    // any number of calls with consecutive pieces of the text, cut anywhere.  The text is split into records, turned into
    // blocks and compressed on the device; identifiers come back for the host's Deflate.  The container is the one
    // add_sequence would have produced for the same reads.  Not to be mixed with add_sequence / add_batch on one object.
    void add_fastq_text(const uint8_t* text, size_t n);
    void finish();                         // flushes, writes the empty terminator block; InvalidState if called twice
    const CompressionStats& stats() const { return stats_; }  // (the out_* fields are final after finish())
    // the model identifiers written to the metadata (acid ids first), available after the first block was processed
    const std::vector<ModelIdentifier>& retained_models() const { return retained_; }

private:
    struct Batch {  // SoA batch of whole blocks
        std::vector<uint8_t> acids, quals, names;
        std::vector<uint64_t> read_off{0}, name_off{0};
        std::vector<uint32_t> block_first{0};
        void clear() {
            acids.clear();
            quals.clear();
            names.clear();
            read_off.assign(1, 0);
            name_off.assign(1, 0);
            block_first.assign(1, 0);
        }
    };
    struct Result {  // one compressed batch, ready to be written
        std::shared_ptr<PinnedBuf> buf;  // page-locked, pooled
        uint64_t out_bytes = 0, prefix_total = 0, payload_bytes = 0, acid_switches = 0, q_switches = 0, blocks = 0;
    };
    struct Worker {  // one device: its context, its uploaded models; one job at a time (a job may change threads)
        DeviceModels dev;
        std::mutex mu;
        std::condition_variable cv;
        bool busy = false;
        void acquire() {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [this] { return !busy; });
            busy = true;
        }
        void release() {
            {
                std::lock_guard<std::mutex> lk(mu);
                busy = false;
            }
            cv.notify_one();
        }
    };
    size_t consume_text(const uint8_t* buf, size_t total, bool final);
    Result compress_parsed(Worker& w, uint32_t n_blocks, uint64_t n_reads, uint64_t n_symbols, uint64_t n_name_bytes) const;
    Result compress_parsed_ids(Worker& w, uint32_t n_blocks, uint64_t n_reads, uint64_t n_symbols, uint64_t n_name_bytes) const;
    void make_block();
    void flush_batch();  // hands the batch under construction to the next device
    void commit(bool all);  // writes finished batches in order (the reference's IdnBlockLock, idn/common.rs:10-57)
    Result compress_batch(Worker& w, const Batch& b) const;
    void initialize();  // CompressorInitializer::initialize (idn/compressor_initializer.rs:33-74)
    std::vector<ModelIdentifier> best_models(ModelType type, size_t model_num, const std::vector<uint32_t>& sizes,
                                             const std::vector<size_t>& cols, size_t n_cols, size_t n_reads, class Clustering& clustering);

    Sink sink_;
    IdnCompressorParams params_;
    std::vector<std::unique_ptr<Worker>> workers_;  // one per entry of params_.devices
    size_t next_worker_ = 0;
    mutable PinnedPool pool_;
    // Batches in flight, in block order.  A writer thread takes the results off the front as they complete and hands them
    // to the sink (ONE thread, in order: this replaces IdnBlockLock, common.rs:10-57), so the thread that adds sequences or
    // text does not spend its time in the sink; it only waits when more than two batches per device are pending.
    std::deque<std::future<Result>> pending_;
    std::mutex wmu_;                // pending_, writer_stop_, writer_err_, the out_* fields of stats_
    std::condition_variable wcv_;
    std::thread writer_;
    bool writer_stop_ = false;
    std::exception_ptr writer_err_;  // what a job or the sink threw; rethrown by the next add_* / finish
    void submit(std::future<Result> f);
    void writer_loop();
    CompressionStats stats_;
    std::vector<ModelIdentifier> retained_;
    bool initialized_ = false, finished_ = false;
    Batch cur_;  // SoA batch under construction
    uint64_t cur_block_len_ = 0;
    std::vector<uint8_t> text_;  // add_fastq_text: what the calls so far left unconsumed (at most about a block's worth of text)
    bool text_mode_ = false;
};

struct IdnDecompressorParams {
    ModelProvider model_provider;
    uint32_t thread_num = 0;
    std::vector<int32_t> devices{0};  // batches of `batch_blocks` blocks go round robin to these GPUs, results come back in order
    uint32_t batch_blocks = 32;
    // inflate the Identifiers slices on the device (idn_gpu_inflate_names) instead of with zlib on thread_num host threads;
    // a batch with a Brotli slice falls back to the host
    bool identifiers_on_device = false;
};

class IdnDecompressor {
public:
    using Source = std::function<size_t(uint8_t*, size_t)>;  // reads up to n bytes, returns the count (0 = end of input)
    IdnDecompressor(Source source, IdnDecompressorParams params);  // IdnDecompressor::with_params
    // the container in memory: the blocks are uploaded from where they lie (no copy into the library's buffers; full link
    // rate when the memory is page-locked).  [data, data + len) must stay valid while the object lives.
    IdnDecompressor(const uint8_t* data, size_t len, IdnDecompressorParams params);
    ~IdnDecompressor();
    std::optional<FastqSequence> next_sequence();  // None at the end of the file
    uint8_t version() const { return version_; }

    // the decoded sequences of the next batch as one SoA batch instead of one FastqSequence at a time (what a FASTQ writer
    // consumes); false at the end of the file.  Do not mix with next_sequence on one object.
    struct DecodedBatch {
        std::vector<uint8_t> acids, quals, names;
        std::vector<uint64_t> read_off{0}, name_off{0};
        bool any_names = false;
        std::shared_ptr<PinnedBuf> text;  // next_fastq_text: the FASTQ text (page-locked, pooled)
        size_t text_len = 0;
    };
    bool next_batch(DecodedBatch& out);
    // the FASTQ text of the next batch of sequences, formatted on the device as FastqWriter does (fastq/writer.rs:190-245);
    // false at the end of the file.  Do not mix with next_sequence / next_batch on one object.
    bool next_fastq_text(std::shared_ptr<PinnedBuf>& out, size_t& len, bool title_with_separator = false);

private:
    struct RawBatch {  // container bytes of some blocks, as read from the source
        std::shared_ptr<PinnedBuf> buf;  // page-locked, pooled: the device reads it at the link's rate
        const uint8_t* base = nullptr;   // buf->p, or the position of the first payload in the caller's memory
        size_t used = 0;                 // bytes from base to the end of the last payload
        std::vector<uint64_t> off;
        std::vector<uint32_t> len, crc;
    };
    struct Worker {
        DeviceModels dev;
        std::mutex mu;
    };
    void initialize();  // header + metadata (idn/decompressor.rs:304-374)
    bool read_raw(RawBatch& rb);  // false once the terminator block was seen (and rb holds no block)
    DecodedBatch decode_batch(Worker& w, const RawBatch& rb) const;
    DecodedBatch decode_text(Worker& w, const RawBatch& rb, bool title_with_separator) const;  // text in DecodedBatch::acids
    // identifiers_on_device: idn_gpu_inflate_names of the batch indexed last; false when it holds a Brotli slice
    bool inflate_names_device(Worker& w, const RawBatch& rb, const std::vector<uint64_t>& off, const std::vector<uint32_t>& block_first,
                              uint64_t n_reads, DecodedBatch& out, bool fetch, uint64_t* n_name_bytes) const;
    void inflate_names(const RawBatch& rb, const std::vector<uint64_t>& off, const std::vector<uint32_t>& block_first, uint64_t n_reads,
                       DecodedBatch& out) const;
    void prefetch();
    void read_exact(uint8_t* dst, size_t n, const char* what);

    Source source_;
    const uint8_t* mem_ = nullptr;  // the in-memory form
    size_t mem_len_ = 0, mem_pos_ = 0;
    IdnDecompressorParams params_;
    std::vector<std::unique_ptr<Worker>> workers_;
    size_t next_worker_ = 0;
    mutable PinnedPool pool_;
    std::deque<std::future<DecodedBatch>> pending_;
    int text_mode_ = 0;  // 0 sequences / batches, 1 text, 2 text with the title repeated on the separator line
    bool initialized_ = false, eof_ = false;
    uint8_t version_ = 0;
    std::deque<FastqSequence> queue_;
};

}  // namespace idencomp
