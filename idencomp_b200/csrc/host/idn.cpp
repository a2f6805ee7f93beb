// idn.cpp -- see idn.hpp.  Host orchestration only: every symbol goes through the C-ABI of libidn_gpu.so.
#include "idn.hpp"

#include "clustering.hpp"

#include <dlfcn.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <numeric>

namespace idencomp {

namespace {

template <class W>
struct WorkerLease {  // a ctx is single-owner: one job at a time per worker
    W& w;
    bool adopted;
    explicit WorkerLease(W& w_, bool already_acquired = false) : w(w_), adopted(already_acquired) {
        if (!adopted) w.acquire();
    }
    ~WorkerLease() { w.release(); }
};

constexpr char kMagic[8] = {'I', 'D', 'E', 'N', 'C', 'O', 'M', 'P'};  // idn/data.rs:3-8

void put_u32be(std::vector<uint8_t>& b, uint32_t v) {
    b.push_back((uint8_t)(v >> 24));
    b.push_back((uint8_t)(v >> 16));
    b.push_back((uint8_t)(v >> 8));
    b.push_back((uint8_t)v);
}
uint32_t get_u32be(const uint8_t* p) { return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3]; }

// names slice: raw Deflate at flate2's default level (compressor_block.rs:146-206).  zlib and miniz_oxide emit
// different but equally valid streams, so this slice is compared after inflation (DESIGN.md section 7).
std::vector<uint8_t> deflate_raw(const uint8_t* src, size_t n) {
    z_stream z;
    std::memset(&z, 0, sizeof z);
    if (deflateInit2(&z, 6, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) throw IdnError(IDN_E_IO, "deflateInit2 failed");
    std::vector<uint8_t> out(deflateBound(&z, (uLong)n) + 64);
    z.next_in = const_cast<Bytef*>(src);
    z.avail_in = (uInt)n;
    z.next_out = out.data();
    z.avail_out = (uInt)out.size();
    int rc = deflate(&z, Z_FINISH);
    deflateEnd(&z);
    if (rc != Z_STREAM_END) throw IdnError(IDN_E_IO, "deflate failed");
    out.resize(out.size() - z.avail_out);
    return out;
}

std::vector<uint8_t> inflate_raw(const uint8_t* src, size_t n) {
    z_stream z;
    std::memset(&z, 0, sizeof z);
    if (inflateInit2(&z, -15) != Z_OK) throw IdnError(IDN_E_IO, "inflateInit2 failed");
    std::vector<uint8_t> out;
    z.next_in = const_cast<Bytef*>(src);
    z.avail_in = (uInt)n;
    int rc;
    do {
        size_t old = out.size();
        out.resize(old + 65536);
        z.next_out = out.data() + old;
        z.avail_out = 65536;
        rc = inflate(&z, Z_NO_FLUSH);
        out.resize(old + 65536 - z.avail_out);
    } while (rc == Z_OK);
    inflateEnd(&z);
    if (rc != Z_STREAM_END) throw IdnError(IDN_E_SERIALIZE, "identifiers slice does not inflate");
    return out;
}

// Brotli for the identifiers of quality 8-9 (compressor_block.rs:160-170: buffer 4096, quality 11, lgwin 20).  The image
// ships libbrotlienc/libbrotlidec without headers, so the four entry points are bound at run time; when the libraries
// are absent the quality 8-9 identifier path fails with Unsupported.  The byte stream of the C encoder differs from the
// Rust crate's (as zlib's does from miniz_oxide's): this slice is compared after decompression.
struct Brotli {
    using EncFn = int (*)(int quality, int lgwin, int mode, size_t in_size, const uint8_t* in, size_t* out_size, uint8_t* out);
    using BoundFn = size_t (*)(size_t);
    using CreateFn = void* (*)(void*, void*, void*);
    using StreamFn = int (*)(void* state, size_t* avail_in, const uint8_t** next_in, size_t* avail_out, uint8_t** next_out, size_t* total_out);
    using DestroyFn = void (*)(void*);
    EncFn enc = nullptr;
    BoundFn bound = nullptr;
    CreateFn create = nullptr;
    StreamFn stream = nullptr;
    DestroyFn destroy = nullptr;
    Brotli() {
        void* e = dlopen("libbrotlienc.so.1", RTLD_NOW | RTLD_LOCAL);
        void* d = dlopen("libbrotlidec.so.1", RTLD_NOW | RTLD_LOCAL);
        if (e) {
            enc = (EncFn)dlsym(e, "BrotliEncoderCompress");
            bound = (BoundFn)dlsym(e, "BrotliEncoderMaxCompressedSize");
        }
        if (d) {
            create = (CreateFn)dlsym(d, "BrotliDecoderCreateInstance");
            stream = (StreamFn)dlsym(d, "BrotliDecoderDecompressStream");
            destroy = (DestroyFn)dlsym(d, "BrotliDecoderDestroyInstance");
        }
    }
    static Brotli& get() {
        static Brotli b;
        return b;
    }
    std::vector<uint8_t> compress(const uint8_t* src, size_t n) const {
        if (!enc || !bound) throw IdnError(IDN_E_UNSUPPORTED, "Brotli identifier slices (quality 8-9) need libbrotlienc.so.1");
        size_t cap = bound(n) + 64;
        std::vector<uint8_t> out(cap);
        if (!enc(11, 20, 0, n, src, &cap, out.data())) throw IdnError(IDN_E_IO, "Brotli compression failed");
        out.resize(cap);
        return out;
    }
    std::vector<uint8_t> decompress(const uint8_t* src, size_t n) const {
        if (!create || !stream || !destroy) throw IdnError(IDN_E_UNSUPPORTED, "Brotli identifier slices need libbrotlidec.so.1");
        void* st = create(nullptr, nullptr, nullptr);
        if (!st) throw IdnError(IDN_E_IO, "BrotliDecoderCreateInstance failed");
        std::vector<uint8_t> out(std::max<size_t>(65536, 8 * n));
        size_t avail_in = n, total = 0;
        const uint8_t* next_in = src;
        int rc;
        for (;;) {
            size_t avail_out = out.size() - total;
            uint8_t* next_out = out.data() + total;
            rc = stream(st, &avail_in, &next_in, &avail_out, &next_out, nullptr);
            total = out.size() - avail_out;
            if (rc != 3) break;  // BROTLI_DECODER_RESULT_NEEDS_MORE_OUTPUT
            out.resize(out.size() * 2);
        }
        destroy(st);
        if (rc != 1) throw IdnError(IDN_E_SERIALIZE, "identifiers slice is not a valid Brotli stream");  // 1 = SUCCESS
        out.resize(total);
        return out;
    }
};

}  // namespace

// ---- IDN_HOST_TRACE=1: wall time per stage of the host mirror, summed over threads, printed when an object closes -----------
namespace {
struct Trace {
    static constexpr int kN = 17;
    const char* name[kN] = {"parse_chunk", "first_block_select", "names_fetch", "names_deflate", "compress_parsed", "compress_blocks",
                            "sink", "read_raw", "index_blocks", "names_inflate", "decode", "wait_worker", "open", "initialize", "wait_result",
                            "close", "names_inflate_device"};
    std::atomic<uint64_t> ns[kN];
    std::atomic<uint64_t> calls[kN];
    bool on = std::getenv("IDN_HOST_TRACE") != nullptr;
    Trace() {
        for (int i = 0; i < kN; i++) ns[i] = calls[i] = 0;
    }
    void print(const char* who) {
        if (!on) return;
        std::fprintf(stderr, "[idn_host trace] %s:", who);
        for (int i = 0; i < kN; i++)
            if (calls[i]) std::fprintf(stderr, " %s %.1f ms/%llu", name[i], ns[i].exchange(0) / 1e6, (unsigned long long)calls[i].exchange(0));
        std::fprintf(stderr, "\n");
    }
};
Trace g_trace;
struct Span {
    int k;
    std::chrono::steady_clock::time_point t0;
    explicit Span(int k_) : k(k_) {
        if (g_trace.on) t0 = std::chrono::steady_clock::now();
    }
    ~Span() {
        if (!g_trace.on) return;
        g_trace.ns[k] += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
        g_trace.calls[k]++;
    }
};
std::atomic<size_t> g_raw_hint{1 << 20};  // bytes of the largest batch of container bytes read so far (sizes the next buffer)
enum { T_PARSE, T_SELECT, T_NFETCH, T_NDEFLATE, T_CPARSED, T_CBLOCKS, T_SINK, T_READRAW, T_INDEX, T_NINFLATE, T_DECODE, T_WAIT, T_OPEN, T_INIT, T_WAITRES, T_CLOSE,
       T_NINFLATE_DEV };
}  // namespace

// ---- page-locked buffers -------------------------------------------------------------------------------------------------
void PinnedBuf::ensure(size_t n) {
    if (n <= cap) return;
    idn_gpu_host_free(p);
    p = nullptr;
    cap = 0;
    void* q = nullptr;
    const size_t want = n + n / 8 + 4096;
    if (idn_gpu_host_alloc(want, &q) != IDN_OK) throw IdnError(IDN_E_IO, "cannot allocate " + std::to_string(want) + " bytes of page-locked host memory");
    p = static_cast<uint8_t*>(q);
    cap = want;
}

void PinnedBuf::ensure_keep(size_t n, size_t used) {
    if (n <= cap) return;
    void* q = nullptr;
    const size_t want = n + n / 2 + 4096;
    if (idn_gpu_host_alloc(want, &q) != IDN_OK) throw IdnError(IDN_E_IO, "cannot allocate " + std::to_string(want) + " bytes of page-locked host memory");
    if (used) std::memcpy(q, p, used);
    idn_gpu_host_free(p);
    p = static_cast<uint8_t*>(q);
    cap = want;
}

PinnedPool::State& PinnedPool::state() {
    static State* st = new State;  // never destroyed: at process exit the CUDA runtime may be gone before static destructors run
    return *st;
}

std::shared_ptr<PinnedBuf> PinnedPool::get(size_t n) {
    // Sizes are rounded up to a size class (1 MB at least) and a buffer is never regrown for a larger request: requests of
    // about the same size then find each other's buffers whatever order the worker threads ask in, and the pool stops
    // allocating once it has seen the peak number of buffers in flight per size class.
    size_t cls = 1 << 20;
    while (cls < n) cls <<= 1;
    if (cls > (1 << 20)) {  // eighths of the power of two above n: at most 12.5 % over
        const size_t step = cls >> 4;
        cls = (n + step - 1) / step * step;
    }
    State& st = state();
    std::unique_ptr<PinnedBuf> b;
    {
        std::lock_guard<std::mutex> lk(st.mu);
        size_t pick = st.free_.size();
        for (size_t i = 0; i < st.free_.size(); i++)
            if (st.free_[i]->cap >= n && (pick == st.free_.size() || st.free_[i]->cap < st.free_[pick]->cap)) pick = i;
        if (pick < st.free_.size()) {
            b = std::move(st.free_[pick]);
            st.free_.erase(st.free_.begin() + pick);
        }
    }
    if (!b) {
        b = std::make_unique<PinnedBuf>();
        void* q = nullptr;
        if (idn_gpu_host_alloc(cls, &q) != IDN_OK) throw IdnError(IDN_E_IO, "cannot allocate " + std::to_string(cls) + " bytes of page-locked host memory");
        b->p = static_cast<uint8_t*>(q);
        b->cap = cls;
    }
    return std::shared_ptr<PinnedBuf>(b.release(), [](PinnedBuf* q) {
        State& s2 = state();
        std::lock_guard<std::mutex> lk(s2.mu);
        s2.free_.emplace_back(q);
    });
}

void PinnedPool::trim() {
    State& st = state();
    std::lock_guard<std::mutex> lk(st.mu);
    st.free_.clear();
}

// device contexts between uses: a context's staging and work buffers on the device are sized by the batches it has seen,
// and allocating them again for every compressor costs more than compressing a few GB
namespace {
struct CachedCtx {
    int32_t first;  // device
    idn_gpu_ctx* second;
    std::vector<std::pair<ModelIdentifier, idn_model_t>> resident;  // models left on it
};
struct CtxCache {
    std::mutex mu;
    std::vector<CachedCtx> free_;
    static constexpr size_t kKeepPerDevice = 8;
};
CtxCache& ctx_cache() {
    static CtxCache* c = new CtxCache;
    return *c;
}
}  // namespace

void release_cached_resources() {
    PinnedPool::trim();
    CtxCache& c = ctx_cache();
    std::lock_guard<std::mutex> lk(c.mu);
    for (auto& e : c.free_) idn_gpu_destroy(e.second);  // (with the models left on it)
    c.free_.clear();
}

// ---- DeviceModels ---------------------------------------------------------------------------------------------------
DeviceModels::~DeviceModels() {
    if (!ctx_) return;
    CtxCache& c = ctx_cache();
    std::lock_guard<std::mutex> lk(c.mu);
    size_t same = 0;
    for (auto& e : c.free_) same += e.first == device_;
    if (!broken_ && same < CtxCache::kKeepPerDevice) c.free_.push_back(CachedCtx{device_, ctx_, std::move(resident_)});
    else idn_gpu_destroy(ctx_);  // (frees its models too)
}
void DeviceModels::open(int32_t device) {
    if (ctx_) return;
    device_ = device;
    {
        CtxCache& c = ctx_cache();
        std::lock_guard<std::mutex> lk(c.mu);
        for (size_t i = c.free_.size(); i-- > 0;)  // the one released last: objects opened and closed in the same order get the
            if (c.free_[i].first == device) {        // contexts they had before, with the buffers of their role already sized
                ctx_ = c.free_[i].second;
                resident_ = std::move(c.free_[i].resident);
                c.free_.erase(c.free_.begin() + i);
                return;
            }
    }
    int32_t rc = idn_gpu_create(device, &ctx_);
    if (rc) throw IdnError(rc, "no usable CUDA device (this implementation has no CPU fallback)");
}
void DeviceModels::raise(int32_t rc) const {
    if (rc == IDN_E_CUDA) broken_ = true;
    throw IdnError(rc, ctx_ ? idn_gpu_last_error(ctx_) : "no device context");
}
void DeviceModels::upload(const ModelProvider& provider) {
    constexpr size_t kKeepResident = 64;  // models a context keeps beyond the ones in use
    handles_.clear();
    std::vector<char> used(resident_.size(), 0);
    for (size_t i = 0; i < provider.len(); i++) {
        const ModelIdentifier& id = provider[i].identifier();
        size_t k = 0;
        while (k < resident_.size() && resident_[k].first != id) k++;
        if (k == resident_.size()) {
            idn_model_t h = -1;
            int32_t rc = upload_model(ctx_, provider[i], &h);
            if (rc) raise(rc);
            resident_.emplace_back(id, h);
            used.push_back(0);
        }
        used[k] = 1;
        handles_.push_back(resident_[k].second);
    }
    // the oldest unused ones go when the context holds too many
    for (size_t k = 0; k < resident_.size() && resident_.size() > provider.len() + kKeepResident;) {
        if (used[k]) {
            k++;
            continue;
        }
        idn_gpu_model_release(ctx_, resident_[k].second);
        resident_.erase(resident_.begin() + k);
        used.erase(used.begin() + k);
    }
}

IdnCompressorParamsBuilder& IdnCompressorParamsBuilder::quality(uint8_t v) {
    if (v < 1 || v > 9) throw std::invalid_argument("compression quality must be between 1 and 9");
    p_.quality = v;
    return *this;
}

// ---- IdnCompressor ---------------------------------------------------------------------------------------------------
IdnCompressor::IdnCompressor(Sink sink, IdnCompressorParams params) : sink_(std::move(sink)), params_(std::move(params)) {
    if (params_.fast) params_.quality = 1;  // IdnCompressorParamsBuilder::fast (idn/compressor.rs:244-251)
    if (params_.mode != IDN_MODE_COMPAT && params_.mode != IDN_MODE_NATIVE) throw IdnError(IDN_E_INVALID_STATE, "unknown container mode");
    if (params_.identifiers_on_device && params_.include_identifiers && params_.quality >= 8)
        throw IdnError(IDN_E_UNSUPPORTED, "identifiers_on_device: quality 8-9 codes identifiers with Brotli, which has no device codec");
    if (params_.devices.empty()) params_.devices.assign(1, 0);
    if (params_.batch_blocks == 0) params_.batch_blocks = 1;
    for (int32_t d : params_.devices) {
        workers_.push_back(std::make_unique<Worker>());
        workers_.back()->dev.open(d);
        if (params_.mode == IDN_MODE_NATIVE) {
            int32_t rc = idn_gpu_set_lane_symbols(workers_.back()->dev.ctx(), params_.lane_symbols);
            if (rc) workers_.back()->dev.raise(rc);
        }
    }
}

IdnCompressor::~IdnCompressor() {
    if (writer_.joinable()) {  // the writer drains what is pending (jobs still running hold references to this object)
        {
            std::lock_guard<std::mutex> lk(wmu_);
            writer_stop_ = true;
        }
        wcv_.notify_all();
        writer_.join();
    }
    for (auto& f : pending_)
        if (f.valid()) f.wait();
}

void IdnCompressor::add_sequence(FastqSequence seq) {
    if (seq.acids.size() != seq.quality_scores.size()) throw IdnError(IDN_E_INVALID_STATE, "acids and quality scores differ in length");
    const uint64_t ro[2] = {0, seq.acids.size()}, no[2] = {0, seq.identifier.size()};
    add_batch(1, ro, seq.acids.data(), seq.quality_scores.data(), no, reinterpret_cast<const uint8_t*>(seq.identifier.data()));
}

void IdnCompressor::add_batch(uint64_t n_reads, const uint64_t* read_off, const uint8_t* acids, const uint8_t* quals,
                              const uint64_t* name_off, const uint8_t* names) {
    if (finished_) throw IdnError(IDN_E_INVALID_STATE, "add_sequence after finish");
    if (text_mode_) throw IdnError(IDN_E_INVALID_STATE, "add_sequence after add_fastq_text");
    uint64_t r = 0;
    while (r < n_reads) {
        // the run of reads [r, e) that goes into the batch under construction: block forming per read exactly as
        // IdnCompressor::add_sequence does it (idn/compressor.rs:517-544); a full batch ends the run
        uint64_t e = r;
        const size_t sym0 = cur_.acids.size();
        const uint64_t base = read_off[r];
        bool dispatched = false;
        while (e < n_reads && !dispatched) {
            const uint64_t len = read_off[e + 1] - read_off[e];
            if (len > params_.max_block_total_len / 2)  // idn/compressor.rs:542-544
                throw IdnError(IDN_E_SEQUENCE_TOO_LONG, "sequence too long: " + std::to_string(len) + " > " + std::to_string(params_.max_block_total_len / 2));
            if (cur_block_len_ + len > params_.max_block_total_len) {  // :526-540
                const uint32_t n = (uint32_t)(cur_.read_off.size() - 1);
                if (n != cur_.block_first.back()) {
                    cur_.block_first.push_back(n);
                    cur_block_len_ = 0;
                    if (cur_.block_first.size() - 1 >= params_.batch_blocks) {
                        dispatched = true;  // the run ends in front of read e; the batch goes out below
                        break;
                    }
                }
            }
            cur_.read_off.push_back(sym0 + (read_off[e + 1] - base));
            const uint64_t nl = (params_.include_identifiers && name_off) ? name_off[e + 1] - name_off[e] : 0;
            cur_.name_off.push_back(cur_.name_off.back() + nl);
            cur_block_len_ += len;
            stats_.in_symbols += len;
            stats_.in_reads++;
            stats_.in_identifier_bytes += name_off ? name_off[e + 1] - name_off[e] : 0;
            e++;
        }
        if (e > r) {
            cur_.acids.insert(cur_.acids.end(), acids + read_off[r], acids + read_off[e]);
            cur_.quals.insert(cur_.quals.end(), quals + read_off[r], quals + read_off[e]);
            if (params_.include_identifiers && name_off && names) cur_.names.insert(cur_.names.end(), names + name_off[r], names + name_off[e]);
        }
        if (dispatched) flush_batch();
        r = e;
    }
}

void IdnCompressor::make_block() {
    const uint32_t n_reads = (uint32_t)(cur_.read_off.size() - 1);
    if (n_reads == cur_.block_first.back()) return;  // nothing since the last block
    cur_.block_first.push_back(n_reads);
    cur_block_len_ = 0;
    if (cur_.block_first.size() - 1 >= params_.batch_blocks) flush_batch();
}

std::vector<ModelIdentifier> IdnCompressor::best_models(ModelType type, size_t model_num, const std::vector<uint32_t>& sizes,
                                                        const std::vector<size_t>& cols, size_t n_cols, size_t n_reads,
                                                        Clustering& clustering) {
    // cost matrix of this type's models only
    const size_t n = cols.size();
    std::vector<uint32_t> cost(n_reads * n);
    for (size_t r = 0; r < n_reads; r++)
        for (size_t k = 0; k < n; k++) cost[r * n + k] = sizes[r * n_cols + cols[k]];
    std::vector<size_t> pick = params_.quality >= 2 ? clustering.make_clusters(cost, n_reads, n, model_num, nullptr)  // CLUSTERING_THRESHOLD
                                                    : rank_models(cost, n_reads, n, model_num);
    std::vector<ModelIdentifier> ids;
    for (size_t k : pick) ids.push_back(params_.model_provider[cols[k]].identifier());
    (void)type;
    return ids;
}

void IdnCompressor::initialize() {
    ModelProvider& mp = params_.model_provider;
    DeviceModels& dev0 = workers_[0]->dev;  // the file-level selection runs on the first device
    std::vector<size_t> of_type[2];
    for (size_t i = 0; i < mp.len(); i++) of_type[(size_t)mp[i].model_type()].push_back(i);
    if (of_type[0].empty() || of_type[1].empty()) throw IdnError(IDN_E_INVALID_STATE, "the model provider needs at least one model per type");
    const size_t model_num = ((size_t)params_.quality + 1) / 2;  // compressor_initializer.rs:56
    std::vector<ModelIdentifier> ids;
    if (of_type[0].size() == 1 && of_type[1].size() == 1) {  // "Only one model registered" (model_chooser.rs:37-40)
        ids = {mp[of_type[0][0]].identifier(), mp[of_type[1][0]].identifier()};
    } else {
        // cost matrix over the reads of the FIRST block with every model of the provider (a6 on the device)
        dev0.upload(mp);
        const uint64_t n_reads = cur_.block_first.size() > 1 ? cur_.block_first[1] : cur_.read_off.size() - 1;
        std::vector<uint32_t> sizes(n_reads * mp.len());
        idn_batch b{};
        b.n_reads = n_reads;
        b.n_symbols = cur_.read_off[n_reads];
        b.acids = cur_.acids.data();
        b.quals = cur_.quals.data();
        b.read_off = cur_.read_off.data();
        if (n_reads) {
            int32_t rc = idn_gpu_score(dev0.ctx(), &b, dev0.handles().data(), (uint32_t)mp.len(), sizes.data());
            if (rc) dev0.raise(rc);
        }
        // ONE Clustering (one random stream) serves the acid models and then the q-score models, as the reference's
        // ModelChooser does (model_chooser.rs:14-24, compressor_initializer.rs:57-64)
        Clustering clustering;
        for (int t = 0; t < 2; t++) {
            std::vector<ModelIdentifier> got;
            if (of_type[t].size() == 1) got = {mp[of_type[t][0]].identifier()};
            else got = best_models((ModelType)t, model_num, sizes, of_type[t], mp.len(), n_reads, clustering);
            ids.insert(ids.end(), got.begin(), got.end());
        }
    }
    mp.filter_by_identifiers(ids);  // acid ids first, then q-score ids (compressor_initializer.rs:57-74)
    if (mp.len() > IDN_MAX_MODELS) throw IdnError(IDN_E_UNSUPPORTED, "too many retained models");
    for (auto& w : workers_) w->dev.upload(mp);  // every device holds the retained models
    retained_ = ids;
    // header + metadata (writer_idn.rs:25-59, data.rs:3-33)
    std::vector<uint8_t> h(kMagic, kMagic + 8);
    h.push_back((uint8_t)(params_.mode == IDN_MODE_NATIVE ? 2 : 1));
    h.push_back(1);  // item_num
    h.push_back(0);  // IdnMetadataItem::Models
    h.push_back((uint8_t)ids.size());
    for (auto& id : ids) h.insert(h.end(), id.begin(), id.end());
    sink_(h.data(), h.size());
    stats_.out_bytes += h.size();
    initialized_ = true;
}

// identifiers slices on host threads, like write_identifiers (compressor_block.rs:146-206): names joined by '\n', Deflate
// (Brotli from quality 8 on), one slice per block
static void identifier_slices(uint8_t quality, uint32_t thread_num, uint32_t n_blocks, const uint32_t* block_first, const uint8_t* names,
                              const uint64_t* name_off, std::vector<std::vector<uint8_t>>& name_slices, std::vector<uint32_t>& prefix) {
    const bool brotli = quality >= 8;  // BROTLI_THRESHOLD (compressor_block.rs:146)
    if (brotli && !Brotli::get().enc) throw IdnError(IDN_E_UNSUPPORTED, "Brotli identifier slices (quality 8-9) need libbrotlienc.so.1");
    auto one = [&](uint32_t b) {
        std::vector<uint8_t> joined;
        for (uint32_t r = block_first[b]; r < block_first[b + 1]; r++) {
            if (r > block_first[b]) joined.push_back('\n');
            joined.insert(joined.end(), names + name_off[r], names + name_off[r + 1]);
        }
        std::vector<uint8_t> z = brotli ? Brotli::get().compress(joined.data(), joined.size()) : deflate_raw(joined.data(), joined.size());
        std::vector<uint8_t> s;
        s.push_back(0x00);  // IdnSliceHeader::Identifiers (data.rs:46-47)
        put_u32be(s, (uint32_t)z.size());
        s.push_back(brotli ? 0 : 1);  // IdnIdentifierCompression::{Brotli = 0, Deflate = 1} (data.rs:57-61)
        s.insert(s.end(), z.begin(), z.end());
        name_slices[b] = std::move(s);
    };
    if (thread_num > 1) {  // thread_num workers take the blocks in turn
        std::vector<std::future<void>> jobs;
        std::atomic<uint32_t> next{0};
        for (uint32_t t = 0; t < std::min<uint32_t>(thread_num, n_blocks); t++)
            jobs.push_back(std::async(std::launch::async, [&] {
                for (uint32_t b = next++; b < n_blocks; b = next++) one(b);
            }));
        for (auto& j : jobs) j.get();
    } else {
        for (uint32_t b = 0; b < n_blocks; b++) one(b);
    }
    for (uint32_t b = 0; b < n_blocks; b++) prefix[b] = (uint32_t)name_slices[b].size();
}

// one batch on one device: identifiers slices on host threads, everything else through the C-ABI
IdnCompressor::Result IdnCompressor::compress_batch(Worker& w, const Batch& bt) const {
    WorkerLease<Worker> lease(w);
    Result res;
    const uint32_t n_blocks = (uint32_t)(bt.block_first.size() - 1);
    const uint64_t n_reads = bt.block_first.back();
    std::vector<std::vector<uint8_t>> name_slices(n_blocks);
    std::vector<uint32_t> prefix(n_blocks, 0);
    std::shared_ptr<PinnedBuf> dev_slices;  // identifiers_on_device: the slices back to back ...
    std::vector<uint64_t> slice_off;        // ... block k's at slice_off[k]
    if (params_.include_identifiers && params_.identifiers_on_device) {
        Span sp(T_NDEFLATE);
        const uint8_t* names = bt.names.empty() ? reinterpret_cast<const uint8_t*>("") : bt.names.data();
        const uint64_t cap = idn_gpu_deflate_names_bound(bt.name_off[n_reads] - bt.name_off[0], n_reads, n_blocks);
        dev_slices = pool_.get(cap);
        slice_off.resize(n_blocks + 1);
        int32_t rc = idn_gpu_deflate_names(w.dev.ctx(), names, bt.name_off.data(), bt.block_first.data(), n_blocks, dev_slices->p, cap, slice_off.data());
        if (rc) w.dev.raise(rc);
        for (uint32_t k = 0; k < n_blocks; k++) prefix[k] = (uint32_t)(slice_off[k + 1] - slice_off[k]);
    } else if (params_.include_identifiers) {
        identifier_slices(params_.quality, params_.thread_num, n_blocks, bt.block_first.data(), bt.names.data(), bt.name_off.data(), name_slices, prefix);
    }
    res.prefix_total = std::accumulate(prefix.begin(), prefix.end(), (uint64_t)0);
    idn_batch b{};
    b.n_reads = n_reads;
    b.n_symbols = bt.read_off[n_reads];
    b.n_blocks = n_blocks;
    b.acids = bt.acids.data();
    b.quals = bt.quals.data();
    b.read_off = bt.read_off.data();
    b.block_first_read = bt.block_first.data();
    if (params_.include_identifiers) {
        b.names = bt.names.empty() ? reinterpret_cast<const uint8_t*>("") : bt.names.data();
        b.name_off = bt.name_off.data();
    }
    // capacity: what containers need in practice (1.25 B per symbol is beyond uniformly random input) and, should a batch
    // ever need more, the library's worst-case bound
    const uint64_t bound = idn_gpu_compress_bound(n_reads, b.n_symbols, n_blocks, res.prefix_total);
    uint64_t cap = std::min<uint64_t>(bound, b.n_symbols + b.n_symbols / 4 + 24 * n_reads + 64ull * n_blocks + res.prefix_total + 4096);
    std::vector<uint64_t> block_off(n_blocks + 1);
    idn_compress_stats st{};
    Span sp_c(T_CBLOCKS);
    for (;;) {
        res.buf = pool_.get(cap);
        int32_t rc = idn_gpu_compress_blocks(w.dev.ctx(), &b, params_.mode, w.dev.handles().data(), (uint32_t)w.dev.handles().size(),
                                             params_.fast ? 1 : 0, params_.include_identifiers ? prefix.data() : nullptr, res.buf->p,
                                             cap, block_off.data(), nullptr, &st);
        if (rc == IDN_E_NOSPACE && cap < bound) {
            cap = bound;
            continue;
        }
        if (rc) w.dev.raise(rc);
        break;
    }
    for (uint32_t k = 0; k < n_blocks; k++)
        if (prefix[k]) std::memcpy(res.buf->p + block_off[k] + 8, dev_slices ? dev_slices->p + slice_off[k] : name_slices[k].data(), prefix[k]);
    res.out_bytes = st.out_bytes;
    res.payload_bytes = st.payload_bytes;
    res.acid_switches = st.acid_switches;
    res.q_switches = st.q_switches;
    res.blocks = n_blocks;
    return res;
}

void IdnCompressor::flush_batch() {
    const uint32_t n_blocks = (uint32_t)(cur_.block_first.size() - 1);
    if (n_blocks == 0) return;
    if (!initialized_) initialize();
    // the batch goes to the next device; up to two batches per device are in flight, results are written in block order
    Worker* w = workers_[next_worker_++ % workers_.size()].get();
    auto job = std::make_shared<Batch>(std::move(cur_));
    cur_ = Batch();
    submit(std::async(std::launch::async, [this, w, job] { return compress_batch(*w, *job); }));
    commit(false);
}

void IdnCompressor::submit(std::future<Result> f) {
    {
        std::lock_guard<std::mutex> lk(wmu_);
        pending_.push_back(std::move(f));
        if (!writer_.joinable()) writer_ = std::thread([this] { writer_loop(); });
    }
    wcv_.notify_all();
}

// the writer thread: results in block order to the sink.  After an error it keeps taking results off the queue (without
// writing them), so that nobody waits for ever and every job has finished before the object goes away.
void IdnCompressor::writer_loop() {
    std::unique_lock<std::mutex> lk(wmu_);
    for (;;) {
        wcv_.wait(lk, [this] { return writer_stop_ || !pending_.empty(); });
        if (pending_.empty()) break;  // (stop requested and nothing left)
        std::future<Result> f = std::move(pending_.front());  // the entry stays in the queue until it is written: commit() counts it
        const bool failed = writer_err_ != nullptr;
        lk.unlock();
        std::exception_ptr err;
        Result r;
        try {
            {
                Span spw(T_WAIT);
                r = f.get();  // rethrows what the job threw
            }
            if (!failed) {
                Span sp(T_SINK);
                sink_(r.buf->p, r.out_bytes);
            }
        } catch (...) {
            err = std::current_exception();
        }
        lk.lock();
        if (err && !writer_err_) writer_err_ = err;
        if (!err && !failed) {
            stats_.out_bytes += r.out_bytes;
            stats_.out_identifier_bytes += r.prefix_total;
            stats_.out_payload_bytes += r.payload_bytes;
            stats_.acid_model_switches += r.acid_switches;
            stats_.q_score_model_switches += r.q_switches;
            stats_.blocks += r.blocks;
        }
        r = Result();  // the page-locked buffer goes back to the pool before the next wait
        pending_.pop_front();
        wcv_.notify_all();
    }
}

// waits until at most two batches per device are pending (all = false) or everything is written (all = true); rethrows
// what a job or the sink threw
void IdnCompressor::commit(bool all) {
    const size_t keep = all ? 0 : 2 * workers_.size();
    std::unique_lock<std::mutex> lk(wmu_);
    {
        Span spw(T_WAIT);
        wcv_.wait(lk, [&] { return pending_.size() <= keep; });
    }
    if (writer_err_) {
        std::exception_ptr e = writer_err_;
        if (all) writer_err_ = nullptr;  // reported once by finish(); an add_* after an error keeps failing
        std::rethrow_exception(e);
    }
}

// ---- FASTQ text in (row f1 wired into the API) -------------------------------------------------------------------------
void IdnCompressor::add_fastq_text(const uint8_t* text, size_t n) {
    if (finished_) throw IdnError(IDN_E_INVALID_STATE, "add_fastq_text after finish");
    if (!text_mode_ && (cur_.read_off.size() > 1 || initialized_)) throw IdnError(IDN_E_INVALID_STATE, "add_fastq_text after add_sequence");
    text_mode_ = true;
    // The caller's buffer is read in place (no copy of the bulk of the text); only what a call leaves unconsumed -- a cut
    // record and the reads of the last, possibly unfinished block: at most a block's worth of text -- is kept in text_
    // and put in front of the next call's text.
    size_t pos = 0;
    while (!text_.empty() && pos < n) {
        // carry-over from the call before: complete it with the head of the new text up to one chunk and process that
        const size_t take = (size_t)std::min<uint64_t>(n - pos, std::max<uint64_t>(params_.text_chunk_bytes, text_.size()) );
        const size_t carried = text_.size();
        text_.insert(text_.end(), text + pos, text + pos + take);
        pos += take;
        const size_t used = consume_text(text_.data(), text_.size(), false);
        const size_t tail = text_.size() - used;
        if (used > 0 && tail <= take) {  // the unconsumed tail lies inside the caller's buffer: go on from there
            pos -= tail;
            text_.clear();
        } else {
            text_.erase(text_.begin(), text_.begin() + used);
            if (used == 0 && text_.size() == carried + take && pos == n) break;  // not one block yet: wait for more text
        }
    }
    if (text_.empty()) {
        while (n - pos >= params_.text_chunk_bytes) {
            const size_t used = consume_text(text + pos, n - pos, false);
            if (used == 0) break;
            pos += used;
        }
        text_.assign(text + pos, text + n);
    }
}

static const char* fastq_error_name(int32_t kind) {
    switch (kind) {
        case 1: return "InvalidFormat";
        case 2: return "InvalidAcid";
        case 3: return "InvalidQualityScore";
        case 4: return "AcidAndQualityScoreLengthMismatch";
        case 5: return "EofReached";
        default: return "";
    }
}

// processes as many chunks of [buf, buf + total) as hold complete blocks (everything when final); returns the bytes consumed
size_t IdnCompressor::consume_text(const uint8_t* buf, size_t total, bool final) {
    uint64_t chunk = params_.text_chunk_bytes;
    size_t text_pos_ = 0;
    for (;;) {
        const size_t avail = total - text_pos_;
        if (avail == 0 && !(final && !initialized_)) break;
        size_t len = (size_t)std::min<uint64_t>(avail, chunk);
        const bool last = final && len == avail;
        if (!last) {  // a chunk of a longer input ends on a line boundary
            while (len > 0 && buf[text_pos_ + len - 1] != '\n') len--;
            if (len == 0) {
                if (chunk >= avail && !final) break;  // not even one line yet: wait for more text
                chunk *= 2;
                continue;
            }
        }
        Worker* w = workers_[next_worker_++ % workers_.size()].get();
        {
            Span sp(T_WAIT);
            w->acquire();  // released by the job below
        }
        idn_fastq_chunk ck{};
        Span sp_parse(T_PARSE);
        int32_t rc = idn_gpu_fastq_parse_chunk(w->dev.ctx(), buf + text_pos_, len, last ? 1 : 0, params_.max_block_total_len, &ck);
        if (rc) {
            std::string what = idn_gpu_last_error(w->dev.ctx());
            if (ck.error_kind) what = std::string("FastqReaderError::") + fastq_error_name(ck.error_kind) + ": " + what;
            if (rc == IDN_E_CUDA) w->dev.mark_broken();
            w->release();
            throw IdnError(rc, what);
        }
        if (ck.n_blocks == 0) {  // not one complete block in this chunk
            w->release();
            if (last) {
                text_pos_ += len;
                break;
            }
            if (chunk > avail) break;  // wait for more text
            chunk *= 2;
            continue;
        }
        if (!initialized_) {
            Span sp_sel(T_SELECT);
            // file-level model selection on the reads of the first block (compressor_initializer.rs:53-74): they are on the
            // device; bring them back once and go through the same initialize() as the add_sequence path
            ModelProvider& mp = params_.model_provider;
            size_t n_a = 0, n_q = 0;
            for (size_t i = 0; i < mp.len(); i++) (mp[i].model_type() == ModelType::Acids ? n_a : n_q)++;
            if (n_a > 1 || n_q > 1) {
                std::vector<uint32_t> bf(ck.n_blocks + 1);
                Batch first;
                first.read_off.assign(ck.n_reads + 1, 0);
                first.acids.resize(ck.n_symbols + 1);
                first.quals.resize(ck.n_symbols + 1);
                rc = idn_gpu_fastq_chunk_fetch(w->dev.ctx(), nullptr, nullptr, bf.data(), first.read_off.data(), first.acids.data(), first.quals.data());
                if (rc) {
                    w->release();
                    w->dev.raise(rc);
                }
                first.block_first = {0, bf[1]};
                std::swap(cur_, first);
                try {
                    initialize();
                } catch (...) {
                    w->release();
                    throw;
                }
                std::swap(cur_, first);
            } else {
                try {
                    initialize();
                } catch (...) {
                    w->release();
                    throw;
                }
            }
        }
        text_pos_ += ck.consumed_text;
        stats_.in_symbols += ck.n_symbols;
        stats_.in_reads += ck.n_reads;
        stats_.in_identifier_bytes += ck.n_name_bytes;
        const uint32_t nb = ck.n_blocks;
        const uint64_t nr = ck.n_reads, ns = ck.n_symbols, nn = ck.n_name_bytes;
        submit(std::async(std::launch::async, [this, w, nb, nr, ns, nn] { return compress_parsed(*w, nb, nr, ns, nn); }));
        commit(false);
        if (last) break;
    }
    return text_pos_;
}

// second half of a text chunk (the worker is already leased): identifiers to the host and through Deflate, the block
// kernels on the parsed symbols where they lie, container bytes back
IdnCompressor::Result IdnCompressor::compress_parsed(Worker& w, uint32_t n_blocks, uint64_t n_reads, uint64_t n_symbols,
                                                     uint64_t n_name_bytes) const {
    WorkerLease<Worker> lease(w, true);
    Result res;
    if (params_.include_identifiers && params_.identifiers_on_device) return compress_parsed_ids(w, n_blocks, n_reads, n_symbols, n_name_bytes);
    std::vector<std::vector<uint8_t>> name_slices(n_blocks);
    std::vector<uint32_t> prefix(n_blocks, 0);
    if (params_.include_identifiers) {
        auto names = pool_.get(n_name_bytes + 1);
        auto name_off = pool_.get((n_reads + 1) * 8);
        uint64_t* no = reinterpret_cast<uint64_t*>(name_off->p);
        std::vector<uint32_t> block_first(n_blocks + 1);
        {
            Span sp(T_NFETCH);
            int32_t rc = idn_gpu_fastq_chunk_fetch(w.dev.ctx(), names->p, no, block_first.data(), nullptr, nullptr, nullptr);
            if (rc) w.dev.raise(rc);
        }
        Span sp(T_NDEFLATE);
        identifier_slices(params_.quality, params_.thread_num, n_blocks, block_first.data(), names->p, no, name_slices, prefix);
    }
    res.prefix_total = std::accumulate(prefix.begin(), prefix.end(), (uint64_t)0);
    const uint64_t bound = idn_gpu_compress_bound(n_reads, n_symbols, n_blocks, res.prefix_total);
    uint64_t cap = std::min<uint64_t>(bound, n_symbols + n_symbols / 4 + 24 * n_reads + 64ull * n_blocks + res.prefix_total + 4096);
    std::vector<uint64_t> block_off(n_blocks + 1);
    idn_compress_stats st{};
    Span sp_c(T_CPARSED);
    for (;;) {
        res.buf = pool_.get(cap);
        int32_t rc = idn_gpu_compress_parsed(w.dev.ctx(), params_.mode, w.dev.handles().data(), (uint32_t)w.dev.handles().size(), params_.fast ? 1 : 0,
                                             params_.include_identifiers ? 1 : 0, params_.include_identifiers ? prefix.data() : nullptr,
                                             res.buf->p, cap, block_off.data(), nullptr, &st);
        if (rc == IDN_E_NOSPACE && cap < bound) {
            cap = bound;
            continue;
        }
        if (rc) w.dev.raise(rc);
        break;
    }
    for (uint32_t k = 0; k < n_blocks; k++)
        if (prefix[k]) std::memcpy(res.buf->p + block_off[k] + 8, name_slices[k].data(), prefix[k]);
    res.out_bytes = st.out_bytes;
    res.payload_bytes = st.payload_bytes;
    res.acid_switches = st.acid_switches;
    res.q_switches = st.q_switches;
    res.blocks = n_blocks;
    return res;
}

// compress_parsed with identifiers_on_device: the library Deflates the names where the parse left them and puts the slices
// into the container; the slice lengths are read back from their headers for the statistics
IdnCompressor::Result IdnCompressor::compress_parsed_ids(Worker& w, uint32_t n_blocks, uint64_t n_reads, uint64_t n_symbols,
                                                         uint64_t n_name_bytes) const {
    Result res;
    const uint64_t ids_bound = idn_gpu_deflate_names_bound(n_name_bytes, n_reads, n_blocks);
    const uint64_t bound = idn_gpu_compress_bound(n_reads, n_symbols, n_blocks, ids_bound);
    uint64_t cap = std::min<uint64_t>(bound, n_symbols + n_symbols / 4 + 24 * n_reads + 64ull * n_blocks + n_name_bytes / 2 + 4096);
    std::vector<uint64_t> block_off(n_blocks + 1);
    idn_compress_stats st{};
    Span sp_c(T_CPARSED);
    for (;;) {
        res.buf = pool_.get(cap);
        int32_t rc = idn_gpu_compress_parsed_ids(w.dev.ctx(), params_.mode, w.dev.handles().data(), (uint32_t)w.dev.handles().size(),
                                                 params_.fast ? 1 : 0, res.buf->p, cap, block_off.data(), nullptr, &st);
        if (rc == IDN_E_NOSPACE && cap < bound) {
            cap = bound;
            continue;
        }
        if (rc) w.dev.raise(rc);
        break;
    }
    for (uint32_t k = 0; k < n_blocks; k++) {  // 0x00 | u32be n | 0x01 | n bytes
        const uint8_t* h = res.buf->p + block_off[k] + 9;
        res.prefix_total += 6 + ((uint64_t)h[0] << 24 | (uint64_t)h[1] << 16 | (uint64_t)h[2] << 8 | h[3]);
    }
    res.out_bytes = st.out_bytes;
    res.payload_bytes = st.payload_bytes;
    res.acid_switches = st.acid_switches;
    res.q_switches = st.q_switches;
    res.blocks = n_blocks;
    return res;
}

void IdnCompressor::finish() {
    if (finished_) throw IdnError(IDN_E_INVALID_STATE, "finish called twice");
    if (text_mode_) {
        consume_text(text_.data(), text_.size(), true);
        text_.clear();
    }
    make_block();  // flush the partial block (idn/compressor.rs:575-578)
    flush_batch();
    if (!initialized_) initialize();  // empty file: header + metadata still get written
    commit(true);
    const uint8_t terminator[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // an empty block marks the end (:579)
    sink_(terminator, 8);
    stats_.out_bytes += 8;
    finished_ = true;
    g_trace.print("compressor");
}

// ---- IdnDecompressor -------------------------------------------------------------------------------------------------
IdnDecompressor::IdnDecompressor(Source source, IdnDecompressorParams params) : source_(std::move(source)), params_(std::move(params)) {
    Span sp(T_OPEN);
    if (params_.devices.empty()) params_.devices.assign(1, 0);
    if (params_.batch_blocks == 0) params_.batch_blocks = 1;
    for (int32_t d : params_.devices) {
        workers_.push_back(std::make_unique<Worker>());
        workers_.back()->dev.open(d);
    }
}
IdnDecompressor::IdnDecompressor(const uint8_t* data, size_t len, IdnDecompressorParams params)
    : IdnDecompressor(Source([this](uint8_t* dst, size_t n) {
                          const size_t k = std::min(n, mem_len_ - mem_pos_);
                          std::memcpy(dst, mem_ + mem_pos_, k);
                          mem_pos_ += k;
                          return k;
                      }),
                      std::move(params)) {
    mem_ = data;
    mem_len_ = len;
}
IdnDecompressor::~IdnDecompressor() {
    {
        Span sp(T_CLOSE);
        for (auto& f : pending_)
            if (f.valid()) f.wait();
        pending_.clear();
        workers_.clear();  // contexts back to the cache
    }
    g_trace.print("decompressor");
}

void IdnDecompressor::read_exact(uint8_t* dst, size_t n, const char* what) {
    size_t got = 0;
    while (got < n) {
        size_t k = source_(dst + got, n - got);
        if (k == 0) throw IdnError(IDN_E_IO, std::string("unexpected end of input while reading ") + what);
        got += k;
    }
}

void IdnDecompressor::initialize() {
    Span sp(T_INIT);
    uint8_t h[9];
    read_exact(h, 9, "the header");
    if (std::memcmp(h, kMagic, 8) != 0) throw IdnError(IDN_E_SERIALIZE, "not an IDN file (bad magic)");
    version_ = h[8];
    if (version_ != 1 && version_ != 2)  // idn/decompressor.rs:317-319 (version 2 = this implementation's native format)
        throw IdnError(IDN_E_INVALID_VERSION, "unsupported IDN version " + std::to_string(version_));
    uint8_t item_num;
    read_exact(&item_num, 1, "the metadata");
    std::vector<ModelIdentifier> ids;
    for (uint8_t i = 0; i < item_num; i++) {
        uint8_t kind;
        read_exact(&kind, 1, "a metadata item");
        if (kind != 0) throw IdnError(IDN_E_SERIALIZE, "unknown metadata item");
        uint8_t n;
        read_exact(&n, 1, "the model list");
        for (uint8_t k = 0; k < n; k++) {
            ModelIdentifier id;
            read_exact(id.data(), 32, "a model identifier");
            ids.push_back(id);
        }
    }
    if (!params_.model_provider.has_all_models(ids)) {  // IdnDecompressorError::UnknownModel (idn/decompressor.rs:340-350)
        for (auto& id : ids)
            if (!params_.model_provider.has_all_models({id})) throw IdnError(IDN_E_UNKNOWN_MODEL, "unknown model " + to_hex(id));
    }
    params_.model_provider.filter_by_identifiers(ids);
    for (auto& w : workers_) w->dev.upload(params_.model_provider);
    initialized_ = true;
}

bool IdnDecompressor::read_raw(RawBatch& rb) {
    // block headers + payloads of up to batch_blocks blocks into one buffer (idn/decompressor.rs:387-428)
    Span sp(T_READRAW);
    bool more = true;
    rb.used = 0;
    if (mem_) {  // the payloads stay where they are: offsets from the first one, headers in between
        size_t first = 0;
        while (rb.off.size() < params_.batch_blocks) {
            uint8_t h[8];
            read_exact(h, 8, "a block header");
            uint32_t n = get_u32be(h), c = get_u32be(h + 4);
            if (n == 0) {
                more = false;
                break;
            }
            if (n > mem_len_ - mem_pos_) throw IdnError(IDN_E_IO, "unexpected end of input while reading a block");
            if (rb.off.empty()) first = mem_pos_;
            rb.off.push_back(mem_pos_ - first);
            rb.len.push_back(n);
            rb.crc.push_back(c);
            mem_pos_ += n;
            rb.used = mem_pos_ - first;
        }
        rb.base = mem_ + first;
        return more;
    }
    rb.buf = pool_.get(g_raw_hint.load());
    while (rb.off.size() < params_.batch_blocks) {
        uint8_t h[8];
        read_exact(h, 8, "a block header");
        uint32_t n = get_u32be(h), c = get_u32be(h + 4);
        if (n == 0) {  // terminator (:422-425)
            more = false;
            break;
        }
        rb.off.push_back(rb.used);
        rb.len.push_back(n);
        rb.crc.push_back(c);
        rb.buf->ensure_keep(rb.used + n, rb.used);
        read_exact(rb.buf->p + rb.used, n, "a block");
        rb.used += n;
    }
    for (size_t h = g_raw_hint.load(); h < rb.used && !g_raw_hint.compare_exchange_weak(h, rb.used);) {}
    rb.base = rb.buf->p;
    return more;
}

// identifiers: leading Identifiers slices of every block, inflated on the host (decompressor_block.rs:146-192)
void IdnDecompressor::inflate_names(const RawBatch& rb, const std::vector<uint64_t>& off, const std::vector<uint32_t>& block_first,
                                    uint64_t n_reads, DecodedBatch& out) const {
    const uint32_t n_blocks = (uint32_t)rb.off.size();
    out.name_off.assign(n_reads + 1, 0);
    // blocks inflate independently: thread_num host threads take them in turn, the pieces are stitched in block order
    std::vector<std::vector<uint8_t>> text(n_blocks);
    std::vector<uint8_t> has(n_blocks, 0);
    auto one = [&](uint32_t b) {
        const uint8_t* p = rb.base + off[b];
        size_t pos = 0;
        while (pos < rb.len[b] && p[pos] == 0x00) {
            if (pos + 6 > rb.len[b]) throw IdnError(IDN_E_SERIALIZE, "truncated identifiers slice");
            uint32_t n = get_u32be(p + pos + 1);
            uint8_t comp = p[pos + 5];
            if (n > rb.len[b] - pos - 6) throw IdnError(IDN_E_SERIALIZE, "truncated identifiers slice");
            if (comp > 1) throw IdnError(IDN_E_SERIALIZE, "unknown identifier compression");
            std::vector<uint8_t> t = comp == 0 ? Brotli::get().decompress(p + pos + 6, n) : inflate_raw(p + pos + 6, n);
            if (has[b]) text[b].push_back('\n');
            text[b].insert(text[b].end(), t.begin(), t.end());
            has[b] = 1;
            pos += 6 + (size_t)n;
        }
    };
    // one identifier per sequence, in order (identifiers_as_lines): split at '\n' inside the block's job -- the line lengths
    // of the block's reads and the text without its separators -- so that only a prefix sum over blocks stays serial
    std::vector<std::vector<uint32_t>> lens(n_blocks);
    auto split = [&](uint32_t b) {
        one(b);
        if (!has[b]) return;
        std::vector<uint8_t>& t = text[b];
        const uint64_t want = block_first[b + 1] - block_first[b];
        lens[b].reserve(want);
        size_t s0 = 0, w = 0;
        while (lens[b].size() < want) {
            const uint8_t* nl = static_cast<const uint8_t*>(std::memchr(t.data() + s0, '\n', t.size() - s0));
            const size_t e = nl ? (size_t)(nl - t.data()) : t.size();
            if (w != s0) std::memmove(t.data() + w, t.data() + s0, e - s0);
            w += e - s0;
            lens[b].push_back((uint32_t)(e - s0));
            if (!nl) break;
            s0 = e + 1;
        }
        t.resize(w);
    };
    auto for_blocks = [&](auto&& fn) {
        if (params_.thread_num > 1 && n_blocks > 1) {
            std::vector<std::future<void>> jobs;
            std::atomic<uint32_t> next{0};
            for (uint32_t t = 0; t < std::min<uint32_t>(params_.thread_num, n_blocks); t++)
                jobs.push_back(std::async(std::launch::async, [&] {
                    for (uint32_t b = next++; b < n_blocks; b = next++) fn(b);
                }));
            std::exception_ptr err;
            for (auto& j : jobs) {
                try {
                    j.get();
                } catch (...) {
                    if (!err) err = std::current_exception();
                }
            }
            if (err) std::rethrow_exception(err);
        } else {
            for (uint32_t b = 0; b < n_blocks; b++) fn(b);
        }
    };
    for_blocks(split);
    std::vector<uint64_t> base(n_blocks + 1, 0);
    for (uint32_t b = 0; b < n_blocks; b++) {
        base[b + 1] = base[b] + text[b].size();
        out.any_names = out.any_names || has[b];
    }
    out.names.resize(base[n_blocks]);
    for_blocks([&](uint32_t b) {
        if (!text[b].empty()) std::memcpy(out.names.data() + base[b], text[b].data(), text[b].size());
        uint64_t at = base[b], r = block_first[b];
        for (uint32_t n : lens[b]) out.name_off[++r] = (at += n);
        for (; r < block_first[b + 1]; r++) out.name_off[r + 1] = at;  // sequences without an identifier
    });
}

// identifiers_on_device: the batch's Identifiers slices inflated on the device, from the container bytes idn_gpu_index_blocks
// left there; the names stay on the device for the _ids decode calls (and come back when `fetch`).  A Brotli slice makes
// the library decline (IDN_E_UNSUPPORTED): false, and the batch takes the host's inflate_names.
bool IdnDecompressor::inflate_names_device(Worker& w, const RawBatch& rb, const std::vector<uint64_t>& off,
                                           const std::vector<uint32_t>& block_first, uint64_t n_reads, DecodedBatch& out, bool fetch,
                                           uint64_t* n_name_bytes) const {
    Span sp(T_NINFLATE_DEV);
    const uint32_t n_blocks = (uint32_t)rb.off.size();
    uint64_t n_bytes = 0;
    int32_t bad = -1;
    idn_inflate_stats st{};
    int32_t rc = idn_gpu_inflate_names(w.dev.ctx(), nullptr, off.data(), rb.len.data(), n_blocks, block_first.data(), n_reads, &n_bytes, &bad, &st);
    if (rc == IDN_E_UNSUPPORTED) return false;
    if (rc) w.dev.raise(rc);
    out.any_names = st.n_streams > 0;
    *n_name_bytes = n_bytes;
    if (fetch) {
        out.names.resize(n_bytes);
        out.name_off.assign(n_reads + 1, 0);
        rc = idn_gpu_inflate_names_fetch(w.dev.ctx(), out.names.data(), out.name_off.data());
        if (rc) w.dev.raise(rc);
    }
    return true;
}

IdnDecompressor::DecodedBatch IdnDecompressor::decode_batch(Worker& w, const RawBatch& rb) const {
    std::lock_guard<std::mutex> lock(w.mu);
    DecodedBatch out;
    const uint32_t n_blocks = (uint32_t)rb.off.size();
    if (n_blocks == 0) return out;
    std::vector<uint64_t> off = rb.off;
    off.push_back(rb.used);
    const int32_t mode = version_ == 2 ? IDN_MODE_NATIVE : IDN_MODE_COMPAT;
    const auto& handles = w.dev.handles();
    idn_block_index_totals tot{};
    std::vector<uint32_t> block_first(n_blocks + 1);
    int32_t rc;
    {
        Span sp(T_INDEX);
        rc = idn_gpu_index_blocks(w.dev.ctx(), rb.base, off.data(), rb.len.data(), n_blocks, mode, handles.data(), (uint32_t)handles.size(), &tot,
                                  block_first.data());
    }
    if (rc) w.dev.raise(rc);
    // next_batch / next_sequence hand the names out: the device's come back to the host
    uint64_t dev_name_bytes = 0;
    const bool on_dev = params_.identifiers_on_device && inflate_names_device(w, rb, off, block_first, tot.n_reads, out, true, &dev_name_bytes);
    if (!on_dev) {
        Span sp(T_NINFLATE);
        inflate_names(rb, off, block_first, tot.n_reads, out);
    }
    Span sp_d(T_DECODE);
    out.acids.resize(tot.n_symbols + 1);
    out.quals.resize(tot.n_symbols + 1);
    out.read_off.assign(tot.n_reads + 1, 0);
    int32_t bad = -1;
    if (out.names.empty()) out.names.push_back(0);
    if (on_dev) {
        // the block CRCs read the names where the inflate left them
        rc = idn_gpu_decompress_blocks_ids(w.dev.ctx(), nullptr, off.data(), rb.len.data(), rb.crc.data(), n_blocks, mode, handles.data(),
                                           (uint32_t)handles.size(), out.acids.data(), out.quals.data(), out.read_off.data(), tot.n_reads,
                                           tot.n_symbols, &bad);
    } else {
        // with identifiers the call is not pipelined and can use the bytes idn_gpu_index_blocks left on the device (blocks == NULL)
        rc = idn_gpu_decompress_blocks(w.dev.ctx(), out.any_names ? nullptr : rb.base, off.data(), rb.len.data(), rb.crc.data(), n_blocks, mode,
                                       handles.data(), (uint32_t)handles.size(), out.any_names ? out.names.data() : nullptr,
                                       out.any_names ? out.name_off.data() : nullptr, out.acids.data(), out.quals.data(), out.read_off.data(),
                                       tot.n_reads, tot.n_symbols, &bad);
    }
    if (rc) w.dev.raise(rc);
    out.acids.resize(tot.n_symbols);
    out.quals.resize(tot.n_symbols);
    if (!out.any_names) out.names.clear();
    return out;
}

// the same with the FASTQ text formatted on the device: the symbols never cross PCIe
IdnDecompressor::DecodedBatch IdnDecompressor::decode_text(Worker& w, const RawBatch& rb, bool title_with_separator) const {
    std::lock_guard<std::mutex> lock(w.mu);
    DecodedBatch out;
    const uint32_t n_blocks = (uint32_t)rb.off.size();
    if (n_blocks == 0) return out;
    std::vector<uint64_t> off = rb.off;
    off.push_back(rb.used);
    const int32_t mode = version_ == 2 ? IDN_MODE_NATIVE : IDN_MODE_COMPAT;
    const auto& handles = w.dev.handles();
    idn_block_index_totals tot{};
    std::vector<uint32_t> block_first(n_blocks + 1);
    int32_t rc;
    {
        Span sp(T_INDEX);
        rc = idn_gpu_index_blocks(w.dev.ctx(), rb.base, off.data(), rb.len.data(), n_blocks, mode, handles.data(), (uint32_t)handles.size(), &tot,
                                  block_first.data());
    }
    if (rc) w.dev.raise(rc);
    // the names of the device path never leave it
    uint64_t dev_name_bytes = 0;
    const bool on_dev = params_.identifiers_on_device && inflate_names_device(w, rb, off, block_first, tot.n_reads, out, false, &dev_name_bytes);
    if (!on_dev) {
        Span sp(T_NINFLATE);
        inflate_names(rb, off, block_first, tot.n_reads, out);
    }
    Span sp_d(T_DECODE);
    if (out.names.empty()) out.names.push_back(0);
    const uint64_t name_bytes = on_dev ? dev_name_bytes : out.any_names ? out.name_off[tot.n_reads] : 0;
    const uint64_t cap = 2 * tot.n_symbols + 6 * tot.n_reads + name_bytes * (title_with_separator ? 2 : 1) + 64;
    uint64_t text_len = 0, n_reads = 0;
    int32_t bad = -1;
    if (on_dev) {
        out.text = pool_.get(cap);
        rc = idn_gpu_decompress_to_fastq_ids(w.dev.ctx(), nullptr, off.data(), rb.len.data(), rb.crc.data(), n_blocks, mode, handles.data(),
                                             (uint32_t)handles.size(), tot.n_reads, tot.n_symbols, title_with_separator ? 1 : 0, out.text->p, cap,
                                             &text_len, &n_reads, &bad);
    } else {
        out.text = pool_.get(cap);
        // blocks == NULL: the bytes idn_gpu_index_blocks just uploaded are still on the device
        rc = idn_gpu_decompress_to_fastq(w.dev.ctx(), nullptr, off.data(), rb.len.data(), rb.crc.data(), n_blocks, mode, handles.data(),
                                         (uint32_t)handles.size(), out.any_names ? out.names.data() : nullptr,
                                         out.any_names ? out.name_off.data() : nullptr, tot.n_reads, tot.n_symbols, title_with_separator ? 1 : 0,
                                         out.text->p, cap, &text_len, &n_reads, &bad);
    }
    if (rc) w.dev.raise(rc);
    out.text_len = text_len;
    out.read_off.assign(1, n_reads);  // [0] = sequences in the text
    return out;
}

bool IdnDecompressor::next_fastq_text(std::shared_ptr<PinnedBuf>& out, size_t& len, bool title_with_separator) {
    if (!initialized_) initialize();
    text_mode_ = title_with_separator ? 2 : 1;
    prefetch();
    if (pending_.empty()) return false;
    DecodedBatch b;
    {
        Span sp(T_WAITRES);
        b = pending_.front().get();
    }
    pending_.pop_front();
    prefetch();
    out = std::move(b.text);
    len = b.text_len;
    return true;
}

// keeps up to two batches per device in flight (the reference reads and dispatches block jobs ahead the same way,
// idn/decompressor.rs:387-428)
void IdnDecompressor::prefetch() {
    while (!eof_ && pending_.size() < 2 * workers_.size()) {
        auto rb = std::make_shared<RawBatch>();
        eof_ = !read_raw(*rb);
        if (rb->off.empty()) break;
        Worker* w = workers_[next_worker_++ % workers_.size()].get();
        const int tm = text_mode_;
        pending_.push_back(std::async(std::launch::async, [this, w, rb, tm] { return tm ? decode_text(*w, *rb, tm == 2) : decode_batch(*w, *rb); }));
    }
}

bool IdnDecompressor::next_batch(DecodedBatch& out) {
    if (!initialized_) initialize();
    prefetch();
    if (pending_.empty()) return false;
    out = pending_.front().get();
    pending_.pop_front();
    prefetch();
    return true;
}

std::optional<FastqSequence> IdnDecompressor::next_sequence() {
    while (queue_.empty()) {
        DecodedBatch b;
        if (!next_batch(b)) return std::nullopt;
        const uint64_t n = b.read_off.size() - 1;
        for (uint64_t r = 0; r < n; r++) {
            FastqSequence s;
            if (b.any_names) s.identifier.assign(b.names.begin() + b.name_off[r], b.names.begin() + b.name_off[r + 1]);
            s.acids.assign(b.acids.begin() + b.read_off[r], b.acids.begin() + b.read_off[r + 1]);
            s.quality_scores.assign(b.quals.begin() + b.read_off[r], b.quals.begin() + b.read_off[r + 1]);
            queue_.push_back(std::move(s));
        }
    }
    FastqSequence s = std::move(queue_.front());
    queue_.pop_front();
    return s;
}

}  // namespace idencomp
