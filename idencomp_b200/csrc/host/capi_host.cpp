// capi_host.cpp -- flat C view (include/idn_host.h) of the C++ host mirror.
#include "../../../include/idn_host.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>

#include "clustering.hpp"
#include "idn.hpp"
#include "model.hpp"

using namespace idencomp;

struct idn_host_model {
    std::shared_ptr<const Model> m;
};

namespace {
thread_local std::string g_err;

int32_t set_err(int32_t code, const std::string& what) {
    g_err = what;
    return code;
}

template <class F>
int32_t guarded(F&& f) {
    try {
        return f();
    } catch (const IdnError& e) {
        return set_err(e.code, e.what());
    } catch (const ModelError& e) {
        return set_err(IDN_E_SERIALIZE, e.what());
    } catch (const std::exception& e) {
        return set_err(IDN_E_INVALID_STATE, e.what());
    }
}
}  // namespace

extern "C" const char* idn_host_last_error(void) { return g_err.c_str(); }

extern "C" int32_t idn_host_model_load(const char* path, idn_host_model** out) {
    if (!path || !out) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *out = nullptr;
    return guarded([&] {
        *out = new idn_host_model{std::make_shared<const Model>(Model::read_file(path))};
        return (int32_t)IDN_OK;
    });
}

extern "C" int32_t idn_host_model_from_bytes(const uint8_t* data, size_t n, idn_host_model** out) {
    if (!data || !out) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *out = nullptr;
    return guarded([&] {
        *out = new idn_host_model{std::make_shared<const Model>(Model::read_msgpack(data, n))};
        return (int32_t)IDN_OK;
    });
}

extern "C" int32_t idn_host_model_new(int32_t model_type, const char* spec_name, uint32_t n_ctx, const float* probs,
                                      const uint32_t* spec_keys, const uint32_t* spec_ctx, uint64_t n_specs,
                                      idn_host_model** out) {
    if (!spec_name || !out || (n_ctx && !probs) || (n_specs && (!spec_keys || !spec_ctx)))
        return set_err(IDN_E_INVALID_ARG, "NULL argument");
    if (model_type != IDN_MODEL_ACID && model_type != IDN_MODEL_QSCORE) return set_err(IDN_E_INVALID_ARG, "bad model type");
    *out = nullptr;
    return guarded([&] {
        ModelType t = (ModelType)model_type;
        size_t nsym = symbols_of(t);
        std::vector<ModelContext> ctxs(n_ctx);
        for (uint32_t i = 0; i < n_ctx; i++) ctxs[i].symbol_prob.assign(probs + i * nsym, probs + (i + 1) * nsym);
        for (uint64_t i = 0; i < n_specs; i++) {
            if (spec_ctx[i] >= n_ctx) throw ModelError("context index out of range");
            ctxs[spec_ctx[i]].specs.push_back(spec_keys[i]);
        }
        *out = new idn_host_model{std::make_shared<const Model>(Model(t, ContextSpecType::parse(spec_name), std::move(ctxs)))};
        return (int32_t)IDN_OK;
    });
}

extern "C" int32_t idn_host_model_empty(int32_t model_type, idn_host_model** out) {
    if (!out) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    return guarded([&] {
        *out = new idn_host_model{std::make_shared<const Model>(Model::empty((ModelType)model_type))};
        return (int32_t)IDN_OK;
    });
}

extern "C" void idn_host_model_free(idn_host_model* m) { delete m; }
extern "C" int32_t idn_host_model_type(const idn_host_model* m) { return (int32_t)m->m->model_type(); }
extern "C" uint32_t idn_host_model_len(const idn_host_model* m) { return (uint32_t)m->m->len(); }
extern "C" const char* idn_host_model_spec_name(const idn_host_model* m) { return m->m->context_spec_type().name.c_str(); }
extern "C" void idn_host_model_identifier(const idn_host_model* m, uint8_t out[32]) {
    std::memcpy(out, m->m->identifier().data(), 32);
}

extern "C" uint64_t idn_host_model_cum_table(const idn_host_model* m, uint16_t* out, uint64_t cap) {
    uint64_t need = (uint64_t)(m->m->len() + 1) * (symbols_of(m->m->model_type()) + 1);
    if (!out || cap < need) return need;
    std::vector<uint16_t> t = m->m->cum_table();
    std::memcpy(out, t.data(), t.size() * 2);
    return need;
}

extern "C" int32_t idn_host_model_upload(idn_gpu_ctx* ctx, const idn_host_model* m, idn_model_t* handle) {
    if (!ctx || !m || !handle) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    return guarded([&] {
        int32_t rc = upload_model(ctx, *m->m, handle);
        if (rc) g_err = idn_gpu_last_error(ctx);
        return rc;
    });
}

extern "C" int32_t idn_host_quantise(const float* probs, uint32_t nsym, uint32_t scale_bits, uint32_t* cum_out) {
    if (!probs || !cum_out) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    return guarded([&] {
        std::vector<uint32_t> c = quantise(probs, nsym, scale_bits);
        std::memcpy(cum_out, c.data(), c.size() * 4);
        return (int32_t)IDN_OK;
    });
}

// ---- IdnCompressor / IdnDecompressor ---------------------------------------------------------------------------------

struct idn_host_compressor {
    std::vector<uint8_t> out;
    uint8_t* ext = nullptr;  // idn_host_compressor_set_output: the caller's buffer
    uint64_t ext_cap = 0, ext_len = 0;
    std::unique_ptr<IdnCompressor> c;
};

struct idn_host_decoded {
    uint32_t version = 0;
    std::vector<uint64_t> read_off{0}, name_off{0};
    std::vector<uint8_t> acids, quals, names;
};

static ModelProvider provider_of(const idn_host_model* const* models, uint32_t n) {
    std::vector<std::shared_ptr<const Model>> v;
    for (uint32_t i = 0; i < n; i++) v.push_back(models[i]->m);
    return ModelProvider(std::move(v));
}

extern "C" void idn_host_params_default(idn_host_params* p) {
    IdnCompressorParams d;
    p->max_block_total_len = d.max_block_total_len;
    p->thread_num = d.thread_num;
    p->include_identifiers = d.include_identifiers;
    p->quality = d.quality;
    p->fast = d.fast;
    p->device = d.devices[0];
    p->mode = d.mode;
    p->batch_blocks = d.batch_blocks;
    p->lane_symbols = d.lane_symbols;
    p->text_chunk_bytes = d.text_chunk_bytes;
    p->n_devices = 0;
    for (int32_t& v : p->devices) v = 0;
    p->identifiers_on_device = d.identifiers_on_device;
}

extern "C" int32_t idn_host_compressor_new(const idn_host_model* const* models, uint32_t n_models, const idn_host_params* params,
                                           idn_host_compressor** out) {
    if (!out || !params || (n_models && !models)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *out = nullptr;
    return guarded([&] {
        if (params->quality < 1 || params->quality > 9) throw IdnError(IDN_E_INVALID_ARG, "compression quality must be between 1 and 9");
        IdnCompressorParams p = IdnCompressorParamsBuilder()
                                    .model_provider(provider_of(models, n_models))
                                    .max_block_total_len(params->max_block_total_len)
                                    .thread_num(params->thread_num)
                                    .include_identifiers(params->include_identifiers != 0)
                                    .quality((uint8_t)params->quality)
                                    .fast(params->fast != 0)
                                    .devices(params->n_devices ? std::vector<int32_t>(params->devices, params->devices + std::min<uint32_t>(params->n_devices, 16))
                                                               : std::vector<int32_t>{params->device})
                                    .mode(params->mode)
                                    .batch_blocks(params->batch_blocks)
                                    .lane_symbols(params->lane_symbols)
                                    .text_chunk_bytes(params->text_chunk_bytes ? params->text_chunk_bytes : (256ull << 20))
                                    .identifiers_on_device(params->identifiers_on_device != 0)
                                    .build();
        auto h = std::make_unique<idn_host_compressor>();
        idn_host_compressor* raw = h.get();
        h->c = std::make_unique<IdnCompressor>([raw](const uint8_t* d, size_t n) {
            if (raw->ext) {
                if (raw->ext_len + n > raw->ext_cap) throw IdnError(IDN_E_NOSPACE, "the output buffer is too small");
                std::memcpy(raw->ext + raw->ext_len, d, n);
                raw->ext_len += n;
            } else {
                raw->out.insert(raw->out.end(), d, d + n);
            }
        }, std::move(p));
        *out = h.release();
        return (int32_t)IDN_OK;
    });
}

extern "C" int32_t idn_host_compressor_add(idn_host_compressor* c, const uint8_t* name, uint64_t name_len, const uint8_t* acids,
                                           const uint8_t* quals, uint64_t len) {
    if (!c || (len && (!acids || !quals))) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    return guarded([&] {
        FastqSequence s;
        if (name && name_len) s.identifier.assign(reinterpret_cast<const char*>(name), name_len);
        s.acids.assign(acids, acids + len);
        s.quality_scores.assign(quals, quals + len);
        c->c->add_sequence(std::move(s));
        return (int32_t)IDN_OK;
    });
}

extern "C" int32_t idn_host_compressor_add_batch(idn_host_compressor* c, uint64_t n_reads, const uint64_t* read_off,
                                                 const uint8_t* acids, const uint8_t* quals, const uint64_t* name_off,
                                                 const uint8_t* names) {
    if (!c || (n_reads && !read_off)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    return guarded([&] {
        c->c->add_batch(n_reads, read_off, acids, quals, name_off && names ? name_off : nullptr, name_off && names ? names : nullptr);
        return (int32_t)IDN_OK;
    });
}

extern "C" int32_t idn_host_compressor_add_text(idn_host_compressor* c, const uint8_t* text, uint64_t n) {
    if (!c || (n && !text)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    return guarded([&] {
        if (!c->ext && c->out.capacity() < c->out.size() + n / 3) c->out.reserve(c->out.size() + n / 3 + (1u << 20));  // the in-memory writer
        c->c->add_fastq_text(text, n);
        return (int32_t)IDN_OK;
    });
}

extern "C" int32_t idn_host_decompress_text_ex(const idn_host_model* const* models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                            uint32_t thread_num, int32_t title_with_separator, const uint8_t* idn, uint64_t idn_len,
                                            uint8_t** text, uint64_t* text_len, const idn_host_decompress_params* dparams) {
    if (!text || !text_len || (!idn && idn_len) || (n_models && !models)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *text = nullptr;
    *text_len = 0;
    return guarded([&] {
        IdnDecompressorParams p;
        p.model_provider = provider_of(models, n_models);
        p.identifiers_on_device = dparams && dparams->identifiers_on_device;
        p.thread_num = thread_num;
        if (device >= 0) {
            p.devices.assign(1, device);
        } else {
            p.devices.clear();
            for (int32_t d = 0; d < -device; d++) p.devices.push_back(d);
        }
        p.batch_blocks = batch_blocks ? batch_blocks : 32;
        uint64_t pos = 0;
        IdnDecompressor d([&](uint8_t* dst, size_t n) {
            size_t k = (size_t)std::min<uint64_t>(n, idn_len - pos);
            std::memcpy(dst, idn + pos, k);
            pos += k;
            return k;
        }, std::move(p));
        // pieces are appended to one malloc'd buffer that doubles when it runs out (starts at 3.2 x the container)
        size_t cap = (size_t)(idn_len * 3.2) + (1u << 20), used = 0;
        uint8_t* buf = static_cast<uint8_t*>(std::malloc(cap));
        if (!buf) throw IdnError(IDN_E_IO, "out of memory");
        try {
            std::shared_ptr<PinnedBuf> piece;
            size_t n = 0;
            while (d.next_fastq_text(piece, n, title_with_separator != 0)) {
                if (used + n > cap) {
                    while (used + n > cap) cap *= 2;
                    uint8_t* nb = static_cast<uint8_t*>(std::realloc(buf, cap));
                    if (!nb) throw IdnError(IDN_E_IO, "out of memory");
                    buf = nb;
                }
                std::memcpy(buf + used, piece->p, n);
                used += n;
            }
        } catch (...) {
            std::free(buf);
            throw;
        }
        *text = buf;
        *text_len = used;
        return (int32_t)IDN_OK;
    });
}
extern "C" void idn_host_text_free(uint8_t* text) { std::free(text); }
extern "C" void idn_host_release_cached(void) { release_cached_resources(); }

// the same into the caller's buffer (page-locked and touched, if the caller wants the full rate); IDN_E_NOSPACE with
// *text_len = bytes written so far when it is too small
extern "C" int32_t idn_host_decompress_text_into_ex(const idn_host_model* const* models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                                 uint32_t thread_num, int32_t title_with_separator, const uint8_t* idn, uint64_t idn_len,
                                                 uint8_t* text, uint64_t cap, uint64_t* text_len, const idn_host_decompress_params* dparams) {
    if (!text_len || (!text && cap) || (!idn && idn_len) || (n_models && !models)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *text_len = 0;
    return guarded([&] {
        IdnDecompressorParams p;
        p.model_provider = provider_of(models, n_models);
        p.identifiers_on_device = dparams && dparams->identifiers_on_device;
        p.thread_num = thread_num;
        if (device >= 0) {
            p.devices.assign(1, device);
        } else {
            p.devices.clear();
            for (int32_t d = 0; d < -device; d++) p.devices.push_back(d);
        }
        p.batch_blocks = batch_blocks ? batch_blocks : 32;
        IdnDecompressor d(idn, (size_t)idn_len, std::move(p));
        std::shared_ptr<PinnedBuf> piece;
        size_t n = 0;
        uint64_t used = 0;
        while (d.next_fastq_text(piece, n, title_with_separator != 0)) {
            if (used + n > cap) {
                *text_len = used;
                throw IdnError(IDN_E_NOSPACE, "the text buffer is too small");
            }
            std::memcpy(text + used, piece->p, n);
            used += n;
        }
        *text_len = used;
        return (int32_t)IDN_OK;
    });
}

// streaming form: every call hands out the FASTQ text of the next batch of blocks where the device wrote it (page-locked
// memory of the library, valid until the next call on this reader); a writer passes the pieces to write() as they come
struct idn_host_text_reader {
    std::unique_ptr<IdnDecompressor> d;
    const uint8_t* idn = nullptr;
    uint64_t idn_len = 0, pos = 0;
    std::shared_ptr<PinnedBuf> piece;
    bool sep = false;
};
extern "C" int32_t idn_host_text_reader_new_ex(const idn_host_model* const* models, uint32_t n_models, const int32_t* devices, uint32_t n_devices,
                                            uint32_t batch_blocks, uint32_t thread_num, int32_t title_with_separator, const uint8_t* idn,
                                            uint64_t idn_len, idn_host_text_reader** out, const idn_host_decompress_params* dparams) {
    if (!out || (!idn && idn_len) || (n_models && !models) || (n_devices && !devices)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *out = nullptr;
    return guarded([&] {
        auto r = std::make_unique<idn_host_text_reader>();
        IdnDecompressorParams p;
        p.model_provider = provider_of(models, n_models);
        p.identifiers_on_device = dparams && dparams->identifiers_on_device;
        p.thread_num = thread_num;
        if (n_devices) p.devices.assign(devices, devices + n_devices);
        p.batch_blocks = batch_blocks ? batch_blocks : 32;
        r->idn = idn;
        r->idn_len = idn_len;
        r->sep = title_with_separator != 0;
        r->d = std::make_unique<IdnDecompressor>(idn, (size_t)idn_len, std::move(p));
        *out = r.release();
        return (int32_t)IDN_OK;
    });
}
// *len = 0 and *text = NULL at the end of the container
extern "C" int32_t idn_host_text_reader_next(idn_host_text_reader* r, const uint8_t** text, uint64_t* len) {
    if (!r || !text || !len) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *text = nullptr;
    *len = 0;
    return guarded([&] {
        size_t n = 0;
        r->piece.reset();
        if (r->d->next_fastq_text(r->piece, n, r->sep)) {
            *text = r->piece->p;
            *len = n;
        }
        return (int32_t)IDN_OK;
    });
}
extern "C" void idn_host_text_reader_free(idn_host_text_reader* r) { delete r; }

// the compressor writes into the caller's buffer instead of the library's growing one (set before the first add)
extern "C" int32_t idn_host_compressor_set_output(idn_host_compressor* c, uint8_t* buf, uint64_t cap) {
    if (!c || (!buf && cap)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    c->ext = buf;
    c->ext_cap = cap;
    c->ext_len = 0;
    return IDN_OK;
}

extern "C" int32_t idn_host_compressor_finish(idn_host_compressor* c) {
    if (!c) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    return guarded([&] {
        c->c->finish();
        return (int32_t)IDN_OK;
    });
}

extern "C" uint64_t idn_host_compressor_output(const idn_host_compressor* c, const uint8_t** data) {
    if (c->ext) {
        if (data) *data = c->ext;
        return c->ext_len;
    }
    if (data) *data = c->out.data();
    return c->out.size();
}

extern "C" uint32_t idn_host_compressor_retained(const idn_host_compressor* c, uint8_t* ids, uint32_t cap) {
    const auto& r = c->c->retained_models();
    for (uint32_t i = 0; i < r.size() && i < cap && ids; i++) std::memcpy(ids + 32 * i, r[i].data(), 32);
    return (uint32_t)r.size();
}

extern "C" void idn_host_compressor_stats(const idn_host_compressor* c, uint64_t out[9]) {
    const CompressionStats& s = c->c->stats();
    const uint64_t v[9] = {s.in_symbols, s.in_reads, s.in_identifier_bytes, s.out_bytes, s.out_identifier_bytes, s.out_payload_bytes,
                           s.blocks, s.acid_model_switches, s.q_score_model_switches};
    std::memcpy(out, v, sizeof v);
}

extern "C" void idn_host_compressor_free(idn_host_compressor* c) { delete c; }

extern "C" int32_t idn_host_decompress_ex(const idn_host_model* const* models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                       const uint8_t* idn, uint64_t idn_len, idn_host_decoded** out, const idn_host_decompress_params* dparams) {
    if (!out || (!idn && idn_len) || (n_models && !models)) return set_err(IDN_E_INVALID_ARG, "NULL argument");
    *out = nullptr;
    return guarded([&] {
        IdnDecompressorParams p;
        p.model_provider = provider_of(models, n_models);
        p.identifiers_on_device = dparams && dparams->identifiers_on_device;
        if (device >= 0) {
            p.devices.assign(1, device);
        } else {
            p.devices.clear();
            for (int32_t d = 0; d < -device; d++) p.devices.push_back(d);
        }
        p.batch_blocks = batch_blocks ? batch_blocks : 32;
        uint64_t pos = 0;
        IdnDecompressor d([&](uint8_t* dst, size_t n) {
            size_t k = (size_t)std::min<uint64_t>(n, idn_len - pos);
            std::memcpy(dst, idn + pos, k);
            pos += k;
            return k;
        }, std::move(p));
        auto res = std::make_unique<idn_host_decoded>();
        IdnDecompressor::DecodedBatch b;
        while (d.next_batch(b)) {  // whole batches: no per-sequence objects on this path
            const uint64_t n = b.read_off.size() - 1, s0 = res->acids.size(), n0 = res->names.size();
            res->acids.insert(res->acids.end(), b.acids.begin(), b.acids.end());
            res->quals.insert(res->quals.end(), b.quals.begin(), b.quals.end());
            if (b.any_names) res->names.insert(res->names.end(), b.names.begin(), b.names.end());
            for (uint64_t r = 1; r <= n; r++) {
                res->read_off.push_back(s0 + b.read_off[r]);
                res->name_off.push_back(n0 + (b.any_names ? b.name_off[r] : 0));
            }
        }
        res->version = d.version();
        *out = res.release();
        return (int32_t)IDN_OK;
    });
}

extern "C" uint64_t idn_host_decoded_reads(const idn_host_decoded* d) { return d->read_off.size() - 1; }
extern "C" uint32_t idn_host_decoded_version(const idn_host_decoded* d) { return d->version; }
extern "C" const uint64_t* idn_host_decoded_read_off(const idn_host_decoded* d) { return d->read_off.data(); }
extern "C" const uint8_t* idn_host_decoded_acids(const idn_host_decoded* d) { return d->acids.data(); }
extern "C" const uint8_t* idn_host_decoded_quals(const idn_host_decoded* d) { return d->quals.data(); }
extern "C" const uint64_t* idn_host_decoded_name_off(const idn_host_decoded* d) { return d->name_off.data(); }
extern "C" const uint8_t* idn_host_decoded_names(const idn_host_decoded* d) { return d->names.data(); }
extern "C" void idn_host_decoded_free(idn_host_decoded* d) { delete d; }

struct idn_host_clustering {
    Clustering c;
};
extern "C" idn_host_clustering* idn_host_clustering_new(void) { return new idn_host_clustering(); }
extern "C" void idn_host_clustering_free(idn_host_clustering* c) { delete c; }

extern "C" uint32_t idn_host_cluster(idn_host_clustering* state, const uint32_t* cost, uint64_t n_values, uint32_t n_centroids,
                                     uint32_t num_clusters, uint32_t* centroids_out, uint32_t* value_cluster_out) {
    std::vector<uint32_t> c(cost, cost + n_values * n_centroids);
    std::vector<std::vector<size_t>> members;
    Clustering fresh;
    std::vector<size_t> best = (state ? state->c : fresh).make_clusters(c, n_values, n_centroids, num_clusters, &members);
    for (size_t k = 0; k < best.size(); k++) {
        if (centroids_out) centroids_out[k] = (uint32_t)best[k];
        if (value_cluster_out)
            for (size_t v : members[k]) value_cluster_out[v] = (uint32_t)k;
    }
    return (uint32_t)best.size();
}

// known-answer hooks for the restated third-party generators (clustering.hpp)
extern "C" void idn_host_splitmix64(uint64_t seed, uint32_t n, uint64_t* out) {
    SplitMix64 g(seed);
    for (uint32_t i = 0; i < n; i++) out[i] = g.next_u64();
}
extern "C" void idn_host_xoshiro256pp(const uint64_t* state4, uint64_t seed, uint32_t n, uint64_t* out) {
    Xoshiro256PlusPlus g = state4 ? Xoshiro256PlusPlus(state4) : Xoshiro256PlusPlus(seed);
    for (uint32_t i = 0; i < n; i++) out[i] = g.next_u64();
}
// rand 0.8.5 `index::sample(&mut Xoshiro256PlusPlus::seed_from_u64(seed), length, amount)`, amount < 12; with draws != NULL the
// generator is replaced by the given u32 sequence (hand-computed cases)
extern "C" uint32_t idn_host_sample_indices(uint64_t seed, uint32_t length, uint32_t amount, uint32_t* out) {
    if (amount > length || amount >= 12) return 0;
    Xoshiro256PlusPlus g(seed);
    std::vector<uint32_t> v = sample_floyd(g, length, amount);
    for (size_t i = 0; i < v.size(); i++) out[i] = v[i];
    return (uint32_t)v.size();
}
extern "C" uint32_t idn_host_gen_range(uint64_t seed, uint32_t high, uint32_t n, uint32_t* out) {
    Xoshiro256PlusPlus g(seed);
    for (uint32_t i = 0; i < n; i++) out[i] = g.gen_range_inclusive(high);
    return n;
}

extern "C" uint32_t idn_host_rank(const uint32_t* cost, uint64_t n_values, uint32_t n_models, uint32_t model_num, uint32_t* models_out) {
    std::vector<uint32_t> c(cost, cost + n_values * n_models);
    std::vector<size_t> best = rank_models(c, n_values, n_models, model_num);
    for (size_t k = 0; k < best.size(); k++) models_out[k] = (uint32_t)best[k];
    return (uint32_t)best.size();
}

// the forms without decompressor parameters: the defaults (identifiers inflated on the host)
extern "C" int32_t idn_host_decompress_text(const idn_host_model* const* models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                            uint32_t thread_num, int32_t title_with_separator, const uint8_t* idn, uint64_t idn_len,
                                            uint8_t** text, uint64_t* text_len) {
    return idn_host_decompress_text_ex(models, n_models, device, batch_blocks, thread_num, title_with_separator, idn, idn_len, text, text_len, nullptr);
}

extern "C" int32_t idn_host_decompress_text_into(const idn_host_model* const* models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                                 uint32_t thread_num, int32_t title_with_separator, const uint8_t* idn, uint64_t idn_len,
                                                 uint8_t* text, uint64_t cap, uint64_t* text_len) {
    return idn_host_decompress_text_into_ex(models, n_models, device, batch_blocks, thread_num, title_with_separator, idn, idn_len, text, cap, text_len, nullptr);
}

extern "C" int32_t idn_host_text_reader_new(const idn_host_model* const* models, uint32_t n_models, const int32_t* devices, uint32_t n_devices,
                                            uint32_t batch_blocks, uint32_t thread_num, int32_t title_with_separator, const uint8_t* idn,
                                            uint64_t idn_len, idn_host_text_reader** out) {
    return idn_host_text_reader_new_ex(models, n_models, devices, n_devices, batch_blocks, thread_num, title_with_separator, idn, idn_len, out, nullptr);
}

extern "C" int32_t idn_host_decompress(const idn_host_model* const* models, uint32_t n_models, int32_t device, uint32_t batch_blocks,
                                       const uint8_t* idn, uint64_t idn_len, idn_host_decoded** out) {
    return idn_host_decompress_ex(models, n_models, device, batch_blocks, idn, idn_len, out, nullptr);
}
