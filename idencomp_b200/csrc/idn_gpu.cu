// idn_gpu.cu -- host side of libidn_gpu.so: the C-ABI declared in include/idn_gpu.h.
//
// Owns the device context (stream, workspaces, uploaded model tables) and sequences the kernels of
// idn_kernels.cuh.  There is no CPU fallback anywhere in this file: every entry point needs a CUDA device.
#include "../../include/idn_gpu.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <string>
#include <vector>

#include "idn_fastq.cuh"
#include "idn_native.cuh"
#include "idn_deflate.cuh"
#include "idn_inflate.cuh"

using namespace idn;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            e = cudaMalloc(&p, n);
            want = n;
        }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
};

struct ModelSlot {
    bool used = false;
    int32_t spec_tuple[5] = {0, 0, 0, 0, 0};  // kind, acid order, q order, position bits, q max
    ModelDev dev{};
    void* d_map = nullptr;
    void* d_hkeys = nullptr;
    void* d_hvals = nullptr;
    void* d_enc = nullptr;
    void* d_dec = nullptr;
    void* d_adirect = nullptr;
    void* d_aenc = nullptr;
    void* d_qwin = nullptr;
    void free_all() {
        cudaFree(d_map);
        cudaFree(d_hkeys);
        cudaFree(d_hvals);
        cudaFree(d_enc);
        cudaFree(d_dec);
        cudaFree(d_adirect);
        cudaFree(d_aenc);
        cudaFree(d_qwin);
        d_qwin = d_aenc = nullptr;
        d_map = d_hkeys = d_hvals = d_enc = d_dec = d_adirect = nullptr;
        used = false;
    }
};

constexpr uint32_t kMaxSlots = 1024;
constexpr uint64_t kDenseSpecLimit = 1ull << 22;  // dense u16 map up to 8 MB, hash above
constexpr uint64_t kDirectSpecLimit = 1ull << 19;  // acid decode rows stored per spec (8 B each) up to 4 MB

}  // namespace

struct idn_gpu_pipe;  // idn_pipeline.inc

struct idn_gpu_ctx {
    int device = 0;
    idn_gpu_pipe* pipe = nullptr;       // streams, events and double-buffered staging of the pipelined host-pointer calls
    uint32_t pipe_blocks = 32;          // blocks per sub-chunk of a host-pointer call (idn_gpu_set_pipeline_blocks)
    bool pipe_blocks_set = false;       // set by the caller: taken as is; otherwise long reads get larger sub-chunks (pipe_sub_blocks)
    uint32_t* pipe_err_out = nullptr;   // where compress_blocks_dev leaves its error flags for the pipeline (device)
    cudaStream_t stream = nullptr;  // used by the host-pointer entry points
    cudaEvent_t ev = nullptr;
    std::string err;
    uint64_t launches = 0;
    // optional per-kernel timing (idn_gpu_profile): an event after every launch; a kernel's time is the gap to the
    // previous event on the same stream (kernels of one call are serialised on one stream)
    bool profiling = false;
    std::vector<cudaEvent_t> prof_pool;
    size_t prof_used = 0;
    struct ProfMark {
        const char* name;  // nullptr = start of a call
        cudaEvent_t ev;
    };
    std::vector<ProfMark> prof_marks;
    // host wall-clock phases of the host-pointer entry points (reported by idn_gpu_profile_read as "host:<phase>")
    struct HostPhase {
        const char* name;
        uint64_t n;
        double ms;
    };
    std::vector<HostPhase> host_phases;
    std::vector<ModelSlot> slots;
    ModelDev* d_models = nullptr;  // [kMaxSlots], mirrors slots[].dev
    ModelDev d_models_host0{};     // all-zero placeholder for the by-value model parameters of the non-uniform kernels
    int sm_count = 148;
    int32_t walk_mode = 0;  // idn_gpu_set_walk
    uint32_t* d_crc_tab = nullptr;  // [256]
    uint32_t* d_xpow = nullptr;     // [64]
    uint32_t* d_crc_back = nullptr;  // [256 + 2 * kCrcLenTab]: Tinv (backward CRC step) | {x^(8n), x^(16n)} for n < kCrcLenTab
    bool enc_crc = true;             // IDN_NO_ENC_CRC=1: the per-read CRC partials of a compress call come from crc_read_kernel
    // workspaces of the *_dev paths
    DevBuf w_scratch, w_paylen, w_sizes, w_chosen, w_tiles, w_sliceoff, w_readblock, w_small, w_crcpart, w_crclen;
    DevBuf w_walkdone, w_blockadj;
    DevBuf w_lanefirst, w_laneoff, w_laneblock, w_blkinfo, w_nhdr, w_lanesym;  // native mode
    uint32_t lane_syms = 2048;  // lane quantum of the native format (tools/lane_sweep.sh: decode is 17 % faster than at 4096 for +0.5 % size)
    // FASTQ text <-> symbols (idn_fastq.cuh): results of the last parse stay here until the next one
    DevBuf f_text, f_tilecnt, f_tilebase, f_linestart, f_linefn, f_linestate, f_tilefn, f_tilestate, f_recscan, f_title, f_namelo,
        f_namelen, f_readlen, f_readoff, f_nameoff, f_names, f_acids, f_quals, f_err, f_fmtoff, f_fmttext;
    idn_fastq_info f_info{};
    uint64_t f_consumed = 0;       // bytes of the last parsed text that belong to complete records (partial parse)
    DevBuf f_blockfirst, f_nxt;    // blocks formed over the parsed reads (idn_gpu_fastq_parse_chunk)
    uint32_t f_blocks = 0;         // blocks idn_gpu_compress_parsed codes
    uint64_t f_reads_used = 0;     // = block_first[f_blocks]
    DevBuf w_index;  // decode-side per-read index
    DevBuf w_blk;    // decode-side per-block counters
    // staging of the host-pointer paths
    DevBuf s_acids, s_quals, s_readoff, s_blockfirst, s_prefix, s_names, s_nameoff, s_out, s_blockoff, s_crc, s_stats,
        s_sizes, s_blocks, s_blocklen, s_aout, s_qout, s_offout, s_status, s_idx;
    DevBuf w_bucket, w_list;       // per-read selection: reads bucketed by model pair (cnt | base | cursor, read list)
    // identifiers Deflate (idn_deflate.cuh): per-block tables, joined names, candidates, tokens, segment records, slices
    DevBuf z_blk, z_joined, z_cand, z_tok, z_ntok, z_rec, z_segblock, z_segoff, z_out;
    // identifiers Inflate (idn_inflate.cuh): streams, chunks, their state and 16-bit output, the joined text, the names
    DevBuf i_misc, i_streams, i_chunks, i_cs, i_ss, i_scratch, i_text, i_bstream, i_names, i_nameoff;
    uint32_t inflate_range = idn::inf::kDefaultRange;  // idn_gpu_set_inflate_range
    double inflate_ratio = 12.0;   // 16-bit scratch entries per compressed byte of a chunk (grows when a call outgrows it)
    bool names_valid = false;      // the last idn_gpu_inflate_names succeeded: i_names / i_nameoff hold ...
    uint32_t names_blocks = 0;     // ... the names of that many blocks ...
    uint64_t names_reads = 0, names_bytes = 0;  // ... and reads, and their size
    bool names_any = false;        // some block had an Identifiers slice
    bool bucket_pairs = true;      // IDN_NO_BUCKETS=1: the run-time generic kernels over all reads instead (for comparison)
    uint64_t resident_bytes = 0;   // container bytes idn_gpu_index_blocks / the decoder left in s_blocks ...
    uint32_t resident_blocks = 0;  // ... and how many blocks they are (0: nothing a decode call may reuse)
};

namespace {

int32_t fail(idn_gpu_ctx* c, int32_t code, const char* fmt, ...) {
    if (c) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        c->err = buf;
    }
    return code;
}

#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            (void)cudaGetLastError();                                                                  \
            return fail(ctx, IDN_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                        __LINE__);                                                                     \
        }                                                                                              \
    } while (0)

#define LAUNCHED(name)                                                                             \
    do {                                                                                           \
        ctx->launches++;                                                                           \
        if (ctx->profiling) prof_mark(ctx, name, st);                                              \
        cudaError_t e__ = cudaGetLastError();                                                      \
        if (e__ != cudaSuccess)                                                                    \
            return fail(ctx, IDN_E_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                       \
    } while (0)

void prof_mark(idn_gpu_ctx* c, const char* name, cudaStream_t st) {
    if (c->prof_used == c->prof_pool.size()) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        c->prof_pool.push_back(e);
    }
    cudaEvent_t e = c->prof_pool[c->prof_used++];
    cudaEventRecord(e, st);
    c->prof_marks.push_back({name, e});
}
#define PROF_BEGIN()                                  \
    do {                                              \
        if (ctx->profiling) prof_mark(ctx, nullptr, st); \
    } while (0)

// wait for a stream without spinning: several ctx (one host thread each) share the host's cores with the caller's own
// threads, and a spinning cudaStreamSynchronize per thread starves them (8 ranks x 3 ctx on a 32-core host)
cudaError_t sync_stream(idn_gpu_ctx* c, cudaStream_t st) {
    cudaError_t e = cudaEventRecord(c->ev, st);
    if (e != cudaSuccess) return e;
    return cudaEventSynchronize(c->ev);
}

struct HostTimer {
    idn_gpu_ctx* c;
    std::chrono::steady_clock::time_point t0;
    explicit HostTimer(idn_gpu_ctx* ctx) : c(ctx), t0(std::chrono::steady_clock::now()) {}
    void lap(const char* name) {
        if (!c->profiling) return;
        auto t1 = std::chrono::steady_clock::now();
        double ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
        t0 = t1;
        for (auto& h : c->host_phases)
            if (strcmp(h.name, name) == 0) {
                h.n++;
                h.ms += ms;
                return;
            }
        c->host_phases.push_back({name, 1, ms});
    }
};

uint32_t host_hash32(uint32_t k) {
    k ^= k >> 16;
    k *= 0x7feb352dU;
    k ^= k >> 15;
    k *= 0x846ca68bU;
    k ^= k >> 16;
    return k;
}

cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

int32_t sync_models(idn_gpu_ctx* ctx) {
    std::vector<ModelDev> host(kMaxSlots);
    memset(host.data(), 0, sizeof(ModelDev) * kMaxSlots);
    for (size_t i = 0; i < ctx->slots.size(); i++)
        if (ctx->slots[i].used) host[i] = ctx->slots[i].dev;
    CU(cudaMemcpy(ctx->d_models, host.data(), sizeof(ModelDev) * kMaxSlots, cudaMemcpyHostToDevice));
    return IDN_OK;
}

int32_t check_models(idn_gpu_ctx* ctx, const idn_model_t* models, uint32_t n_models) {
    if (!models && n_models) return fail(ctx, IDN_E_INVALID_ARG, "models is NULL");
    if (n_models > IDN_MAX_MODELS) return fail(ctx, IDN_E_INVALID_ARG, "more than %d models", IDN_MAX_MODELS);
    for (uint32_t i = 0; i < n_models; i++)
        if (models[i] < 0 || (size_t)models[i] >= ctx->slots.size() || !ctx->slots[models[i]].used)
            return fail(ctx, IDN_E_UNKNOWN_MODEL, "model handle %d is not live", (int)models[i]);
    return IDN_OK;
}

// small per-call parameter block living in w_small (device):
struct SmallParams {
    int32_t model_ids[256];            // container index -> slot
    uint8_t model_type[256];           // container index -> IDN_MODEL_ACID / IDN_MODEL_QSCORE
    uint32_t cand_cols[2 * kMaxCand];  // candidate -> column of the score matrix
    int32_t cand_model[2 * kMaxCand];  // candidate -> slot
    uint8_t cand_index[2 * kMaxCand];  // candidate -> SwitchModel index
    uint32_t n_cand[2];
    uint32_t has_sizes[2];
    int32_t score_ids[256];  // score-matrix column -> slot
    uint32_t err;            // bit 0: invalid symbol
    uint32_t native_split;   // native decode: some block of the call cuts long reads into pieces
    uint32_t pad[2];
    unsigned long long stats[8];
    int32_t status[4];
};

}  // namespace

// Kernels specialised at compile time for the (acid spec type, q-score spec type) pairs of the bundled same-sequencer
// model files; every other pair runs the run-time-generic kernels (DynSpecs).  kind: 0 generic, 1 light.
//                          acids: kind ao qo pb qm      q-scores: kind ao qo pb qm
using SP0 = StaticSpecs<1, 8, 0, 0, 1, 0, 0, 2, 6, 0>;   // light_ao8_qo0_pb0_qm1  + generic_ao0_qo2_pb6   (HiSeq: ERR174310, SRR2962693, SRR19549058)
using SP1 = StaticSpecs<1, 8, 0, 0, 1, 0, 2, 1, 6, 0>;   // light_ao8_qo0_pb0_qm1  + generic_ao2_qo1_pb6   (NovaSeq: SRR8861483)
using SP2 = StaticSpecs<0, 8, 0, 0, 0, 1, 0, 4, 0, 16>;  // generic_ao8_qo0_pb0    + light_ao0_qo4_pb0_qm16 (Sequel II: m64187e)
using SP3 = StaticSpecs<1, 4, 3, 2, 8, 1, 0, 4, 3, 16>;  // light_ao4_qo3_pb2_qm8  + light_ao0_qo4_pb3_qm16 (NovaSeq: SRR18908372)
using SP4 = StaticSpecs<0, 4, 1, 2, 0, 1, 0, 4, 3, 16>;  // generic_ao4_qo1_pb2    + light_ao0_qo4_pb3_qm16 (HiSeq 2500: SRR5373739)
using SP5 = StaticSpecs<0, 8, 0, 0, 0, 1, 2, 4, 2, 8>;   // generic_ao8_qo0_pb0    + light_ao2_qo4_pb2_qm8  (iSeq 100: ERR5462922)
using SP6 = StaticSpecs<0, 8, 0, 0, 0, 1, 0, 3, 0, 32>;  // generic_ao8_qo0_pb0    + light_ao0_qo3_pb0_qm32 (HiSeq 2500: SRR16141966)
using SP7 = StaticSpecs<0, 8, 0, 0, 0, 1, 0, 4, 3, 16>;  // generic_ao8_qo0_pb0    + light_ao0_qo4_pb3_qm16 (HiSeq 2500: SRR19609907)
// (the one remaining same-sequencer pair of the reference's models/, SRR20210997 = light_ao8_qo0_pb0_qm1 + generic_ao3_qo3_pb0,
// has a 2^27-spec q-score space served by the hashed map: it runs the run-time-generic kernels)
constexpr int kNumStaticPairs = 8;
static const int32_t kStaticPairs[kNumStaticPairs][10] = {
    {1, 8, 0, 0, 1, 0, 0, 2, 6, 0}, {1, 8, 0, 0, 1, 0, 2, 1, 6, 0}, {0, 8, 0, 0, 0, 1, 0, 4, 0, 16}, {1, 4, 3, 2, 8, 1, 0, 4, 3, 16},
    {0, 4, 1, 2, 0, 1, 0, 4, 3, 16}, {0, 8, 0, 0, 0, 1, 2, 4, 2, 8}, {0, 8, 0, 0, 0, 1, 0, 3, 0, 32}, {0, 8, 0, 0, 0, 1, 0, 4, 3, 16}};

static int static_pair_index(const idn_gpu_ctx* ctx, int32_t acid_slot, int32_t q_slot) {
    // the specialised kernels index the dense spec -> row table without looking (ctx_row<true>)
    if (!ctx->slots[acid_slot].dev.map || !ctx->slots[q_slot].dev.map || !ctx->slots[acid_slot].dev.adirect || !ctx->slots[q_slot].dev.qwin) return -1;
#ifndef IDN_NO_AENC
    if (!ctx->slots[acid_slot].dev.aenc) return -1;
#endif
    for (int i = 0; i < kNumStaticPairs; i++) {
        bool same = true;
        for (int k = 0; k < 5; k++)
            same = same && ctx->slots[acid_slot].spec_tuple[k] == kStaticPairs[i][k] && ctx->slots[q_slot].spec_tuple[k] == kStaticPairs[i][5 + k];
        if (same) return i;
    }
    return -1;
}

extern "C" int32_t idn_gpu_kernel_variant(const idn_gpu_ctx* ctx, idn_model_t acid_model, idn_model_t q_model) {
    if (!ctx) return -1;
    for (idn_model_t h : {acid_model, q_model})
        if (h < 0 || (size_t)h >= ctx->slots.size() || !ctx->slots[h].used) return -1;
    if (ctx->slots[acid_model].dev.type != IDN_MODEL_ACID || ctx->slots[q_model].dev.type != IDN_MODEL_QSCORE) return -1;
    return static_pair_index(ctx, acid_model, q_model);
}
extern "C" int32_t idn_gpu_kernel_variant_count(void) { return kNumStaticPairs; }

// launch KERNEL<true, SPi> for a specialised pair, KERNEL<true, DynSpecs> otherwise
// IDN_DEBUG_SMEM=<bytes>: dynamic shared memory added to these launches, an occupancy knob for experiments
static unsigned debug_smem() {
    static const unsigned v = [] { const char* e = getenv("IDN_DEBUG_SMEM"); return e ? (unsigned)atoi(e) : 0u; }();
    return v;
}
#define IDN_LAUNCH_UNIFORM(idx, KERNEL, grid, st, ...)                                         \
    switch (idx) {                                                                             \
        case 0: KERNEL<true, SP0><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        case 1: KERNEL<true, SP1><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        case 2: KERNEL<true, SP2><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        case 3: KERNEL<true, SP3><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        case 4: KERNEL<true, SP4><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        case 5: KERNEL<true, SP5><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        case 6: KERNEL<true, SP6><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        case 7: KERNEL<true, SP7><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
        default: KERNEL<true, DynSpecs><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;             \
    }

// the list kernels over one bucket of reads (per-read model selection, see bucket_scatter_kernel)
#define IDN_LAUNCH_LIST(idx, KERNEL, grid, st, ...)                                            \
    switch (idx) {                                                                             \
        case 0: KERNEL<SP0><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        case 1: KERNEL<SP1><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        case 2: KERNEL<SP2><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        case 3: KERNEL<SP3><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        case 4: KERNEL<SP4><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        case 5: KERNEL<SP5><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        case 6: KERNEL<SP6><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        case 7: KERNEL<SP7><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                         \
        default: KERNEL<DynSpecs><<<grid, 128, debug_smem(), st>>>(__VA_ARGS__); break;                   \
    }

// ======================================================================================================
// lifecycle
// ======================================================================================================
extern "C" int32_t idn_gpu_abi_version(void) { return IDN_GPU_ABI_VERSION; }

extern "C" int32_t idn_gpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

static void make_crc_tables(uint32_t* tab, uint32_t* xpow) {
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i;
        for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1) ? 0xEDB88320u : 0);
        tab[i] = c;
    }
    // reflected polynomial arithmetic: bit 31 is x^0.  x^8 = 0x00800000.
    auto mul = [](uint32_t a, uint32_t b) {
        uint32_t p = 0;
        for (int i = 0; i < 32; i++) {
            if (b & 0x80000000u) p ^= a;
            a = (a >> 1) ^ ((a & 1) ? 0xEDB88320u : 0);
            b <<= 1;
        }
        return p;
    };
    xpow[0] = 0x00800000u;
    for (int k = 1; k < 64; k++) xpow[k] = mul(xpow[k - 1], xpow[k - 1]);
}

// Tables of the backward CRC the encoder runs (it visits a read's symbols last to first; EncCrc in idn_kernels.cuh):
// Tinv undoes one "advance by a zero byte" step, xlen[n] = {x^(8n), x^(16n)} mod P bring the result back into place.
static void make_crc_back_tables(const uint32_t* tab, const uint32_t* xpow, uint32_t* back /*[256 + 2 * kCrcLenTab]*/) {
    uint32_t rtop[256];
    for (uint32_t i = 0; i < 256; i++) rtop[tab[i] >> 24] = i;  // the top bytes of the table are a permutation
    uint32_t* tinv = back;
    for (uint32_t t = 0; t < 256; t++) tinv[t] = (tab[rtop[t]] << 8) | rtop[t];
    auto mul = [](uint32_t a, uint32_t b) {
        uint32_t p = 0;
        for (int i = 0; i < 32; i++) {
            if (b & 0x80000000u) p ^= a;
            a = (a >> 1) ^ ((a & 1) ? 0xEDB88320u : 0);
            b <<= 1;
        }
        return p;
    };
    uint32_t* xlen = back + 256;
    uint32_t x = 0x80000000u;  // x^0
    for (uint32_t n = 0; n < kCrcLenTab; n++) {
        xlen[2 * n] = x;
        xlen[2 * n + 1] = mul(x, x);
        x = mul(x, xpow[0]);
    }
}

extern "C" int32_t idn_gpu_create(int32_t device, idn_gpu_ctx** out) {
    if (!out) return IDN_E_INVALID_ARG;
    *out = nullptr;
    int n = idn_gpu_device_count();
    if (n <= 0 || device < 0 || device >= n) return IDN_E_CUDA;  // no CPU fallback
    idn_gpu_ctx* ctx = new idn_gpu_ctx();
    ctx->device = device;
    if (const char* pb = getenv("IDN_PIPE_BLOCKS")) {
        ctx->pipe_blocks = std::max(1, atoi(pb));
        ctx->pipe_blocks_set = true;
    }
    if (getenv("IDN_NO_BUCKETS")) ctx->bucket_pairs = false;
    if (const char* w = getenv("IDN_WALK")) ctx->walk_mode = strcmp(w, "serial") == 0 ? 1 : (strcmp(w, "fast") == 0 ? 2 : 0);
    auto bail = [&](const char* what) {
        fprintf(stderr, "idn_gpu_create: %s failed: %s\n", what, cudaGetErrorString(cudaGetLastError()));
        delete ctx;
        return (int32_t)IDN_E_CUDA;
    };
    if (cudaSetDevice(device) != cudaSuccess) return bail("cudaSetDevice");
    if (cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return bail("cudaDeviceGetAttribute");
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail("cudaStreamCreate");
    if (cudaEventCreateWithFlags(&ctx->ev, cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) return bail("cudaEventCreate");
    if (cudaMalloc(&ctx->d_models, sizeof(ModelDev) * kMaxSlots) != cudaSuccess) return bail("cudaMalloc");
    if (cudaMemset(ctx->d_models, 0, sizeof(ModelDev) * kMaxSlots) != cudaSuccess) return bail("cudaMemset");
    uint32_t tab[256], xpow[64];
    make_crc_tables(tab, xpow);
    if (cudaMalloc(&ctx->d_crc_tab, sizeof tab) != cudaSuccess) return bail("cudaMalloc");
    if (cudaMalloc(&ctx->d_xpow, sizeof xpow) != cudaSuccess) return bail("cudaMalloc");
    if (cudaMemcpy(ctx->d_crc_tab, tab, sizeof tab, cudaMemcpyHostToDevice) != cudaSuccess) return bail("cudaMemcpy");
    if (cudaMemcpy(ctx->d_xpow, xpow, sizeof xpow, cudaMemcpyHostToDevice) != cudaSuccess) return bail("cudaMemcpy");
    {
        std::vector<uint32_t> back(256 + 2 * kCrcLenTab);
        make_crc_back_tables(tab, xpow, back.data());
        if (cudaMalloc(&ctx->d_crc_back, back.size() * 4) != cudaSuccess) return bail("cudaMalloc");
        if (cudaMemcpy(ctx->d_crc_back, back.data(), back.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) return bail("cudaMemcpy");
    }
    if (getenv("IDN_NO_ENC_CRC")) ctx->enc_crc = false;
    *out = ctx;
    return IDN_OK;
}

static void pipe_destroy(idn_gpu_pipe* p);  // idn_pipeline.inc

extern "C" void idn_gpu_destroy(idn_gpu_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto& s : ctx->slots)
        if (s.used) s.free_all();
    DevBuf* bufs[] = {&ctx->w_scratch, &ctx->w_paylen,  &ctx->w_sizes,   &ctx->w_chosen,     &ctx->w_tiles,  &ctx->w_sliceoff,
                      &ctx->w_readblock, &ctx->w_small, &ctx->w_crcpart, &ctx->w_crclen,     &ctx->w_index,  &ctx->w_blk,
                      &ctx->w_lanefirst, &ctx->w_laneoff, &ctx->w_laneblock, &ctx->w_blkinfo, &ctx->w_nhdr, &ctx->w_lanesym, &ctx->w_walkdone, &ctx->w_blockadj,
                      &ctx->f_text, &ctx->f_tilecnt, &ctx->f_tilebase, &ctx->f_linestart, &ctx->f_linefn, &ctx->f_linestate, &ctx->f_tilefn,
                      &ctx->f_tilestate, &ctx->f_recscan, &ctx->f_title, &ctx->f_namelo, &ctx->f_namelen, &ctx->f_readlen, &ctx->f_readoff,
                      &ctx->f_nameoff, &ctx->f_names, &ctx->f_acids, &ctx->f_quals, &ctx->f_err, &ctx->f_fmtoff, &ctx->f_fmttext,
                      &ctx->f_blockfirst, &ctx->f_nxt, &ctx->w_bucket, &ctx->w_list,
                      &ctx->s_acids,   &ctx->s_quals,   &ctx->s_readoff, &ctx->s_blockfirst, &ctx->s_prefix, &ctx->s_names,
                      &ctx->s_nameoff, &ctx->s_out,     &ctx->s_blockoff, &ctx->s_crc,       &ctx->s_stats,  &ctx->s_sizes,
                      &ctx->s_blocks,  &ctx->s_blocklen, &ctx->s_aout,    &ctx->s_qout,    &ctx->s_offout,     &ctx->s_status, &ctx->s_idx,
                      &ctx->z_blk, &ctx->z_joined, &ctx->z_cand, &ctx->z_tok, &ctx->z_ntok, &ctx->z_rec, &ctx->z_segblock,
                      &ctx->z_segoff, &ctx->z_out, &ctx->i_misc, &ctx->i_streams, &ctx->i_chunks, &ctx->i_cs, &ctx->i_ss,
                      &ctx->i_scratch, &ctx->i_text, &ctx->i_bstream, &ctx->i_names, &ctx->i_nameoff};
    for (DevBuf* b : bufs) b->release();
    pipe_destroy(ctx->pipe);
    cudaFree(ctx->d_models);
    cudaFree(ctx->d_crc_tab);
    cudaFree(ctx->d_xpow);
    cudaFree(ctx->d_crc_back);
    if (ctx->ev) cudaEventDestroy(ctx->ev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" int32_t idn_gpu_host_alloc(uint64_t bytes, void** p) {
    if (!p) return IDN_E_INVALID_ARG;
    *p = nullptr;
    if (cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        (void)cudaGetLastError();
        *p = nullptr;
        return IDN_E_CUDA;
    }
    return IDN_OK;
}
extern "C" void idn_gpu_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

extern "C" int32_t idn_gpu_set_walk(idn_gpu_ctx* ctx, int32_t mode) {
    if (!ctx) return IDN_E_INVALID_ARG;
    if (mode < 0 || mode > 2) return fail(ctx, IDN_E_INVALID_ARG, "walk mode %d", mode);
    ctx->walk_mode = mode;
    return IDN_OK;
}

extern "C" int32_t idn_gpu_set_lane_symbols(idn_gpu_ctx* ctx, uint32_t lane_syms) {
    if (!ctx) return IDN_E_INVALID_ARG;
    if (lane_syms == 0) return fail(ctx, IDN_E_INVALID_ARG, "lane_syms must be positive");
    ctx->lane_syms = lane_syms;
    return IDN_OK;
}

extern "C" const char* idn_gpu_last_error(const idn_gpu_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }
extern "C" uint64_t idn_gpu_launch_count(const idn_gpu_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ======================================================================================================
// models
// ======================================================================================================
extern "C" int32_t idn_gpu_model_upload(idn_gpu_ctx* ctx, int32_t model_type, int32_t spec_kind, int32_t acid_order,
                                        int32_t q_order, int32_t pos_bits, int32_t q_max, uint32_t n_ctx,
                                        const uint16_t* cum, const uint32_t* spec_keys, const uint32_t* spec_ctx,
                                        uint64_t n_specs, idn_model_t* handle) {
    if (!ctx || !handle || !cum) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    if (model_type != IDN_MODEL_ACID && model_type != IDN_MODEL_QSCORE)
        return fail(ctx, IDN_E_INVALID_ARG, "bad model type %d", model_type);
    if (n_ctx > 65536) return fail(ctx, IDN_E_UNSUPPORTED, "model has %u contexts (limit 65536, check_model sequence_compressor.rs:209-219)", n_ctx);
    if (n_specs && (!spec_keys || !spec_ctx)) return fail(ctx, IDN_E_INVALID_ARG, "NULL spec table");
    CU(cudaSetDevice(ctx->device));
    const SpecBuild sb = make_spec(spec_kind, acid_order, q_order, pos_bits, q_max);
    const SpecDev spec = sb.spec;
    const uint32_t bits = sb.total_bits;
    if (!sb.ok)
        return fail(ctx, IDN_E_UNSUPPORTED, "unsupported context spec type (kind %d ao %d qo %d pb %d qmax %d)", spec_kind,
                    acid_order, q_order, pos_bits, q_max);
    const uint64_t spec_num = 1ull << bits;
    const uint32_t nsym = model_type == IDN_MODEL_ACID ? kAcidSyms : kQSyms;
    const uint32_t n_rows = n_ctx + 1;
    const uint32_t total = 1u << kScaleBits;

    // validate the integer tables (Context::as_integer_cum_freqs asserts, context.rs:366-367)
    for (uint32_t r = 0; r < n_rows; r++) {
        const uint16_t* row = cum + (size_t)r * (nsym + 1);
        if (row[0] != 0 || row[nsym] != total) return fail(ctx, IDN_E_INVALID_ARG, "cum row %u does not span [0, 2^14]", r);
        for (uint32_t s = 0; s < nsym; s++)
            if (row[s + 1] <= row[s]) return fail(ctx, IDN_E_INVALID_ARG, "cum row %u has a zero frequency", r);
    }
    for (uint64_t i = 0; i < n_specs; i++) {
        if (spec_keys[i] >= spec_num) return fail(ctx, IDN_E_INVALID_ARG, "spec key %u out of range", spec_keys[i]);
        if (spec_ctx[i] >= n_ctx) return fail(ctx, IDN_E_INVALID_ARG, "context index %u out of range", spec_ctx[i]);
    }

    // Row order: contexts sorted by the position field of their specs (stable; models without position bits keep their
    // order).  A context of the bundled models belongs to ONE position bin in 99 % of the cases, a position bin owns a few
    // dozen contexts, and the reads of a thread block advance in lock step: with this numbering the rows a block touches at
    // any moment are neighbours in memory (a few KB that stay in L1) instead of being scattered over the whole table.
    // Row numbers never leave the device, so this changes no result.
    std::vector<uint32_t> new_of_old(n_ctx);  // 0-based context -> 0-based row - 1
    std::vector<uint16_t> cum_sorted;
    std::vector<uint32_t> ctx_sorted;
    if (spec.pb > 0 && n_ctx > 1 && !getenv("IDN_NO_ROW_SORT")) {
        std::vector<uint32_t> key(n_ctx, 0xffffffffu);
        for (uint64_t i = 0; i < n_specs; i++) key[spec_ctx[i]] = std::min(key[spec_ctx[i]], spec_keys[i] & ((1u << spec.pb) - 1u));
        std::vector<uint32_t> order(n_ctx);
        for (uint32_t i = 0; i < n_ctx; i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
        for (uint32_t r = 0; r < n_ctx; r++) new_of_old[order[r]] = r;
        cum_sorted.resize((size_t)n_rows * (nsym + 1));
        memcpy(cum_sorted.data(), cum, (size_t)(nsym + 1) * 2);  // row 0 = the dummy context
        for (uint32_t c = 0; c < n_ctx; c++)
            memcpy(cum_sorted.data() + (size_t)(new_of_old[c] + 1) * (nsym + 1), cum + (size_t)(c + 1) * (nsym + 1), (size_t)(nsym + 1) * 2);
        ctx_sorted.resize(n_specs);
        for (uint64_t i = 0; i < n_specs; i++) ctx_sorted[i] = new_of_old[spec_ctx[i]];
        cum = cum_sorted.data();
        spec_ctx = ctx_sorted.data();
    }
    // index of a spec in the dense per-spec tables: position-major (idn_device.cuh: spec_table_index)
    auto tix = [&](uint32_t sp) { return (size_t)spec_table_index(spec, sp); };

    ModelSlot slot;
    struct SlotGuard {  // every error exit below releases what was allocated so far
        ModelSlot* s;
        ~SlotGuard() {
            if (s) s->free_all();
        }
    } guard{&slot};
    slot.dev.spec = spec;
    slot.spec_tuple[0] = spec_kind;
    slot.spec_tuple[1] = acid_order;
    slot.spec_tuple[2] = q_order;
    slot.spec_tuple[3] = pos_bits;
    slot.spec_tuple[4] = spec_kind == IDN_SPEC_LIGHT ? q_max : 0;
    slot.dev.type = (uint32_t)model_type;
    slot.dev.nsym = nsym;
    slot.dev.n_rows = n_rows;

    // spec -> row (RansEncModel::from_model map, sequence_compressor.rs:31-40): dense u16 or open-addressing hash
    if (n_specs == 0) {
        // model without contexts: every spec is the dummy row
    } else if (spec_num <= kDenseSpecLimit && n_ctx < 65536) {  // row numbers 0 .. 65535 fit the u16 table; a model with exactly
                                                                 // 65 536 contexts (the reference's limit) goes through the hash
        std::vector<uint16_t> map(spec_num, 0);
        for (uint64_t i = 0; i < n_specs; i++) map[tix(spec_keys[i])] = (uint16_t)(spec_ctx[i] + 1);
        CU(cudaMalloc(&slot.d_map, spec_num * sizeof(uint16_t)));
        CU(cudaMemcpy(slot.d_map, map.data(), spec_num * sizeof(uint16_t), cudaMemcpyHostToDevice));
        slot.dev.map = (const uint16_t*)slot.d_map;
    } else {
        uint64_t capn = 16;
        while (capn < 2 * n_specs) capn <<= 1;
        std::vector<uint32_t> hk(capn, 0xffffffffu);
        std::vector<uint32_t> hv(capn, 0);
        for (uint64_t i = 0; i < n_specs; i++) {
            uint32_t h = host_hash32(spec_keys[i]) & (uint32_t)(capn - 1);
            while (hk[h] != 0xffffffffu && hk[h] != spec_keys[i]) h = (h + 1) & (uint32_t)(capn - 1);
            hk[h] = spec_keys[i];
            hv[h] = spec_ctx[i] + 1;
        }
        CU(cudaMalloc(&slot.d_hkeys, capn * sizeof(uint32_t)));
        CU(cudaMalloc(&slot.d_hvals, capn * sizeof(uint32_t)));
        CU(cudaMemcpy(slot.d_hkeys, hk.data(), capn * sizeof(uint32_t), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(slot.d_hvals, hv.data(), capn * sizeof(uint32_t), cudaMemcpyHostToDevice));
        slot.dev.hkeys = (const uint32_t*)slot.d_hkeys;
        slot.dev.hvals = (const uint32_t*)slot.d_hvals;
        slot.dev.hmask = (uint32_t)(capn - 1);
    }

    // encoder entries: RansEncSymbolInit (ryg rans_byte.h) folded into {rcp_freq, start | freq<<14 | rcp_shift<<28}
    std::vector<uint2> enc((size_t)n_rows * nsym);
    for (uint32_t r = 0; r < n_rows; r++) {
        const uint16_t* row = cum + (size_t)r * (nsym + 1);
        for (uint32_t s = 0; s < nsym; s++) {
            uint32_t start = row[s], freq = (uint32_t)row[s + 1] - row[s];
            uint32_t rcp = 0xffffffffu, rshift = 0;
            if (freq >= 2) {
                uint32_t shift = 0;
                while (freq > (1u << shift)) shift++;
                rcp = (uint32_t)(((1ull << (shift + 31)) + freq - 1) / freq);
                rshift = shift - 1;
            }
            enc[(size_t)r * nsym + s] = make_uint2(rcp, start | (freq << 14) | (rshift << 28));
        }
    }
    CU(cudaMalloc(&slot.d_enc, enc.size() * sizeof(uint2)));
    CU(cudaMemcpy(slot.d_enc, enc.data(), enc.size() * sizeof(uint2), cudaMemcpyHostToDevice));
    slot.dev.enc = (const uint2*)slot.d_enc;

    // decoder rows: cumulative frequencies searched directly (no 2^14-entry LUT per context)
    std::vector<uint8_t> dec;
    if (model_type == IDN_MODEL_ACID) {
        dec.resize((size_t)n_rows * 8);
        for (uint32_t r = 0; r < n_rows; r++)
            for (uint32_t k = 0; k < 4; k++) {
                uint16_t c = cum[(size_t)r * 6 + 1 + k];
                memcpy(dec.data() + (size_t)r * 8 + 2 * k, &c, 2);
            }
    } else {
        dec.assign((size_t)n_rows * kQRowBytes, 0);
        for (uint32_t r = 0; r < n_rows; r++) {
            const uint16_t* row = cum + (size_t)r * 95;
            uint8_t* d = dec.data() + (size_t)r * kQRowBytes;
#ifndef IDN_QROW352
            uint16_t* wins = reinterpret_cast<uint16_t*>(d + kQLutBytes);  // window g = starts of the symbols 4g .. 4g+7
            for (uint32_t g = 0; g < (uint32_t)kQWindows; g++)
                for (uint32_t t = 0; t < 8; t++) wins[8 * g + t] = 4 * g + t < 94 ? row[4 * g + t] : (uint16_t)total;
#else
            uint16_t* starts = reinterpret_cast<uint16_t*>(d + kQLutBytes);
            for (uint32_t sidx = 0; sidx < (uint32_t)kQStarts; sidx++) starts[sidx] = sidx < 94 ? row[sidx] : (uint16_t)total;
#endif
            uint32_t sidx = 0;
            for (uint32_t k = 0; k < (uint32_t)kQLutBytes; k++) {  // the symbol that owns slot 128 k, in units of 4 symbols
                while (row[sidx + 1] <= 128 * k) sidx++;
                d[k] = (uint8_t)(sidx >> 2);
            }
        }
    }
    CU(cudaMalloc(&slot.d_dec, dec.size()));
    CU(cudaMemcpy(slot.d_dec, dec.data(), dec.size(), cudaMemcpyHostToDevice));
    slot.dev.dec = (const uint8_t*)slot.d_dec;
    // q-score window rows (kQWinBytes per row): bucket LUT and starts window in one 16-byte gather
    if (model_type == IDN_MODEL_QSCORE && (size_t)n_rows * kQWinBytes <= ((size_t)256 << 20)) {
        std::vector<uint16_t> win((size_t)n_rows * (kQWinBytes / 2));
        for (uint32_t r = 0; r < n_rows; r++) {
            const uint16_t* row = cum + (size_t)r * 95;
            uint32_t sidx = 0;
            for (uint32_t k = 0; k < 128; k++) {
                while (row[sidx + 1] <= 128 * k) sidx++;  // the symbol that owns slot 128 k
                uint16_t* e = win.data() + ((size_t)r * 128 + k) * 8;
                e[0] = (uint16_t)sidx;
                for (uint32_t t = 0; t < 7; t++) e[1 + t] = sidx + t < 94 ? row[sidx + t] : (uint16_t)total;
            }
        }
        CU(cudaMalloc(&slot.d_qwin, win.size() * 2));
        CU(cudaMemcpy(slot.d_qwin, win.data(), win.size() * 2, cudaMemcpyHostToDevice));
        slot.dev.qwin = (const uint4*)slot.d_qwin;
    }
    // acid decode rows per spec: the decoder's spec -> row -> cum-freqs chain becomes one gather
    if (model_type == IDN_MODEL_ACID && slot.dev.map && spec_num <= kDirectSpecLimit) {  // (dense models only: the specialised kernels want both)
        std::vector<uint64_t> direct(spec_num);
        uint64_t row0;
        memcpy(&row0, dec.data(), 8);
        std::fill(direct.begin(), direct.end(), row0);
        for (uint64_t i = 0; i < n_specs; i++) memcpy(&direct[tix(spec_keys[i])], dec.data() + (size_t)(spec_ctx[i] + 1) * 8, 8);
        CU(cudaMalloc(&slot.d_adirect, spec_num * 8));
        CU(cudaMemcpy(slot.d_adirect, direct.data(), spec_num * 8, cudaMemcpyHostToDevice));
        slot.dev.adirect = (const uint2*)slot.d_adirect;
#ifndef IDN_NO_AENC
        // the encoder entries per spec, [spec][5]: spec -> row -> entry is one gather in the encoder and the scorer
        std::vector<uint2> aenc(spec_num * kAcidSyms);
        for (uint64_t sp = 0; sp < spec_num; sp++)
            for (uint32_t k = 0; k < kAcidSyms; k++) aenc[sp * kAcidSyms + k] = enc[k];  // row 0 = the dummy context
        for (uint64_t i = 0; i < n_specs; i++)
            for (uint32_t k = 0; k < kAcidSyms; k++)
                aenc[tix(spec_keys[i]) * kAcidSyms + k] = enc[(size_t)(spec_ctx[i] + 1) * kAcidSyms + k];
        CU(cudaMalloc(&slot.d_aenc, aenc.size() * sizeof(uint2)));
        CU(cudaMemcpy(slot.d_aenc, aenc.data(), aenc.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        slot.dev.aenc = (const uint2*)slot.d_aenc;
#endif
    }
    slot.used = true;

    size_t idx = ctx->slots.size();
    for (size_t i = 0; i < ctx->slots.size(); i++)
        if (!ctx->slots[i].used) {
            idx = i;
            break;
        }
    if (idx >= kMaxSlots) return fail(ctx, IDN_E_UNSUPPORTED, "too many live models");
    guard.s = nullptr;  // the context owns the buffers from here on
    if (idx == ctx->slots.size()) ctx->slots.push_back(slot);
    else ctx->slots[idx] = slot;
    *handle = (idn_model_t)idx;
    return sync_models(ctx);
}

extern "C" int32_t idn_gpu_model_release(idn_gpu_ctx* ctx, idn_model_t h) {
    if (!ctx) return IDN_E_INVALID_ARG;
    if (h < 0 || (size_t)h >= ctx->slots.size() || !ctx->slots[h].used)
        return fail(ctx, IDN_E_UNKNOWN_MODEL, "model handle %d is not live", (int)h);
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    ctx->slots[h].free_all();
    return sync_models(ctx);
}

// ======================================================================================================
// scoring
// ======================================================================================================
static int32_t check_batch(idn_gpu_ctx* ctx, const idn_batch* b) {
    if (!b) return fail(ctx, IDN_E_INVALID_ARG, "batch is NULL");
    if (b->n_reads && !b->read_off) return fail(ctx, IDN_E_INVALID_ARG, "read_off is NULL");
    if (b->n_symbols && (!b->acids || !b->quals)) return fail(ctx, IDN_E_INVALID_ARG, "symbol arrays are NULL");
    if (b->n_reads >= (1ull << 32) - 1) return fail(ctx, IDN_E_INVALID_ARG, "too many reads in one batch");
    if ((b->names != nullptr) != (b->name_off != nullptr)) return fail(ctx, IDN_E_INVALID_ARG, "names and name_off go together");
    return IDN_OK;
}

static int32_t upload_small(idn_gpu_ctx* ctx, const SmallParams& sp, cudaStream_t st) {
    CU(ctx->w_small.ensure(sizeof(SmallParams)));
    // pageable source: cudaMemcpyAsync stages it before returning, so `sp` may live on the caller's stack
    CU(cudaMemcpyAsync(ctx->w_small.p, &sp, sizeof sp, cudaMemcpyHostToDevice, st));
    return IDN_OK;
}

// K2 over `n` models (slots ids[0..n)): packs of up to 4 models per launch (measured: 4 per pass at 56 registers beats 8
// per pass at 85 by 1.36x, 2 per pass ties), columns col0.. of the [reads][n_cols] matrix
static int32_t launch_score(idn_gpu_ctx* ctx, const int32_t* ids, uint32_t n, const idn_batch* batch, uint32_t n_cols,
                            uint32_t* sizes, uint32_t* err, cudaStream_t st) {
    const uint64_t R = batch->n_reads;
    const unsigned grid = (unsigned)((R + 127) / 128);
    for (uint32_t k0 = 0; k0 < n;) {
        const uint32_t left = n - k0;
        if (left > 2) {
            ModelPack<4> P;
            P.n = left < 4 ? left : 4;
            for (uint32_t k = 0; k < 4; k++) P.m[k] = ctx->slots[ids[k0 + (k < P.n ? k : 0)]].dev;
            bool dense = true;
            for (uint32_t k = 0; k < 4; k++) dense = dense && P.m[k].map;
            if (dense) score_multi_kernel<4, true><<<grid, 128, 0, st>>>(P, batch->acids, batch->quals, batch->read_off, R, n_cols, k0, sizes, err);
            else score_multi_kernel<4, false><<<grid, 128, 0, st>>>(P, batch->acids, batch->quals, batch->read_off, R, n_cols, k0, sizes, err);
            k0 += P.n;
        } else {
            ModelPack<2> P;
            P.n = left;
            for (uint32_t k = 0; k < 2; k++) P.m[k] = ctx->slots[ids[k0 + (k < P.n ? k : 0)]].dev;
            bool dense = true;
            for (uint32_t k = 0; k < 2; k++) dense = dense && P.m[k].map;
            if (dense) score_multi_kernel<2, true><<<grid, 128, 0, st>>>(P, batch->acids, batch->quals, batch->read_off, R, n_cols, k0, sizes, err);
            else score_multi_kernel<2, false><<<grid, 128, 0, st>>>(P, batch->acids, batch->quals, batch->read_off, R, n_cols, k0, sizes, err);
            k0 += P.n;
        }
        LAUNCHED("score");
    }
    return IDN_OK;
}

extern "C" int32_t idn_gpu_score_dev(idn_gpu_ctx* ctx, const idn_batch* batch, const idn_model_t* models,
                                     uint32_t n_models, uint32_t* sizes, void* stream) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_batch(ctx, batch);
    if (rc) return rc;
    rc = check_models(ctx, models, n_models);
    if (rc) return rc;
    if (n_models == 0 || batch->n_reads == 0) return IDN_OK;
    if (!sizes) return fail(ctx, IDN_E_INVALID_ARG, "sizes is NULL");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = as_stream(stream);
    PROF_BEGIN();
    SmallParams sp;
    memset(&sp, 0, sizeof sp);
    for (uint32_t i = 0; i < n_models; i++) sp.score_ids[i] = models[i];
    rc = upload_small(ctx, sp, st);
    if (rc) return rc;
    SmallParams* dsp = ctx->w_small.as<SmallParams>();
    return launch_score(ctx, sp.score_ids, n_models, batch, n_models, sizes, &dsp->err, st);
}

extern "C" int32_t idn_gpu_score(idn_gpu_ctx* ctx, const idn_batch* b, const idn_model_t* models, uint32_t n_models,
                                 uint32_t* sizes) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_batch(ctx, b);
    if (rc) return rc;
    if (n_models == 0 || b->n_reads == 0) return check_models(ctx, models, n_models);
    if (!sizes) return fail(ctx, IDN_E_INVALID_ARG, "sizes is NULL");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    CU(ctx->s_acids.ensure(b->n_symbols + 16));
    CU(ctx->s_quals.ensure(b->n_symbols + 16));
    CU(ctx->s_readoff.ensure((b->n_reads + 1) * 8));
    CU(ctx->s_sizes.ensure(b->n_reads * n_models * 4));
    CU(cudaMemcpyAsync(ctx->s_acids.p, b->acids, b->n_symbols, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->s_quals.p, b->quals, b->n_symbols, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->s_readoff.p, b->read_off, (b->n_reads + 1) * 8, cudaMemcpyHostToDevice, st));
    idn_batch d = *b;
    d.acids = ctx->s_acids.as<uint8_t>();
    d.quals = ctx->s_quals.as<uint8_t>();
    d.read_off = ctx->s_readoff.as<uint64_t>();
    d.names = nullptr;
    d.name_off = nullptr;
    d.block_first_read = nullptr;
    rc = idn_gpu_score_dev(ctx, &d, models, n_models, ctx->s_sizes.as<uint32_t>(), st);
    if (rc) return rc;
    uint32_t err = 0;
    CU(cudaMemcpyAsync(sizes, ctx->s_sizes.p, b->n_reads * n_models * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&err, &ctx->w_small.as<SmallParams>()->err, 4, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    if (err & 1) return fail(ctx, IDN_E_INVALID_SYMBOL, "input holds an acid > 4 or a quality score > 93");
    return IDN_OK;
}

// ======================================================================================================
// compression
// ======================================================================================================
extern "C" uint64_t idn_gpu_compress_bound(uint64_t n_reads, uint64_t n_symbols, uint32_t n_blocks, uint64_t prefix_total) {
    // per read: two switches (4) + sequence header (9) + payload (<= 4*len + 8); per block: header 8 + fast switches 4
    // (the native format needs less per read but 30 bytes of headers per block)
    return 4 * n_symbols + 21 * n_reads + 32ull * n_blocks + prefix_total;
}

static int32_t idn_gpu_block_crc_dev_impl(idn_gpu_ctx* ctx, const idn_batch* batch, uint32_t* block_crc, uint8_t* out,
                                          const unsigned long long* block_off, uint64_t out_cap, cudaStream_t st, bool have_partials = false);
static int32_t compress_native_dev(idn_gpu_ctx* ctx, const idn_batch* batch, SmallParams& sp, int32_t fast,
                                   const uint32_t* prefix_len, uint8_t* out, uint64_t out_cap, uint64_t* block_off,
                                   uint32_t* block_crc, idn_compress_stats* stats_dev, cudaStream_t st);


extern "C" int32_t idn_gpu_compress_blocks_dev(idn_gpu_ctx* ctx, const idn_batch* batch, int32_t mode,
                                               const idn_model_t* models, uint32_t n_models, int32_t fast,
                                               const uint32_t* prefix_len, uint8_t* out, uint64_t out_cap,
                                               uint64_t* block_off, uint32_t* block_crc, idn_compress_stats* stats_dev,
                                               void* stream) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_batch(ctx, batch);
    if (rc) return rc;
    rc = check_models(ctx, models, n_models);
    if (rc) return rc;
    if (mode != IDN_MODE_COMPAT && mode != IDN_MODE_NATIVE) return fail(ctx, IDN_E_UNSUPPORTED, "unknown mode %d", mode);
    if (!batch->block_first_read || !block_off || (!out && out_cap)) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    if (batch->n_blocks == 0) return fail(ctx, IDN_E_INVALID_ARG, "batch has no blocks");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = as_stream(stream);
    PROF_BEGIN();
    const uint64_t R = batch->n_reads, S = batch->n_symbols;
    const uint32_t B = batch->n_blocks;
    const bool fuse_crc = ctx->enc_crc && batch->names == nullptr && R > 0;  // compat mode only (the native path returns above this use)

    // candidate lists per type, in provider order (model_provider.rs:210-238)
    SmallParams sp;
    memset(&sp, 0, sizeof sp);
    uint32_t n_score = 0;
    for (uint32_t i = 0; i < n_models; i++) {
        uint32_t t = ctx->slots[models[i]].dev.type;
        if (sp.n_cand[t] >= (uint32_t)kMaxCand) return fail(ctx, IDN_E_UNSUPPORTED, "more than %d models of one type", kMaxCand);
        uint32_t k = sp.n_cand[t]++;
        sp.cand_model[t * kMaxCand + k] = models[i];
        sp.cand_index[t * kMaxCand + k] = (uint8_t)i;
    }
    if (R > 0 && (sp.n_cand[0] == 0 || sp.n_cand[1] == 0))
        return fail(ctx, IDN_E_INVALID_STATE, "need at least one acid model and one quality score model");
    if (fast && n_models != 2) return fail(ctx, IDN_E_INVALID_STATE, "fast mode needs exactly 2 models (compressor_block.rs:96)");
    for (uint32_t t = 0; t < 2; t++) {
        sp.has_sizes[t] = !fast && sp.n_cand[t] > 1;
        if (sp.has_sizes[t])
            for (uint32_t k = 0; k < sp.n_cand[t]; k++) {
                sp.cand_cols[t * kMaxCand + k] = n_score;
                sp.score_ids[n_score++] = sp.cand_model[t * kMaxCand + k];
            }
    }
    if (mode == IDN_MODE_NATIVE) return compress_native_dev(ctx, batch, sp, fast, prefix_len, out, out_cap, block_off, block_crc, stats_dev, st);
    rc = upload_small(ctx, sp, st);
    if (rc) return rc;
    SmallParams* dsp = ctx->w_small.as<SmallParams>();

    CU(ctx->w_scratch.ensure(4 * S + kSlotExtra * R + 16));
    CU(ctx->w_paylen.ensure((R + 1) * 4));
    CU(ctx->w_sliceoff.ensure((R + 2) * 8));
    CU(ctx->w_readblock.ensure((R + 1) * 4));
    const uint32_t n_tiles = (uint32_t)((R + kScanTile - 1) / kScanTile);
    CU(ctx->w_tiles.ensure(((size_t)n_tiles + 2) * 8));
    uint8_t* chosen = nullptr;
    uint8_t* switched = nullptr;
    if (!fast) {
        CU(ctx->w_chosen.ensure(4 * R + 16));
        chosen = ctx->w_chosen.as<uint8_t>();
        switched = chosen + 2 * R;
    }

    if (R > 0) {
        if (n_score) {  // K2
            CU(ctx->w_sizes.ensure(R * n_score * 4));
            rc = launch_score(ctx, sp.score_ids, n_score, batch, n_score, ctx->w_sizes.as<uint32_t>(), &dsp->err, st);
            if (rc) return rc;
        }
        if (!fast && n_score == 0) {  // one candidate per type: no choice to make
            CU(cudaMemsetAsync(chosen, 0, 4 * R, st));
            switch_single_kernel<<<(B + 127) / 128, 128, 0, st>>>(batch->block_first_read, B, switched, R);
            LAUNCHED("switch_single");
        } else if (!fast) {  // K3
            switch_kernel<<<2 * B, 32, 0, st>>>(ctx->w_sizes.as<uint32_t>(), n_score, dsp->cand_cols, dsp->n_cand,
                                                dsp->has_sizes, batch->block_first_read, B, chosen, switched, R);
            LAUNCHED("switch");
        }
        EncodeArgs ea;  // K4
        ea.models = ctx->d_models;
        ea.acids = batch->acids;
        ea.quals = batch->quals;
        ea.n_symbols = S;
        ea.read_off = batch->read_off;
        ea.n_reads = R;
        ea.fixed_acid = sp.cand_model[0];
        ea.fixed_q = sp.cand_model[kMaxCand];
        ea.chosen = chosen;
        ea.cand_model = dsp->cand_model;
        ea.scratch = ctx->w_scratch.as<uint8_t>();
        ea.pay_len = ctx->w_paylen.as<uint32_t>();
        ea.err = &dsp->err;
        ea.switched = switched;
        ea.cand_index = dsp->cand_index;
        // no identifiers in the block CRC: the encoder leaves the per-read partials crc(acids | quals) itself (it walks the
        // symbols anyway, backwards: EncCrc), and the pass of crc_read_kernel over the input is not needed
        ea.crc_back = nullptr;
        ea.xpow = ctx->d_xpow;
        ea.part_crc = nullptr;
        ea.part_len = nullptr;
        if (fuse_crc) {
            CU(ctx->w_crcpart.ensure((R + 1) * 4));
            CU(ctx->w_crclen.ensure((R + 1) * 8));
            ea.crc_back = ctx->d_crc_back;
            ea.part_crc = ctx->w_crcpart.as<uint32_t>();
            ea.part_len = ctx->w_crclen.as<unsigned long long>();
        }
        const bool uniform = !chosen || (sp.n_cand[0] == 1 && sp.n_cand[1] == 1);
        const ModelDev& hma = ctx->slots[sp.cand_model[0]].dev;
        const ModelDev& hmq = ctx->slots[sp.cand_model[kMaxCand]].dev;
        const unsigned egrid = (unsigned)((R + 127) / 128);
        const uint32_t n_pairs = sp.n_cand[0] * sp.n_cand[1];
        if (uniform) {
            IDN_LAUNCH_UNIFORM(static_pair_index(ctx, sp.cand_model[0], sp.cand_model[kMaxCand]), encode_kernel, egrid, st, ea, hma, hmq)
            LAUNCHED("encode");
        } else if (ctx->bucket_pairs && n_pairs <= kMaxPairs && R < 0xffffffffull) {
            // reads bucketed by the pair they chose; one launch of the uniform (specialised where bundled) kernel per pair
            CU(ctx->w_bucket.ensure(3 * kMaxPairs * 4));
            CU(ctx->w_list.ensure(R * 4 + 16));
            uint32_t* cnt = ctx->w_bucket.as<uint32_t>();
            uint32_t *base = cnt + kMaxPairs, *cursor = cnt + 2 * kMaxPairs;
            CU(cudaMemsetAsync(cnt, 0, kMaxPairs * 4, st));
            const EncodePairKey key{chosen, R, sp.n_cand[1]};
            const unsigned bgrid = (unsigned)((R + 255) / 256);
            bucket_count_kernel<<<bgrid, 256, 0, st>>>(key, R, n_pairs, cnt);
            LAUNCHED("bucket_count");
            bucket_base_kernel<<<1, 32, 0, st>>>(cnt, n_pairs, base, cursor);
            LAUNCHED("bucket_base");
            bucket_scatter_kernel<<<bgrid, 256, 0, st>>>(key, R, n_pairs, cursor, ctx->w_list.as<uint32_t>());
            LAUNCHED("bucket_scatter");
            ReadList rl{ctx->w_list.as<uint32_t>(), nullptr, nullptr};
            const unsigned lgrid = (unsigned)std::min<uint64_t>(egrid, (uint64_t)ctx->sm_count * IDN_ENC_MINB);
            for (uint32_t a = 0; a < sp.n_cand[0]; a++)
                for (uint32_t q = 0; q < sp.n_cand[1]; q++) {
                    const int32_t ia = sp.cand_model[a], iq = sp.cand_model[kMaxCand + q];
                    rl.base = base + a * sp.n_cand[1] + q;
                    rl.count = cnt + a * sp.n_cand[1] + q;
                    IDN_LAUNCH_LIST(static_pair_index(ctx, ia, iq), encode_list_kernel, lgrid, st, ea, ctx->slots[ia].dev, ctx->slots[iq].dev, rl)
                    LAUNCHED("encode");
                }
        } else {
            encode_kernel<false, DynSpecs><<<egrid, 128, 0, st>>>(ea, hma, hmq);
            LAUNCHED("encode");
        }
    }

    // slice offsets: exclusive scan of per-read slice sizes
    SliceSize fn{ctx->w_paylen.as<uint32_t>(), switched, R};
    unsigned long long* tiles = ctx->w_tiles.as<unsigned long long>();
    unsigned long long* slice_off = ctx->w_sliceoff.as<unsigned long long>();
    if (n_tiles) {
        scan_reduce_kernel<<<n_tiles, kScanBlock, 0, st>>>(fn, R, tiles);
        LAUNCHED("scan_reduce");
    }
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(tiles, n_tiles);
    LAUNCHED("scan_tiles");
    if (n_tiles) {
        scan_apply_kernel<<<n_tiles, kScanBlock, 0, st>>>(fn, R, tiles, slice_off);
        LAUNCHED("scan_apply");
    } else {
        CU(cudaMemsetAsync(slice_off, 0, 8, st));
    }
    CU(ctx->w_blockadj.ensure(((size_t)B + 1) * 8));
    block_layout_kernel<<<1, 32, 0, st>>>(slice_off, batch->block_first_read, B, prefix_len, fast,
                                          reinterpret_cast<unsigned long long*>(block_off), out, out_cap, dsp->stats,
                                          ctx->w_blockadj.as<unsigned long long>());
    LAUNCHED("block_layout");
    if (R > 0) {
        read_block_kernel<<<B, 256, 0, st>>>(batch->block_first_read, B, ctx->w_readblock.as<uint32_t>());
        LAUNCHED("read_block");
        AssembleArgs aa;
        aa.read_off = batch->read_off;
        aa.n_reads = R;
        aa.pay_len = ctx->w_paylen.as<uint32_t>();
        aa.scratch = ctx->w_scratch.as<uint8_t>();
        aa.slice_off = slice_off;
        aa.block_adj = ctx->w_blockadj.as<unsigned long long>();
        aa.read_block = ctx->w_readblock.as<uint32_t>();
        aa.chosen = chosen;
        aa.switched = switched;
        aa.cand_index = dsp->cand_index;
        aa.out = out;
        aa.out_cap = out_cap;
        assemble_kernel<<<(unsigned)((R + 127) / 128), 128, 0, st>>>(aa);
        LAUNCHED("assemble");
        stats_kernel<<<592, 256, 0, st>>>(ctx->w_paylen.as<uint32_t>(), switched, R, dsp->stats);
        LAUNCHED("stats");
    }
    // K7: block CRCs into the block headers
    rc = idn_gpu_block_crc_dev_impl(ctx, batch, block_crc, out, reinterpret_cast<unsigned long long*>(block_off), out_cap, st, fuse_crc);
    if (rc) return rc;
    if (stats_dev) {
        finish_stats_kernel<<<1, 32, 0, st>>>(dsp->stats, &dsp->err, reinterpret_cast<unsigned long long*>(stats_dev), ctx->pipe_err_out);
        LAUNCHED("finish_stats");
    }
    return IDN_OK;
}

// per-read CRC partials: thread per read, or warp per read when the reads are long (avg_len = symbols per read, a hint)
static int32_t launch_crc_read(idn_gpu_ctx* ctx, const uint8_t* acids, const uint8_t* quals, const unsigned long long* read_off,
                               const uint8_t* names, const unsigned long long* name_off, uint64_t n_reads,
                               const unsigned long long* n_reads_dev, const int32_t* status, uint64_t grid_reads, uint64_t avg_len,
                               cudaStream_t st, const uint32_t* run_flag = nullptr) {
    if (avg_len >= 1024) {
        crc_read_warp_kernel<<<(unsigned)((grid_reads * 32 + 127) / 128), 128, 0, st>>>(
            acids, quals, read_off, names, name_off, n_reads, n_reads_dev, status, ctx->d_crc_tab, ctx->d_xpow,
            ctx->w_crcpart.as<uint32_t>(), ctx->w_crclen.as<unsigned long long>(), run_flag);
    } else {
        const uint64_t tiles = (grid_reads + kCrcThreads - 1) / kCrcThreads;
        const unsigned cgrid = (unsigned)std::min<uint64_t>(tiles ? tiles : 1, (uint64_t)ctx->sm_count * 2);
        crc_read_kernel<<<cgrid, kCrcThreads, 0, st>>>(acids, quals, read_off, names, name_off, n_reads, n_reads_dev,
                                                                             status, ctx->d_crc_tab, ctx->d_xpow,
                                                                             ctx->w_crcpart.as<uint32_t>(),
                                                                             ctx->w_crclen.as<unsigned long long>(), run_flag);
    }
    LAUNCHED("crc_read");
    return IDN_OK;
}

static int32_t idn_gpu_block_crc_dev_impl(idn_gpu_ctx* ctx, const idn_batch* batch, uint32_t* block_crc, uint8_t* out,
                                          const unsigned long long* block_off, uint64_t out_cap, cudaStream_t st, bool have_partials) {
    const uint64_t R = batch->n_reads;
    CU(ctx->w_crcpart.ensure((R + 1) * 4));
    CU(ctx->w_crclen.ensure((R + 1) * 8));
    if (R > 0 && !have_partials) {  // (have_partials: the encoder of this call left them)
        int32_t rc = launch_crc_read(ctx, batch->acids, batch->quals, reinterpret_cast<const unsigned long long*>(batch->read_off),
                                     batch->names, reinterpret_cast<const unsigned long long*>(batch->name_off), R, nullptr, nullptr, R,
                                     batch->n_symbols / R, st);
        if (rc) return rc;
    }
    crc_block_kernel<<<batch->n_blocks, 256, 0, st>>>(ctx->w_crcpart.as<uint32_t>(), ctx->w_crclen.as<unsigned long long>(),
                                                      batch->block_first_read, batch->n_blocks, ctx->d_xpow, block_crc, out,
                                                      block_off, out_cap);
    LAUNCHED("crc_block");
    return IDN_OK;
}

// ======================================================================================================
// native multi-lane format (container version 2, idn_native.cuh)
// ======================================================================================================
template <class Fn>
static int32_t scan_u64(idn_gpu_ctx* ctx, Fn fn, uint64_t n, unsigned long long* out, cudaStream_t st) {
    const uint32_t n_tiles = (uint32_t)((n + kScanTile - 1) / kScanTile);
    CU(ctx->w_tiles.ensure(((size_t)n_tiles + 2) * 8));
    unsigned long long* tiles = ctx->w_tiles.as<unsigned long long>();
    if (n_tiles) {
        scan_reduce_kernel<<<n_tiles, kScanBlock, 0, st>>>(fn, n, tiles);
        LAUNCHED("scan_reduce");
    }
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(tiles, n_tiles);
    LAUNCHED("scan_tiles");
    if (n_tiles) {
        scan_apply_kernel<<<n_tiles, kScanBlock, 0, st>>>(fn, n, tiles, out);
        LAUNCHED("scan_apply");
    } else {
        CU(cudaMemsetAsync(out, 0, 8, st));
    }
    return IDN_OK;
}

static int32_t compress_native_dev(idn_gpu_ctx* ctx, const idn_batch* batch, SmallParams& sp, int32_t fast,
                                   const uint32_t* prefix_len, uint8_t* out, uint64_t out_cap, uint64_t* block_off,
                                   uint32_t* block_crc, idn_compress_stats* stats_dev, cudaStream_t st) {
    const uint64_t R = batch->n_reads, S = batch->n_symbols;
    const uint32_t B = batch->n_blocks;
    const uint32_t Q = ctx->lane_syms;
    int32_t rc = upload_small(ctx, sp, st);
    if (rc) return rc;
    SmallParams* dsp = ctx->w_small.as<SmallParams>();
    // lanes per block <= 1 + its symbols / Q (a lane starts the block or changes the quantum); without cut reads also <= reads
    uint64_t lane_cap = S / Q + 2ull * B + 1;
    if (Q < kNativeMinSplitQ && lane_cap > R) lane_cap = R;
    CU(ctx->w_readblock.ensure((R + 1) * 4));
    CU(ctx->w_sliceoff.ensure((R + 2) * 8));          // lane_scan
    CU(ctx->w_lanefirst.ensure((lane_cap + 2) * 4));
    CU(ctx->w_lanesym.ensure((lane_cap + 2) * 8));
    CU(ctx->w_paylen.ensure((lane_cap + 1) * 4));     // lane_len
    CU(ctx->w_laneoff.ensure((lane_cap + 2) * 8));
    CU(ctx->w_laneblock.ensure((lane_cap + 1) * 4));
    CU(ctx->w_blkinfo.ensure(((size_t)B + 2) * 4 * 3));
    CU(ctx->w_scratch.ensure(4 * S + kLaneSlotExtra * (lane_cap + 1) + 16));
    uint32_t* read_block = ctx->w_readblock.as<uint32_t>();
    unsigned long long* lane_scan = ctx->w_sliceoff.as<unsigned long long>();
    uint32_t* lane_first = ctx->w_lanefirst.as<uint32_t>();
    unsigned long long* lane_sym = ctx->w_lanesym.as<unsigned long long>();
    uint32_t* lane_len = ctx->w_paylen.as<uint32_t>();
    unsigned long long* lane_off = ctx->w_laneoff.as<unsigned long long>();
    uint32_t* lane_block = ctx->w_laneblock.as<uint32_t>();
    uint32_t* blk_width = ctx->w_blkinfo.as<uint32_t>();
    uint32_t* blk_const = blk_width + B + 2;
    uint32_t* blk_lane0 = blk_const + B + 2;
    const unsigned long long* n_lanes_dev = lane_scan + R;
    unsigned long long* boff = reinterpret_cast<unsigned long long*>(block_off);

    LaneCount lf{batch->read_off, batch->block_first_read, read_block, Q};
    if (R > 0) {
        read_block_kernel<<<B, 256, 0, st>>>(batch->block_first_read, B, read_block);
        LAUNCHED("read_block");
    }
    rc = scan_u64(ctx, lf, R, lane_scan, st);
    if (rc) return rc;
    uint8_t* lane_choice = nullptr;
    const bool uniform = sp.n_cand[0] == 1 && sp.n_cand[1] == 1;
    (void)fast;  // one model pair per lane either way; fast only restricts the provider to 2 models
    if (R > 0) {
        lane_scatter_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(lf, R, lane_scan, lane_first, lane_sym);
        LAUNCHED("lane_scatter");
        uint32_t n_score = 0;
        for (uint32_t t = 0; t < 2; t++)
            if (sp.has_sizes[t]) n_score += sp.n_cand[t];
        if (n_score) {
            CU(ctx->w_sizes.ensure(R * n_score * 4));
            CU(ctx->w_chosen.ensure(2 * lane_cap + 16));
            lane_choice = ctx->w_chosen.as<uint8_t>();
            rc = launch_score(ctx, sp.score_ids, n_score, batch, n_score, ctx->w_sizes.as<uint32_t>(), &dsp->err, st);
            if (rc) return rc;
            lane_choose_kernel<<<(unsigned)((2 * lane_cap + 127) / 128), 128, 0, st>>>(
                ctx->w_sizes.as<uint32_t>(), n_score, dsp->cand_cols, dsp->n_cand, dsp->has_sizes, lane_first, lane_sym, batch->read_off, R,
                n_lanes_dev, lane_cap, lane_choice);
            LAUNCHED("lane_choose");
        }
        EncodeLaneArgs ea;
        ea.models = ctx->d_models;
        ea.acids = batch->acids;
        ea.quals = batch->quals;
        ea.n_symbols = S;
        ea.read_off = batch->read_off;
        ea.n_reads = R;
        ea.lane_first = lane_first;
        ea.lane_sym = lane_sym;
        ea.n_lanes_dev = n_lanes_dev;
        ea.lane_cap = lane_cap;
        ea.lane_choice = lane_choice;
        ea.cand_model = dsp->cand_model;
        ea.scratch = ctx->w_scratch.as<uint8_t>();
        ea.lane_len = lane_len;
        ea.err = &dsp->err;
        const ModelDev& hma = ctx->slots[sp.cand_model[0]].dev;
        const ModelDev& hmq = ctx->slots[sp.cand_model[kMaxCand]].dev;
        const unsigned grid = (unsigned)((lane_cap + 127) / 128);
        const uint32_t n_pairs = sp.n_cand[0] * sp.n_cand[1];
        if (uniform) {
            IDN_LAUNCH_UNIFORM(static_pair_index(ctx, sp.cand_model[0], sp.cand_model[kMaxCand]), encode_lane_kernel, grid, st, ea, hma, hmq)
            LAUNCHED("encode_lane");
        } else if (ctx->bucket_pairs && lane_choice && n_pairs <= kMaxPairs && lane_cap < 0xffffffffull) {
            // lanes bucketed by the pair lane_choose_kernel picked; one launch of the uniform kernel per pair (see the compat path)
            CU(ctx->w_bucket.ensure(3 * kMaxPairs * 4));
            CU(ctx->w_list.ensure(lane_cap * 4 + 16));
            uint32_t* cnt = ctx->w_bucket.as<uint32_t>();
            uint32_t *base = cnt + kMaxPairs, *cursor = cnt + 2 * kMaxPairs;
            CU(cudaMemsetAsync(cnt, 0, kMaxPairs * 4, st));
            const EncodeLanePairKey key{lane_choice, n_lanes_dev, lane_cap, sp.n_cand[1]};
            const unsigned bgrid = (unsigned)((lane_cap + 255) / 256);
            bucket_count_kernel<<<bgrid, 256, 0, st>>>(key, lane_cap, n_pairs, cnt);
            LAUNCHED("bucket_count");
            bucket_base_kernel<<<1, 32, 0, st>>>(cnt, n_pairs, base, cursor);
            LAUNCHED("bucket_base");
            bucket_scatter_kernel<<<bgrid, 256, 0, st>>>(key, lane_cap, n_pairs, cursor, ctx->w_list.as<uint32_t>());
            LAUNCHED("bucket_scatter");
            ReadList rl{ctx->w_list.as<uint32_t>(), nullptr, nullptr};
            const unsigned lgrid = (unsigned)std::min<uint64_t>(grid, (uint64_t)ctx->sm_count * IDN_LANE_MINB);
            for (uint32_t a = 0; a < sp.n_cand[0]; a++)
                for (uint32_t q = 0; q < sp.n_cand[1]; q++) {
                    const int32_t ia = sp.cand_model[a], iq = sp.cand_model[kMaxCand + q];
                    rl.base = base + a * sp.n_cand[1] + q;
                    rl.count = cnt + a * sp.n_cand[1] + q;
                    IDN_LAUNCH_LIST(static_pair_index(ctx, ia, iq), encode_lane_list_kernel, lgrid, st, ea, ctx->slots[ia].dev, ctx->slots[iq].dev, rl)
                    LAUNCHED("encode_lane");
                }
        } else {
            encode_lane_kernel<false, DynSpecs><<<grid, 128, 0, st>>>(ea, hma, hmq);
            LAUNCHED("encode_lane");
        }
    }
    LaneLenFn ll{lane_len, n_lanes_dev};
    rc = scan_u64(ctx, ll, lane_cap, lane_off, st);
    if (rc) return rc;
    native_block_info_kernel<<<B, 256, 0, st>>>(batch->read_off, batch->block_first_read, B, lane_scan, Q, blk_width, blk_const,
                                                blk_lane0);
    LAUNCHED("native_block_info");
    native_layout_kernel<<<1, 32, 0, st>>>(batch->block_first_read, B, prefix_len, blk_width, blk_lane0, lane_off, boff, out,
                                           out_cap, dsp->stats);
    LAUNCHED("native_layout");
    if (R > 0) {
        lane_block_kernel<<<B, 256, 0, st>>>(blk_lane0, B, lane_block);
        LAUNCHED("lane_block");
        NativeAssembleArgs aa;
        aa.read_off = batch->read_off;
        aa.block_first = batch->block_first_read;
        aa.n_blocks = B;
        aa.prefix_len = prefix_len;
        aa.blk_width = blk_width;
        aa.blk_const_len = blk_const;
        aa.blk_lane0 = blk_lane0;
        aa.lane_first = lane_first;
        aa.lane_sym = lane_sym;
        aa.lane_len = lane_len;
        aa.lane_off = lane_off;
        aa.lane_choice = lane_choice;
        aa.cand_index = dsp->cand_index;
        aa.n_lanes_dev = n_lanes_dev;
        aa.lane_cap = lane_cap;
        aa.lane_syms = Q;
        aa.block_off = boff;
        aa.out = out;
        aa.out_cap = out_cap;
        native_header_kernel<<<B, 256, 0, st>>>(aa);
        LAUNCHED("native_header");
        native_copy_kernel<<<(unsigned)((lane_cap * 32 + 255) / 256), 256, 0, st>>>(aa, ctx->w_scratch.as<uint8_t>(), lane_block);
        LAUNCHED("native_copy");
    }
    rc = idn_gpu_block_crc_dev_impl(ctx, batch, block_crc, out, boff, out_cap, st);
    if (rc) return rc;
    if (stats_dev) {
        finish_stats_kernel<<<1, 32, 0, st>>>(dsp->stats, &dsp->err, reinterpret_cast<unsigned long long*>(stats_dev), ctx->pipe_err_out);
        LAUNCHED("finish_stats");
    }
    return IDN_OK;
}

// upload a host batch into the staging buffers; returns the device view
static int32_t stage_batch(idn_gpu_ctx* ctx, const idn_batch* b, idn_batch* d, cudaStream_t st) {
    CU(ctx->s_acids.ensure(b->n_symbols + 16));
    CU(ctx->s_quals.ensure(b->n_symbols + 16));
    CU(ctx->s_readoff.ensure((b->n_reads + 1) * 8));
    CU(ctx->s_blockfirst.ensure(((size_t)b->n_blocks + 1) * 4));
    if (b->n_symbols) {
        CU(cudaMemcpyAsync(ctx->s_acids.p, b->acids, b->n_symbols, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->s_quals.p, b->quals, b->n_symbols, cudaMemcpyHostToDevice, st));
    }
    if (b->n_reads) {
        CU(cudaMemcpyAsync(ctx->s_readoff.p, b->read_off, (b->n_reads + 1) * 8, cudaMemcpyHostToDevice, st));
    } else {
        CU(cudaMemsetAsync(ctx->s_readoff.p, 0, 8, st));
    }
    CU(cudaMemcpyAsync(ctx->s_blockfirst.p, b->block_first_read, ((size_t)b->n_blocks + 1) * 4, cudaMemcpyHostToDevice, st));
    *d = *b;
    d->acids = ctx->s_acids.as<uint8_t>();
    d->quals = ctx->s_quals.as<uint8_t>();
    d->read_off = ctx->s_readoff.as<uint64_t>();
    d->block_first_read = ctx->s_blockfirst.as<uint32_t>();
    d->names = nullptr;
    d->name_off = nullptr;
    if (b->names && b->n_reads) {
        uint64_t nbytes = b->name_off[b->n_reads];
        CU(ctx->s_names.ensure(nbytes + 16));
        CU(ctx->s_nameoff.ensure((b->n_reads + 1) * 8));
        if (nbytes) CU(cudaMemcpyAsync(ctx->s_names.p, b->names, nbytes, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ctx->s_nameoff.p, b->name_off, (b->n_reads + 1) * 8, cudaMemcpyHostToDevice, st));
        d->names = ctx->s_names.as<uint8_t>();
        d->name_off = ctx->s_nameoff.as<uint64_t>();
    }
    return IDN_OK;
}

static int32_t check_host_batch(idn_gpu_ctx* ctx, const idn_batch* b, bool need_blocks, bool every_read = true) {
    int32_t rc = check_batch(ctx, b);
    if (rc) return rc;
    if (b->n_reads) {
        if (b->read_off[0] != 0 || b->read_off[b->n_reads] != b->n_symbols)
            return fail(ctx, IDN_E_INVALID_ARG, "read_off does not span [0, n_symbols]");
        for (uint64_t r = 0; every_read && r < b->n_reads; r++) {
            if (b->read_off[r + 1] < b->read_off[r]) return fail(ctx, IDN_E_INVALID_ARG, "read_off is not monotone");
            if (b->read_off[r + 1] - b->read_off[r] > (1ull << 26))
                return fail(ctx, IDN_E_SEQUENCE_TOO_LONG, "read %llu is longer than 2^26 symbols", (unsigned long long)r);
        }
    } else if (b->n_symbols) {
        return fail(ctx, IDN_E_INVALID_ARG, "symbols without reads");
    }
    if (need_blocks) {
        if (!b->block_first_read || b->n_blocks == 0) return fail(ctx, IDN_E_INVALID_ARG, "batch has no blocks");
        if (b->block_first_read[0] != 0 || b->block_first_read[b->n_blocks] != b->n_reads)
            return fail(ctx, IDN_E_INVALID_ARG, "block_first_read does not span [0, n_reads]");
        for (uint32_t i = 0; i < b->n_blocks; i++)
            if (b->block_first_read[i + 1] < b->block_first_read[i])
                return fail(ctx, IDN_E_INVALID_ARG, "block_first_read is not monotone");
    }
    return IDN_OK;
}

static int32_t compress_blocks_pipelined(idn_gpu_ctx* ctx, const idn_batch* b, int32_t mode, const idn_model_t* models,
                                         uint32_t n_models, int32_t fast, const uint32_t* prefix_len, uint8_t* out, uint64_t out_cap,
                                         uint64_t* block_off, uint32_t* block_crc, idn_compress_stats* stats);

extern "C" int32_t idn_gpu_compress_blocks(idn_gpu_ctx* ctx, const idn_batch* b, int32_t mode, const idn_model_t* models,
                                           uint32_t n_models, int32_t fast, const uint32_t* prefix_len, uint8_t* out,
                                           uint64_t out_cap, uint64_t* block_off, uint32_t* block_crc,
                                           idn_compress_stats* stats) {
    if (!ctx) return IDN_E_INVALID_ARG;
    // the tables that frame the batch are checked here; the reads of each sub-chunk are checked inside the pipeline while
    // the device is busy with the sub-chunks before it
    int32_t rc = check_host_batch(ctx, b, true, false);
    if (rc) return rc;
    rc = check_models(ctx, models, n_models);
    if (rc) return rc;
    if (!block_off || (!out && out_cap)) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    if (mode != IDN_MODE_COMPAT && mode != IDN_MODE_NATIVE) return fail(ctx, IDN_E_UNSUPPORTED, "unknown mode %d", mode);
    CU(cudaSetDevice(ctx->device));
    // sub-chunks of whole blocks flow through upload / kernels / download streams (idn_pipeline.inc)
    return compress_blocks_pipelined(ctx, b, mode, models, n_models, fast, prefix_len, out, out_cap, block_off, block_crc, stats);
}

extern "C" int32_t idn_gpu_block_crc(idn_gpu_ctx* ctx, const idn_batch* b, uint32_t* block_crc) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_host_batch(ctx, b, true);
    if (rc) return rc;
    if (!block_crc) return fail(ctx, IDN_E_INVALID_ARG, "block_crc is NULL");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    idn_batch d;
    rc = stage_batch(ctx, b, &d, st);
    if (rc) return rc;
    CU(ctx->s_crc.ensure((size_t)b->n_blocks * 4));
    rc = idn_gpu_block_crc_dev_impl(ctx, &d, ctx->s_crc.as<uint32_t>(), nullptr, nullptr, 0, st);
    if (rc) return rc;
    CU(cudaMemcpyAsync(block_crc, ctx->s_crc.p, (size_t)b->n_blocks * 4, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    return IDN_OK;
}

// ======================================================================================================
// decompression
// ======================================================================================================
namespace {
// per-read index arrays carved out of w_index for `cap` entries
size_t index_bytes(uint64_t cap) { return (cap + 2) * (8 + 8 + 4 + 4 + 1 + 1) + 64; }
ReadIndexDev carve_index(void* base, uint64_t cap) {
    ReadIndexDev ix;
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    ix.pay_off = reinterpret_cast<unsigned long long*>(p);
    p += (cap + 2) * 8;
    ix.sym_off = reinterpret_cast<unsigned long long*>(p);
    p += (cap + 2) * 8;
    ix.pay_len = reinterpret_cast<uint32_t*>(p);
    p += (cap + 2) * 4;
    ix.seq_len = reinterpret_cast<uint32_t*>(p);
    p += (cap + 2) * 4;
    ix.am = p;
    p += cap + 2;
    ix.qm = p;
    return ix;
}
// per-block counters of the decode side, carved out of w_blk: each [B + 2] u64
struct BlockCounters {
    unsigned long long *reads, *syms, *slots;
};
BlockCounters carve_counters(void* base, uint32_t B) {
    BlockCounters c;
    c.reads = reinterpret_cast<unsigned long long*>(base);
    c.syms = c.reads + B + 2;
    c.slots = c.syms + B + 2;
    return c;
}
}  // namespace

// shared by idn_gpu_index_blocks and the decoder: slot bases, the slice walk, and the scans.  Leaves in w_blk the
// exclusive scans reads[0..B] / syms[0..B] ([B] = totals) and slots[0..B]; the per-read index in w_index.
static int32_t index_walk(idn_gpu_ctx* ctx, const uint8_t* blocks, const unsigned long long* block_off,
                          const uint32_t* block_len, uint32_t B, uint64_t blocks_bytes, const SmallParams* dsp,
                          uint32_t n_models, cudaStream_t st) {
    CU(ctx->w_blk.ensure(((size_t)B + 2) * 8 * 3));
    BlockCounters bc = carve_counters(ctx->w_blk.p, B);
    const uint64_t cap = blocks_bytes / 17 + B + 1;  // every Sequence slice takes at least 17 bytes
    CU(ctx->w_index.ensure(index_bytes(cap)));
    ReadIndexDev ix = carve_index(ctx->w_index.p, cap);
    slot_count_kernel<<<(B + 127) / 128, 128, 0, st>>>(block_off, block_len, B, bc.slots);
    LAUNCHED("slot_count");
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(bc.slots, B);
    LAUNCHED("scan_tiles");
    slot_cap_check_kernel<<<1, 32, 0, st>>>(bc.slots + B, cap, const_cast<int32_t*>(dsp->status));
    LAUNCHED("slot_cap_check");
    CU(ctx->w_walkdone.ensure((size_t)B + 16));
    const bool fast = ctx->walk_mode == 0 ? B < kWalkFastMaxBlocks : ctx->walk_mode == 2;
    uint8_t* done = fast ? ctx->w_walkdone.as<uint8_t>() : nullptr;
    if (done) {
        walk_fast_kernel<<<B, kWalkFastThreads, 0, st>>>(blocks, block_off, block_len, B, blocks_bytes, dsp->model_type, n_models,
                                                         bc.slots, ix, bc.reads, bc.syms, done, dsp->status);
        LAUNCHED("walk_fast");
    }
    walk_kernel<<<B, 32, 0, st>>>(blocks, block_off, block_len, B, blocks_bytes, dsp->model_type, n_models, bc.slots, ix, bc.reads,
                                  bc.syms, const_cast<int32_t*>(dsp->status), done);
    LAUNCHED("walk");
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(bc.reads, B);
    LAUNCHED("scan_tiles");
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(bc.syms, B);
    LAUNCHED("scan_tiles");
    return IDN_OK;
}

static void fill_decode_params(idn_gpu_ctx* ctx, SmallParams* sp, const idn_model_t* models, uint32_t n_models) {
    memset(sp, 0, sizeof *sp);
    for (uint32_t i = 0; i < n_models; i++) {
        sp->model_ids[i] = models[i];
        sp->model_type[i] = (uint8_t)ctx->slots[models[i]].dev.type;
    }
    sp->status[1] = -1;
}

static int32_t decompress_native_dev(idn_gpu_ctx* ctx, const uint8_t* blocks, const unsigned long long* boff,
                                     const uint32_t* block_len, const uint32_t* block_crc, uint32_t n_blocks,
                                     uint64_t blocks_bytes, const idn_model_t* models, uint32_t n_models, uint8_t* acids_out,
                                     uint8_t* quals_out, uint64_t* read_off_out, uint64_t out_reads_cap,
                                     uint64_t out_symbols_cap, int32_t* status_dev, SmallParams* dsp, cudaStream_t st) {
    CU(ctx->w_blk.ensure(((size_t)n_blocks + 2) * 8 * 3));
    BlockCounters bc = carve_counters(ctx->w_blk.p, n_blocks);  // reads, syms, slots (= lanes here)
    CU(ctx->w_nhdr.ensure(((size_t)n_blocks + 1) * sizeof(NativeBlockHdr)));
    NativeBlockHdr* hdr = ctx->w_nhdr.as<NativeBlockHdr>();
    // lanes <= reads, plus one per kNativeMinSplitQ symbols when long reads are cut into pieces (idn_native.cuh)
    const uint64_t lane_cap = out_reads_cap + out_symbols_cap / kNativeMinSplitQ + n_blocks + 2;
    CU(ctx->w_index.ensure(index_bytes(lane_cap)));
    CU(ctx->w_lanesym.ensure((lane_cap + 2) * 8));
    ReadIndexDev rix = carve_index(ctx->w_index.p, lane_cap);
    NativeIndex ix{rix.pay_off, rix.pay_len, rix.sym_off, ctx->w_lanesym.as<unsigned long long>(), rix.am, rix.qm, lane_cap};
    CU(ctx->w_readblock.ensure(((size_t)n_blocks + 2) * 4));
    uint32_t* block_first = ctx->w_readblock.as<uint32_t>();
    unsigned long long* roff = reinterpret_cast<unsigned long long*>(read_off_out);
    if (!roff) {
        CU(ctx->w_sliceoff.ensure((out_reads_cap + 2) * 8));
        roff = ctx->w_sliceoff.as<unsigned long long>();
    }
    native_hdr_kernel<<<n_blocks, 32, 0, st>>>(blocks, boff, block_len, n_blocks, blocks_bytes, n_models, dsp->model_type, hdr,
                                               bc.reads, bc.syms, bc.slots, dsp->status, &dsp->native_split);
    LAUNCHED("native_hdr");
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(bc.reads, n_blocks);
    LAUNCHED("scan_tiles");
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(bc.syms, n_blocks);
    LAUNCHED("scan_tiles");
    scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(bc.slots, n_blocks);
    LAUNCHED("scan_tiles");
    index_check_kernel<<<(n_blocks + 1 + 255) / 256, 256, 0, st>>>(bc.reads, bc.syms, n_blocks, out_reads_cap, out_symbols_cap,
                                                                 block_first, dsp->status);
    LAUNCHED("index_check");
    native_fill_kernel<<<n_blocks + 1, kScanBlock, 0, st>>>(blocks, hdr, n_blocks, bc.reads, bc.syms, bc.slots, roff, ix,
                                                            block_first, dsp->status);
    LAUNCHED("native_fill");
    if (out_reads_cap) {
        DecodeLaneArgs da;
        da.models = ctx->d_models;
        da.model_ids = dsp->model_ids;
        da.payload = blocks;
        da.ix = ix;
        da.n_lanes_dev = bc.slots + n_blocks;
        da.read_off = roff;
        da.status = dsp->status;
        da.split_flag = &dsp->native_split;
        da.acids_out = acids_out;
        da.quals_out = quals_out;
        da.out_dq = (long long)(quals_out - acids_out);
        da.err = &dsp->err;
        da.part_crc = nullptr;
        da.part_len = nullptr;
        da.crc_tab = da.xpow = nullptr;
        if (block_crc) {  // the lane decoder leaves the per-read CRC partials for crc_verify_kernel
            CU(ctx->w_crcpart.ensure((out_reads_cap + 1) * 4));
            CU(ctx->w_crclen.ensure((out_reads_cap + 1) * 8));
            da.part_crc = ctx->w_crcpart.as<uint32_t>();
            da.part_len = ctx->w_crclen.as<unsigned long long>();
            da.crc_tab = ctx->d_crc_tab;
            da.xpow = ctx->d_xpow;
            // empty reads that no lane visits keep the partial of an empty read
            CU(cudaMemsetAsync(da.part_crc, 0, (out_reads_cap + 1) * 4, st));
            CU(cudaMemsetAsync(da.part_len, 0, (out_reads_cap + 1) * 8, st));
        }
        int ua = -1, uq = -1, na = 0, nq = 0;
        for (uint32_t i = 0; i < n_models; i++) {
            if (ctx->slots[models[i]].dev.type == IDN_MODEL_ACID) { ua = models[i]; na++; } else { uq = models[i]; nq++; }
        }
        // one thread per lane; the kernel strides, so a call with more lanes than this estimate (many cut reads) still decodes
        const uint64_t lanes_est = std::min<uint64_t>(lane_cap, out_reads_cap + out_symbols_cap / 1024 + n_blocks);
        const unsigned grid = (unsigned)std::max<uint64_t>(1, (lanes_est + 127) / 128);
        if (na == 1 && nq == 1) {
            IDN_LAUNCH_UNIFORM(static_pair_index(ctx, ua, uq), decode_lane_kernel, grid, st, da, ctx->slots[ua].dev, ctx->slots[uq].dev)
            LAUNCHED("decode_lane");
        } else if (ctx->bucket_pairs && n_models * n_models <= kMaxPairs && lane_cap < 0xffffffffull) {
            // lanes bucketed by the model pair of the lane table; one launch of the uniform kernel per (acid, q-score) pair
            const uint32_t n_pairs = n_models * n_models;
            CU(ctx->w_bucket.ensure(3 * kMaxPairs * 4));
            CU(ctx->w_list.ensure(lane_cap * 4 + 16));
            uint32_t* cnt = ctx->w_bucket.as<uint32_t>();
            uint32_t *base = cnt + kMaxPairs, *cursor = cnt + 2 * kMaxPairs;
            CU(cudaMemsetAsync(cnt, 0, kMaxPairs * 4, st));
            const DecodeLanePairKey key{ix.am, ix.qm, da.n_lanes_dev, dsp->status, n_models};
            const unsigned bgrid = (unsigned)((lane_cap + 255) / 256);
            bucket_count_kernel<<<bgrid, 256, 0, st>>>(key, lane_cap, n_pairs, cnt);
            LAUNCHED("bucket_count");
            bucket_base_kernel<<<1, 32, 0, st>>>(cnt, n_pairs, base, cursor);
            LAUNCHED("bucket_base");
            bucket_scatter_kernel<<<bgrid, 256, 0, st>>>(key, lane_cap, n_pairs, cursor, ctx->w_list.as<uint32_t>());
            LAUNCHED("bucket_scatter");
            ReadList rl{ctx->w_list.as<uint32_t>(), nullptr, nullptr};
            const unsigned lgrid = (unsigned)std::min<uint64_t>(grid, (uint64_t)ctx->sm_count * IDN_LANE_MINB);
            for (uint32_t a = 0; a < n_models; a++) {
                if (ctx->slots[models[a]].dev.type != IDN_MODEL_ACID) continue;
                for (uint32_t q = 0; q < n_models; q++) {
                    if (ctx->slots[models[q]].dev.type == IDN_MODEL_ACID) continue;
                    rl.base = base + a * n_models + q;
                    rl.count = cnt + a * n_models + q;
                    IDN_LAUNCH_LIST(static_pair_index(ctx, models[a], models[q]), decode_lane_list_kernel, lgrid, st, da, ctx->slots[models[a]].dev,
                                    ctx->slots[models[q]].dev, rl)
                    LAUNCHED("decode_lane");
                }
            }
        } else {
            decode_lane_kernel<false, DynSpecs><<<grid, 128, 0, st>>>(da, ctx->d_models_host0, ctx->d_models_host0);
            LAUNCHED("decode_lane");
        }
        if (block_crc) {
            // blocks that cut reads into pieces: the per-read CRC partials come from a pass over the decoded symbols (a no-op otherwise)
            int32_t rc = launch_crc_read(ctx, acids_out, quals_out, roff, nullptr, nullptr, 0, bc.reads + n_blocks, dsp->status, out_reads_cap,
                                         out_reads_cap ? out_symbols_cap / out_reads_cap : 0, st, &dsp->native_split);
            if (rc) return rc;
        }
    }
    if (block_crc && out_reads_cap) {
        crc_verify_kernel<<<n_blocks, 256, 0, st>>>(ctx->w_crcpart.as<uint32_t>(), ctx->w_crclen.as<unsigned long long>(),
                                                    block_first, n_blocks, ctx->d_xpow, block_crc, dsp->status);
        LAUNCHED("crc_verify");
    }
    finish_decode_kernel<<<1, 32, 0, st>>>(dsp->status, &dsp->err, bc.reads + n_blocks, bc.syms + n_blocks,
                                           reinterpret_cast<unsigned long long*>(read_off_out), status_dev);
    LAUNCHED("finish_decode");
    return IDN_OK;
}

extern "C" int32_t idn_gpu_decompress_blocks_dev(idn_gpu_ctx* ctx, const uint8_t* blocks, const uint64_t* block_off,
                                                 const uint32_t* block_len, const uint32_t* block_crc, uint32_t n_blocks, uint64_t blocks_bytes,
                                                 int32_t mode, const idn_model_t* models, uint32_t n_models,
                                                 uint8_t* acids_out, uint8_t* quals_out, uint64_t* read_off_out,
                                                 uint64_t out_reads_cap, uint64_t out_symbols_cap, int32_t* status_dev,
                                                 void* stream) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_models(ctx, models, n_models);
    if (rc) return rc;
    if (mode != IDN_MODE_COMPAT && mode != IDN_MODE_NATIVE) return fail(ctx, IDN_E_UNSUPPORTED, "unknown mode %d", mode);
    if (!block_off || !status_dev || (!blocks && blocks_bytes)) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    if (out_reads_cap >= (1ull << 32) - 2) return fail(ctx, IDN_E_INVALID_ARG, "out_reads_cap too large");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = as_stream(stream);
    PROF_BEGIN();
    SmallParams sp;
    fill_decode_params(ctx, &sp, models, n_models);
    rc = upload_small(ctx, sp, st);
    if (rc) return rc;
    SmallParams* dsp = ctx->w_small.as<SmallParams>();
    const unsigned long long* boff = reinterpret_cast<const unsigned long long*>(block_off);
    if (mode == IDN_MODE_NATIVE && n_blocks)
        return decompress_native_dev(ctx, blocks, boff, block_len, block_crc, n_blocks, blocks_bytes, models, n_models, acids_out,
                                     quals_out, read_off_out, out_reads_cap, out_symbols_cap, status_dev, dsp, st);
    if (n_blocks) {
        rc = index_walk(ctx, blocks, boff, block_len, n_blocks, blocks_bytes, dsp, n_models, st);
        if (rc) return rc;
    } else {
        CU(ctx->w_blk.ensure(2 * 8 * 3));
        CU(cudaMemsetAsync(ctx->w_blk.p, 0, 2 * 8 * 3, st));
        CU(ctx->w_index.ensure(index_bytes(1)));
    }
    BlockCounters bc = carve_counters(ctx->w_blk.p, n_blocks);
    ReadIndexDev ix = carve_index(ctx->w_index.p, blocks_bytes / 17 + n_blocks + 1);
    CU(ctx->w_readblock.ensure(((size_t)n_blocks + 2) * 4));
    uint32_t* block_first = ctx->w_readblock.as<uint32_t>();
    unsigned long long* roff = reinterpret_cast<unsigned long long*>(read_off_out);
    if (!roff) {  // the CRC kernels need the per-read symbol offsets even when the caller does not
        CU(ctx->w_sliceoff.ensure((out_reads_cap + 2) * 8));
        roff = ctx->w_sliceoff.as<unsigned long long>();
    }
    // capacity check on the device; on failure the later kernels are no-ops
    index_check_kernel<<<(n_blocks + 1 + 255) / 256, 256, 0, st>>>(bc.reads, bc.syms, n_blocks, out_reads_cap, out_symbols_cap,
                                                                 block_first, dsp->status);
    LAUNCHED("index_check");
    DecodeArgs da;
    da.models = ctx->d_models;
    da.model_ids = dsp->model_ids;
    da.payload = blocks;
    da.ix = ix;
    da.blk_read_base = bc.reads;
    da.blk_sym_base = bc.syms;
    da.slot_base = bc.slots;
    da.n_blocks = n_blocks;
    da.n_reads = 0;
    da.status = dsp->status;
    da.acids_out = acids_out;
    da.quals_out = quals_out;
    da.out_dq = (long long)(quals_out - acids_out);
    da.read_off_out = roff;
    da.read_status = nullptr;
    da.err = &dsp->err;
    da.part_crc = nullptr;
    da.part_len = nullptr;
    da.crc_tab = da.xpow = nullptr;
    const bool want_crc = block_crc && n_blocks && out_reads_cap;
    if (want_crc) {  // the decoder leaves the per-read CRC partials for crc_verify_kernel
        CU(ctx->w_crcpart.ensure((out_reads_cap + 1) * 4));
        CU(ctx->w_crclen.ensure((out_reads_cap + 1) * 8));
        da.part_crc = ctx->w_crcpart.as<uint32_t>();
        da.part_len = ctx->w_crclen.as<unsigned long long>();
        da.crc_tab = ctx->d_crc_tab;
        da.xpow = ctx->d_xpow;
    }
    if (out_reads_cap && n_blocks) {
        // one acid + one q-score model: every read uses that pair (the walk rejects anything else)
        int ua = -1, uq = -1, na = 0, nq = 0;
        for (uint32_t i = 0; i < n_models; i++) {
            if (ctx->slots[models[i]].dev.type == IDN_MODEL_ACID) { ua = models[i]; na++; } else { uq = models[i]; nq++; }
        }
        const unsigned grid = (unsigned)((out_reads_cap + 127) / 128);
        if (na == 1 && nq == 1) {
            IDN_LAUNCH_UNIFORM(static_pair_index(ctx, ua, uq), decode_kernel, grid, st, da, ctx->slots[ua].dev, ctx->slots[uq].dev)
            LAUNCHED("decode");
        } else if (ctx->bucket_pairs && n_models * n_models <= kMaxPairs && out_reads_cap < 0xffffffffull) {
            // reads bucketed by the model pair the walk recorded; one launch of the uniform kernel per (acid, q-score) pair
            const uint32_t n_pairs = n_models * n_models;
            CU(ctx->w_bucket.ensure(3 * kMaxPairs * 4));
            CU(ctx->w_list.ensure(out_reads_cap * 4 + 16));
            uint32_t* cnt = ctx->w_bucket.as<uint32_t>();
            uint32_t *base = cnt + kMaxPairs, *cursor = cnt + 2 * kMaxPairs;
            CU(cudaMemsetAsync(cnt, 0, kMaxPairs * 4, st));
            const DecodePairKey key{da, n_models};
            const unsigned bgrid = (unsigned)((out_reads_cap + 255) / 256);
            bucket_count_kernel<<<bgrid, 256, 0, st>>>(key, out_reads_cap, n_pairs, cnt);
            LAUNCHED("bucket_count");
            bucket_base_kernel<<<1, 32, 0, st>>>(cnt, n_pairs, base, cursor);
            LAUNCHED("bucket_base");
            bucket_scatter_kernel<<<bgrid, 256, 0, st>>>(key, out_reads_cap, n_pairs, cursor, ctx->w_list.as<uint32_t>());
            LAUNCHED("bucket_scatter");
            ReadList rl{ctx->w_list.as<uint32_t>(), nullptr, nullptr};
            const unsigned lgrid = (unsigned)std::min<uint64_t>(grid, (uint64_t)ctx->sm_count * IDN_DEC_MINB);
            for (uint32_t a = 0; a < n_models; a++) {
                if (ctx->slots[models[a]].dev.type != IDN_MODEL_ACID) continue;
                for (uint32_t q = 0; q < n_models; q++) {
                    if (ctx->slots[models[q]].dev.type == IDN_MODEL_ACID) continue;
                    rl.base = base + a * n_models + q;
                    rl.count = cnt + a * n_models + q;
                    IDN_LAUNCH_LIST(static_pair_index(ctx, models[a], models[q]), decode_list_kernel, lgrid, st, da, ctx->slots[models[a]].dev,
                                    ctx->slots[models[q]].dev, rl)
                    LAUNCHED("decode");
                }
            }
        } else {
            decode_kernel<false, DynSpecs><<<grid, 128, 0, st>>>(da, ctx->d_models_host0, ctx->d_models_host0);
            LAUNCHED("decode");
        }
    }
    // CRC of the decoded symbols per block, compared with the header value (decompressor_block.rs:131-144)
    if (want_crc) {
        crc_verify_kernel<<<n_blocks, 256, 0, st>>>(ctx->w_crcpart.as<uint32_t>(), ctx->w_crclen.as<unsigned long long>(),
                                                    block_first, n_blocks, ctx->d_xpow, block_crc, dsp->status);
        LAUNCHED("crc_verify");
    }
    finish_decode_kernel<<<1, 32, 0, st>>>(dsp->status, &dsp->err, bc.reads + n_blocks, bc.syms + n_blocks,
                                           reinterpret_cast<unsigned long long*>(read_off_out), status_dev);
    LAUNCHED("finish_decode");
    return IDN_OK;
}

// block b = blocks[block_off[b] .. block_off[b] + len_b), len_b = block_len ? block_len[b] : block_off[b+1] - block_off[b];
// block_off[n_blocks] = size of the `blocks` region.  With block_len the region may hold other bytes between
// blocks (e.g. the 8-byte block headers of a container chunk copied as is).
static int32_t check_block_table(idn_gpu_ctx* ctx, const uint64_t* block_off, const uint32_t* block_len, uint32_t n_blocks) {
    for (uint32_t i = 0; i < n_blocks; i++) {
        if (block_off[i + 1] < block_off[i]) return fail(ctx, IDN_E_INVALID_ARG, "block_off is not monotone");
        if (block_len && block_off[i] + block_len[i] > block_off[n_blocks])
            return fail(ctx, IDN_E_SERIALIZE, "block %u runs past the end of the input", i);
        // blocks must be disjoint: the per-read index is sized from the bytes of the region (index_walk)
        if (block_len && i + 1 < n_blocks && block_off[i] + block_len[i] > block_off[i + 1])
            return fail(ctx, IDN_E_INVALID_ARG, "block %u overlaps block %u", i, i + 1);
    }
    return IDN_OK;
}

static int32_t status_to_error(idn_gpu_ctx* ctx, const int32_t st[4]) {
    switch (st[0]) {
        case IDN_OK: return IDN_OK;
        case IDN_E_SERIALIZE: return fail(ctx, st[0], "malformed slice in block %d", st[1]);
        case IDN_E_INVALID_MODEL_INDEX: return fail(ctx, st[0], "SwitchModel index out of range in block %d", st[1]);
        case IDN_E_NO_ACTIVE_MODEL: return fail(ctx, st[0], "sequence slice before any SwitchModel in block %d", st[1]);
        case IDN_E_CHECKSUM: return fail(ctx, st[0], "checksum mismatch in block %d", st[1]);
        case IDN_E_NOSPACE: return fail(ctx, st[0], "output capacity too small (%d reads needed)", st[2]);
        case IDN_E_INVALID_ARG: return fail(ctx, st[0], "the blocks of the table overlap");
        default: return fail(ctx, st[0], "decode failed with status %d in block %d", st[0], st[1]);
    }
}

extern "C" int32_t idn_gpu_index_blocks(idn_gpu_ctx* ctx, const uint8_t* blocks, const uint64_t* block_off,
                                        const uint32_t* block_len, uint32_t n_blocks, int32_t mode, const idn_model_t* models, uint32_t n_models, idn_block_index_totals* totals,
                                        uint32_t* block_first_read) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_models(ctx, models, n_models);
    if (rc) return rc;
    if (!totals || !block_off) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    totals->n_reads = totals->n_symbols = 0;
    if (block_first_read) block_first_read[0] = 0;
    if (n_blocks == 0) return IDN_OK;
    int32_t rc0 = check_block_table(ctx, block_off, block_len, n_blocks);
    if (rc0) return rc0;
    if (!blocks && block_off[n_blocks]) return fail(ctx, IDN_E_INVALID_ARG, "blocks is NULL");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    uint64_t nbytes = block_off[n_blocks];
    CU(ctx->s_blocks.ensure(nbytes + 16));
    CU(ctx->s_blockoff.ensure(((size_t)n_blocks + 1) * 8));
    CU(ctx->s_blocklen.ensure(((size_t)n_blocks + 1) * 4));
    ctx->resident_blocks = 0;
    if (nbytes) CU(cudaMemcpyAsync(ctx->s_blocks.p, blocks, nbytes, cudaMemcpyHostToDevice, st));
    ctx->resident_bytes = nbytes;
    ctx->resident_blocks = n_blocks;
    CU(cudaMemcpyAsync(ctx->s_blockoff.p, block_off, ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, st));
    if (block_len) CU(cudaMemcpyAsync(ctx->s_blocklen.p, block_len, (size_t)n_blocks * 4, cudaMemcpyHostToDevice, st));
    SmallParams sp;
    fill_decode_params(ctx, &sp, models, n_models);
    rc = upload_small(ctx, sp, st);
    if (rc) return rc;
    SmallParams* dsp = ctx->w_small.as<SmallParams>();
    if (mode == IDN_MODE_NATIVE) {
        CU(ctx->w_blk.ensure(((size_t)n_blocks + 2) * 8 * 3));
        BlockCounters nbc = carve_counters(ctx->w_blk.p, n_blocks);
        CU(ctx->w_nhdr.ensure(((size_t)n_blocks + 1) * sizeof(NativeBlockHdr)));
        native_hdr_kernel<<<n_blocks, 32, 0, st>>>(ctx->s_blocks.as<uint8_t>(), ctx->s_blockoff.as<unsigned long long>(),
                                                   block_len ? ctx->s_blocklen.as<uint32_t>() : nullptr, n_blocks, nbytes, n_models,
                                                   dsp->model_type, ctx->w_nhdr.as<NativeBlockHdr>(), nbc.reads, nbc.syms,
                                                   nbc.slots, dsp->status, &dsp->native_split);
        LAUNCHED("native_hdr");
        scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(nbc.reads, n_blocks);
        LAUNCHED("scan_tiles");
        scan_tiles_kernel<<<1, kScanBlock, 0, st>>>(nbc.syms, n_blocks);
        LAUNCHED("scan_tiles");
    } else if (mode == IDN_MODE_COMPAT) {
        rc = index_walk(ctx, ctx->s_blocks.as<uint8_t>(), ctx->s_blockoff.as<unsigned long long>(),
                        block_len ? ctx->s_blocklen.as<uint32_t>() : nullptr, n_blocks, nbytes, dsp, n_models, st);
        if (rc) return rc;
    } else {
        return fail(ctx, IDN_E_UNSUPPORTED, "unknown mode %d", mode);
    }
    std::vector<unsigned long long> hr(n_blocks + 1), hsym(n_blocks + 1);
    int32_t hst[4];
    BlockCounters bc = carve_counters(ctx->w_blk.p, n_blocks);
    CU(cudaMemcpyAsync(hr.data(), bc.reads, ((size_t)n_blocks + 1) * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hsym.data(), bc.syms, ((size_t)n_blocks + 1) * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hst, dsp->status, sizeof hst, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    if (hst[0]) return status_to_error(ctx, hst);
    totals->n_reads = hr[n_blocks];
    totals->n_symbols = hsym[n_blocks];
    if (block_first_read)
        for (uint32_t i = 0; i <= n_blocks; i++) block_first_read[i] = (uint32_t)hr[i];
    return IDN_OK;
}

#include "idn_pipeline.inc"

// The unpipelined decode of a call: container bytes and tables to the device, the *_dev path into the staging buffers
// s_aout / s_qout / s_offout (the results STAY on the device), the block CRCs checked -- with the identifiers when the
// caller passes them (sequence.rs:381-394; they are left staged in s_names / s_nameoff).
static int32_t decompress_to_staging(idn_gpu_ctx* ctx, const uint8_t* blocks, const uint64_t* block_off, const uint32_t* block_len,
                                     const uint32_t* block_crc, uint32_t n_blocks, int32_t mode, const idn_model_t* models,
                                     uint32_t n_models, const uint8_t* names, const uint64_t* name_off, uint64_t out_reads_cap,
                                     uint64_t out_symbols_cap, uint64_t* R_out, uint64_t* S_out, int32_t* bad_block, bool ids = false) {
    if (!ctx) return IDN_E_INVALID_ARG;
    if (bad_block) *bad_block = -1;
    if (!block_off) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    if ((names != nullptr) != (name_off != nullptr)) return fail(ctx, IDN_E_INVALID_ARG, "names and name_off go together");
    // ids: the names idn_gpu_inflate_names left on the device (i_names / i_nameoff) instead of host ones
    if (ids && (!ctx->names_valid || ctx->names_blocks != n_blocks))
        return fail(ctx, IDN_E_INVALID_ARG, "no idn_gpu_inflate_names call of these blocks precedes this call");
    int32_t rc0 = check_block_table(ctx, block_off, block_len, n_blocks);
    if (rc0) return rc0;
    const uint64_t nbytes = n_blocks ? block_off[n_blocks] : 0;
    // blocks == NULL: the container bytes the last idn_gpu_index_blocks call on this context uploaded (same table)
    const bool resident = !blocks && nbytes && ctx->resident_blocks == n_blocks && ctx->resident_bytes == nbytes;
    if (!blocks && nbytes && !resident) return fail(ctx, IDN_E_INVALID_ARG, "blocks is NULL and the context holds no indexed blocks of this table");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (!resident) {
        ctx->resident_blocks = 0;
        CU(ctx->s_blocks.ensure(nbytes + 16));
    }
    CU(ctx->s_blockoff.ensure(((size_t)n_blocks + 1) * 8));
    CU(ctx->s_crc.ensure(((size_t)n_blocks + 1) * 4));
    CU(ctx->s_aout.ensure(out_symbols_cap + 16));
    CU(ctx->s_qout.ensure(out_symbols_cap + 16));
    CU(ctx->s_offout.ensure((out_reads_cap + 1) * 8));
    CU(ctx->s_status.ensure(64));
    HostTimer ht(ctx);
    if (nbytes && !resident) CU(cudaMemcpyAsync(ctx->s_blocks.p, blocks, nbytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->s_blockoff.p, block_off, ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, st));
    CU(ctx->s_blocklen.ensure(((size_t)n_blocks + 1) * 4));
    if (block_len && n_blocks) CU(cudaMemcpyAsync(ctx->s_blocklen.p, block_len, (size_t)n_blocks * 4, cudaMemcpyHostToDevice, st));
    // names join the block CRC (sequence.rs:381-394): when given, the device verifies symbols only and the name bytes are
    // folded in on the host below; otherwise the device compares against the header directly.
    const bool host_crc = names != nullptr || (ids && ctx->names_any);
    if (block_crc && !host_crc && n_blocks)
        CU(cudaMemcpyAsync(ctx->s_crc.p, block_crc, (size_t)n_blocks * 4, cudaMemcpyHostToDevice, st));
    int32_t rc = idn_gpu_decompress_blocks_dev(ctx, ctx->s_blocks.as<uint8_t>(), ctx->s_blockoff.as<uint64_t>(),
                                               block_len ? ctx->s_blocklen.as<uint32_t>() : nullptr, (block_crc && !host_crc) ? ctx->s_crc.as<uint32_t>() : nullptr, n_blocks, nbytes,
                                               mode, models, n_models, ctx->s_aout.as<uint8_t>(), ctx->s_qout.as<uint8_t>(),
                                               ctx->s_offout.as<uint64_t>(), out_reads_cap, out_symbols_cap,
                                               ctx->s_status.as<int32_t>(), st);
    if (rc) return rc;
    int32_t hst[4];
    unsigned long long tot[2];
    CU(cudaMemcpyAsync(hst, ctx->s_status.p, sizeof hst, cudaMemcpyDeviceToHost, st));
    BlockCounters bc = carve_counters(ctx->w_blk.p, n_blocks);
    CU(cudaMemcpyAsync(&tot[0], bc.reads + n_blocks, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&tot[1], bc.syms + n_blocks, 8, cudaMemcpyDeviceToHost, st));
    ht.lap("host:d_enqueue");
    CU(sync_stream(ctx, st));
    ht.lap("host:d_wait_h2d_kernels");
    if (hst[0]) {
        if (bad_block) *bad_block = hst[1];
        return status_to_error(ctx, hst);
    }
    const uint64_t R = tot[0], S = tot[1];
    *R_out = R;
    *S_out = S;
    if (ids && R != ctx->names_reads)
        return fail(ctx, IDN_E_INVALID_ARG, "the blocks hold %llu reads, the inflated names %llu", (unsigned long long)R,
                    (unsigned long long)ctx->names_reads);
    if (host_crc && n_blocks) {
        // CRC with names on the device: stage names and run the CRC kernels over the decoded batch
        idn_batch d;
        memset(&d, 0, sizeof d);
        d.n_reads = R;
        d.n_symbols = S;
        d.n_blocks = n_blocks;
        d.acids = ctx->s_aout.as<uint8_t>();
        d.quals = ctx->s_qout.as<uint8_t>();
        d.read_off = ctx->s_offout.as<uint64_t>();
        d.block_first_read = ctx->w_readblock.as<uint32_t>();
        if (ids) {
            d.names = ctx->i_names.as<uint8_t>();
            d.name_off = ctx->i_nameoff.as<uint64_t>();
        } else {
            uint64_t nb = R ? name_off[R] : 0;
            CU(ctx->s_names.ensure(nb + 16));
            CU(ctx->s_nameoff.ensure((R + 1) * 8));
            if (nb) CU(cudaMemcpyAsync(ctx->s_names.p, names, nb, cudaMemcpyHostToDevice, st));
            CU(cudaMemcpyAsync(ctx->s_nameoff.p, name_off, (R + 1) * 8, cudaMemcpyHostToDevice, st));
            d.names = ctx->s_names.as<uint8_t>();
            d.name_off = ctx->s_nameoff.as<uint64_t>();
        }
        if (!block_crc) {
            CU(sync_stream(ctx, st));
            return IDN_OK;
        }
        rc = idn_gpu_block_crc_dev_impl(ctx, &d, ctx->s_crc.as<uint32_t>(), nullptr, nullptr, 0, st);
        if (rc) return rc;
        std::vector<uint32_t> got(n_blocks);
        CU(cudaMemcpyAsync(got.data(), ctx->s_crc.p, (size_t)n_blocks * 4, cudaMemcpyDeviceToHost, st));
        CU(sync_stream(ctx, st));
        for (uint32_t i = 0; i < n_blocks; i++)
            if (got[i] != block_crc[i]) {
                if (bad_block) *bad_block = (int32_t)i;
                return fail(ctx, IDN_E_CHECKSUM, "checksum mismatch in block %u", i);
            }
    }
    return IDN_OK;
}



extern "C" int32_t idn_gpu_set_pipeline_blocks(idn_gpu_ctx* ctx, uint32_t blocks) {
    if (!ctx) return IDN_E_INVALID_ARG;
    if (blocks == 0) return fail(ctx, IDN_E_INVALID_ARG, "blocks per sub-chunk must be positive");
    ctx->pipe_blocks = blocks;
    ctx->pipe_blocks_set = true;
    return IDN_OK;
}

static int32_t decompress_blocks_staged(idn_gpu_ctx* ctx, const uint8_t* blocks, const uint64_t* block_off, const uint32_t* block_len,
                                        const uint32_t* block_crc, uint32_t n_blocks, int32_t mode, const idn_model_t* models,
                                        uint32_t n_models, const uint8_t* names, const uint64_t* name_off, uint8_t* acids_out,
                                        uint8_t* quals_out, uint64_t* read_off_out, uint64_t out_reads_cap, uint64_t out_symbols_cap,
                                        int32_t* bad_block, bool ids);

extern "C" int32_t idn_gpu_decompress_blocks(idn_gpu_ctx* ctx, const uint8_t* blocks, const uint64_t* block_off,
                                             const uint32_t* block_len, const uint32_t* block_crc, uint32_t n_blocks, int32_t mode,
                                             const idn_model_t* models, uint32_t n_models, const uint8_t* names,
                                             const uint64_t* name_off, uint8_t* acids_out, uint8_t* quals_out,
                                             uint64_t* read_off_out, uint64_t out_reads_cap, uint64_t out_symbols_cap,
                                             int32_t* bad_block) {
    if (!ctx) return IDN_E_INVALID_ARG;
    if (bad_block) *bad_block = -1;
    if (!block_off || !read_off_out) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    if ((names != nullptr) != (name_off != nullptr)) return fail(ctx, IDN_E_INVALID_ARG, "names and name_off go together");
    if (out_symbols_cap && (!acids_out || !quals_out)) return fail(ctx, IDN_E_INVALID_ARG, "NULL output");
    int32_t rc0 = check_block_table(ctx, block_off, block_len, n_blocks);
    if (rc0) return rc0;
    CU(cudaSetDevice(ctx->device));
    if (!names && n_blocks && blocks) {
        // no names on the device (the block CRCs cover the symbols only): sub-chunks of whole blocks flow through upload /
        // kernels / download streams; a sub-chunk that outgrows its share of the staging sends the call down the path below
        int32_t rcm = check_models(ctx, models, n_models);
        if (rcm) return rcm;
        if (mode != IDN_MODE_COMPAT && mode != IDN_MODE_NATIVE) return fail(ctx, IDN_E_UNSUPPORTED, "unknown mode %d", mode);
        bool retry_simple = false;
        int32_t rcp = decompress_blocks_pipelined(ctx, blocks, block_off, block_len, block_crc, n_blocks, mode, models, n_models, acids_out,
                                                  quals_out, read_off_out, out_reads_cap, out_symbols_cap, bad_block, &retry_simple);
        if (rcp || !retry_simple) return rcp;
    }
    return decompress_blocks_staged(ctx, blocks, block_off, block_len, block_crc, n_blocks, mode, models, n_models, names, name_off, acids_out,
                                    quals_out, read_off_out, out_reads_cap, out_symbols_cap, bad_block, false);
}

// the unpipelined decode of idn_gpu_decompress_blocks(_ids) with its results copied to the caller's buffers
static int32_t decompress_blocks_staged(idn_gpu_ctx* ctx, const uint8_t* blocks, const uint64_t* block_off, const uint32_t* block_len,
                                        const uint32_t* block_crc, uint32_t n_blocks, int32_t mode, const idn_model_t* models,
                                        uint32_t n_models, const uint8_t* names, const uint64_t* name_off, uint8_t* acids_out,
                                        uint8_t* quals_out, uint64_t* read_off_out, uint64_t out_reads_cap, uint64_t out_symbols_cap,
                                        int32_t* bad_block, bool ids) {
    cudaStream_t st = ctx->stream;
    uint64_t R = 0, S = 0;
    int32_t rc = decompress_to_staging(ctx, blocks, block_off, block_len, block_crc, n_blocks, mode, models, n_models, names, name_off,
                                       out_reads_cap, out_symbols_cap, &R, &S, bad_block, ids);
    if (rc) return rc;
    if (S) {
        CU(cudaMemcpyAsync(acids_out, ctx->s_aout.p, S, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(quals_out, ctx->s_qout.p, S, cudaMemcpyDeviceToHost, st));
    }
    CU(cudaMemcpyAsync(read_off_out, ctx->s_offout.p, (R + 1) * 8, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    return IDN_OK;
}

extern "C" int32_t idn_gpu_decompress_reads(idn_gpu_ctx* ctx, const uint8_t* payload, uint64_t payload_bytes,
                                            const idn_read_index* index, const idn_model_t* models, uint32_t n_models,
                                            uint8_t* acids_out, uint8_t* quals_out, uint32_t* read_status) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_models(ctx, models, n_models);
    if (rc) return rc;
    if (!index) return fail(ctx, IDN_E_INVALID_ARG, "index is NULL");
    const uint64_t R = index->n_reads;
    if (R == 0) return IDN_OK;
    if (!index->pay_off || !index->pay_len || !index->seq_len || !index->out_off || !index->acid_model || !index->q_model)
        return fail(ctx, IDN_E_INVALID_ARG, "NULL index array");
    if (!payload && payload_bytes) return fail(ctx, IDN_E_INVALID_ARG, "payload is NULL");
    uint64_t S = 0;
    for (uint64_t r = 0; r < R; r++) {
        // (not pay_off + pay_len > payload_bytes: that sum wraps for an offset near 2^64)
        if (index->pay_len[r] > payload_bytes || index->pay_off[r] > payload_bytes - index->pay_len[r]) return fail(ctx, IDN_E_SERIALIZE, "read %llu payload out of range", (unsigned long long)r);
        if (index->out_off[r] != S) return fail(ctx, IDN_E_INVALID_ARG, "out_off is not the exclusive scan of seq_len");
        S += index->seq_len[r];
        if (index->acid_model[r] >= n_models || index->q_model[r] >= n_models)
            return fail(ctx, IDN_E_INVALID_MODEL_INDEX, "read %llu names model index out of range", (unsigned long long)r);
        if (ctx->slots[models[index->acid_model[r]]].dev.type != IDN_MODEL_ACID ||
            ctx->slots[models[index->q_model[r]]].dev.type != IDN_MODEL_QSCORE)
            return fail(ctx, IDN_E_INVALID_MODEL_INDEX, "read %llu names a model of the wrong type", (unsigned long long)r);
    }
    if (index->out_off[R] != S) return fail(ctx, IDN_E_INVALID_ARG, "out_off[n_reads] != sum of seq_len");
    if (S && (!acids_out || !quals_out)) return fail(ctx, IDN_E_INVALID_ARG, "NULL output");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    SmallParams sp;
    memset(&sp, 0, sizeof sp);
    for (uint32_t i = 0; i < n_models; i++) sp.model_ids[i] = models[i];
    rc = upload_small(ctx, sp, st);
    if (rc) return rc;
    SmallParams* dsp = ctx->w_small.as<SmallParams>();
    ctx->resident_blocks = 0;
    CU(ctx->s_blocks.ensure(payload_bytes + 16));
    CU(ctx->w_index.ensure(index_bytes(R)));
    CU(ctx->s_aout.ensure(S + 16));
    CU(ctx->s_qout.ensure(S + 16));
    CU(ctx->s_idx.ensure((R + 1) * 4));
    ReadIndexDev ix = carve_index(ctx->w_index.p, R);
    if (payload_bytes) CU(cudaMemcpyAsync(ctx->s_blocks.p, payload, payload_bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ix.pay_off, index->pay_off, R * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ix.sym_off, index->out_off, (R + 1) * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ix.pay_len, index->pay_len, R * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ix.seq_len, index->seq_len, R * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ix.am, index->acid_model, R, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ix.qm, index->q_model, R, cudaMemcpyHostToDevice, st));
    DecodeArgs da;
    da.models = ctx->d_models;
    da.model_ids = dsp->model_ids;
    da.payload = ctx->s_blocks.as<uint8_t>();
    da.ix = ix;
    da.blk_read_base = nullptr;
    da.blk_sym_base = nullptr;
    da.slot_base = nullptr;
    da.n_blocks = 0;
    da.n_reads = R;
    da.status = nullptr;
    da.acids_out = ctx->s_aout.as<uint8_t>();
    da.quals_out = ctx->s_qout.as<uint8_t>();
    da.out_dq = (long long)(da.quals_out - da.acids_out);
    da.read_off_out = nullptr;
    da.read_status = ctx->s_idx.as<uint32_t>();
    da.err = &dsp->err;
    da.part_crc = nullptr;
    da.part_len = nullptr;
    da.crc_tab = da.xpow = nullptr;
    decode_kernel<false, DynSpecs><<<(unsigned)((R + 127) / 128), 128, 0, st>>>(da, ctx->d_models_host0, ctx->d_models_host0);
    LAUNCHED("decode");
    uint32_t err = 0;
    if (S) {
        CU(cudaMemcpyAsync(acids_out, ctx->s_aout.p, S, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(quals_out, ctx->s_qout.p, S, cudaMemcpyDeviceToHost, st));
    }
    if (read_status) CU(cudaMemcpyAsync(read_status, ctx->s_idx.p, R * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&err, &dsp->err, 4, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    if (err & 1) return fail(ctx, IDN_E_SERIALIZE, "a sequence payload ended before its symbols were decoded");
    return IDN_OK;
}

// ======================================================================================================
// workload generator (bench/test utility)
// ======================================================================================================
extern "C" int32_t idn_gpu_synth_reads_dev(idn_gpu_ctx* ctx, idn_model_t acid_model, idn_model_t q_model,
                                           const uint64_t* read_off, uint64_t n_reads, uint64_t first_read_index,
                                           uint64_t seed, uint32_t n_ppm, uint8_t* acids, uint8_t* quals, void* stream) {
    if (!ctx) return IDN_E_INVALID_ARG;
    idn_model_t pair[2] = {acid_model, q_model};
    int32_t rc = check_models(ctx, pair, 2);
    if (rc) return rc;
    if (ctx->slots[acid_model].dev.type != IDN_MODEL_ACID || ctx->slots[q_model].dev.type != IDN_MODEL_QSCORE)
        return fail(ctx, IDN_E_INVALID_ARG, "need an acid model and a quality score model, in that order");
    if (n_reads == 0) return IDN_OK;
    if (!read_off || !acids || !quals) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = as_stream(stream);
    PROF_BEGIN();
    synth_kernel<<<(unsigned)((n_reads + 127) / 128), 128, 0, st>>>(
        ctx->d_models, acid_model, q_model, reinterpret_cast<const unsigned long long*>(read_off), n_reads, first_read_index,
        seed, n_ppm, acids, quals);
    LAUNCHED("synth");
    return IDN_OK;
}

// ======================================================================================================
// per-kernel timing
// ======================================================================================================
extern "C" int32_t idn_gpu_profile(idn_gpu_ctx* ctx, int32_t enable) {
    if (!ctx) return IDN_E_INVALID_ARG;
    ctx->profiling = enable != 0;
    ctx->prof_marks.clear();
    ctx->prof_used = 0;
    return IDN_OK;
}

extern "C" int32_t idn_gpu_profile_read(idn_gpu_ctx* ctx, char* buf, uint64_t cap) {
    if (!ctx || !buf || cap == 0) return IDN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    struct Acc {
        const char* name;
        uint64_t n;
        double ms;
    };
    std::vector<Acc> acc;
    for (size_t i = 1; i < ctx->prof_marks.size(); i++) {
        const auto& m = ctx->prof_marks[i];
        if (!m.name) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->prof_marks[i - 1].ev, m.ev) != cudaSuccess) {
            (void)cudaGetLastError();
            continue;
        }
        size_t k = 0;
        while (k < acc.size() && strcmp(acc[k].name, m.name) != 0) k++;
        if (k == acc.size()) acc.push_back({m.name, 0, 0.0});
        acc[k].n++;
        acc[k].ms += ms;
    }
    std::string out;
    char line[160];
    for (auto& a : acc) {
        snprintf(line, sizeof line, "%s %llu %.6f\n", a.name, (unsigned long long)a.n, a.ms);
        out += line;
    }
    for (auto& hph : ctx->host_phases) {
        snprintf(line, sizeof line, "%s %llu %.6f\n", hph.name, (unsigned long long)hph.n, hph.ms);
        out += line;
    }
    ctx->host_phases.clear();
    ctx->prof_marks.clear();
    ctx->prof_used = 0;
    if (out.size() + 1 > cap) return fail(ctx, IDN_E_NOSPACE, "profile text needs %zu bytes", out.size() + 1);
    memcpy(buf, out.c_str(), out.size() + 1);
    return IDN_OK;
}

// ======================================================================================================
// FASTQ text <-> symbol arrays on the device (SURVEY.md section 8f, row f1)
// ======================================================================================================
static const char* fastq_err_name(uint32_t e) {
    switch (e) {
        case kFqInvalidFormat: return "invalid format (title without '@' or separator line without '+')";
        case kFqInvalidAcid: return "invalid acid";
        case kFqInvalidQualityScore: return "invalid quality score";
        case kFqLengthMismatch: return "acid and quality score lengths differ";
        case kFqEof: return "end of input inside a record";
        default: return "ok";
    }
}

// partial: the text is a chunk of a longer input that ends on a line boundary; a record cut short at its end is left to
// the next chunk (ctx->f_consumed = where it starts) instead of being an error
static int32_t fastq_parse_dev_impl(idn_gpu_ctx* ctx, const uint8_t* text, uint64_t n, idn_fastq_info* info, cudaStream_t st, bool partial) {
    if (!ctx || !info || (!text && n)) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    ctx->f_consumed = n;
    PROF_BEGIN();
    memset(info, 0, sizeof *info);
    ctx->f_info = *info;
    const uint64_t n_tiles = (n + kFqTile - 1) / kFqTile;
    CU(ctx->f_tilecnt.ensure((n_tiles + 1) * 8));
    CU(ctx->f_tilebase.ensure((n_tiles + 2) * 8));
    CU(ctx->f_err.ensure(16));
    unsigned long long* tile_cnt = ctx->f_tilecnt.as<unsigned long long>();
    unsigned long long* tile_base = ctx->f_tilebase.as<unsigned long long>();
    unsigned long long* first_err = ctx->f_err.as<unsigned long long>();
    CU(cudaMemsetAsync(first_err, 0xff, 8, st));
    uint64_t n_newlines = 0;
    uint8_t last = '\n';
    if (n) {
        fq_count_kernel<<<(unsigned)n_tiles, 256, 0, st>>>(text, n, tile_cnt);
        LAUNCHED("fq_count");
        int32_t rc = scan_u64(ctx, TileCntFn{tile_cnt}, n_tiles, tile_base, st);
        if (rc) return rc;
        CU(cudaMemcpyAsync(&n_newlines, tile_base + n_tiles, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(&last, text + n - 1, 1, cudaMemcpyDeviceToHost, st));
        CU(sync_stream(ctx, st));
    }
    const uint64_t n_lines = n_newlines + (n > 0 && last != '\n' ? 1 : 0);
    info->n_lines = n_lines;
    CU(ctx->f_linestart.ensure((n_newlines + 2) * 8));
    unsigned long long* line_start = ctx->f_linestart.as<unsigned long long>();
    uint64_t n_reads = 0;
    if (n_lines) {
        fq_scatter_kernel<<<(unsigned)n_tiles, 256, 0, st>>>(text, n, tile_base, line_start);
        LAUNCHED("fq_scatter");
        const uint64_t f_tiles = (n_lines + kFstTile - 1) / kFstTile;
        CU(ctx->f_linefn.ensure(n_lines + 16));
        CU(ctx->f_linestate.ensure(n_lines + 16));
        CU(ctx->f_tilefn.ensure(f_tiles + 16));
        CU(ctx->f_tilestate.ensure(f_tiles + 16));
        CU(ctx->f_recscan.ensure((n_lines + 2) * 8));
        uint8_t* line_fn = ctx->f_linefn.as<uint8_t>();
        uint8_t* line_state = ctx->f_linestate.as<uint8_t>();
        fst_reduce_kernel<<<(unsigned)f_tiles, 256, 0, st>>>(text, n, line_start, n_lines, n_newlines, line_fn, ctx->f_tilefn.as<uint8_t>());
        LAUNCHED("fst_reduce");
        fst_tiles_kernel<<<1, 256, 0, st>>>(ctx->f_tilefn.as<uint8_t>(), f_tiles, ctx->f_tilestate.as<uint8_t>());
        LAUNCHED("fst_tiles");
        fst_apply_kernel<<<(unsigned)f_tiles, 256, 0, st>>>(line_fn, n_lines, ctx->f_tilestate.as<uint8_t>(), line_state);
        LAUNCHED("fst_apply");
        TitleFlag tf{line_state, line_fn};
        unsigned long long* rec_scan = ctx->f_recscan.as<unsigned long long>();
        int32_t rc = scan_u64(ctx, tf, n_lines, rec_scan, st);
        if (rc) return rc;
        CU(cudaMemcpyAsync(&n_reads, rec_scan + n_lines, 8, cudaMemcpyDeviceToHost, st));
        CU(sync_stream(ctx, st));
        CU(ctx->f_title.ensure((n_reads + 1) * 8));
        if (n_reads) {
            fq_titles_kernel<<<(unsigned)((n_lines + 255) / 256), 256, 0, st>>>(tf, n_lines, rec_scan, ctx->f_title.as<unsigned long long>());
            LAUNCHED("fq_titles");
        }
        if (partial && n_reads) {  // a last record with fewer than four lines belongs to the next chunk
            if (last != '\n') return fail(ctx, IDN_E_INVALID_ARG, "a chunk of a longer FASTQ input must end on a line boundary");
            unsigned long long t_last = 0;
            CU(cudaMemcpyAsync(&t_last, ctx->f_title.as<unsigned long long>() + (n_reads - 1), 8, cudaMemcpyDeviceToHost, st));
            CU(sync_stream(ctx, st));
            if (t_last + 3 >= n_lines) {
                unsigned long long off = 0;
                CU(cudaMemcpyAsync(&off, line_start + t_last, 8, cudaMemcpyDeviceToHost, st));
                CU(sync_stream(ctx, st));
                ctx->f_consumed = off;
                n_reads--;
            }
        }
    }
    info->n_reads = n_reads;
    CU(ctx->f_namelo.ensure((n_reads + 1) * 8));
    CU(ctx->f_namelen.ensure((n_reads + 1) * 4));
    CU(ctx->f_readlen.ensure((n_reads + 1) * 4));
    CU(ctx->f_readoff.ensure((n_reads + 2) * 8));
    CU(ctx->f_nameoff.ensure((n_reads + 2) * 8));
    FastqView V{text, n, line_start, n_lines, n_newlines, ctx->f_title.as<unsigned long long>(), n_reads};
    unsigned long long* read_off = ctx->f_readoff.as<unsigned long long>();
    unsigned long long* name_off = ctx->f_nameoff.as<unsigned long long>();
    if (n_reads) {
        fq_lengths_kernel<<<(unsigned)((n_reads + 127) / 128), 128, 0, st>>>(V, ctx->f_namelo.as<unsigned long long>(),
                                                                           ctx->f_namelen.as<uint32_t>(), ctx->f_readlen.as<uint32_t>(),
                                                                           first_err);
        LAUNCHED("fq_lengths");
    }
    int32_t rc = scan_u64(ctx, U32Fn{ctx->f_readlen.as<uint32_t>()}, n_reads, read_off, st);
    if (rc) return rc;
    rc = scan_u64(ctx, U32Fn{ctx->f_namelen.as<uint32_t>()}, n_reads, name_off, st);
    if (rc) return rc;
    unsigned long long tot[2] = {0, 0}, ferr = ~0ull;
    CU(cudaMemcpyAsync(&tot[0], read_off + n_reads, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&tot[1], name_off + n_reads, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&ferr, first_err, 8, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    info->n_symbols = tot[0];
    info->n_name_bytes = tot[1];
    if (ferr == ~0ull && n_reads) {
        CU(ctx->f_names.ensure(tot[1] + 16));
        CU(ctx->f_acids.ensure(tot[0] + 16));
        CU(ctx->f_quals.ensure(tot[0] + 16));
        fq_convert_kernel<<<(unsigned)((n_reads + 127) / 128), 128, 0, st>>>(V, ctx->f_namelo.as<unsigned long long>(), name_off, read_off,
                                                                           ctx->f_names.as<uint8_t>(), ctx->f_acids.as<uint8_t>(),
                                                                           ctx->f_quals.as<uint8_t>(), first_err);
        LAUNCHED("fq_convert");
        CU(cudaMemcpyAsync(&ferr, first_err, 8, cudaMemcpyDeviceToHost, st));
        CU(sync_stream(ctx, st));
    }
    if (ferr != ~0ull) {
        info->error_kind = (int32_t)(ferr & 0xff);
        info->bad_record = ferr >> 8;
        ctx->f_info = *info;
        return fail(ctx, IDN_E_SERIALIZE, "FASTQ record %llu: %s", (unsigned long long)info->bad_record, fastq_err_name((uint32_t)(ferr & 0xff)));
    }
    ctx->f_info = *info;
    return IDN_OK;
}

extern "C" int32_t idn_gpu_fastq_parse_dev(idn_gpu_ctx* ctx, const uint8_t* text, uint64_t n, idn_fastq_info* info, void* stream) {
    return fastq_parse_dev_impl(ctx, text, n, info, as_stream(stream), false);
}

extern "C" int32_t idn_gpu_fastq_parse(idn_gpu_ctx* ctx, const uint8_t* text, uint64_t n, idn_fastq_info* info) {
    if (!ctx || !info || (!text && n)) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    CU(ctx->f_text.ensure(n + 16));
    if (n) CU(cudaMemcpyAsync(ctx->f_text.p, text, n, cudaMemcpyHostToDevice, ctx->stream));
    return idn_gpu_fastq_parse_dev(ctx, ctx->f_text.as<uint8_t>(), n, info, ctx->stream);
}

extern "C" int32_t idn_gpu_fastq_batch_dev(idn_gpu_ctx* ctx, idn_batch* out) {
    if (!ctx || !out) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    memset(out, 0, sizeof *out);
    out->n_reads = ctx->f_info.n_reads;
    out->n_symbols = ctx->f_info.n_symbols;
    out->acids = ctx->f_acids.as<uint8_t>();
    out->quals = ctx->f_quals.as<uint8_t>();
    out->read_off = ctx->f_readoff.as<uint64_t>();
    out->names = ctx->f_names.as<uint8_t>();
    out->name_off = ctx->f_nameoff.as<uint64_t>();
    return IDN_OK;
}

extern "C" int32_t idn_gpu_fastq_fetch(idn_gpu_ctx* ctx, uint8_t* acids, uint8_t* quals, uint64_t* read_off, uint8_t* names,
                                       uint64_t* name_off) {
    if (!ctx) return IDN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const idn_fastq_info& f = ctx->f_info;
    if (f.error_kind) return fail(ctx, IDN_E_INVALID_STATE, "the last parse failed");
    if (acids && f.n_symbols) CU(cudaMemcpyAsync(acids, ctx->f_acids.p, f.n_symbols, cudaMemcpyDeviceToHost, st));
    if (quals && f.n_symbols) CU(cudaMemcpyAsync(quals, ctx->f_quals.p, f.n_symbols, cudaMemcpyDeviceToHost, st));
    if (read_off) CU(cudaMemcpyAsync(read_off, ctx->f_readoff.p, (f.n_reads + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (names && f.n_name_bytes) CU(cudaMemcpyAsync(names, ctx->f_names.p, f.n_name_bytes, cudaMemcpyDeviceToHost, st));
    if (name_off) CU(cudaMemcpyAsync(name_off, ctx->f_nameoff.p, (f.n_reads + 1) * 8, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    return IDN_OK;
}

extern "C" int32_t idn_gpu_fastq_format_dev(idn_gpu_ctx* ctx, const idn_batch* batch, int32_t title_with_separator, uint8_t* text,
                                            uint64_t cap, uint64_t* n_out_dev, void* stream) {
    if (!ctx) return IDN_E_INVALID_ARG;
    int32_t rc = check_batch(ctx, batch);
    if (rc) return rc;
    if (!n_out_dev || (!text && cap)) return fail(ctx, IDN_E_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = as_stream(stream);
    PROF_BEGIN();
    const uint64_t R = batch->n_reads;
    CU(ctx->f_fmtoff.ensure((R + 2) * 8));
    CU(ctx->f_err.ensure(16));
    unsigned long long* off = ctx->f_fmtoff.as<unsigned long long>();
    FormatSize fs{batch->read_off, batch->name_off, title_with_separator};
    rc = scan_u64(ctx, fs, R, off, st);
    if (rc) return rc;
    CU(cudaMemsetAsync(ctx->f_err.p, 0, 8, st));
    if (R) {
        fq_format_kernel<<<(unsigned)((R + 127) / 128), 128, 0, st>>>(batch->acids, batch->quals, batch->read_off, batch->names,
                                                                    batch->name_off, R, title_with_separator, off, text, cap,
                                                                    ctx->f_err.as<uint32_t>());
        LAUNCHED("fq_format");
    }
    CU(cudaMemcpyAsync(n_out_dev, off + R, 8, cudaMemcpyDeviceToDevice, st));
    return IDN_OK;
}

extern "C" int32_t idn_gpu_fastq_format(idn_gpu_ctx* ctx, const idn_batch* b, int32_t title_with_separator, uint8_t* text, uint64_t cap,
                                        uint64_t* n_out) {
    if (!ctx || !n_out) return IDN_E_INVALID_ARG;
    int32_t rc = check_host_batch(ctx, b, false);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    idn_batch h = *b;
    uint32_t bf[2] = {0, (uint32_t)b->n_reads};
    h.block_first_read = bf;
    h.n_blocks = 1;
    idn_batch d;
    rc = stage_batch(ctx, &h, &d, st);
    if (rc) return rc;
    CU(ctx->f_fmttext.ensure(cap + 16));
    CU(ctx->s_stats.ensure(64));
    rc = idn_gpu_fastq_format_dev(ctx, &d, title_with_separator, ctx->f_fmttext.as<uint8_t>(), cap, ctx->s_stats.as<uint64_t>(), st);
    if (rc) return rc;
    uint64_t need = 0;
    uint32_t err = 0;
    CU(cudaMemcpyAsync(&need, ctx->s_stats.p, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&err, ctx->f_err.p, 4, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    *n_out = need;
    if (err & 1) return fail(ctx, IDN_E_INVALID_SYMBOL, "input holds an acid > 4 or a quality score > 93");
    if (need > cap) return fail(ctx, IDN_E_NOSPACE, "FASTQ text needs %llu bytes, capacity is %llu", (unsigned long long)need, (unsigned long long)cap);
    if (need) CU(cudaMemcpyAsync(text, ctx->f_fmttext.p, need, cudaMemcpyDeviceToHost, st));
    CU(sync_stream(ctx, st));
    return IDN_OK;
}

#include "idn_textpath.inc"
