// idn_kernels.cuh -- the CUDA kernels of the hot path (sm_100a).  See DESIGN.md for the launch plan.
//
//   K2  score_kernel      ModelTester::compute_size           idn/model_chooser.rs:215-243
//   K3  switch_kernel     get_best_model_for + switch_to_*    idn/model_chooser.rs:168-198, compressor_block.rs:232-280
//   K4  encode_kernel     SequenceCompressor::compress        sequence_compressor.rs:82-155, compressor.rs:83-98
//       layout/assemble   BlockWriter                         idn/writer_block.rs:27-82
//   K5  decode_kernel     SequenceDecompressor::decompress    sequence_compressor.rs:231-278, compressor.rs:173-193
//       walk_fast_kernel / walk_kernel   IdnBlockDecompressor slice walk   idn/decompressor_block.rs:115-129,194-239
//   K7  crc kernels       crc32 over name|acids|quals         writer_block.rs:64, sequence.rs:381-394
#pragma once
#include "idn_device.cuh"

namespace idn {

// ---------------------------------------------------------------------------------------------------
// byte readers / writers on 4-byte words (threads walk their read sequentially; word access keeps the
// divergent traffic at one 32-byte sector per 32 bytes instead of one per byte)
// ---------------------------------------------------------------------------------------------------
// Sequential byte readers over aligned 4-byte words: the cursor (word pointer + byte lane) moves by one byte per call and
// a word is loaded only when its first byte is asked for, so nothing outside [first byte read, last byte read] rounded
// to words is ever touched.
struct BackReader {  // bytes at decreasing addresses
    const uint32_t* wp;  // word that holds the next byte
    uint32_t word;
    int lane;            // byte of `word` the next get() returns, + 4 while that word is not loaded yet
    __device__ __forceinline__ void start(const uint8_t* last) {  // the next get() returns *last
        const uintptr_t a = reinterpret_cast<uintptr_t>(last);
        wp = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        lane = (int)(a & 3) + 4;
        word = 0;
    }
    __device__ __forceinline__ uint32_t get() {
        if (lane >= 4) {
            word = __ldg(wp);
            lane -= 4;
        }
        const uint32_t b = (word >> (8 * lane)) & 0xffu;
        if (--lane < 0) {
            lane = 7;
            wp--;
        }
        return b;
    }
};

struct FwdReader {  // bytes at increasing addresses
    const uint32_t* wp;
    uint32_t word;
    int lane;  // byte of `word` the next get() returns, - 4 while that word is not loaded yet
    __device__ __forceinline__ void start(const uint8_t* first) {  // the next get() returns *first
        const uintptr_t a = reinterpret_cast<uintptr_t>(first);
        wp = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        lane = (int)(a & 3) - 4;
        word = 0;
    }
    __device__ __forceinline__ uint32_t get() {
        if (lane < 0) {
            word = __ldg(wp);
            lane += 4;
        }
        const uint32_t b = (word >> (8 * lane)) & 0xffu;
        if (++lane == 4) {
            lane = -4;
            wp++;
        }
        return b;
    }
};

// The 16 bytes at the 16-byte aligned address c of a byte array [base, base + n): one vector load when the chunk lies
// inside the array, byte loads (zeros outside) at its two ends.
__device__ __forceinline__ uint4 load_chunk16(const uint8_t* __restrict__ base, unsigned long long n, const uint8_t* c) {
    if (c >= base && c + 16 <= base + n) return __ldg(reinterpret_cast<const uint4*>(c));
    uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 16; j++)
        if (c + j >= base && c + j < base + n) w[j >> 2] |= (uint32_t)__ldg(c + j) << (8 * (j & 3));
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// The acids and the quality scores of a read, one position per call, last position first.  Both arrays are read at the
// same offsets, so one cursor serves both; the symbols come in aligned 16-byte chunks (one vector load per stream per 16
// positions: a thread's loads are 32 scattered sectors per warp request whatever their width, and the encoder is bound by
// the number of such requests) that are consumed from the top word down.  When the two arrays disagree in their
// alignment modulo 16 the reader falls back to byte loads.
struct SymBackReader {
    const uint8_t *abase, *qbase;  // the arrays (kernel parameters: constant-bank operands, no registers)
    unsigned long long n;          // their length
    const uint8_t* c;              // acid-side address of the chunk below the one in the registers / of the next byte (slow)
    uint32_t ca, cq;               // current words, next byte in bits 24..31
    uint32_t a0, a1, a2, q0, q1, q2;  // the words of the chunk still to come: x2 next
    uint32_t left;                 // bytes of the chunk not yet returned
    bool vec;
    __device__ __forceinline__ void load() {
        const uint4 va = load_chunk16(abase, n, c), vq = load_chunk16(qbase, n, qbase + (c - abase));
        ca = va.w; a2 = va.z; a1 = va.y; a0 = va.x;
        cq = vq.w; q2 = vq.z; q1 = vq.y; q0 = vq.x;
        c -= 16;
        left = 16;
    }
    __device__ __forceinline__ void next_word() {
        ca = a2; a2 = a1; a1 = a0;
        cq = q2; q2 = q1; q1 = q0;
    }
    // the first call of get() returns position off + len - 1; nothing is loaded when len == 0
    __device__ __forceinline__ void start(const uint8_t* acids, const uint8_t* quals, unsigned long long n_symbols, long long off,
                                          uint32_t len) {
        abase = acids;
        qbase = quals;
        n = n_symbols;
        vec = ((reinterpret_cast<uintptr_t>(acids) ^ reinterpret_cast<uintptr_t>(quals)) & 15) == 0;
        ca = cq = a0 = a1 = a2 = q0 = q1 = q2 = 0;
        left = 0;
        const uint8_t* last = acids + off + (long long)len - 1;
        c = last;
        if (!vec || len == 0) return;
        const uint32_t k = (uint32_t)(reinterpret_cast<uintptr_t>(last) & 15);  // byte of its chunk the first get() returns
        c = last - k;
        load();
        for (uint32_t t = 3; t > (k >> 2); t--) next_word();  // drop the words above the one that holds byte k
        const uint32_t sh = 8 * (3 - (k & 3));
        ca <<= sh;
        cq <<= sh;
        left = k + 1;
    }
    __device__ __forceinline__ void get(uint32_t& a, uint32_t& q) {
        if (!vec) {
            a = __ldg(c);
            q = __ldg(qbase + (c - abase));
            c--;
            return;
        }
        if (left == 0) load();  // lazily: never touches a chunk that holds no byte of the read
        a = ca >> 24;
        q = cq >> 24;
        ca <<= 8;
        cq <<= 8;
        left--;
        if ((left & 3) == 0 && left != 0) next_word();
    }
    // vec only, at a word boundary ((left & 3) == 0): the next four bytes in ca / cq (first one in bits 24..31), taken
    // by the caller before it calls skip_word().  The caller guarantees that their chunk lies inside the arrays (above it
    // lies the chunk already read, so only its lower end is in question).
    __device__ __forceinline__ void peek_word() {
        if (left == 0) {
            const uint4 va = __ldg(reinterpret_cast<const uint4*>(c)), vq = __ldg(reinterpret_cast<const uint4*>(qbase + (c - abase)));
            ca = va.w; a2 = va.z; a1 = va.y; a0 = va.x;
            cq = vq.w; q2 = vq.z; q1 = vq.y; q0 = vq.x;
            c -= 16;
            left = 16;
        }
    }
    __device__ __forceinline__ void skip_word() {
        left -= 4;
        next_word();  // (when left reaches 0 the next peek_word() reloads all of them)
    }
};

// writes bytes at decreasing addresses, 4 at a time.  `end` must be 4-byte aligned.  Bytes wait in a 64-bit
// accumulator (oldest highest); drain() stores a word once four are there, so at most 7 may be pending before it.
struct BackWriter {
    uint32_t* wptr;  // next word to fill is wptr[-1]
    unsigned long long acc;
    uint32_t nbits;  // pending bytes * 8
    __device__ __forceinline__ void init(uint8_t* end) {
        wptr = reinterpret_cast<uint32_t*>(end);
        acc = 0;
        nbits = 0;
    }
    // bytes written so far, given the `end` the writer was started at (not kept: two registers across the hot loop)
    __device__ __forceinline__ uint32_t bytes(const uint8_t* end) const {
        return (uint32_t)(reinterpret_cast<const uint32_t*>(end) - wptr) * 4u + (nbits >> 3);
    }
    // appends kbits / 8 bytes given in emission order, first emitted byte highest
    __device__ __forceinline__ void push_bits(uint32_t bytes_be, uint32_t kbits) {
        acc = (acc << kbits) | bytes_be;
        nbits += kbits;
    }
    __device__ __forceinline__ void drain() {
        if (nbits >= 32) {
            nbits -= 32;
            *--wptr = (uint32_t)(acc >> nbits);  // the first byte pushed lands at the highest address
        }
    }
    __device__ __forceinline__ void push_u32_le(uint32_t x) {  // RansEncFlush: x stored little-endian below ptr
        acc = (acc << 32) | x;
        nbits += 32;
        drain();
    }
    __device__ __forceinline__ void finish() {  // leftover bytes sit in the low bytes of acc, oldest highest
        uint8_t* p = reinterpret_cast<uint8_t*>(wptr);
        const uint32_t n = nbits >> 3;
        for (uint32_t k = 0; k < n; k++) p[-1 - (int)k] = (uint8_t)(acc >> (8 * (n - 1 - k)));
    }
};

// writes one byte per call at increasing addresses starting anywhere: bytes are collected into aligned words; the
// partial words at the two ends of the range (shared with the neighbouring reads) are written byte by byte
struct FwdWriter {
    uint8_t* wbase;  // aligned address of the word being filled
    uint32_t acc, lane, first;  // lane = byte of the word the next push fills; first = first lane this range owns
    __device__ __forceinline__ void init(uint8_t* dst) {
        lane = (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 3);
        first = lane;
        wbase = dst - lane;
        acc = 0;
    }
    __device__ __forceinline__ void push(uint32_t b) {
        acc |= b << (8 * lane);
        if (++lane == 4) {
            if (first == 0) {
                *reinterpret_cast<uint32_t*>(wbase) = acc;
            } else {
                for (uint32_t k = first; k < 4; k++) wbase[k] = (uint8_t)(acc >> (8 * k));
                first = 0;
            }
            wbase += 4;
            acc = 0;
            lane = 0;
        }
    }
    __device__ __forceinline__ void finish() {
        for (uint32_t k = first; k < lane; k++) wbase[k] = (uint8_t)(acc >> (8 * k));
    }
};

// ---------------------------------------------------------------------------------------------------
// K2: forward single-state scorer   ModelTester::compute_size, idn/model_chooser.rs:215-243
// ---------------------------------------------------------------------------------------------------
// K2, several models at once: one thread per read walks the read ONCE and advances every candidate model per
// position (symbols, the N/zero test and the position counter are shared; the M table-gather chains are independent,
// which gives the memory system M requests in flight per thread).  The models travel by value in the kernel
// parameter space, so their constants cost no registers.
template <int M>
struct ModelPack {
    ModelDev m[M];
    uint32_t n;
};

// kDense: every model of the pack has the dense spec -> row table (no hash fallback in the loop)
template <int M, bool kDense>
__global__ void __launch_bounds__(128)
score_multi_kernel(const ModelPack<M> P, const uint8_t* __restrict__ acids, const uint8_t* __restrict__ quals,
                   const uint64_t* __restrict__ read_off, uint64_t n_reads, uint32_t n_cols, uint32_t col0,
                   uint32_t* __restrict__ sizes, uint32_t* __restrict__ err) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    uint64_t off = read_off[r];
    uint32_t len = (uint32_t)(read_off[r + 1] - off);
    uint32_t pbmax = 0;
#pragma unroll
    for (int k = 0; k < M; k++)
        if (k < (int)P.n) pbmax = max(pbmax, P.m[k].spec.pb);
    PosFwd pf;
    pf.init(len, pbmax);
    GenFwd g[M];
    uint32_t x[M], bytes[M];
#pragma unroll
    for (int k = 0; k < M; k++) {
        g[k].init();
        x[k] = kRansL;
        bytes[k] = 0;
    }
    FwdReader ra, rq;
    ra.start(acids + off);
    rq.start(quals + off);
    bool bad = false;
#pragma unroll 1
    for (uint32_t i = 0; i < len; i++) {
        uint32_t a = ra.get(), q = rq.get();
        if (a > 4 || q > 93) {
            bad = true;
            a = a > 4 ? 0 : a;
            q = q > 93 ? 0 : q;
        }
        const bool z = a * q == 0;
        uint2 e[M];
#pragma unroll
        for (int k = 0; k < M; k++)
            if (k < (int)P.n) {
                const ModelDev& m = P.m[k];
                if (m.aenc) {  // acid model with the encoder entries per spec: one gather instead of two
                    e[k] = __ldg(m.aenc + (g[k].index(m.spec, pf.pos, pbmax - m.spec.pb) * kAcidSyms + a));
                } else {
                    const uint32_t row = gen_row<kDense>(m, m.spec, g[k], pf.pos, pbmax - m.spec.pb);
                    e[k] = __ldg(m.enc + (row * m.nsym + (m.type == 0 ? a : q)));
                }
            }
#pragma unroll
        for (int k = 0; k < M; k++)
            if (k < (int)P.n) {
                rans_put_count(x[k], e[k], bytes[k]);
                g[k].update(P.m[k].spec, a, q, z);
            }
        pf.advance();
    }
#pragma unroll
    for (int k = 0; k < M; k++)
        if (k < (int)P.n) sizes[r * n_cols + col0 + k] = bytes[k] + 4;
    if (bad) atomicOr(err, 1u);
}

// ---------------------------------------------------------------------------------------------------
// K3: greedy per-read model choice inside each block.  One warp per (block, model type).
// The choice for read r depends on the model active after read r-1, so the warp composes per-chunk
// transition functions: lane l simulates its chunk for every possible incoming state, a 32-step
// sequential pass picks the true incoming state of every lane, and each lane then replays its chunk.
// State space: "none" (block start) or one of the candidate models of the type (<= kMaxCand).
// ---------------------------------------------------------------------------------------------------
constexpr int kMaxCand = 16;

__device__ __forceinline__ uint32_t pick_model(const uint32_t* __restrict__ sz, uint32_t n_cand, uint32_t cur) {
    // first minimum of size + (k == cur ? 0 : 2)   (Iterator::min_by keeps the first; penalty model_chooser.rs:175-186)
    uint32_t best = 0, best_len = 0xffffffffu;
    for (uint32_t k = 0; k < n_cand; k++) {
        uint32_t l = sz[k] + (k == cur ? 0u : 2u);
        if (l < best_len) {
            best_len = l;
            best = k;
        }
    }
    return best;
}

// sizes: [n_reads][n_models] (all models); cand[type][k] = column of candidate k of that type.
// chosen[type][r] = candidate index (0..n_cand-1) ; switched[type][r] = 1 when a SwitchModel slice precedes r.
__global__ void __launch_bounds__(32)
switch_kernel(const uint32_t* __restrict__ sizes_all, uint32_t n_models, const uint32_t* __restrict__ cand,
              const uint32_t* __restrict__ n_cand2, const uint32_t* __restrict__ has_sizes,
              const uint32_t* __restrict__ block_first, uint32_t n_blocks, uint8_t* __restrict__ chosen,
              uint8_t* __restrict__ switched, uint64_t n_reads) {
    uint32_t b = blockIdx.x >> 1, type = blockIdx.x & 1;
    if (b >= n_blocks) return;
    uint32_t n_cand = n_cand2[type];
    const uint32_t* sizes = has_sizes[type] ? sizes_all : nullptr;  // single candidate: nothing to compare
    const uint32_t* cols = cand + type * kMaxCand;
    uint32_t lane = threadIdx.x;
    uint64_t r0 = block_first[b], r1 = block_first[b + 1];
    uint64_t n = r1 - r0, per = (n + 31) / 32;
    uint64_t c0 = r0 + lane * per, c1 = c0 + per;
    if (c0 > r1) c0 = r1;
    if (c1 > r1) c1 = r1;
    uint8_t* ch = chosen + (size_t)type * n_reads;
    uint8_t* sw = switched + (size_t)type * n_reads;
    const uint32_t NONE = 0xffu;

    uint32_t sz[kMaxCand];
    // phase 1: out[s] = state after the chunk when entering with state s (s = n_cand means NONE)
    uint32_t out[kMaxCand + 1];
    for (uint32_t s = 0; s <= n_cand; s++) out[s] = s == n_cand ? NONE : s;
    for (uint64_t r = c0; r < c1; r++) {
        for (uint32_t k = 0; k < n_cand; k++) sz[k] = sizes ? sizes[r * n_models + cols[k]] : 0u;
        // the result depends on cur only through "is cur == k"; evaluate once per distinct incoming state
        uint32_t res[kMaxCand + 1];
        for (uint32_t s = 0; s <= n_cand; s++) res[s] = pick_model(sz, n_cand, s == n_cand ? NONE : s);
        for (uint32_t s = 0; s <= n_cand; s++) {
            uint32_t cur = out[s];
            out[s] = res[cur == NONE ? n_cand : cur];
        }
    }
    // phase 2: lane l+1 enters with the state lane l leaves with (lane 0 enters with NONE)
    uint32_t in_state = NONE;
    for (uint32_t l = 0; l < 31; l++) {
        uint32_t my_out = out[in_state == NONE ? n_cand : in_state];
        uint32_t from_l = __shfl_sync(0xffffffffu, my_out, l);
        if (lane == l + 1) in_state = from_l;
    }
    // phase 3: replay
    uint32_t cur = in_state;
    for (uint64_t r = c0; r < c1; r++) {
        for (uint32_t k = 0; k < n_cand; k++) sz[k] = sizes ? sizes[r * n_models + cols[k]] : 0u;
        uint32_t best = pick_model(sz, n_cand, cur);
        ch[r] = (uint8_t)best;
        sw[r] = best != cur;
        cur = best;
    }
}

// one candidate per type: nothing to choose; only the first read of every block carries the two SwitchModel slices
// (chosen / switched were cleared by the caller)
__global__ void switch_single_kernel(const uint32_t* __restrict__ block_first, uint32_t n_blocks, uint8_t* __restrict__ switched,
                                     uint64_t n_reads) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks || block_first[b + 1] == block_first[b]) return;
    switched[block_first[b]] = 1;
    switched[n_reads + block_first[b]] = 1;
}

// ---------------------------------------------------------------------------------------------------
// K4: two-state per-read rANS encode.  One thread per read, symbols walked last -> first.
// Writes the payload right-aligned into the read's scratch slot [slot_end - pay_len, slot_end).
// ---------------------------------------------------------------------------------------------------
struct EncodeArgs {
    const ModelDev* models;
    const uint8_t* acids;
    const uint8_t* quals;
    uint64_t n_symbols;
    const uint64_t* read_off;
    uint64_t n_reads;
    // model choice: either fixed (fast / single model per type) or per read
    int32_t fixed_acid, fixed_q;        // indices into models[], used when chosen == nullptr
    const uint8_t* chosen;              // [2][n_reads] candidate index per type, or nullptr
    const int32_t* cand_model;          // [2][kMaxCand] candidate -> models[] index
    uint8_t* scratch;                   // slot of read r ends at 4*read_off[r+1] + kSlotExtra*(r+1)
    uint32_t* pay_len;                  // [n_reads]
    uint32_t* err;
    const uint8_t* switched;            // [2][n_reads]: a SwitchModel slice precedes the read's Sequence slice, or nullptr
    const uint8_t* cand_index;          // [2][kMaxCand] candidate -> SwitchModel index
    // optional: the per-read CRC-32 partials crc(acids | quals) for crc_block_kernel, computed on the way (EncCrc)
    const uint32_t* crc_back;           // [256 + 2 * kCrcLenTab] (make_crc_back_tables), or nullptr
    const uint32_t* xpow;               // [64]
    uint32_t* part_crc;
    unsigned long long* part_len;
};
// the reads of one launch of a *_list_kernel: list[*base .. *base + *count), one bucket of bucket_scatter_kernel (the reads
// that chose this launch's model pair)
struct ReadList {
    const uint32_t* list;
    const uint32_t* base;
    const uint32_t* count;
};
// scratch bytes per read besides 4 per symbol: two flushed states (8) + Sequence slice header (9) + two SwitchModel
// slices (4), rounded up to keep the slot ends word-aligned
constexpr unsigned long long kSlotExtra = 24;

// State of one rANS output stream under construction (a read in compat mode, a lane in native mode).
struct EncStream {
    uint32_t x0, x1;  // state 0 = acids, state 1 = quality scores (compressor.rs:95-96)
    BackWriter out;
    bool bad;         // an input symbol was out of range
    __device__ __forceinline__ void begin(uint8_t* slot_end) {
        x0 = x1 = kRansL;
        out.init(slot_end);
        bad = false;
    }
    __device__ __forceinline__ void flush_states() {  // flush_all: state 0 then state 1
        out.push_u32_le(x0);
        out.push_u32_le(x1);
    }
    __device__ __forceinline__ void flush() {
        flush_states();
        out.finish();
    }
    __device__ __forceinline__ uint32_t total(const uint8_t* slot_end) const { return out.bytes(slot_end); }  // bytes emitted so far
};

// CRC-32 of a byte string whose bytes arrive LAST TO FIRST (the encoder's order).  With L = "advance the register by one
// zero byte" (c -> tab[c & 0xff] ^ (c >> 8), linear over GF(2)) the register after the string b_0 .. b_{n-1} is
// L^n(ff..f) ^ XOR_i L^(n-1-i)(tab[b_i]).  Keeping B = L^-(n-i)(contribution of b_i .. b_{n-1}) turns the backward walk into
// B <- Linv(B) ^ Linv(tab[b]) = (B << 8) ^ tinv[B >> 24] ^ b  -- tab[b] = L(b), so Linv(tab[b]) is the byte itself: one
// shift and one look-up per byte -- and crc = ~L^n(B ^ ff..f), where L^n is the multiplication by x^(8n) mod P (gf2_mul).
// Linv(v) = v << 8 for v < 2^24 (tinv[0] = 0), so four bytes w = b_i b_{i+1} b_{i+2} b_{i+3} (b_i in bits 24..31) step
// B <- Linv^4(B) ^ w.  For acids | quals of one read (two strings of n bytes walked in lock step):
// crc = ~(x^(8n) * Bq  ^  x^(16n) * (Ba ^ ff..f)).
constexpr uint32_t kCrcLenTab = 1024;  // read lengths whose x^(8n), x^(16n) come from a table
__device__ __forceinline__ uint32_t gf2_mul(uint32_t a, uint32_t b);  // (K7 section below)
__device__ __forceinline__ uint32_t x8n_mod_p(unsigned long long n, const uint32_t* __restrict__ xpow);
struct EncCrc {
    const uint32_t* tinv;  // shared memory [256], or nullptr: no CRC
    uint32_t ba, bq;
    __device__ __forceinline__ void add(uint32_t a, uint32_t q) {
        ba = (ba << 8) ^ tinv[ba >> 24] ^ a;
        bq = (bq << 8) ^ tinv[bq >> 24] ^ q;
    }
    __device__ __forceinline__ void add_word(uint32_t wa, uint32_t wq) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            ba = (ba << 8) ^ tinv[ba >> 24];
            bq = (bq << 8) ^ tinv[bq >> 24];
        }
        ba ^= wa;
        bq ^= wq;
    }
};

// Pushes the positions p1-1 .. p0 of one read onto the stream (the whole read: p0 = 0, p1 = len)
//   SequenceCompressor::compress, sequence_compressor.rs:82-155
// The generators always see the true symbols in front of a position, so a piece of a read (native format, long reads cut
// into lanes) is coded with the same contexts as inside the whole read.
//
// The loop is software-pipelined over three positions because only the 32-bit rANS states are serial in the encoder:
// while position i is coded, the encoder entry of position i-1 is being gathered and the context row of position i-2
// is being looked up, so the two dependent L2 gathers per symbol (spec -> row -> entry) overlap with arithmetic.
template <class P>
__device__ __forceinline__ void encode_read_body(const ModelDev& ma, const ModelDev& mq, const uint8_t* __restrict__ acids,
                                                 const uint8_t* __restrict__ quals, unsigned long long n_symbols, long long off,
                                                 uint32_t len, uint32_t p0, uint32_t p1, EncStream& S, EncCrc& C) {
    constexpr SpecDev ksa = P::sa(), ksq = P::sq();  // compile-time generator parameters of a specialised pair
    const SpecDev& sa = P::kStatic ? ksa : ma.spec;
    const SpecDev& sq = P::kStatic ? ksq : mq.spec;
#ifndef IDN_NO_SYM16
    SymBackReader rs;
    rs.start(acids, quals, n_symbols, off, p1);  // nothing is loaded when p1 == 0
#else
    (void)n_symbols;
    BackReader ra, rq;
    ra.start(acids + off + p1 - 1);  // nothing is loaded before the first get()
    rq.start(quals + off + p1 - 1);
#endif
    GenBack ga, gq;
    ga.clear(sa);
    gq.clear(sq);
    uint32_t raw_a = 0;  // raw symbols travel in two more shift registers (entry k = position j - k)
    unsigned long long raw_q = 0;
    auto shift_in = [&](uint32_t a, uint32_t q) {
        const bool z = a * q == 0;
        ga.shift_in(sa, a, q, z);
        gq.shift_in(sq, a, q, z);
        raw_a = (raw_a >> 3) | (a << (3 * kHist));
        raw_q = (raw_q >> 7) | ((unsigned long long)q << (7 * kHist));
    };
    // pulls position `front` into the windows (zeros in front of the read: front < 0); called for p1-1, p1-2, ... in turn
    auto pull = [&](int32_t front) {
        uint32_t a = 0, q = 0;
        if (front >= 0) {
#ifndef IDN_NO_SYM16
            rs.get(a, q);
#else
            a = ra.get();
            q = rq.get();
#endif
            if (a > 4 || q > 93) {
                S.bad = true;
                a = a > 4 ? 0 : a;
                q = q > 93 ? 0 : q;
            }
            if (C.tinv) C.add(a, q);  // uniform per launch; whole reads only (every position is pulled exactly once, last to first)
        }
        shift_in(a, q);
    };
#pragma unroll 1
    for (int t = 0; t < kHist; t++) pull((int32_t)p1 - 1 - t);  // entry k = symbol at p1 - k
    ga.init_state(sa);
    gq.init_state(sq);
    const uint32_t pbmax = sa.pb > sq.pb ? sa.pb : sq.pb;
    const uint32_t psa = pbmax - sa.pb, psq = pbmax - sq.pb;
    PosBack pb;
    pb.init_at(len, pbmax, p1);

    // acid side: models with a small dense spec space carry the encoder entries per spec (ModelDev::aenc), i.e. the "row" of
    // the acid side is the spec itself and spec -> row -> entry is one gather
#ifndef IDN_NO_AENC
    const bool direct_a = P::kStatic || ma.aenc != nullptr;
#else
    const bool direct_a = false;
#endif
    const uint2* __restrict__ enc_a = direct_a ? ma.aenc : ma.enc;
    uint32_t row_a, row_q;
    // generator stage, once position j - kHist is in the windows: moves the generators to position j (entry 0 = symbol j)
    // and looks the two rows up
    auto gen_step = [&]() {
        ga.step_back(sa);
        gq.step_back(sq);
        pb.retreat();
        row_a = direct_a ? ga.index(sa, pb.pos, psa) : gen_row<P::kStatic>(ma, sa, ga, pb.pos, psa);
        row_q = gen_row<P::kStatic>(mq, sq, gq, pb.pos, psq);
    };
    auto rows_next = [&](int32_t j) {  // j = p1-1, p1-2, ... in turn (reads are shorter than 2^31)
        row_a = row_q = 0;
        if (j >= (int32_t)p0) {
            pull(j - kHist);
            gen_step();
        }
    };
    // entries of the position the generators stand at
    auto entries = [&](uint2& ea_, uint2& eq_) {
        ea_ = ldg_stream8(enc_a + (row_a * kAcidSyms + (raw_a & 7u)));
        eq_ = __ldg(mq.enc + (row_q * kQSyms + ((uint32_t)raw_q & 127u)));
    };
    uint2 ea = make_uint2(0, 0), eq = make_uint2(0, 0);
    auto put = [&]() {
        rans_put_bf(S.x0, ea, S.out);  // put_at(0, acid) then put_at(1, q)   compressor.rs:95-96
        rans_put_bf(S.x1, eq, S.out);
        S.out.drain();
    };
    // prologue: rows of position p1-1, its entries, rows of position p1-2
    rows_next((int32_t)p1 - 1);  // generators at p1-1, entry 0 = symbol p1-1
    if (p1 > p0) entries(ea, eq);
    rows_next((int32_t)p1 - 2);  // generators at p1-2
#ifndef IDN_NO_SYM16
    // Coding position i gathers the entries of i-1 when i > p0, moves the generators to i-2 when i-2 >= p0 and pulls
    // position i-2-kHist when it is >= 0.  While i >= wlim (i = the last position coded), the next four positions
    // i-1 .. i-4 do all three, and once the reader stands at a word boundary the four symbols they pull are one word of
    // each array: that interior runs one word per iteration without the per-position tests; the head (down to the first
    // word boundary) and the tail run position by position.  The interior also stays above the chunk that holds the
    // first byte of an array that is not 16-byte aligned (so its loads need no bounds test): its pulls must not reach
    // below position `skip` of the read.
    const long long skip = (long long)((0 - reinterpret_cast<uintptr_t>(acids)) & 15) - off;
    uint32_t wlim = p0 > kHist ? p0 : kHist;
    if (skip > 0 && (uint32_t)skip + kHist > wlim) wlim = (uint32_t)skip + kHist;
    wlim += 4 + 2;  // the lowest pull of a word step: (i - 4) - 2 - kHist
#endif
    uint32_t i = p1;
#pragma unroll 1
    while (i > p0) {
#ifndef IDN_NO_SYM16
        // (one word per pass of the outer loop, not a loop of its own: the threads of a warp reach their first word
        // boundary up to three positions apart, and an inner loop would run their interiors one after the other)
        if (rs.vec && (rs.left & 3) == 0 && i >= wlim) {
            rs.peek_word();
            // some acid > 4 or quality score > 93: flag the read and zero those bytes, as pull() does
            if ((((rs.ca & 0x7f7f7f7fu) + 0x7b7b7b7bu) | rs.ca | ((rs.cq & 0x7f7f7f7fu) + 0x22222222u) | rs.cq) & 0x80808080u) {
                S.bad = true;
                uint32_t ca = 0, cq = 0;
#pragma unroll 1
                for (int k = 0; k < 32; k += 8) {
                    const uint32_t a = (rs.ca >> k) & 0xffu, q = (rs.cq >> k) & 0xffu;
                    ca |= (a > 4 ? 0u : a) << k;
                    cq |= (q > 93 ? 0u : q) << k;
                }
                rs.ca = ca;
                rs.cq = cq;
            }
            if (C.tinv) C.add_word(rs.ca, rs.cq);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                uint2 ea_n, eq_n;
                entries(ea_n, eq_n);  // of position i-2-k
                shift_in(__byte_perm(rs.ca, 0, 0x4443 - k), __byte_perm(rs.cq, 0, 0x4443 - k));
                gen_step();  // generators to i-3-k
                put();       // position i-1-k
                ea = ea_n;
                eq = eq_n;
            }
            rs.skip_word();
            i -= 4;
            continue;
        }
#endif
        i--;
        // entries of position i-1 (generators stand at i-1: entry 0), gathered while position i is coded
        uint2 ea_n = make_uint2(0, 0), eq_n = make_uint2(0, 0);
        if (i > p0) entries(ea_n, eq_n);
        rows_next((int32_t)i - 2);  // generators to i-2
        put();
        ea = ea_n;
        eq = eq_n;
    }
}

// kUniform: every read of the batch uses the same model pair; its parameters then live in the kernel parameter
// space (constant bank operands) instead of ~40 registers per thread, which is what bounds occupancy here.
// resident CTAs per SM the uniform kernels are compiled for: 8 x 128 threads = 64 registers per thread.  Round 1 ran 9
// (56 registers); the 16-byte symbol chunks of round 2 need the room (9 CTAs spill: encode 12.1 vs 7.9 ms per 3 GB).
#ifndef IDN_ENC_MINB
#define IDN_ENC_MINB 8
#endif
#ifndef IDN_DEC_MINB
#define IDN_DEC_MINB 8
#endif
template <bool kUniform, class P>
__device__ __forceinline__ void encode_one(const EncodeArgs& A, const ModelDev& MA, const ModelDev& MQ, uint64_t r, const uint32_t* s_back) {
    int32_t ia = A.fixed_acid, iq = A.fixed_q;
    if (!kUniform && A.chosen) {
        ia = A.cand_model[A.chosen[r]];
        iq = A.cand_model[kMaxCand + A.chosen[A.n_reads + r]];
    }
    const ModelDev& ma = kUniform ? MA : A.models[ia];
    const ModelDev& mq = kUniform ? MQ : A.models[iq];
    const long long off = (long long)A.read_off[r];
    const uint32_t len = (uint32_t)(A.read_off[r + 1] - A.read_off[r]);
    EncStream S;
    S.begin(A.scratch + 4ull * A.read_off[r + 1] + kSlotExtra * (r + 1));
    EncCrc C{A.crc_back ? s_back : nullptr, 0u, 0u};
    encode_read_body<P>(ma, mq, A.acids, A.quals, A.n_symbols, off, len, 0, len, S, C);
    if (A.crc_back) {  // crc(acids | quals) of the read, as crc_read_kernel computes it
        uint32_t x1, x2;  // x^(8 len), x^(16 len) mod P
        if (len < kCrcLenTab) {
            const uint2 x = __ldg(reinterpret_cast<const uint2*>(A.crc_back + 256) + len);
            x1 = x.x;
            x2 = x.y;
        } else {
            x1 = x8n_mod_p(len, A.xpow);
            x2 = gf2_mul(x1, x1);
        }
        A.part_crc[r] = len ? ~(gf2_mul(x1, C.bq) ^ gf2_mul(x2, ~C.ba)) : 0u;
        A.part_len[r] = 2ull * len;
    }
    S.flush_states();
    const uint32_t plen = S.total(A.scratch + 4ull * A.read_off[r + 1] + kSlotExtra * (r + 1));
    A.pay_len[r] = plen;
    // the read's slices, complete, in front of the payload (the writer walks down): [01 acid idx][01 q idx] 02 u32be
    // length u32be seq_len   (data.rs:57-84, compressor_block.rs:103-110), so that assembly is one copy per read
    S.out.push_u32_le(__byte_perm(len, 0, 0x0123));
    S.out.push_u32_le(__byte_perm(plen, 0, 0x0123));
    S.out.push_bits(2u, 8);
    S.out.drain();
    if (A.switched) {
        if (A.switched[A.n_reads + r]) {
            S.out.push_bits(((uint32_t)A.cand_index[kMaxCand + A.chosen[A.n_reads + r]] << 8) | 1u, 16);
            S.out.drain();
        }
        if (A.switched[r]) {  // acid first (compressor_block.rs:103-104)
            S.out.push_bits(((uint32_t)A.cand_index[A.chosen[r]] << 8) | 1u, 16);
            S.out.drain();
        }
    }
    S.out.finish();
    if (S.bad) atomicOr(A.err, 1u);
}

template <bool kUniform, class P>
__global__ void __launch_bounds__(128, kUniform ? IDN_ENC_MINB : 1)
encode_kernel(EncodeArgs A, const ModelDev MA, const ModelDev MQ) {
    __shared__ uint32_t s_back[256];
    if (A.crc_back) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s_back[i] = A.crc_back[i];
        __syncthreads();
    }
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= A.n_reads) return;
    encode_one<kUniform, P>(A, MA, MQ, r, s_back);
}

// Per-read model selection: one launch per model pair over the reads that chose it (a fixed grid strides over the bucket,
// whose size only the device knows), so that those reads run the uniform -- and, for the bundled pairs, the compile-time
// specialised -- arithmetic instead of the run-time generic one.
template <class P>
__global__ void __launch_bounds__(128, IDN_ENC_MINB)
encode_list_kernel(EncodeArgs A, const ModelDev MA, const ModelDev MQ, ReadList L) {
    __shared__ uint32_t s_back[256];
    if (A.crc_back) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s_back[i] = A.crc_back[i];
        __syncthreads();
    }
    const uint32_t n = *L.count;
    const uint32_t* __restrict__ list = L.list + *L.base;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        encode_one<true, P>(A, MA, MQ, list[i], s_back);
}

// ---------------------------------------------------------------------------------------------------
// Buckets of reads by model pair (per-read selection): count, exclusive scan, scatter.  KeyFn(r) = pair number of read r
// or 0xffffffff (no such read).  The order inside a bucket depends on the order the CTAs arrive in; the output does not
// (every read writes its own slot).
// ---------------------------------------------------------------------------------------------------
constexpr uint32_t kMaxPairs = 1024;

struct EncodePairKey {  // compress side: the candidates the greedy switcher chose
    const uint8_t* chosen;  // [2][n_reads]
    uint64_t n_reads;
    uint32_t n_q;
    __device__ __forceinline__ uint32_t operator()(uint64_t r) const {
        return r < n_reads ? (uint32_t)chosen[r] * n_q + chosen[n_reads + r] : 0xffffffffu;
    }
};

template <class KeyFn>
__global__ void __launch_bounds__(256)
bucket_count_kernel(KeyFn key, uint64_t n, uint32_t n_pairs, uint32_t* __restrict__ cnt) {
    __shared__ uint32_t hist[kMaxPairs];
    for (uint32_t k = threadIdx.x; k < n_pairs; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t k = r < n ? key(r) : 0xffffffffu;
    if (k < n_pairs) atomicAdd(&hist[k], 1u);
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < n_pairs; j += blockDim.x)
        if (hist[j]) atomicAdd(&cnt[j], hist[j]);
}

// cnt[n_pairs] -> base[n_pairs] (exclusive scan), cursor = base
__global__ void bucket_base_kernel(const uint32_t* __restrict__ cnt, uint32_t n_pairs, uint32_t* __restrict__ base, uint32_t* __restrict__ cursor) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t acc = 0;
    for (uint32_t k = 0; k < n_pairs; k++) {
        base[k] = cursor[k] = acc;
        acc += cnt[k];
    }
}

template <class KeyFn>
__global__ void __launch_bounds__(256)
bucket_scatter_kernel(KeyFn key, uint64_t n, uint32_t n_pairs, uint32_t* __restrict__ cursor, uint32_t* __restrict__ list) {
    __shared__ uint32_t hist[kMaxPairs];
    for (uint32_t k = threadIdx.x; k < n_pairs; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t k = r < n ? key(r) : 0xffffffffu;
    uint32_t rank = 0;
    if (k < n_pairs) rank = atomicAdd(&hist[k], 1u);
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < n_pairs; j += blockDim.x)
        if (hist[j]) hist[j] = atomicAdd(&cursor[j], hist[j]);  // the CTA's range in bucket j
    __syncthreads();
    if (k < n_pairs) list[hist[k] + rank] = (uint32_t)r;
}

// ---------------------------------------------------------------------------------------------------
// exclusive scan over u64 (three launches; sizes of a few million elements)
// ---------------------------------------------------------------------------------------------------
constexpr int kScanBlock = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanBlock * kScanItems;

__device__ __forceinline__ unsigned long long block_exclusive_scan(unsigned long long v, unsigned long long* total,
                                                                  unsigned long long* smem /*[kScanBlock/32]*/) {
    uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned long long inc = v;
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += o;
    }
    if (lane == 31) smem[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        unsigned long long s = lane < kScanBlock / 32 ? smem[lane] : 0;
        unsigned long long sinc = s;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long o = __shfl_up_sync(0xffffffffu, sinc, d);
            if (lane >= (uint32_t)d) sinc += o;
        }
        if (lane < kScanBlock / 32) smem[lane] = sinc - s;
        if (lane == kScanBlock / 32 - 1) *total = sinc;
    }
    __syncthreads();
    unsigned long long r = inc - v + smem[wid];
    __syncthreads();
    return r;
}

// per-read slice size -> per-tile sums
template <class SizeFn>
__global__ void __launch_bounds__(kScanBlock)
scan_reduce_kernel(SizeFn fn, uint64_t n, unsigned long long* __restrict__ tile_sum) {
    __shared__ unsigned long long smem[kScanBlock / 32];
    __shared__ unsigned long long total;
    uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    unsigned long long v = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; k++)
        if (base + k < n) v += fn(base + k);
    block_exclusive_scan(v, &total, smem);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// single block: exclusive scan of tile sums in place; grand total to tile_sum[n_tiles]
__global__ void __launch_bounds__(kScanBlock)
scan_tiles_kernel(unsigned long long* __restrict__ tile_sum, uint32_t n_tiles) {
    __shared__ unsigned long long smem[kScanBlock / 32];
    __shared__ unsigned long long total;
    unsigned long long carry = 0;
    for (uint32_t base = 0; base < n_tiles; base += kScanBlock) {
        uint32_t i = base + threadIdx.x;
        unsigned long long v = i < n_tiles ? tile_sum[i] : 0;
        unsigned long long ex = block_exclusive_scan(v, &total, smem);
        if (i < n_tiles) tile_sum[i] = carry + ex;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) tile_sum[n_tiles] = carry;
}

template <class SizeFn>
__global__ void __launch_bounds__(kScanBlock)
scan_apply_kernel(SizeFn fn, uint64_t n, const unsigned long long* __restrict__ tile_sum,
                  unsigned long long* __restrict__ out /*[n+1]*/) {
    __shared__ unsigned long long smem[kScanBlock / 32];
    __shared__ unsigned long long total;
    uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    unsigned long long item[kScanItems], v = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; k++) {
        item[k] = base + k < n ? fn(base + k) : 0;
        v += item[k];
    }
    unsigned long long ex = block_exclusive_scan(v, &total, smem) + tile_sum[blockIdx.x];
#pragma unroll
    for (int k = 0; k < kScanItems; k++) {
        if (base + k < n) out[base + k] = ex;
        ex += item[k];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) out[n] = tile_sum[gridDim.x];
}

// ---------------------------------------------------------------------------------------------------
// compat-mode container layout (writer_block.rs:27-82, data.rs:35-84)
//   block b: [u32be length][u32be crc][prefix_len[b] bytes reserved][fast: 01 00 01 01] then per read
//            [01 idx]* [02 u32be len u32be seq_len payload]
// slice_off[r] = offset of read r's first slice byte counted over all reads' slices only (scan of
// slice sizes); block overheads are added per block through block_base[b].
// ---------------------------------------------------------------------------------------------------
struct SliceSize {
    const uint32_t* pay_len;
    const uint8_t* switched;  // [2][n_reads] or nullptr
    uint64_t n_reads;
    __device__ __forceinline__ unsigned long long operator()(uint64_t r) const {
        unsigned long long s = 9ull + pay_len[r];
        if (switched) s += 2u * switched[r] + 2u * switched[n_reads + r];
        return s;
    }
};

// block b's length field: its slices, the reserved prefix and the fast-mode marker (an empty block has no marker)
__device__ __forceinline__ unsigned long long block_length(const unsigned long long* __restrict__ slice_off,
                                                           const uint32_t* __restrict__ block_first, uint32_t b,
                                                           const uint32_t* __restrict__ prefix_len, int fast) {
    const unsigned long long body = slice_off[block_first[b + 1]] - slice_off[block_first[b]];
    const bool empty = block_first[b + 1] == block_first[b];
    return body + (prefix_len ? prefix_len[b] : 0) + ((fast && !empty) ? 4 : 0);
}

// block layout, step 1 of 3: thread per block, block_off[b] = the bytes of block b (header + length); step 2 is the
// exclusive scan of block_off by scan_tiles_kernel, step 3 block_layout_kernel
__global__ void block_size_kernel(const unsigned long long* __restrict__ slice_off, const uint32_t* __restrict__ block_first,
                                  uint32_t n_blocks, const uint32_t* __restrict__ prefix_len, int fast,
                                  unsigned long long* __restrict__ block_off /*[n_blocks+1]*/) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < n_blocks) block_off[b] = 8 + block_length(slice_off, block_first, b, prefix_len, fast);
}

// thread per block, after the scan: block_adj, the length field and the fast-mode marker of block b at block_off[b];
// thread 0 also leaves the container size in stats[0] (out_bytes / required_bytes).  Launch with at least one thread.
__global__ void block_layout_kernel(const unsigned long long* __restrict__ slice_off, const uint32_t* __restrict__ block_first,
                                    uint32_t n_blocks, const uint32_t* __restrict__ prefix_len, int fast,
                                    const unsigned long long* __restrict__ block_off /*[n_blocks+1], scanned*/,
                                    uint8_t* __restrict__ out, uint64_t out_cap, unsigned long long* __restrict__ stats /*[8]*/,
                                    unsigned long long* __restrict__ block_adj /*[n_blocks]: slice_off[r] + block_adj[b] = where read r's slices go*/) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b == 0) stats[0] = block_off[n_blocks];
    if (b >= n_blocks) return;
    const unsigned long long pos = block_off[b];
    const uint32_t prefix = prefix_len ? prefix_len[b] : 0;
    block_adj[b] = pos + 8 + prefix + (fast ? 4 : 0) - slice_off[block_first[b]];
    if (pos + 8 <= out_cap) {
        const uint32_t l = (uint32_t)block_length(slice_off, block_first, b, prefix_len, fast);
        out[pos + 0] = (uint8_t)(l >> 24);
        out[pos + 1] = (uint8_t)(l >> 16);
        out[pos + 2] = (uint8_t)(l >> 8);
        out[pos + 3] = (uint8_t)l;
        const uint64_t f = pos + 8 + prefix;
        if (fast && block_first[b + 1] != block_first[b] && f + 4 <= out_cap) {  // compressor_block.rs:95-99
            out[f + 0] = 1;
            out[f + 1] = 0;
            out[f + 2] = 1;
            out[f + 3] = 1;
        }
    }
}

struct AssembleArgs {
    const uint64_t* read_off;
    uint64_t n_reads;
    const uint32_t* pay_len;
    const uint8_t* scratch;
    const unsigned long long* slice_off;
    const unsigned long long* block_adj;  // [n_blocks], block_layout_kernel
    const uint32_t* read_block;  // [n_reads] block of each read
    const uint8_t* chosen;    // [2][n_reads] or nullptr
    const uint8_t* switched;  // [2][n_reads] or nullptr
    const uint8_t* cand_index;  // [2][kMaxCand] candidate -> SwitchModel index (position in models[])
    uint8_t* out;
    uint64_t out_cap;
    uint32_t lanes_log2;  // lanes per read: 1..5 (assemble_lanes_log2)
};

constexpr int kAssembleBlock = 256;

// the 16 bytes at address s (any alignment) from the aligned 16-byte loads that hold them; a load whose 16 bytes hold none
// of the wanted source range [vlo, vhi) is left out (its bytes read as 0), so nothing outside that range's aligned cover
// is touched
__device__ __forceinline__ uint4 load_unaligned16(uintptr_t s, uintptr_t vlo, uintptr_t vhi) {
    const uintptr_t a = s & ~(uintptr_t)15;
    const uint32_t off = (uint32_t)(s & 15);
    uint4 lo = make_uint4(0, 0, 0, 0), hi = make_uint4(0, 0, 0, 0);
    if (a + 16 > vlo && a < vhi) lo = __ldg(reinterpret_cast<const uint4*>(a));
    if (off && a + 32 > vlo && a + 16 < vhi) hi = __ldg(reinterpret_cast<const uint4*>(a + 16));
    // words w0 .. w7 = lo | hi; drop off / 4 words, then funnel-shift by the byte rest
    uint32_t w0 = lo.x, w1 = lo.y, w2 = lo.z, w3 = lo.w, w4 = hi.x, w5 = hi.y, w6 = hi.z, w7 = hi.w;
    if (off & 8) {
        w0 = w2, w1 = w3, w2 = w4, w3 = w5, w4 = w6, w5 = w7;
    }
    if (off & 4) {
        w0 = w1, w1 = w2, w2 = w3, w3 = w4, w4 = w5;
    }
    const uint32_t sh = 8 * (off & 3);
    return make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                      __funnelshift_r(w3, w4, sh));
}

// bytes [k0, k1) of the 16-byte destination chunk at d (the bytes around them belong to somebody else)
__device__ __forceinline__ void store_bytes16(uint8_t* d, uint4 v, uint32_t k0, uint32_t k1) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (uint32_t k = 0; k < 16; k++)
        if (k >= k0 && k < k1) d[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
}

// destination chunk c of a read (assemble_kernel): its address, its bytes [k0, k1) to write and their values
struct AssembleChunk {
    uintptr_t a;
    uint4 v;
    uint32_t k0, k1;
};
__device__ __forceinline__ AssembleChunk assemble_chunk(uint32_t c, uint32_t n_chunks, uintptr_t c0, uintptr_t d, uintptr_t e,
                                                        uintptr_t s, uintptr_t pe, bool fits, bool prev_fits) {
    AssembleChunk x;
    x.a = c0 + 16ull * c;
    x.v = make_uint4(0, 0, 0, 0);
    x.k0 = x.k1 = 0;
    if (c >= n_chunks) return x;
    const uintptr_t a = x.a;
    // chunk bytes [0, split) belong to the previous read, [split, k_end) to this one
    const uint32_t split = a < d ? (uint32_t)(d - a) : 0u;
    const uint32_t k_end = a + 16 <= e ? 16u : (uint32_t)(e - a);
    x.k0 = (split && prev_fits) ? 0u : split;
    x.k1 = fits ? k_end : split;
    if (x.k1 > split) x.v = load_unaligned16(s + (a - d), s + (a + split - d), s + (a + k_end - d));  // chunk byte k <- s + (a + k - d)
    if (split && x.k0 == 0) {
        const uint4 p = load_unaligned16(pe - split, pe - split, pe);
        // bytes below split from p
        const uint32_t m0 = split >= 4 ? 0xffffffffu : (1u << (8 * split)) - 1;
        const uint32_t m1 = split >= 8 ? 0xffffffffu : split <= 4 ? 0u : (1u << (8 * (split - 4))) - 1;
        const uint32_t m2 = split >= 12 ? 0xffffffffu : split <= 8 ? 0u : (1u << (8 * (split - 8))) - 1;
        const uint32_t m3 = split <= 12 ? 0u : (1u << (8 * (split - 12))) - 1;
        x.v.x = (p.x & m0) | (x.v.x & ~m0);
        x.v.y = (p.y & m1) | (x.v.y & ~m1);
        x.v.z = (p.z & m2) | (x.v.z & ~m2);
        x.v.w = (p.w & m3) | (x.v.w & ~m3);
    }
    return x;
}

// Lanes per read for assemble_kernel: two passes of two 16-byte chunks per lane for a read of the call's mean length at
// about one byte of slices per symbol, 2 lanes (reads of up to ~100 symbols) to 32 (a warp per read, which loops over
// long reads).  Few lanes per read keep many reads -- many independent loads -- in each warp (on hiseq100, 8 lanes per
// read: 3.3 ms, 4: 2.9 ms, 2: 2.2 ms).
inline uint32_t assemble_lanes_log2(uint64_t n_symbols, uint64_t n_reads) {
    const uint64_t mean = n_reads ? n_symbols / n_reads : 0;
    const uint64_t chunks = (mean + 9 + 15) / 16 + 1;
    uint32_t l2 = 1;
    while (l2 < 5 && (4ull << l2) < chunks) l2++;
    return l2;
}

// Copies the reads' finished slices from their scratch slots into the container.  Within a block the slices of
// consecutive reads lie back to back, so the container body is cut into aligned 16-byte destination chunks, and a chunk
// belongs to the read that holds its LAST byte: its leading bytes, when it has any before the read's first byte, are the
// last bytes of the read before (whose slot ends at 4*read_off[r] + kSlotExtra*r; every read has at least 17 bytes of
// slices, so no chunk reaches two reads back).  A group of 2^lanes_log2 lanes owns a read and moves its chunks as whole
// 16-byte stores, two per lane and pass, each built by funnel shifts from two aligned 16-byte loads per source read; consecutive lanes take
// consecutive chunks, so a warp instruction covers a few hundred contiguous destination bytes instead of 32 scattered
// words.  Bytes are written one by one only where a chunk holds bytes that are not slices of the block: the first chunk
// of a block's first read, the tail of its last read (the last read also owns the chunk that holds its last byte), and
// the reads that do not fit the capacity.  A read is written completely or not at all: never at or past out_cap
// (IDN_E_NOSPACE is reported by the host from stats).
__global__ void __launch_bounds__(kAssembleBlock, 6)
assemble_kernel(AssembleArgs A) {
    const uint64_t t = (uint64_t)blockIdx.x * kAssembleBlock + threadIdx.x;
    const uint64_t r = t >> A.lanes_log2;
    const uint32_t lanes = 1u << A.lanes_log2, j = (uint32_t)t & (lanes - 1);
    if (r >= A.n_reads) return;
    const uint32_t blk = A.read_block[r];
    const bool first = r == 0 || A.read_block[r - 1] != blk;
    const bool last = r + 1 == A.n_reads || A.read_block[r + 1] != blk;
    const unsigned long long dst = A.slice_off[r] + A.block_adj[blk];
    uint32_t nsw = 0;
    if (A.switched) nsw = A.switched[r] + A.switched[A.n_reads + r];
    const uint32_t total = 2u * nsw + 9u + A.pay_len[r];  // the encoder left the read's slices complete in its scratch slot
    const bool fits = dst + total <= A.out_cap;
    const bool prev_fits = !first && dst <= A.out_cap;  // the read before ends at dst
    if (!fits && !prev_fits) return;
    const uintptr_t out = reinterpret_cast<uintptr_t>(A.out);
    const uintptr_t scr = reinterpret_cast<uintptr_t>(A.scratch);
    const uintptr_t d = out + dst, e = d + total;                                        // this read's destination bytes
    const uintptr_t s = scr + 4ull * A.read_off[r + 1] + kSlotExtra * (r + 1) - total;  // and their source
    const uintptr_t pe = scr + 4ull * A.read_off[r] + kSlotExtra * r;                   // end of the previous read's source
    const uintptr_t c0 = d & ~(uintptr_t)15;
    const uint32_t n_chunks = (uint32_t)(((e & ~(uintptr_t)15) - c0) >> 4) + ((last && (e & 15)) ? 1u : 0u);
    // two chunks per lane and pass: both chunks' loads are in flight before the first store
#pragma unroll 1
    for (uint32_t c = j; c < n_chunks; c += 2 * lanes) {
        AssembleChunk x[2];
#pragma unroll
        for (int u = 0; u < 2; u++) x[u] = assemble_chunk(c + u * lanes, n_chunks, c0, d, e, s, pe, fits, prev_fits);
#pragma unroll
        for (int u = 0; u < 2; u++) {
            uint8_t* dp = reinterpret_cast<uint8_t*>(x[u].a);
            if (x[u].k0 == 0 && x[u].k1 == 16) *reinterpret_cast<uint4*>(dp) = x[u].v;
            else if (x[u].k1 > x[u].k0) store_bytes16(dp, x[u].v, x[u].k0, x[u].k1);
        }
    }
}

// read -> block map (one thread per block fills its range; blocks are large, so use a grid-stride loop)
__global__ void read_block_kernel(const uint32_t* __restrict__ block_first, uint32_t n_blocks,
                                  uint32_t* __restrict__ read_block) {
    uint32_t b = blockIdx.x;
    if (b >= n_blocks) return;
    for (uint64_t r = block_first[b] + threadIdx.x; r < block_first[b + 1]; r += blockDim.x) read_block[r] = b;
}

// stats: payload bytes and switch counts (one pass, block reduce + atomics)
__global__ void __launch_bounds__(256)
stats_kernel(const uint32_t* __restrict__ pay_len, const uint8_t* __restrict__ switched, uint64_t n_reads,
             unsigned long long* __restrict__ stats) {
    unsigned long long pay = 0, sa = 0, sq = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * blockDim.x) {
        pay += pay_len[r];
        if (switched) {
            sa += switched[r];
            sq += switched[n_reads + r];
        }
    }
    for (int d = 16; d > 0; d >>= 1) {
        pay += __shfl_down_sync(0xffffffffu, pay, d);
        sa += __shfl_down_sync(0xffffffffu, sa, d);
        sq += __shfl_down_sync(0xffffffffu, sq, d);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&stats[1], sa);
        atomicAdd(&stats[2], sq);
        atomicAdd(&stats[3], pay);
    }
}

// stats[0] = bytes the container needs, [1] acid switches, [2] q switches, [3] payload bytes
// -> idn_compress_stats {out_bytes, acid_switches, q_switches, payload_bytes, required_bytes}
__global__ void finish_stats_kernel(const unsigned long long* __restrict__ stats, const uint32_t* __restrict__ err,
                                    unsigned long long* __restrict__ out, uint32_t* __restrict__ err_out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    out[0] = stats[0];
    out[1] = stats[1];
    out[2] = stats[2];
    out[3] = stats[3];
    out[4] = stats[0];
    if (err_out) {  // the pipelined host-pointer path reads the flags next to the stats (a u64 slot)
        err_out[0] = *err;
        err_out[1] = 0;
    }
}

// ---------------------------------------------------------------------------------------------------
// K7: CRC-32 (IEEE, reflected 0xEDB88320) of name|acids|quals per read, combined per block.
// Per-read partials are combined with the GF(2) "multiply by x^(8n) mod P" operator, which is associative,
// so a block's CRC is a tree reduction over (crc, length) pairs.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t gf2_mul(uint32_t a, uint32_t b) {  // a*b mod P, reflected representation
    uint32_t p = 0;
#pragma unroll 4
    for (int i = 0; i < 32; i++) {
        p ^= (0u - (b >> 31)) & a;
        a = (a >> 1) ^ ((0u - (a & 1u)) & 0xEDB88320u);
        b <<= 1;
    }
    return p;
}

// x^(8n) mod P via the table xpow[k] = x^(8 * 2^k) mod P
__device__ __forceinline__ uint32_t x8n_mod_p(unsigned long long n, const uint32_t* __restrict__ xpow) {
    uint32_t r = 0x80000000u;  // the polynomial "1"
    for (int k = 0; n; k++, n >>= 1)
        if (n & 1) r = gf2_mul(r, xpow[k]);
    return r;
}

struct CrcPair {
    uint32_t crc;
    unsigned long long len;
};
// crc of A|B from crc(A), crc(B), len(B)  (zlib crc32_combine)
__device__ __forceinline__ CrcPair crc_concat(CrcPair a, CrcPair b, const uint32_t* __restrict__ xpow) {
    if (b.len == 0) return a;
    if (a.len == 0) return b;
    CrcPair o;
    o.crc = gf2_mul(x8n_mod_p(b.len, xpow), a.crc) ^ b.crc;
    o.len = a.len + b.len;
    return o;
}

__device__ __forceinline__ uint32_t crc_bytes(const uint8_t* __restrict__ base, unsigned long long off, uint32_t n,
                                              const uint32_t* __restrict__ tab /*smem[256]*/) {
    uint32_t c = 0xffffffffu;
    const uint8_t* p = base + off;
    while (n && (reinterpret_cast<uintptr_t>(p) & 3)) {  // head up to a word boundary
        c = tab[(c ^ *p++) & 0xffu] ^ (c >> 8);
        n--;
    }
    const uint32_t* w = reinterpret_cast<const uint32_t*>(p);
    for (; n >= 4; n -= 4) {  // a word at a time: xor it in, then four table steps
        c ^= __ldg(w++);
        c = tab[c & 0xffu] ^ (c >> 8);
        c = tab[c & 0xffu] ^ (c >> 8);
        c = tab[c & 0xffu] ^ (c >> 8);
        c = tab[c & 0xffu] ^ (c >> 8);
    }
    p = reinterpret_cast<const uint8_t*>(w);
    for (; n; n--) c = tab[(c ^ *p++) & 0xffu] ^ (c >> 8);
    return ~c;
}

// CRC tables of the thread-per-read kernel: one copy of the 256-entry table per lane (entry i of lane l at
// [i * 32 + l]), so that the 32 look-ups of a warp never share a bank, whatever the data.
constexpr int kCrcThreads = 1024;
__device__ __forceinline__ uint32_t crc_step(uint32_t c, const uint32_t* __restrict__ rtab /*+ lane*/) {
    return rtab[(c & 0xffu) << 5] ^ (c >> 8);
}
__device__ __forceinline__ uint32_t crc_bytes_rep(const uint8_t* __restrict__ base, unsigned long long off, uint32_t n,
                                                  const uint32_t* __restrict__ rtab) {
    uint32_t c = 0xffffffffu;
    const uint8_t* p = base + off;
    while (n && (reinterpret_cast<uintptr_t>(p) & 3)) {  // head up to a word boundary
        c = crc_step(c ^ *p++, rtab);
        n--;
    }
    const uint32_t* w = reinterpret_cast<const uint32_t*>(p);
    for (; n >= 4; n -= 4) {
        c ^= __ldg(w++);
        c = crc_step(c, rtab);
        c = crc_step(c, rtab);
        c = crc_step(c, rtab);
        c = crc_step(c, rtab);
    }
    p = reinterpret_cast<const uint8_t*>(w);
    for (; n; n--) c = crc_step(c ^ *p++, rtab);
    return ~c;
}
// two byte strings of the same length and alignment (the acids and the quality scores of a read) in lock step: two
// independent look-up chains per thread
__device__ __forceinline__ void crc_bytes_rep2(const uint8_t* __restrict__ pa, const uint8_t* __restrict__ pq, uint32_t n,
                                               const uint32_t* __restrict__ rtab, uint32_t& crc_a, uint32_t& crc_q) {
    uint32_t ca = 0xffffffffu, cq = 0xffffffffu;
    while (n && (reinterpret_cast<uintptr_t>(pa) & 3)) {
        ca = crc_step(ca ^ *pa++, rtab);
        cq = crc_step(cq ^ *pq++, rtab);
        n--;
    }
    const uint32_t* wa = reinterpret_cast<const uint32_t*>(pa);
    const uint32_t* wq = reinterpret_cast<const uint32_t*>(pq);
    for (; n >= 4; n -= 4) {
        ca ^= __ldg(wa++);
        cq ^= __ldg(wq++);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            ca = crc_step(ca, rtab);
            cq = crc_step(cq, rtab);
        }
    }
    pa = reinterpret_cast<const uint8_t*>(wa);
    pq = reinterpret_cast<const uint8_t*>(wq);
    for (; n; n--) {
        ca = crc_step(ca ^ *pa++, rtab);
        cq = crc_step(cq ^ *pq++, rtab);
    }
    crc_a = ~ca;
    crc_q = ~cq;
}

// one thread per read: partial = crc(name|acids|quals), length = name_len + 2*len.  The CTAs walk the reads in tiles of
// kCrcThreads (grid-stride), so the 32 KB of tables are filled once per CTA.
// n_reads_dev / status (optional) serve the decode path, where the read count only exists on the device.
__global__ void __launch_bounds__(kCrcThreads)
crc_read_kernel(const uint8_t* __restrict__ acids, const uint8_t* __restrict__ quals,
                const unsigned long long* __restrict__ read_off, const uint8_t* __restrict__ names,
                const unsigned long long* __restrict__ name_off, uint64_t n_reads,
                const unsigned long long* __restrict__ n_reads_dev, const int32_t* __restrict__ status,
                const uint32_t* __restrict__ crc_tab, const uint32_t* __restrict__ xpow_g,
                uint32_t* __restrict__ part_crc, unsigned long long* __restrict__ part_len,
                const uint32_t* __restrict__ run_flag /* optional: the kernel does nothing while *run_flag == 0 */) {
    __shared__ uint32_t tab[256 * 32];
    __shared__ uint32_t xpow[64];
    if (status && status[0] != 0) return;
    if (run_flag && *run_flag == 0) return;
    if (n_reads_dev) n_reads = *n_reads_dev;
    for (int i = threadIdx.x; i < 256 * 32; i += blockDim.x) tab[i] = crc_tab[i >> 5];
    for (int i = threadIdx.x; i < 64; i += blockDim.x) xpow[i] = xpow_g[i];
    __syncthreads();
    const uint32_t* rtab = tab + (threadIdx.x & 31);
    const bool same_align = ((reinterpret_cast<uintptr_t>(acids) ^ reinterpret_cast<uintptr_t>(quals)) & 3) == 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * blockDim.x) {
        unsigned long long off = read_off[r];
        uint32_t len = (uint32_t)(read_off[r + 1] - off);
        CrcPair p{0, 0};
        if (names && name_off) {
            uint32_t nl = (uint32_t)(name_off[r + 1] - name_off[r]);
            p.crc = crc_bytes_rep(names, name_off[r], nl, rtab);
            p.len = nl;
        }
        CrcPair a{0, len}, q{0, len};
        if (same_align) {
            crc_bytes_rep2(acids + off, quals + off, len, rtab, a.crc, q.crc);
        } else {
            a.crc = crc_bytes_rep(acids, off, len, rtab);
            q.crc = crc_bytes_rep(quals, off, len, rtab);
        }
        p = crc_concat(crc_concat(p, a, xpow), q, xpow);
        part_crc[r] = p.crc;
        part_len[r] = p.len;
    }
}

// CRC of n bytes by one warp: every lane takes a contiguous slice, the lanes combine in order (result in lane 0)
__device__ __forceinline__ CrcPair crc_bytes_warp(const uint8_t* __restrict__ base, unsigned long long off, uint32_t n,
                                                  const uint32_t* __restrict__ tab, const uint32_t* __restrict__ xpow, uint32_t lane) {
    const uint32_t chunk = (n + 31) / 32;
    const uint32_t lo = min(lane * chunk, n), hi = min(lo + chunk, n);
    CrcPair p{0, hi - lo};
    if (hi > lo) p.crc = crc_bytes(base, off + lo, hi - lo, tab);
    for (int d = 1; d < 32; d <<= 1) {
        CrcPair o;
        o.crc = __shfl_down_sync(0xffffffffu, p.crc, d);
        o.len = __shfl_down_sync(0xffffffffu, p.len, d);
        if ((lane & (2 * d - 1)) == 0) p = crc_concat(p, o, xpow);
    }
    return p;
}

// long reads: one warp per read (the thread-per-read kernel would walk tens of kilobytes per thread)
__global__ void __launch_bounds__(128)
crc_read_warp_kernel(const uint8_t* __restrict__ acids, const uint8_t* __restrict__ quals,
                     const unsigned long long* __restrict__ read_off, const uint8_t* __restrict__ names,
                     const unsigned long long* __restrict__ name_off, uint64_t n_reads,
                     const unsigned long long* __restrict__ n_reads_dev, const int32_t* __restrict__ status,
                     const uint32_t* __restrict__ crc_tab, const uint32_t* __restrict__ xpow_g,
                     uint32_t* __restrict__ part_crc, unsigned long long* __restrict__ part_len,
                     const uint32_t* __restrict__ run_flag) {
    __shared__ uint32_t tab[256];
    __shared__ uint32_t xpow[64];
    if (status && status[0] != 0) return;
    if (run_flag && *run_flag == 0) return;
    if (n_reads_dev) n_reads = *n_reads_dev;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = crc_tab[i];
    for (int i = threadIdx.x; i < 64; i += blockDim.x) xpow[i] = xpow_g[i];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= n_reads) return;
    unsigned long long off = read_off[r];
    uint32_t len = (uint32_t)(read_off[r + 1] - off);
    CrcPair p{0, 0};
    if (names && name_off) p = crc_bytes_warp(names, name_off[r], (uint32_t)(name_off[r + 1] - name_off[r]), tab, xpow, lane);
    CrcPair a = crc_bytes_warp(acids, off, len, tab, xpow, lane);
    CrcPair q = crc_bytes_warp(quals, off, len, tab, xpow, lane);
    if (lane == 0) {
        p = crc_concat(crc_concat(p, a, xpow), q, xpow);
        part_crc[r] = p.crc;
        part_len[r] = p.len;
    }
}

// ordered tree reduction of the per-read partials of reads [r0, r1) by one 256-thread block; result in thread 0
__device__ __forceinline__ uint32_t block_crc_reduce(const uint32_t* __restrict__ part_crc,
                                                     const unsigned long long* __restrict__ part_len, uint64_t r0,
                                                     uint64_t r1, const uint32_t* __restrict__ xpow, uint32_t* s_crc,
                                                     unsigned long long* s_len) {
    uint64_t n = r1 - r0, per = (n + blockDim.x - 1) / blockDim.x;
    uint64_t c0 = r0 + threadIdx.x * per, c1 = c0 + per;
    if (c0 > r1) c0 = r1;
    if (c1 > r1) c1 = r1;
    CrcPair acc{0, 0};
    // reads of one length are the rule: keep x^(8 len) mod P of the previous length instead of rebuilding it per read
    unsigned long long last_len = 0;
    uint32_t last_pow = 0x80000000u;
    for (uint64_t r = c0; r < c1; r++) {
        const CrcPair nxt{part_crc[r], part_len[r]};
        if (nxt.len == 0) continue;
        if (acc.len == 0) {
            acc = nxt;
            continue;
        }
        if (nxt.len != last_len) {
            last_len = nxt.len;
            last_pow = x8n_mod_p(nxt.len, xpow);
        }
        acc.crc = gf2_mul(last_pow, acc.crc) ^ nxt.crc;
        acc.len += nxt.len;
    }
    s_crc[threadIdx.x] = acc.crc;
    s_len[threadIdx.x] = acc.len;
    __syncthreads();
    for (uint32_t d = 1; d < blockDim.x; d <<= 1) {  // ordered pairwise combine: [i] <- [i] ++ [i+d]
        CrcPair m{0, 0};
        bool act = (threadIdx.x % (2 * d)) == 0 && threadIdx.x + d < blockDim.x;
        if (act)
            m = crc_concat(CrcPair{s_crc[threadIdx.x], s_len[threadIdx.x]},
                           CrcPair{s_crc[threadIdx.x + d], s_len[threadIdx.x + d]}, xpow);
        __syncthreads();
        if (act) {
            s_crc[threadIdx.x] = m.crc;
            s_len[threadIdx.x] = m.len;
        }
        __syncthreads();
    }
    return s_crc[0];
}

// one thread block per container block: CRC into block_crc[] and/or the block header in `out`
__global__ void __launch_bounds__(256)
crc_block_kernel(const uint32_t* __restrict__ part_crc, const unsigned long long* __restrict__ part_len,
                 const uint32_t* __restrict__ block_first, uint32_t n_blocks, const uint32_t* __restrict__ xpow_g,
                 uint32_t* __restrict__ block_crc, uint8_t* __restrict__ out,
                 const unsigned long long* __restrict__ block_off, uint64_t out_cap) {
    __shared__ uint32_t xpow[64];
    __shared__ uint32_t s_crc[256];
    __shared__ unsigned long long s_len[256];
    for (int i = threadIdx.x; i < 64; i += blockDim.x) xpow[i] = xpow_g[i];
    __syncthreads();
    uint32_t b = blockIdx.x;
    if (b >= n_blocks) return;
    uint32_t c = block_crc_reduce(part_crc, part_len, block_first[b], block_first[b + 1], xpow, s_crc, s_len);
    if (threadIdx.x == 0) {
        if (block_crc) block_crc[b] = c;
        if (out && block_off && block_off[b] + 8 <= out_cap) {
            uint8_t* p = out + block_off[b] + 4;
            p[0] = (uint8_t)(c >> 24);
            p[1] = (uint8_t)(c >> 16);
            p[2] = (uint8_t)(c >> 8);
            p[3] = (uint8_t)c;
        }
    }
}

// decode side: compare with the block header value (IdnBlockDecompressor::check_checksum, decompressor_block.rs:131-144)
__global__ void __launch_bounds__(256)
crc_verify_kernel(const uint32_t* __restrict__ part_crc, const unsigned long long* __restrict__ part_len,
                  const uint32_t* __restrict__ block_first, uint32_t n_blocks, const uint32_t* __restrict__ xpow_g,
                  const uint32_t* __restrict__ expect, int32_t* __restrict__ status) {
    __shared__ uint32_t xpow[64];
    __shared__ uint32_t s_crc[256];
    __shared__ unsigned long long s_len[256];
    if (status[0] != 0 && status[0] != 6) return;
    for (int i = threadIdx.x; i < 64; i += blockDim.x) xpow[i] = xpow_g[i];
    __syncthreads();
    uint32_t b = blockIdx.x;
    if (b >= n_blocks) return;
    uint32_t c = block_crc_reduce(part_crc, part_len, block_first[b], block_first[b + 1], xpow, s_crc, s_len);
    if (threadIdx.x == 0 && c != expect[b]) {
        atomicCAS(&status[0], 0, 6);  // IDN_E_CHECKSUM
        atomicMin(&status[3], (int32_t)b);
    }
}

// ---------------------------------------------------------------------------------------------------
// container slice walk (decode side)   IdnBlockDecompressor::next_sequence_internal, decompressor_block.rs:115-129
// The chain "slice header -> next slice header" is serial inside a block, so ONE WARP walks one block and blocks
// run in parallel.  The warp stages the block through shared memory in tiles (coalesced 16-byte loads); lane 0
// follows the chain inside the tile (shared-memory latency per hop instead of a global round trip) and only
// records (offset, length, seq_len, models) per Sequence slice; the whole warp then turns those records into
// index entries (prefix sum of seq_len, coalesced stores).  A single pass suffices because the entries of block
// b are stored at slot_base[b] + i, slot_base = exclusive scan of the per-block upper bound len_b / 17 + 1
// (a Sequence slice is at least 9 header + 8 flush bytes); the decoder maps read -> (block, i) by binary search.
// ---------------------------------------------------------------------------------------------------
constexpr int kWalkTile = 8192;
constexpr int kWalkMaxEnt = 512;  // > kWalkTile / 17

__device__ __forceinline__ uint32_t load_u32be(const uint8_t* p) {
    return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3];
}

// Decode-side errors are reported for the first failing block in file order, whichever thread block gets there first.
// A block whose slices (compat) or lane table (native) are malformed records (block << 32 | code) with atomicMin in
// status[4..5] (~0 = none); index_check_kernel then cuts the call at that block, so the blocks in front of it are still
// decoded and checked, and finish_decode_kernel reports the lowest block among that failure, the checksum mismatches
// (status[3]) and the rANS stream errors (status[6]).
__device__ __forceinline__ unsigned long long fail_key(const int32_t* status) {
    return *reinterpret_cast<const volatile unsigned long long*>(status + 4);
}
__device__ __forceinline__ void fail_block(int32_t* status, uint32_t b, int32_t code) {
    atomicMin(reinterpret_cast<unsigned long long*>(status + 4), ((unsigned long long)b << 32) | (uint32_t)code);
}

struct ReadIndexDev {  // per-read index, strided by block (see above) or dense (idn_gpu_decompress_reads)
    unsigned long long* pay_off;  // absolute offset of the rANS payload in `payload`
    uint32_t* pay_len;
    uint32_t* seq_len;
    unsigned long long* sym_off;  // offset of the read's symbols, relative to its block's first symbol
    uint8_t* am;                  // container model indices
    uint8_t* qm;
};

// upper bound of Sequence slices per block -> slot counts (scanned by scan_tiles_kernel)
__global__ void slot_count_kernel(const unsigned long long* __restrict__ block_off, const uint32_t* __restrict__ block_len,
                                  uint32_t n_blocks, unsigned long long* __restrict__ slot_cnt) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    unsigned long long n = block_len ? block_len[b] : block_off[b + 1] - block_off[b];
    slot_cnt[b] = n / 17 + 1;
}

// The per-read index holds `cap` entries = blocks_bytes / 17 + n_blocks + 1, enough for any set of DISJOINT blocks inside
// the input region.  Blocks that overlap (only a caller of the _dev entry points can pass such a table; the host-pointer
// calls reject it) could ask for more: refuse the call instead of writing past the index.
__global__ void slot_cap_check_kernel(const unsigned long long* __restrict__ slot_total, unsigned long long cap,
                                      int32_t* __restrict__ status) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && *slot_total > cap) {
        status[0] = 12;  // IDN_E_INVALID_ARG
        status[1] = -1;
    }
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// stage kWalkTile + 16 bytes starting at the 16-byte aligned absolute address A into `tile` (asynchronously where the
// 16-byte chunk lies completely inside the caller's buffer, byte by byte with zero fill at its two ends)
__device__ __forceinline__ void walk_stage(uint8_t* tile, uintptr_t A, uintptr_t lo16, uintptr_t hi16, uintptr_t buf_lo,
                                           uintptr_t buf_hi, uint32_t lane) {
#pragma unroll 1
    for (uint32_t k = lane; k < kWalkTile / 16 + 1; k += 32) {
        uintptr_t addr = A + 16ull * k;
        if (addr >= lo16 && addr + 16 <= hi16) {
            cp_async16(tile + 16 * k, reinterpret_cast<const void*>(addr));
        } else {
            uint32_t w[4] = {0, 0, 0, 0};
            for (int j = 0; j < 16; j++) {
                uintptr_t p = addr + j;
                if (p >= buf_lo && p < buf_hi) w[j >> 2] |= (uint32_t)(*reinterpret_cast<const uint8_t*>(p)) << (8 * (j & 3));
            }
            *reinterpret_cast<uint4*>(tile + 16 * k) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
    cp_async_commit();
}

__global__ void __launch_bounds__(32)
walk_kernel(const uint8_t* __restrict__ blocks, const unsigned long long* __restrict__ block_off,
            const uint32_t* __restrict__ block_len, uint32_t n_blocks, unsigned long long blocks_bytes,
            const uint8_t* __restrict__ model_type /*[n_models] by container index*/, uint32_t n_models,
            const unsigned long long* __restrict__ slot_base, ReadIndexDev ix, unsigned long long* __restrict__ blk_reads,
            unsigned long long* __restrict__ blk_syms, int32_t* __restrict__ status /*SmallParams::status*/,
            const uint8_t* __restrict__ done /*blocks walk_fast_kernel has indexed, or nullptr*/) {
    __shared__ __align__(16) uint8_t tiles[2][kWalkTile + 32];
    __shared__ uint16_t plist[kWalkMaxEnt];  // tile offsets of the slice headers found in the current tile
    const uint32_t b = blockIdx.x, lane = threadIdx.x;
    if (b >= n_blocks) return;
    if (status[0] == 12) return;  // slot_cap_check_kernel refused the block table
    if (done && done[b]) return;
    const unsigned long long boff = block_off[b];
    const unsigned long long n = block_len ? block_len[b] : block_off[b + 1] - boff;
    int32_t st = 0;
    if (boff > blocks_bytes || n > blocks_bytes - boff || n > 0xffffffffull) st = 3;  // runs past the input: malformed
    // 16-byte chunks that lie completely inside the caller's buffer may be copied as vectors
    const uintptr_t buf_lo = reinterpret_cast<uintptr_t>(blocks), buf_hi = buf_lo + blocks_bytes;
    const uintptr_t lo16 = (buf_lo + 15) & ~(uintptr_t)15, hi16 = buf_hi & ~(uintptr_t)15;
    const uintptr_t blk_abs = buf_lo + boff;

    unsigned long long pos = 0;  // block-relative position of the next slice header
    unsigned long long n_reads = 0, n_syms = 0;
    uint32_t mdl = 0xffffu;      // active models: acid | q << 8, 0xff = none yet (container indices are < 255)
    const unsigned long long slot0 = slot_base[b];
    uint32_t cur = 0;
    uintptr_t A = blk_abs & ~(uintptr_t)15;  // absolute address of tile[0] of the current buffer
    if (st == 0 && n > 0) walk_stage(tiles[0], A, lo16, hi16, buf_lo, buf_hi, lane);
    while (st == 0 && pos < n) {
        // prefetch the tile that follows on the assumption that the walk ends within 16 bytes of this tile's end
        const uintptr_t A_next = A + kWalkTile - 16;
        walk_stage(tiles[cur ^ 1], A_next, lo16, hi16, buf_lo, buf_hi, lane);
        cp_async_wait<1>();
        __syncwarp();
        const uint8_t* tile = tiles[cur];
        const uint32_t* tw = reinterpret_cast<const uint32_t*>(tile);
        // block positions [t_lo, t_lo + kStaged) are staged in tile[]; t_lo may lie before the block (alignment)
        const long long t_lo = (long long)(A - blk_abs);
        const uint32_t kStaged = kWalkTile + 16;
        const uint32_t p0 = (uint32_t)((long long)pos - t_lo);  // tile offset of the first header
        const unsigned long long left = n - pos;                // bytes of the block from pos on
        // clamped, so that a bound accepted in 32 bits is always a true bound; rejections are rechecked in 64 bits
        const uint32_t n_off = p0 + (uint32_t)(left > 0x40000000ull ? 0x40000000ull : left);
        // ---- lane 0 chases the chain and does nothing else: one thread's dependent-instruction latency bounds this
        // loop, so validation, model tracking and index building are left to the whole warp below ----
        uint32_t n_hdr = 0, p_end = p0;
        if (lane == 0) {
            // the dependent chain per hop is p -> shared-memory load -> byte permute -> add: a Sequence slice (the rule) goes
            // straight to p + 9 + length, every other slice type takes the side exit
            uint32_t p = p0;
            while (p < n_off && n_hdr < (uint32_t)kWalkMaxEnt && p + 9 <= kStaged) {
                const uint32_t wi = p >> 2, sh = p & 3;
                const uint32_t W0 = tw[wi], W1 = tw[wi + 1];
                const uint32_t w1 = __byte_perm(W0, W1, 0x1234u + sh * 0x1111u);  // bytes p+1 .. p+4, big endian
                const uint32_t kind = (W0 >> (8 * sh)) & 0xffu;
                plist[n_hdr++] = (uint16_t)p;
                if (kind == 2 && w1 <= 0x7fff0000u) {  // Sequence: 9 + length
                    p = p + 9u + w1;
                    continue;
                }
                // SwitchModel: 2; Identifiers: 6 + length; anything else, or a length that cannot be real, stops the
                // chain here (the warp reports it)
                uint32_t step = kind == 1 ? 2u : 6u + w1;
                if (kind > 2 || w1 > 0x7fff0000u) step = 0x7fffffffu;
                p = p + step > p ? p + step : 0x7fffffffu;
            }
            p_end = p;
        }
        n_hdr = __shfl_sync(0xffffffffu, n_hdr, 0);
        p_end = __shfl_sync(0xffffffffu, p_end, 0);
        // ---- the warp: re-read every header, validate, track the active models, emit index entries ----
        for (uint32_t base = 0; base < n_hdr && st == 0; base += 32) {
            const uint32_t i = base + lane;
            const bool have = i < n_hdr;
            uint32_t kind = 0xff, w1 = 0, w2 = 0, p = 0, bad = 0;
            if (have) {
                p = plist[i];
                const uint32_t wi = p >> 2, sh = p & 3;
                const uint32_t W0 = tw[wi], W1 = tw[wi + 1], W2 = tw[wi + 2];
                const uint32_t sel = 0x1234u + sh * 0x1111u;
                kind = (W0 >> (8 * sh)) & 0xffu;
                w1 = __byte_perm(W0, W1, sel);
                w2 = __byte_perm(W1, W2, sel);
                const unsigned long long room = n - (unsigned long long)((long long)p + t_lo);  // bytes from this header on
                if (kind == 2) {  // Sequence: u32 length, u32 seq_len, payload   (data.rs:79-84, decompressor_block.rs:216-239)
                    if (room < 9 || w1 > room - 9 || w1 < 8) bad = 3;
                } else if (kind == 1) {  // SwitchModel: u8 index   (decompressor_block.rs:194-214)
                    if (room < 2) bad = 3;
                    else if ((w1 >> 24) >= n_models || (w1 >> 24) >= 255) bad = 7;
                } else if (kind == 0) {  // Identifiers: u32 length, u8 compression, data -- names stay on the host
                    if (room < 6 || w1 > room - 6) bad = 3;
                } else {
                    bad = 3;
                }
            }
            // active models at every header: inclusive scan of "the right operand overrides what it sets"
            uint32_t set = 0xffffu;  // what this slice sets: acid | q << 8, 0xff = nothing
            if (have && kind == 1 && !bad) {
                const uint32_t idx = w1 >> 24;
                set = model_type[idx] == 0 ? (0xff00u | idx) : (0x00ffu | (idx << 8));
            }
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, set, d);
                if (lane >= (uint32_t)d) {
                    const uint32_t a = (set & 0xffu) != 0xffu ? (set & 0xffu) : (o & 0xffu);
                    const uint32_t q = (set & 0xff00u) != 0xff00u ? (set & 0xff00u) : (o & 0xff00u);
                    set = a | q;
                }
            }
            uint32_t act = ((set & 0xffu) != 0xffu ? (set & 0xffu) : (mdl & 0xffu)) |
                           ((set & 0xff00u) != 0xff00u ? (set & 0xff00u) : (mdl & 0xff00u));
            if (have && kind == 2 && !bad && ((act & 0xffu) == 0xffu || (act >> 8) == 0xffu)) bad = 8;  // NoActiveModel
            mdl = __shfl_sync(0xffffffffu, act, 31);
            // the first bad header decides the status (headers are in chain order)
            const uint32_t bad_mask = __ballot_sync(0xffffffffu, bad != 0);
            if (bad_mask) st = __shfl_sync(0xffffffffu, (int32_t)bad, __ffs(bad_mask) - 1);
            const uint32_t ok_before = bad_mask ? ((1u << (__ffs(bad_mask) - 1)) - 1) : 0xffffffffu;
            const bool is_seq = have && kind == 2 && ((ok_before >> lane) & 1u);
            const uint32_t seq_mask = __ballot_sync(0xffffffffu, is_seq);
            unsigned long long sl = is_seq ? w2 : 0, inc = sl;
            for (int d = 1; d < 32; d <<= 1) {
                unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= (uint32_t)d) inc += o;
            }
            if (is_seq) {
                const unsigned long long slot = slot0 + n_reads + __popc(seq_mask & ((1u << lane) - 1));
                ix.pay_off[slot] = boff + (unsigned long long)(t_lo + (long long)p + 9);
                ix.pay_len[slot] = w1;
                ix.seq_len[slot] = w2;
                ix.sym_off[slot] = n_syms + inc - sl;
                ix.am[slot] = (uint8_t)(act & 0xffu);
                ix.qm[slot] = (uint8_t)(act >> 8);
            }
            n_syms += __shfl_sync(0xffffffffu, inc, 31);
            n_reads += __popc(seq_mask);
        }
        if (st == 0) {
            if (p_end >= 0x7fffffffu) st = 3;  // the chain stopped on a header the warp did not flag: cannot happen, but never walk on
            else pos = (unsigned long long)((long long)p_end + t_lo);
        }
        __syncwarp();
        if (st != 0 || pos >= n) break;
        // the prefetched tile serves when the next header starts inside it (and the walk can make progress)
        const long long nt_lo = (long long)(A_next - blk_abs);
        if ((long long)pos >= nt_lo && (long long)pos + 9 <= nt_lo + kWalkTile + 16) {
            A = A_next;
            cur ^= 1;
        } else {
            cp_async_wait<0>();  // the speculative copy must land before its buffer is reused
            __syncwarp();
            A = (blk_abs + pos) & ~(uintptr_t)15;
            walk_stage(tiles[cur], A, lo16, hi16, buf_lo, buf_hi, lane);
        }
    }
    cp_async_wait<0>();
    if (lane == 0) {
        blk_reads[b] = n_reads;
        blk_syms[b] = n_syms;
        if (st != 0) fail_block(status, b, st);
    }
}

// ---------------------------------------------------------------------------------------------------
// Parallel slice walk.  The chain "header -> next header" of a block is serial, but a chain can be entered at any true
// slice boundary, and a false boundary almost never survives a few hops (every hop must find a legal slice type and a
// length that stays inside the block).  128 threads cut the block into segments; each looks for the first Sequence
// header in its segment that survives kWalkDepth hops, follows the chain from there up to the next thread's start and
// counts; the pieces are accepted only if they join exactly (thread t ends where the next start lies, the last ends
// at the block's end) and every header on the way is valid.  Then a prefix sum gives every piece its first read
// ordinal / symbol offset / active models and the pieces are walked again to write the index.
// Cost: two passes of small scattered reads over the container, i.e. DRAM-access-rate bound (~2.2 us per MB measured),
// while the serial walk costs ~1.2 us per KB of the LARGEST block whatever the number of blocks: the host picks this
// kernel for calls of fewer than kWalkFastMaxBlocks blocks (the e2e path's 32-block calls: 3.9 -> 0.2 ms).
// Anything else -- a malformed block, a false start that survived (slice look-alikes inside an Identifiers slice), a
// Sequence slice before any SwitchModel -- leaves done[b] = 0 and walk_kernel does that block the serial way, which
// also keeps every error code where it was.
// ---------------------------------------------------------------------------------------------------
constexpr int kWalkFastThreads = 128;
constexpr int kWalkDepth = 6;
constexpr uint32_t kWalkFastMaxBlocks = 512;
constexpr int kWalkFixRounds = 8;  // false starts dropped per block before the serial walk takes over
constexpr unsigned long long kWalkNone = ~0ull;

struct WalkHdr {
    uint32_t kind, w1, w2;
};

// the 9 bytes at absolute address a (kind, u32be, u32be); bytes outside the caller's buffer read as zero
__device__ __forceinline__ WalkHdr walk_load_hdr(uintptr_t a, uintptr_t buf_lo, uintptr_t buf_hi) {
    const uintptr_t A = a & ~(uintptr_t)7;
    unsigned long long q0 = 0, q1 = 0;
    if (A >= buf_lo && A + 16 <= buf_hi) {
        q0 = __ldg(reinterpret_cast<const unsigned long long*>(A));
        q1 = __ldg(reinterpret_cast<const unsigned long long*>(A + 8));
    } else {
        for (int j = 0; j < 16; j++) {
            const uintptr_t pa = A + j;
            unsigned long long v = (pa >= buf_lo && pa < buf_hi) ? *reinterpret_cast<const uint8_t*>(pa) : 0;
            if (j < 8) q0 |= v << (8 * j);
            else q1 |= v << (8 * (j - 8));
        }
    }
    const uint32_t sh = 8 * (uint32_t)(a & 7);
    const unsigned long long lo = sh ? (q0 >> sh) | (q1 << (64 - sh)) : q0;  // bytes a .. a+7
    const uint32_t b8 = (uint32_t)(q1 >> sh) & 0xffu;                        // byte a+8
    WalkHdr h;
    h.kind = (uint32_t)lo & 0xffu;
    h.w1 = __byte_perm((uint32_t)(lo >> 8), 0, 0x0123);
    h.w2 = __byte_perm((uint32_t)(lo >> 40) | (b8 << 24), 0, 0x0123);
    return h;
}

// size of the slice whose header is h with `room` bytes left in the block, 0 when it is not a legal slice
// (the same rules as walk_kernel)
__device__ __forceinline__ unsigned long long walk_slice_size(const WalkHdr& h, unsigned long long room, uint32_t n_models) {
    if (h.kind == 2) return (room < 9 || h.w1 < 8 || h.w1 > room - 9) ? 0 : 9ull + h.w1;
    if (h.kind == 1) return (room < 2 || (h.w1 >> 24) >= n_models || (h.w1 >> 24) >= 255) ? 0 : 2ull;
    if (h.kind == 0) return (room < 6 || h.w1 > room - 6) ? 0 : 6ull + h.w1;
    return 0;
}

__global__ void __launch_bounds__(kWalkFastThreads)
walk_fast_kernel(const uint8_t* __restrict__ blocks, const unsigned long long* __restrict__ block_off,
                 const uint32_t* __restrict__ block_len, uint32_t n_blocks, unsigned long long blocks_bytes,
                 const uint8_t* __restrict__ model_type, uint32_t n_models, const unsigned long long* __restrict__ slot_base,
                 ReadIndexDev ix, unsigned long long* __restrict__ blk_reads, unsigned long long* __restrict__ blk_syms,
                 uint8_t* __restrict__ done, const int32_t* __restrict__ status) {
    __shared__ unsigned long long s_start[kWalkFastThreads];
    __shared__ unsigned long long s_syms[kWalkFastThreads];
    __shared__ uint32_t s_cnt[kWalkFastThreads];
    __shared__ uint32_t s_set[kWalkFastThreads];   // models set inside the piece: acid | q << 8, 0xff = none
    __shared__ int s_fail, s_giveup;
    const uint32_t b = blockIdx.x, t = threadIdx.x;
    if (b >= n_blocks) return;
    if (t == 0) done[b] = 0;
    if (status[0] == 12) return;  // uniform: written by an earlier kernel of the stream
    const unsigned long long boff = block_off[b];
    const unsigned long long n = block_len ? block_len[b] : block_off[b + 1] - boff;
    if (boff > blocks_bytes || n > blocks_bytes - boff || n > 0xffffffffull) return;  // walk_kernel reports it
    const uintptr_t buf_lo = reinterpret_cast<uintptr_t>(blocks), buf_hi = buf_lo + blocks_bytes;
    const uintptr_t blk = buf_lo + boff;
    const uint8_t* bytes = blocks + boff;

    // 1. a start per segment
    const unsigned long long seg = max(64ull, (n + kWalkFastThreads - 1) / kWalkFastThreads);
    const unsigned long long g0 = min(n, (unsigned long long)t * seg), g1 = min(n, g0 + seg);
    unsigned long long start = kWalkNone;
    if (t == 0) {
        start = 0;
    } else {
        for (unsigned long long p = g0; p < g1; p++) {
            if (__ldg(bytes + p) != 2) continue;
            unsigned long long q = p;
            bool good = true;
            for (int hop = 0; hop < kWalkDepth && q < n; hop++) {
                const unsigned long long sz = walk_slice_size(walk_load_hdr(blk + q, buf_lo, buf_hi), n - q, n_models);
                if (!sz) {
                    good = false;
                    break;
                }
                q += sz;
            }
            if (good) {
                start = p;
                break;
            }
        }
    }
    s_start[t] = start;
    if (t == 0) {
        s_fail = kWalkFastThreads;
        s_giveup = 0;
    }
    __syncthreads();

    // 2. count along the piece [start, next), next = the following thread's start.  A start that only LOOKS true can
    // survive the hop test by landing on a true header (e.g. a payload that ends "02 00 00" in front of a header
    // "02 00 ..." reads as a Sequence slice of 512 bytes): then the piece before it overshoots it.  Thread 0 starts at
    // the true beginning, so the lowest thread whose piece does not end at `next` is on the true chain and its overshoot
    // proves that `next` is false: that start is dropped and the piece is extended, one false start per round.
    unsigned long long next = n, piece_next = kWalkNone;
    uint32_t cnt = 0, set = 0xffffu, need = 0;  // need bit 0 / 1: a Sequence slice came before the piece set an acid / q model
    unsigned long long syms = 0, p = 0;
    uint32_t state = 0;  // 0 joins, 1 valid headers but the piece ends past `next`, 2 an invalid header
    bool all_ok = false;
    for (int round = 0; round < kWalkFixRounds; round++) {
        start = s_start[t];
        next = n;  // where the following piece starts
        for (uint32_t j = t + 1; j < (uint32_t)kWalkFastThreads; j++)
            if (s_start[j] != kWalkNone) {
                next = s_start[j];
                break;
            }
        if (start == kWalkNone) {
            state = 0;
            cnt = 0;
            syms = 0;
            set = 0xffffu;
            need = 0;
        } else if (next != piece_next) {  // first round, or the piece grew
            piece_next = next;
            cnt = 0;
            syms = 0;
            set = 0xffffu;
            need = 0;
            state = 0;
            p = start;
            while (p < next) {
                const WalkHdr h = walk_load_hdr(blk + p, buf_lo, buf_hi);
                const unsigned long long sz = walk_slice_size(h, n - p, n_models);
                if (!sz) {
                    state = 2;
                    break;
                }
                if (h.kind == 2) {
                    cnt++;
                    syms += h.w2;
                    need |= ((set & 0xffu) == 0xffu ? 1u : 0u) | ((set >> 8) == 0xffu ? 2u : 0u);
                } else if (h.kind == 1) {
                    const uint32_t idx = h.w1 >> 24;
                    set = model_type[idx] == 0 ? ((set & 0xff00u) | idx) : ((set & 0x00ffu) | (idx << 8));
                }
                p += sz;
            }
            if (state == 0 && p != next) state = 1;
        }
        if (state) atomicMin(&s_fail, (int)t);
        __syncthreads();
        const int f = s_fail;
        __syncthreads();  // everybody has read s_fail before thread f resets it
        if (f == kWalkFastThreads) {
            all_ok = true;
            break;
        }
        if ((int)t == f) {
            if (state == 1 && next != n) {
                for (uint32_t j = t + 1; j < (uint32_t)kWalkFastThreads; j++)
                    if (s_start[j] == next) {
                        s_start[j] = kWalkNone;
                        break;
                    }
            } else {
                s_giveup = 1;  // a bad header on the true chain, or a chain that runs past the block: walk_kernel reports it
            }
            s_fail = kWalkFastThreads;
        }
        __syncthreads();
        if (s_giveup) return;  // done[b] stays 0
    }
    if (!all_ok) return;
    s_cnt[t] = cnt;
    s_syms[t] = syms;
    s_set[t] = set;
    __syncthreads();

    // 3. what the piece starts with: reads and symbols before it, models active when it is entered
    unsigned long long first_read = 0, first_sym = 0;
    uint32_t act = 0xffffu;
    for (uint32_t j = 0; j < t; j++) {
        first_read += s_cnt[j];
        first_sym += s_syms[j];
        const uint32_t sj = s_set[j];
        act = ((sj & 0xffu) != 0xffu ? (sj & 0xffu) : (act & 0xffu)) | ((sj & 0xff00u) != 0xff00u ? (sj & 0xff00u) : (act & 0xff00u));
    }
    const bool active_ok = !(((need & 1u) && (act & 0xffu) == 0xffu) || ((need & 2u) && (act >> 8) == 0xffu));
    if (!__syncthreads_and(active_ok)) return;  // NoActiveModel: walk_kernel reports it

    // 4. the index entries of the piece
    if (start != kWalkNone) {
        const unsigned long long slot0 = slot_base[b] + first_read;
        unsigned long long i = 0, so = first_sym;
        p = start;
        while (p < next) {
            const WalkHdr h = walk_load_hdr(blk + p, buf_lo, buf_hi);
            if (h.kind == 2) {
                ix.pay_off[slot0 + i] = boff + p + 9;
                ix.pay_len[slot0 + i] = h.w1;
                ix.seq_len[slot0 + i] = h.w2;
                ix.sym_off[slot0 + i] = so;
                ix.am[slot0 + i] = (uint8_t)(act & 0xffu);
                ix.qm[slot0 + i] = (uint8_t)(act >> 8);
                so += h.w2;
                i++;
            } else if (h.kind == 1) {
                const uint32_t idx = h.w1 >> 24;
                act = model_type[idx] == 0 ? ((act & 0xff00u) | idx) : ((act & 0x00ffu) | (idx << 8));
            }
            p += walk_slice_size(h, n - p, n_models);
        }
    }
    if (t == kWalkFastThreads - 1) {
        blk_reads[b] = first_read + cnt;
        blk_syms[b] = first_sym + syms;
        done[b] = 1;
    }
}

// totals against the caller's capacities + u32 block_first for the CRC kernels; on failure every later kernel of the
// call is a no-op.  A block f that failed its walk / lane table cuts the call: the scans of reads, symbols and index slots
// (lanes) stop at f, so the decoders and the CRC check see blocks [0, f) only.
__global__ void __launch_bounds__(256)
index_check_kernel(unsigned long long* __restrict__ blk_reads, unsigned long long* __restrict__ blk_syms,
                   unsigned long long* __restrict__ blk_slots, uint32_t n_blocks, uint64_t reads_cap, uint64_t syms_cap,
                   uint32_t* __restrict__ block_first, int32_t* __restrict__ status) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long key = fail_key(status);
    const uint32_t f = key == ~0ull ? n_blocks : (uint32_t)(key >> 32);  // (entry f itself is never written here)
    if (i <= n_blocks) {
        if (i > f) {
            blk_reads[i] = blk_reads[f];
            blk_syms[i] = blk_syms[f];
            blk_slots[i] = blk_slots[f];
        }
        if (block_first) block_first[i] = (uint32_t)blk_reads[i < f ? i : f];
    }
    if (i != 0) return;
    status[3] = 0x7fffffff;  // first block with a checksum mismatch
    if (status[0] != 0) return;
    if (blk_reads[f] > reads_cap || blk_syms[f] > syms_cap) {
        if (f < n_blocks) {  // the blocks in front of the failing one do not fit: its failure stands
            status[0] = (int32_t)(uint32_t)key;
            status[1] = (int32_t)f;
            return;
        }
        status[0] = 11;  // IDN_E_NOSPACE
        status[1] = -1;
        status[2] = (int32_t)(blk_reads[n_blocks] > 0x7fffffffull ? 0x7fffffff : blk_reads[n_blocks]);
    }
}

struct IdentU64 {
    const unsigned long long* v;
    __device__ __forceinline__ unsigned long long operator()(uint64_t i) const { return v[i]; }
};

// ---------------------------------------------------------------------------------------------------
// K5: two-state per-read rANS decode.  One thread per read.
// status bits: 1 = payload exhausted / malformed, 2 = the stream does not end cleanly (final states != L or bytes left
// over).  Both fail the call with IDN_E_SERIALIZE, in compat and in native mode alike: a valid encoder output always ends
// with both states back at L and every payload byte consumed (RansEncFlush / RansDecInit symmetry), so anything else is a
// garbled payload even when no block CRC was supplied to catch it.
// ---------------------------------------------------------------------------------------------------
struct DecodeArgs {
    const ModelDev* models;
    const int32_t* model_ids;  // container index -> models[]
    const uint8_t* payload;
    ReadIndexDev ix;
    // block-strided index (walk_kernel): read r -> block b by binary search over blk_read_base[0..n_blocks], entry at
    // slot_base[b] + (r - blk_read_base[b]); nullptr = dense index, entry r, sym_off absolute
    const unsigned long long* blk_read_base;
    const unsigned long long* blk_sym_base;
    const unsigned long long* slot_base;
    uint32_t n_blocks;
    uint64_t n_reads;                       // dense form only
    const int32_t* status;                  // when set and != 0 the kernel does nothing
    uint8_t* acids_out;
    uint8_t* quals_out;
    long long out_dq;                       // quals_out - acids_out
    unsigned long long* read_off_out;       // optional [n_reads+1]: absolute symbol offset of every read
    uint32_t* read_status;  // optional
    uint32_t* err;
    int32_t* err_block;     // optional (block-strided index): atomicMin of the block of a read whose stream fails
    // optional: CRC-32 partial of every decoded read (acids | quals), the input of crc_verify_kernel, computed while the
    // symbols are in registers instead of by a second pass over the output (K7 fused into K5)
    uint32_t* part_crc;
    unsigned long long* part_len;
    const uint32_t* crc_tab;  // [256]
    const uint32_t* xpow;     // [64]
};

// State of one rANS input stream being consumed (a read in compat mode, a lane in native mode).
//
// The payload is read through a 64-bit window: `w` holds the next `bits` (>= 32 at the top of every position) unread
// payload bits, next byte lowest; one position consumes at most 4 bytes (two per state), so one conditional refill per
// position suffices, and the word that refill shifts in was loaded one refill earlier (`nextw`), i.e. the payload load
// is never on the state -> slot -> symbol -> context chain.  Renormalisation is branch-free: the number of bytes a state
// needs (0, 1 or 2: x >= 2^9 after RansDecAdvanceStep) picks a byte-permute selector that shifts the state and drops
// the bytes in at once.  Past the end of the payload the window is fed zeros; finish() reports that afterwards.
struct DecStream {
    uint32_t xq, xa;          // decoder state 0 = quality scores, state 1 = acids (compressor.rs:181-182)
    unsigned long long w;     // unread payload bytes, next byte in bits 0..7
    uint32_t bits;            // valid bits in w
    uint32_t nextw;           // the word that follows the window
    const uint32_t* wp;       // the word after nextw
    int32_t wleft;            // payload words from wp on (<= 0: past the end, zeros are fed)
    uint32_t lowest;          // minimum over the renormalised states; < L: the stream is malformed
    uint32_t st, cur;         // set by finish(): st bit 0 = the payload ran out / is malformed, cur = bytes consumed
    __device__ __forceinline__ uint32_t load_word() {
        uint32_t v = 0;
        if (wleft > 0) v = __ldg(wp);
        wp++;
        wleft--;
        return v;
    }
    __device__ __forceinline__ void begin(const uint8_t* payload, unsigned long long off, uint32_t len) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(payload + off);
        const uint32_t skip = (uint32_t)(a & 3);
        wp = reinterpret_cast<const uint32_t*>(a - skip);
        wleft = len < 8 ? 0 : (int32_t)((skip + len + 3) >> 2);  // a valid stream holds at least the two flushed states
        const uint32_t w0 = load_word(), w1 = load_word(), w2 = load_word();
        nextw = load_word();
        const uint32_t sh = 8 * skip;
        xq = __funnelshift_r(w0, w1, sh);  // RansDecInit x2: little-endian state 0, then state 1
        xa = __funnelshift_r(w1, w2, sh);
        w = w2 >> sh;
        bits = 32 - sh;
        lowest = 0xffffffffu;
        st = 0;
        cur = 0;
    }
    __device__ __forceinline__ void refill() {
        if (bits < 32) {
            w |= (unsigned long long)nextw << bits;
            bits += 32;
            nextw = load_word();
        }
    }
    // RansDecRenorm: while (x < L) x = (x << 8) | *ptr++   -- at most two rounds here
    __device__ __forceinline__ void renorm(uint32_t& x) {
        const bool one = x < kRansL, two = x < (1u << 15);
        const uint32_t sel = two ? 0x5401u : (one ? 0x6540u : 0x7654u);  // [w1 w0 x0 x1] / [w0 x0 x1 x2] / x
        const uint32_t sh = two ? 16u : (one ? 8u : 0u);
        x = __byte_perm((uint32_t)w, x, sel);
        w >>= sh;
        bits -= sh;
    }
    __device__ __forceinline__ void renorm_all() {  // state 0 then state 1 (compressor.rs:188-189)
        renorm(xq);
        renorm(xa);
        lowest = min(lowest, min(xq, xa));
    }
    __device__ __forceinline__ void finish(const uint8_t* payload, unsigned long long off, uint32_t len) {
        const uint32_t skip = (uint32_t)(reinterpret_cast<uintptr_t>(payload + off) & 3);
        const int32_t nw = len < 8 ? 0 : (int32_t)((skip + len + 3) >> 2);
        const int32_t in_window = nw - wleft - 1;  // words shifted into the window so far (nextw is not)
        const int32_t used = 4 * in_window - (int32_t)skip - (int32_t)(bits >> 3);
        cur = (uint32_t)used;
        st = (len < 8 || used > (int32_t)len || lowest < kRansL) ? 1u : 0u;
    }
    // a valid stream ends with both states back at L and every byte consumed
    __device__ __forceinline__ bool clean_end(uint32_t len) const { return xq == kRansL && xa == kRansL && cur == len; }
};

// Decoded symbols of consecutive positions.  Bytes at the ragged ends of a read (the words it shares with its neighbours),
// whole words in between; full words are collected four at a time and leave as ONE 16-byte store per stream wherever the
// two output addresses are 16-byte aligned together.  A thread's stores are 32 scattered sectors per warp request, and
// the codec kernels are bound by the number of such requests (l1tex data-pipe wavefronts, profiles/r2_ncu_*.md): 16 bytes
// per request instead of 4 cuts the store requests of the decoder fourfold and fills a 32-byte sector in two writes
// instead of eight (less read-modify-write traffic at the DRAM).  IDN_NO_SYM16 keeps the round-1 word stores for A/B runs.
struct SymWriter {
    uint8_t* pa;     // acids; the quality scores go to pa + dq
    long long dq;    // quals_out - acids_out: a kernel parameter (constant-bank operand, no registers)
#ifndef IDN_NO_SYM16
    uint32_t an_lo, an_hi;    // pending acid words as nibbles (an acid is 0..4): word k of the pending four in bits 16k..16k+15
    uint32_t q0, q1, q2, q3;  // pending quality-score words, oldest first: the last `nw` count
    uint32_t nw;              // pending words (0..3); they end at pa; bit 31 = "pa and pa + dq share their phase modulo 16"
#endif
    __device__ __forceinline__ void init(uint8_t* a, long long dq_) {
        pa = a;
        dq = dq_;
#ifndef IDN_NO_SYM16
        an_lo = an_hi = q0 = q1 = q2 = q3 = 0;
        nw = (dq_ & 15) == 0 ? 0x80000000u : 0u;
#endif
    }
    __device__ __forceinline__ bool aligned() const {
        return ((reinterpret_cast<uintptr_t>(pa) | (uintptr_t)dq) & 3) == 0;
    }
#ifndef IDN_NO_SYM16
    // four acids as nibbles (16 bits) <-> one byte each
    static __device__ __forceinline__ uint32_t pack4(uint32_t w) {
        const uint32_t t = w | (w >> 4);          // byte 0 = b0 | b1 << 4, byte 2 = b2 | b3 << 4
        return __byte_perm(t, 0, 0x4420);         // bytes 0 and 2 -> bits 0..15
    }
    static __device__ __forceinline__ uint32_t unpack4(uint32_t n16) {  // n16 in bits 0..15
        const uint32_t t = __byte_perm(n16, 0, 0x4140);  // byte 0 -> byte 0, byte 1 -> byte 2
        return (t | (t << 4)) & 0x0f0f0f0fu;
    }
    // the pending words, one store each (end of a read / lane, or a byte store is about to open a gap)
    __device__ __forceinline__ void flush() {
        const uint32_t k = nw & 3u;
        uint32_t* wa = reinterpret_cast<uint32_t*>(pa);
        uint32_t* wq = reinterpret_cast<uint32_t*>(pa + dq);
        if (k == 3) {
            wa[-3] = unpack4(an_lo >> 16);
            wq[-3] = q1;
        }
        if (k >= 2) {
            wa[-2] = unpack4(an_hi & 0xffffu);
            wq[-2] = q2;
        }
        if (k >= 1) {
            wa[-1] = unpack4(an_hi >> 16);
            wq[-1] = q3;
        }
        nw &= 0x80000000u;
    }
#else
    __device__ __forceinline__ void flush() {}
#endif
    __device__ __forceinline__ void put(uint32_t a, uint32_t q) {
#ifndef IDN_NO_SYM16
        if (nw & 3u) flush();
#endif
        pa[0] = (uint8_t)a;
        pa[dq] = (uint8_t)q;
        pa++;
    }
    __device__ __forceinline__ void put4(uint32_t wa, uint32_t wq) {  // both addresses are word-aligned
#ifdef IDN_ABL_NOSTORE
        if (wa != 0xdeadbeefu) { pa += 4; return; }
#endif
#ifndef IDN_NO_SYM16
        if ((nw & 3u) || (nw && (reinterpret_cast<uintptr_t>(pa) & 15) == 0)) {
            an_lo = __funnelshift_r(an_lo, an_hi, 16);
            an_hi = __byte_perm(an_hi, pack4(wa), 0x5432);  // (an_hi >> 16) | pack << 16
            q0 = q1; q1 = q2; q2 = q3; q3 = wq;
            pa += 4;
            nw++;
            if ((nw & 7u) == 4) {
                *reinterpret_cast<uint4*>(pa - 16) = make_uint4(unpack4(an_lo & 0xffffu), unpack4(an_lo >> 16),
                                                                unpack4(an_hi & 0xffffu), unpack4(an_hi >> 16));
                *reinterpret_cast<uint4*>(pa + dq - 16) = make_uint4(q0, q1, q2, q3);
                nw &= 0x80000000u;
            }
            return;
        }
#endif
        *reinterpret_cast<uint32_t*>(pa) = wa;
        *reinterpret_cast<uint32_t*>(pa + dq) = wq;
        pa += 4;
    }
};

// Pops one read (positions 0 .. len-1) from the stream   SequenceDecompressor::decompress, sequence_compressor.rs:231-278
// crc_tab: shared-memory CRC table, or nullptr; ca / cq: running (pre-inversion) CRC registers of the two symbol streams
struct DecCrc {
    const uint32_t* tab;
    uint32_t ca, cq;
};

// positions p0 .. p1-1 of a read of `len` symbols (the whole read: p0 = 0, p1 = len).  p0 > 0 (native format, a lane that
// starts inside a long read): hist[0 .. kHist) are the acids and hist[kHist .. 2 kHist) the quality scores of the kHist
// positions in front of p0, from which the generator states are rebuilt (no legal spec type looks further back).
template <class P>
__device__ __forceinline__ void decode_read_body(const ModelDev& ma, const ModelDev& mq, uint32_t len, uint32_t p0, uint32_t p1,
                                                 const uint8_t* __restrict__ hist, DecStream& D, SymWriter& O, DecCrc& C) {
    constexpr SpecDev ksa = P::sa(), ksq = P::sq();
    const SpecDev& sa = P::kStatic ? ksa : ma.spec;
    const SpecDev& sq = P::kStatic ? ksq : mq.spec;
    GenFwd ga, gq;
    ga.init();
    gq.init();
    const uint32_t pbmax = sa.pb > sq.pb ? sa.pb : sq.pb;
    const uint32_t psa = pbmax - sa.pb, psq = pbmax - sq.pb;
    PosFwd pf;
    pf.init_at(len, pbmax, p0);
    if (p0) {
#pragma unroll 1
        for (int k = 0; k < kHist; k++) {
            uint32_t ha = __ldg(hist + k), hq = __ldg(hist + kHist + k);
            ha = ha > 4 ? 0 : ha;   // (a garbled history cannot index outside the tables; the CRC / clean-end checks report it)
            hq = hq > 93 ? 0 : hq;
            const bool hz = ha * hq == 0;
            ga.update(sa, ha, hq, hz);
            gq.update(sq, ha, hq, hz);
        }
    }
    auto step = [&](uint32_t& va, uint32_t& vq) {
        D.refill();
        uint2 pk;  // cum[1..4] of the acid context
        if (P::kStatic || ma.adirect) pk = ldg_stream8(ma.adirect + ga.index(sa, pf.pos, psa));
        else pk = __ldg(reinterpret_cast<const uint2*>(ma.dec) + gen_row(ma, sa, ga, pf.pos, psa));
#if defined(IDN_ABL_ROW1)
        const uint32_t row_q = 1;
#elif defined(IDN_ABL_NOQMAP)
        const uint32_t row_q = (gq.spec(sq, pf.pos, psq) * 2654435761u >> 22) + 1;
#else
        const uint32_t row_q = gen_row<P::kStatic>(mq, sq, gq, pf.pos, psq);
#endif
        const uint32_t slot_q = D.xq & kSlotMask, slot_a = D.xa & kSlotMask;
        uint32_t start, freq;
#ifndef IDN_NO_QWIN
        if (P::kQWin) vq = q_find_win(mq.qwin + row_q * (uint32_t)(kQWinBytes / 16), mq.dec + row_q * (uint32_t)kQRowBytes, slot_q, start, freq);
        else
#endif
            vq = q_find(mq.dec + row_q * (uint32_t)kQRowBytes, slot_q, start, freq);
        D.xq = freq * (D.xq >> kScaleBits) + slot_q - start;  // RansDecAdvanceStep
        va = acid_find(pk, slot_a, start, freq);
        D.xa = freq * (D.xa >> kScaleBits) + slot_a - start;
        D.renorm_all();
        if (C.tab) {  // uniform per launch
            C.ca = C.tab[(C.ca ^ va) & 0xffu] ^ (C.ca >> 8);
            C.cq = C.tab[(C.cq ^ vq) & 0xffu] ^ (C.cq >> 8);
        }
        const bool z = va * vq == 0;
        ga.update(sa, va, vq, z);
        gq.update(sq, va, vq, z);
        pf.advance();
    };
    uint32_t i = p0, va, vq;
#pragma unroll 1
    for (; i < p1 && !O.aligned(); i++) {  // up to the first word boundary (everything, if the two outputs disagree)
        step(va, vq);
        O.put(va, vq);
    }
#pragma unroll 1
    for (; i + 4 <= p1; i += 4) {
        uint32_t wa, wq;
        step(wa, wq);
        step(va, vq);
        wa = __byte_perm(wa, va, 0x3240);
        wq = __byte_perm(wq, vq, 0x3240);
        step(va, vq);
        wa = __byte_perm(wa, va, 0x3410);
        wq = __byte_perm(wq, vq, 0x3410);
        step(va, vq);
        wa = __byte_perm(wa, va, 0x4210);
        wq = __byte_perm(wq, vq, 0x4210);
        O.put4(wa, wq);
    }
#pragma unroll 1
    for (; i < p1; i++) {
        step(va, vq);
        O.put(va, vq);
    }
}

// largest b < n_blocks with base[b] <= v (base: an exclusive scan per block)
__device__ __forceinline__ uint32_t block_of(const unsigned long long* __restrict__ base, uint32_t n_blocks, unsigned long long v) {
    uint32_t lo = 0, hi = n_blocks;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(base + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// block and index slot of read r of a block-strided index; false past the last read
__device__ __forceinline__ bool decode_locate(const DecodeArgs& A, uint64_t r, unsigned long long& slot, unsigned long long& sym_base) {
    const unsigned long long R = A.blk_read_base[A.n_blocks];
    if (r >= R) return false;
    const uint32_t lo = block_of(A.blk_read_base, A.n_blocks, r);
    slot = A.slot_base[lo] + (r - A.blk_read_base[lo]);
    sym_base = A.blk_sym_base[lo];
    return true;
}

template <bool kUniform, class P>
__device__ __forceinline__ void decode_one(const DecodeArgs& A, const ModelDev& MA, const ModelDev& MQ, uint64_t r, const uint32_t* s_tab,
                                           const uint32_t* s_xpow) {
    DecCrc C{A.part_crc ? s_tab : nullptr, 0xffffffffu, 0xffffffffu};
    unsigned long long slot = r, sym_base = 0;
    if (A.blk_read_base) {
        if (!decode_locate(A, r, slot, sym_base)) return;
        const unsigned long long R = A.blk_read_base[A.n_blocks];
        if (r == R - 1 && A.read_off_out) A.read_off_out[R] = A.blk_sym_base[A.n_blocks];
    } else if (r >= A.n_reads) {
        return;
    }
    const ModelDev& ma = kUniform ? MA : A.models[A.model_ids[A.ix.am[slot]]];
    const ModelDev& mq = kUniform ? MQ : A.models[A.model_ids[A.ix.qm[slot]]];
    const uint32_t len = A.ix.seq_len[slot];
    const unsigned long long ooff = sym_base + A.ix.sym_off[slot];
    if (A.read_off_out) A.read_off_out[r] = ooff;
    DecStream D;
    D.begin(A.payload, A.ix.pay_off[slot], A.ix.pay_len[slot]);
    SymWriter O;
    O.init(A.acids_out + ooff, A.out_dq);
    decode_read_body<P>(ma, mq, len, 0, len, nullptr, D, O, C);
    O.flush();
    const uint32_t plen = A.ix.pay_len[slot];
    D.finish(A.payload, A.ix.pay_off[slot], plen);
    uint32_t st = D.st;
    if (!(st & 1) && !D.clean_end(plen)) st |= 2;
    if (A.read_status) A.read_status[r] = st;
    if (st) {
        atomicOr(A.err, 1u);
        if (A.err_block) atomicMin(A.err_block, (int32_t)block_of(A.blk_read_base, A.n_blocks, r));
    }
    if (A.part_crc) {  // crc(acids | quals) of this read, as crc_read_kernel would compute it
        const CrcPair p = crc_concat(CrcPair{~C.ca, len}, CrcPair{~C.cq, len}, s_xpow);
        A.part_crc[r] = len ? p.crc : 0u;
        A.part_len[r] = 2ull * len;
    }
}

template <bool kUniform, class P>
__global__ void __launch_bounds__(128, kUniform ? IDN_DEC_MINB : 1)
decode_kernel(DecodeArgs A, const ModelDev MA, const ModelDev MQ) {
    __shared__ uint32_t s_tab[256];
    __shared__ uint32_t s_xpow[64];
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (A.status && A.status[0] != 0) return;
    if (A.part_crc) {
        for (int k = threadIdx.x; k < 256; k += blockDim.x) s_tab[k] = A.crc_tab[k];
        for (int k = threadIdx.x; k < 64; k += blockDim.x) s_xpow[k] = A.xpow[k];
        __syncthreads();
    }
    decode_one<kUniform, P>(A, MA, MQ, r, s_tab, s_xpow);
}

// one model pair's bucket of reads (block-strided index only), see encode_list_kernel
template <class P>
__global__ void __launch_bounds__(128, IDN_DEC_MINB)
decode_list_kernel(DecodeArgs A, const ModelDev MA, const ModelDev MQ, ReadList L) {
    __shared__ uint32_t s_tab[256];
    __shared__ uint32_t s_xpow[64];
    if (A.status && A.status[0] != 0) return;
    if (A.part_crc) {
        for (int k = threadIdx.x; k < 256; k += blockDim.x) s_tab[k] = A.crc_tab[k];
        for (int k = threadIdx.x; k < 64; k += blockDim.x) s_xpow[k] = A.xpow[k];
        __syncthreads();
    }
    const uint32_t n = *L.count;
    const uint32_t* __restrict__ list = L.list + *L.base;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        decode_one<true, P>(A, MA, MQ, list[i], s_tab, s_xpow);
}

// decompress side: the model pair the slice walk recorded for read r (container model indices; a pair that is not
// (acid model, q-score model) in that order never reaches the decoder: the walk rejects it)
struct DecodePairKey {
    DecodeArgs A;
    uint32_t n_models;
    __device__ __forceinline__ uint32_t operator()(uint64_t r) const {
        if (A.status && A.status[0] != 0) return 0xffffffffu;
        unsigned long long slot, sym_base;
        if (!decode_locate(A, r, slot, sym_base)) return 0xffffffffu;
        return (uint32_t)A.ix.am[slot] * n_models + A.ix.qm[slot];
    }
};

// final status word of a device-side decompress call
__global__ void finish_decode_kernel(const int32_t* __restrict__ status, const uint32_t* __restrict__ err,
                                     const unsigned long long* __restrict__ n_reads_total,
                                     const unsigned long long* __restrict__ n_syms_total,
                                     unsigned long long* __restrict__ read_off_out, int32_t* __restrict__ status_dev) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int32_t code = status[0];
    uint64_t R = *n_reads_total;
    int32_t blk = status[1];
    if (code != 11 && code != 12) {
        // block failures: the lowest block wins; within one block a malformed walk / lane table before a checksum mismatch
        // before a stream that runs out or does not end cleanly (IDN_E_SERIALIZE)
        unsigned long long best = ~0ull;
        int32_t best_code = 0;
        auto take = [&](unsigned long long b, unsigned rank, int32_t c) {
            const unsigned long long k = b << 2 | rank;
            if (k < best) {
                best = k;
                best_code = c;
            }
        };
        const unsigned long long key = fail_key(status);
        if (key != ~0ull) take(key >> 32, 0, (int32_t)(uint32_t)key);
        if (code == 6) take((uint32_t)status[3], 1, 6);
        if (status[6] != 0x7fffffff) take((uint32_t)status[6], 2, 3);
        if (best_code) {
            code = best_code;
            blk = (int32_t)(best >> 2);
        } else if (*err & 1u) {
            code = 3;  // a payload ran out: IDN_E_SERIALIZE
        }
    }
    status_dev[0] = code;
    status_dev[1] = blk;
    status_dev[2] = code == 11 ? status[2] : (int32_t)(R > 0x7fffffffull ? 0x7fffffff : R);
    status_dev[3] = (int32_t)(*n_syms_total & 0x7fffffffull);
    if (code == 0 && R == 0 && read_off_out) read_off_out[0] = 0;
}

// ---------------------------------------------------------------------------------------------------
// Workload generator (bench/test utility, not on the reference's path): model-driven synthetic reads.
// Every symbol is drawn from the model's own distribution for the context the generators are in
// (SURVEY.md 8d), so the coder sees the statistics the models were trained on instead of the uniform
// dummy context.  One thread per read; RNG = SplitMix64 keyed by (seed, read index).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long& s) {
    unsigned long long z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__global__ void __launch_bounds__(128)
synth_kernel(const ModelDev* __restrict__ models, int32_t ia, int32_t iq, const unsigned long long* __restrict__ read_off,
             uint64_t n_reads, uint64_t first_read_index, unsigned long long seed, uint32_t n_ppm,
             uint8_t* __restrict__ acids, uint8_t* __restrict__ quals) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const ModelDev& ma = models[ia];
    const ModelDev& mq = models[iq];
    unsigned long long off = read_off[r];
    uint32_t len = (uint32_t)(read_off[r + 1] - off);
    unsigned long long s = seed ^ ((first_read_index + r + 1) * 0xD1B54A32D192ED03ull);
    const SpecDev sa = ma.spec, sq = mq.spec;
    GenFwd ga, gq;
    ga.init();
    gq.init();
    const uint32_t pbmax = sa.pb > sq.pb ? sa.pb : sq.pb;
    const uint32_t psa = pbmax - sa.pb, psq = pbmax - sq.pb;
    PosFwd pf;
    pf.init(len, pbmax);
    FwdWriter oa, oq;
    oa.init(acids + off);
    oq.init(quals + off);
    uint32_t prev_q = 0;
    for (uint32_t i = 0; i < len; i++) {
        unsigned long long u = splitmix64(s);
        uint32_t slot_a = (uint32_t)u & kSlotMask, slot_q = (uint32_t)(u >> 14) & kSlotMask;
        uint32_t start, freq;
        uint32_t row_a = gen_row(ma, sa, ga, pf.pos, psa);
        uint32_t row_q = gen_row(mq, sq, gq, pf.pos, psq);
        uint2 pk = __ldg(reinterpret_cast<const uint2*>(ma.dec) + row_a);
        uint32_t a = acid_find(pk, slot_a, start, freq);
        uint32_t q = q_find(mq.dec + row_q * (uint32_t)kQRowBytes, slot_q, start, freq);
        // a context the model never saw maps to the uniform dummy row; drawing from it would leave the statistics the
        // model was trained on for good (uniform symbols lead to more unseen contexts), which real reads do not do:
        // keep the previous quality score and draw a plain base instead
        if (row_a == 0) a = 1 + (slot_a & 3u);
        if (row_q == 0 && i > 0) q = prev_q;
        if ((uint32_t)((u >> 32) % 1000000u) < n_ppm) {  // an N call with the Illumina "no call" quality '#'
            a = 0;
            q = 2;
        }
        prev_q = q;
        oa.push(a);
        oq.push(q);
        const bool z = a * q == 0;
        ga.update(sa, a, q, z);
        gq.update(sq, a, q, z);
        pf.advance();
    }
    oa.finish();
    oq.finish();
}

}  // namespace idn
