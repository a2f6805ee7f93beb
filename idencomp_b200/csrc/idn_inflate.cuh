// idn_inflate.cuh -- raw Inflate (RFC 1951) of the Identifiers slices on the device (included by idn_gpu.cu).
//
// Acceptance is zlib's (inflateInit2(-15), the host's inflate_raw): an over-subscribed code is an error, an incomplete
// code is an error except a single code of length 1 for the literal/length and distance codes, a distance code without
// codes is fine until a distance is decoded, a distance reaching before the start of the stream, literal/length
// symbols 286/287 and distance symbols 30/31 are errors, bytes after the final block are ignored.  Every input read is
// bounds-checked: bytes past the slice read as zero and a decode that consumed more bits than the slice holds fails.
//
// Parallel decode: each slice (a stream) is cut into ranges of `range` compressed bytes.  In every range but the first
// one warp looks for a block start (inf_find_kernel): the byte after a byte-aligned 00 00 FF FF (the end of an empty
// stored block: sync / full flushes, the device encoder's segment joins), or a bit where a dynamic-block header passes
// full validation (complete codes, end-of-block present; the block finder of rapidgzip, Knespel & Brunst 2023).  From
// its candidate a warp decodes (inf_decode_kernel) without the 32 KiB history: a back-reference before the chunk's start
// becomes a marker 0x8000 | (32768 + offset) naming that byte, so chunk output is 16-bit per byte.  A chunk stops at the
// first block boundary at or past the next chunk's candidate.  inf_join_kernel walks each stream's chunks in order: a
// chunk is used only when the verified decode before it ended exactly on its start bit; any other chunk is decoded again
// from that end (serially, one warp per stream).  inf_resolve_kernel then writes the bytes chunk after chunk, each step
// parallel over the chunk and reading the already resolved 32 KiB before it.  inf_split_*_kernel cut each block's text
// into names the way the host's inflate_names does.
//
// The decoder runs warp-redundant: every lane walks the same bits with the same state (the loads broadcast), lane 0
// writes literals, the warp builds the Huffman tables in shared memory and copies matches (an overlapping copy with
// distance d < length reads out[p - d + (j mod d)], so no lane waits for another).
#pragma once

#include <cstdint>

namespace idn {
namespace inf {

constexpr uint32_t kLutBits = 10;
constexpr uint32_t kWarps = 4;                 // decoder warps per CTA
constexpr uint64_t kNone = ~0ull;               // no candidate / no stop
constexpr uint32_t kDefaultRange = 4096;        // compressed bytes per range (tools/names_inflate_bench.py --sweep, DESIGN section 5)

enum : uint32_t { ST_ERR = 1u, ST_FINAL = 2u, ST_DONE = 4u };

struct Stream {
    unsigned long long in_off;  // Deflate bytes in the container buffer
    uint32_t in_len;
    uint32_t block;
    uint32_t first_chunk, n_chunks;
};

struct Chunk {
    uint32_t stream, k;         // k-th range of its stream
};

// per chunk: candidate start bit, end bit, output length, status, offset of its output in the stream
struct ChunkState {
    unsigned long long cand, end, olen, off;
    uint32_t status, used;
};

struct HufTab {
    uint16_t lut[1u << kLutBits];  // (symbol << 4) | length for codes of <= kLutBits bits, 0 = longer or invalid
    uint16_t cnt[16];
    uint16_t sym[288];             // symbols by (length, value)
};

struct WarpSmem {
    HufTab lit, dist;              // the code-length code is built into `dist` before the distance code replaces it
    uint8_t lens[32 + 316];        // code-length code at [0, 19); literal/length and distance lengths from 32 on
    int32_t flag;
    int32_t fixed;                 // the tables hold the fixed code
};

__constant__ uint16_t c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
                                     4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// LSB-first bit reader over in[0, n); bytes past n read as zero, `pos` counts consumed bits
struct BitIn {
    const uint8_t* p;
    uint64_t n, byte, buf, pos;
    int cnt;
    __device__ void init(const uint8_t* p_, uint64_t n_, uint64_t bit) {
        p = p_;
        n = n_;
        byte = bit >> 3;
        buf = 0;
        cnt = 0;
        pos = bit & ~7ull;
        refill();
        get((int)(bit & 7));
    }
    __device__ __forceinline__ void refill() {
        while (cnt <= 56) {
            const uint64_t b = byte < n ? p[byte] : 0;
            buf |= b << cnt;
            cnt += 8;
            byte++;
        }
    }
    __device__ __forceinline__ uint32_t get(int k) {
        const uint32_t v = (uint32_t)(buf & ((1ull << k) - 1));
        buf >>= k;
        cnt -= k;
        pos += k;
        return v;
    }
    __device__ __forceinline__ bool over() const { return pos > 8 * n; }
};

// canonical decode of the bits `v` (LSB first); -1 when no code of <= 15 bits matches
__device__ __forceinline__ int huf_slow(const HufTab& t, uint32_t v, int* len) {
    int code = 0, first = 0, index = 0;
    for (int l = 1; l <= 15; l++) {
        code |= (v >> (l - 1)) & 1;
        const int count = t.cnt[l];
        if (code - first < count) {
            *len = l;
            return t.sym[index + code - first];
        }
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

__device__ __forceinline__ int huf_decode(const HufTab& t, BitIn& br) {
    br.refill();
    const uint32_t v = (uint32_t)br.buf;
    const uint32_t e = t.lut[v & ((1u << kLutBits) - 1)];
    if (e) {
        br.get((int)(e & 15));
        return (int)(e >> 4);
    }
    int len = 0;
    const int s = huf_slow(t, v, &len);
    if (s >= 0) br.get(len);
    return s;
}

// Builds `t` from lens[0, n) with zlib's rules (inftrees.c): over-subscribed -> invalid; incomplete -> invalid unless
// (not `codes` and the longest code has 1 bit); no codes at all -> valid, every decode fails.  Warp-collective.
__device__ bool huf_build(HufTab& t, const uint8_t* lens, int n, bool codes, int32_t* flag, int lane) {
    if (lane == 0) {
        for (int l = 0; l < 16; l++) t.cnt[l] = 0;
        for (int s = 0; s < n; s++) t.cnt[lens[s]]++;
        t.cnt[0] = 0;
        int max = 15;
        while (max >= 1 && t.cnt[max] == 0) max--;
        int left = 1;
        bool ok = true;
        for (int l = 1; l <= 15; l++) {
            left <<= 1;
            left -= t.cnt[l];
            if (left < 0) ok = false;
        }
        if (ok && max > 0 && left > 0 && (codes || max != 1)) ok = false;
        uint16_t offs[16];
        offs[1] = 0;
        for (int l = 1; l < 15; l++) offs[l + 1] = offs[l] + t.cnt[l];
        if (ok)
            for (int s = 0; s < n; s++)
                if (lens[s]) t.sym[offs[lens[s]]++] = (uint16_t)s;
        *flag = ok;
    }
    __syncwarp();
    const bool ok = *flag != 0;
    if (ok)
        for (uint32_t j = lane; j < (1u << kLutBits); j += 32) {
            int len = 0;
            const int s = huf_slow(t, j, &len);
            t.lut[j] = (s >= 0 && len <= (int)kLutBits) ? (uint16_t)((s << 4) | len) : 0;
        }
    __syncwarp();
    return ok;
}

// Decodes blocks from br.pos until a block boundary at or past `stop`, the end of a final block, or an error.  Output
// (16-bit, markers for bytes before the start) goes to out[0, cap); *olen counts all of it, also past cap.
__device__ uint32_t inflate_run(WarpSmem& sm, BitIn& br, uint64_t stop, uint16_t* __restrict__ out, uint64_t cap, uint64_t* olen_out,
                                uint64_t* end_out, int lane) {
    uint64_t olen = 0;
    uint32_t st = 0;
    for (;;) {
        if (br.pos >= stop) break;
        br.refill();
        const uint32_t bfinal = br.get(1), type = br.get(2);
        if (type == 0) {
            br.get((int)((8 - (br.pos & 7)) & 7));
            br.refill();
            const uint32_t len = br.get(16), nlen = br.get(16);
            if (br.over() || len != (~nlen & 0xffffu) || br.pos + 8ull * len > 8 * br.n) {
                st = ST_ERR;
                break;
            }
            const uint64_t at = br.pos >> 3;
            for (uint32_t j = lane; j < len; j += 32)
                if (olen + j < cap) out[olen + j] = br.p[at + j];
            olen += len;
            br.init(br.p, br.n, br.pos + 8ull * len);
            __syncwarp();
        } else if (type == 3) {
            st = ST_ERR;
            break;
        } else {
            if (type == 1) {
                if (!sm.fixed) {
                    for (int s = lane; s < 288; s += 32) sm.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
                    __syncwarp();
                    huf_build(sm.lit, sm.lens, 288, false, &sm.flag, lane);
                    for (int s = lane; s < 32; s += 32) sm.lens[s] = 5;
                    __syncwarp();
                    huf_build(sm.dist, sm.lens, 32, false, &sm.flag, lane);
                    if (lane == 0) sm.fixed = 1;
                    __syncwarp();
                }
            } else {
                if (lane == 0) sm.fixed = 0;
                const uint32_t nlen = br.get(5) + 257, ndist = br.get(5) + 1, ncl = br.get(4) + 4;
                if (nlen > 286 || ndist > 30) {
                    st = ST_ERR;
                    break;
                }
                if (lane < 19) sm.lens[lane] = 0;
                __syncwarp();
                for (uint32_t i = 0; i < ncl; i++) {
                    if ((i & 7) == 0) br.refill();
                    const uint32_t v = br.get(3);
                    if (lane == 0) sm.lens[c_clorder[i]] = (uint8_t)v;
                }
                __syncwarp();
                if (br.over() || !huf_build(sm.dist, sm.lens, 19, true, &sm.flag, lane)) {
                    st = ST_ERR;
                    break;
                }
                // code lengths: every lane decodes, lane 0 stores
                uint32_t i = 0;
                bool bad = false;
                while (i < nlen + ndist) {
                    const int s = huf_decode(sm.dist, br);
                    if (s < 0) {
                        bad = true;
                        break;
                    }
                    uint32_t rep = 1;
                    if (s == 16) {
                        if (i == 0) {
                            bad = true;
                            break;
                        }
                        rep = 3 + br.get(2);
                    } else if (s == 17) {
                        rep = 3 + br.get(3);
                    } else if (s == 18) {
                        rep = 11 + br.get(7);
                    }
                    if (i + rep > nlen + ndist) {
                        bad = true;
                        break;
                    }
                    if (lane == 0) {
                        // lengths live past the code-length slots: lit at [32, 32 + nlen), dist right after
                        const uint8_t val = s == 16 ? sm.lens[32 + i - 1] : (s < 16 ? (uint8_t)s : 0);
                        for (uint32_t r = 0; r < rep; r++) sm.lens[32 + i + r] = val;
                    }
                    __syncwarp();
                    i += rep;
                }
                if (bad || br.over() || sm.lens[32 + 256] == 0) {
                    st = ST_ERR;
                    break;
                }
                if (!huf_build(sm.lit, sm.lens + 32, (int)nlen, false, &sm.flag, lane) ||
                    !huf_build(sm.dist, sm.lens + 32 + nlen, (int)ndist, false, &sm.flag, lane)) {
                    st = ST_ERR;
                    break;
                }
            }
            // symbols of the block
            for (;;) {
                const int s = huf_decode(sm.lit, br);
                if (s < 0 || s >= 286) {
                    st = ST_ERR;
                    break;
                }
                if (s < 256) {
                    if (lane == 0 && olen < cap) out[olen] = (uint16_t)s;
                    olen++;
                } else if (s == 256) {
                    break;
                } else {
                    const uint32_t len = c_lbase[s - 257] + br.get(c_lext[s - 257]);
                    const int ds = huf_decode(sm.dist, br);
                    if (ds < 0 || ds >= 30) {
                        st = ST_ERR;
                        break;
                    }
                    br.refill();
                    const uint32_t d = c_dbase[ds] + br.get(c_dext[ds]);
                    __syncwarp();
                    for (uint32_t j = lane; j < len; j += 32) {
                        const int64_t q = (int64_t)olen - (int64_t)d + (int64_t)(j % d);
                        uint16_t v;
                        if (q < 0) v = (uint16_t)(0x8000u | (uint32_t)(q + 32768));
                        else v = (uint64_t)q < cap ? out[q] : 0;
                        if (olen + j < cap) out[olen + j] = v;
                    }
                    __syncwarp();
                    olen += len;
                }
                if (br.over()) {
                    st = ST_ERR;
                    break;
                }
            }
            if (st) break;
            if (br.over()) {
                st = ST_ERR;
                break;
            }
        }
        if (bfinal) {
            st = ST_FINAL;
            break;
        }
    }
    *olen_out = olen;
    *end_out = br.pos;
    return st;
}

// Does a dynamic-block header with complete codes and an end-of-block code start at bit `bit`?  (one lane, registers)
__device__ bool dyn_header_ok(const uint8_t* in, uint64_t n, uint64_t bit) {
    BitIn br;
    br.init(in, n, bit);
    br.get(1);
    if (br.get(2) != 2) return false;
    const uint32_t nlen = br.get(5) + 257, ndist = br.get(5) + 1, ncl = br.get(4) + 4;
    if (nlen > 286 || ndist > 30) return false;
    uint8_t cl[19];
    for (int i = 0; i < 19; i++) cl[i] = 0;
    br.refill();
    for (uint32_t i = 0; i < ncl; i++) {
        if ((i & 7) == 0) br.refill();
        cl[c_clorder[i]] = (uint8_t)br.get(3);
    }
    int cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 19; i++) cnt[cl[i]]++;
    int left = 1;
    for (int l = 1; l < 8; l++) {
        left = (left << 1) - cnt[l];
        if (left < 0) return false;
    }
    if (left != 0) return false;
    // canonical decode of the code lengths with the (complete) code-length code
    int lc[16], dc[16];
    for (int l = 0; l < 16; l++) lc[l] = dc[l] = 0;
    uint32_t i = 0, prev = 0;
    bool eob = false;
    while (i < nlen + ndist) {
        br.refill();
        int code = 0, first = 0, s = -1;
        for (int l = 1; l < 8; l++) {
            code |= (int)br.get(1);
            const int c = cnt[l];
            if (code - first < c) {
                int k = code - first;
                for (int x = 0; x < 19; x++)
                    if (cl[x] == l && k-- == 0) {
                        s = x;
                        break;
                    }
                break;
            }
            first = (first + c) << 1;
            code <<= 1;
        }
        if (s < 0) return false;
        uint32_t rep = 1, v = (uint32_t)s;
        if (s == 16) {
            if (i == 0) return false;
            v = prev;
            rep = 3 + br.get(2);
        } else if (s == 17) {
            v = 0;
            rep = 3 + br.get(3);
        } else if (s == 18) {
            v = 0;
            rep = 11 + br.get(7);
        }
        if (i + rep > nlen + ndist) return false;
        for (uint32_t r = 0; r < rep; r++, i++) {
            if (i < nlen) {
                lc[v]++;
                if (i == 256 && v) eob = true;
            } else {
                dc[v]++;
            }
        }
        prev = v;
    }
    if (!eob || br.over()) return false;
    int ll = 1, dl = 1;
    for (int l = 1; l < 16; l++) {
        ll = (ll << 1) - lc[l];
        dl = (dl << 1) - dc[l];
        if (ll < 0 || dl < 0) return false;
    }
    return ll == 0 && dl == 0;
}

// ---- kernels -------------------------------------------------------------------------------------------------------------

// blocks' leading Identifiers slices (0x00 | u32be n | compression | n bytes), as inflate_names walks them.  count pass
// (out == nullptr): n_slices[b] and flags[b] (1 malformed, 2 Brotli); fill pass: the stream records from first[b] on.
__global__ void inf_walk_kernel(const uint8_t* __restrict__ blocks, const unsigned long long* __restrict__ block_off,
                                const uint32_t* __restrict__ block_len, uint32_t B, uint32_t* __restrict__ n_slices,
                                uint32_t* __restrict__ flags, const unsigned long long* __restrict__ first, Stream* __restrict__ out) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const uint8_t* p = blocks + block_off[b];
    const uint64_t len = block_len ? block_len[b] : block_off[b + 1] - block_off[b];
    uint64_t pos = 0;
    uint32_t k = 0, f = 0;
    while (pos < len && p[pos] == 0x00) {
        if (pos + 6 > len) {
            f |= 1;
            break;
        }
        const uint32_t n = ((uint32_t)p[pos + 1] << 24) | ((uint32_t)p[pos + 2] << 16) | ((uint32_t)p[pos + 3] << 8) | p[pos + 4];
        const uint8_t comp = p[pos + 5];
        if (n > len - pos - 6 || comp > 1) {
            f |= 1;
            break;
        }
        if (comp == 0) f |= 2;
        if (out) {
            Stream s;
            s.in_off = block_off[b] + pos + 6;
            s.in_len = n;
            s.block = b;
            s.first_chunk = s.n_chunks = 0;
            out[first[b] + k] = s;
        }
        k++;
        pos += 6 + (uint64_t)n;
    }
    if (!out) {
        n_slices[b] = k;
        flags[b] = f;
    }
}

// one warp per chunk of range >= 1: the first candidate bit of its range, or kNone
__global__ void __launch_bounds__(128) inf_find_kernel(const uint8_t* __restrict__ blocks, const Stream* __restrict__ streams,
                                                       const Chunk* __restrict__ chunks, uint32_t n_chunks, uint32_t range,
                                                       ChunkState* __restrict__ cs) {
    const uint32_t c = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, lane = threadIdx.x & 31;
    if (c >= n_chunks) return;
    const Chunk ch = chunks[c];
    const Stream s = streams[ch.stream];
    uint64_t found = kNone;
    if (ch.k == 0) {
        found = 0;
    } else {
        const uint8_t* in = blocks + s.in_off;
        const uint64_t lo = (uint64_t)ch.k * range * 8, hi = min((uint64_t)(ch.k + 1) * range, (uint64_t)s.in_len) * 8;
        for (uint64_t base = lo; base < hi && found == kNone; base += 32) {
            const uint64_t bit = base + lane;
            bool ok = false;
            if (bit < hi) {
                if ((bit & 7) == 0 && bit >= 32) {
                    const uint64_t y = bit >> 3;
                    ok = in[y - 4] == 0 && in[y - 3] == 0 && in[y - 2] == 0xff && in[y - 1] == 0xff;
                }
                if (!ok) ok = dyn_header_ok(in, s.in_len, bit);
            }
            const uint32_t m = __ballot_sync(0xffffffffu, ok);
            if (m) found = base + (__ffs(m) - 1);
        }
    }
    if (lane == 0) {
        ChunkState z;
        z.cand = found;
        z.end = z.olen = z.off = 0;
        z.status = 0;
        z.used = 0;
        cs[c] = z;
    }
}

// start of the next chunk of the stream that has a candidate (the stop bit of chunk c), or kNone
__device__ __forceinline__ uint64_t next_cand(const ChunkState* cs, const Stream& s, uint32_t c) {
    for (uint32_t j = c + 1; j < s.first_chunk + s.n_chunks; j++)
        if (cs[j].cand != kNone) return cs[j].cand;
    return kNone;
}

// one warp per chunk with a candidate: the speculative decode into its slot of `cap` 16-bit entries
__global__ void __launch_bounds__(kWarps * 32) inf_decode_kernel(const uint8_t* __restrict__ blocks, const Stream* __restrict__ streams,
                                                                 const Chunk* __restrict__ chunks, uint32_t n_chunks, ChunkState* __restrict__ cs,
                                                                 uint16_t* __restrict__ scratch, uint64_t cap) {
    __shared__ WarpSmem smem[kWarps];
    const uint32_t w = threadIdx.x / 32, lane = threadIdx.x & 31, c = blockIdx.x * kWarps + w;
    if (c >= n_chunks) return;
    const uint64_t start = cs[c].cand;
    if (start == kNone) return;
    WarpSmem& sm = smem[w];
    if (lane == 0) sm.fixed = 0;
    __syncwarp();
    const Stream s = streams[chunks[c].stream];
    BitIn br;
    br.init(blocks + s.in_off, s.in_len, start);
    uint64_t olen = 0, end = 0;
    const uint32_t st = inflate_run(sm, br, next_cand(cs, s, c), scratch + (uint64_t)c * cap, cap, &olen, &end, lane);
    if (lane == 0) {
        cs[c].end = end;
        cs[c].olen = olen;
        cs[c].status = st | ST_DONE;
    }
}

// per-stream results of the join
struct StreamState {
    unsigned long long len, pos;  // output bytes; position of the stream's text in the joined buffer
    uint32_t status;              // ST_ERR
    uint32_t pad;
};

// stats[0] speculative chunks decoded, [1] of them joined, [2] bytes decoded serially, [3] largest used output
// one warp per stream: walk the chunks in order, re-decode what does not join, place outputs
__global__ void __launch_bounds__(kWarps * 32) inf_join_kernel(const uint8_t* __restrict__ blocks, const Stream* __restrict__ streams,
                                                               uint32_t n_streams, ChunkState* __restrict__ cs, uint16_t* __restrict__ scratch,
                                                               uint64_t cap, StreamState* __restrict__ ss, unsigned long long* __restrict__ stats) {
    __shared__ WarpSmem smem[kWarps];
    const uint32_t w = threadIdx.x / 32, lane = threadIdx.x & 31, si = blockIdx.x * kWarps + w;
    if (si >= n_streams) return;
    WarpSmem& sm = smem[w];
    if (lane == 0) sm.fixed = 0;
    __syncwarp();
    const Stream s = streams[si];
    uint64_t e = 0, off = 0, spec = 0, joined = 0, serial = 0, maxlen = 0;
    bool final = false, err = false;
    for (uint32_t c = s.first_chunk; c < s.first_chunk + s.n_chunks; c++) {
        ChunkState x = cs[c];
        if (x.status & ST_DONE && c != s.first_chunk) spec++;
        if (final || err || x.cand == kNone) {
            if (lane == 0) {
                cs[c].used = 0;
                cs[c].olen = 0;
            }
            continue;
        }
        if (x.cand == e && (x.status & ST_DONE) && !(x.status & ST_ERR)) {
            if (c != s.first_chunk) joined++;
        } else if (x.cand == e && (x.status & ST_ERR)) {
            err = true;  // the verified chain fails here
        } else {
            // serial repair: chunk c again, from where the verified decode ended
            BitIn br;
            br.init(blocks + s.in_off, s.in_len, e);
            uint64_t olen = 0, end = 0;
            const uint32_t st = inflate_run(sm, br, next_cand(cs, s, c), scratch + (uint64_t)c * cap, cap, &olen, &end, lane);
            x.status = st | ST_DONE;
            x.olen = olen;
            x.end = end;
            serial += olen;
            if (st & ST_ERR) err = true;
        }
        if (err) break;
        if (x.status & ST_FINAL) final = true;
        if (lane == 0) {
            cs[c].used = 1;
            cs[c].olen = x.olen;
            cs[c].off = off;
        }
        off += x.olen;
        maxlen = max(maxlen, (uint64_t)x.olen);
        e = x.end;
    }
    if (lane == 0) {
        ss[si].len = off;
        ss[si].status = (err || !final) ? ST_ERR : 0;
        atomicAdd(&stats[0], spec);
        atomicAdd(&stats[1], joined);
        atomicAdd(&stats[2], serial);
        atomicMax(&stats[3], maxlen);
    }
}

// one CTA per stream: chunk outputs to bytes, in order, markers read from the bytes already written before the chunk;
// a '\n' follows every stream (between the slices of a block it is the separator inflate_names puts there)
__global__ void __launch_bounds__(256) inf_resolve_kernel(const Stream* __restrict__ streams, uint32_t n_streams,
                                                          const ChunkState* __restrict__ cs, const uint16_t* __restrict__ scratch,
                                                          uint64_t cap, StreamState* __restrict__ ss, uint8_t* __restrict__ text) {
    const uint32_t si = blockIdx.x;
    if (si >= n_streams) return;
    const Stream s = streams[si];
    const uint64_t base = ss[si].pos;
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    for (uint32_t c = s.first_chunk; c < s.first_chunk + s.n_chunks; c++) {
        const ChunkState x = cs[c];
        if (!x.used) continue;
        const uint16_t* src = scratch + (uint64_t)c * cap;
        const uint64_t at = base + x.off;
        for (uint64_t i = threadIdx.x; i < x.olen; i += blockDim.x) {
            const uint32_t v = src[i];
            uint8_t b;
            if (v < 0x8000u) {
                b = (uint8_t)v;
            } else {
                const int64_t q = (int64_t)x.off + (int64_t)(v & 0x7fffu) - 32768;  // stream-relative source
                if (q < 0) {
                    bad = 1;  // distance too far back
                    b = 0;
                } else {
                    b = text[base + q];
                }
            }
            text[at + i] = b;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        text[base + ss[si].len] = '\n';
        if (bad) ss[si].status |= ST_ERR;
    }
}

// per block: text range [tb, te) in `text`, lines wanted = reads of the block; writes name bytes used to nb[b]
// and the end of line L - 1 (L = lines used) to cut[b]
__device__ __forceinline__ void block_text(const StreamState* ss, const unsigned long long* bstream, uint32_t b, uint64_t* tb, uint64_t* te) {
    const uint64_t f = bstream[b], l = bstream[b + 1];
    if (f == l) {
        *tb = *te = 0;
        return;
    }
    *tb = ss[f].pos;
    *te = ss[l - 1].pos + ss[l - 1].len;
}

// block-wide: for the tile [t0, t0 + 256) of the block's text, each thread's byte, whether it is '\n', and the count of
// '\n' before it in the tile; returns the tile's total
__device__ __forceinline__ uint32_t tile_nl(const uint8_t* text, uint64_t p, uint64_t te, bool* is_nl, uint32_t* before, uint32_t* wsum) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    *is_nl = p < te && text[p] == '\n';
    const uint32_t m = __ballot_sync(0xffffffffu, *is_nl);
    if (lane == 0) wsum[warp] = __popc(m);
    __syncthreads();
    uint32_t pre = 0, tot = 0;
    for (uint32_t k = 0; k < blockDim.x / 32; k++) {
        if (k < warp) pre += wsum[k];
        tot += wsum[k];
    }
    *before = pre + __popc(m & ((1u << lane) - 1));
    __syncthreads();
    return tot;
}

__global__ void __launch_bounds__(256) inf_split_count_kernel(const StreamState* __restrict__ ss, const unsigned long long* __restrict__ bstream,
                                                              const uint32_t* __restrict__ bfr, const uint8_t* __restrict__ text,
                                                              unsigned long long* __restrict__ nb) {
    __shared__ uint32_t wsum[8];
    __shared__ unsigned long long cut;
    const uint32_t b = blockIdx.x;
    uint64_t tb, te;
    block_text(ss, bstream, b, &tb, &te);
    const uint64_t want = bfr[b + 1] - bfr[b];
    if (threadIdx.x == 0) cut = te;
    __syncthreads();
    if (bstream[b] == bstream[b + 1] || want == 0) {
        if (threadIdx.x == 0) nb[b] = 0;
        return;
    }
    // end of line want - 1: the newline with index want - 1, else the text's end
    uint64_t seen = 0;
    for (uint64_t t0 = tb; t0 < te; t0 += blockDim.x) {
        bool nl;
        uint32_t before;
        const uint32_t tot = tile_nl(text, t0 + threadIdx.x, te, &nl, &before, wsum);
        if (nl && seen + before == want - 1) cut = t0 + threadIdx.x;
        seen += tot;
        __syncthreads();
        if (seen >= want) break;
    }
    if (threadIdx.x == 0) {
        const uint64_t lines = min(want, seen + 1);
        nb[b] = (cut - tb) - (lines - 1);
    }
}

__global__ void __launch_bounds__(256) inf_split_write_kernel(const StreamState* __restrict__ ss, const unsigned long long* __restrict__ bstream,
                                                              const uint32_t* __restrict__ bfr, const uint8_t* __restrict__ text,
                                                              const unsigned long long* __restrict__ nbase, uint8_t* __restrict__ names,
                                                              unsigned long long* __restrict__ name_off) {
    __shared__ uint32_t wsum[8];
    const uint32_t b = blockIdx.x;
    uint64_t tb, te;
    block_text(ss, bstream, b, &tb, &te);
    const uint64_t first = bfr[b], want = bfr[b + 1] - first, base = nbase[b], nbytes = nbase[b + 1] - base;
    if (b == 0 && threadIdx.x == 0) name_off[0] = 0;
    uint64_t lines = 0;  // lines whose end was written
    if (bstream[b] != bstream[b + 1] && want) {
        uint64_t seen = 0;
        for (uint64_t t0 = tb; t0 < te && seen < want; t0 += blockDim.x) {
            bool nl;
            uint32_t before;
            const uint64_t p = t0 + threadIdx.x;
            const uint32_t tot = tile_nl(text, p, te, &nl, &before, wsum);
            const uint64_t li = seen + before;  // line of byte p
            if (p < te && li < want) {
                const uint64_t o = base + (p - tb) - li;
                if (!nl) names[o] = text[p];
                else if (li < want - 1) name_off[first + li + 1] = o;
            }
            seen += tot;
        }
        lines = min(want, seen + 1);
    }
    // the last line used and every read without a line end at the block's last name byte
    for (uint64_t r = (lines ? lines - 1 : 0) + threadIdx.x; r < want; r += blockDim.x) name_off[first + r + 1] = base + nbytes;
}

}  // namespace inf
}  // namespace idn
