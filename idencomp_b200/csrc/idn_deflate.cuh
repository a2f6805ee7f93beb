// idn_deflate.cuh -- raw Deflate (RFC 1951) of the Identifiers slice on the device (included by idn_gpu.cu).
//
// The reference joins the names of a block with '\n' and Deflates them (write_identifiers, compressor_block.rs:146-206).
// Here the joined text of every block is cut into segments of kSeg bytes; one CTA codes one segment as one Deflate block
// with its own Huffman tables (dynamic, or fixed when that is smaller).  Every segment but the last of a block is followed
// by an empty stored block (000, pad, 00 00 FF FF, as pigz does), so each segment's output ends on a byte and a slice is
// the byte concatenation of its segments: a scan over segment lengths places them, no bit stitching is needed.
//
// Matches: each warp owns kPart bytes of the segment and walks them (after a warm-up over the kWarm bytes before them,
// which may lie in the previous segment of the same block) 32 positions at a time; a position's candidate is the latest
// earlier position with the same 4-byte hash, from the warp's own table or an earlier lane of the same step.  Each thread
// then parses its kSub bytes greedily (minimum match 4, matches clipped at the sub-range end).  Tables are written by the
// highest lane of a group of equal hashes, histograms are counts, bits are OR-ed into zeroed words: the output depends on
// the block's names only, never on scheduling, the other blocks of the call or the device.
#pragma once

#include <cstdint>

namespace idn {
namespace dfl {

constexpr uint32_t kSeg = 65536;             // input bytes per segment (one CTA, one Deflate block)
constexpr uint32_t kThreads = 256;
constexpr uint32_t kSub = kSeg / kThreads;   // bytes each thread parses
constexpr uint32_t kWarps = kThreads / 32;
constexpr uint32_t kPart = kSeg / kWarps;    // bytes whose candidates one warp finds
constexpr uint32_t kWarm = 4096;             // history a warp's table sees before its part
constexpr uint32_t kHashBits = 11;           // table of 2048 entries per warp
// literal/length alphabet: 288 symbols as RFC 1951 3.2.6 defines the fixed code (286 and 287 never occur, but the fixed
// code's canonical assignment counts them: without them every 9-bit code would come out 4 too small)
constexpr uint32_t kLit = 288, kDist = 30, kHdrBytes = 288;

// what the analysis pass leaves for the emit pass of one segment
struct SegRec {
    uint32_t hdr_bits;  // block header (BFINAL, BTYPE and, for a dynamic block, the code length tables)
    uint32_t bits;      // header + tokens + end-of-block code
    uint8_t len[kLit + kDist + 2];  // code lengths: literal/length [0, 288), distance [288, 318)
    uint8_t hdr[kHdrBytes];
};

__device__ __forceinline__ uint32_t len_sym(uint32_t l, uint32_t& eb, uint32_t& ev) {  // l in 3..258
    if (l == 258) { eb = 0; ev = 0; return 285; }
    const uint32_t l3 = l - 3;
    if (l3 < 8) { eb = 0; ev = 0; return 257 + l3; }
    eb = 31 - __clz(l3) - 2;
    ev = l3 & ((1u << eb) - 1);
    return 257 + 4 * (eb + 1) + ((l3 >> eb) - 4);
}

__device__ __forceinline__ uint32_t dist_sym(uint32_t d, uint32_t& eb, uint32_t& ev) {  // d in 1..32768
    const uint32_t d1 = d - 1;
    if (d1 < 4) { eb = 0; ev = 0; return d1; }
    eb = 31 - __clz(d1) - 1;
    ev = d1 & ((1u << eb) - 1);
    return 2 * (eb + 1) + ((d1 >> eb) & 1);
}

__device__ __forceinline__ uint32_t fixed_len(uint32_t s) { return s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8; }

// scratch of one code builder (shared memory)
struct TreeScratch {
    uint32_t w[2 * kLit];
    uint16_t par[2 * kLit];
    uint16_t sym[kLit];
    uint16_t bl[2 * kLit];
};

// Code lengths (<= limit) over freq[0, n), one thread.  At least two symbols get a code, as zlib's build_tree does, so
// that every code is complete.  Huffman depths by the two-queue method over symbols sorted by (freq, symbol), then the
// depth counts are limited (JPEG Annex K.3) and the lengths handed out longest-first to the rarest symbols.
__device__ void build_lengths(const uint32_t* freq, int n, int limit, uint8_t* len, TreeScratch& t) {
    int m = 0;
    for (int s = 0; s < n; s++) {
        len[s] = 0;
        if (freq[s]) t.sym[m++] = (uint16_t)s;
    }
    for (int s = 0; m < 2; s++)
        if (!freq[s]) t.sym[m++] = (uint16_t)s;
    auto wt = [&](int s) { return freq[s] ? freq[s] : 1u; };
    for (int i = 1; i < m; i++) {  // insertion sort by (weight, symbol)
        const uint16_t x = t.sym[i];
        const uint32_t wx = wt(x);
        int j = i - 1;
        while (j >= 0 && (wt(t.sym[j]) > wx || (wt(t.sym[j]) == wx && t.sym[j] > x))) {
            t.sym[j + 1] = t.sym[j];
            j--;
        }
        t.sym[j + 1] = x;
    }
    for (int i = 0; i < m; i++) t.w[i] = wt(t.sym[i]);
    int li = 0, ii = m, nn = m;
    for (int k = 0; k < m - 1; k++) {
        const int a = (li < m && (ii >= nn || t.w[li] <= t.w[ii])) ? li++ : ii++;
        const int b = (li < m && (ii >= nn || t.w[li] <= t.w[ii])) ? li++ : ii++;
        t.w[nn] = t.w[a] + t.w[b];
        t.par[a] = t.par[b] = (uint16_t)nn;
        nn++;
    }
    t.w[nn - 1] = 0;  // now depths: parents come after their children
    for (int x = nn - 2; x >= 0; x--) t.w[x] = t.w[t.par[x]] + 1;
    int maxd = 0;
    for (int d = 0; d < 2 * kLit; d++) t.bl[d] = 0;
    for (int i = 0; i < m; i++) {
        t.bl[t.w[i]]++;
        maxd = max(maxd, (int)t.w[i]);
    }
    for (int i = maxd; i > limit; i--) {
        while (t.bl[i] > 0) {
            int j = i - 2;
            while (t.bl[j] == 0) j--;
            t.bl[i] -= 2;
            t.bl[i - 1] += 1;
            t.bl[j + 1] += 2;
            t.bl[j] -= 1;
        }
    }
    int idx = 0;
    for (int l = min(maxd, limit); l >= 1; l--)
        for (int c = 0; c < t.bl[l]; c++) len[t.sym[idx++]] = (uint8_t)l;
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for LSB-first output
__device__ void canon_codes(const uint8_t* len, int n, uint16_t* code) {
    uint32_t cnt[16] = {0}, next[16];
    for (int s = 0; s < n; s++) cnt[len[s]]++;
    cnt[0] = 0;
    uint32_t c = 0;
    next[0] = 0;
    for (int b = 1; b < 16; b++) {
        c = (c + cnt[b - 1]) << 1;
        next[b] = c;
    }
    for (int s = 0; s < n; s++)
        code[s] = len[s] ? (uint16_t)(__brev(next[len[s]]++) >> (32 - len[s])) : 0;
}

// bits OR-ed into zeroed 32-bit words: the result does not depend on the order of the writers
struct BitOut {
    uint32_t* w;
    unsigned long long wi;
    unsigned long long acc;
    uint32_t nb;
    __device__ void init(uint32_t* words, unsigned long long bitpos) {
        w = words;
        wi = bitpos >> 5;
        nb = (uint32_t)(bitpos & 31);
        acc = 0;
    }
    __device__ __forceinline__ void put(uint32_t v, uint32_t n) {  // n <= 16
        acc |= (unsigned long long)v << nb;
        nb += n;
        if (nb >= 32) {
            if ((uint32_t)acc) atomicOr(w + wi, (uint32_t)acc);
            wi++;
            acc >>= 32;
            nb -= 32;
        }
    }
    __device__ void flush() {
        if (nb && (uint32_t)acc) atomicOr(w + wi, (uint32_t)acc);
        nb = 0;
    }
};

__device__ __forceinline__ uint32_t tok_bits(uint32_t tk, const uint8_t* len) {
    if (!(tk & 0x80000000u)) return len[tk];
    uint32_t eb, ev, db, dv;
    const uint32_t ls = len_sym(((tk >> 16) & 0xff) + 3, eb, ev);
    const uint32_t ds = dist_sym((tk & 0x7fff) + 1, db, dv);
    return len[ls] + eb + len[kLit + ds] + db;
}

// ---- kernels ----------------------------------------------------------------------------------------------------------

// name_off must not decrease over [0, R]
__global__ void dfl_check_kernel(const unsigned long long* __restrict__ name_off, uint64_t R, uint32_t* __restrict__ bad) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < R && name_off[r + 1] < name_off[r]) atomicOr(bad, 1u);
}

// joined length and segment count of every block; a block table that is not monotone inside [0, R] is flagged
__global__ void dfl_block_kernel(const unsigned long long* __restrict__ name_off, const uint32_t* __restrict__ bfr, uint32_t B, uint64_t R,
                                 unsigned long long* __restrict__ L, unsigned long long* __restrict__ nseg, uint32_t* __restrict__ bad) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const uint32_t f = bfr[b], e = bfr[b + 1];
    unsigned long long l = 0;
    if (e < f || e > R) {
        atomicOr(bad, 1u);
    } else if (e > f) {
        l = name_off[e] - name_off[f] + (e - f - 1);
        if (l >= (1ull << 31)) atomicOr(bad, 2u);
    }
    L[b] = l;
    nseg[b] = l ? (l + kSeg - 1) / kSeg : 1;
}

// out[0] = 0, out[i + 1] = out[i] + in[i] + add; one CTA of 1024 threads
__global__ void __launch_bounds__(1024) dfl_scan_kernel(const unsigned long long* __restrict__ in, uint32_t n, unsigned long long add,
                                                        unsigned long long* __restrict__ out) {
    __shared__ unsigned long long ws[32];
    __shared__ unsigned long long carry;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        carry = 0;
        out[0] = 0;
    }
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + tid;
        unsigned long long x = i < n ? in[i] + add : 0;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= (uint32_t)o) x += y;
        }
        if (lane == 31) ws[warp] = x;
        __syncthreads();
        if (warp == 0) {
            unsigned long long t = ws[lane];
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= (uint32_t)o) t += y;
            }
            ws[lane] = t;
        }
        __syncthreads();
        const unsigned long long incl = carry + (warp ? ws[warp - 1] : 0) + x;
        if (i < n) out[i + 1] = incl;
        __syncthreads();
        if (tid == 1023) carry = incl;
        __syncthreads();
    }
}

// names of every block joined by '\n' into one buffer (block b at J[b])
__global__ void dfl_join_kernel(const uint8_t* __restrict__ names, const unsigned long long* __restrict__ name_off,
                                const uint32_t* __restrict__ bfr, uint32_t B, uint64_t R, const unsigned long long* __restrict__ J,
                                uint8_t* __restrict__ joined) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    uint32_t lo = 0, hi = B - 1;  // last block with bfr[b] <= r
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (bfr[mid] <= r) lo = mid; else hi = mid - 1;
    }
    const uint32_t f = bfr[lo];
    const unsigned long long src = name_off[r], n = name_off[r + 1] - src;
    uint8_t* dst = joined + J[lo] + (src - name_off[f]) + (r - f);
    for (unsigned long long i = 0; i < n; i++) dst[i] = names[src + i];
    if (r + 1 < bfr[lo + 1]) dst[n] = '\n';
}

__global__ void dfl_segmap_kernel(const unsigned long long* __restrict__ segfirst, uint32_t B, uint32_t* __restrict__ segblock) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    for (unsigned long long s = segfirst[b]; s < segfirst[b + 1]; s++) segblock[s] = b;
}

struct AnalyseSmem {
    uint8_t text[kSeg + kWarm];
    union {
        uint16_t tab[kWarps][1u << kHashBits];
        struct {
            TreeScratch t[2];
            uint8_t rsym[kLit + kDist];
            uint8_t rext[kLit + kDist];
            uint32_t clf[19];
            uint8_t cll[19];
            uint16_t clc[19];
        } h;
    } u;
    uint32_t hist[kLit + kDist];
    uint8_t len[kLit + kDist];
};

// one CTA per segment: candidates, greedy parse into tokens, histograms, code lengths, block header, size in bits
__global__ void __launch_bounds__(kThreads, 2)
dfl_analyse_kernel(const uint8_t* __restrict__ joined, const unsigned long long* __restrict__ J, const unsigned long long* __restrict__ L,
                   const unsigned long long* __restrict__ segfirst, const uint32_t* __restrict__ segblock, uint16_t* __restrict__ cand,
                   uint32_t* __restrict__ tok, uint16_t* __restrict__ ntok, SegRec* __restrict__ rec) {
    extern __shared__ __align__(16) uint8_t dfl_smem[];
    AnalyseSmem& sm = *reinterpret_cast<AnalyseSmem*>(dfl_smem);
    const uint32_t s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t b = segblock[s];
    const unsigned long long bstart = J[b], bend = bstart + L[b];
    const unsigned long long s0 = bstart + (s - segfirst[b]) * (unsigned long long)kSeg;
    const unsigned long long s1 = min(s0 + kSeg, bend);
    const bool last = s1 == bend;
    const unsigned long long w0 = s0 - bstart > kWarm ? s0 - kWarm : bstart;
    for (uint32_t i = tid; i < (uint32_t)(s1 - w0); i += kThreads) sm.text[i] = joined[w0 + i];
    for (uint32_t i = tid; i < kLit + kDist; i += kThreads) sm.hist[i] = i == 256;  // end of block
    for (uint32_t i = tid; i < kWarps * (1u << kHashBits); i += kThreads) (&sm.u.tab[0][0])[i] = 0;
    __syncthreads();

    {  // candidates of this warp's part
        const unsigned long long ps = s0 + warp * (unsigned long long)kPart, pe = min(ps + kPart, s1);
        if (ps < pe) {
            const unsigned long long ws = ps - w0 > kWarm ? ps - kWarm : w0;
            uint16_t* tb = sm.u.tab[warp];
            for (unsigned long long base = ws; base < pe; base += 32) {
                const unsigned long long p = base + lane;
                const bool valid = p < pe && p + 4 <= s1;
                uint32_t h = 0;
                if (valid) {
                    const uint8_t* x = sm.text + (p - w0);
                    const uint32_t v = x[0] | (x[1] << 8) | (x[2] << 16) | ((uint32_t)x[3] << 24);
                    h = (v * 2654435761u) >> (32 - kHashBits);
                }
                const uint32_t grp = __match_any_sync(0xffffffffu, valid ? h : (0x10000u + lane));
                const uint32_t e = valid ? tb[h] : 0;
                const uint32_t below = grp & ((1u << lane) - 1);
                unsigned long long c = 0;
                if (valid && below) c = base + (31 - __clz(below)) + 1;
                else if (valid && e) c = ws + e;  // (+1: 0 = none)
                if (p >= ps && p < pe) cand[p] = c ? (uint16_t)(p + 1 - c) : 0;
                __syncwarp();
                if (valid && (grp >> lane) == 1u) tb[h] = (uint16_t)(p - ws + 1);
                __syncwarp();
            }
        }
    }
    __syncthreads();

    {  // greedy parse of this thread's sub-range
        const unsigned long long a = s0 + tid * (unsigned long long)kSub, e = min(a + kSub, s1);
        uint32_t nt = 0;
        for (unsigned long long p = a; p < e;) {
            const uint32_t d = cand[p];
            const uint8_t* x = sm.text + (p - w0);
            uint32_t n = 0;
            if (d) {
                const uint32_t mx = (uint32_t)min(258ull, e - p);
                const uint8_t* y = x - d;
                while (n < mx && x[n] == y[n]) n++;
            }
            if (n >= 4) {
                tok[a + nt++] = 0x80000000u | ((n - 3) << 16) | (d - 1);
                uint32_t eb, ev;
                atomicAdd(&sm.hist[len_sym(n, eb, ev)], 1u);
                atomicAdd(&sm.hist[kLit + dist_sym(d, eb, ev)], 1u);
                p += n;
            } else {
                tok[a + nt++] = x[0];
                atomicAdd(&sm.hist[x[0]], 1u);
                p++;
            }
        }
        ntok[(size_t)s * kThreads + tid] = (uint16_t)nt;
    }
    __syncthreads();

    if (tid == 0) build_lengths(sm.hist, kLit, 15, sm.len, sm.u.h.t[0]);
    if (tid == 32) build_lengths(sm.hist + kLit, kDist, 15, sm.len + kLit, sm.u.h.t[1]);
    __syncthreads();
    if (tid != 0) return;

    // run-length code of the code lengths (RFC 1951 3.2.7), one sequence over HLIT + HDIST values
    uint32_t hlit = kLit, hdist = kDist;
    while (hlit > 257 && sm.len[hlit - 1] == 0) hlit--;
    while (hdist > 1 && sm.len[kLit + hdist - 1] == 0) hdist--;
    auto seq = [&](uint32_t i) { return i < hlit ? sm.len[i] : sm.len[kLit + i - hlit]; };
    const uint32_t nseq = hlit + hdist;
    uint32_t nr = 0;
    for (uint32_t i = 0; i < 19; i++) sm.u.h.clf[i] = 0;
    for (uint32_t i = 0; i < nseq;) {
        const uint8_t v = seq(i);
        uint32_t run = 1;
        while (i + run < nseq && seq(i + run) == v) run++;
        i += run;
        if (v == 0) {
            while (run >= 11) {
                const uint32_t k = min(run, 138u);
                sm.u.h.rsym[nr] = 18, sm.u.h.rext[nr++] = (uint8_t)(k - 11);
                run -= k;
            }
            if (run >= 3) {
                sm.u.h.rsym[nr] = 17, sm.u.h.rext[nr++] = (uint8_t)(run - 3);
                run = 0;
            }
        } else {
            sm.u.h.rsym[nr] = v, sm.u.h.rext[nr++] = 0;
            run--;
            while (run >= 3) {
                const uint32_t k = min(run, 6u);
                sm.u.h.rsym[nr] = 16, sm.u.h.rext[nr++] = (uint8_t)(k - 3);
                run -= k;
            }
        }
        for (; run > 0; run--) sm.u.h.rsym[nr] = v, sm.u.h.rext[nr++] = 0;
    }
    for (uint32_t i = 0; i < nr; i++) sm.u.h.clf[sm.u.h.rsym[i]]++;
    build_lengths(sm.u.h.clf, 19, 7, sm.u.h.cll, sm.u.h.t[0]);
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint32_t hclen = 19;
    while (hclen > 4 && sm.u.h.cll[order[hclen - 1]] == 0) hclen--;
    unsigned long long hdr = 3 + 5 + 5 + 4 + 3 * hclen;
    for (uint32_t i = 0; i < nr; i++) {
        const uint32_t r = sm.u.h.rsym[i];
        hdr += sm.u.h.cll[r] + (r == 16 ? 2 : r == 17 ? 3 : r == 18 ? 7 : 0);
    }
    // cost of the tokens under the dynamic and the fixed code (extra bits are the same for both)
    unsigned long long dyn = hdr, fix = 3, extra = 0;
    for (uint32_t i = 0; i < kLit; i++) {
        dyn += (unsigned long long)sm.hist[i] * sm.len[i];
        fix += (unsigned long long)sm.hist[i] * fixed_len(i);
        if (i >= 265 && i < 285) extra += (unsigned long long)sm.hist[i] * ((i - 261) / 4);
    }
    for (uint32_t i = 0; i < kDist; i++) {
        dyn += (unsigned long long)sm.hist[kLit + i] * sm.len[kLit + i];
        fix += (unsigned long long)sm.hist[kLit + i] * 5;
        if (i >= 4) extra += (unsigned long long)sm.hist[kLit + i] * (i / 2 - 1);
    }
    SegRec& R = rec[s];
    const bool fixed = fix <= dyn;
    for (uint32_t i = 0; i < kHdrBytes; i++) R.hdr[i] = 0;
    if (fixed) {
        for (uint32_t i = 0; i < kLit; i++) R.len[i] = (uint8_t)fixed_len(i);
        for (uint32_t i = 0; i < kDist; i++) R.len[kLit + i] = 5;
        R.hdr[0] = (uint8_t)((last ? 1 : 0) | (1 << 1));
        R.hdr_bits = 3;
        R.bits = (uint32_t)(fix + extra);
        return;
    }
    for (uint32_t i = 0; i < kLit + kDist; i++) R.len[i] = sm.len[i];
    R.hdr_bits = (uint32_t)hdr;
    R.bits = (uint32_t)(dyn + extra);
    canon_codes(sm.u.h.cll, 19, sm.u.h.clc);
    unsigned long long acc = 0;
    uint32_t nb = 0, o = 0;
    auto put = [&](uint32_t v, uint32_t n) {
        acc |= (unsigned long long)v << nb;
        nb += n;
        while (nb >= 8) {
            R.hdr[o++] = (uint8_t)acc;
            acc >>= 8;
            nb -= 8;
        }
    };
    put((last ? 1 : 0) | (2 << 1), 3);
    put(hlit - 257, 5);
    put(hdist - 1, 5);
    put(hclen - 4, 4);
    for (uint32_t i = 0; i < hclen; i++) put(sm.u.h.cll[order[i]], 3);
    for (uint32_t i = 0; i < nr; i++) {
        const uint32_t r = sm.u.h.rsym[i];
        put(sm.u.h.clc[r], sm.u.h.cll[r]);
        if (r >= 16) put(sm.u.h.rext[i], r == 16 ? 2 : r == 17 ? 3 : 7);
    }
    if (nb) R.hdr[o] = (uint8_t)acc;
}

// byte sizes of the segments of each block (relative offsets in segoff) and of its Deflate stream (dlen)
__global__ void dfl_place_kernel(const unsigned long long* __restrict__ segfirst, uint32_t B, const SegRec* __restrict__ rec,
                                 unsigned long long* __restrict__ segoff, unsigned long long* __restrict__ dlen) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    unsigned long long rel = 0;
    for (unsigned long long s = segfirst[b]; s < segfirst[b + 1]; s++) {
        const unsigned long long bits = rec[s].bits;
        segoff[s] = rel;
        rel += s + 1 == segfirst[b + 1] ? (bits + 7) / 8 : (bits + 3 + 7) / 8 + 4;  // + empty stored block
    }
    dlen[b] = rel;
}

// slice headers (IdnSliceHeader::Identifiers, u32be length, IdnIdentifierCompression::Deflate) and absolute segment offsets
__global__ void dfl_head_kernel(const unsigned long long* __restrict__ segfirst, uint32_t B, const unsigned long long* __restrict__ dlen,
                                const unsigned long long* __restrict__ slice_off, unsigned long long* __restrict__ segoff,
                                uint8_t* __restrict__ z) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const unsigned long long o = slice_off[b];
    const uint32_t n = (uint32_t)dlen[b];
    z[o] = 0x00;
    z[o + 1] = (uint8_t)(n >> 24);
    z[o + 2] = (uint8_t)(n >> 16);
    z[o + 3] = (uint8_t)(n >> 8);
    z[o + 4] = (uint8_t)n;
    z[o + 5] = 0x01;
    for (unsigned long long s = segfirst[b]; s < segfirst[b + 1]; s++) segoff[s] += o + 6;
}

// one CTA per segment: header, tokens, end of block and (not the last segment of a block) the empty stored block
__global__ void __launch_bounds__(kThreads)
dfl_emit_kernel(const unsigned long long* __restrict__ J, const unsigned long long* __restrict__ segfirst, const uint32_t* __restrict__ segblock,
                const uint32_t* __restrict__ tok, const uint16_t* __restrict__ ntok, const SegRec* __restrict__ rec,
                const unsigned long long* __restrict__ segoff, uint32_t* __restrict__ zw) {
    __shared__ uint8_t len[kLit + kDist];
    __shared__ uint16_t code[kLit + kDist];
    __shared__ uint32_t wsum[kWarps];
    const uint32_t s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const SegRec& R = rec[s];
    for (uint32_t i = tid; i < kLit + kDist; i += kThreads) len[i] = R.len[i];
    __syncthreads();
    if (tid == 0) canon_codes(len, kLit, code);
    if (tid == 32) canon_codes(len + kLit, kDist, code + kLit);
    const uint32_t b = segblock[s];
    const bool last = s + 1 == segfirst[b + 1];
    const unsigned long long a = J[b] + (s - segfirst[b]) * (unsigned long long)kSeg + tid * (unsigned long long)kSub;
    const uint32_t nt = ntok[(size_t)s * kThreads + tid];
    const uint32_t* tk = tok + a;
    uint32_t bits = 0;
    for (uint32_t i = 0; i < nt; i++) bits += tok_bits(tk[i], len);
    uint32_t x = bits;  // exclusive scan over the CTA
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= (uint32_t)o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    uint32_t before = x - bits;
    for (uint32_t w = 0; w < warp; w++) before += wsum[w];
    const unsigned long long seg_bit = segoff[s] * 8;
    BitOut out;
    if (tid == 0) {
        out.init(zw, seg_bit);
        for (uint32_t i = 0; i < R.hdr_bits; i += 8) out.put(R.hdr[i >> 3], min(8u, R.hdr_bits - i));
        out.flush();
    }
    out.init(zw, seg_bit + R.hdr_bits + before);
    for (uint32_t i = 0; i < nt; i++) {
        const uint32_t t = tk[i];
        if (!(t & 0x80000000u)) {
            out.put(code[t], len[t]);
            continue;
        }
        uint32_t eb, ev, db, dv;
        const uint32_t ls = len_sym(((t >> 16) & 0xff) + 3, eb, ev);
        const uint32_t ds = dist_sym((t & 0x7fff) + 1, db, dv);
        out.put(code[ls], len[ls]);
        if (eb) out.put(ev, eb);
        out.put(code[kLit + ds], len[kLit + ds]);
        if (db) out.put(dv, db);
    }
    if (tid == kThreads - 1) {
        out.put(code[256], len[256]);
        out.flush();
        if (!last) {  // 000 (BFINAL = 0, stored), pad to a byte, LEN = 0000, NLEN = FFFF
            const unsigned long long q = (seg_bit + R.bits + 3 + 7) & ~7ull;
            out.init(zw, q + 16);
            out.put(0xffffu, 16);
            out.flush();
        }
    } else {
        out.flush();
    }
}

// the slices of block b to out[block_off[b] + 8, ...): the room the block kernels reserved after the block header
__global__ void dfl_copy_slices_kernel(const uint8_t* __restrict__ z, const unsigned long long* __restrict__ slice_off,
                                       const unsigned long long* __restrict__ block_off, uint8_t* __restrict__ out) {
    const uint32_t b = blockIdx.x;
    const unsigned long long o = slice_off[b], n = slice_off[b + 1] - o;
    uint8_t* dst = out + block_off[b] + 8;
    for (unsigned long long i = threadIdx.x; i < n; i += blockDim.x) dst[i] = z[o + i];
}

}  // namespace dfl
}  // namespace idn
