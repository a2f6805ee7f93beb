// idn_fastq.cuh -- FASTQ text <-> symbol arrays on the device ("next" row f1 of SURVEY.md section 8f).
//
//   parse    FastqReader::read_sequence   idencomp/src/fastq/reader.rs:166-282, byte tables fastq/consts.rs:28-98
//   format   FastqWriter::write_sequence  idencomp/src/fastq/writer.rs:190-245
//
// The reference reads line by line (read_until + one table lookup per byte), which cannot feed the codec kernels.
// Here: newline index (count / scan / scatter), a scan over the LINES that composes the reader's four-state machine
// (title -> acids -> separator -> quality scores; blank lines are skipped only where a title is expected, exactly as
// parse_title does), then one thread per record validates and converts.  Same acceptance rules as the reference:
// the title starts with '@' and is trimmed, acids are ATCGN, the separator line starts with '+', quality scores are
// '!'..'~', both symbol lines have one length, a record that ends early is an error.  (Rust's trim() also strips
// non-ASCII Unicode white space; here ASCII white space only.)  The reader reports the first error in file order.
#pragma once
#include "idn_kernels.cuh"

namespace idn {

constexpr int kFqTile = 4096;  // bytes per thread block in the newline passes (256 threads x 16 bytes)

enum FastqErr : uint32_t {  // FastqReaderError variants (fastq/reader.rs:20-40)
    kFqOk = 0,
    kFqInvalidFormat = 1,
    kFqInvalidAcid = 2,
    kFqInvalidQualityScore = 3,
    kFqLengthMismatch = 4,
    kFqEof = 5,  // a record ends before its fourth line
};

__device__ __forceinline__ bool is_ascii_ws(uint8_t c) { return c == ' ' || (c >= 9 && c <= 13); }

// number of '\n' per tile
__global__ void __launch_bounds__(256)
fq_count_kernel(const uint8_t* __restrict__ text, unsigned long long n, unsigned long long* __restrict__ tile_cnt) {
    __shared__ uint32_t warp_cnt[8];
    const unsigned long long base = (unsigned long long)blockIdx.x * kFqTile + threadIdx.x * 16ull;
    uint32_t c = 0;
    for (int k = 0; k < 16; k++)
        if (base + k < n && text[base + k] == '\n') c++;
    for (int d = 16; d > 0; d >>= 1) c += __shfl_down_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0) warp_cnt[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < 8; w++) t += warp_cnt[w];
        tile_cnt[blockIdx.x] = t;
    }
}

struct TileCntFn {
    const unsigned long long* v;
    __device__ __forceinline__ unsigned long long operator()(uint64_t i) const { return v[i]; }
};

// line_start[k + 1] = position after the k-th '\n'; line_start[0] = 0.  Thread order inside a tile = byte order.
__global__ void __launch_bounds__(256)
fq_scatter_kernel(const uint8_t* __restrict__ text, unsigned long long n, const unsigned long long* __restrict__ tile_base,
                  unsigned long long* __restrict__ line_start) {
    __shared__ uint32_t warp_cnt[8];
    const unsigned long long base = (unsigned long long)blockIdx.x * kFqTile + threadIdx.x * 16ull;
    uint32_t mask = 0;
    for (int k = 0; k < 16; k++)
        if (base + k < n && text[base + k] == '\n') mask |= 1u << k;
    uint32_t c = __popc(mask), inc = c;
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if ((threadIdx.x & 31) >= (uint32_t)d) inc += o;
    }
    if ((threadIdx.x & 31) == 31) warp_cnt[threadIdx.x >> 5] = inc;
    __syncthreads();
    uint32_t before = inc - c;
    for (uint32_t w = 0; w < (threadIdx.x >> 5); w++) before += warp_cnt[w];
    unsigned long long k0 = tile_base[blockIdx.x] + before;
    if (blockIdx.x == 0 && threadIdx.x == 0) line_start[0] = 0;
    while (mask) {
        int k = __ffs(mask) - 1;
        mask &= mask - 1;
        line_start[++k0] = base + k + 1;
    }
}

// The reader as a state machine over lines: state = which line of a record is expected (0 title, 1 acids,
// 2 separator, 3 quality scores).  A blank line is skipped when a title is expected (parse_title's loop), every other
// line advances.  A line is a function state -> state, packed 2 bits per input state; composition is associative, so
// the state in front of every line is an exclusive scan.
__device__ __forceinline__ uint32_t fst_compose(uint32_t f, uint32_t g) {  // first f, then g
    uint32_t r = 0;
    for (int s = 0; s < 4; s++) r |= ((g >> (2 * ((f >> (2 * s)) & 3))) & 3) << (2 * s);
    return r;
}
constexpr uint32_t kFstIdentity = 0xE4;  // 3,2,1,0 -> themselves
constexpr uint32_t kFstAdvance = 0x39;   // 0->1, 1->2, 2->3, 3->0
constexpr uint32_t kFstBlank = 0x38;     // as advance, but 0->0

__device__ __forceinline__ uint32_t fq_line_fn(const uint8_t* __restrict__ text, unsigned long long lo, unsigned long long hi) {
    for (unsigned long long p = lo; p < hi; p++)
        if (!is_ascii_ws(text[p])) return kFstAdvance;
    return kFstBlank;
}

constexpr int kFstItems = 8;
constexpr int kFstTile = 256 * kFstItems;

// line k spans [line_start[k], line_end(k)) with line_end = line_start[k + 1] - 1 for terminated lines, n for the last
__device__ __forceinline__ unsigned long long fq_line_end(const unsigned long long* __restrict__ line_start, uint64_t k,
                                                          uint64_t n_lines, uint64_t n_newlines, unsigned long long n) {
    return k < n_newlines ? line_start[k + 1] - 1 : n;
}

__global__ void __launch_bounds__(256)
fst_reduce_kernel(const uint8_t* __restrict__ text, unsigned long long n, const unsigned long long* __restrict__ line_start,
                  uint64_t n_lines, uint64_t n_newlines, uint8_t* __restrict__ line_fn, uint8_t* __restrict__ tile_fn) {
    __shared__ uint8_t s_fn[256];
    uint64_t base = (uint64_t)blockIdx.x * kFstTile + (uint64_t)threadIdx.x * kFstItems;
    uint32_t f = kFstIdentity;
    for (int k = 0; k < kFstItems; k++) {
        uint64_t l = base + k;
        if (l < n_lines) {
            uint32_t g = fq_line_fn(text, line_start[l], fq_line_end(line_start, l, n_lines, n_newlines, n));
            line_fn[l] = (uint8_t)g;
            f = fst_compose(f, g);
        }
    }
    s_fn[threadIdx.x] = (uint8_t)f;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = kFstIdentity;
        for (int i = 0; i < 256; i++) t = fst_compose(t, s_fn[i]);
        tile_fn[blockIdx.x] = (uint8_t)t;
    }
}

// exclusive scan of the tile functions applied to the start state 0 -> state in front of every tile.  One CTA: every
// thread composes a contiguous run of tiles, thread 0 chains the 256 results, every thread replays its run.
__global__ void __launch_bounds__(256)
fst_tiles_kernel(const uint8_t* __restrict__ tile_fn, uint64_t n_tiles, uint8_t* __restrict__ tile_state) {
    __shared__ uint8_t s_fn[256];
    __shared__ uint8_t s_state[257];
    const uint64_t per = (n_tiles + 255) / 256;
    const uint64_t t0 = threadIdx.x * per, t1 = t0 + per < n_tiles ? t0 + per : n_tiles;
    uint32_t f = kFstIdentity;
    for (uint64_t t = t0; t < t1; t++) f = fst_compose(f, tile_fn[t]);
    s_fn[threadIdx.x] = (uint8_t)f;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (int i = 0; i < 256; i++) {
            s_state[i] = (uint8_t)s;
            s = (s_fn[i] >> (2 * s)) & 3;
        }
        s_state[256] = (uint8_t)s;
    }
    __syncthreads();
    uint32_t s = s_state[threadIdx.x];
    for (uint64_t t = t0; t < t1; t++) {
        tile_state[t] = (uint8_t)s;
        s = (tile_fn[t] >> (2 * s)) & 3;
    }
    if (threadIdx.x == 0) tile_state[n_tiles] = s_state[256];
}

// state in front of every line; is_title[l] = the line is the title of a record
__global__ void __launch_bounds__(256)
fst_apply_kernel(const uint8_t* __restrict__ line_fn, uint64_t n_lines, const uint8_t* __restrict__ tile_state,
                 uint8_t* __restrict__ line_state) {
    __shared__ uint8_t s_fn[256];
    uint64_t base = (uint64_t)blockIdx.x * kFstTile + (uint64_t)threadIdx.x * kFstItems;
    uint32_t f = kFstIdentity;
    for (int k = 0; k < kFstItems; k++)
        if (base + k < n_lines) f = fst_compose(f, line_fn[base + k]);
    s_fn[threadIdx.x] = (uint8_t)f;
    __syncthreads();
    // state in front of this thread's first line: tile state through the functions of the threads before it
    uint32_t s = tile_state[blockIdx.x];
    for (uint32_t i = 0; i < threadIdx.x; i++) s = (s_fn[i] >> (2 * s)) & 3;
    for (int k = 0; k < kFstItems; k++) {
        uint64_t l = base + k;
        if (l < n_lines) {
            line_state[l] = (uint8_t)s;
            s = (line_fn[l] >> (2 * s)) & 3;
        }
    }
}

struct TitleFlag {  // 1 for lines that open a record: a title is expected and the line is not blank
    const uint8_t* line_state;
    const uint8_t* line_fn;
    __device__ __forceinline__ unsigned long long operator()(uint64_t l) const {
        return line_state[l] == 0 && line_fn[l] == kFstAdvance;
    }
};

__global__ void __launch_bounds__(256)
fq_titles_kernel(TitleFlag fn, uint64_t n_lines, const unsigned long long* __restrict__ rec_scan, unsigned long long* __restrict__ title_line) {
    uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_lines) return;
    if (fn(l)) title_line[rec_scan[l]] = l;
}

struct FastqView {
    const uint8_t* text;
    unsigned long long n;
    const unsigned long long* line_start;
    uint64_t n_lines, n_newlines;
    const unsigned long long* title_line;  // [n_reads]
    uint64_t n_reads;
};

// per record: trimmed name span and symbol count; a title without '@'.  Every other check is fq_convert_kernel's, so
// that a record's checks run in the reference's order and the lowest record wins the atomicMin.
__global__ void __launch_bounds__(128)
fq_lengths_kernel(FastqView V, unsigned long long* __restrict__ name_lo, uint32_t* __restrict__ name_len,
                  uint32_t* __restrict__ read_len, unsigned long long* __restrict__ first_err) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= V.n_reads) return;
    const uint64_t t = V.title_line[r];
    unsigned long long lo = V.line_start[t], hi = fq_line_end(V.line_start, t, V.n_lines, V.n_newlines, V.n);
    uint32_t err = kFqOk;
    if (V.text[lo] != '@') err = kFqInvalidFormat;  // line.starts_with('@') on the untrimmed line (reader.rs:199-201)
    lo++;
    while (lo < hi && is_ascii_ws(V.text[lo])) lo++;  // line[1..].trim()
    while (hi > lo && is_ascii_ws(V.text[hi - 1])) hi--;
    name_lo[r] = lo;
    name_len[r] = err ? 0 : (uint32_t)(hi - lo);
    uint32_t len = 0;
    if (t + 3 < V.n_lines)  // a record cut short is fq_convert_kernel's to report
        len = (uint32_t)(fq_line_end(V.line_start, t + 1, V.n_lines, V.n_newlines, V.n) - V.line_start[t + 1]);
    read_len[r] = len;
    if (err) atomicMin(first_err, (r << 8) | err);
}

struct U32Fn {
    const uint32_t* v;
    __device__ __forceinline__ unsigned long long operator()(uint64_t i) const { return v[i]; }
};

// The last record, cut short at the end of the text: the lines it has are checked in the reference's order before
// EofReached.  Only its error matters, so nothing is written.  Kept out of line so that it costs fq_convert_kernel no
// registers.
__device__ __noinline__ uint32_t fq_cut_short_err(FastqView V, uint64_t t) {
    if (t + 1 >= V.n_lines) return kFqEof;
    const unsigned long long a_lo = V.line_start[t + 1], a_hi = fq_line_end(V.line_start, t + 1, V.n_lines, V.n_newlines, V.n);
    for (unsigned long long p = a_lo; p < a_hi; p++) {
        const uint8_t c = V.text[p];
        if (c != 'A' && c != 'C' && c != 'T' && c != 'G' && c != 'N') return kFqInvalidAcid;
    }
    if (t + 2 >= V.n_lines) return kFqEof;
    const unsigned long long s_lo = V.line_start[t + 2], s_hi = fq_line_end(V.line_start, t + 2, V.n_lines, V.n_newlines, V.n);
    if (s_hi == s_lo || V.text[s_lo] != '+') return kFqInvalidFormat;
    return kFqEof;
}

// per record: name bytes, acids and quality scores through the reference's byte tables.  The checks run in the
// reference's order: acids, the separator, every byte of the quality line, then the lengths.
__global__ void __launch_bounds__(128)
fq_convert_kernel(FastqView V, const unsigned long long* __restrict__ name_lo, const unsigned long long* __restrict__ name_off,
                  const unsigned long long* __restrict__ read_off, uint8_t* __restrict__ names, uint8_t* __restrict__ acids,
                  uint8_t* __restrict__ quals, unsigned long long* __restrict__ first_err) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= V.n_reads) return;
    const uint64_t t = V.title_line[r];
    if (t + 3 >= V.n_lines) {
        atomicMin(first_err, (r << 8) | fq_cut_short_err(V, t));
        return;
    }
    const uint32_t nl = (uint32_t)(name_off[r + 1] - name_off[r]);
    for (uint32_t i = 0; i < nl; i++) names[name_off[r] + i] = V.text[name_lo[r] + i];
    const unsigned long long a_lo = V.line_start[t + 1], a_hi = fq_line_end(V.line_start, t + 1, V.n_lines, V.n_newlines, V.n);
    const unsigned long long s_lo = V.line_start[t + 2], s_hi = fq_line_end(V.line_start, t + 2, V.n_lines, V.n_newlines, V.n);
    const unsigned long long q_lo = V.line_start[t + 3], q_hi = fq_line_end(V.line_start, t + 3, V.n_lines, V.n_newlines, V.n);
    uint32_t err = kFqOk;
    const uint32_t len = (uint32_t)(a_hi - a_lo);
    FwdReader ra, rq;
    ra.start(V.text + a_lo);
    rq.start(V.text + q_lo);
    FwdWriter oa, oq;
    oa.init(acids + read_off[r]);
    oq.init(quals + read_off[r]);
    for (uint32_t i = 0; i < len; i++) {
        uint32_t c = ra.get(), a;
        // FASTQ_BYTE_TO_ACID (consts.rs:41-51): N=0 A=1 C=2 T=3 G=4 (sequence.rs:401-413)
        if (c == 'A') a = 1; else if (c == 'C') a = 2; else if (c == 'T') a = 3; else if (c == 'G') a = 4; else if (c == 'N') a = 0;
        else {
            a = 0;
            if (!err) err = kFqInvalidAcid;
        }
        oa.push(a);
    }
    oa.finish();
    if (!err && (s_hi == s_lo || V.text[s_lo] != '+')) err = kFqInvalidFormat;  // parse_separator (reader.rs:236-247)
    const uint32_t qlen = (uint32_t)(q_hi - q_lo);
    const uint32_t m = qlen < len ? qlen : len;
    for (uint32_t i = 0; i < m; i++) {
        uint32_t c = rq.get();
        if (c < '!' || c > '~') {  // FASTQ_VALID_Q_SCORE_BYTES (consts.rs:53-63)
            if (!err) err = kFqInvalidQualityScore;
            c = '!';
        }
        oq.push(c - '!');
    }
    for (uint32_t i = m; i < len; i++) oq.push(0);
    oq.finish();
    if (!err && qlen > len) {  // the reference converts the whole line before it compares the lengths
        for (uint32_t i = len; i < qlen; i++) {
            uint8_t c = V.text[q_lo + i];
            if (c < '!' || c > '~') {
                err = kFqInvalidQualityScore;
                break;
            }
        }
    }
    if (!err && qlen != len) err = kFqLengthMismatch;
    if (err) atomicMin(first_err, (r << 8) | err);
}

// ---- format: "@name\nACGT\n+[name]\n!!!!\n" per record (writer.rs:190-245) ----
struct FormatSize {
    const uint64_t* read_off;
    const uint64_t* name_off;  // may be nullptr: empty names
    int title_with_separator;
    __device__ __forceinline__ unsigned long long operator()(uint64_t r) const {
        unsigned long long len = read_off[r + 1] - read_off[r];
        unsigned long long nl = name_off ? name_off[r + 1] - name_off[r] : 0;
        return 1 + nl + 1 + len + 1 + 1 + (title_with_separator ? nl : 0) + 1 + len + 1;
    }
};

__global__ void __launch_bounds__(128)
fq_format_kernel(const uint8_t* __restrict__ acids, const uint8_t* __restrict__ quals, const uint64_t* __restrict__ read_off,
                 const uint8_t* __restrict__ names, const uint64_t* __restrict__ name_off, uint64_t n_reads,
                 int title_with_separator, const unsigned long long* __restrict__ text_off, uint8_t* __restrict__ text,
                 uint64_t cap, uint32_t* __restrict__ err) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    if (text_off[r + 1] > cap) return;
    const unsigned long long off = read_off[r];
    const uint32_t len = (uint32_t)(read_off[r + 1] - off);
    const unsigned long long no = name_off ? name_off[r] : 0;
    const uint32_t nl = name_off ? (uint32_t)(name_off[r + 1] - no) : 0;
    FwdWriter w;
    w.init(text + text_off[r]);
    w.push('@');
    for (uint32_t i = 0; i < nl; i++) w.push(names[no + i]);
    w.push('\n');
    bool bad = false;
    FwdReader ra, rq;
    ra.start(acids + off);
    rq.start(quals + off);
    for (uint32_t i = 0; i < len; i++) {
        uint32_t a = ra.get();
        if (a > 4) {
            bad = true;
            a = 0;
        }
        w.push(a == 0 ? 'N' : a == 1 ? 'A' : a == 2 ? 'C' : a == 3 ? 'T' : 'G');  // FASTQ_ACID_TO_BYTE (consts.rs:77-87)
    }
    w.push('\n');
    w.push('+');
    if (title_with_separator)
        for (uint32_t i = 0; i < nl; i++) w.push(names[no + i]);
    w.push('\n');
    for (uint32_t i = 0; i < len; i++) {
        uint32_t q = rq.get();
        if (q > 93) {
            bad = true;
            q = 0;
        }
        w.push('!' + q);
    }
    w.push('\n');
    w.finish();
    if (bad) atomicOr(err, 1u);
}

}  // namespace idn
