// idn_native.cuh -- the GPU-native multi-lane block format (container version 2).  See DESIGN.md section 8.
//
// Same tables, context specs, scale bits and symbol order inside a read as the reference format; only stream
// segmentation and framing change (SURVEY.md section 7): instead of one rANS stream + 9-byte slice header + 8 flush
// bytes per read, a block carries one NativeLanes slice whose reads are cut into lanes of about `lane_syms` symbols,
// each lane one 2-state rANS stream over whole reads (generators restart at every read, states run on).
//
//   0x03                                  slice kind NativeLanes (new in version 2)
//   u32be body_len                        bytes that follow this field
//   u32be n_reads | u32be n_lanes | u32be lane_syms | u8 len_width (0, 2 or 4) | u32be const_len
//   n_reads x len_width bytes             read lengths, big endian (absent when len_width == 0: all = const_len)
//   n_lanes x {u8 acid model, u8 q model} container model indices per lane
//   n_lanes x u32be                       lane payload lengths
//   lane payloads, back to back
//
// Lane partition (recomputed by the decoder from the lengths).  A read is ONE piece, unless lane_syms >= 256 and the read
// is longer than lane_syms: then it is cut into ceil(len / lane_syms) pieces of lane_syms symbols (the last one shorter).
// With o_p the block-relative offset of the first symbol of piece p, a new lane starts at the first piece of the block and
// at every piece with o_p / lane_syms != o_(p-1) / lane_syms.  A lane is thus a contiguous range of the block's symbol
// stream; bit 7 of len_width is set when some read of the block is cut (then there may be more lanes than reads).
// Lane payload: [16 history bytes][state 1 (q) LE][state 0 (acid) LE][renormalisation bytes]; the symbols of the lane are
// pushed last -> first, every position with the contexts it has inside its whole read.  The history bytes exist only
// when the lane starts inside a read: the acids and then the quality scores of the 8 positions in front of the lane, from
// which the decoder rebuilds the generator states (no legal spec type looks further back than 8 symbols; long reads thus
// decode with as many independent chains as they have lanes instead of one chain of 10-20 k positions per read).
// Model choice per lane: argmin of the summed forward scores of the reads that have a symbol in the lane.
#pragma once
#include "idn_kernels.cuh"

namespace idn {

constexpr uint32_t kNativeHdrFixed = 1 + 4 + 4 + 4 + 4 + 1 + 4;  // kind .. const_len = 22 bytes

__device__ __forceinline__ void store_u32be(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24);
    p[1] = (uint8_t)(v >> 16);
    p[2] = (uint8_t)(v >> 8);
    p[3] = (uint8_t)v;
}

// ---------------------------------------------------------------------------------------------------
// compress side
// ---------------------------------------------------------------------------------------------------
constexpr uint32_t kNativeMinSplitQ = 256;  // reads are only cut into pieces when the lane quantum is at least this
constexpr uint32_t kNativeHistBytes = 2 * kHist;

__host__ __device__ __forceinline__ uint32_t native_pieces(uint32_t len, uint32_t Q) {
    return (Q >= kNativeMinSplitQ && len > Q) ? (len + Q - 1) / Q : 1u;
}

// number of lanes read r opens: its first piece if it crosses into a new quantum (or starts the block), and every
// further piece
struct LaneCount {
    const uint64_t* read_off;
    const uint32_t* block_first;
    const uint32_t* read_block;
    uint32_t lane_syms;
    __device__ __forceinline__ bool first_piece_opens(uint64_t r) const {
        const uint32_t b = read_block[r];
        const uint64_t r0 = block_first[b];
        if (r == r0) return true;
        const uint64_t base = read_off[r0];
        const uint32_t plen = (uint32_t)(read_off[r] - read_off[r - 1]);
        const uint64_t prev_last = (read_off[r - 1] - base) + (uint64_t)(native_pieces(plen, lane_syms) - 1) * lane_syms;
        return (read_off[r] - base) / lane_syms != prev_last / lane_syms;
    }
    __device__ __forceinline__ unsigned long long operator()(uint64_t r) const {
        const uint32_t len = (uint32_t)(read_off[r + 1] - read_off[r]);
        return (first_piece_opens(r) ? 1u : 0u) + native_pieces(len, lane_syms) - 1;
    }
};

// lane_first[l] = the read lane l starts in, lane_sym[l] = absolute offset of its first symbol (scatter by the scanned
// counts); terminators lane_first[n_lanes] = n_reads, lane_sym[n_lanes] = n_symbols
__global__ void __launch_bounds__(256)
lane_scatter_kernel(LaneCount fn, uint64_t n_reads, const unsigned long long* __restrict__ lane_scan /*[n_reads+1]*/,
                    uint32_t* __restrict__ lane_first, unsigned long long* __restrict__ lane_sym) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r == 0) {
        lane_first[lane_scan[n_reads]] = (uint32_t)n_reads;
        lane_sym[lane_scan[n_reads]] = fn.read_off[n_reads];
    }
    if (r >= n_reads) return;
    unsigned long long l = lane_scan[r];
    const uint32_t len = (uint32_t)(fn.read_off[r + 1] - fn.read_off[r]);
    const uint32_t pc = native_pieces(len, fn.lane_syms);
    if (fn.first_piece_opens(r)) {
        lane_first[l] = (uint32_t)r;
        lane_sym[l] = fn.read_off[r];
        l++;
    }
    for (uint32_t j = 1; j < pc; j++, l++) {
        lane_first[l] = (uint32_t)r;
        lane_sym[l] = fn.read_off[r] + (unsigned long long)j * fn.lane_syms;
    }
}

// per-lane model choice: argmin over the candidates of a type of the summed forward scores of the reads that have a symbol
// in the lane (first minimum wins, as everywhere in the reference's choosers); one thread per (lane, type)
__global__ void __launch_bounds__(128)
lane_choose_kernel(const uint32_t* __restrict__ sizes, uint32_t n_cols, const uint32_t* __restrict__ cand_cols,
                   const uint32_t* __restrict__ n_cand2, const uint32_t* __restrict__ has_sizes,
                   const uint32_t* __restrict__ lane_first, const unsigned long long* __restrict__ lane_sym,
                   const uint64_t* __restrict__ read_off, uint64_t n_reads, const unsigned long long* __restrict__ n_lanes_dev,
                   uint64_t lane_cap, uint8_t* __restrict__ lane_choice /*[2][lane_cap]*/) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t l = t >> 1;
    uint32_t type = (uint32_t)t & 1;
    if (l >= *n_lanes_dev) return;
    uint32_t best = 0;
    if (has_sizes[type]) {
        const unsigned long long a = lane_sym[l], b = lane_sym[l + 1];
        unsigned long long best_sum = ~0ull;
        for (uint32_t k = 0; k < n_cand2[type]; k++) {
            uint32_t col = cand_cols[type * kMaxCand + k];
            unsigned long long sum = 0;
            for (uint64_t r = lane_first[l]; r < n_reads && read_off[r] < b; r++)
                if (read_off[r + 1] > a) sum += sizes[r * n_cols + col];
            if (sum < best_sum) {
                best_sum = sum;
                best = k;
            }
        }
    }
    lane_choice[(size_t)type * lane_cap + l] = (uint8_t)best;
}

struct EncodeLaneArgs {
    const ModelDev* models;
    const uint8_t* acids;
    const uint8_t* quals;
    uint64_t n_symbols;
    const uint64_t* read_off;
    uint64_t n_reads;
    const uint32_t* lane_first;   // [n_lanes+1] read the lane starts in
    const unsigned long long* lane_sym;  // [n_lanes+1] absolute offset of the lane's first symbol
    const unsigned long long* n_lanes_dev;
    uint64_t lane_cap;            // stride of the [2][lane_cap] arrays
    const uint8_t* lane_choice;   // [2][lane_cap] candidate index per type, or nullptr (single pair)
    const int32_t* cand_model;    // [2][kMaxCand] candidate -> models[] index
    uint8_t* scratch;             // slot of lane l ends at 4 * lane_sym[l+1] + kLaneSlotExtra * (l+1)
    uint32_t* lane_len;           // [n_lanes]
    uint32_t* err;
};
constexpr unsigned long long kLaneSlotExtra = 8 + kNativeHistBytes;  // two flushed states + the history of a lane that starts inside a read

#ifndef IDN_LANE_MINB
#define IDN_LANE_MINB 8
#endif
template <bool kUniform, class P>
__device__ __forceinline__ void encode_lane_one(const EncodeLaneArgs& A, const ModelDev& MA, const ModelDev& MQ, uint64_t l64) {
    const uint32_t l = (uint32_t)l64;
    const uint32_t r_lo = A.lane_first[l];
    int32_t ia = 0, iq = 0;
    if (!kUniform) {
        ia = A.cand_model[A.lane_choice ? A.lane_choice[l] : 0];
        iq = A.cand_model[kMaxCand + (A.lane_choice ? A.lane_choice[A.lane_cap + l] : 0)];
    }
    const ModelDev& ma = kUniform ? MA : A.models[ia];
    const ModelDev& mq = kUniform ? MQ : A.models[iq];
    EncStream S;
    EncCrc C{nullptr, 0u, 0u};  // (the native path takes its CRC partials from crc_read_kernel)
    S.begin(A.scratch + 4ull * A.lane_sym[l + 1] + kLaneSlotExtra * ((unsigned long long)l + 1));
    if (A.lane_sym[l + 1] > A.lane_sym[l]) {
        // the last read with a symbol in the lane, then down to the first
        uint32_t r = A.lane_first[l + 1] < A.n_reads ? A.lane_first[l + 1] : (uint32_t)A.n_reads - 1;
        while (r > r_lo && A.read_off[r] >= A.lane_sym[l + 1]) r--;
#pragma unroll 1
        for (;; r--) {
            const unsigned long long a = A.lane_sym[l], b = A.lane_sym[l + 1];
            const unsigned long long ro = A.read_off[r], re = A.read_off[r + 1];
            if (re > a && ro < b) {
                const uint32_t p0 = (uint32_t)((a > ro ? a : ro) - ro), p1 = (uint32_t)((b < re ? b : re) - ro);
                encode_read_body<P>(ma, mq, A.acids, A.quals, A.n_symbols, (long long)ro, (uint32_t)(re - ro), p0, p1, S, C);
            }
            if (r == r_lo) break;
        }
    }
    S.flush_states();
    {
        const unsigned long long a = A.lane_sym[l], b = A.lane_sym[l + 1];
        if (b > a && a > A.read_off[r_lo]) {
            // the lane starts inside a read: the symbols of the kHist positions in front of it go in front of the stream,
            // acids then quality scores in position order (the writer walks down: last word first)
            const uint8_t* ha = A.acids + a - kHist;
            const uint8_t* hq = A.quals + a - kHist;
            auto word = [](const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); };
            S.out.push_u32_le(word(hq + 4));
            S.out.push_u32_le(word(hq));
            S.out.push_u32_le(word(ha + 4));
            S.out.push_u32_le(word(ha));
        }
    }
    S.out.finish();
    A.lane_len[l] = S.total(A.scratch + 4ull * A.lane_sym[l + 1] + kLaneSlotExtra * ((unsigned long long)l + 1));
    if (S.bad) atomicOr(A.err, 1u);
}

template <bool kUniform, class P>
__global__ void __launch_bounds__(128, kUniform ? IDN_LANE_MINB : 1)
encode_lane_kernel(EncodeLaneArgs A, const ModelDev MA, const ModelDev MQ) {
    // (register budget: the per-position loop inside encode_read_body is what counts, so the lane bounds are re-read from
    // memory per read instead of being kept in registers across it)
    const uint64_t l64 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l64 >= *A.n_lanes_dev) return;
    encode_lane_one<kUniform, P>(A, MA, MQ, l64);
}

// per-lane model selection: the lanes that chose one model pair (a bucket of bucket_scatter_kernel), see encode_list_kernel
template <class P>
__global__ void __launch_bounds__(128, IDN_LANE_MINB)
encode_lane_list_kernel(EncodeLaneArgs A, const ModelDev MA, const ModelDev MQ, ReadList L) {
    const uint32_t n = *L.count;
    const uint32_t* __restrict__ list = L.list + *L.base;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        encode_lane_one<true, P>(A, MA, MQ, list[i]);
}

struct EncodeLanePairKey {  // compress side: the candidates lane_choose_kernel picked
    const uint8_t* lane_choice;  // [2][lane_cap]
    const unsigned long long* n_lanes_dev;
    uint64_t lane_cap;
    uint32_t n_q;
    __device__ __forceinline__ uint32_t operator()(uint64_t l) const {
        return l < *n_lanes_dev ? (uint32_t)lane_choice[l] * n_q + lane_choice[lane_cap + l] : 0xffffffffu;
    }
};

struct LaneLenFn {
    const uint32_t* lane_len;
    const unsigned long long* n_lanes_dev;
    __device__ __forceinline__ unsigned long long operator()(uint64_t l) const { return l < *n_lanes_dev ? lane_len[l] : 0; }
};

// per block: min / max read length (one CTA per block) -> len_width, and the lane range of the block
__global__ void __launch_bounds__(256)
native_block_info_kernel(const uint64_t* __restrict__ read_off, const uint32_t* __restrict__ block_first, uint32_t n_blocks,
                         const unsigned long long* __restrict__ lane_scan /*[n_reads+1]*/, uint32_t lane_syms,
                         uint32_t* __restrict__ blk_width /* bit 7: a read of the block is cut into pieces */,
                         uint32_t* __restrict__ blk_const_len, uint32_t* __restrict__ blk_lane0 /*[n_blocks+1]*/) {
    __shared__ uint32_t s_min[256], s_max[256];
    uint32_t b = blockIdx.x;
    if (b >= n_blocks) return;
    uint64_t r0 = block_first[b], r1 = block_first[b + 1];
    uint32_t mn = 0xffffffffu, mx = 0;
    for (uint64_t r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
        uint32_t len = (uint32_t)(read_off[r + 1] - read_off[r]);
        mn = min(mn, len);
        mx = max(mx, len);
    }
    s_min[threadIdx.x] = mn;
    s_max[threadIdx.x] = mx;
    __syncthreads();
    for (uint32_t d = 128; d > 0; d >>= 1) {
        if (threadIdx.x < d) {
            s_min[threadIdx.x] = min(s_min[threadIdx.x], s_min[threadIdx.x + d]);
            s_max[threadIdx.x] = max(s_max[threadIdx.x], s_max[threadIdx.x + d]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        mn = s_min[0];
        mx = s_max[0];
        bool is_const = r1 == r0 || mn == mx;
        blk_width[b] = (is_const ? 0u : (mx < 65536u ? 2u : 4u)) | ((r1 > r0 && native_pieces(mx, lane_syms) > 1) ? 0x80u : 0u);
        blk_const_len[b] = (is_const && r1 > r0) ? mn : 0u;
        blk_lane0[b] = (uint32_t)lane_scan[r0];
        if (b == n_blocks - 1) blk_lane0[n_blocks] = (uint32_t)lane_scan[r1];
    }
}

// sequential over blocks (hundreds): block offsets and block headers of the native container
__global__ void __launch_bounds__(32)
native_layout_kernel(const uint32_t* __restrict__ block_first, uint32_t n_blocks, const uint32_t* __restrict__ prefix_len,
                     const uint32_t* __restrict__ blk_width, const uint32_t* __restrict__ blk_lane0,
                     const unsigned long long* __restrict__ lane_off /*[n_lanes+1]*/, unsigned long long* __restrict__ block_off,
                     uint8_t* __restrict__ out, uint64_t out_cap, unsigned long long* __restrict__ stats) {
    if (threadIdx.x != 0) return;
    unsigned long long pos = 0;
    for (uint32_t b = 0; b < n_blocks; b++) {
        block_off[b] = pos;
        unsigned long long n_reads = block_first[b + 1] - block_first[b];
        unsigned long long n_lanes = blk_lane0[b + 1] - blk_lane0[b];
        unsigned long long pre = prefix_len ? prefix_len[b] : 0;
        unsigned long long length = pre;
        if (n_reads)
            length += kNativeHdrFixed + n_reads * (blk_width[b] & 0x7fu) + n_lanes * 6 + (lane_off[blk_lane0[b + 1]] - lane_off[blk_lane0[b]]);
        if (pos + 8 <= out_cap) store_u32be(out + pos, (uint32_t)length);
        pos += 8 + length;
    }
    block_off[n_blocks] = pos;
    stats[0] = pos;
    stats[3] = lane_off[blk_lane0[n_blocks]];  // payload bytes
}

struct NativeAssembleArgs {
    const uint64_t* read_off;
    const uint32_t* block_first;
    uint32_t n_blocks;
    const uint32_t* prefix_len;
    const uint32_t* blk_width;
    const uint32_t* blk_const_len;
    const uint32_t* blk_lane0;
    const uint32_t* lane_first;
    const unsigned long long* lane_sym;
    const uint32_t* lane_len;
    const unsigned long long* lane_off;
    const uint8_t* lane_choice;   // [2][lane_cap] or nullptr
    const uint8_t* cand_index;    // [2][kMaxCand] candidate -> container model index
    const unsigned long long* n_lanes_dev;
    uint64_t lane_cap;
    uint32_t lane_syms;
    const unsigned long long* block_off;
    uint8_t* out;
    uint64_t out_cap;
};

// one CTA per block: the NativeLanes slice header and its three tables
__global__ void __launch_bounds__(256)
native_header_kernel(NativeAssembleArgs A) {
    uint32_t b = blockIdx.x;
    if (b >= A.n_blocks) return;
    const uint64_t r0 = A.block_first[b], r1 = A.block_first[b + 1];
    const uint32_t n_reads = (uint32_t)(r1 - r0);
    if (n_reads == 0) return;
    const uint32_t l0 = A.blk_lane0[b], l1 = A.blk_lane0[b + 1], n_lanes = l1 - l0;
    const uint32_t w = A.blk_width[b] & 0x7fu;
    const unsigned long long pay = A.lane_off[l1] - A.lane_off[l0];
    const unsigned long long body = kNativeHdrFixed - 5 + (unsigned long long)n_reads * w + 6ull * n_lanes + pay;
    unsigned long long base = A.block_off[b] + 8 + (A.prefix_len ? A.prefix_len[b] : 0);
    if (base + 5 + body > A.out_cap) return;  // IDN_E_NOSPACE is reported by the host from stats
    uint8_t* p = A.out + base;
    if (threadIdx.x == 0) {
        p[0] = 3;
        store_u32be(p + 1, (uint32_t)body);
        store_u32be(p + 5, n_reads);
        store_u32be(p + 9, n_lanes);
        store_u32be(p + 13, A.lane_syms);
        p[17] = (uint8_t)A.blk_width[b];
        store_u32be(p + 18, A.blk_const_len[b]);
    }
    uint8_t* t_len = p + kNativeHdrFixed;
    uint8_t* t_mdl = t_len + (size_t)n_reads * w;
    uint8_t* t_ll = t_mdl + 2ull * n_lanes;
    if (w)
        for (uint32_t i = threadIdx.x; i < n_reads; i += blockDim.x) {
            uint32_t len = (uint32_t)(A.read_off[r0 + i + 1] - A.read_off[r0 + i]);
            if (w == 2) {
                t_len[2 * i] = (uint8_t)(len >> 8);
                t_len[2 * i + 1] = (uint8_t)len;
            } else {
                store_u32be(t_len + 4ull * i, len);
            }
        }
    for (uint32_t i = threadIdx.x; i < n_lanes; i += blockDim.x) {
        uint32_t ca = A.lane_choice ? A.lane_choice[l0 + i] : 0, cq = A.lane_choice ? A.lane_choice[A.lane_cap + l0 + i] : 0;
        t_mdl[2 * i] = A.cand_index[ca];
        t_mdl[2 * i + 1] = A.cand_index[kMaxCand + cq];
        store_u32be(t_ll + 4ull * i, A.lane_len[l0 + i]);
    }
}

// one warp per lane: payload copy from the scratch slot to its place in the block
__global__ void __launch_bounds__(256)
native_copy_kernel(NativeAssembleArgs A, const uint8_t* __restrict__ scratch, const uint32_t* __restrict__ lane_block) {
    uint64_t l = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t lane = threadIdx.x & 31;
    if (l >= *A.n_lanes_dev) return;
    uint32_t b = lane_block[l];
    const uint32_t n_reads = A.block_first[b + 1] - A.block_first[b];
    const uint32_t l0 = A.blk_lane0[b], n_lanes = A.blk_lane0[b + 1] - l0;
    unsigned long long dst = A.block_off[b] + 8 + (A.prefix_len ? A.prefix_len[b] : 0) + kNativeHdrFixed +
                             (unsigned long long)n_reads * (A.blk_width[b] & 0x7fu) + 6ull * n_lanes + (A.lane_off[l] - A.lane_off[l0]);
    const uint32_t n = A.lane_len[l];
    if (dst + n > A.out_cap) return;
    const uint8_t* src = scratch + 4ull * A.lane_sym[l + 1] + kLaneSlotExtra * (l + 1) - n;
    uint8_t* d = A.out + dst;
    // head bytes up to a 4-byte boundary of the destination, then words assembled from two aligned source words
    uint32_t head = (uint32_t)((4 - (reinterpret_cast<uintptr_t>(d) & 3)) & 3);
    if (head > n) head = n;
    if (lane < head) d[lane] = src[lane];
    const uint32_t words = (n - head) >> 2;
    const uint8_t* s2 = src + head;
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(s2) & 3);
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(s2 - sh);
    uint32_t* dw = reinterpret_cast<uint32_t*>(d + head);
    for (uint32_t i = lane; i < words; i += 32) {
        uint32_t lo = sw[i];
        uint32_t v = sh ? __funnelshift_r(lo, sw[i + 1], 8 * sh) : lo;
        dw[i] = v;
    }
    const uint32_t done = head + 4 * words;
    if (lane < n - done) d[done + lane] = src[done + lane];
}

// lane -> block map (block ranges of lanes are contiguous)
__global__ void lane_block_kernel(const uint32_t* __restrict__ blk_lane0, uint32_t n_blocks, uint32_t* __restrict__ lane_block) {
    uint32_t b = blockIdx.x;
    if (b >= n_blocks) return;
    for (uint32_t l = blk_lane0[b] + threadIdx.x; l < blk_lane0[b + 1]; l += blockDim.x) lane_block[l] = b;
}

// ---------------------------------------------------------------------------------------------------
// decompress side
// ---------------------------------------------------------------------------------------------------
struct NativeBlockHdr {  // what the header kernel leaves per block
    unsigned long long tab;  // absolute offset of the read length table in `blocks`
    uint32_t n_reads, n_lanes, lane_syms, width, const_len;
    uint32_t split;          // bit 7 of len_width: some read of the block is cut into pieces
};

// one warp per block: find the NativeLanes slice, validate its framing, count symbols
__global__ void __launch_bounds__(32)
native_hdr_kernel(const uint8_t* __restrict__ blocks, const unsigned long long* __restrict__ block_off,
                  const uint32_t* __restrict__ block_len, uint32_t n_blocks, unsigned long long blocks_bytes, uint32_t n_models,
                  const uint8_t* __restrict__ model_type, NativeBlockHdr* __restrict__ hdr,
                  unsigned long long* __restrict__ blk_reads, unsigned long long* __restrict__ blk_syms,
                  unsigned long long* __restrict__ blk_lanes, int32_t* __restrict__ status, uint32_t* __restrict__ split_flag) {
    const uint32_t b = blockIdx.x, lane = threadIdx.x;
    if (b >= n_blocks) return;
    const unsigned long long boff = block_off[b];
    const unsigned long long n = block_len ? block_len[b] : block_off[b + 1] - boff;
    int32_t st = 0;
    NativeBlockHdr h{0, 0, 0, 0, 0, 0, 0};
    if (boff > blocks_bytes || n > blocks_bytes - boff) st = 3;
    const uint8_t* p = blocks + boff;
    unsigned long long pos = 0, body_end = 0;
    bool found = false;
    if (st == 0 && lane == 0) {
        while (pos < n) {
            uint8_t kind = p[pos];
            if (kind == 0) {  // Identifiers slice: names stay on the host
                if (pos + 6 > n) { st = 3; break; }
                unsigned long long len = load_u32be(p + pos + 1);
                if (len > n - pos - 6) { st = 3; break; }
                pos += 6 + len;
            } else if (kind == 3) {
                if (found || pos + kNativeHdrFixed > n) { st = 3; break; }
                unsigned long long body = load_u32be(p + pos + 1);
                if (body > n - pos - 5 || body < kNativeHdrFixed - 5) { st = 3; break; }
                h.n_reads = load_u32be(p + pos + 5);
                h.n_lanes = load_u32be(p + pos + 9);
                h.lane_syms = load_u32be(p + pos + 13);
                h.width = p[pos + 17] & 0x7fu;
                h.split = p[pos + 17] >> 7;
                h.const_len = load_u32be(p + pos + 18);
                h.tab = boff + pos + kNativeHdrFixed;
                body_end = pos + 5 + body;
                unsigned long long need = kNativeHdrFixed - 5 + (unsigned long long)h.n_reads * h.width + 6ull * h.n_lanes;
                if ((h.width != 0 && h.width != 2 && h.width != 4) || h.lane_syms == 0 || need > body ||
                    (!h.split && h.n_lanes > h.n_reads) || (h.split && h.lane_syms < kNativeMinSplitQ) ||
                    (h.n_reads > 0) != (h.n_lanes > 0)) { st = 3; break; }
                found = true;
                pos = body_end;
            } else {
                st = 3;  // compat slices do not belong in a version 2 block
                break;
            }
        }
    }
    st = __shfl_sync(0xffffffffu, st, 0);
    h.n_reads = __shfl_sync(0xffffffffu, h.n_reads, 0);
    h.n_lanes = __shfl_sync(0xffffffffu, h.n_lanes, 0);
    h.width = __shfl_sync(0xffffffffu, h.width, 0);
    h.const_len = __shfl_sync(0xffffffffu, h.const_len, 0);
    h.split = __shfl_sync(0xffffffffu, h.split, 0);
    h.lane_syms = __shfl_sync(0xffffffffu, h.lane_syms, 0);
    h.tab = __shfl_sync(0xffffffffu, h.tab, 0);
    body_end = __shfl_sync(0xffffffffu, body_end, 0);
    unsigned long long syms = 0, pay = 0;
    if (st == 0 && h.n_reads) {
        const uint8_t* t_len = blocks + h.tab;
        const uint8_t* t_mdl = t_len + (size_t)h.n_reads * h.width;
        const uint8_t* t_ll = t_mdl + 2ull * h.n_lanes;
        if (h.width == 0) {
            if (lane == 0) syms = (unsigned long long)h.n_reads * h.const_len;  // summed over the warp below
        } else {
            for (uint32_t i = lane; i < h.n_reads; i += 32)
                syms += h.width == 2 ? (((uint32_t)t_len[2 * i] << 8) | t_len[2 * i + 1]) : load_u32be(t_len + 4ull * i);
        }
        bool bad = false, short_lane = false;
        for (uint32_t i = lane; i < h.n_lanes; i += 32) {
            uint32_t ll = load_u32be(t_ll + 4ull * i);
            pay += ll;
            uint32_t ma = t_mdl[2 * i], mq = t_mdl[2 * i + 1];
            if (ma >= n_models || mq >= n_models || model_type[ma] != 0 || model_type[mq] != 1) bad = true;
            if (ll < 8) short_lane = true;  // a lane holds at least its two flushed states (the decoder checks the history bytes)
        }
        for (int d = 16; d > 0; d >>= 1) {
            syms += __shfl_down_sync(0xffffffffu, syms, d);
            pay += __shfl_down_sync(0xffffffffu, pay, d);
        }
        bad = __any_sync(0xffffffffu, bad);
        short_lane = __any_sync(0xffffffffu, short_lane);
        if (lane == 0) {
            unsigned long long used = h.tab - boff + (unsigned long long)h.n_reads * h.width + 6ull * h.n_lanes + pay;
            if (bad) st = 7;  // IDN_E_INVALID_MODEL_INDEX
            if (short_lane || used != body_end) st = 3;
        }
        st = __shfl_sync(0xffffffffu, st, 0);
    }
    if (lane == 0) {
        hdr[b] = h;
        if (st == 0 && h.split) atomicOr(split_flag, 1u);
        blk_reads[b] = st == 0 ? h.n_reads : 0;
        blk_syms[b] = st == 0 ? syms : 0;
        blk_lanes[b] = st == 0 ? h.n_lanes : 0;
        if (st != 0) {
            int old = atomicCAS(&status[0], 0, st);
            if (old == 0) status[1] = (int32_t)b;
        }
    }
}

struct NativeIndex {  // per lane, global lane numbering
    unsigned long long* pay_off;     // absolute offset of the lane payload in `blocks`
    uint32_t* pay_len;
    unsigned long long* first_read;  // [n_lanes + 1]  global index of the read the lane starts in
    unsigned long long* sym_start;   // [n_lanes + 1]  absolute offset of the lane's first symbol in the output
    uint8_t* am;
    uint8_t* qm;
    unsigned long long cap;          // entries the arrays hold
};

// one CTA per block: read offsets (scan of the lengths), lane partition (recomputed from the lengths: pieces, quanta),
// lane payload offsets (scan of the lane lengths).  Sequential tiles of 256 with a running carry.
__global__ void __launch_bounds__(256)
native_fill_kernel(const uint8_t* __restrict__ blocks, const NativeBlockHdr* __restrict__ hdr, uint32_t n_blocks,
                   const unsigned long long* __restrict__ blk_read_base, const unsigned long long* __restrict__ blk_sym_base,
                   const unsigned long long* __restrict__ blk_lane_base, unsigned long long* __restrict__ read_off_out,
                   NativeIndex ix, uint32_t* __restrict__ block_first, int32_t* __restrict__ status) {
    __shared__ unsigned long long smem[kScanBlock / 32];
    __shared__ unsigned long long total;
    __shared__ int lane_mismatch;
    __shared__ int32_t s_status;
    const uint32_t b = blockIdx.x;
    // other CTAs of this launch may set status[0] while this one runs: every thread must take the same exit (barriers follow)
    if (threadIdx.x == 0) s_status = status[0];
    __syncthreads();
    if (s_status != 0) return;
    if (blk_lane_base[n_blocks] + 1 > ix.cap) {  // more lanes than the index holds: refuse (uniform over the launch)
        if (b == 0 && threadIdx.x == 0) {
            int old = atomicCAS(&status[0], 0, 11);  // IDN_E_NOSPACE
            if (old == 0) status[1] = -1;
        }
        return;
    }
    if (b == n_blocks) {  // terminators
        if (threadIdx.x == 0) {
            block_first[n_blocks] = (uint32_t)blk_read_base[n_blocks];
            read_off_out[blk_read_base[n_blocks]] = blk_sym_base[n_blocks];
            ix.first_read[blk_lane_base[n_blocks]] = blk_read_base[n_blocks];
            ix.sym_start[blk_lane_base[n_blocks]] = blk_sym_base[n_blocks];
        }
        return;
    }
    const NativeBlockHdr h = hdr[b];
    const unsigned long long rbase = blk_read_base[b], sbase = blk_sym_base[b], lbase = blk_lane_base[b];
    const uint32_t Q = h.lane_syms;
    if (threadIdx.x == 0) {
        block_first[b] = (uint32_t)rbase;
        lane_mismatch = 0;
    }
    __syncthreads();
    const uint8_t* t_len = blocks + h.tab;
    const uint8_t* t_mdl = t_len + (size_t)h.n_reads * h.width;
    const uint8_t* t_ll = t_mdl + 2ull * h.n_lanes;
    const unsigned long long pay0 = h.tab + (unsigned long long)h.n_reads * h.width + 6ull * h.n_lanes;
    // reads: offsets + the lanes they open.  The first piece of a read opens a lane when its quantum differs from the
    // quantum of the piece before it (the LAST piece of the read before); every further piece opens one.
    unsigned long long carry = 0;         // symbols before this tile
    unsigned long long lane_carry = 0;    // lanes opened before this tile
    unsigned long long prev_q_carry = 0;  // quantum of the last piece of the last read of the previous tile
    bool any_cut = false;
    for (uint32_t base = 0; base < h.n_reads; base += kScanBlock) {
        uint32_t i = base + threadIdx.x;
        unsigned long long len = 0;
        if (i < h.n_reads)
            len = h.width == 0 ? h.const_len
                               : (h.width == 2 ? (((uint32_t)t_len[2 * i] << 8) | t_len[2 * i + 1]) : load_u32be(t_len + 4ull * i));
        unsigned long long ex = block_exclusive_scan(len, &total, smem);
        unsigned long long off = carry + ex;  // block-relative symbol offset of read i
        unsigned long long tile_syms = total;
        __syncthreads();
        const uint32_t pc = native_pieces((uint32_t)len, Q);
        any_cut = any_cut || pc > 1;
        const unsigned long long q_first = off / Q, q_last = (off + (unsigned long long)(pc - 1) * Q) / Q;
        // quantum of the piece before: the previous thread's last piece, or the carried one for the first thread of the tile
        unsigned long long pq = __shfl_up_sync(0xffffffffu, q_last, 1);
        __shared__ unsigned long long warp_last_q[kScanBlock / 32];
        if ((threadIdx.x & 31) == 31) warp_last_q[threadIdx.x >> 5] = q_last;
        __syncthreads();
        if ((threadIdx.x & 31) == 0) pq = threadIdx.x == 0 ? prev_q_carry : warp_last_q[(threadIdx.x >> 5) - 1];
        const bool opens = i < h.n_reads && ((i == 0) || (q_first != pq));
        unsigned long long cnt = 0;
        if (i < h.n_reads) cnt = (opens ? 1u : 0u) + pc - 1;
        unsigned long long lex = block_exclusive_scan(cnt, &total, smem);
        unsigned long long tile_lanes = total;
        if (i < h.n_reads) {
            read_off_out[rbase + i] = sbase + off;
            unsigned long long l = lane_carry + lex;
            if (opens) {
                if (l < h.n_lanes) {
                    ix.first_read[lbase + l] = rbase + i;
                    ix.sym_start[lbase + l] = sbase + off;
                } else {
                    lane_mismatch = 1;
                }
                l++;
            }
            for (uint32_t j = 1; j < pc; j++, l++) {
                if (l < h.n_lanes) {
                    ix.first_read[lbase + l] = rbase + i;
                    ix.sym_start[lbase + l] = sbase + off + (unsigned long long)j * Q;
                } else {
                    lane_mismatch = 1;
                }
            }
        }
        // carry the quantum of the last piece of the last read of this tile
        __shared__ unsigned long long last_q;
        if (threadIdx.x == kScanBlock - 1) last_q = q_last;
        __syncthreads();
        prev_q_carry = last_q;
        carry += tile_syms;
        lane_carry += tile_lanes;
        __syncthreads();
    }
    if (threadIdx.x == 0 && lane_carry != h.n_lanes) lane_mismatch = 1;
    if (__syncthreads_or(any_cut) != (int)(h.split != 0) && threadIdx.x == 0) lane_mismatch = 1;  // the flag must tell the truth
    // lanes: payload offsets + models
    unsigned long long pcarry = 0;
    for (uint32_t base = 0; base < h.n_lanes; base += kScanBlock) {
        uint32_t i = base + threadIdx.x;
        unsigned long long ll = i < h.n_lanes ? load_u32be(t_ll + 4ull * i) : 0;
        unsigned long long ex = block_exclusive_scan(ll, &total, smem);
        if (i < h.n_lanes) {
            ix.pay_off[lbase + i] = pay0 + pcarry + ex;
            ix.pay_len[lbase + i] = (uint32_t)ll;
            ix.am[lbase + i] = t_mdl[2 * i];
            ix.qm[lbase + i] = t_mdl[2 * i + 1];
        }
        pcarry += total;
        __syncthreads();
    }
    __syncthreads();
    if (threadIdx.x == 0 && lane_mismatch) {
        int old = atomicCAS(&status[0], 0, 3);  // the lane table does not match the partition of the lengths
        if (old == 0) status[1] = (int32_t)b;
    }
}

struct DecodeLaneArgs {
    const ModelDev* models;
    const int32_t* model_ids;  // container index -> models[]
    const uint8_t* payload;
    NativeIndex ix;
    const unsigned long long* n_lanes_dev;
    const unsigned long long* read_off;  // [n_reads+1] absolute symbol offsets (native_fill_kernel)
    const int32_t* status;
    const uint32_t* split_flag;  // some block of the call cuts reads into pieces: the per-read CRC partials come from a pass
                                 // over the output instead (crc_read kernels), a read's symbols being decoded by several threads
    uint8_t* acids_out;
    uint8_t* quals_out;
    long long out_dq;  // quals_out - acids_out
    uint32_t* err;
    // optional: per-read CRC-32 partials (acids | quals) for crc_verify_kernel, as in DecodeArgs
    uint32_t* part_crc;
    unsigned long long* part_len;
    const uint32_t* crc_tab;
    const uint32_t* xpow;
};

template <bool kUniform, class P>
__device__ __forceinline__ void decode_lane_one(const DecodeLaneArgs& A, const ModelDev& MA, const ModelDev& MQ, unsigned long long l64, DecCrc& C,
                                                const uint32_t* s_xpow) {
    // (register budget: the per-position loop inside decode_read_body is what counts, so the lane bounds and the
    // payload address are re-read from the index per read instead of being kept in registers across it)
    const uint32_t l = (uint32_t)l64;
    const ModelDev& ma = kUniform ? MA : A.models[A.model_ids[A.ix.am[l]]];
    const ModelDev& mq = kUniform ? MQ : A.models[A.model_ids[A.ix.qm[l]]];
    uint32_t r = (uint32_t)A.ix.first_read[l];
    // (first_read <= n_reads and read_off holds n_reads + 1 entries)
    const bool mid = A.ix.sym_start[l + 1] > A.ix.sym_start[l] && A.ix.sym_start[l] > A.read_off[r];  // the lane starts inside read r
    const bool bad = mid && A.ix.pay_len[l] < kNativeHistBytes + 8;
    const uint32_t lead = (mid && !bad) ? kNativeHistBytes : 0u;  // history bytes in front of the stream
    DecStream D;
    D.begin(A.payload + A.ix.pay_off[l], lead, bad ? 0u : A.ix.pay_len[l] - lead);
    SymWriter O;
    O.init(A.acids_out + A.ix.sym_start[l], A.out_dq);
    // the reads with a symbol in [a, b): the loop ends by itself at the last read (read_off[n_reads] >= b)
#pragma unroll 1
    for (;; r++) {
        const unsigned long long a = A.ix.sym_start[l], b = A.ix.sym_start[l + 1];
        const unsigned long long o = A.read_off[r];
        if (o >= b) break;
        const unsigned long long o_next = A.read_off[r + 1];
        if (o_next > a) {
            const uint32_t len = (uint32_t)(o_next - o);
            const uint32_t p0 = (uint32_t)((a > o ? a : o) - o), p1 = (uint32_t)((b < o_next ? b : o_next) - o);
            decode_read_body<P>(ma, mq, len, p0, p1, A.payload + A.ix.pay_off[l], D, O, C);
            if (C.tab) {  // whole reads only (no block of the call cuts reads)
                const CrcPair p = crc_concat(CrcPair{~C.ca, len}, CrcPair{~C.cq, len}, s_xpow);
                A.part_crc[r] = len ? p.crc : 0u;
                A.part_len[r] = 2ull * len;
                C.ca = C.cq = 0xffffffffu;
            }
        }
    }
    O.flush();
    const uint32_t plen = A.ix.pay_len[l] - lead;
    D.finish(A.payload + A.ix.pay_off[l], lead, plen);
    if (bad || (D.st & 1) || !D.clean_end(plen)) atomicOr(A.err, 1u);
}

template <bool kUniform, class P>
__global__ void __launch_bounds__(128, kUniform ? IDN_LANE_MINB : 1)
decode_lane_kernel(DecodeLaneArgs A, const ModelDev MA, const ModelDev MQ) {
    __shared__ uint32_t s_tab[256];
    __shared__ uint32_t s_xpow[64];
    if (A.status[0] != 0) return;
    DecCrc C{nullptr, 0xffffffffu, 0xffffffffu};
    if (A.part_crc && *A.split_flag == 0) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s_tab[i] = A.crc_tab[i];
        for (int i = threadIdx.x; i < 64; i += blockDim.x) s_xpow[i] = A.xpow[i];
        __syncthreads();
        C.tab = s_tab;
    }
    const unsigned long long n_lanes = *A.n_lanes_dev;
    // (grid-stride: a call whose blocks cut long reads into pieces may hold more lanes than the launch has threads)
#pragma unroll 1
    for (unsigned long long l64 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; l64 < n_lanes; l64 += (unsigned long long)gridDim.x * blockDim.x)
        decode_lane_one<kUniform, P>(A, MA, MQ, l64, C, s_xpow);
}

// the lanes of one model pair, see decode_list_kernel
template <class P>
__global__ void __launch_bounds__(128, IDN_LANE_MINB)
decode_lane_list_kernel(DecodeLaneArgs A, const ModelDev MA, const ModelDev MQ, ReadList L) {
    __shared__ uint32_t s_tab[256];
    __shared__ uint32_t s_xpow[64];
    if (A.status[0] != 0) return;
    DecCrc C{nullptr, 0xffffffffu, 0xffffffffu};
    if (A.part_crc && *A.split_flag == 0) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s_tab[i] = A.crc_tab[i];
        for (int i = threadIdx.x; i < 64; i += blockDim.x) s_xpow[i] = A.xpow[i];
        __syncthreads();
        C.tab = s_tab;
    }
    const uint32_t n = *L.count;
    const uint32_t* __restrict__ list = L.list + *L.base;
#pragma unroll 1
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        decode_lane_one<true, P>(A, MA, MQ, list[i], C, s_xpow);
}

struct DecodeLanePairKey {  // decompress side: the model pair of lane l from the lane table (container model indices)
    const uint8_t* am;
    const uint8_t* qm;
    const unsigned long long* n_lanes_dev;
    const int32_t* status;
    uint32_t n_models;
    __device__ __forceinline__ uint32_t operator()(uint64_t l) const {
        if (status[0] != 0 || l >= *n_lanes_dev) return 0xffffffffu;
        return (uint32_t)am[l] * n_models + qm[l];
    }
};

}  // namespace idn
