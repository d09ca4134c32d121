// Device-side gzip writer: byte ranges ("cells") of a device buffer -> one RFC 1952 member per non-empty cell,
// members laid out cell after cell (SURVEY 8 f-1, the deflate half; the inflate half is gz_kernels.cuh).
//
// A cell is cut into pieces of kPiece bytes, and every piece is one independent job of one CTA:
//
//   deflate_plan_kernel    pieces per cell -> first piece of every cell (exclusive scan); no pieces at all when the
//                          producer of the cells raised an error
//   deflate_piece_kernel   LZ77 + dynamic Huffman of one piece into its own scratch slot, or a stored block when that
//                          is not smaller; the piece ends byte-aligned (an empty stored block, as Z_SYNC_FLUSH writes
//                          it), so pieces concatenate byte-wise.  Also the CRC-32 of the piece.
//   deflate_layout_kernel  exclusive scan of the piece sizes (header in front of a cell's first piece, trailer
//                          behind its last) and the CRC-32 prefix over all pieces
//   deflate_cells_kernel   member offsets of the cells, gzip header and "03 00" + CRC-32 + ISIZE of every member
//   deflate_gather_kernel  the piece bytes into place
//
// BGZF (the blocked gzip of htslib and bgzip) is a layout of the same pieces.  deflate_split_kernel cuts every cell
// into blocks of at most kBgzfBlock bytes (three pieces), the five kernels above run over the blocks as if they were
// cells -- so no back-reference crosses a block start and every block is a member of its own -- with htslib's
// 18-byte header (the BC extra field holds the block's size), and deflate_cell_offsets_kernel gives every cell the
// offset of its first block.  A cell is then a run of whole BGZF blocks; the 28-byte EOF block is the caller's.
//
// LZ77 of a piece: back-references reach into the kHist bytes of the same cell in front of the piece (never into
// another cell), at most 32 KiB back, lengths 3..258.  Candidates come from a hash table of 4-byte prefixes in
// shared memory that is filled in rounds of 256 positions: a position sees the latest earlier position of its hash
// from the rounds before its own, chosen with atomicMax, so the parse does not depend on thread timing and the
// same input always gives the same bytes.  The greedy parse is then split over the 32 lanes of warp 0, one
// kSeg-byte segment each; a match that would run past its segment's end is cut there (or becomes literals when
// fewer than 3 bytes are left).  Warps 1..7 sum the piece's CRC-32 meanwhile.
//
// Huffman: literal/length and distance histograms in shared memory; code lengths from the sorted weights with the
// in-place minimum-redundancy algorithm of Moffat and Katajainen (one lane), limited to 15 bits (7 for the
// code-length code) by moving the deepest codes up until the Kraft sum is 1.  Every lane counts the bits of its
// tokens; a warp scan places them; every lane writes its own bit range of the scratch slot (words it shares with a
// neighbour with atomicOr).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "crc32.cuh"

namespace frb {
namespace dfl {

constexpr unsigned kPiece = 16384;           // input bytes per piece
constexpr unsigned kHist = 16384;            // bytes of the cell in front of a piece that matches may reach
constexpr unsigned kPieceCap = kPiece + 64;  // scratch bytes per piece (a stored piece takes kPiece + 5)
constexpr int kHashBits = 13;
constexpr int kThreads = 256;
constexpr int kLanes = 32;                   // parse segments per piece (warp 0)
constexpr unsigned kSeg = kPiece / kLanes;
constexpr int kMaxMatch = 258;
constexpr unsigned kWindow = 32768;
constexpr int kHeaderBytes = 10, kTrailerBytes = 10;  // gzip header; final empty block (2) + CRC-32 + ISIZE
constexpr unsigned kBgzfBlock = 3 * kPiece;  // BGZF: input bytes per block (at most 49,195 bytes written)
constexpr int kBgzfHeaderBytes = 18;         // gzip header with the 6-byte BC extra field
constexpr int kBgzfEofBytes = 28;            // the empty block that ends a BGZF file

struct PieceInfo {
    unsigned out;    // bytes of the piece in its scratch slot
    unsigned in;     // input bytes
    unsigned crc;    // CRC-32 of the input bytes
    unsigned flags;  // bit 0: first piece of its cell, bit 1: last piece
};

// order in which a dynamic header gives the code lengths of the code-length code (RFC 1951 3.2.7)
__device__ __constant__ unsigned char c_dfl_cl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct Smem {
    unsigned tab[1 << kHashBits];            // latest position + 1 of every 4-byte hash (0: none)
    unsigned char in[kHist + kPiece + 8];    // history, then the piece
    unsigned short tok[kPiece];              // candidate + 1 per position; after the parse: 0 literal, else distance
                                             // (and the length in the slot behind it)
    unsigned lfreq[288], dfreq[32], clfreq[19];
    unsigned char llen[288], dlen[32], cllen[19];
    unsigned short lcode[288], dcode[32], clcode[19];
    unsigned short cltok[288 + 32];          // run-length coded code lengths: symbol | extra << 5
    unsigned keys[288], sorted[288], A[288], cnt[32];      // code builder of warp 0
    unsigned dkeys[32], dsorted[32], dA[32], dcnt[32];     // code builder of warp 1
    unsigned long long lane_bits[kLanes];    // bits of the tokens in front of every lane's segment
    unsigned long long tok_bits;             // bits of all tokens
    unsigned wcrc[8];
    unsigned wlen[8];
    unsigned n_cltok, hlit, hdist, hclen, header_bits;
};

// ---- symbols ----------------------------------------------------------------------------------------------------
// length 3..258 -> index 0..28 of the length codes (symbol 257 + index), extra bits and their value
__device__ __forceinline__ void len_code(unsigned len, unsigned& idx, unsigned& nextra, unsigned& extra) {
    const unsigned x = len - 3;
    if (x < 8) {
        idx = x, nextra = 0, extra = 0;
    } else if (x == 255) {
        idx = 28, nextra = 0, extra = 0;
    } else {
        const unsigned e = 31 - __clz(x) - 2;
        idx = 4 * e + 4 + ((x >> e) & 3), nextra = e, extra = x & ((1u << e) - 1);
    }
}
// distance 1..32768 -> code 0..29, extra bits and their value
__device__ __forceinline__ void dist_code(unsigned dist, unsigned& idx, unsigned& nextra, unsigned& extra) {
    const unsigned x = dist - 1;
    if (x < 4) {
        idx = x, nextra = 0, extra = 0;
    } else {
        const unsigned e = 31 - __clz(x) - 1;
        idx = 2 * e + 2 + ((x >> e) & 1), nextra = e, extra = x & ((1u << e) - 1);
    }
}

// ---- bit output ---------------------------------------------------------------------------------------------------
// Bits [b0, b1) of a zeroed, word-aligned buffer, LSB first.  The first and the last word may be shared with the
// writer of the neighbouring range: those two take atomicOr, the words between plain stores.
struct BitSink {
    unsigned* w;
    unsigned long long first, last, word;
    unsigned long long acc;
    int n;
    __device__ BitSink(unsigned* out, unsigned long long b0, unsigned long long b1)
        : w(out), first(b0 >> 5), last(b1 > b0 ? (b1 - 1) >> 5 : b0 >> 5), word(b0 >> 5), acc(0), n(static_cast<int>(b0 & 31)) {}
    __device__ __forceinline__ void store(unsigned v) {
        if (word == first || word == last) atomicOr(w + word, v);
        else w[word] = v;
        ++word;
    }
    __device__ __forceinline__ void put(unsigned v, int len) {  // len <= 32, v < 2^len
        acc |= static_cast<unsigned long long>(v) << n;
        n += len;
        if (n >= 32) {
            store(static_cast<unsigned>(acc));
            acc >>= 32;
            n -= 32;
        }
    }
    __device__ __forceinline__ void flush() {
        if (n > 0) store(static_cast<unsigned>(acc));
    }
};

__device__ __forceinline__ unsigned rev(unsigned code, unsigned len) { return __brev(code) >> (32 - len); }

// ---- Huffman codes --------------------------------------------------------------------------------------------------
// Minimum-redundancy code lengths in place (Moffat & Katajainen, 1995): A[0, n) holds weights in ascending order and
// is overwritten with the code length of each.  n >= 2.
__device__ inline void min_redundancy(unsigned* A, int n) {
    A[0] += A[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < n - 1; ++next) {
        if (leaf >= n || A[root] < A[leaf]) {
            A[next] = A[root];
            A[root++] = next;
        } else {
            A[next] = A[leaf++];
        }
        if (leaf >= n || (root < next && A[root] < A[leaf])) {
            A[next] += A[root];
            A[root++] = next;
        } else {
            A[next] += A[leaf++];
        }
    }
    A[n - 2] = 0;
    for (int next = n - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
    int avbl = 1, used = 0, dpth = 0, next = n - 1;
    root = n - 2;
    while (avbl > 0) {
        while (root >= 0 && static_cast<int>(A[root]) == dpth) ++used, --root;
        while (avbl > used) A[next--] = dpth, --avbl;
        avbl = 2 * used, ++dpth, used = 0;
    }
}

// One warp: code lengths of at most maxlen bits for freq[0, n) into len[], canonical codes (bit-reversed, ready for
// LSB-first output) into code[].  At least two symbols get a code, so that every code is complete.
__device__ inline void build_code(unsigned* freq, int n, int maxlen, unsigned char* len, unsigned short* code,
                                  unsigned* keys, unsigned* sorted, unsigned* A, unsigned* cnt) {
    const int lane = threadIdx.x & 31;
    if (lane == 0) {
        int used = 0;
        for (int s = 0; s < n; ++s) used += freq[s] != 0;
        if (used < 2) freq[0] = max(freq[0], 1u), freq[1] = max(freq[1], 1u);
    }
    __syncwarp();
    int m = 0;  // used symbols, compacted in symbol order as (weight << 9) | symbol
    for (int base = 0; base < n; base += 32) {
        const int s = base + lane;
        const unsigned f = s < n ? freq[s] : 0u;
        const unsigned ballot = __ballot_sync(0xFFFFFFFFu, f != 0);
        if (f) keys[m + __popc(ballot & ((1u << lane) - 1))] = (f << 9) | static_cast<unsigned>(s);
        if (s < n) len[s] = 0;
        m += __popc(ballot);
    }
    __syncwarp();
    for (int i = lane; i < m; i += 32) {  // rank sort, ascending (keys are distinct)
        const unsigned k = keys[i];
        int r = 0;
        for (int j = 0; j < m; ++j) r += keys[j] < k;
        sorted[r] = k;
    }
    __syncwarp();
    if (lane == 0) {
        for (int i = 0; i < m; ++i) A[i] = sorted[i] >> 9;
        min_redundancy(A, m);
        for (int l = 0; l < 32; ++l) cnt[l] = 0;
        for (int i = 0; i < m; ++i) cnt[min(A[i], 31u)]++;
        for (int l = maxlen + 1; l < 32; ++l) cnt[maxlen] += cnt[l], cnt[l] = 0;
        unsigned total = 0;
        for (int l = 1; l <= maxlen; ++l) total += cnt[l] << (maxlen - l);
        while (total != (1u << maxlen)) {  // over-full after the clamp: move codes down until the Kraft sum is 1
            cnt[maxlen]--;
            for (int l = maxlen - 1; l > 0; --l)
                if (cnt[l]) {
                    cnt[l]--;
                    cnt[l + 1] += 2;
                    break;
                }
            total--;
        }
        int j = 0;  // the rarest symbols get the longest codes
        for (int l = maxlen; l >= 1; --l)
            for (unsigned k = 0; k < cnt[l]; ++k) len[sorted[j++] & 511] = static_cast<unsigned char>(l);
        unsigned next[16];  // canonical codes (RFC 1951 3.2.2); cnt[0] = 0
        unsigned c = 0;
        for (int l = 1; l <= maxlen; ++l) {
            c = (c + cnt[l - 1]) << 1;
            next[l] = c;
        }
        for (int s = 0; s < n; ++s)
            if (len[s]) code[s] = static_cast<unsigned short>(rev(next[len[s]]++, len[s]));
    }
    __syncwarp();
}

// ---- kernels ------------------------------------------------------------------------------------------------------
// BGZF: block_off[0, n_blocks] = the cells cut into blocks of at most kBgzfBlock bytes, cell after cell; entries
// behind the last block repeat the end offset (empty blocks: no output).  first_block[c] = blocks in front of cell c
// (n_cells + 1 entries; the last is the block count).  A cell list that is not ordered, or reaches beyond max_bytes,
// or a raised *skip, gives no blocks at all (every offset 0).  One block.
__global__ void __launch_bounds__(1024) deflate_split_kernel(const unsigned long long* __restrict__ cell_off, unsigned n_cells,
                                                             unsigned long long max_bytes, const int* __restrict__ skip,
                                                             unsigned long long* __restrict__ block_off, unsigned n_blocks,
                                                             unsigned* __restrict__ first_block) {
    __shared__ unsigned s_sum[1024];
    __shared__ unsigned s_bad;
    const unsigned t = threadIdx.x;
    if (t == 0) s_bad = (skip && *skip) || cell_off[n_cells] - cell_off[0] > max_bytes || cell_off[n_cells] < cell_off[0];
    __syncthreads();
    const unsigned per = (n_cells + 1023) / 1024, c0 = min(n_cells, t * per), c1 = min(n_cells, c0 + per);
    unsigned local = 0;
    for (unsigned c = c0; c < c1; ++c) {
        if (cell_off[c + 1] < cell_off[c]) s_bad = 1;
        local += static_cast<unsigned>((cell_off[c + 1] - cell_off[c] + kBgzfBlock - 1) / kBgzfBlock);
    }
    s_sum[t] = local;
    __syncthreads();
    for (unsigned d = 1; d < 1024; d <<= 1) {
        const unsigned v = t >= d ? s_sum[t - d] : 0u;
        __syncthreads();
        s_sum[t] += v;
        __syncthreads();
    }
    const bool bad = s_bad != 0 || s_sum[1023] > n_blocks;
    unsigned run = bad ? 0u : s_sum[t] - local;
    for (unsigned c = c0; c < c1; ++c) {
        first_block[c] = run;
        if (bad) continue;
        const unsigned long long a = cell_off[c], len = cell_off[c + 1] - a;
        for (unsigned long long j = 0; j * kBgzfBlock < len; ++j) block_off[run++] = a + j * kBgzfBlock;
    }
    const unsigned total = bad ? 0u : s_sum[1023];
    const unsigned long long end = bad ? 0ull : cell_off[n_cells];
    if (t == 1023) first_block[n_cells] = total;
    for (unsigned b = total + t; b <= n_blocks; b += 1024) block_off[b] = end;
}

// first_piece[c] = pieces in front of cell c (n_cells + 1 entries; the last is the piece count).  A cell list that is
// not ordered, or reaches beyond max_bytes, or a raised *skip, gives no pieces: the caller reports its own error.
__global__ void __launch_bounds__(1024) deflate_plan_kernel(const unsigned long long* __restrict__ cell_off, unsigned n_cells,
                                                            unsigned long long max_bytes, const int* __restrict__ skip,
                                                            unsigned* __restrict__ first_piece) {
    __shared__ unsigned s_sum[1024];
    __shared__ unsigned s_bad;
    const unsigned t = threadIdx.x;
    if (t == 0) s_bad = (skip && *skip) || cell_off[n_cells] - cell_off[0] > max_bytes || cell_off[n_cells] < cell_off[0];
    __syncthreads();
    const unsigned per = (n_cells + 1023) / 1024, c0 = min(n_cells, t * per), c1 = min(n_cells, c0 + per);
    unsigned local = 0;
    for (unsigned c = c0; c < c1; ++c) {
        if (cell_off[c + 1] < cell_off[c]) s_bad = 1;
        local += static_cast<unsigned>((cell_off[c + 1] - cell_off[c] + kPiece - 1) / kPiece);
    }
    s_sum[t] = local;
    __syncthreads();
    for (unsigned d = 1; d < 1024; d <<= 1) {
        const unsigned v = t >= d ? s_sum[t - d] : 0u;
        __syncthreads();
        s_sum[t] += v;
        __syncthreads();
    }
    const bool bad = s_bad != 0;
    unsigned run = bad ? 0u : s_sum[t] - local;
    for (unsigned c = c0; c < c1; ++c) {
        first_piece[c] = run;
        if (!bad) run += static_cast<unsigned>((cell_off[c + 1] - cell_off[c] + kPiece - 1) / kPiece);
    }
    if (t == 1023) first_piece[n_cells] = bad ? 0u : s_sum[1023];
}

// One CTA per piece (grid-stride).  Scratch slot p: kPieceCap bytes at scratch + p * kPieceCap.
__global__ void __launch_bounds__(kThreads, 2) deflate_piece_kernel(const unsigned char* __restrict__ src,
                                                                    const unsigned long long* __restrict__ cell_off,
                                                                    unsigned n_cells, const unsigned* __restrict__ first_piece,
                                                                    unsigned char* __restrict__ scratch,
                                                                    PieceInfo* __restrict__ info, gz::CrcPowers pw) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    Smem& S = *reinterpret_cast<Smem*>(s_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned n_pieces = first_piece[n_cells];
    for (unsigned p = blockIdx.x; p < n_pieces; p += gridDim.x) {
        // ---- the piece: its cell (the last cell whose first piece is <= p), history, bytes ----
        unsigned lo = 0, hi = n_cells;  // first_piece[lo] <= p < first_piece[hi]
        while (hi - lo > 1) {
            const unsigned mid = (lo + hi) >> 1;
            if (first_piece[mid] <= p) lo = mid;
            else hi = mid;
        }
        const unsigned cell = lo, k = p - first_piece[cell];
        const unsigned long long cell_len = cell_off[cell + 1] - cell_off[cell];
        const unsigned long long start = cell_off[cell] + static_cast<unsigned long long>(k) * kPiece;
        const unsigned len = static_cast<unsigned>(min(static_cast<unsigned long long>(kPiece), cell_len - static_cast<unsigned long long>(k) * kPiece));
        const unsigned hist = k ? kHist : 0u;
        const unsigned total = hist + len;
        const unsigned char* const from = src + start - hist;
        for (unsigned i = tid; i < total; i += kThreads) S.in[i] = from[i];
        for (unsigned i = tid; i < (1u << kHashBits); i += kThreads) S.tab[i] = 0;
        for (unsigned i = tid; i < 288; i += kThreads) S.lfreq[i] = 0;
        if (tid < 32) S.dfreq[tid] = 0;
        if (tid < 19) S.clfreq[tid] = 0;
        unsigned* const out = reinterpret_cast<unsigned*>(scratch + static_cast<unsigned long long>(p) * kPieceCap);
        for (unsigned i = tid; i < kPieceCap / 4; i += kThreads) out[i] = 0;
        __syncthreads();
        auto hash4 = [&](unsigned q) {
            const unsigned v = S.in[q] | (S.in[q + 1] << 8) | (S.in[q + 2] << 16) | (static_cast<unsigned>(S.in[q + 3]) << 24);
            return (v * 0x9E3779B1u) >> (32 - kHashBits);
        };
        // ---- history: every position at once (the table keeps the latest) ----
        for (unsigned q = tid; q < hist; q += kThreads)
            if (q + 3 < total) atomicMax(&S.tab[hash4(q)], q + 1);
        __syncthreads();
        // ---- the piece in rounds: candidates from the rounds before, then this round's positions go in ----
        for (unsigned r = 0; r < len; r += kThreads) {
            const unsigned i = r + tid, q = hist + i;
            unsigned h = 0;
            const bool hashed = i < len && q + 3 < total;
            if (hashed) {
                h = hash4(q);
                const unsigned c = S.tab[h];
                S.tok[i] = static_cast<unsigned short>(c && q - (c - 1) <= kWindow ? c : 0u);
            } else if (i < len) {
                S.tok[i] = 0;
            }
            __syncthreads();
            if (hashed) atomicMax(&S.tab[h], q + 1);
            __syncthreads();
        }
        // ---- greedy parse (warp 0, one segment per lane); CRC-32 of the piece (warps 1..7) ----
        if (warp == 0) {
            const unsigned s0 = min(len, lane * kSeg), s1 = min(len, s0 + kSeg);
            unsigned i = s0;
            while (i < s1) {
                const unsigned c = S.tok[i];
                unsigned m = 0;
                if (c) {
                    const unsigned char* a = S.in + (c - 1);
                    const unsigned char* b = S.in + hist + i;
                    const unsigned lim = min(static_cast<unsigned>(kMaxMatch), s1 - i);
                    while (m < lim && a[m] == b[m]) ++m;
                }
                if (m >= 3) {
                    const unsigned dist = hist + i - (c - 1);
                    unsigned li, ln, lx, di, dn, dx;
                    len_code(m, li, ln, lx);
                    dist_code(dist, di, dn, dx);
                    atomicAdd(&S.lfreq[257 + li], 1u);
                    atomicAdd(&S.dfreq[di], 1u);
                    S.tok[i] = static_cast<unsigned short>(dist);
                    S.tok[i + 1] = static_cast<unsigned short>(m);
                    i += m;
                } else {
                    atomicAdd(&S.lfreq[S.in[hist + i]], 1u);
                    S.tok[i] = 0;
                    ++i;
                }
            }
        } else {
            const unsigned u = tid - 32, chunk = (len + kThreads - 33) / (kThreads - 32);
            const unsigned a = min(len, u * chunk), n = min(len, a + chunk) - a;
            unsigned crc = n ? gz::crc_bytes(S.in + hist + a, n) : 0u;
            unsigned l = n;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {  // (crc, len) of lane L joins in front of lane L + d's
                const unsigned ocrc = __shfl_down_sync(0xFFFFFFFFu, crc, d);
                const unsigned olen = __shfl_down_sync(0xFFFFFFFFu, l, d);
                if ((lane & (2 * d - 1)) == 0) {
                    crc = gz::crc_join(pw, crc, ocrc, olen);
                    l += olen;
                }
            }
            if (lane == 0) S.wcrc[warp] = crc, S.wlen[warp] = l;
        }
        if (tid == 0) S.lfreq[256] = 1;  // end of block
        __syncthreads();
        // ---- codes: literal/length (warp 0) and distance (warp 1) at the same time, then the code-length code ----
        if (warp == 0) build_code(S.lfreq, 286, 15, S.llen, S.lcode, S.keys, S.sorted, S.A, S.cnt);
        else if (warp == 1) build_code(S.dfreq, 30, 15, S.dlen, S.dcode, S.dkeys, S.dsorted, S.dA, S.dcnt);
        __syncthreads();
        if (tid == 0) {  // code lengths, run-length coded (RFC 1951 3.2.7)
            unsigned nl = 286, nd = 30;
            while (nl > 257 && !S.llen[nl - 1]) --nl;
            while (nd > 1 && !S.dlen[nd - 1]) --nd;
            const unsigned all = nl + nd;
            auto L = [&](unsigned j) -> unsigned { return j < nl ? S.llen[j] : S.dlen[j - nl]; };
            unsigned nt = 0;
            auto emit = [&](unsigned sym, unsigned extra) {
                S.cltok[nt++] = static_cast<unsigned short>(sym | (extra << 5));
                S.clfreq[sym]++;
            };
            for (unsigned j = 0; j < all;) {
                const unsigned v = L(j);
                unsigned run = 1;
                while (j + run < all && L(j + run) == v) ++run;
                j += run;
                if (v == 0) {
                    while (run >= 11) {
                        const unsigned r = min(run, 138u);
                        emit(18, r - 11);
                        run -= r;
                    }
                    if (run >= 3) emit(17, run - 3), run = 0;
                    while (run--) emit(0, 0);
                } else {
                    emit(v, 0);
                    --run;
                    while (run >= 3) {
                        const unsigned r = min(run, 6u);
                        emit(16, r - 3);
                        run -= r;
                    }
                    while (run--) emit(v, 0);
                }
            }
            S.n_cltok = nt, S.hlit = nl, S.hdist = nd;
        }
        __syncthreads();
        if (warp == 0) build_code(S.clfreq, 19, 7, S.cllen, S.clcode, S.keys, S.sorted, S.A, S.cnt);
        __syncthreads();
        // ---- bits of every lane's tokens, placed by a warp scan ----
        if (warp == 0) {
            if (lane == 0) {
                unsigned hc = 19;
                while (hc > 4 && !S.cllen[c_dfl_cl_order[hc - 1]]) --hc;
                unsigned bits = 3 + 14 + 3 * hc;
                for (unsigned j = 0; j < S.n_cltok; ++j) {
                    const unsigned sym = S.cltok[j] & 31;
                    bits += S.cllen[sym] + (sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
                }
                S.hclen = hc, S.header_bits = bits;
            }
            const unsigned s0 = min(len, lane * kSeg), s1 = min(len, s0 + kSeg);
            unsigned long long bits = 0;
            for (unsigned i = s0; i < s1;) {
                const unsigned d = S.tok[i];
                if (!d) {
                    bits += S.llen[S.in[hist + i]];
                    ++i;
                } else {
                    const unsigned m = S.tok[i + 1];
                    unsigned li, ln, lx, di, dn, dx;
                    len_code(m, li, ln, lx);
                    dist_code(d, di, dn, dx);
                    bits += S.llen[257 + li] + ln + S.dlen[di] + dn;
                    i += m;
                }
            }
            unsigned long long incl = bits;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned long long o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
                if (lane >= d) incl += o;
            }
            S.lane_bits[lane] = incl - bits;
            if (lane == 31) S.tok_bits = incl;
        }
        __syncthreads();
        const unsigned long long hb = S.header_bits;
        const unsigned long long eob = hb + S.tok_bits;               // where the end-of-block code goes
        const unsigned long long after = eob + S.llen[256] + 3;      // behind the empty stored block's 3 header bits
        const unsigned dyn_bytes = static_cast<unsigned>((after + 7) / 8 + 4);
        const bool dynamic = dyn_bytes < len + 5;
        if (dynamic) {
            if (warp == 0) {
                if (lane == 0) {  // block header: BFINAL 0, BTYPE 10, HLIT, HDIST, HCLEN, code-length code, lengths
                    BitSink w(out, 0, hb);
                    w.put(4, 3);
                    w.put(S.hlit - 257, 5);
                    w.put(S.hdist - 1, 5);
                    w.put(S.hclen - 4, 4);
                    for (unsigned j = 0; j < S.hclen; ++j) w.put(S.cllen[c_dfl_cl_order[j]], 3);
                    for (unsigned j = 0; j < S.n_cltok; ++j) {
                        const unsigned sym = S.cltok[j] & 31, extra = S.cltok[j] >> 5;
                        w.put(S.clcode[sym], S.cllen[sym]);
                        if (sym >= 16) w.put(extra, sym == 16 ? 2 : sym == 17 ? 3 : 7);
                    }
                    w.flush();
                }
                const unsigned s0 = min(len, lane * kSeg), s1 = min(len, s0 + kSeg);
                const unsigned long long b0 = hb + S.lane_bits[lane];
                const unsigned long long b1 = lane < 31 ? hb + S.lane_bits[lane + 1] : eob;
                if (s1 > s0) {
                    BitSink w(out, b0, b1);
                    for (unsigned i = s0; i < s1;) {
                        const unsigned d = S.tok[i];
                        if (!d) {
                            const unsigned b = S.in[hist + i];
                            w.put(S.lcode[b], S.llen[b]);
                            ++i;
                        } else {
                            const unsigned m = S.tok[i + 1];
                            unsigned li, ln, lx, di, dn, dx;
                            len_code(m, li, ln, lx);
                            dist_code(d, di, dn, dx);
                            w.put(S.lcode[257 + li], S.llen[257 + li]);
                            if (ln) w.put(lx, ln);
                            w.put(S.dcode[di], S.dlen[di]);
                            if (dn) w.put(dx, dn);
                            i += m;
                        }
                    }
                    w.flush();
                }
                if (lane == 0) {  // end of block, then an empty stored block: 3 bits, pad to the byte, 00 00 FF FF
                    const unsigned pad = static_cast<unsigned>((8 - (after & 7)) & 7);
                    BitSink w(out, eob, after + pad + 32);
                    w.put(S.lcode[256], S.llen[256]);
                    w.put(0, 3);
                    if (pad) w.put(0, pad);
                    w.put(0xFFFF0000u, 32);
                    w.flush();
                }
            }
        } else {  // stored block: 00, LEN, NLEN, the bytes (already byte-aligned: no empty block behind it)
            unsigned char* const ob = reinterpret_cast<unsigned char*>(out);
            if (tid == 0) {
                ob[0] = 0;
                ob[1] = static_cast<unsigned char>(len), ob[2] = static_cast<unsigned char>(len >> 8);
                ob[3] = static_cast<unsigned char>(~len), ob[4] = static_cast<unsigned char>(~len >> 8);
            }
            for (unsigned i = tid; i < len; i += kThreads) ob[5 + i] = S.in[hist + i];
        }
        if (tid == 0) {
            unsigned crc = S.wcrc[1];
            for (int w = 2; w < kThreads / 32; ++w) crc = gz::crc_join(pw, crc, S.wcrc[w], S.wlen[w]);
            const bool last = static_cast<unsigned long long>(k + 1) * kPiece >= cell_len;
            info[p] = PieceInfo{dynamic ? dyn_bytes : len + 5, len, crc, (k == 0 ? 1u : 0u) | (last ? 2u : 0u)};
        }
        __syncthreads();  // shared memory is refilled for the next piece
    }
}

// start[p] = output bytes in front of piece p's part (header of `hdr` bytes / trailer included), start[n] = all;
// crc_pre[p] = CRC-32 of the input of pieces [0, p).  One block.
__global__ void __launch_bounds__(1024) deflate_layout_kernel(const PieceInfo* __restrict__ info,
                                                              const unsigned* __restrict__ first_piece, unsigned n_cells,
                                                              unsigned long long* __restrict__ start,
                                                              unsigned* __restrict__ crc_pre, gz::CrcPowers pw, int hdr) {
    __shared__ unsigned long long s_sum[1024], s_len[1024];
    __shared__ unsigned s_crc[1024];
    const unsigned t = threadIdx.x, n = first_piece[n_cells];
    const unsigned per = (n + 1023) / 1024, p0 = min(n, t * per), p1 = min(n, p0 + per);
    const unsigned xfull = gz::crc_xpow8(pw, kPiece);
    auto size = [&](const PieceInfo& f) {
        return static_cast<unsigned long long>(f.out) + ((f.flags & 1) ? hdr : 0) + ((f.flags & 2) ? kTrailerBytes : 0);
    };
    auto join = [&](unsigned crc, const PieceInfo& f) {
        return gz::crc_mul(f.in == kPiece ? xfull : gz::crc_xpow8(pw, f.in), crc) ^ f.crc;
    };
    unsigned long long sum = 0, len = 0;
    unsigned crc = 0;
    for (unsigned p = p0; p < p1; ++p) {
        const PieceInfo f = info[p];
        sum += size(f);
        crc = join(crc, f);
        len += f.in;
    }
    s_sum[t] = sum, s_len[t] = len, s_crc[t] = crc;
    __syncthreads();
    for (unsigned d = 1; d < 1024; d <<= 1) {  // inclusive scans: sums, and (crc, len) under the join
        unsigned long long a = 0, l2 = 0;
        unsigned c2 = 0;
        if (t >= d) a = s_sum[t - d], c2 = s_crc[t - d], l2 = s_len[t - d];
        __syncthreads();
        if (t >= d) {
            s_sum[t] += a;
            s_crc[t] = gz::crc_join(pw, c2, s_crc[t], s_len[t]);
            s_len[t] += l2;
        }
        __syncthreads();
    }
    unsigned long long run = t ? s_sum[t - 1] : 0ull;
    unsigned rc = t ? s_crc[t - 1] : 0u;
    for (unsigned p = p0; p < p1; ++p) {
        const PieceInfo f = info[p];
        start[p] = run, crc_pre[p] = rc;
        run += size(f);
        rc = join(rc, f);
    }
    if (t == 1023) start[n] = s_sum[1023], crc_pre[n] = s_crc[1023];
}

// Member offsets (n_cells + 1), gzip header and trailer of every non-empty cell.  bgzf: htslib's header, whose BC
// field holds the member's size - 1 (the cells are BGZF blocks here).
__global__ void __launch_bounds__(128) deflate_cells_kernel(const unsigned long long* __restrict__ cell_off, unsigned n_cells,
                                                            const unsigned* __restrict__ first_piece,
                                                            const unsigned long long* __restrict__ start,
                                                            const unsigned* __restrict__ crc_pre, unsigned char* __restrict__ out,
                                                            unsigned long long* __restrict__ out_off, gz::CrcPowers pw, bool bgzf) {
    const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > n_cells) return;
    const unsigned a = first_piece[c];
    out_off[c] = start[a];
    if (c == n_cells) return;
    const unsigned b = first_piece[c + 1];
    if (a == b) return;
    const unsigned long long len = cell_off[c + 1] - cell_off[c];
    unsigned char* const h = out + start[a];
    if (bgzf) {
        const unsigned bsize = static_cast<unsigned>(start[b] - start[a] - 1);
        const unsigned char head[kBgzfHeaderBytes] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0,
                                                      static_cast<unsigned char>(bsize), static_cast<unsigned char>(bsize >> 8)};
        for (int i = 0; i < kBgzfHeaderBytes; ++i) h[i] = head[i];
    } else {
        const unsigned char head[kHeaderBytes] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 3};  // zlib's, wbits = 31
        for (int i = 0; i < kHeaderBytes; ++i) h[i] = head[i];
    }
    const unsigned crc = crc_pre[b] ^ gz::crc_mul(gz::crc_xpow8(pw, len), crc_pre[a]);
    const unsigned isize = static_cast<unsigned>(len);
    unsigned char* const e = out + start[b] - kTrailerBytes;
    e[0] = 3, e[1] = 0;  // final empty block with fixed codes
    for (int i = 0; i < 4; ++i) e[2 + i] = static_cast<unsigned char>(crc >> (8 * i)), e[6 + i] = static_cast<unsigned char>(isize >> (8 * i));
}

// Piece bytes into place (behind a header of `hdr` bytes for a cell's first piece).  One CTA per piece (grid-stride).
__global__ void __launch_bounds__(256) deflate_gather_kernel(const unsigned* __restrict__ first_piece, unsigned n_cells,
                                                             const PieceInfo* __restrict__ info,
                                                             const unsigned long long* __restrict__ start,
                                                             const unsigned char* __restrict__ scratch, unsigned char* __restrict__ out,
                                                             int hdr) {
    const unsigned n = first_piece[n_cells];
    for (unsigned p = blockIdx.x; p < n; p += gridDim.x) {
        const PieceInfo f = info[p];
        const unsigned char* const s = scratch + static_cast<unsigned long long>(p) * kPieceCap;
        unsigned char* const d = out + start[p] + ((f.flags & 1) ? hdr : 0);
        for (unsigned i = threadIdx.x; i < f.out; i += blockDim.x) d[i] = s[i];
    }
}

// BGZF: out_off[c] = output offset of cell c's first block (n_cells + 1 entries), from the blocks' offsets.
__global__ void __launch_bounds__(128) deflate_cell_offsets_kernel(const unsigned* __restrict__ first_block, unsigned n_cells,
                                                                   const unsigned long long* __restrict__ block_out,
                                                                   unsigned long long* __restrict__ out_off) {
    const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c <= n_cells) out_off[c] = block_out[first_block[c]];
}

}  // namespace dfl
}  // namespace frb
