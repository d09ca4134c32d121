// Device-side gzip inflate of ONE stream in parallel (SURVEY 8 f-1; the reference inflates with a single
// zlib thread, gzip.open F:159 / F:776).
//
// DEFLATE is a serial bit stream: a block can only be decoded once its first bit is known, and a match may
// reach 32 KiB back into output that another decoder has not produced yet.  Both are dealt with the way
// parallel host decompressors do it (pugz, rapidgzip), here with one warp per chunk of the compressed bytes:
//
//   gz_find_kernel     for every chunk boundary: the first bit at or after it where a dynamic-Huffman block
//                      starts -- every bit position is tried in parallel (block type, code-length code complete,
//                      literal/length and distance codes valid, first symbols decodable).
//   gz_decode_kernel   one warp per chunk, from its block start to the next chunk's: lane 0 walks the Huffman
//                      codes, all lanes copy matches and build tables.  Output is 16-bit symbols: a byte, or a
//                      MARKER (0x8000 + offset) for a match that reaches into the 32 KiB before the chunk.
//   gz_tailmap/groupwin/windows   the last 32 KiB in front of every chunk.  (The 32 KiB behind a chunk are its last
//                      symbols with their markers looked up in the 32 KiB in front of it: a chain over all chunks,
//                      cut into groups whose maps compose.)
//   gz_resolve_kernel  every symbol of every chunk to its byte, markers through the chunk's window; all chunks in
//                      parallel, output contiguous.
//
// A false block start (a bit pattern inside a block that passes every check) shows when the chunk in front of it
// does not stop exactly there: the host then inflates that file with zlib instead.  gzip members may follow each
// other (multi-member files, BGZF); trailers are skipped, ISIZE is checked against the bytes produced.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "crc32.cuh"

namespace frb {
namespace gz {

constexpr int kLitBits = 10;                 // one-step look-up of literal/length codes up to this length
constexpr int kDistBits = 9;
constexpr unsigned kWindow = 32768;
constexpr unsigned kMarker = 0x8000;         // symbol >= kMarker: byte at offset (symbol - kMarker) of the window
constexpr int kFindThreads = 128;
constexpr int kFindWindow = 8192;            // bit positions per round of the finder
constexpr int kDecodeWarps = 4;              // warps (= chunks) per decode CTA

enum : int {
    GZ_OK = 0,
    GZ_END = 1,          // the stream ended (last member complete, no bytes left)
    GZ_ERR_DATA = -1,    // invalid deflate / gzip data
    GZ_ERR_SPACE = -2,   // staging area of the chunk too small
    GZ_ERR_TRUNC = -3,   // the data ends inside a member
};

struct Chunk {
    unsigned long long start_bit;  // first bit of the block the chunk starts with
    unsigned long long stop_bit;   // a block must begin exactly here: stop (~0: run to the end of the data)
    unsigned long long end_bit;    // where decoding stopped
    unsigned long long out_off;    // symbols in front of this chunk (exclusive sum of n_out)
    unsigned long long stage_off;  // first symbol of the chunk's staging area
    unsigned int stage_cap;
    unsigned int n_out;
    int status;
    unsigned int found;            // a block start was found for this chunk
    unsigned int isize_ok;         // every member trailer passed agreed with the bytes produced
    unsigned int member_start;     // a gzip member begins with this chunk's first block: nothing in front to refer to
};

// A member trailer the decoder passed: the member ends `local_end` symbols into chunk `chunk`.
struct Trailer {
    unsigned int chunk, local_end, crc, isize;
    unsigned long long comp_end;   // byte behind the trailer in the piece buffer (which FILE of a batch ends here)
};

// ---- bit access ---------------------------------------------------------------------------------------------
// 64 bits starting at absolute bit `pos` (LSB first, as deflate packs them).  The buffer is word aligned and
// padded with 64 zero bytes behind its `nbytes`, so the three aligned 32-bit loads never leave it.
__device__ __forceinline__ unsigned long long bits64(const unsigned char* __restrict__ d, unsigned long long pos) {
    const unsigned* const w = reinterpret_cast<const unsigned*>(d) + (pos >> 5);
    const unsigned sh = static_cast<unsigned>(pos & 31);
    const unsigned long long lo = static_cast<unsigned long long>(w[0]) | (static_cast<unsigned long long>(w[1]) << 32);
    return sh ? (lo >> sh) | (static_cast<unsigned long long>(w[2]) << (64 - sh)) : lo;
}
// n <= 32 bits starting at absolute bit `pos`; positions at or behind the end of the data read as 0.
__device__ __forceinline__ unsigned peek(const unsigned char* __restrict__ d, unsigned long long nbytes,
                                         unsigned long long pos, int n) {
    if ((pos >> 3) >= nbytes) return 0;
    const unsigned* const w = reinterpret_cast<const unsigned*>(d) + (pos >> 5);
    const unsigned long long v = static_cast<unsigned long long>(w[0]) | (static_cast<unsigned long long>(w[1]) << 32);
    return static_cast<unsigned>((v >> (pos & 31)) & (n == 32 ? 0xFFFFFFFFull : ((1ull << n) - 1)));
}

__device__ __forceinline__ unsigned rev_bits(unsigned code, int len) { return __brev(code) >> (32 - len); }

// Canonical code over lens[0, n): returns 0 complete, > 0 incomplete (unused code space), < 0 over-subscribed.
// count[l] = codes of length l.
__device__ __forceinline__ int code_space(const unsigned char* lens, int n, unsigned short* count) {
    for (int l = 0; l <= 15; ++l) count[l] = 0;
    for (int s = 0; s < n; ++s) count[lens[s]]++;
    int left = 1;
    for (int l = 1; l <= 15; ++l) {
        left <<= 1;
        left -= count[l];
        if (left < 0) return left;
    }
    return left;
}

// zlib's rule for a literal/length or distance code (inftrees.c): never over-subscribed; incomplete only as a
// single code of length 1 -- or, for distances, no code at all.
__device__ __forceinline__ bool code_ok(const unsigned char* lens, int n, unsigned short* count, bool may_be_empty) {
    const int left = code_space(lens, n, count);
    if (left < 0) return false;
    if (left == 0) return true;
    const int used = n - count[0];
    return (used == 1 && count[1] == 1) || (used == 0 && may_be_empty);
}

__device__ __constant__ unsigned short c_len_base[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43,
                                                         51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__device__ __constant__ unsigned char c_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3,
                                                         3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__device__ __constant__ unsigned short c_dist_base[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257,
                                                          385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193,
                                                          12289, 16385, 24577};
__device__ __constant__ unsigned char c_dist_extra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7,
                                                          8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__device__ __constant__ unsigned char c_cl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// Header of a dynamic block at bit `pos` (just behind BFINAL/BTYPE): code lengths of the literal/length code
// into lens[0, 288) and of the distance code into lens[288, 320).  Applies zlib's validity rules (inflate.c /
// inftrees.c: complete code-length code; literal/length and distance codes complete, or incomplete with a single
// code; no repeat without a previous length; end-of-block code present).  Returns the bit behind the header or 0.
__device__ inline unsigned long long dynamic_header(const unsigned char* __restrict__ d, unsigned long long nbytes,
                                                    unsigned long long pos, unsigned char* lens, int* n_lit, int* n_dist) {
    const unsigned h = peek(d, nbytes, pos, 14);
    const int hlit = (h & 31) + 257, hdist = ((h >> 5) & 31) + 1, hclen = ((h >> 10) & 15) + 4;
    if (hlit > 286 || hdist > 30) return 0;
    pos += 14;
    unsigned char cl[19];
#pragma unroll
    for (int i = 0; i < 19; ++i) cl[i] = 0;
    for (int i = 0; i < hclen; ++i, pos += 3) cl[c_cl_order[i]] = static_cast<unsigned char>(peek(d, nbytes, pos, 3));
    unsigned short count[16];
    if (code_space(cl, 19, count) != 0) return 0;  // the code-length code must be complete
    // canonical decode of the code-length code, bit by bit (at most 7 bits)
    unsigned short offs[8], sym[19];
    offs[1] = 0;
    for (int l = 1; l < 7; ++l) offs[l + 1] = offs[l] + count[l];
    for (int s = 0; s < 19; ++s)
        if (cl[s]) sym[offs[cl[s]]++] = static_cast<unsigned short>(s);
    const int total = hlit + hdist;
    int idx = 0;
    unsigned char prev = 0;
    // code space left (in units of 2^-15) while the lengths come in: an over-subscribed code is given up at once --
    // what bits that are not a block header turn into after a few dozen lengths
    int room[2] = {1 << 15, 1 << 15};
    while (idx < total) {
        unsigned bits = peek(d, nbytes, pos, 7 + 7);
        int code = 0, first = 0, index = 0, s = -1, used = 0;
        for (int l = 1; l <= 7; ++l) {
            code |= bits & 1;
            bits >>= 1;
            const int c = count[l];
            if (code - c < first) {
                s = sym[index + (code - first)];
                used = l;
                break;
            }
            index += c;
            first += c;
            first <<= 1;
            code <<= 1;
        }
        if (s < 0) return 0;
        if (s < 16) {
            lens[idx < hlit ? idx : 288 + (idx - hlit)] = prev = static_cast<unsigned char>(s);
            if (s && (room[idx >= hlit] -= (1 << 15) >> s) < 0) return 0;
            ++idx;
            pos += used;
        } else {
            int rep;
            unsigned char val = 0;
            if (s == 16) {
                if (idx == 0) return 0;
                val = prev;
                rep = 3 + ((bits)&3);
                pos += used + 2;
            } else if (s == 17) {
                rep = 3 + (bits & 7);
                pos += used + 3;
            } else {
                rep = 11 + (bits & 127);
                pos += used + 7;
            }
            if (idx + rep > total) return 0;
            for (; rep; --rep, ++idx) {
                lens[idx < hlit ? idx : 288 + (idx - hlit)] = val;
                if (val && (room[idx >= hlit] -= (1 << 15) >> val) < 0) return 0;
            }
            prev = val;
        }
    }
    if ((pos >> 3) > nbytes) return 0;
    if (lens[256] == 0) return 0;  // no end-of-block code
    for (int i = hlit; i < 288; ++i) lens[i] = 0;
    for (int i = hdist; i < 32; ++i) lens[288 + i] = 0;
    if (!code_ok(lens, hlit, count, false) || !code_ok(lens + 288, hdist, count, true)) return 0;
    *n_lit = hlit, *n_dist = hdist;
    return pos;
}

// Slow exact decode of one symbol of a canonical code (count / sorted symbols), puff.c's loop; -1 = no such code.
__device__ __forceinline__ int decode_slow(unsigned bits, const unsigned short* count, const unsigned short* sorted,
                                           int* used) {
    int code = 0, first = 0, index = 0;
    for (int l = 1; l <= 15; ++l) {
        code |= bits & 1;
        bits >>= 1;
        const int c = count[l];
        if (code - c < first) {
            *used = l;
            return sorted[index + (code - first)];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

__device__ inline unsigned long long member_header(const unsigned char* __restrict__ d, unsigned long long nbytes,
                                                   unsigned long long pos);

// Is a dynamic block likely to start at bit `pos`?  Header valid, and the first symbols decode (no unused code, no
// distance beyond the window).  One thread, local scratch only.
// The test in three steps of rising cost, so that the finder can run each step on a dense list of survivors:
//   block_head_ok   block type and code counts (the first 13 bits)
//   block_kraft_ok  the code-length code is complete (Kraft sum of its up to 19 three-bit lengths)
//   block_body_ok   the code lengths decode to valid codes and the first symbols decode
__device__ __forceinline__ bool block_head_ok(unsigned v, bool any_final) {
    // BTYPE = 10; BFINAL = 0 -- a last block is only looked for behind a member header (any_final)
    return (v & (any_final ? 6u : 7u)) == 4u && ((v >> 3) & 31u) <= 29u && ((v >> 8) & 31u) <= 29u;
}
__device__ __forceinline__ bool block_kraft_ok(const unsigned char* __restrict__ d, unsigned long long pos) {
    const int hclen = static_cast<int>((bits64(d, pos) >> 13) & 15) + 4;
    const unsigned long long cl = bits64(d, pos + 17);
    unsigned kraft = 0;
    for (int i = 0; i < hclen; ++i) {
        const unsigned l = static_cast<unsigned>(cl >> (3 * i)) & 7u;
        kraft += l ? (128u >> l) : 0u;
    }
    return kraft == 128u;
}
__device__ inline bool block_body_ok(const unsigned char* __restrict__ d, unsigned long long nbytes, unsigned long long pos);

__device__ inline bool plausible_block_start(const unsigned char* __restrict__ d, unsigned long long nbytes,
                                             unsigned long long pos, bool any_final = false) {
    return block_head_ok(static_cast<unsigned>(bits64(d, pos)), any_final) && block_kraft_ok(d, pos) &&
           block_body_ok(d, nbytes, pos);
}

__device__ inline bool block_body_ok(const unsigned char* __restrict__ d, unsigned long long nbytes, unsigned long long pos) {
    unsigned char lens[320];
    int n_lit, n_dist;
    unsigned long long p = dynamic_header(d, nbytes, pos + 3, lens, &n_lit, &n_dist);
    if (!p) return false;
    unsigned short lcount[16], dcount[16], lsorted[288], dsorted[32], offs[16];
    code_space(lens, n_lit, lcount);
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + lcount[l];
    for (int s = 0; s < n_lit; ++s)
        if (lens[s]) lsorted[offs[lens[s]]++] = static_cast<unsigned short>(s);
    code_space(lens + 288, n_dist, dcount);
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + dcount[l];
    for (int s = 0; s < n_dist; ++s)
        if (lens[288 + s]) dsorted[offs[lens[288 + s]]++] = static_cast<unsigned short>(s);
    unsigned produced = 0;
    for (int k = 0; k < 1024; ++k) {  // the first symbols of the block
        if ((p >> 3) >= nbytes) return false;
        int used;
        int s = decode_slow(peek(d, nbytes, p, 15), lcount, lsorted, &used);
        if (s < 0) return false;
        p += used;
        if (s < 256) {
            ++produced;
            continue;
        }
        if (s == 256) return true;
        s -= 257;
        if (s >= 29) return false;
        p += c_len_extra[s];
        const int ds = decode_slow(peek(d, nbytes, p, 15), dcount, dsorted, &used);
        if (ds < 0 || ds >= 30) return false;
        p += used;
        const unsigned dist = c_dist_base[ds] + peek(d, nbytes, p, c_dist_extra[ds]);
        p += c_dist_extra[ds];
        if (dist > produced + kWindow) return false;
        produced += 3;
    }
    return true;
}

// chunk c (> 0 or search_first): first plausible block start at or after byte c * stride (bit granular), before
// `limit_bit`.  One CTA per chunk; the threads try consecutive bit positions.
__global__ void __launch_bounds__(kFindThreads) gz_find_kernel(const unsigned char* __restrict__ d, unsigned long long nbytes,
                                                               Chunk* chunks, unsigned n_chunks, unsigned long long stride,
                                                               unsigned long long first_byte, unsigned first_chunk,
                                                               unsigned tail_chunk, unsigned long long tail_reach) {
    const unsigned c = blockIdx.x + first_chunk;
    if (c >= n_chunks) return;
    __shared__ unsigned long long s_best;
    if (threadIdx.x == 0) s_best = ~0ull;
    __syncthreads();
    const unsigned long long from = (first_byte + static_cast<unsigned long long>(c) * stride) * 8;
    // search one stride and a half: a start behind that belongs to the next chunk anyway
    // (the chunk behind the piece, whose start closes the piece's last chunk, looks through the overlap the piece
    // buffer carries: tail_reach bytes)
    const bool tail = c == tail_chunk;
    const unsigned long long reach = tail ? tail_reach : stride + stride / 2;
    const unsigned long long to = min((first_byte + static_cast<unsigned long long>(c) * stride + reach) * 8, nbytes * 8);
    // kFindWindow bit positions per round, in three passes: every position gets the 13-bit test; the survivors
    // (one in nine) are collected and shared out over ALL threads for the Kraft sum; what is left of them (a few
    // dozen) is collected again for the expensive part.  Done in place, a single survivor in a warp keeps the other
    // 31 lanes waiting through its code lengths and trial decode: 3.5e9 warp instructions per piece at ten active
    // lanes, most of them that wait.
    __shared__ unsigned short s_a[kFindWindow], s_b[kFindWindow];
    __shared__ unsigned s_na, s_nb;
    for (unsigned long long base = from; base < to; base += kFindWindow) {
        if (threadIdx.x == 0) s_na = 0, s_nb = 0;
        __syncthreads();
        for (int r = 0; r < kFindWindow / kFindThreads; ++r) {
            const unsigned rel = r * kFindThreads + threadIdx.x;
            const unsigned long long p = base + rel;
            if (p >= to) break;
            if (block_head_ok(static_cast<unsigned>(bits64(d, p)), false)) s_a[atomicAdd(&s_na, 1u)] = static_cast<unsigned short>(rel);
            // a gzip member header (files of many small members, BGZF): the first block of a member may be its
            // last, and nothing in front of it is referred to
            if ((p & 7) == 0) {
                const unsigned long long b = p >> 3;
                if (b + 18 < nbytes && d[b] == 0x1f && d[b + 1] == 0x8b && d[b + 2] == 8) {
                    const unsigned long long hb = member_header(d, nbytes, b);
                    if (hb && plausible_block_start(d, nbytes, hb * 8, true)) atomicMin(&s_best, (hb * 8) << 1);
                }
            }
        }
        __syncthreads();
        const unsigned na = s_na;
        for (unsigned i = threadIdx.x; i < na; i += kFindThreads)
            if (block_kraft_ok(d, base + s_a[i])) s_b[atomicAdd(&s_nb, 1u)] = s_a[i];
        __syncthreads();
        const unsigned nb = s_nb;
        for (unsigned i = threadIdx.x; i < nb; i += kFindThreads) {
            const unsigned long long p = base + s_b[i];
            if (block_body_ok(d, nbytes, p)) atomicMin(&s_best, (p << 1) | 1ull);
        }
        __syncthreads();
        if (s_best != ~0ull) break;
    }
    if (threadIdx.x == 0) {  // s_best = (bit << 1) | 1, or bit << 1 for the first block of a member
        const unsigned long long best = s_best >> 1;
        chunks[c].found = s_best != ~0ull && (tail || best < (first_byte + static_cast<unsigned long long>(c + 1) * stride) * 8);
        chunks[c].start_bit = best;
        chunks[c].member_start = s_best != ~0ull && (s_best & 1) == 0;
    }
}

// stop_bit of every found chunk = start of the next found chunk; chunks without a start are skipped (the chunk in
// front of them decodes through).  One thread.
// has_tail: chunks[n_chunks] is the search result for the first block start behind the piece (where the piece's
// last chunk stops); without one found the piece cannot be closed (*fail = 1).
__global__ void gz_link_kernel(Chunk* chunks, unsigned n_chunks, unsigned long long stage_per_chunk, int has_tail,
                               unsigned* fail) {
    if (threadIdx.x || blockIdx.x) return;
    unsigned long long next = ~0ull;
    if (has_tail) {
        if (chunks[n_chunks].found) next = chunks[n_chunks].start_bit;
        else *fail = 1;
    }
    // a chunk that absorbs k skipped neighbours also gets their staging areas (areas are consecutive)
    unsigned long long cap = 0;
    for (int c = static_cast<int>(n_chunks) - 1; c >= 0; --c) {
        cap += stage_per_chunk;
        chunks[c].stage_off = static_cast<unsigned long long>(c) * stage_per_chunk;
        chunks[c].n_out = 0;
        chunks[c].status = GZ_OK;
        chunks[c].isize_ok = 1;
        chunks[c].end_bit = 0;
        if (chunks[c].found) {
            chunks[c].stop_bit = next;
            chunks[c].stage_cap = static_cast<unsigned>(cap < 0xFFFFFFFFull ? cap : 0xFFFFFFFFull);
            next = chunks[c].start_bit;
            cap = 0;
        } else {
            chunks[c].stage_cap = 0;
        }
    }
}

// Shared-memory tables of one decoding warp.
struct WarpTables {
    unsigned short lit[1 << kLitBits];    // (symbol << 4) | code length, 0 = longer code or none
    unsigned short dist[1 << kDistBits];
    unsigned short lcount[16], dcount[16];
    unsigned short lsorted[288], dsorted[32];
    unsigned char lens[320];
};

// gzip member header at byte `pos` (RFC 1952): returns the byte behind it, 0 = not a gzip header / truncated.
__device__ inline unsigned long long member_header(const unsigned char* __restrict__ d, unsigned long long nbytes,
                                                   unsigned long long pos) {
    if (pos + 10 > nbytes) return 0;
    if (d[pos] != 0x1f || d[pos + 1] != 0x8b || d[pos + 2] != 8) return 0;
    const unsigned flg = d[pos + 3];
    if (flg & 0xE0) return 0;
    pos += 10;
    if (flg & 4) {  // FEXTRA
        if (pos + 2 > nbytes) return 0;
        pos += 2 + (d[pos] | (d[pos + 1] << 8));
    }
    for (int k = 0; k < 2; ++k)  // FNAME, FCOMMENT
        if (flg & (8 << k)) {
            while (pos < nbytes && d[pos]) ++pos;
            ++pos;
        }
    if (flg & 2) pos += 2;  // FHCRC
    return pos <= nbytes ? pos : 0;
}

// One warp per chunk.  Lane 0 reads bits and walks the codes; the warp copies matches, builds tables.
__global__ void __launch_bounds__(kDecodeWarps * 32) gz_decode_kernel(const unsigned char* __restrict__ d,
                                                                      unsigned long long nbytes, Chunk* chunks,
                                                                      unsigned n_chunks, unsigned short* stage,
                                                                      Trailer* trailers, unsigned trailer_cap,
                                                                      unsigned* trailer_n, const unsigned* link_failed) {
    __shared__ WarpTables s_tab[kDecodeWarps];
    if (*link_failed) return;  // no block start behind the piece: the host inflates this file
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned c = blockIdx.x * kDecodeWarps + w;
    if (c >= n_chunks || !chunks[c].found) return;
    WarpTables& T = s_tab[w];
    const unsigned long long stop = chunks[c].stop_bit;
    unsigned short* const out = stage + chunks[c].stage_off;
    const unsigned cap = chunks[c].stage_cap;
    unsigned long long pos = chunks[c].start_bit;
    unsigned n = 0;             // symbols produced
    // output index of the first byte of the member being decoded, once one began in this chunk
    unsigned known_from = chunks[c].member_start ? 0u : ~0u;
    unsigned long long member_out0 = 0;  // symbols of this chunk when the current member began (for ISIZE)
    int status = GZ_OK;
    unsigned isize_ok = 1;

    for (;;) {  // blocks
        if (pos == stop) break;
        if (stop != ~0ull && pos > stop) { status = GZ_ERR_DATA; break; }  // ran past the next chunk's start
        if ((pos >> 3) >= nbytes) { status = GZ_ERR_TRUNC; break; }
        const unsigned hdr = peek(d, nbytes, pos, 3);
        const unsigned bfinal = hdr & 1, btype = hdr >> 1;
        pos += 3;
        if (btype == 3) { status = GZ_ERR_DATA; break; }
        if (btype == 0) {  // stored
            pos = (pos + 7) & ~7ull;
            const unsigned long long b = pos >> 3;
            if (b + 4 > nbytes) { status = GZ_ERR_TRUNC; break; }
            const unsigned len = d[b] | (d[b + 1] << 8), nlen = d[b + 2] | (d[b + 3] << 8);
            if ((len ^ nlen) != 0xFFFFu) { status = GZ_ERR_DATA; break; }
            if (b + 4 + len > nbytes) { status = GZ_ERR_TRUNC; break; }
            if (n + len > cap) { status = GZ_ERR_SPACE; break; }
            for (unsigned i = lane; i < len; i += 32) out[n + i] = d[b + 4 + i];
            n += len;
            pos = (b + 4 + len) * 8;
            __syncwarp();
        } else {
            // ---- code lengths ----
            int n_lit = 288, n_dist = 30;
            if (btype == 1) {
                for (int i = lane; i < 320; i += 32)
                    T.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : i < 288 + 30 ? 5 : 0;
            } else {
                unsigned long long p2 = 0;
                if (lane == 0) p2 = dynamic_header(d, nbytes, pos, T.lens, &n_lit, &n_dist);
                p2 = __shfl_sync(0xFFFFFFFFu, p2, 0);
                n_lit = __shfl_sync(0xFFFFFFFFu, n_lit, 0);
                n_dist = __shfl_sync(0xFFFFFFFFu, n_dist, 0);
                if (!p2) { status = (pos >> 3) + 40 > nbytes ? GZ_ERR_TRUNC : GZ_ERR_DATA; break; }
                pos = p2;
            }
            __syncwarp();
            // ---- tables: canonical codes by lane 0, look-up fill by all lanes ----
            for (int i = lane; i < (1 << kLitBits); i += 32) T.lit[i] = 0;
            for (int i = lane; i < (1 << kDistBits); i += 32) T.dist[i] = 0;
            __syncwarp();
            if (lane == 0) {
                unsigned short offs[16];
                code_space(T.lens, n_lit, T.lcount);
                offs[1] = 0;
                for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + T.lcount[l];
                for (int s = 0; s < n_lit; ++s)
                    if (T.lens[s]) T.lsorted[offs[T.lens[s]]++] = static_cast<unsigned short>(s);
                code_space(T.lens + 288, n_dist, T.dcount);
                offs[1] = 0;
                for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + T.dcount[l];
                for (int s = 0; s < n_dist; ++s)
                    if (T.lens[288 + s]) T.dsorted[offs[T.lens[288 + s]]++] = static_cast<unsigned short>(s);
            }
            __syncwarp();
            // the k-th symbol (in sorted order) of length l has code first[l] + (k - index[l]); every lane takes
            // sorted positions lane, lane + 32, ...
            {
                unsigned first = 0, index = 0;
                unsigned lfirst[16], lindex[16];
                for (int l = 1; l <= 15; ++l) {
                    lfirst[l] = first, lindex[l] = index;
                    index += T.lcount[l];
                    first = (first + T.lcount[l]) << 1;
                }
                const unsigned n_codes = index;
                for (unsigned k = lane; k < n_codes; k += 32) {
                    const unsigned s = T.lsorted[k];
                    const int l = T.lens[s];
                    if (l > kLitBits) continue;
                    const unsigned r = rev_bits(lfirst[l] + (k - lindex[l]), l);
                    for (unsigned e = r; e < (1u << kLitBits); e += 1u << l) T.lit[e] = static_cast<unsigned short>((s << 4) | l);
                }
                first = 0, index = 0;
                for (int l = 1; l <= 15; ++l) {
                    lfirst[l] = first, lindex[l] = index;
                    index += T.dcount[l];
                    first = (first + T.dcount[l]) << 1;
                }
                const unsigned n_dcodes = index;
                for (unsigned k = lane; k < n_dcodes; k += 32) {
                    const unsigned s = T.dsorted[k];
                    const int l = T.lens[288 + s];
                    if (l > kDistBits) continue;
                    const unsigned r = rev_bits(lfirst[l] + (k - lindex[l]), l);
                    for (unsigned e = r; e < (1u << kDistBits); e += 1u << l) T.dist[e] = static_cast<unsigned short>((s << 4) | l);
                }
            }
            __syncwarp();
            // ---- symbols ----
            // lane 0 keeps a 64-bit bit buffer fed with aligned 32-bit words
            unsigned long long buf = 0;
            int cnt = 0;
            unsigned long long wpos = 0;  // next 32-bit word to load
            const unsigned* const d32 = reinterpret_cast<const unsigned*>(d);
            const unsigned long long nwords = (nbytes + 3) >> 2;  // the buffer is padded to whole words
            if (lane == 0) {
                wpos = pos >> 5;
                buf = (wpos < nwords ? d32[wpos] : 0u) >> (pos & 31);
                cnt = 32 - static_cast<int>(pos & 31);
                ++wpos;
            }
            for (;;) {
                // op: 0 literal(s) done by lane 0, 1 match, 2 end of block, < 0 error
                int op = 0;
                unsigned mlen = 0, mdist = 0;
                if (lane == 0) {
                    // a run of literals without involving the other lanes
                    for (;;) {
                        if (cnt <= 32) {
                            // more than two words of padding taken in: the block runs past the end of the data
                            if (wpos > nwords + 2) { op = GZ_ERR_TRUNC; break; }
                            buf |= static_cast<unsigned long long>(wpos < nwords ? d32[wpos] : 0u) << cnt;
                            cnt += 32;
                            ++wpos;
                        }
                        unsigned e = T.lit[buf & ((1u << kLitBits) - 1)];
                        int used = e & 15;
                        int s = e >> 4;
                        if (e == 0) {
                            s = decode_slow(static_cast<unsigned>(buf), T.lcount, T.lsorted, &used);
                            if (s < 0) { op = GZ_ERR_DATA; break; }
                        }
                        buf >>= used, cnt -= used;
                        if (s < 256) {
                            if (n >= cap) { op = GZ_ERR_SPACE; break; }
                            out[n++] = static_cast<unsigned short>(s);
                            continue;
                        }
                        if (s == 256) { op = 2; break; }
                        s -= 257;
                        if (s >= 29) { op = GZ_ERR_DATA; break; }
                        mlen = c_len_base[s] + (static_cast<unsigned>(buf) & ((1u << c_len_extra[s]) - 1));
                        buf >>= c_len_extra[s], cnt -= c_len_extra[s];
                        if (cnt <= 32) {
                            buf |= static_cast<unsigned long long>(wpos < nwords ? d32[wpos] : 0u) << cnt;
                            cnt += 32;
                            ++wpos;
                        }
                        e = T.dist[buf & ((1u << kDistBits) - 1)];
                        used = e & 15;
                        int ds = e >> 4;
                        if (e == 0) {
                            ds = decode_slow(static_cast<unsigned>(buf), T.dcount, T.dsorted, &used);
                            if (ds < 0) { op = GZ_ERR_DATA; break; }
                        }
                        buf >>= used, cnt -= used;
                        if (ds >= 30) { op = GZ_ERR_DATA; break; }
                        mdist = c_dist_base[ds] + (static_cast<unsigned>(buf) & ((1u << c_dist_extra[ds]) - 1));
                        buf >>= c_dist_extra[ds], cnt -= c_dist_extra[ds];
                        op = 1;
                        break;
                    }
                }
                op = __shfl_sync(0xFFFFFFFFu, op, 0);
                if (op == 2 || op < 0) {
                    if (op < 0) status = op;
                    break;
                }
                mlen = __shfl_sync(0xFFFFFFFFu, mlen, 0);
                mdist = __shfl_sync(0xFFFFFFFFu, mdist, 0);
                n = __shfl_sync(0xFFFFFFFFu, n, 0);
                if (n + mlen > cap) { status = GZ_ERR_SPACE; break; }
                // A match that starts in front of the member (possible only for the chunk's first member, whose
                // beginning lies in an earlier chunk) is a marker into the 32 KiB before the chunk.
                __syncwarp();  // lane 0's literals are visible to the lanes that copy
                const long long src0 = static_cast<long long>(n) - static_cast<long long>(mdist);
                if (src0 < 0 && (mdist > n + kWindow || known_from != ~0u)) { status = GZ_ERR_DATA; break; }
                if (known_from != ~0u && src0 < static_cast<long long>(known_from)) { status = GZ_ERR_DATA; break; }
                for (unsigned i = lane; i < mlen; i += 32) {
                    const long long src = src0 + static_cast<long long>(i % mdist);
                    out[n + i] = src >= 0 ? __ldcg(out + src) : static_cast<unsigned short>(kMarker + (src + kWindow));
                }
                n += mlen;
                __syncwarp();
            }
            // where the bit buffer stands
            unsigned long long endpos = 0;
            if (lane == 0) endpos = wpos * 32 - cnt;
            pos = __shfl_sync(0xFFFFFFFFu, endpos, 0);
            n = __shfl_sync(0xFFFFFFFFu, n, 0);
            if (status != GZ_OK) break;
        }
        if (bfinal) {
            // member trailer (CRC32, ISIZE), then another member or the end of the data
            const unsigned long long b = (pos + 7) >> 3;
            if (b + 8 > nbytes) { status = GZ_ERR_TRUNC; break; }
            const unsigned isize = d[b + 4] | (d[b + 5] << 8) | (d[b + 6] << 16) | (static_cast<unsigned>(d[b + 7]) << 24);
            // bytes of the member produced by THIS chunk can be checked only when the member began here
            if (known_from != ~0u && static_cast<unsigned>(n - member_out0) != isize) isize_ok = 0;
            if (lane == 0) {  // CRC32 and ISIZE of the whole member are checked once the text is there (gz_crc_*)
                const unsigned t = atomicAdd(trailer_n, 1u);
                if (t < trailer_cap) {
                    const unsigned crc = d[b] | (d[b + 1] << 8) | (d[b + 2] << 16) | (static_cast<unsigned>(d[b + 3]) << 24);
                    trailers[t] = Trailer{c, n, crc, isize, b + 8};
                }
            }
            unsigned long long nb = b + 8;
            while (nb < nbytes && d[nb] == 0) ++nb;  // zero padding between / behind members (gzip tolerates it)
            if (nb >= nbytes) {
                pos = nbytes * 8;
                status = GZ_END;
                break;
            }
            const unsigned long long hb = member_header(d, nbytes, nb);
            if (!hb) { status = GZ_ERR_DATA; break; }
            pos = hb * 8;
            known_from = n;
            member_out0 = n;
        }
    }
    if (lane == 0) {
        chunks[c].end_bit = pos;
        chunks[c].n_out = n;
        chunks[c].status = status;
        chunks[c].isize_ok = isize_ok;
    }
}

// out_off = exclusive sum of n_out over the found chunks; *total = all symbols; *bad = first chunk whose end does
// not meet its successor's start or that failed (~0 none).  One block.
__global__ void __launch_bounds__(1024) gz_offsets_kernel(Chunk* chunks, unsigned n_chunks, unsigned long long* total,
                                                          unsigned* bad) {
    __shared__ unsigned long long s_sum[1024];
    __shared__ unsigned s_bad;
    const unsigned t = threadIdx.x;
    if (t == 0) s_bad = 0xFFFFFFFFu;
    __syncthreads();
    const unsigned per = (n_chunks + 1023) / 1024;
    unsigned long long local = 0;
    for (unsigned c = t * per; c < min(n_chunks, (t + 1) * per); ++c) {
        if (!chunks[c].found) continue;
        local += chunks[c].n_out;
        const bool ok = (chunks[c].status == GZ_OK && chunks[c].end_bit == chunks[c].stop_bit) ||
                        (chunks[c].status == GZ_END);
        if (!ok || !chunks[c].isize_ok) atomicMin(&s_bad, c);
    }
    s_sum[t] = local;
    __syncthreads();
    for (unsigned dlt = 1; dlt < 1024; dlt <<= 1) {
        const unsigned long long v = t >= dlt ? s_sum[t - dlt] : 0;
        __syncthreads();
        s_sum[t] += v;
        __syncthreads();
    }
    unsigned long long run = s_sum[t] - local;
    for (unsigned c = t * per; c < min(n_chunks, (t + 1) * per); ++c) {
        chunks[c].out_off = run;
        if (chunks[c].found) run += chunks[c].n_out;
    }
    if (t == 1023) *total = s_sum[1023];
    if (t == 0) *bad = s_bad;
}

// ---- the 32 KiB in front of every chunk -----------------------------------------------------------------------
// The window behind chunk c is a function of the window in front of it: entry j is a byte of the chunk's own
// output, or entry m of the window in front (a marker).  Such maps compose, so the chain over thousands of chunks
// is cut into groups of kGroup chunks:
//   gz_tailmap_kernel   one CTA per group, chunk after chunk: map from the window in front of the GROUP to the
//                       window behind each of its chunks (32 Ki entries of 16 bits, running map in shared memory)
//   gz_groupwin_kernel  one CTA, group after group: the window in front of every group (and behind the last one)
//   gz_windows_kernel   all chunks in parallel: window in front of the chunk = map of the chunk before it applied
//                       to its group's window
constexpr unsigned kGroup = 64;

__global__ void __launch_bounds__(1024) gz_tailmap_kernel(const Chunk* __restrict__ chunks, unsigned n_chunks,
                                                          const unsigned short* __restrict__ stage,
                                                          unsigned short* __restrict__ maps, int* __restrict__ prev_found) {
    extern __shared__ unsigned short s_map[];  // 2 x 32 Ki entries
    unsigned short* cur = s_map;
    unsigned short* nxt = s_map + kWindow;
    for (unsigned i = threadIdx.x; i < kWindow; i += 1024) cur[i] = static_cast<unsigned short>(kMarker + i);  // identity
    __syncthreads();
    const unsigned c0 = blockIdx.x * kGroup, c1 = min(n_chunks, c0 + kGroup);
    int prev = -1;
    for (unsigned c = c0; c < c1; ++c) {
        if (threadIdx.x == 0) prev_found[c] = prev;
        if (!chunks[c].found) continue;
        const unsigned n = chunks[c].n_out;
        const unsigned short* const sym = stage + chunks[c].stage_off;
        unsigned short* const mc = maps + static_cast<unsigned long long>(c) * kWindow;
        for (unsigned j = threadIdx.x; j < kWindow; j += 1024) {
            const long long p = static_cast<long long>(n) - kWindow + j;  // output position; negative: the window in front
            unsigned short e;
            if (p < 0) {
                e = cur[p + kWindow];
            } else {
                const unsigned short sy = sym[p];
                e = sy >= kMarker ? cur[sy - kMarker] : sy;
            }
            nxt[j] = e;
            mc[j] = e;
        }
        __syncthreads();
        unsigned short* t = cur;
        cur = nxt;
        nxt = t;
        prev = static_cast<int>(c);
    }
}

// group_win[g] = the 32 KiB in front of group g; win_out = the 32 KiB behind the last chunk.
__global__ void __launch_bounds__(1024) gz_groupwin_kernel(const Chunk* __restrict__ chunks, unsigned n_chunks,
                                                           const unsigned short* __restrict__ maps,
                                                           const unsigned char* __restrict__ win_in,
                                                           unsigned char* __restrict__ group_win,
                                                           unsigned char* __restrict__ win_out) {
    extern __shared__ unsigned char s_win[];  // 2 x 32 KiB
    unsigned char* cur = s_win;
    unsigned char* nxt = s_win + kWindow;
    for (unsigned i = threadIdx.x; i < kWindow; i += 1024) cur[i] = win_in[i];
    __syncthreads();
    const unsigned n_groups = (n_chunks + kGroup - 1) / kGroup;
    for (unsigned g = 0; g < n_groups; ++g) {
        unsigned char* const gw = group_win + static_cast<unsigned long long>(g) * kWindow;
        for (unsigned i = threadIdx.x; i < kWindow / 16; i += 1024) reinterpret_cast<uint4*>(gw)[i] = reinterpret_cast<const uint4*>(cur)[i];
        // last found chunk of the group
        int last = -1;
        for (int c = static_cast<int>(min(n_chunks, (g + 1) * kGroup)) - 1; c >= static_cast<int>(g * kGroup); --c)
            if (chunks[c].found) {
                last = c;
                break;
            }
        if (last < 0) continue;
        const unsigned short* const m = maps + static_cast<unsigned long long>(last) * kWindow;
        for (unsigned j = threadIdx.x; j < kWindow; j += 1024) {
            const unsigned short e = m[j];
            nxt[j] = e >= kMarker ? cur[e - kMarker] : static_cast<unsigned char>(e);
        }
        __syncthreads();
        unsigned char* t = cur;
        cur = nxt;
        nxt = t;
    }
    for (unsigned i = threadIdx.x; i < kWindow; i += 1024) win_out[i] = cur[i];
}

// windows[c] = the 32 KiB in front of chunk c.  grid.x = chunk.
__global__ void __launch_bounds__(256) gz_windows_kernel(const Chunk* __restrict__ chunks, const unsigned short* __restrict__ maps,
                                                         const int* __restrict__ prev_found,
                                                         const unsigned char* __restrict__ group_win,
                                                         unsigned char* __restrict__ windows) {
    const unsigned c = blockIdx.x;
    if (!chunks[c].found) return;
    const unsigned char* const gw = group_win + static_cast<unsigned long long>(c / kGroup) * kWindow;
    unsigned char* const wc = windows + static_cast<unsigned long long>(c) * kWindow;
    const int prev = prev_found[c];
    if (prev < 0) {
        for (unsigned i = threadIdx.x; i < kWindow / 16; i += 256) reinterpret_cast<uint4*>(wc)[i] = reinterpret_cast<const uint4*>(gw)[i];
        return;
    }
    const unsigned short* const m = maps + static_cast<unsigned long long>(prev) * kWindow;
    for (unsigned j = threadIdx.x; j < kWindow; j += 256) {
        const unsigned short e = m[j];
        wc[j] = e >= kMarker ? gw[e - kMarker] : static_cast<unsigned char>(e);
    }
}

// Every symbol to its byte.  grid.y = chunk, grid.x strides over the chunk's symbols.
__global__ void __launch_bounds__(256) gz_resolve_kernel(const Chunk* __restrict__ chunks, const unsigned short* __restrict__ stage,
                                                         const unsigned char* __restrict__ windows,
                                                         unsigned char* __restrict__ out, unsigned long long out_cap) {
    const unsigned c = blockIdx.y;
    if (!chunks[c].found) return;
    const unsigned n = chunks[c].n_out;
    const unsigned short* const sym = stage + chunks[c].stage_off;
    const unsigned char* const win = windows + static_cast<unsigned long long>(c) * kWindow;
    unsigned char* const dst = out + chunks[c].out_off;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned short s = sym[i];
        if (chunks[c].out_off + i < out_cap) dst[i] = s >= kMarker ? win[s - kMarker] : static_cast<unsigned char>(s);
    }
}

// Position behind the last '\n' of buf[0, n) (0 if there is none) and whether a '\r' occurs at all.
__global__ void __launch_bounds__(1024) gz_text_kernel(const unsigned char* __restrict__ buf, unsigned long long n,
                                                       unsigned long long* last_nl_end, unsigned* has_cr) {
    unsigned long long best = 0;
    unsigned cr = 0;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; i < n; i += stride) {
        const unsigned char b = buf[i];
        if (b == '\n') best = i + 1;
        cr |= b == '\r';
    }
    if (best) atomicMax(last_nl_end, best);
    if (cr) atomicOr(has_cr, 1u);
}

// ---- CRC-32 of the inflated text (RFC 1952 trailer check) -------------------------------------------------------
// Standard CRC-32 values combine like zlib's crc32_combine: crc(A || B) = x^(8 |B|) * crc(A) + crc(B) in
// GF(2)[x] / P (reflected bit order, bit 31 = x^0).  So the text is summed in 4 KiB blocks by warps (gz_crc_blocks),
// the block sums are prefix-combined (gz_crc_scan: F[b] = crc of text[0, 4096 b)), and every member end e gets
// F(e) from F[e / 4096] and the bytes behind it (gz_crc_ends); a member [a, e) then has
// crc = F(e) + x^(8 (e - a)) * F(a), which gz_crc_check compares with the trailer, as it does ISIZE.
constexpr unsigned kCrcBlock = 4096;

// blk[b] = crc32 of text[4096 b, min(4096 (b + 1), n)): one warp per block, 128 bytes per lane
__global__ void __launch_bounds__(256) gz_crc_blocks_kernel(const unsigned char* __restrict__ text, unsigned long long n,
                                                            unsigned* __restrict__ blk, CrcPowers pw) {
    const int lane = threadIdx.x & 31;
    const unsigned long long n_blocks = (n + kCrcBlock - 1) / kCrcBlock;
    for (unsigned long long b = blockIdx.x * 8ull + (threadIdx.x >> 5); b < n_blocks; b += gridDim.x * 8ull) {
        const unsigned long long base = b * kCrcBlock + lane * 128ull;
        unsigned len = base < n ? static_cast<unsigned>(n - base < 128 ? n - base : 128) : 0u;
        unsigned crc = len ? crc_bytes(text + base, len) : 0u;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {  // (crc, len) of lane L joins in front of lane L + d's
            const unsigned ocrc = __shfl_down_sync(0xFFFFFFFFu, crc, d);
            const unsigned olen = __shfl_down_sync(0xFFFFFFFFu, len, d);
            if ((lane & (2 * d - 1)) == 0) {
                crc = crc_join(pw, crc, ocrc, olen);
                len += olen;
            }
        }
        if (lane == 0) blk[b] = crc;
    }
}

// F[b] = crc32 of text[0, 4096 b) for b <= n_blocks (exclusive prefix; F[n_blocks] = the whole text).  One block.
__global__ void __launch_bounds__(1024) gz_crc_scan_kernel(const unsigned* __restrict__ blk, unsigned long long n,
                                                           unsigned* __restrict__ F, CrcPowers pw) {
    __shared__ unsigned s_crc[1024];
    __shared__ unsigned long long s_len[1024];
    const unsigned t = threadIdx.x;
    const unsigned long long n_blocks = (n + kCrcBlock - 1) / kCrcBlock;
    const unsigned long long per = (n_blocks + 1023) / 1024;
    const unsigned long long b0 = t * per, b1 = b0 + per < n_blocks ? b0 + per : n_blocks;
    const unsigned x4k = crc_xpow8(pw, kCrcBlock);
    auto block_len = [&](unsigned long long b) { return b + 1 < n_blocks ? kCrcBlock : n - b * kCrcBlock; };
    unsigned crc = 0;
    unsigned long long len = 0;
    for (unsigned long long b = b0; b < b1; ++b) {
        const unsigned long long l = block_len(b);
        crc = (l == kCrcBlock ? crc_mul(x4k, crc) : crc_mul(crc_xpow8(pw, l), crc)) ^ blk[b];
        len += l;
    }
    s_crc[t] = crc, s_len[t] = len;
    __syncthreads();
    for (unsigned d = 1; d < 1024; d <<= 1) {  // inclusive scan of (crc, len) under the join
        unsigned c2 = 0;
        unsigned long long l2 = 0;
        if (t >= d) c2 = s_crc[t - d], l2 = s_len[t - d];
        __syncthreads();
        if (t >= d) {
            s_crc[t] = crc_join(pw, c2, s_crc[t], s_len[t]);
            s_len[t] += l2;
        }
        __syncthreads();
    }
    unsigned run = t ? s_crc[t - 1] : 0u;  // everything in front of this thread's blocks
    for (unsigned long long b = b0; b < b1; ++b) {
        F[b] = run;
        const unsigned long long l = block_len(b);
        run = (l == kCrcBlock ? crc_mul(x4k, run) : crc_mul(crc_xpow8(pw, l), run)) ^ blk[b];
    }
    if (b0 < n_blocks && b1 == n_blocks) F[n_blocks] = run;
    if (n_blocks == 0 && t == 0) F[0] = 0u;
}

// end[i] = absolute end of trailer i in the piece's text (chunk offset + local end)
__global__ void gz_trailer_ends_kernel(const Trailer* __restrict__ tr, unsigned n_tr, const Chunk* __restrict__ chunks,
                                       unsigned long long* __restrict__ end, unsigned* __restrict__ idx) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_tr) return;
    end[i] = chunks[tr[i].chunk].out_off + tr[i].local_end;
    idx[i] = i;
}

// Fe[i] = crc32 of text[0, end[i]) for the trailers in text order
__global__ void __launch_bounds__(128) gz_crc_ends_kernel(const unsigned char* __restrict__ text,
                                                          const unsigned long long* __restrict__ end, unsigned n_tr,
                                                          const unsigned* __restrict__ F, unsigned* __restrict__ Fe, CrcPowers pw) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_tr) return;
    const unsigned long long e = end[i], b = e / kCrcBlock;
    const unsigned rest = static_cast<unsigned>(e - b * kCrcBlock);
    Fe[i] = rest ? crc_join(pw, F[b], crc_bytes(text + b * kCrcBlock, rest), rest) : F[b];
}

// Every member that ends in this piece against its trailer.  carry_crc / carry_len: the part of the first member
// that earlier pieces produced.  result[0] = members that disagree, result[1] / result[2..3] = crc / length of the
// open member behind the last trailer (the next piece's carry).
__global__ void __launch_bounds__(128) gz_crc_check_kernel(const Trailer* __restrict__ tr, const unsigned* __restrict__ idx,
                                                           const unsigned long long* __restrict__ end,
                                                           const unsigned* __restrict__ Fe, unsigned n_tr,
                                                           const unsigned* __restrict__ F, unsigned long long n,
                                                           unsigned carry_crc, unsigned long long carry_len,
                                                           unsigned* __restrict__ result, CrcPowers pw) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long n_blocks = (n + kCrcBlock - 1) / kCrcBlock;
    if (i < n_tr) {
        const Trailer t = tr[idx[i]];
        const unsigned long long a = i ? end[i - 1] : 0ull, e = end[i];
        unsigned crc = Fe[i] ^ (i ? crc_mul(crc_xpow8(pw, e - a), Fe[i - 1]) : 0u);  // crc32 of text[a, e)
        unsigned long long len = e - a;
        if (i == 0) {
            crc = crc_join(pw, carry_crc, crc, len);
            len += carry_len;
        }
        if (crc != t.crc || static_cast<unsigned>(len) != t.isize) atomicAdd(&result[0], 1u);
    }
    if (i == 0) {  // what is open behind the last trailer
        const unsigned long long a = n_tr ? end[n_tr - 1] : 0ull;
        unsigned crc = F[n_blocks] ^ (n_tr ? crc_mul(crc_xpow8(pw, n - a), Fe[n_tr - 1]) : 0u);
        unsigned long long len = n - a;
        if (!n_tr) {
            crc = crc_join(pw, carry_crc, crc, len);
            len += carry_len;
        }
        result[1] = crc;
        result[2] = static_cast<unsigned>(len), result[3] = static_cast<unsigned>(len >> 32);
    }
}

}  // namespace gz
}  // namespace frb
