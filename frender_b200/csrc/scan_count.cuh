// Shared by the two scan kernels (scan_spec_kernel.cuh: tally of whole files; scan_ws_kernel.cuh: per-read outputs,
// -s, instrumentation): tile geometry and the counter warps' work on one tile.
//
// A counter thread owns 15 segments of 16 bytes (240 contiguous bytes).  The odd segment count is what makes the
// shared-memory loads conflict-free with compile-time register indices: lane l reads segment j at bank group
// (15 l + j) mod 8 = (j - l) mod 8, so the eight lanes of a 128-bit load phase hit eight different bank groups.
// (Round 1 used 16 segments and rotated the segment order per lane at run time, which cost 36 instructions per
// segment for the dynamic placement of each 16-bit mask against 19 here.)
#pragma once
#include "scan_common.cuh"

namespace frb {

constexpr int kWsGroup = 128;                 // counter threads
constexpr unsigned kNoTile = 0xFFFFFFFFu;
constexpr unsigned kNoGuess = 0xFFu;

// Tile geometry.  SEG = 16-byte segments per counter thread (odd: see above), PW = extractor warps,
// CTAS = resident CTAs per SM the shared memory and registers are budgeted for.
template <int SEG, int PW, int CTAS, int NLCAP, int STAGES, int RC = 56, int RW = 104>
struct WsGeom {
    static_assert(SEG % 2 == 1, "an odd segment count keeps the 128-bit shared loads conflict-free");
    static constexpr int stages = STAGES;
    static constexpr int seg = SEG;
    static constexpr int per_thread = SEG * 16;
    static constexpr int words = (per_thread + 31) / 32;     // 32-byte mask words per thread
    static constexpr int tile = kWsGroup * per_thread;
    static constexpr int buf = tile + kHalo;
    static constexpr int nl_cap = NLCAP;
    static constexpr int xwarps = PW;                        // extractor warps
    static constexpr int xgroup = PW * 32;
    static constexpr int threads = kWsGroup + xgroup + 32;  // + the committer warp
    static constexpr int ctas = CTAS;
    // per-thread register budget that keeps CTAS resident (registers are allocated per 4 warps)
    static constexpr int maxreg = (65536 / (CTAS * ((threads + 127) / 128 * 128))) / 8 * 8;
    // With 3 CTAs per SM the launch budget (80) is re-split inside the CTA: the counter warpgroup gives
    // registers back (setmaxnreg.dec) and the extractor/committer warpgroup takes them (setmaxnreg.inc).
    static constexpr bool split_regs = CTAS == 3 && threads == 256;
    static constexpr int regs_count = RC, regs_work = RW;  // their mean is the launch budget (80)
    static constexpr int smem = STAGES * buf + STAGES * nl_cap * (int)sizeof(uint16_t);
    static constexpr bool wide = false;  // keys of up to 21 symbols in one word
};
using WsTile = WsGeom<15, 3, 3, 1280, 2>;  // 30 KiB tiles, two stages, 3 CTAs per SM
// The same geometry for a wide context: keys of up to 42 symbols as (lo, hi), WideSlot table.
struct WsTileWide : WsTile {
    static constexpr bool wide = true;
};

// status[1 + t] of the speculative path: newlines of the tile (bits 0-19), unterminated last line (bit 20),
// guessed list index of the first header end (bits 24-31, kNoGuess = none)
__host__ __device__ __forceinline__ unsigned long long spec_info(unsigned total, unsigned vnl, unsigned guess) {
    return static_cast<unsigned long long>(total) | (static_cast<unsigned long long>(vnl) << 20) |
           (static_cast<unsigned long long>(guess) << 24);
}

// (1 << (f & 31)) - 1 in one instruction (BMSK)
__device__ __forceinline__ unsigned bits_below(unsigned f) {
    unsigned m;
    asm("bmsk.wrap.b32 %0, 0, %1;" : "=r"(m) : "r"(f));
    return m;
}

template <int N>
__device__ __forceinline__ void group_sync(int id) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(N) : "memory");
}


// What the counters know about a tile when they hand it on.
struct TileMeta {
    unsigned total;  // newlines in the tile
    unsigned vnl;    // 1 if the chunk ends in this tile without a final '\n' (that last line still is a line, F:169)
    unsigned halo;   // buffer position where the line that straddles the tile start begins (kUnknown: further back)
    unsigned guess;  // list index of the first header-line end as the text suggests it, or kNoGuess
};

// The counter warps' work on one staged tile (all 128 counter threads call it): bytes past the bulk copy's last
// 16-byte multiple, newline mask of the thread's 15 segments, scan over the group, ordered list of newline
// positions in `nl`, start of the straddling line, guess of the line phase.  kPublish: the tile's newline count
// goes to status[t] the moment it is known (the general kernel's look-back waits for it).  The returned values
// are complete in warp 0.
template <class G, bool kPublish>
__device__ __forceinline__ TileMeta count_tile(const ScanArgs& a, unsigned char* buf, uint16_t* nl, unsigned* s_cwarp,
                                               unsigned t, bool may_guess, volatile unsigned long long* status,
                                               int ct = threadIdx.x) {  // ct: index among the 128 counter threads
    constexpr int kWsTile = G::tile, kWsNlCap = G::nl_cap, kWsPerThread = G::per_thread;
    const int lane = ct & 31, warp = ct >> 5;
    const unsigned long long tile_off = static_cast<unsigned long long>(t) * kWsTile;
    const unsigned long long left = a.nbytes - tile_off;
    const unsigned valid = static_cast<unsigned>(left < kWsTile ? left : kWsTile);
    {   // bytes past the last 16-byte multiple of the bulk copy (final tile only)
        const unsigned halo = t ? kHalo : 0;
        const unsigned avail = valid + halo, bulk = avail & ~15u;
        if (avail != bulk) {
            if (ct < static_cast<int>(avail - bulk))
                buf[(kHalo - halo) + bulk + ct] = a.data[tile_off - halo + bulk + ct];
            group_sync<kWsGroup>(1);
        }
    }
    // Newline mask of this thread's bytes as 32-byte words, MIRRORED: byte k of word q (thread byte
    // 32q + k) sits at bit 31 - k, so the first newline of a word is its highest set bit.
    constexpr int kWords = G::words;
    unsigned w[kWords];
    const uint4* t4 = reinterpret_cast<const uint4*>(buf + kHalo) + ct * G::seg;
#pragma unroll
    for (int q = 0; q < kWords; ++q) {
        if (2 * q + 1 < G::seg) w[q] = eq_mask32_rev(t4[2 * q], t4[2 * q + 1], a.pat_nl);
        else w[q] = eq_mask16_rev_hi(t4[2 * q], a.pat_nl);
    }
    // bytes in front of a.skip (a carried tail was put in front of an aligned buffer) are not text
    const long long sk = static_cast<long long>(a.skip) - static_cast<long long>(tile_off);
    if (sk > 0) {
        const long long ns = sk - static_cast<long long>(ct) * kWsPerThread;  // bytes of this thread to ignore
        if (ns > 0) {
#pragma unroll
            for (int q = 0; q < kWords; ++q) {
                const long long n = ns - 32 * q;  // leading bytes of word q to ignore = its top n bits
                w[q] = n <= 0 ? w[q] : (n >= 32 ? 0u : (w[q] & (0xFFFFFFFFu >> n)));
            }
        }
    }
    {
        const int nv = static_cast<int>(valid) - ct * kWsPerThread;
        if (nv < kWsPerThread) {
#pragma unroll
            for (int q = 0; q < kWords; ++q) {
                const int n = nv - 32 * q;  // bytes of word q that exist: keep the top n bits
                w[q] = n <= 0 ? 0u : (n >= 32 ? w[q] : (w[q] & ~(0xFFFFFFFFu >> n)));
            }
        }
    }
    unsigned cnt = 0;
#pragma unroll
    for (int q = 0; q < kWords; ++q) cnt += __popc(w[q]);
    unsigned incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned n = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += n;
    }
    if (lane == 31) s_cwarp[warp] = incl;
    group_sync<kWsGroup>(1);
    unsigned wbase = 0, total = 0;
#pragma unroll
    for (int k = 0; k < kWsGroup / 32; ++k) {
        const unsigned v = s_cwarp[k];
        if (k < warp) wbase += v;
        total += v;
    }
    // Thread 32: not the thread that arrives on the mbarrier afterwards
    if (kPublish && ct == 32) status[t] = (t == 0 ? kFlagInc : kFlagAgg) | total;
    // a last line without '\n' still is a line (F:161 iterates it; F:169 rstrip)
    const unsigned vnl = (t == a.n_tiles - 1 && valid > 0 && sk < static_cast<long long>(valid) && buf[kHalo + valid - 1] != '\n') ? 1u : 0u;
    {   // ordered list of newline positions; which of them end header lines is decided later
        unsigned idx = wbase + incl - cnt;
        unsigned pos0 = kHalo + ct * kWsPerThread;
        // A list that does not fit is never read (the tile goes to scan_redo_kernel), so one range check per
        // thread is enough.  Straight-line code for the first two newlines of a 32-byte word -- a third one
        // means lines shorter than 16 bytes -- keeps the warp out of a data-dependent loop.
        if (wbase + incl <= static_cast<unsigned>(kWsNlCap)) {
            auto store_if = [](uint16_t* p, unsigned value, unsigned cond) {  // predicated store, no branch
                asm volatile(
                    "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.shared.u16 [%0], %1;\n\t}"
                    ::"r"(smem_addr(p)), "h"(static_cast<unsigned short>(value)), "r"(cond)
                    : "memory");
            };
#pragma unroll
            for (int q = 0; q < kWords; ++q) {
                // f = index of the highest set bit = 31 - byte offset of the first newline left
                const unsigned m = w[q];
                const unsigned f1 = 31 - __clz(m);              // FLO; 0xFFFFFFFF when m == 0
                store_if(nl + idx, pos0 + 31 - f1, m);
                unsigned m2 = m & bits_below(f1);               // m == 0 stays 0
                const unsigned f2 = 31 - __clz(m2);
                store_if(nl + idx + 1, pos0 + 31 - f2, m2);
                m2 &= bits_below(f2);
                if (m2) {
                    unsigned k = idx + 2;
                    do {
                        const unsigned f = 31 - __clz(m2);
                        nl[k++] = static_cast<uint16_t>(pos0 + 31 - f);
                        m2 &= ~(1u << f);
                    } while (m2);
                }
                idx += __popc(m);
                pos0 += 32;
            }
        }
        if (ct == 0 && vnl && total < static_cast<unsigned>(kWsNlCap)) nl[total] = static_cast<uint16_t>(kHalo + valid);
    }
    // start of the line that straddles the tile start: behind the last newline of the halo -- or at a.skip, where
    // the text begins (in this tile: sk >= 0; inside the halo: -kHalo < sk < 0)
    unsigned halo_start = kHalo + static_cast<unsigned>(sk > 0 ? sk : 0);
    if (warp == 0 && t != 0 && sk < 0) {
        unsigned m = newline_mask16(reinterpret_cast<const uint4*>(buf)[lane], a.pat_nl);
        const long long text0 = kHalo + sk;  // buffer position of a.skip (<= 0: the whole halo is text)
        if (text0 > 0) {
            const long long cut = text0 - lane * 16;  // leading bytes of this lane's segment in front of the text
            m = cut >= 16 ? 0u : (cut > 0 ? (m & (0xFFFFu << cut)) : m);
        }
        const unsigned any = __ballot_sync(0xFFFFFFFFu, m != 0);
        const int top = 31 - __clz(any);  // -1: no newline in the halo
        const unsigned mine = lane * 16 + (31 - __clz(m)) + 1;
        halo_start = any ? __shfl_sync(0xFFFFFFFFu, mine, top & 31) : (text0 > 0 ? static_cast<unsigned>(text0) : kUnknown);
    }
    group_sync<kWsGroup>(1);  // list complete (also protects s_cwarp)
    unsigned g = kNoGuess;
    if (warp == 0) {
        // Which list entries end header lines?  The reference goes by line COUNT (F:161); in well-formed FASTQ
        // the answer shows in the tile itself: a line that starts with '@' whose second successor starts with
        // '+' and fourth with '@' is a header line, and exactly one of the first four lines may fit.  The keys
        // are extracted on this guess; it is always checked against the count before a result stands.
        if (may_guess && total >= 9 && halo_start != kUnknown && total + vnl <= static_cast<unsigned>(kWsNlCap)) {
            const unsigned c = lane & 7;  // lane c < 8 looks at the first byte of the tile's line c
            const unsigned first = buf[c ? nl[c - 1] + 1u : halo_start];
            const unsigned at = __ballot_sync(0xFFFFFFFFu, first == '@') & 0xFFu;
            const unsigned plus = __ballot_sync(0xFFFFFFFFu, first == '+') & 0xFFu;
            const unsigned hits = at & (plus >> 2) & (at >> 4) & 0xFu;
            if (__popc(hits) == 1) g = __ffs(hits) - 1;
        }
    }
    return TileMeta{total, vnl, halo_start, g};
}

}  // namespace frb
