// Hot path A, shared pieces: arguments, mbarrier / bulk-copy PTX helpers, byte-compare primitives, the
// two key rules (reference frender.py:169 for scan, F:778 for demux) and the decoupled look-back over
// per-tile newline counts.  The kernel itself is scan_ws_kernel.cuh.
#pragma once
#include "common.cuh"

namespace frb {

constexpr int kHalo = 512;           // bytes staged in front of every tile (start of the straddling line)
constexpr unsigned kUnknown = 0xFFFFu;
constexpr int kRuleOffsetsOnly = 2;  // internal: no key, record offsets only
constexpr int kRuleRuntime = -1;     // parse_header<>: take the rule from ScanArgs

#define kFlagAgg (1ULL << 62)
#define kFlagInc (2ULL << 62)
#define kValMask ((1ULL << 62) - 1)

struct ScanArgs {
    const unsigned char* data;      // chunk, 16-byte aligned, begins at a line start
    unsigned long long nbytes;
    unsigned long long line_base;   // lines of the file before this chunk (ignored if use_carry)
    unsigned long long read_limit;  // reads with ordinal >= limit are not tallied (-s, F:163-165)
    unsigned long long pos_base;    // added to the read ordinal to form `first`
    Slot* table;
    unsigned long long table_mask;
    unsigned long long* status;     // [0] tile counter, [1 + t] look-back word of tile t
    DevState* st;
    unsigned long long* keys_out;     // optional: key of read r at [r - first read of chunk]
    unsigned long long* rec_off_out;  // optional: chunk offset of the record start, same index
    unsigned long long out_cap;       // entries available in keys_out / rec_off_out
    unsigned int n_tiles;
    int use_carry;
    int rule;
    unsigned long long* timing;  // optional: per-role clock64 sums (instrumented instantiation only)
    unsigned long long* tile_first;  // speculative path: first read ordinal of every tile of the file
    unsigned long long tile_base;  // speculative path: tiles of this file before the chunk (composite positions)
    const unsigned long long* skip_ptr;  // device value: bytes at the start of `data` that are not text (the
                                         // demux stream keeps `data` aligned and puts a carried tail in front)
    unsigned long long skip;     // ... its value inside the kernels (filled in by them)
    int negate;                  // speculative path: take the chunk's guessed keys out of the table again
    int composite;               // scan_redo_kernel: record composite positions, leave n_reads / line_carry alone
    unsigned int* redo;          // tiles left to scan_redo_kernel, capacity n_tiles
    unsigned int tile_bytes;     // tile size of the kernel that filled status[] (for scan_redo_kernel)
    int no_guess;                // A-B: never guess the line phase from the text
    // '\n' and ' ' replicated over a word.  Kernel parameters, not literals: with the pattern in a register the
    // byte compare is three instructions per word (LOP3 takes one immediate; as a literal next to the 0x7f..
    // mask the pattern costs a fourth).
    unsigned int pat_nl, pat_sp;
};

// ---- PTX helpers: mbarrier + TMA bulk copy ------------------------------------------------
__device__ __forceinline__ unsigned smem_addr(const void* p) {
    return static_cast<unsigned>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
// Arrival without release semantics, issued only once `dep` is available.  A releasing arrival waits for the
// arriving thread's outstanding global loads and atomics; the extractors always have some in flight (table
// updates), and what the arrival has to order -- their shared-memory loads of the tile stage against the bulk
// copy that refills it -- is ordered by the register dependency: `dep` is computed from the loaded values, so
// the loads have returned when the arrival issues.
__device__ __forceinline__ void mbar_arrive_relaxed_after(unsigned long long* bar, unsigned dep) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0x9E3779B9;\n\t"
        "@p mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];\n\t"
        "@!p mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];\n\t}"
        ::"r"(smem_addr(bar)), "r"(dep)
        : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    // whole spin loop in one asm block (the form ptxas knows), then an explicit warp reconvergence:
    // lanes leave the loop at different times and the warp-collective code that follows
    // (shuffles, ballots) must not run on a partial warp.
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "FRB_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra FRB_DONE_%=;\n\t"
        "bra FRB_WAIT_%=;\n\t"
        "FRB_DONE_%=:\n\t}"
        ::"r"(smem_addr(bar)), "r"(parity)
        : "memory");
    // not __syncwarp(): nvcc sees straight-line code here and drops it
    asm volatile("bar.warp.sync 0xffffffff;" ::: "memory");
}
// non-blocking probe: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(unsigned long long* bar, unsigned parity) {
    unsigned done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_addr(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
// single-thread wait (no warp reconvergence: the caller is one elected lane)
__device__ __forceinline__ void mbar_wait_one(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "FRB_WAIT1_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra FRB_DONE1_%=;\n\t"
        "bra FRB_WAIT1_%=;\n\t"
        "FRB_DONE1_%=:\n\t}"
        ::"r"(smem_addr(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}

#define kFoldLsb3 0x1249249249249249ULL  // bit 0 of every 3-bit group

// ---- byte-compare primitives ---------------------------------------------------------------
// bit 7 of every byte of w that equals the byte replicated in `pat` (pattern bytes < 0x80); exact (no borrow
// leaks).  (w & 0x7f..) ^ pat is the low seven bits of w ^ pat, and bit 7 of w ^ pat is bit 7 of w.
__device__ __forceinline__ unsigned eq_flags(unsigned w, unsigned pat) {
    const unsigned t = ((w & 0x7F7F7F7Fu) ^ pat) + 0x7F7F7F7Fu;
    return ~(t | w) & 0x80808080u;
}
// 16-bit mask (bit i = byte i) of the bytes of v equal to the byte replicated in `pat`.
// The flags (0x80 per equal byte) are gathered with byte dot products: weights 1,2,4,8 for the first word
// of a pair and 16,32,64,128 for the second give mask8 * 128, on the multiply pipe instead of the ALU.
__device__ __forceinline__ unsigned eq_mask16(const uint4 v, unsigned pat) {
    unsigned lo = __dp4a(eq_flags(v.x, pat), 0x08040201u, 0u);
    lo = __dp4a(eq_flags(v.y, pat), 0x80402010u, lo);
    unsigned hi = __dp4a(eq_flags(v.z, pat), 0x08040201u, 0u);
    hi = __dp4a(eq_flags(v.w, pat), 0x80402010u, hi);
    return (lo >> 7) | (hi << 1);
}
__device__ __forceinline__ unsigned newline_mask16(const uint4 v, unsigned pat_nl) { return eq_mask16(v, pat_nl); }
// Mirrored mask of 32 bytes (v0 = bytes 0-15, v1 = bytes 16-31): byte k -> bit 31 - k.  With a thread's mask
// words mirrored, the first newline of a word is its highest set bit, which FLO finds in one instruction
// (find-first-set is a bit reverse + FLO).  The four byte-dot-product chains each deliver eight flags at bits
// 7-14; the fields do not overlap once shifted, so they are joined with shift-adds (LEA).
__device__ __forceinline__ unsigned eq_mask32_rev(const uint4 v0, const uint4 v1, unsigned pat) {
    unsigned a = __dp4a(eq_flags(v0.x, pat), 0x10204080u, 0u);
    a = __dp4a(eq_flags(v0.y, pat), 0x01020408u, a);   // bytes 0-7:   byte k at bit 14 - k
    unsigned b = __dp4a(eq_flags(v0.z, pat), 0x10204080u, 0u);
    b = __dp4a(eq_flags(v0.w, pat), 0x01020408u, b);   // bytes 8-15
    unsigned c = __dp4a(eq_flags(v1.x, pat), 0x10204080u, 0u);
    c = __dp4a(eq_flags(v1.y, pat), 0x01020408u, c);   // bytes 16-23
    unsigned d = __dp4a(eq_flags(v1.z, pat), 0x10204080u, 0u);
    d = __dp4a(eq_flags(v1.w, pat), 0x01020408u, d);   // bytes 24-31
    return (a << 17) + ((b << 9) + ((c << 1) + (d >> 7)));
}
__device__ __forceinline__ unsigned eq_mask16_rev_hi(const uint4 v0, unsigned pat) {  // bytes 0-15 only
    unsigned a = __dp4a(eq_flags(v0.x, pat), 0x10204080u, 0u);
    a = __dp4a(eq_flags(v0.y, pat), 0x01020408u, a);
    unsigned b = __dp4a(eq_flags(v0.z, pat), 0x10204080u, 0u);
    b = __dp4a(eq_flags(v0.w, pat), 0x01020408u, b);
    return (a << 17) + (b << 9);
}

// Number of ' ' in buf[sb, eb) for lines that end within 112 bytes of their 16-byte-aligned start,
// else -1.  Fully unrolled and branch-free: seven independent 16-byte shared loads in flight.
__device__ __forceinline__ int count_spaces_fast(const unsigned char* buf, unsigned sb, unsigned eb, unsigned pat_sp) {
    const unsigned a0 = sb & ~15u;
    if (eb - a0 > 112u) return -1;
    unsigned cnt = 0;
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        const unsigned p = a0 + 16u * i;
        if (i >= 4 && p >= eb) break;  // ordinary header lines span 5 segments; the loads stay batched
        const uint4 v = *reinterpret_cast<const uint4*>(buf + (p < eb ? p : a0));
        unsigned m = eq_mask16(v, pat_sp);
        const unsigned lo_cut = sb > p ? sb - p : 0u;                  // bytes of this segment before the line
        const unsigned hi_cut = eb > p ? (eb - p < 16u ? eb - p : 16u) : 0u;  // bytes of it inside [.., eb)
        m &= (0xFFFFu << lo_cut) & ((1u << hi_cut) - 1u);
        cnt += __popc(m);
    }
    return static_cast<int>(cnt);
}

// Same result as count_spaces_fast with fewer instructions: every 16-byte segment the line touches is
// counted whole with byte dot products (flag word . 0x01010101, four instructions per word, no positional
// mask), then the bytes of the first segment in front of the line and of the last segment behind it are
// taken off again with two positional masks.
__device__ __forceinline__ int count_spaces_sum(const unsigned char* buf, unsigned sb, unsigned eb, unsigned pat_sp) {
    const unsigned a0 = sb & ~15u;
    const unsigned span = eb - a0;  // >= 22 on the fast path
    if (span > 112u) return -1;
    const unsigned last = (span - 1u) >> 4;  // segment holding the last byte of the line, 1..6
    unsigned acc = 0;
    uint4 v0 = make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        if (i >= 5 && static_cast<unsigned>(i) > last) break;  // ordinary header lines span 5 or 6 segments
        const bool in = static_cast<unsigned>(i) <= last;
        const uint4 v = *reinterpret_cast<const uint4*>(buf + a0 + (in ? 16u * i : 0u));
        if (i == 0) v0 = v;
        const unsigned wt = in ? 0x01010101u : 0u;
        acc = __dp4a(eq_flags(v.x, pat_sp), wt, acc);
        acc = __dp4a(eq_flags(v.y, pat_sp), wt, acc);
        acc = __dp4a(eq_flags(v.z, pat_sp), wt, acc);
        acc = __dp4a(eq_flags(v.w, pat_sp), wt, acc);
    }
    const unsigned head = eq_mask16(v0, pat_sp) & ((1u << (sb - a0)) - 1u);
    const uint4 vl = *reinterpret_cast<const uint4*>(buf + a0 + 16u * last);
    const unsigned tail = eq_mask16(vl, pat_sp) >> (span - 16u * last);  // bytes at and behind eb (1..16)
    return static_cast<int>((acc >> 7) - __popc(head) - __popc(tail));
}

// shared-memory LUT entry of byte c for parse_header: bits 0-2 symbol code, bit 3 = c ends the key
// when walking back from the end of the line (':' always, ' ' under the scan rule).  Nothing above bit 3.
__device__ __forceinline__ unsigned char lut_entry(unsigned c, int rule) {
    const bool delim = (c == ':') || (rule == FRB_RULE_SCAN && c == ' ');
    return static_cast<unsigned char>(enc_read(c) | (delim ? 0x08u : 0u));
}

// Exact, byte-serial statement of both key rules over one header line (no trailing newline).
// Used for the rare lines the fast path declines (second space, key > 21, line not in smem).
__host__ __device__ inline int parse_serial(const unsigned char* s, unsigned long long len, int rule,
                                            unsigned long long* key_out) {
    unsigned long long i = 0;
    if (rule == FRB_RULE_SCAN) {
        while (i < len && s[i] != ' ') ++i;
        if (i >= len) return FRB_ERR_BAD_HEADER;  // split(" ")[1] -> IndexError, F:169
        ++i;
    }
    unsigned long long k = 0;
    int n = 0;
    bool bad = false, too_long = false;
    for (; i < len; ++i) {
        unsigned c = s[i];
        if (rule == FRB_RULE_SCAN && c == ' ') break;
        if (c == ':') {
            k = 0, n = 0, bad = false, too_long = false;
            continue;
        }
        unsigned code = enc_read(c);
        bad |= (code == 0);
        if (n >= kMaxSyms) too_long = true;
        else k |= static_cast<unsigned long long>(code) << (3 * n);
        ++n;
    }
    if (bad) return FRB_ERR_BAD_ALPHABET;
    if (too_long) return FRB_ERR_KEY_TOO_LONG;
    *key_out = k;
    return 0;
}

// Key of the header line occupying buffer positions [sb, eb) (sb == kUnknown: starts before
// the staged bytes).  Buffer position p is chunk offset tile_off + p - kHalo.
// RULE: a compile-time rule, or kRuleRuntime to take a.rule; SUM: count spaces with count_spaces_sum.
template <int RULE = kRuleRuntime, bool SUM = false>
__device__ __forceinline__ int parse_header(const unsigned char* buf, const unsigned char* lut, unsigned sb,
                                            unsigned eb, const ScanArgs& a, unsigned long long tile_off,
                                            unsigned long long* key_out, unsigned long long* start_out) {
    const int rule = RULE == kRuleRuntime ? a.rule : RULE;
    const bool scan_rule = (rule == FRB_RULE_SCAN);
    if (rule == kRuleOffsetsOnly) {  // record boundaries only (R1 side of the demux router)
        if (sb != kUnknown) {
            *start_out = tile_off + sb - kHalo;
        } else {
            unsigned long long s_g = tile_off + eb - kHalo;
            while (s_g > a.skip && a.data[s_g - 1] != '\n') --s_g;
            *start_out = s_g;
        }
        *key_out = 0;
        return 0;
    }
    if (sb != kUnknown) *start_out = tile_off + sb - kHalo;
    if (sb != kUnknown && eb - sb > static_cast<unsigned>(kMaxSyms)) {
        // Fast path, branch-free and latency-flat.  With exactly one ' ' in the line the key is the
        // text after the last ':' or ' ' (the 2nd space token runs to the end of the line).  The line
        // has at least 22 bytes, so the 22 bytes before its end all belong to it.
        const int spaces = !scan_rule ? 1 : SUM ? count_spaces_sum(buf, sb, eb, a.pat_sp)
                                               : count_spaces_fast(buf, sb, eb, a.pat_sp);
        const unsigned char* const e = buf + eb;
        unsigned delim = 0, lo = 0, hi = 0, top = 0;
#pragma unroll
        for (int j = 0; j < kMaxSyms + 1; ++j) {  // closest to the end of the line first
            const unsigned v = lut[e[-1 - j]];
            const unsigned code = v & 7u;
            delim += (v >> 3) << j;
            if (j < 10) lo += code << (3 * j);
            else if (j < 20) hi += code << (3 * (j - 10));
            else if (j == 20) top = code;
        }
        if (spaces == 0) return FRB_ERR_BAD_HEADER;
        if (spaces == 1 && delim != 0) {
            const int len = __ffs(delim) - 1;  // symbols in the key, <= 21
            // krev holds the key backwards (symbol j = j-th char from the end)
            const unsigned long long krev = static_cast<unsigned long long>(lo) |
                                            (static_cast<unsigned long long>(hi) << 30) |
                                            (static_cast<unsigned long long>(top) << 60);
            // every one of the len symbols must have a non-zero code
            const unsigned long long want = len ? (kFoldLsb3 & ((1ULL << (3 * len)) - 1ULL)) : 0ULL;
            if (((krev | (krev >> 1) | (krev >> 2)) & want) != want) return FRB_ERR_BAD_ALPHABET;
            // reverse the order of the 3-bit groups: bit-reverse the word, then put the bits of every
            // group back in order
            const unsigned long long r = __brevll(krev) >> 1;  // group j now at group index 20 - j, bits mirrored
            const unsigned long long g = ((r & kFoldLsb3) << 2) | (r & (kFoldLsb3 << 1)) | ((r >> 2) & kFoldLsb3);
            *key_out = len ? (g >> (3 * (kMaxSyms - len))) : 0ULL;
            return 0;
        }
    }
    const unsigned long long e_g = tile_off + eb - kHalo;
    unsigned long long s_g;
    if (sb != kUnknown) {
        s_g = tile_off + sb - kHalo;
    } else {
        s_g = e_g;
        while (s_g > a.skip && a.data[s_g - 1] != '\n') --s_g;
    }
    *start_out = s_g;
    return parse_serial(a.data + s_g, e_g - s_g, rule, key_out);
}

// ---- wide keys (up to 42 symbols: lo = symbols 0..20, hi = symbols 21..41) ---------------------------------------
// parse_serial for a wide context.
__host__ __device__ inline int parse_serial_wide(const unsigned char* s, unsigned long long len, int rule,
                                                 unsigned long long* lo_out, unsigned long long* hi_out) {
    unsigned long long i = 0;
    if (rule == FRB_RULE_SCAN) {
        while (i < len && s[i] != ' ') ++i;
        if (i >= len) return FRB_ERR_BAD_HEADER;
        ++i;
    }
    unsigned long long k0 = 0, k1 = 0;
    int n = 0;
    bool bad = false, too_long = false;
    for (; i < len; ++i) {
        unsigned c = s[i];
        if (rule == FRB_RULE_SCAN && c == ' ') break;
        if (c == ':') {
            k0 = k1 = 0, n = 0, bad = false, too_long = false;
            continue;
        }
        unsigned code = enc_read(c);
        bad |= (code == 0);
        if (n >= kMaxWideSyms) too_long = true;
        else if (n < kMaxSyms) k0 |= static_cast<unsigned long long>(code) << (3 * n);
        else k1 |= static_cast<unsigned long long>(code) << (3 * (n - kMaxSyms));
        ++n;
    }
    if (bad) return FRB_ERR_BAD_ALPHABET;
    if (too_long) return FRB_ERR_KEY_TOO_LONG;
    *lo_out = k0, *hi_out = k1;
    return 0;
}

// The order of the 21 3-bit groups of a word reversed (group j -> group 20 - j).
__device__ __forceinline__ unsigned long long reverse21(unsigned long long w) {
    const unsigned long long r = __brevll(w) >> 1;
    return ((r & kFoldLsb3) << 2) | (r & (kFoldLsb3 << 1)) | ((r >> 2) & kFoldLsb3);
}

// parse_header for a wide context.  The fast path walks back over the last 43 bytes of the line.
template <bool SUM = false>
__device__ __forceinline__ int parse_header_wide(const unsigned char* buf, const unsigned char* lut, unsigned sb,
                                                 unsigned eb, const ScanArgs& a, unsigned long long tile_off,
                                                 unsigned long long* lo_out, unsigned long long* hi_out,
                                                 unsigned long long* start_out) {
    const bool scan_rule = (a.rule == FRB_RULE_SCAN);
    if (sb != kUnknown) *start_out = tile_off + sb - kHalo;
    if (sb != kUnknown && eb - sb > static_cast<unsigned>(kMaxWideSyms)) {
        const int spaces = !scan_rule ? 1 : SUM ? count_spaces_sum(buf, sb, eb, a.pat_sp)
                                               : count_spaces_fast(buf, sb, eb, a.pat_sp);
        const unsigned char* const e = buf + eb;
        unsigned long long delim = 0, r0 = 0, r1 = 0;  // r0 / r1: symbols 0..20 / 21..41 counted from the end
#pragma unroll
        for (int j = 0; j < kMaxWideSyms + 1; ++j) {
            const unsigned v = lut[e[-1 - j]];
            delim |= static_cast<unsigned long long>(v >> 3) << j;
            if (j < kMaxSyms) r0 |= static_cast<unsigned long long>(v & 7u) << (3 * j);
            else if (j < kMaxWideSyms) r1 |= static_cast<unsigned long long>(v & 7u) << (3 * (j - kMaxSyms));
        }
        if (spaces == 0) return FRB_ERR_BAD_HEADER;
        if (spaces == 1 && delim != 0) {
            const int len = __ffsll(static_cast<long long>(delim)) - 1;  // symbols in the key, <= 42
            const unsigned long long want0 = len >= kMaxSyms ? kFoldLsb3 : (len ? (kFoldLsb3 & ((1ULL << (3 * len)) - 1ULL)) : 0ULL);
            const unsigned long long want1 = len > kMaxSyms ? (kFoldLsb3 & ((1ULL << (3 * (len - kMaxSyms))) - 1ULL)) : 0ULL;
            if (((r0 | (r0 >> 1) | (r0 >> 2)) & want0) != want0 || ((r1 | (r1 >> 1) | (r1 >> 2)) & want1) != want1)
                return FRB_ERR_BAD_ALPHABET;
            // the 42 symbols in text order, then shifted down by the 42 - len that are not part of the key
            const unsigned long long f0 = reverse21(r1), f1 = reverse21(r0);
            const int s = kMaxWideSyms - len;
            if (s >= kMaxSyms) {
                *lo_out = f1 >> (3 * (s - kMaxSyms)), *hi_out = 0;
            } else {
                *lo_out = s ? ((f0 >> (3 * s)) | (f1 << (3 * (kMaxSyms - s)))) & ((1ULL << 63) - 1ULL) : f0;
                *hi_out = f1 >> (3 * s);
            }
            return 0;
        }
    }
    const unsigned long long e_g = tile_off + eb - kHalo;
    unsigned long long s_g;
    if (sb != kUnknown) {
        s_g = tile_off + sb - kHalo;
    } else {
        s_g = e_g;
        while (s_g > a.skip && a.data[s_g - 1] != '\n') --s_g;
    }
    *start_out = s_g;
    return parse_serial_wide(a.data + s_g, e_g - s_g, a.rule, lo_out, hi_out);
}

// ---- header parsing in two halves (speculative path) ------------------------------------------------------------
// The tile buffer is wanted back as early as possible (its refill is a long-latency bulk copy), so an extractor
// thread first LOADS what its header line needs -- the up to seven 16-byte segments the line touches (space
// count) into registers, the three segments in front of the line end (the key is in the last 22 bytes) into a
// private shared-memory scratch -- the stage is released, and the arithmetic runs afterwards.
struct HeaderRegs {
    uint4 v[7];       // segments a0 + 16 i of the line, a0 = sb & ~15
    unsigned sb, eb;  // buffer positions of the line start and of its '\n'
    bool fast;        // >= 22 bytes, starts inside the staged bytes, ends within 112 bytes of a0
};

__device__ __forceinline__ unsigned header_load(const unsigned char* buf, unsigned sb, unsigned eb, bool have, bool need5,
                                                bool need6, HeaderRegs& r, uint4* scratch) {
    r.sb = sb, r.eb = eb;
    r.fast = have && sb != kUnknown && eb - sb > static_cast<unsigned>(kMaxSyms) && eb - (sb & ~15u) <= 112u;
    const unsigned a0 = r.fast ? (sb & ~15u) : 0u;
    const unsigned last = r.fast ? (eb - a0 - 1u) >> 4 : 0u;
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        if ((i == 5 && !need5) || (i == 6 && !need6)) {  // warp-uniform
            r.v[i] = make_uint4(0, 0, 0, 0);
            continue;
        }
        r.v[i] = *reinterpret_cast<const uint4*>(buf + a0 + (static_cast<unsigned>(i) <= last ? 16u * i : 0u));
    }
    const unsigned tb = r.fast ? ((eb - 1u) & ~15u) - 32u : 0u;  // >= kHalo - 32 + 16 for a line of >= 22 bytes
    unsigned dep = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const uint4 v = *reinterpret_cast<const uint4*>(buf + tb + 16u * k);
        scratch[k] = v;
        dep ^= v.x;
    }
    // one register of every load: when `dep` is available, every load of the stage has returned
#pragma unroll
    for (int i = 0; i < 7; ++i) dep ^= r.v[i].x;
    return dep;
}

// Key of a header staged by header_load (scan rule).  Lines the fast path declines go to parse_serial on the
// bytes in global memory, as in parse_header.
__device__ __forceinline__ int header_key(const HeaderRegs& r, const uint4* scratch, const unsigned char* lut,
                                          const ScanArgs& a, unsigned long long tile_off, bool need5, bool need6,
                                          unsigned long long* key_out) {
    if (r.fast) {
        const unsigned a0 = r.sb & ~15u, span = r.eb - a0, last = (span - 1u) >> 4;
        unsigned acc = 0;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            if ((i == 5 && !need5) || (i == 6 && !need6)) continue;
            const unsigned wt = static_cast<unsigned>(i) <= last ? 0x01010101u : 0u;
            acc = __dp4a(eq_flags(r.v[i].x, a.pat_sp), wt, acc);
            acc = __dp4a(eq_flags(r.v[i].y, a.pat_sp), wt, acc);
            acc = __dp4a(eq_flags(r.v[i].z, a.pat_sp), wt, acc);
            acc = __dp4a(eq_flags(r.v[i].w, a.pat_sp), wt, acc);
        }
        const unsigned head = eq_mask16(r.v[0], a.pat_sp) & ((1u << (r.sb - a0)) - 1u);
        const unsigned tail = eq_mask16(scratch[2], a.pat_sp) >> (span - 16u * last);  // scratch[2] = segment `last`
        const int spaces = static_cast<int>((acc >> 7) - __popc(head) - __popc(tail));
        const unsigned char* const e = reinterpret_cast<const unsigned char*>(scratch) + (((r.eb - 1u) & 15u) + 33u);
        unsigned delim = 0, lo = 0, hi = 0, top = 0;
#pragma unroll
        for (int j = 0; j < kMaxSyms + 1; ++j) {  // closest to the end of the line first
            const unsigned v = lut[e[-1 - j]];
            const unsigned code = v & 7u;
            delim += (v >> 3) << j;
            if (j < 10) lo += code << (3 * j);
            else if (j < 20) hi += code << (3 * (j - 10));
            else if (j == 20) top = code;
        }
        if (spaces == 0) return FRB_ERR_BAD_HEADER;
        if (spaces == 1 && delim != 0) {
            const int len = __ffs(delim) - 1;  // symbols in the key, <= 21
            const unsigned long long krev = static_cast<unsigned long long>(lo) |
                                            (static_cast<unsigned long long>(hi) << 30) |
                                            (static_cast<unsigned long long>(top) << 60);
            const unsigned long long want = len ? (kFoldLsb3 & ((1ULL << (3 * len)) - 1ULL)) : 0ULL;
            if (((krev | (krev >> 1) | (krev >> 2)) & want) != want) return FRB_ERR_BAD_ALPHABET;
            const unsigned long long rv = __brevll(krev) >> 1;
            const unsigned long long g = ((rv & kFoldLsb3) << 2) | (rv & (kFoldLsb3 << 1)) | ((rv >> 2) & kFoldLsb3);
            *key_out = len ? (g >> (3 * (kMaxSyms - len))) : 0ULL;
            return 0;
        }
    }
    const unsigned long long e_g = tile_off + r.eb - kHalo;
    unsigned long long s_g;
    if (r.sb != kUnknown) {
        s_g = tile_off + r.sb - kHalo;
    } else {
        s_g = e_g;
        while (s_g > a.skip && a.data[s_g - 1] != '\n') --s_g;
    }
    return parse_serial(a.data + s_g, e_g - s_g, FRB_RULE_SCAN, key_out);
}

// Decoupled look-back over per-tile newline counts.  The tile's own count was published by the
// count stage (one pipeline step earlier, see scan_kernel); returns the number of newlines before
// tile t and publishes the tile's inclusive prefix.  Called by one full warp.
// kBlocking = false: a single pass that gives up (returns false) as soon as a needed count is not
// published yet -- used to take the look-back off the critical path without ever stalling a CTA on
// another CTA's progress.
template <bool kBlocking>
__device__ __forceinline__ bool tile_prefix(volatile unsigned long long* status, unsigned t, unsigned total,
                                            int lane, unsigned long long* out) {
    // Windows of 128 predecessors per step (four independent loads per lane, one L2 round trip): with several
    // hundred tiles in flight the nearest inclusive word is usually more than 32 tiles back.  Measured effect
    // on the kernel: +0.7 %; what the look-back mostly waits for is predecessors that are not counted yet.
    constexpr int kSub = 4;
    *out = 0;
    if (t == 0) return true;  // published as inclusive by the count stage
    unsigned long long acc = 0;  // lane-local partial sum, reduced once at the end
    long long idx = static_cast<long long>(t) - 1;
    for (;;) {
        bool done = false;
        for (;;) {  // until every word this step needs has been published
            unsigned long long s[kSub];
#pragma unroll
            for (int m = 0; m < kSub; ++m) {
                const long long j = idx - 32 * m - lane;
                s[m] = (j >= 0) ? status[j] : kFlagInc;
            }
            unsigned long long part = 0;
            bool ready = true;
#pragma unroll
            for (int m = 0; m < kSub; ++m) {
                if (ready && !done) {
                    const unsigned none = __ballot_sync(0xFFFFFFFFu, (s[m] >> 62) == 0);
                    const unsigned inc = __ballot_sync(0xFFFFFFFFu, (s[m] >> 62) == 2);
                    const int first_inc = inc ? (__ffs(inc) - 1) : 32;
                    const unsigned relevant = (first_inc >= 31) ? 0xFFFFFFFFu : ((2u << first_inc) - 1u);
                    if (none & relevant) {
                        ready = false;
                    } else {
                        part += (lane <= first_inc) ? (s[m] & kValMask) : 0ULL;
                        done = first_inc < 32;
                    }
                }
            }
            if (ready) {
                acc += part;
                break;
            }
            done = false;
            if (!kBlocking) return false;
        }
        if (done) break;
        idx -= 32 * kSub;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, d);
    if (lane == 0) status[t] = kFlagInc | (acc + total);
    *out = acc;
    return true;
}

}  // namespace frb
