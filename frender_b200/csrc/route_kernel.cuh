// Hot path C: demux record router (reference loop F:774-810, write_reads F:726-730, grouper F:719-723).
//
// A STREAM of chunks (R1 bytes, R2 bytes, ..., cut anywhere) goes through the device without a host round trip
// in between:
//   scan_ws_kernel (general form) on R2: key of every record under the demux rule (F:778) + record offsets;
//   on R1: record offsets only.  A record that is not complete yet (and the surplus records of the mate that
//   happens to be ahead) stay on the device as the carried tail of the next chunk.
//   route_plan_kernel   pairs = the records both mates have complete (zip() of the 4-line groupers, F:777; a
//                       trailing partial record counts once its file has ended, F:719-723); bytes consumed
//   route_hist_kernel   per record: sink id from the results table (hash look-up), lengths of both mates' records;
//                       per block of 256 records and per sink the bytes of each mate, and every record's offset
//                       inside its (block, sink) cell -- in record order, so the partition is STABLE
//   route_scan_kernel   exclusive sum over the (sink, block) matrix in sink-major order: where every cell starts
//                       in the output; the sinks' own offsets fall out of it
//   route_copy_kernel   one warp per record and mate: 16-byte stores, source realigned with funnel shifts
//   route_carry_kernel  the unconsumed tails to the front of the next chunk's buffers
// Algorithmic bytes = 2 x (R1 + R2): every byte read once by the parser and written once into its sink (the copy
// re-reads the chunk, which is still in L2).
// A single-end stream (Mates = 1, frb_route_set_mates) is the same with R1 alone: the parser takes the keys from the
// R1 headers, the routed records are R1's complete records (no zip), the scan runs on a (S, 1) grid and the copy,
// the carry and the deflate on R1 only -- 2 x R1 algorithmic bytes.
// Index reads (frb_route_set_mates2, Mates = 3 or 4) add the I1 / I2 files as more mates behind R1 (and R2): the key
// still comes from one mate (R2, or R1 in a single-end stream), every other mate is parsed for record offsets only,
// and record i of every mate goes to the sink of record i's key.  The zip() runs over all Mates files; the scan runs
// on a (S, Mates) grid, the carry on (64, Mates), the copy and the deflate once per mate.  Nothing here depends on a
// host-side count: grids are sized by capacity and the kernels take the record counts from device memory.
#pragma once
#include "common.cuh"

namespace frb {

constexpr int kRouteBlock = 256;                    // records per histogram block
constexpr int kRouteMaxMates = 4;                   // R1, R2, I1, I2
// Shared memory a block may have on sm_90 / sm_100 (the opt-in limit): the histogram keeps [Mates][n_sinks] u32
// counters in it, so a stream of m mates takes at most kRouteSmemMax / (4 m) sinks (14,528 at 4 mates).
constexpr unsigned kRouteSmemMax = 227u << 10;

// Device-resident state of the stream (one per context; copied to the host per chunk).  Per-mate arrays: mate m is
// the m-th buffer of frb_route_pushv (R1, R2, then the index reads).
struct RouteState {
    // carried into the next chunk
    unsigned long long skip[kRouteMaxMates];   // where the text begins in the next chunk's buffers (carry area - carry)
    // this chunk
    unsigned long long n[kRouteMaxMates];      // records parsed (a trailing partial one included)
    unsigned long long lines[kRouteMaxMates];  // lines parsed
    unsigned long long pairs;                  // records routed (of every mate)
    unsigned long long used[kRouteMaxMates];   // end of the routed records in the chunk buffers (buffer offsets)
    unsigned long long out[kRouteMaxMates];    // bytes written to the sinks, per mate
    unsigned long long bad;                    // smallest record with a key the results table does not hold (~0: none)
    unsigned long long bad_key;
    int error;                                 // FRB_ERR_* raised by the plan (a record longer than the carry area)
    int done;                                  // one mate has ended and is used up: zip() is over, later chunks are ignored
};

// Per-mate device pointers and sizes of one chunk, passed by value (mates >= Mates are not read).
struct RouteMates {
    unsigned long long* off[kRouteMaxMates];   // record offsets (rec_cap + 1 each)
    unsigned* local[kRouteMaxMates];           // offset of every record inside its (block, sink) cell
    const unsigned char* in[kRouteMaxMates];   // the chunk buffers: [carry area | new bytes]
    unsigned char* next[kRouteMaxMates];       // the next chunk's buffers (the carry goes there)
    unsigned long long end[kRouteMaxMates];    // bytes in the chunk buffers (carry area included)
};

// results-table build: key -> sink id stored in the slot's `count` (keys are unique: the host keeps the last CSV row
// of a repeated key, as a Python dict does, F:660).  The table is filled with ones (no real key has bit 63 of either
// word set); a wide key is claimed with one 128-bit compare-and-swap.  keys_hi: upper key words (wide only).
template <bool Wide>
__global__ void __launch_bounds__(256) route_build_kernel(Slot* table, unsigned long long mask,
                                                          const unsigned long long* __restrict__ keys,
                                                          const unsigned* __restrict__ sinks, unsigned long long n,
                                                          DevState* st, const unsigned long long* __restrict__ keys_hi) {
    using K = KeyWidth<Wide>;
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    typename K::Slot* const tab = reinterpret_cast<typename K::Slot*>(table);
    const auto key = K::at(keys, keys_hi, i);
    unsigned long long h = K::hash(key) & mask;
    for (unsigned probe = 0; probe < kMaxProbe; ++probe) {
        const auto k = K::claim(&tab[h], K::ones(), key);
        if (K::same(k, K::ones()) || K::same(k, key)) {
            tab[h].count = sinks[i];
            return;
        }
        h = (h + 1) & mask;
    }
    raise_error<Wide>(st, FRB_ERR_TABLE_FULL, key);
}

// The parser left n_reads / line_carry of the mate it just scanned in DevState: move them into the stream state
// and clear them for the next launch.
__global__ void route_grab_kernel(DevState* st, RouteState* rs, int mate) {
    if (threadIdx.x || blockIdx.x) return;
    rs->n[mate] = st->n_reads, rs->lines[mate] = st->line_carry;
    st->n_reads = 0, st->line_carry = 0;
}

// pairs, bytes used, and the terminators of the offset lists.  m.end[k] = bytes in the chunk buffers of mate k;
// final bit k: mate k's file ends with this chunk.  The routed records are the ones every mate has complete (the
// zip() of the 4-line groupers, F:777, over Mates files; Mates = 1: R1's complete records).
template <int Mates>
__global__ void route_plan_kernel(RouteState* rs, DevState* st, RouteMates m, int final_chunk,
                                  unsigned long long rec_cap, unsigned long long carry_cap, unsigned long long* tot,
                                  unsigned n_tot) {
    for (unsigned k = threadIdx.x; k < n_tot; k += blockDim.x) tot[k] = 0;  // per-sink bytes, summed by the histogram
    if (threadIdx.x || blockIdx.x) return;
    rs->error = 0;
    if (rs->done) {  // chunks the host had already queued when the shorter mate ran out
        st->err_code = 0;
        rs->pairs = 0;
#pragma unroll
        for (int k = 0; k < Mates; ++k) rs->used[k] = m.end[k];
        return;
    }
    if (st->err_code) {  // raised by the parser (a key outside the alphabet, ...)
        rs->error = st->err_code;
        rs->bad_key = st->err_pos;
        st->err_code = 0;
        rs->pairs = 0;
        return;
    }
#pragma unroll
    for (int k = 0; k < Mates; ++k)
        if (rs->n[k] > rec_cap) {
            rs->error = FRB_ERR_ARG;  // records shorter than 16 bytes
            rs->pairs = 0;
            return;
        }
    // zip() of the 4-line groupers stops at the shorter mate (F:777); a trailing partial record only exists at the
    // end of a file (F:719-723)
    // (the parser counts a last line without '\n' as a line; before the end of the file it is not complete)
    unsigned long long n = ~0ull;
#pragma unroll
    for (int k = 0; k < Mates; ++k) {
        m.off[k][rs->n[k]] = m.end[k];
        const unsigned long long open = (m.end[k] > rs->skip[k] && m.in[k][m.end[k] - 1] != '\n') ? 1 : 0;
        const unsigned long long e = (final_chunk >> k & 1) ? rs->n[k] : (rs->lines[k] - open) / 4;
        n = e < n ? e : n;
    }
    rs->pairs = n;
    rs->bad = ~0ull;
    // a mate that has ended and is used up ends the stream (F:777): what the others still hold is never read
    bool over = false;
#pragma unroll
    for (int k = 0; k < Mates; ++k) {
        rs->used[k] = n ? m.off[k][n] : rs->skip[k];
        over = over || ((final_chunk >> k & 1) && n == rs->n[k]);
    }
    if (over) rs->done = 1;
#pragma unroll
    for (int k = 0; k < Mates; ++k) {
        if (over) rs->used[k] = m.end[k];
        if (m.end[k] - rs->used[k] > carry_cap) rs->error = FRB_ERR_ARG;
    }
}

// sink of every record, its offset inside its (block, sink) cell, and the cells' sizes.  cell[(k * n_sinks + s) *
// n_blocks + b] for mate k.  One warp-step after the other inside a block, so that records of one sink keep their
// order.  key: the keys of the routed records (parsed from the key mate's headers: R2, or R1 in a single-end stream);
// key_hi: their upper words (wide only).
template <bool Wide, int Mates>
__global__ void __launch_bounds__(kRouteBlock) route_hist_kernel(const Slot* __restrict__ table, unsigned long long mask,
                                                                 const unsigned long long* __restrict__ key,
                                                                 const RouteMates m, RouteState* rs, unsigned n_sinks,
                                                                 unsigned n_blocks, unsigned* __restrict__ sink,
                                                                 unsigned long long* __restrict__ cell,
                                                                 unsigned long long* __restrict__ tot,
                                                                 const unsigned long long* __restrict__ key_hi) {
    using K = KeyWidth<Wide>;
    const typename K::Slot* __restrict__ const tab = reinterpret_cast<const typename K::Slot*>(table);
    extern __shared__ unsigned s_acc[];  // [Mates][n_sinks]
    const unsigned long long n = rs->pairs;
    const unsigned b = blockIdx.x;
    if (static_cast<unsigned long long>(b) * kRouteBlock >= n) return;
    for (unsigned i = threadIdx.x; i < Mates * n_sinks; i += kRouteBlock) s_acc[i] = 0;
    __syncthreads();
    const unsigned long long i = static_cast<unsigned long long>(b) * kRouteBlock + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned s = 0xFFFFFFFFu, len[Mates];
#pragma unroll
    for (int k = 0; k < Mates; ++k) len[k] = 0;
    if (i < n) {
        const auto k = K::at(key, key_hi, i);
        unsigned long long h = K::hash(k) & mask;
        for (unsigned probe = 0; probe < kMaxProbe; ++probe) {
            const auto t = K::load(&tab[h]);
            if (K::same(t, k)) {
                s = static_cast<unsigned>(tab[h].count);
                break;
            }
            if (K::is_free(t)) break;
            h = (h + 1) & mask;
        }
        if (s == 0xFFFFFFFFu) {
            atomicMin(&rs->bad, i);
            s = 0;
        }
#pragma unroll
        for (int q = 0; q < Mates; ++q) len[q] = static_cast<unsigned>(m.off[q][i + 1] - m.off[q][i]);
        sink[i] = s;
    }
    for (int w = 0; w < kRouteBlock / 32; ++w) {
        if (warp == w && i < n) {
            const unsigned active = __activemask();
            const unsigned same = __match_any_sync(active, s);
            // bytes of the lower lanes of my sink
            unsigned before[Mates], all[Mates];
#pragma unroll
            for (int q = 0; q < Mates; ++q) before[q] = 0, all[q] = 0;
            for (unsigned bits = same; bits; bits &= bits - 1) {
                const int src = __ffs(bits) - 1;
#pragma unroll
                for (int q = 0; q < Mates; ++q) {
                    const unsigned a = __shfl_sync(same, len[q], src);
                    if (src < lane) before[q] += a;
                    all[q] += a;
                }
            }
#pragma unroll
            for (int q = 0; q < Mates; ++q) m.local[q][i] = s_acc[q * n_sinks + s] + before[q];
            __syncwarp(active);
            if (lane == __ffs(same) - 1) {
#pragma unroll
                for (int q = 0; q < Mates; ++q) s_acc[q * n_sinks + s] += all[q];
            }
        }
        __syncthreads();
    }
    for (unsigned k = threadIdx.x; k < n_sinks; k += kRouteBlock) {
#pragma unroll
        for (int q = 0; q < Mates; ++q) {
            const unsigned v = s_acc[q * n_sinks + k];
            cell[(static_cast<unsigned long long>(q) * n_sinks + k) * n_blocks + b] = v;
            if (v) atomicAdd(&tot[q * n_sinks + k], static_cast<unsigned long long>(v));
        }
    }
}

// Exclusive sum over the (sink, block) matrix of one mate in sink-major order, in place: where every cell starts in
// the output.  Block (s, mate) takes row s: its base is the sum of the totals of the sinks in front (tot[], summed
// by the histogram), then the row's used cells are summed 256 at a time.  sink_off[m][s] = start of sink s
// (n_sinks + 1 entries per mate).
__global__ void __launch_bounds__(kRouteBlock) route_scan_kernel(unsigned long long* cell, unsigned n_sinks, unsigned n_blocks,
                                                                 RouteState* rs, const unsigned long long* __restrict__ tot,
                                                                 unsigned long long* sink_off) {
    __shared__ unsigned long long s_warp[kRouteBlock / 32];
    const unsigned s = blockIdx.x, mate = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long used_blocks = (rs->pairs + kRouteBlock - 1) / kRouteBlock;
    unsigned long long* const row = cell + (static_cast<unsigned long long>(mate) * n_sinks + s) * n_blocks;
    const unsigned long long* const t = tot + static_cast<unsigned long long>(mate) * n_sinks;
    auto block_scan = [&](unsigned long long v, unsigned long long* total) {  // inclusive sum over the block
        unsigned long long incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += o;
        }
        __syncthreads();  // s_warp of the round before has been read
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned long long before = 0, all = 0;
#pragma unroll
        for (int w = 0; w < kRouteBlock / 32; ++w) {
            const unsigned long long x = s_warp[w];
            before += w < warp ? x : 0ull;
            all += x;
        }
        *total = all;
        return incl + before;
    };
    unsigned long long mine = 0, base;
    for (unsigned k = threadIdx.x; k < s; k += kRouteBlock) mine += t[k];
    block_scan(mine, &base);
    if (threadIdx.x == 0) {
        sink_off[static_cast<unsigned long long>(mate) * (n_sinks + 1) + s] = base;
        if (s == n_sinks - 1) {
            const unsigned long long end = base + t[s];
            sink_off[static_cast<unsigned long long>(mate) * (n_sinks + 1) + n_sinks] = end;
            rs->out[mate] = end;
        }
    }
    for (unsigned long long b0 = 0; b0 < used_blocks; b0 += kRouteBlock) {
        const unsigned long long b = b0 + threadIdx.x;
        const unsigned long long v = b < used_blocks ? row[b] : 0ull;
        unsigned long long total;
        const unsigned long long incl = block_scan(v, &total);
        if (b < used_blocks) row[b] = base + incl - v;
        base += total;
    }
}

// One warp per record (of one mate): dst is written with aligned 16-byte stores, the source is read as aligned
// 32-bit words and shifted into place (records start anywhere).
__global__ void __launch_bounds__(256) route_copy_kernel(const RouteState* __restrict__ rs, const unsigned* __restrict__ sink,
                                                         const unsigned* __restrict__ local, const unsigned long long* __restrict__ cell,
                                                         unsigned n_blocks, const unsigned long long* __restrict__ off,
                                                         const unsigned char* __restrict__ in, unsigned char* __restrict__ out) {
    const unsigned long long n = rs->pairs;
    const int lane = threadIdx.x & 31;
    const unsigned long long wstride = static_cast<unsigned long long>(gridDim.x) * (blockDim.x >> 5);
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x >> 5) + (threadIdx.x >> 5); i < n;
         i += wstride) {
        const unsigned long long o = off[i];
        const unsigned len = static_cast<unsigned>(off[i + 1] - o);
        const unsigned char* const src = in + o;
        unsigned char* const dst = out + cell[static_cast<unsigned long long>(sink[i]) * n_blocks + i / kRouteBlock] + local[i];
        // head: bytes up to the first 16-byte boundary of dst
        const unsigned head = min(len, static_cast<unsigned>((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15));
        if (static_cast<unsigned>(lane) < head) dst[lane] = src[lane];
        const unsigned body = (len - head) >> 4;  // whole 16-byte pieces
        const unsigned char* const s0 = src + head;
        const unsigned mis = static_cast<unsigned>(reinterpret_cast<uintptr_t>(s0) & 3);
        const unsigned* const sw = reinterpret_cast<const unsigned*>(s0 - mis);
        uint4* const d4 = reinterpret_cast<uint4*>(dst + head);
        for (unsigned k = lane; k < body; k += 32) {
            const unsigned* const w = sw + 4 * k;
            uint4 v;
            if (mis == 0) {
                v = make_uint4(w[0], w[1], w[2], w[3]);
            } else {
                const unsigned sh = 8 * mis;
                const unsigned a0 = w[0], a1 = w[1], a2 = w[2], a3 = w[3], a4 = w[4];
                v = make_uint4(__funnelshift_r(a0, a1, sh), __funnelshift_r(a1, a2, sh), __funnelshift_r(a2, a3, sh),
                               __funnelshift_r(a3, a4, sh));
            }
            d4[k] = v;
        }
        const unsigned done = head + (body << 4);
        if (done + lane < len) dst[done + lane] = src[done + lane];  // tail: fewer than 16 bytes
    }
}

// The unconsumed tails in front of the next chunk's buffers (they end where the host puts the new bytes), and
// where the text begins there.  Grid (64, mates): blockIdx.y is the mate.
__global__ void __launch_bounds__(1024) route_carry_kernel(RouteState* rs, const RouteMates m, unsigned long long carry_cap) {
    const unsigned k = blockIdx.y;
    const unsigned char* in = nullptr;
    unsigned char* next = nullptr;
    unsigned long long end = 0;
#pragma unroll
    for (unsigned q = 0; q < kRouteMaxMates; ++q)  // selects, not an indexed copy of the parameters in local memory
        if (q == k) in = m.in[q], next = m.next[q], end = m.end[q];
    const unsigned long long c = end - rs->used[k];
    if (rs->error) return;
    const unsigned char* const src = in + rs->used[k];
    unsigned char* const dst = next + (carry_cap - c);
    for (unsigned long long i = blockIdx.x * 1024ull + threadIdx.x; i < c; i += gridDim.x * 1024ull) dst[i] = src[i];
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x == 0) rs->skip[k] = carry_cap - c;  // read by the NEXT chunk's kernels only
}

}  // namespace frb
