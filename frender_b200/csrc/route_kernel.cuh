// Hot path C: demux record router (reference loop F:774-810, write_reads F:726-730, grouper F:719-723).
//
// A STREAM of chunk pairs (R1 bytes, R2 bytes, cut anywhere) goes through the device without a host round trip
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
// re-reads the chunk, which is still in L2).  Nothing here depends on a host-side count: grids are sized by
// capacity and the kernels take the record counts from device memory.
#pragma once
#include "common.cuh"

namespace frb {

constexpr int kRouteBlock = 256;                    // records per histogram block

// Device-resident state of the stream (one per context; the `out` part is copied to the host per chunk).
struct RouteState {
    // carried into the next chunk
    unsigned long long skip1, skip2;      // where the text begins in the next chunk's buffers (carry area - carry)
    // this chunk
    unsigned long long n1, n2;            // records parsed (a trailing partial one included)
    unsigned long long lines1, lines2;    // lines parsed
    unsigned long long pairs;             // records routed
    unsigned long long used1, used2;      // end of the routed records in the chunk buffers (buffer offsets)
    unsigned long long out1, out2;        // bytes written to the sinks, per mate
    unsigned long long bad;               // smallest record with a key the results table does not hold (~0: none)
    unsigned long long bad_key;
    int error;                            // FRB_ERR_* raised by the plan (a record longer than the carry area)
    int done;                             // one mate has ended and is used up: zip() is over, later chunks are ignored
};

// results-table build: key -> sink id stored in Slot.count (keys are unique: the host keeps the
// last CSV row of a repeated key, as a Python dict does, F:660)
__global__ void __launch_bounds__(256) route_build_kernel(Slot* tab, unsigned long long mask,
                                                          const unsigned long long* __restrict__ keys,
                                                          const unsigned* __restrict__ sinks, unsigned long long n,
                                                          DevState* st) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    const unsigned long long key = keys[i];
    unsigned long long h = hash64(key) & mask;
    for (unsigned probe = 0; probe < kMaxProbe; ++probe) {
        const unsigned long long k = atomicCAS(&tab[h].key, kEmpty, key);
        if (k == kEmpty || k == key) {
            tab[h].count = sinks[i];
            return;
        }
        h = (h + 1) & mask;
    }
    raise_error(st, FRB_ERR_TABLE_FULL, key);
}

// route_build_kernel for a wide context: (lo, hi) -> sink id in WideSlot.count, claimed with one 128-bit
// compare-and-swap on a table filled with ones (no real key has bit 63 of either word set).
__global__ void __launch_bounds__(256) route_build_wide_kernel(WideSlot* tab, unsigned long long mask,
                                                               const unsigned long long* __restrict__ keys,
                                                               const unsigned long long* __restrict__ keys_hi,
                                                               const unsigned* __restrict__ sinks, unsigned long long n,
                                                               DevState* st) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    const unsigned long long lo = keys[i], hi = keys_hi[i];
    unsigned long long h = hash64(lo ^ (hi * 0x9E3779B97F4A7C15ULL)) & mask;
    for (unsigned probe = 0; probe < kMaxProbe; ++probe) {
        const Key128 k = atomicCAS(reinterpret_cast<Key128*>(&tab[h].lo), Key128{kEmpty, kEmpty}, Key128{lo, hi});
        if ((k.lo == kEmpty && k.hi == kEmpty) || (k.lo == lo && k.hi == hi)) {
            tab[h].count = sinks[i];
            return;
        }
        h = (h + 1) & mask;
    }
    raise_error_wide(st, FRB_ERR_TABLE_FULL, lo, hi);
}

// The parser left n_reads / line_carry of the mate it just scanned in DevState: move them into the stream state
// and clear them for the next launch.  which = 1 / 2.
__global__ void route_grab_kernel(DevState* st, RouteState* rs, int which) {
    if (threadIdx.x || blockIdx.x) return;
    if (which == 2) rs->n2 = st->n_reads, rs->lines2 = st->line_carry;
    else rs->n1 = st->n_reads, rs->lines1 = st->line_carry;
    st->n_reads = 0, st->line_carry = 0;
}

// pairs, bytes used, and the terminators of the offset lists.  end1 / end2 = bytes in the chunk buffers;
// final bit 0 / 1: the R1 / R2 stream ends with this chunk.
__global__ void route_plan_kernel(RouteState* rs, DevState* st, unsigned long long* off1, unsigned long long* off2,
                                  const unsigned char* __restrict__ in1, const unsigned char* __restrict__ in2,
                                  unsigned long long end1, unsigned long long end2, int final_chunk,
                                  unsigned long long rec_cap, unsigned long long carry_cap, unsigned long long* tot,
                                  unsigned n_tot) {
    for (unsigned k = threadIdx.x; k < n_tot; k += blockDim.x) tot[k] = 0;  // per-sink bytes, summed by the histogram
    if (threadIdx.x || blockIdx.x) return;
    rs->error = 0;
    if (rs->done) {  // chunks the host had already queued when the shorter mate ran out
        st->err_code = 0;
        rs->pairs = 0;
        rs->used1 = end1, rs->used2 = end2;
        return;
    }
    if (st->err_code) {  // raised by the parser (a key outside the alphabet, ...)
        rs->error = st->err_code;
        rs->bad_key = st->err_pos;
        st->err_code = 0;
        rs->pairs = 0;
        return;
    }
    if (rs->n1 > rec_cap || rs->n2 > rec_cap) {
        rs->error = FRB_ERR_ARG;  // records shorter than 16 bytes
        rs->pairs = 0;
        return;
    }
    off1[rs->n1] = end1;
    off2[rs->n2] = end2;
    // zip() of the 4-line groupers stops at the shorter mate (F:777); a trailing partial record only exists at the
    // end of a file (F:719-723)
    // (the parser counts a last line without '\n' as a line; before the end of the file it is not complete)
    const unsigned long long open1 = (end1 > rs->skip1 && in1[end1 - 1] != '\n') ? 1 : 0;
    const unsigned long long open2 = (end2 > rs->skip2 && in2[end2 - 1] != '\n') ? 1 : 0;
    const unsigned long long e1 = (final_chunk & 1) ? rs->n1 : (rs->lines1 - open1) / 4;
    const unsigned long long e2 = (final_chunk & 2) ? rs->n2 : (rs->lines2 - open2) / 4;
    const unsigned long long n = e1 < e2 ? e1 : e2;
    rs->pairs = n;
    rs->used1 = n ? off1[n] : rs->skip1;
    rs->used2 = n ? off2[n] : rs->skip2;
    rs->bad = ~0ull;
    // a mate that has ended and is used up ends the stream (F:777): what the other one still holds is never read
    if (((final_chunk & 1) && n == rs->n1) || ((final_chunk & 2) && n == rs->n2)) {
        rs->done = 1;
        rs->used1 = end1, rs->used2 = end2;
    }
    if (end1 - rs->used1 > carry_cap || end2 - rs->used2 > carry_cap) rs->error = FRB_ERR_ARG;
}

// sink of every record, its offset inside its (block, sink) cell, and the cells' sizes.  cell[(s * n_blocks + b)]
// for mate 1, the same + n_sinks * n_blocks for mate 2.  One warp-step after the other inside a block, so that
// records of one sink keep their order.
__global__ void __launch_bounds__(kRouteBlock) route_hist_kernel(const Slot* __restrict__ tab, unsigned long long mask,
                                                                 const unsigned long long* __restrict__ key2,
                                                                 const unsigned long long* __restrict__ off1,
                                                                 const unsigned long long* __restrict__ off2,
                                                                 RouteState* rs, unsigned n_sinks, unsigned n_blocks,
                                                                 unsigned* __restrict__ sink, unsigned* __restrict__ local1,
                                                                 unsigned* __restrict__ local2,
                                                                 unsigned long long* __restrict__ cell,
                                                                 unsigned long long* __restrict__ tot) {
    extern __shared__ unsigned s_acc[];  // [2][n_sinks]
    const unsigned long long n = rs->pairs;
    const unsigned b = blockIdx.x;
    if (static_cast<unsigned long long>(b) * kRouteBlock >= n) return;
    for (unsigned i = threadIdx.x; i < 2 * n_sinks; i += kRouteBlock) s_acc[i] = 0;
    __syncthreads();
    const unsigned long long i = static_cast<unsigned long long>(b) * kRouteBlock + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned s = 0xFFFFFFFFu, l1 = 0, l2 = 0;
    if (i < n) {
        const unsigned long long key = key2[i];
        unsigned long long h = hash64(key) & mask;
        for (unsigned probe = 0; probe < kMaxProbe; ++probe) {
            const unsigned long long k = tab[h].key;
            if (k == key) {
                s = static_cast<unsigned>(tab[h].count);
                break;
            }
            if (k == kEmpty) break;
            h = (h + 1) & mask;
        }
        if (s == 0xFFFFFFFFu) {
            atomicMin(&rs->bad, i);
            s = 0;
        }
        l1 = static_cast<unsigned>(off1[i + 1] - off1[i]);
        l2 = static_cast<unsigned>(off2[i + 1] - off2[i]);
        sink[i] = s;
    }
    for (int w = 0; w < kRouteBlock / 32; ++w) {
        if (warp == w && i < n) {
            const unsigned active = __activemask();
            const unsigned same = __match_any_sync(active, s);
            // bytes of the lower lanes of my sink
            unsigned before1 = 0, before2 = 0, tot1 = 0, tot2 = 0;
            for (unsigned m = same; m; m &= m - 1) {
                const int src = __ffs(m) - 1;
                const unsigned a1 = __shfl_sync(same, l1, src), a2 = __shfl_sync(same, l2, src);
                if (src < lane) before1 += a1, before2 += a2;
                tot1 += a1, tot2 += a2;
            }
            local1[i] = s_acc[s] + before1;
            local2[i] = s_acc[n_sinks + s] + before2;
            __syncwarp(active);
            if (lane == __ffs(same) - 1) s_acc[s] += tot1, s_acc[n_sinks + s] += tot2;
        }
        __syncthreads();
    }
    for (unsigned k = threadIdx.x; k < n_sinks; k += kRouteBlock) {
        cell[static_cast<unsigned long long>(k) * n_blocks + b] = s_acc[k];
        cell[static_cast<unsigned long long>(n_sinks + k) * n_blocks + b] = s_acc[n_sinks + k];
        if (s_acc[k]) atomicAdd(&tot[k], static_cast<unsigned long long>(s_acc[k]));
        if (s_acc[n_sinks + k]) atomicAdd(&tot[n_sinks + k], static_cast<unsigned long long>(s_acc[n_sinks + k]));
    }
}

// route_hist_kernel for a wide context: key2 holds rec_cap lower words, then rec_cap upper words; the results table
// is a WideSlot table (sink id in `count`, free slots all ones).  Kept apart from the narrow kernel, whose code this
// leaves exactly as it is.
// sink of every record, its offset inside its (block, sink) cell, and the cells' sizes.  cell[(s * n_blocks + b)]
// for mate 1, the same + n_sinks * n_blocks for mate 2.  One warp-step after the other inside a block, so that
// records of one sink keep their order.
__global__ void __launch_bounds__(kRouteBlock) route_hist_wide_kernel(const WideSlot* __restrict__ tab, unsigned long long mask,
                                                                 const unsigned long long* __restrict__ key2,
                                                                 unsigned long long rec_cap,
                                                                 const unsigned long long* __restrict__ off1,
                                                                 const unsigned long long* __restrict__ off2,
                                                                 RouteState* rs, unsigned n_sinks, unsigned n_blocks,
                                                                 unsigned* __restrict__ sink, unsigned* __restrict__ local1,
                                                                 unsigned* __restrict__ local2,
                                                                 unsigned long long* __restrict__ cell,
                                                                 unsigned long long* __restrict__ tot) {
    extern __shared__ unsigned s_acc[];  // [2][n_sinks]
    const unsigned long long n = rs->pairs;
    const unsigned b = blockIdx.x;
    if (static_cast<unsigned long long>(b) * kRouteBlock >= n) return;
    for (unsigned i = threadIdx.x; i < 2 * n_sinks; i += kRouteBlock) s_acc[i] = 0;
    __syncthreads();
    const unsigned long long i = static_cast<unsigned long long>(b) * kRouteBlock + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned s = 0xFFFFFFFFu, l1 = 0, l2 = 0;
    if (i < n) {
        const unsigned long long lo = key2[i], hi = key2[rec_cap + i];
        unsigned long long h = hash64(lo ^ (hi * 0x9E3779B97F4A7C15ULL)) & mask;
        for (unsigned probe = 0; probe < kMaxProbe; ++probe) {
            const ulonglong2 k = *reinterpret_cast<const ulonglong2*>(&tab[h].lo);
            if (k.x == lo && k.y == hi) {
                s = static_cast<unsigned>(tab[h].count);
                break;
            }
            if (k.x == kEmpty) break;
            h = (h + 1) & mask;
        }
        if (s == 0xFFFFFFFFu) {
            atomicMin(&rs->bad, i);
            s = 0;
        }
        l1 = static_cast<unsigned>(off1[i + 1] - off1[i]);
        l2 = static_cast<unsigned>(off2[i + 1] - off2[i]);
        sink[i] = s;
    }
    for (int w = 0; w < kRouteBlock / 32; ++w) {
        if (warp == w && i < n) {
            const unsigned active = __activemask();
            const unsigned same = __match_any_sync(active, s);
            // bytes of the lower lanes of my sink
            unsigned before1 = 0, before2 = 0, tot1 = 0, tot2 = 0;
            for (unsigned m = same; m; m &= m - 1) {
                const int src = __ffs(m) - 1;
                const unsigned a1 = __shfl_sync(same, l1, src), a2 = __shfl_sync(same, l2, src);
                if (src < lane) before1 += a1, before2 += a2;
                tot1 += a1, tot2 += a2;
            }
            local1[i] = s_acc[s] + before1;
            local2[i] = s_acc[n_sinks + s] + before2;
            __syncwarp(active);
            if (lane == __ffs(same) - 1) s_acc[s] += tot1, s_acc[n_sinks + s] += tot2;
        }
        __syncthreads();
    }
    for (unsigned k = threadIdx.x; k < n_sinks; k += kRouteBlock) {
        cell[static_cast<unsigned long long>(k) * n_blocks + b] = s_acc[k];
        cell[static_cast<unsigned long long>(n_sinks + k) * n_blocks + b] = s_acc[n_sinks + k];
        if (s_acc[k]) atomicAdd(&tot[k], static_cast<unsigned long long>(s_acc[k]));
        if (s_acc[n_sinks + k]) atomicAdd(&tot[n_sinks + k], static_cast<unsigned long long>(s_acc[n_sinks + k]));
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
            if (mate == 0) rs->out1 = end;
            else rs->out2 = end;
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

// The unconsumed tails in front of the next chunk's buffers (they end where the host puts the new
// bytes), and where the text begins there.
__global__ void __launch_bounds__(1024) route_carry_kernel(RouteState* rs, const unsigned char* __restrict__ in1,
                                                           const unsigned char* __restrict__ in2, unsigned long long end1,
                                                           unsigned long long end2, unsigned char* __restrict__ next1,
                                                           unsigned char* __restrict__ next2, unsigned long long carry_cap) {
    const unsigned long long c1 = end1 - rs->used1, c2 = end2 - rs->used2;
    if (rs->error) return;
    const unsigned char* const src = blockIdx.y ? in2 + rs->used2 : in1 + rs->used1;
    unsigned char* const dst = blockIdx.y ? next2 + (carry_cap - c2) : next1 + (carry_cap - c1);
    const unsigned long long c = blockIdx.y ? c2 : c1;
    for (unsigned long long i = blockIdx.x * 1024ull + threadIdx.x; i < c; i += gridDim.x * 1024ull) dst[i] = src[i];
    __syncthreads();
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
        // read by the NEXT chunk's kernels only (stream order)
        rs->skip1 = carry_cap - c1;
        rs->skip2 = carry_cap - c2;
    }
}

}  // namespace frb
