// Unique-key table maintenance: clear, compaction to (key,count,first) lists, merge of a list
// into another table (per-file tables -> "total", F:199-205; per-rank totals -> merged total).
#pragma once
#include "common.cuh"

namespace frb {

__global__ void __launch_bounds__(256) clear_table_kernel(Slot* tab, unsigned long long cap) {
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    ulonglong4* t4 = reinterpret_cast<ulonglong4*>(tab);
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; i < cap;
         i += stride)
        t4[i] = make_ulonglong4(kEmpty, ~0ULL, 0ULL, 0ULL);  // key, first, count, aux
}

// Occupied slots (key present, count not taken back to 0 by a negate pass) -> dense arrays in arbitrary order;
// *counter receives their number (the scan kernel does not keep it: knowing who won a slot would mean waiting for
// every compare-and-swap's result).  One atomic per
// block and pass (a per-warp atomic on the one counter was the kernel's bound: 2 M atomics for 2^26 slots).
__global__ void __launch_bounds__(256) compact_table_kernel(const Slot* __restrict__ tab, unsigned long long cap,
                                                            unsigned long long* __restrict__ keys,
                                                            unsigned long long* __restrict__ counts,
                                                            unsigned long long* __restrict__ first,
                                                            unsigned long long* counter,
                                                            unsigned long long out_cap,
                                                            const unsigned long long* __restrict__ tile_first = nullptr) {
    __shared__ unsigned s_warp[8];
    __shared__ unsigned long long s_base;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long cap_up = (cap + 255) & ~255ULL;
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
         i < cap_up; i += stride) {
        ulonglong4 s = make_ulonglong4(kEmpty, 0, 0, 0);
        if (i < cap) s = reinterpret_cast<const ulonglong4*>(tab)[i];
        const bool occ = s.x != kEmpty && s.z != 0;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, occ);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        unsigned before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned v = s_warp[w];
            if (w < warp) before += v;
            total += v;
        }
        if (threadIdx.x == 0 && total) s_base = atomicAdd(counter, static_cast<unsigned long long>(total));
        __syncthreads();
        if (occ) {
            const unsigned long long idx = s_base + before + __popc(m & ((1u << lane) - 1u));
            if (idx < out_cap) {
                keys[idx] = s.x;
                counts[idx] = s.z;
                // composite position (tile << 13 | header index) -> read ordinal
                first[idx] = tile_first ? tile_first[s.y >> kCompositeShift] + (s.y & ((1ULL << kCompositeShift) - 1)) : s.y;
            }
        }
    }
}

__global__ void __launch_bounds__(256) iota_kernel(unsigned* idx, unsigned long long n) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) idx[i] = static_cast<unsigned>(i);
}

__global__ void __launch_bounds__(256) gather2_kernel(const unsigned* __restrict__ perm,
                                                      const unsigned long long* __restrict__ a_in,
                                                      const unsigned long long* __restrict__ b_in,
                                                      unsigned long long* __restrict__ a_out,
                                                      unsigned long long* __restrict__ b_out, unsigned long long n) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) {
        const unsigned p = perm[i];
        a_out[i] = a_in[p];
        b_out[i] = b_in[p];
    }
}

__global__ void __launch_bounds__(256) add_offset_kernel(const unsigned long long* __restrict__ in,
                                                         unsigned long long* __restrict__ out, unsigned long long n,
                                                         unsigned long long off) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) out[i] = in[i] + off;
}

// dst[key] += counts, first = min(first, pos_base + first_in)
__global__ void __launch_bounds__(256) merge_list_kernel(Slot* dst, unsigned long long mask,
                                                         const unsigned long long* __restrict__ keys,
                                                         const unsigned long long* __restrict__ counts,
                                                         const unsigned long long* __restrict__ first,
                                                         unsigned long long n, unsigned long long pos_base,
                                                         unsigned long long* occupied, DevState* st) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) table_add(dst, mask, keys[i], counts[i], first ? pos_base + first[i] : pos_base + i, occupied, st);
}

// Entries sorted by key (ks) with their original positions (perm): every run of equal keys becomes one entry
// (count: +, first: min), appended in arbitrary order.  Runs are at most n_ranks long.
__global__ void __launch_bounds__(256) fold_runs_kernel(const unsigned long long* __restrict__ ks,
                                                        const unsigned* __restrict__ perm,
                                                        const unsigned long long* __restrict__ counts,
                                                        const unsigned long long* __restrict__ first,
                                                        unsigned long long n, unsigned long long* __restrict__ k_out,
                                                        unsigned long long* __restrict__ c_out,
                                                        unsigned long long* __restrict__ f_out,
                                                        unsigned long long* counter) {
    const int lane = threadIdx.x & 31;
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    const unsigned long long key = i < n ? ks[i] : 0ULL;
    const bool head = i < n && (i == 0 || ks[i - 1] != key);
    unsigned long long sum = 0, mn = ~0ULL;
    if (head) {
        for (unsigned long long j = i; j < n && ks[j] == key; ++j) {
            const unsigned p = perm[j];
            sum += counts[p];
            const unsigned long long f = first[p];
            mn = f < mn ? f : mn;
        }
    }
    const unsigned m = __ballot_sync(0xFFFFFFFFu, head);
    if (m) {
        unsigned long long base = 0;
        const int leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(counter, static_cast<unsigned long long>(__popc(m)));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (head) {
            const unsigned long long idx = base + __popc(m & ((1u << lane) - 1u));
            k_out[idx] = key;
            c_out[idx] = sum;
            f_out[idx] = mn;
        }
    }
}

// 32 bits of the key's hash for every entry (what the received parts of a sharded merge are sorted on: four radix
// passes instead of the eight a 64-bit key takes) and the largest `first` among them (significant bits of the
// sort by first appearance that follows).
__global__ void __launch_bounds__(256) hash32_kernel(const unsigned long long* __restrict__ keys,
                                                     const unsigned long long* __restrict__ first, unsigned long long n,
                                                     unsigned* __restrict__ h32, unsigned long long* max_first) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    unsigned long long f = 0;
    if (i < n) {
        h32[i] = static_cast<unsigned>(hash64(keys[i]) >> 8);
        f = first[i];
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, f, d);
        f = o > f ? o : f;
    }
    if ((threadIdx.x & 31) == 0 && f) atomicMax(max_first, f);
}

// Entries sorted by hs = 32 hash bits of their keys (perm = original positions): one output entry per distinct
// KEY (count: +, first: min), appended in arbitrary order.  A run of equal hash bits holds one key from up to
// n_ranks parts -- and now and then a second key with the same 32 bits, which is why the keys themselves are
// compared inside the run.
__global__ void __launch_bounds__(256) fold_hash_runs_kernel(const unsigned* __restrict__ hs, const unsigned* __restrict__ perm,
                                                             const unsigned long long* __restrict__ keys,
                                                             const unsigned long long* __restrict__ counts,
                                                             const unsigned long long* __restrict__ first,
                                                             unsigned long long n, unsigned long long* __restrict__ k_out,
                                                             unsigned long long* __restrict__ c_out,
                                                             unsigned long long* __restrict__ f_out,
                                                             unsigned long long* counter) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    const unsigned h = hs[i];
    // this thread speaks for the key at sorted position i if no earlier position of the run holds the same key
    const unsigned long long key = keys[perm[i]];
    for (unsigned long long j = i; j > 0 && hs[j - 1] == h; --j)
        if (keys[perm[j - 1]] == key) return;
    unsigned long long sum = 0, mn = ~0ULL;
    for (unsigned long long j = i; j < n && hs[j] == h; ++j) {
        const unsigned p = perm[j];
        if (keys[p] != key) continue;
        sum += counts[p];
        const unsigned long long f = first[p];
        mn = f < mn ? f : mn;
    }
    const unsigned long long idx = atomicAdd(counter, 1ULL);
    k_out[idx] = key;
    c_out[idx] = sum;
    f_out[idx] = mn;
}

// Owner rank of a key in the sharded merge: hash bits the table index does not use.
__host__ __device__ __forceinline__ unsigned key_owner(unsigned long long key, unsigned n_ranks) {
    return static_cast<unsigned>((hash64(key) >> 40) % n_ranks);
}

// owner[i] of every list entry + per-owner histogram (shared-memory partial counts, one atomic per block and owner)
__global__ void __launch_bounds__(256) owner_kernel(const unsigned long long* __restrict__ keys, unsigned long long n,
                                                    unsigned n_ranks, unsigned* __restrict__ owner,
                                                    unsigned long long* __restrict__ hist) {
    __shared__ unsigned s_hist[256];
    if (threadIdx.x < n_ranks) s_hist[threadIdx.x] = 0;
    __syncthreads();
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) {
        const unsigned o = key_owner(keys[i], n_ranks);
        owner[i] = o;
        atomicAdd(&s_hist[o], 1u);
    }
    __syncthreads();
    if (threadIdx.x < n_ranks && s_hist[threadIdx.x]) atomicAdd(&hist[threadIdx.x], static_cast<unsigned long long>(s_hist[threadIdx.x]));
}

__global__ void __launch_bounds__(256) gather3_kernel(const unsigned* __restrict__ perm,
                                                      const unsigned long long* __restrict__ a_in,
                                                      const unsigned long long* __restrict__ b_in,
                                                      const unsigned long long* __restrict__ c_in,
                                                      unsigned long long* __restrict__ a_out,
                                                      unsigned long long* __restrict__ b_out,
                                                      unsigned long long* __restrict__ c_out, unsigned long long n) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) {
        const unsigned p = perm[i];
        a_out[i] = a_in[p];
        b_out[i] = b_in[p];
        c_out[i] = c_in[p];
    }
}

// demux_ok (F:504-564): a unique key is "ok" unless some file holds it whose NAME does not fit the key's class.
// One thread per entry of one file's list: find the key in the total list (binary search in the key-sorted view),
// take its class -- read type 0/1/3, or 4 + sample row for a demuxable key -- and look up class x file in the
// match matrix the host made with the reference's regexes (0 no, 1 yes, 2 the regex does not compile).
__global__ void __launch_bounds__(256) demux_ok_kernel(const unsigned long long* __restrict__ fkeys,
                                                       const unsigned long long* __restrict__ fcounts, unsigned long long nf,
                                                       const unsigned long long* __restrict__ sorted_keys,
                                                       const unsigned* __restrict__ sorted_idx, unsigned long long n,
                                                       const unsigned char* __restrict__ type, const int* __restrict__ srow,
                                                       const unsigned char* __restrict__ match, unsigned n_files, unsigned f,
                                                       unsigned char* __restrict__ ok, unsigned char* __restrict__ bad_file,
                                                       int* err_row) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i >= nf || (fcounts && fcounts[i] == 0)) return;
    const unsigned long long key = fkeys[i];
    unsigned long long lo = 0, hi = n;
    while (lo < hi) {
        const unsigned long long mid = (lo + hi) >> 1;
        if (sorted_keys[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    if (lo >= n || sorted_keys[lo] != key) return;  // not part of the total: nothing to flag
    const unsigned idx = sorted_idx[lo];
    const unsigned t = type[idx];
    const unsigned cls = t == 2 ? 4u + static_cast<unsigned>(srow[idx]) : t;
    const unsigned m = match[static_cast<unsigned long long>(cls) * n_files + f];
    if (m == 2) {
        atomicMin(err_row, static_cast<int>(cls) - 4);
    } else if (m == 0) {
        ok[idx] = 0;
        bad_file[f] = 1;
    }
}

// ---- wide context (WideSlot tables, keys as lo / hi arrays) ---------------------------------------------------
__global__ void __launch_bounds__(256) clear_wide_table_kernel(WideSlot* tab, unsigned long long cap) {
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    ulonglong4* t4 = reinterpret_cast<ulonglong4*>(tab);
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; i < cap;
         i += stride)
        t4[i] = make_ulonglong4(kEmpty, 0ULL, ~0ULL, 0ULL);  // lo, hi, first, count
}

// compact_table_kernel for WideSlot tables (no composite positions: a wide context never runs the speculative scan)
__global__ void __launch_bounds__(256) compact_wide_table_kernel(const WideSlot* __restrict__ tab, unsigned long long cap,
                                                                 unsigned long long* __restrict__ keys,
                                                                 unsigned long long* __restrict__ keys_hi,
                                                                 unsigned long long* __restrict__ counts,
                                                                 unsigned long long* __restrict__ first,
                                                                 unsigned long long* counter, unsigned long long out_cap) {
    __shared__ unsigned s_warp[8];
    __shared__ unsigned long long s_base;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long cap_up = (cap + 255) & ~255ULL;
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
         i < cap_up; i += stride) {
        ulonglong4 s = make_ulonglong4(kEmpty, 0, 0, 0);
        if (i < cap) s = reinterpret_cast<const ulonglong4*>(tab)[i];
        const bool occ = s.x != kEmpty && s.w != 0;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, occ);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        unsigned before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned v = s_warp[w];
            if (w < warp) before += v;
            total += v;
        }
        if (threadIdx.x == 0 && total) s_base = atomicAdd(counter, static_cast<unsigned long long>(total));
        __syncthreads();
        if (occ) {
            const unsigned long long idx = s_base + before + __popc(m & ((1u << lane) - 1u));
            if (idx < out_cap) keys[idx] = s.x, keys_hi[idx] = s.y, counts[idx] = s.w, first[idx] = s.z;
        }
    }
}

__global__ void __launch_bounds__(256) gather1_kernel(const unsigned* __restrict__ perm,
                                                      const unsigned long long* __restrict__ in,
                                                      unsigned long long* __restrict__ out, unsigned long long n) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) out[i] = in[perm[i]];
}

// dst[(lo, hi)] += counts, first = min(first, pos_base + first_in)
__global__ void __launch_bounds__(256) merge_wide_list_kernel(WideSlot* dst, unsigned long long mask,
                                                              const unsigned long long* __restrict__ keys,
                                                              const unsigned long long* __restrict__ keys_hi,
                                                              const unsigned long long* __restrict__ counts,
                                                              const unsigned long long* __restrict__ first,
                                                              unsigned long long n, unsigned long long pos_base,
                                                              unsigned long long* occupied, DevState* st) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i < n) table_add_wide(dst, mask, keys[i], keys_hi[i], counts[i], first ? pos_base + first[i] : pos_base + i, occupied, st);
}

// demux_ok_kernel over wide keys: the total is sorted by (hi, lo).
__global__ void __launch_bounds__(256) demux_ok_wide_kernel(const unsigned long long* __restrict__ fkeys,
                                                            const unsigned long long* __restrict__ fkeys_hi,
                                                            const unsigned long long* __restrict__ fcounts, unsigned long long nf,
                                                            const unsigned long long* __restrict__ sorted_lo,
                                                            const unsigned long long* __restrict__ sorted_hi,
                                                            const unsigned* __restrict__ sorted_idx, unsigned long long n,
                                                            const unsigned char* __restrict__ type, const int* __restrict__ srow,
                                                            const unsigned char* __restrict__ match, unsigned n_files, unsigned f,
                                                            unsigned char* __restrict__ ok, unsigned char* __restrict__ bad_file,
                                                            int* err_row) {
    const unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x;
    if (i >= nf || (fcounts && fcounts[i] == 0)) return;
    const unsigned long long klo = fkeys[i], khi = fkeys_hi[i];
    unsigned long long lo = 0, hi = n;
    while (lo < hi) {
        const unsigned long long mid = (lo + hi) >> 1;
        const unsigned long long mh = sorted_hi[mid];
        if (mh < khi || (mh == khi && sorted_lo[mid] < klo)) lo = mid + 1;
        else hi = mid;
    }
    if (lo >= n || sorted_lo[lo] != klo || sorted_hi[lo] != khi) return;
    const unsigned idx = sorted_idx[lo];
    const unsigned t = type[idx];
    const unsigned cls = t == 2 ? 4u + static_cast<unsigned>(srow[idx]) : t;
    const unsigned m = match[static_cast<unsigned long long>(cls) * n_files + f];
    if (m == 2) {
        atomicMin(err_row, static_cast<int>(cls) - 4);
    } else if (m == 0) {
        ok[idx] = 0;
        bad_file[f] = 1;
    }
}

}  // namespace frb
