// Shared device/host definitions: packed-key alphabet, table slot, device control block.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/frender_b200.h"

namespace frb {

// One slot of the open-addressing unique-key table: exactly one 32-byte DRAM sector, so a probe
// and its count/first updates touch a single sector.
struct __align__(32) Slot {
    unsigned long long key;    // packed key, FRB_EMPTY_KEY when free
    unsigned long long first;  // smallest read position seen      (dict insertion order, F:176); next to the key so
                               // that one 16-byte load shows whether an update can lower it at all
    unsigned long long count;  // reads carrying the key           (dict value, F:172-177)
    unsigned long long aux;    // unused
};

// Device-resident control block of a context (zeroed by frb_scan_begin).
struct DevState {
    unsigned long long line_carry;  // lines of the current file consumed by earlier chunks
    unsigned long long n_reads;     // header lines tallied in the current file
    unsigned long long occupied;    // slots claimed in the per-file table
    unsigned long long occupied_total;
    unsigned long long err_pos;     // read ordinal / key of the first error
    unsigned long long scratch;     // generic counter (compaction)
    int err_code;                   // first FRB_ERR_* raised on the device, 0 if none
    int pad;
    unsigned long long chunk_l0;    // lines before the chunk the scan kernel last ran on
    unsigned long long redo_n;      // tiles of that chunk left to scan_redo_kernel
    // speculative (lean) scan path: keys are committed on the text's own line phase and the phase is checked
    // against the newline count afterwards (scan_verify.cuh)
    unsigned long long spec_err_pos;  // composite position of the first parse error seen in a guessed tile
    int spec_err_code;                // ... and its code; promoted to err_code once the guesses are confirmed
    int spec_bad;                     // a guess of the current chunk was wrong: the chunk is redone by count
    unsigned long long err_hi;        // wide context: upper word of the key of the first error (err_pos holds lo)
};

// Slot of a wide context's table (keys of up to 42 symbols, see frender_b200.h): same 32 bytes as Slot, so both
// layouts share one allocation.  (lo, hi) is claimed with one 128-bit compare-and-swap; lo = FRB_EMPTY_KEY is free.
struct __align__(32) WideSlot {
    unsigned long long lo, hi;  // packed key: symbols 0..20 / 21..41
    unsigned long long first;   // smallest read position seen
    unsigned long long count;   // reads carrying the key
};
struct __align__(16) Key128 {
    unsigned long long lo, hi;
};

// Position of a read inside a file as the speculative path records it: (tile index in the file << 13) | index of
// the header among the tile's headers.  Order-preserving in the read ordinal; turned into the ordinal itself when
// the file's table is compacted (first read ordinal of every tile is known once the newline counts are summed).
constexpr int kCompositeShift = 13;  // a 30 KiB tile holds at most 7680 headers (four empty lines each)

constexpr unsigned long long kEmpty = FRB_EMPTY_KEY;
constexpr int kMaxSyms = 21;
constexpr int kMaxWideSyms = 2 * kMaxSyms;
constexpr uint32_t kMaxProbe = 1u << 15;

// Symbol codes.  enc_read(): strict read alphabet, 0 = not allowed.
__host__ __device__ __forceinline__ uint32_t enc_read(uint32_t c) {
    // branch-free: '+'..'T' (0x2B..0x54) index a 3-bit-per-entry table held in two 64-bit words
    // ('+'->6 'A'->1 'C'->2 'G'->3 'N'->5 'T'->4, everything else 0)
    const uint32_t d = c - 0x2Bu;
    const unsigned long long lo = 6ULL;                                              // entries 0..20
    const unsigned long long hi = (1ULL << 3) | (2ULL << 9) | (3ULL << 21) | (5ULL << 42) | (4ULL << 60);  // 21..41
    const unsigned long long word = d < 21u ? lo : hi;
    const uint32_t sh = 3u * (d < 21u ? d : d - 21u);
    return d <= 41u ? static_cast<uint32_t>(word >> (sh & 63u)) & 7u : 0u;
}
__host__ __device__ __forceinline__ char dec_sym(uint32_t code) {
    const char t[8] = {0, 'A', 'C', 'G', 'T', 'N', '+', '?'};
    return t[code & 7];
}

__host__ __device__ __forceinline__ unsigned long long hash64(unsigned long long k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdULL;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ULL;
    k ^= k >> 33;
    return k;
}

// Demux parser: kBadKeyBase + (-FRB_ERR_*) in place of a key whose header line did not parse.  Only the router
// knows whether that record is routed at all (the last record of a chunk may be cut anywhere) and reports it then.
constexpr unsigned long long kBadKeyBase = ~0ULL - 256ULL;

#ifdef __CUDACC__
__device__ __forceinline__ void raise_error(DevState* st, int code, unsigned long long pos) {
    if (atomicCAS(&st->err_code, 0, code) == 0) st->err_pos = pos;
}

// count += cnt, first = min(first, pos) for `key`, inserting it if new.  Linear probing.
// Cold path (collisions, first insertions that lost a race): out of line, so that the many places that
// may need it do not each carry a copy of the probing loop (the scan kernels' SASS has to stay near the
// instruction cache size).
__device__ __noinline__ void table_add(Slot* __restrict__ tab, unsigned long long mask,
                                          unsigned long long key, unsigned long long cnt,
                                          unsigned long long pos, unsigned long long* occupied,
                                          DevState* st) {
    unsigned long long h = hash64(key) & mask;
    for (uint32_t probe = 0; probe < kMaxProbe; ++probe) {
        unsigned long long k = *reinterpret_cast<volatile unsigned long long*>(&tab[h].key);
        if (k == kEmpty) {
            k = atomicCAS(&tab[h].key, kEmpty, key);
            if (k == kEmpty) {
                atomicAdd(occupied, 1ULL);
                k = key;
            }
        }
        if (k == key) {
            atomicAdd(&tab[h].count, cnt);
            atomicMin(&tab[h].first, pos);
            return;
        }
        h = (h + 1) & mask;
    }
    raise_error(st, FRB_ERR_TABLE_FULL, key);
}

// Wide keys: the first error also records the key's upper word.
__device__ __forceinline__ void raise_error_wide(DevState* st, int code, unsigned long long pos, unsigned long long hi) {
    if (atomicCAS(&st->err_code, 0, code) == 0) st->err_pos = pos, st->err_hi = hi;
}

// table_add for a wide context, inlined (a call would spill in the scan kernels).  A key with hi = 0 hashes as its
// narrow twin.  One 16-byte load per probe;
// a free slot is claimed with one 128-bit compare-and-swap on (lo, hi).
__device__ __forceinline__ void table_add_wide(WideSlot* __restrict__ tab, unsigned long long mask, unsigned long long lo,
                                            unsigned long long hi, unsigned long long cnt, unsigned long long pos,
                                            unsigned long long* occupied, DevState* st) {
    unsigned long long h = hash64(lo ^ (hi * 0x9E3779B97F4A7C15ULL)) & mask;
    for (uint32_t probe = 0; probe < kMaxProbe; ++probe) {
        unsigned long long klo, khi;
        asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(klo), "=l"(khi) : "l"(&tab[h].lo));
        if (klo == kEmpty) {
            const Key128 old = atomicCAS(reinterpret_cast<Key128*>(&tab[h].lo), Key128{kEmpty, 0ULL}, Key128{lo, hi});
            klo = old.lo, khi = old.hi;
            if (klo == kEmpty) {
                atomicAdd(occupied, 1ULL);
                klo = lo, khi = hi;
            }
        }
        if (klo == lo && khi == hi) {
            atomicAdd(&tab[h].count, cnt);
            atomicMin(&tab[h].first, pos);
            return;
        }
        h = (h + 1) & mask;
    }
    raise_error_wide(st, FRB_ERR_TABLE_FULL, lo, hi);
}
#endif

}  // namespace frb
