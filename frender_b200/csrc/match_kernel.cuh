// Hot path B: Hamming matcher + classifier + reverse-complement orientation sums.
// One thread per UNIQUE key (F:610 passes the unique dict, not the reads); the packed sample
// sheet sits in shared memory and every thread streams over its rows.
//   mismatches(idx)  = popc( fold3(key ^ row) & field_mask )          (F:226-230, per symbol)
//   fold3(d)         = (d | d>>1 | d>>2) & 0b001001...  -> one bit per differing 3-bit symbol
// N is an ordinary symbol (N==N equal, N!=A); a sheet symbol outside ACGTN is code 7 and can
// never equal a read symbol.  The classifier keeps only what analyze_barcode needs (F:256-284):
// the FIRST matching row per index, the number of rows matching both, and that row.
#pragma once
#include "common.cuh"

namespace frb {

constexpr unsigned long long kFoldLsb = 0x1249249249249249ULL;  // bit 0 of each 3-bit field
constexpr int kMatchThreads = 256;

struct MatchArgs {
    const unsigned long long* keys;    // [n] packed unique keys
    const unsigned long long* counts;  // [n] reads per key
    unsigned long long n;
    const unsigned long long* sheet_fwd;  // [rows] pack(idx1+idx2)
    const unsigned long long* sheet_rc;   // [rows] pack(idx1+revcomp(idx2))
    const int* group;                     // [rows] sample-name group
    const unsigned char* use_rc;          // [rows] or null: pick sheet_rc for that row (F:618-623)
    unsigned rows, l1, l2, n_subs;
    int rc_mode;
    int *m1, *m2, *srow, *m2rc, *srowrc;  // per-key outputs (device, may be null)
    unsigned char *type, *typerc;
    unsigned long long *f_sum, *rc_sum;   // [rows] per group (rc_mode only)
    unsigned* work;                       // [n] indices of the keys with an idx1 match
    unsigned long long* work_n;           // entries in work[]
    DevState* st;
};

__device__ __forceinline__ unsigned long long fold3(unsigned long long d) {
    return (d | (d >> 1) | (d >> 2)) & kFoldLsb;
}

__device__ __forceinline__ void classify_one(int first1, int first2, unsigned both, int both_row, int* m1, int* m2,
                                             int* type, int* srow) {
    if (first1 >= 0 && first2 >= 0) {  // F:259-278
        *m1 = first1;
        *m2 = first2;
        *type = both == 0 ? FRB_TYPE_INDEX_HOP : (both == 1 ? FRB_TYPE_DEMUXABLE : FRB_TYPE_AMBIGUOUS);
        *srow = both == 1 ? both_row : -1;
    } else {  // F:280-284
        *m1 = -1, *m2 = -1, *type = FRB_TYPE_UNDETERMINED, *srow = -1;
    }
}

// ---- pieces every matcher kernel shares ---------------------------------------------------------------------------
// Shape check: idx1 of l1 symbols in 1..5, then '+' and idx2 of l2 symbols in 1..5, then end or another '+' (extra
// parts ignored, F:306); single index: l1 symbols then end.  sym(s) = symbol s of the key, max_syms its capacity.
template <class Sym>
__device__ __forceinline__ bool shape_ok(const MatchArgs& a, unsigned max_syms, Sym sym) {
    bool ok = true;
    const unsigned total = a.l2 ? a.l1 + 1 + a.l2 : a.l1;
    for (unsigned s = 0; s < total; ++s) {
        const unsigned c = sym(s);
        if (a.l2 && s == a.l1) ok &= (c == 6);
        else ok &= (c >= 1 && c <= 5);
    }
    if (total < max_syms) {
        const unsigned nxt = sym(total);
        ok &= a.l2 ? (nxt == 0 || nxt == 6) : (nxt == 0);
    }
    return ok;
}

// A key without an idx1 row is undetermined whatever its idx2 does (F:259, F:280-284).
__device__ __forceinline__ void mark_undetermined(const MatchArgs& a, unsigned long long i) {
    a.m2[i] = -1, a.srow[i] = -1, a.type[i] = FRB_TYPE_UNDETERMINED;
    if (a.rc_mode) a.m2rc[i] = -1, a.srowrc[i] = -1, a.typerc[i] = FRB_TYPE_UNDETERMINED;
}

// Keys of the warp with an idx1 row -> work list, one atomic per warp.  Every lane of the warp calls this.
__device__ __forceinline__ void append_work(const MatchArgs& a, int lane, unsigned long long i, int first1) {
    const unsigned need = __ballot_sync(0xFFFFFFFFu, first1 >= 0);
    if (need) {
        unsigned long long base = 0;
        const int leader = __ffs(need) - 1;
        if (lane == leader) base = atomicAdd(a.work_n, static_cast<unsigned long long>(__popc(need)));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (first1 >= 0) a.work[base + __popc(need & ((1u << lane) - 1u))] = static_cast<unsigned>(i);
    }
}

// Kernel 2's verdict on key i from the rows its sweep found: first idx2 row, rows matching both and the first of
// them (-1: none), as supplied / oriented (f) and reverse-complemented (r, rc_mode only).  rc_mode also adds the
// key's reads to the per-group sums in shared memory (s_f, s_r; s_g = group of every row).
__device__ __forceinline__ void classify_store(const MatchArgs& a, unsigned long long i, int first1, int firstf,
                                               unsigned nf, int rowf, int firstr, unsigned nr, int rowr,
                                               unsigned long long* s_f, unsigned long long* s_r, const int* s_g) {
    int m1, m2, type, srow;
    classify_one(first1, firstf, nf, rowf, &m1, &m2, &type, &srow);
    if (a.rc_mode) {
        int m1r, m2r, typer, srowr;
        classify_one(first1, firstr, nr, rowr, &m1r, &m2r, &typer, &srowr);
        if (m1 < 0) m1 = m1r;  // F:319-323
        if (type == FRB_TYPE_DEMUXABLE && typer == FRB_TYPE_DEMUXABLE && s_g[srow] != s_g[srowr]) {
            type = typer = FRB_TYPE_AMBIGUOUS;  // F:336-349
            srow = srowr = -1;
        }
        const unsigned long long c = a.counts[i];
        if (srow >= 0) atomicAdd(&s_f[s_g[srow]], c);      // F:370-371
        if (srowr >= 0) atomicAdd(&s_r[s_g[srowr]], c);    // F:372-373
        a.m2rc[i] = m2r;
        a.typerc[i] = static_cast<unsigned char>(typer);
        a.srowrc[i] = srowr;
    }
    a.m1[i] = m1;
    a.m2[i] = m2;
    a.type[i] = static_cast<unsigned char>(type);
    a.srow[i] = srow;
}

// The block's per-group sums -> f_sum / rc_sum (rc_mode only).  Every thread of the block calls this.
__device__ __forceinline__ void flush_group_sums(const MatchArgs& a, const unsigned long long* s_f,
                                                 const unsigned long long* s_r) {
    if (a.rc_mode) {
        __syncthreads();
        for (unsigned g = threadIdx.x; g < a.rows; g += blockDim.x) {
            if (s_f[g]) atomicAdd(&a.f_sum[g], s_f[g]);
            if (s_r[g]) atomicAdd(&a.rc_sum[g], s_r[g]);
        }
    }
}

// ---- kernel 1: idx1 sweep over ALL unique keys, fully convergent --------------------------------
// A key whose idx1 matches no row is undetermined whatever its idx2 does (F:259, F:280-284) -- the fate
// of almost every unique key of a real lane (random index pairs dominate the unique set).  Those keys
// are finished here; the others go to a compact work list so that the expensive idx2 / reverse-
// complement sweep (kernel 2) runs with full warps instead of a few live lanes per warp.
__global__ void __launch_bounds__(kMatchThreads) match_idx1_kernel(const MatchArgs a) {
    extern __shared__ __align__(16) unsigned char msmem[];
    unsigned long long* s_a = reinterpret_cast<unsigned long long*>(msmem);
    for (unsigned r = threadIdx.x; r < a.rows; r += blockDim.x) s_a[r] = a.sheet_fwd[r];
    __syncthreads();
    const unsigned long long B1 = ((1ULL << (3 * a.l1)) - 1) & kFoldLsb;
    const unsigned n_subs = a.n_subs;
    const int lane = threadIdx.x & 31;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    const unsigned long long n_up = (a.n + 31) & ~31ULL;
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; i < n_up;
         i += stride) {
        int first1 = -1;
        if (i < a.n) {
            const unsigned long long key = a.keys[i];
            if (a.rows && !shape_ok(a, kMaxSyms, [&](unsigned s) { return static_cast<unsigned>(key >> (3 * s)) & 7u; }))
                raise_error(a.st, FRB_ERR_BAD_LENGTH, key);
            if (a.l1 <= 10) {  // idx1 fits 30 bits: 32-bit compare, one LOP3 folds the three bit planes
                const unsigned m = (1u << (3 * a.l1)) - 1u;
                const unsigned k1 = static_cast<unsigned>(key) & m, b1 = static_cast<unsigned>(B1);
                for (unsigned r = 0; r < a.rows; ++r) {
                    const unsigned d = k1 ^ (static_cast<unsigned>(s_a[r]) & m);
                    const bool h1 = static_cast<unsigned>(__popc((d | (d >> 1) | (d >> 2)) & b1)) <= n_subs;
                    if (h1 && first1 < 0) first1 = r;
                }
            } else {
                for (unsigned r = 0; r < a.rows; ++r) {
                    const bool h1 = static_cast<unsigned>(__popcll(fold3(key ^ s_a[r]) & B1)) <= n_subs;
                    if (h1 && first1 < 0) first1 = r;
                }
            }
            a.m1[i] = first1;
            if (first1 < 0) mark_undetermined(a, i);
        }
        append_work(a, lane, i, first1);
    }
}

// ---- kernel 2: full classification of the keys on the work list ---------------------------------
__global__ void __launch_bounds__(kMatchThreads) match_kernel(const MatchArgs a) {
    extern __shared__ __align__(16) unsigned char msmem[];
    unsigned long long* s_a = reinterpret_cast<unsigned long long*>(msmem);  // idx2 as supplied / oriented
    unsigned long long* s_b = s_a + a.rows;                                  // idx2 reverse-complemented
    unsigned long long* s_f = s_b + a.rows;                                  // per-group forward reads
    unsigned long long* s_r = s_f + a.rows;                                  // per-group rc reads
    int* s_g = reinterpret_cast<int*>(s_r + a.rows);

    for (unsigned r = threadIdx.x; r < a.rows; r += blockDim.x) {
        const bool flip = a.use_rc && a.use_rc[r];
        s_a[r] = flip ? a.sheet_rc[r] : a.sheet_fwd[r];
        s_b[r] = a.sheet_rc[r];
        s_f[r] = 0, s_r[r] = 0;
        s_g[r] = a.group[r];
    }
    __syncthreads();

    // field masks in "one bit per symbol" space
    const unsigned long long B1 = ((1ULL << (3 * a.l1)) - 1) & kFoldLsb;
    const unsigned long long B2 = a.l2 ? ((((1ULL << (3 * a.l2)) - 1) & kFoldLsb) << (3 * (a.l1 + 1))) : 0ULL;
    const unsigned n_subs = a.n_subs;
    const unsigned long long n_work = *a.work_n;

    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    for (unsigned long long j = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; j < n_work;
         j += stride) {
        const unsigned long long i = a.work[j];
        const unsigned long long key = a.keys[i];
        // first idx1 row: from kernel 1, or from the rc pass when this is the oriented second pass of a
        // scan (F:628) -- orientation only changes idx2, and a key the rc pass left without an
        // idx1+idx2 match in either orientation cannot get one from a per-row choice between the two.
        const int first1 = a.m1[i];
        int firstf = -1, firstr = -1, rowf = -1, rowr = -1;
        unsigned nf = 0, nr = 0;
        if (first1 >= 0) {
            for (unsigned r = 0; r < a.rows; ++r) {
                const unsigned long long df = fold3(key ^ s_a[r]);
                const bool h1 = static_cast<unsigned>(__popcll(df & B1)) <= n_subs;
                const bool h2 = a.l2 ? (static_cast<unsigned>(__popcll(df & B2)) <= n_subs) : true;
                if (h2 && firstf < 0) firstf = r;
                if (h1 && h2) {
                    ++nf;
                    if (rowf < 0) rowf = r;
                }
                if (a.rc_mode) {
                    const unsigned long long dr = fold3(key ^ s_b[r]);
                    const bool h3 = static_cast<unsigned>(__popcll(dr & B2)) <= n_subs;
                    if (h3 && firstr < 0) firstr = r;
                    if (h1 && h3) {
                        ++nr;
                        if (rowr < 0) rowr = r;
                    }
                }
            }
        }
        classify_store(a, i, first1, firstf, nf, rowf, firstr, nr, rowr, s_f, s_r, s_g);
    }
    flush_group_sums(a, s_f, s_r);
}

// =================================================================================================
// Candidate rows instead of a sweep over the sheet.  Split an index of l symbols into P = n_subs + 1
// parts: a row within n_subs substitutions of the key agrees EXACTLY with it on at least one part
// (n_subs mismatches cannot touch n_subs + 1 parts).  Per block, a shared-memory hash table maps
// (part number, part value) -> the rows holding that value; a key looks up its P part values, walks the
// short chains and checks every candidate with the full compare of F:226-230.  "First matching row" of the
// reference's ascending sweep is the smallest matching row; a row that agrees on several parts is visited
// through the first of them only.  Same results as the sweep, ~2 candidates per key instead of S rows.
// =================================================================================================
constexpr unsigned kNil = 0xFFFFFFFFu;

struct PartLayout {
    unsigned parts, shift[4], mask[4];  // part p of an index = (idx >> shift[p]) & mask[p]
};
__host__ __device__ inline PartLayout part_layout(unsigned l, unsigned parts) {
    PartLayout L{};
    L.parts = parts;
    for (unsigned p = 0; p < parts && p < 4; ++p) {
        const unsigned b = p * l / parts, e = (p + 1) * l / parts;
        L.shift[p] = 3 * b;
        L.mask[p] = (e - b) >= 10 ? 0x3FFFFFFFu : ((1u << (3 * (e - b))) - 1u);
    }
    return L;
}
// usable when every part is non-empty, the index fits 30 bits and the table fits
__host__ __device__ inline bool parts_usable(unsigned l, unsigned n_subs, unsigned rows, unsigned slots) {
    return l >= 1 && l <= 10 && n_subs <= 3 && n_subs + 1 <= l && static_cast<unsigned long long>(rows) * (n_subs + 1) * 2 <= slots;
}

struct CandTable {
    unsigned* keys;   // [slots] tagged part value + 1, 0 = free
    unsigned* head;   // [slots] first row of the chain
    unsigned* next;   // [rows * parts] next row with the same value of that part
    unsigned* idx;    // [rows] the rows' index values (30 bits)
    unsigned slots;
    PartLayout L;
};
__device__ __forceinline__ unsigned cand_tag(const PartLayout& L, unsigned idx, unsigned p) {
    return (((idx >> L.shift[p]) & L.mask[p]) | (L.parts > 1 ? (p << 30) : 0u)) + 1u;
}
__device__ __forceinline__ unsigned cand_hash(unsigned v, unsigned slots) { return (v * 2654435761u) >> 7 & (slots - 1); }

// all threads of the block; T.idx[] must be filled and visible
__device__ inline void cand_build(const CandTable& T, unsigned rows) {
    for (unsigned i = threadIdx.x; i < T.slots; i += blockDim.x) T.keys[i] = 0, T.head[i] = kNil;
    __syncthreads();
    for (unsigned e = threadIdx.x; e < rows * T.L.parts; e += blockDim.x) {
        const unsigned r = e / T.L.parts, p = e % T.L.parts;
        const unsigned v = cand_tag(T.L, T.idx[r], p);
        unsigned slot = cand_hash(v, T.slots);
        for (;;) {
            const unsigned old = atomicCAS(&T.keys[slot], 0u, v);
            if (old == 0u || old == v) break;
            slot = (slot + 1) & (T.slots - 1);
        }
        T.next[e] = atomicExch(&T.head[slot], r);
    }
    __syncthreads();
}
// f(row) for every row that agrees with `idx` on at least one part, each row once
template <class F>
__device__ __forceinline__ void cand_visit(const CandTable& T, unsigned idx, F&& f) {
    for (unsigned p = 0; p < T.L.parts; ++p) {
        const unsigned v = cand_tag(T.L, idx, p);
        unsigned slot = cand_hash(v, T.slots);
        unsigned k;
        while ((k = T.keys[slot]) != 0u) {
            if (k == v) {
                for (unsigned r = T.head[slot]; r != kNil; r = T.next[r * T.L.parts + p]) {
                    bool earlier = false;  // already visited through a part before p?
                    for (unsigned q = 0; q < p; ++q)
                        earlier |= ((idx ^ T.idx[r]) >> T.L.shift[q] & T.L.mask[q]) == 0u;
                    if (!earlier) f(r);
                }
                break;
            }
            slot = (slot + 1) & (T.slots - 1);
        }
    }
}
__device__ __forceinline__ unsigned hamming30(unsigned a, unsigned b, unsigned field) {
    const unsigned d = a ^ b;
    return static_cast<unsigned>(__popc((d | (d >> 1) | (d >> 2)) & field));
}

// shared-memory footprint of one table
__host__ __device__ inline size_t cand_bytes(unsigned rows, unsigned parts, unsigned slots) {
    return (static_cast<size_t>(slots) * 2 + static_cast<size_t>(rows) * parts + rows) * 4;
}
__device__ inline CandTable cand_carve(unsigned char*& p, unsigned rows, unsigned l, unsigned parts, unsigned slots) {
    CandTable T;
    T.keys = reinterpret_cast<unsigned*>(p);
    T.head = T.keys + slots;
    T.next = T.head + slots;
    T.idx = T.next + static_cast<size_t>(rows) * parts;
    T.slots = slots;
    T.L = part_layout(l, parts);
    p += cand_bytes(rows, parts, slots);
    return T;
}

// ---- kernel 1 with candidates: first idx1 row of every key, work list of the keys that have one ----
__global__ void __launch_bounds__(kMatchThreads) match_idx1_cand_kernel(const MatchArgs a, unsigned slots) {
    extern __shared__ __align__(16) unsigned char msmem[];
    unsigned char* cur = msmem;
    CandTable T = cand_carve(cur, a.rows, a.l1, a.n_subs + 1, slots);
    const unsigned m1mask = (1u << (3 * a.l1)) - 1u;
    for (unsigned r = threadIdx.x; r < a.rows; r += blockDim.x) T.idx[r] = static_cast<unsigned>(a.sheet_fwd[r]) & m1mask;
    __syncthreads();
    cand_build(T, a.rows);
    const unsigned b1 = static_cast<unsigned>(((1ULL << (3 * a.l1)) - 1) & kFoldLsb);
    const unsigned n_subs = a.n_subs;
    const int lane = threadIdx.x & 31;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    const unsigned long long n_up = (a.n + 31) & ~31ULL;
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; i < n_up;
         i += stride) {
        int first1 = -1;
        if (i < a.n) {
            const unsigned long long key = a.keys[i];
            if (!shape_ok(a, kMaxSyms, [&](unsigned s) { return static_cast<unsigned>(key >> (3 * s)) & 7u; }))
                raise_error(a.st, FRB_ERR_BAD_LENGTH, key);
            const unsigned k1 = static_cast<unsigned>(key) & m1mask;
            unsigned best = kNil;
            cand_visit(T, k1, [&](unsigned r) {
                if (hamming30(k1, T.idx[r], b1) <= n_subs && r < best) best = r;
            });
            first1 = best == kNil ? -1 : static_cast<int>(best);
            a.m1[i] = first1;
            if (first1 < 0) mark_undetermined(a, i);
        }
        append_work(a, lane, i, first1);
    }
}

// ---- kernel 2 with candidates: rows whose idx2 matches (as supplied / oriented, and reverse-complemented) ----
__global__ void __launch_bounds__(kMatchThreads) match_cand_kernel(const MatchArgs a, unsigned slots) {
    extern __shared__ __align__(16) unsigned char msmem[];
    unsigned char* cur = msmem;
    unsigned long long* s_f = reinterpret_cast<unsigned long long*>(cur);  // per-group forward reads
    unsigned long long* s_r = s_f + a.rows;                                // per-group rc reads
    int* s_g = reinterpret_cast<int*>(s_r + a.rows);
    unsigned* s_i1 = reinterpret_cast<unsigned*>(s_g + a.rows);            // idx1 of every row
    cur = reinterpret_cast<unsigned char*>(s_i1 + a.rows);
    cur += (16 - (reinterpret_cast<uintptr_t>(cur) & 15)) & 15;
    CandTable Tf = cand_carve(cur, a.rows, a.l2, a.n_subs + 1, slots);
    CandTable Tr = Tf;
    if (a.rc_mode) Tr = cand_carve(cur, a.rows, a.l2, a.n_subs + 1, slots);
    const unsigned m1mask = (1u << (3 * a.l1)) - 1u, m2mask = (1u << (3 * a.l2)) - 1u;
    const unsigned sh2 = 3 * (a.l1 + 1);
    for (unsigned r = threadIdx.x; r < a.rows; r += blockDim.x) {
        const bool flip = a.use_rc && a.use_rc[r];
        const unsigned long long used = flip ? a.sheet_rc[r] : a.sheet_fwd[r];
        s_i1[r] = static_cast<unsigned>(a.sheet_fwd[r]) & m1mask;
        Tf.idx[r] = static_cast<unsigned>(used >> sh2) & m2mask;
        if (a.rc_mode) Tr.idx[r] = static_cast<unsigned>(a.sheet_rc[r] >> sh2) & m2mask;
        s_f[r] = 0, s_r[r] = 0;
        s_g[r] = a.group[r];
    }
    __syncthreads();
    cand_build(Tf, a.rows);
    if (a.rc_mode) cand_build(Tr, a.rows);

    const unsigned b1 = static_cast<unsigned>(((1ULL << (3 * a.l1)) - 1) & kFoldLsb);
    const unsigned b2 = static_cast<unsigned>(((1ULL << (3 * a.l2)) - 1) & kFoldLsb);
    const unsigned n_subs = a.n_subs;
    const unsigned long long n_work = *a.work_n;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    for (unsigned long long j = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; j < n_work;
         j += stride) {
        const unsigned long long i = a.work[j];
        const unsigned long long key = a.keys[i];
        const int first1 = a.m1[i];
        const unsigned k1 = static_cast<unsigned>(key) & m1mask, k2 = static_cast<unsigned>(key >> sh2) & m2mask;
        unsigned firstf = kNil, firstr = kNil, rowf = kNil, rowr = kNil, nf = 0, nr = 0;
        if (first1 >= 0) {
            cand_visit(Tf, k2, [&](unsigned r) {
                if (hamming30(k2, Tf.idx[r], b2) <= n_subs) {        // h2
                    firstf = r < firstf ? r : firstf;
                    if (hamming30(k1, s_i1[r], b1) <= n_subs) {      // h1 && h2
                        ++nf;
                        rowf = r < rowf ? r : rowf;
                    }
                }
            });
            if (a.rc_mode) {
                cand_visit(Tr, k2, [&](unsigned r) {
                    if (hamming30(k2, Tr.idx[r], b2) <= n_subs) {    // h3
                        firstr = r < firstr ? r : firstr;
                        if (hamming30(k1, s_i1[r], b1) <= n_subs) {
                            ++nr;
                            rowr = r < rowr ? r : rowr;
                        }
                    }
                });
            }
        }
        // classify_store written out: called here, it changes how the compiler schedules this kernel's epilogue
        int m1, m2, type, srow;
        classify_one(first1, static_cast<int>(firstf), nf, static_cast<int>(rowf), &m1, &m2, &type, &srow);
        if (a.rc_mode) {
            int m1r, m2r, typer, srowr;
            classify_one(first1, static_cast<int>(firstr), nr, static_cast<int>(rowr), &m1r, &m2r, &typer, &srowr);
            if (m1 < 0) m1 = m1r;  // F:319-323
            if (type == FRB_TYPE_DEMUXABLE && typer == FRB_TYPE_DEMUXABLE && s_g[srow] != s_g[srowr]) {
                type = typer = FRB_TYPE_AMBIGUOUS;  // F:336-349
                srow = srowr = -1;
            }
            const unsigned long long c = a.counts[i];
            if (srow >= 0) atomicAdd(&s_f[s_g[srow]], c);      // F:370-371
            if (srowr >= 0) atomicAdd(&s_r[s_g[srowr]], c);    // F:372-373
            a.m2rc[i] = m2r;
            a.typerc[i] = static_cast<unsigned char>(typer);
            a.srowrc[i] = srowr;
        }
        a.m1[i] = m1;
        a.m2[i] = m2;
        a.type[i] = static_cast<unsigned char>(type);
        a.srow[i] = srow;
    }
    flush_group_sums(a, s_f, s_r);
}

}  // namespace frb

// =================================================================================================
// Wide context: keys of up to 42 symbols as (lo, hi).  Every key is split into an idx1 word (symbols [0, l1)) and
// an idx2 word (symbols [l1 + 1, l1 + 1 + l2)), each <= 21 symbols, and the sweep of match_idx1_kernel /
// match_kernel runs on the split words with one mask per index.  Same shape check, same classification.
// =================================================================================================
namespace frb {

struct WideMatchArgs {
    MatchArgs m;                       // keys / sheet_fwd / sheet_rc hold the lo words
    const unsigned long long* keys_hi;
    const unsigned long long* sheet_fwd_hi;
    const unsigned long long* sheet_rc_hi;
};

// symbols [p, p + l) of the 126-bit key (lo | hi << 63) as one word, l <= 21
__device__ __forceinline__ unsigned long long wide_field(unsigned long long lo, unsigned long long hi, unsigned p, unsigned l) {
    const unsigned __int128 v = static_cast<unsigned __int128>(lo) | (static_cast<unsigned __int128>(hi) << 63);
    return static_cast<unsigned long long>(v >> (3 * p)) & ((1ULL << (3 * l)) - 1ULL);
}

// kernel 1: shape check, first idx1 row, work list
__global__ void __launch_bounds__(kMatchThreads) match_idx1_wide_kernel(const WideMatchArgs w) {
    const MatchArgs& a = w.m;
    extern __shared__ __align__(16) unsigned char msmem[];
    unsigned long long* s_1 = reinterpret_cast<unsigned long long*>(msmem);  // idx1 word of every row
    for (unsigned r = threadIdx.x; r < a.rows; r += blockDim.x) s_1[r] = wide_field(a.sheet_fwd[r], w.sheet_fwd_hi[r], 0, a.l1);
    __syncthreads();
    const unsigned long long B1 = ((1ULL << (3 * a.l1)) - 1) & kFoldLsb;
    const unsigned n_subs = a.n_subs;
    const int lane = threadIdx.x & 31;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    const unsigned long long n_up = (a.n + 31) & ~31ULL;
    for (unsigned long long i = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; i < n_up;
         i += stride) {
        int first1 = -1;
        if (i < a.n) {
            const unsigned long long lo = a.keys[i], hi = w.keys_hi[i];
            if (a.rows &&
                !shape_ok(a, kMaxWideSyms, [&](unsigned s) { return static_cast<unsigned>(wide_field(lo, hi, s, 1)); }))
                raise_error<true>(a.st, FRB_ERR_BAD_LENGTH, Key128{lo, hi});
            const unsigned long long k1 = wide_field(lo, hi, 0, a.l1);
            for (unsigned r = 0; r < a.rows; ++r) {
                const bool h1 = static_cast<unsigned>(__popcll(fold3(k1 ^ s_1[r]) & B1)) <= n_subs;
                if (h1 && first1 < 0) first1 = r;
            }
            a.m1[i] = first1;
            if (first1 < 0) mark_undetermined(a, i);
        }
        append_work(a, lane, i, first1);
    }
}

// kernel 2: full classification of the keys on the work list (rc-mode cross-ambiguity rule and group sums included)
__global__ void __launch_bounds__(kMatchThreads) match_wide_kernel(const WideMatchArgs w) {
    const MatchArgs& a = w.m;
    extern __shared__ __align__(16) unsigned char msmem[];
    unsigned long long* s_1 = reinterpret_cast<unsigned long long*>(msmem);  // idx1
    unsigned long long* s_a = s_1 + a.rows;                                  // idx2 as supplied / oriented
    unsigned long long* s_b = s_a + a.rows;                                  // idx2 reverse-complemented
    unsigned long long* s_f = s_b + a.rows;                                  // per-group forward reads
    unsigned long long* s_r = s_f + a.rows;                                  // per-group rc reads
    int* s_g = reinterpret_cast<int*>(s_r + a.rows);
    const unsigned p2 = a.l1 + 1;
    for (unsigned r = threadIdx.x; r < a.rows; r += blockDim.x) {
        const bool flip = a.use_rc && a.use_rc[r];
        s_1[r] = wide_field(a.sheet_fwd[r], w.sheet_fwd_hi[r], 0, a.l1);
        s_a[r] = flip ? wide_field(a.sheet_rc[r], w.sheet_rc_hi[r], p2, a.l2) : wide_field(a.sheet_fwd[r], w.sheet_fwd_hi[r], p2, a.l2);
        s_b[r] = wide_field(a.sheet_rc[r], w.sheet_rc_hi[r], p2, a.l2);
        s_f[r] = 0, s_r[r] = 0;
        s_g[r] = a.group[r];
    }
    __syncthreads();
    const unsigned long long B1 = ((1ULL << (3 * a.l1)) - 1) & kFoldLsb;
    const unsigned long long B2 = ((1ULL << (3 * a.l2)) - 1) & kFoldLsb;
    const unsigned n_subs = a.n_subs;
    const unsigned long long n_work = *a.work_n;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    for (unsigned long long j = blockIdx.x * static_cast<unsigned long long>(blockDim.x) + threadIdx.x; j < n_work;
         j += stride) {
        const unsigned long long i = a.work[j];
        const unsigned long long lo = a.keys[i], hi = w.keys_hi[i];
        const unsigned long long k1 = wide_field(lo, hi, 0, a.l1), k2 = wide_field(lo, hi, p2, a.l2);
        const int first1 = a.m1[i];
        int firstf = -1, firstr = -1, rowf = -1, rowr = -1;
        unsigned nf = 0, nr = 0;
        if (first1 >= 0) {
            for (unsigned r = 0; r < a.rows; ++r) {
                const bool h1 = static_cast<unsigned>(__popcll(fold3(k1 ^ s_1[r]) & B1)) <= n_subs;
                const bool h2 = a.l2 ? (static_cast<unsigned>(__popcll(fold3(k2 ^ s_a[r]) & B2)) <= n_subs) : true;
                if (h2 && firstf < 0) firstf = r;
                if (h1 && h2) {
                    ++nf;
                    if (rowf < 0) rowf = r;
                }
                if (a.rc_mode) {
                    const bool h3 = static_cast<unsigned>(__popcll(fold3(k2 ^ s_b[r]) & B2)) <= n_subs;
                    if (h3 && firstr < 0) firstr = r;
                    if (h1 && h3) {
                        ++nr;
                        if (rowr < 0) rowr = r;
                    }
                }
            }
        }
        classify_store(a, i, first1, firstf, nf, rowf, firstr, nr, rowr, s_f, s_r, s_g);
    }
    flush_group_sums(a, s_f, s_r);
}

// =================================================================================================
// Which pair of kernels frb_match launches for a sheet shape, and with how much shared memory.
// =================================================================================================
enum MatchPath : int {
    kMatchCand = 0,   // match_idx1_cand_kernel + match_cand_kernel
    kMatchSweep = 1,  // match_idx1_kernel + match_kernel
    kMatchWide = 2,   // match_idx1_wide_kernel + match_wide_kernel
};
constexpr int kMatchSmemMax = 200 * 1024;      // dynamic shared memory allowed to match_kernel and both cand kernels
constexpr int kMatchWideSmemMax = 220 * 1024;  // ... and to match_wide_kernel

struct MatchPlan {
    MatchPath path;
    unsigned slots;     // slots of each candidate table (kMatchCand only, else 0)
    int blocks_per_sm;  // grid of both kernels: at most sm_count * blocks_per_sm blocks of kMatchThreads
};
constexpr MatchPlan kSweepPlan{kMatchSweep, 0, 8};

// Candidate tables whenever both indexes can be split into n_subs + 1 parts and the tables fit (2048 slots while
// rows * parts * 2 <= 2048, else 4096); the sweep for every other narrow shape; wide contexts sweep the split words.
__host__ inline MatchPlan match_plan(unsigned rows, unsigned l1, unsigned l2, unsigned n_subs, bool wide) {
    if (wide) return {kMatchWide, 0, 8};
    const unsigned parts = n_subs + 1;
    const unsigned slots = static_cast<unsigned long long>(rows) * parts * 2 <= 2048 ? 2048u : 4096u;
    if (rows > 0 && l2 > 0 && parts_usable(l1, n_subs, rows, slots) && parts_usable(l2, n_subs, rows, slots))
        return {kMatchCand, slots, 4};
    return kSweepPlan;
}
// dynamic shared memory of kernel 1 (idx1 sweep / table, work list)
__host__ inline size_t match_smem_idx1(const MatchPlan& p, unsigned rows, unsigned n_subs) {
    if (p.path == kMatchCand) return cand_bytes(rows, n_subs + 1, p.slots) + 16;
    return static_cast<size_t>(rows) * 8 + 16;
}
// dynamic shared memory of kernel 2 (classification of the work list)
__host__ inline size_t match_smem_classify(const MatchPlan& p, unsigned rows, unsigned n_subs, bool rc_mode) {
    if (p.path == kMatchCand)
        return static_cast<size_t>(rows) * 24 + 32 + (rc_mode ? 2 : 1) * cand_bytes(rows, n_subs + 1, p.slots);
    if (p.path == kMatchSweep) return static_cast<size_t>(rows) * (4 * 8 + 4) + 16;
    return static_cast<size_t>(rows) * (5 * 8 + 4) + 16;
}

}  // namespace frb
