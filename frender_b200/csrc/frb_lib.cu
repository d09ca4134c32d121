// C-ABI of frender_b200 (see include/frender_b200.h).  Host-side orchestration only: streams,
// staging buffers, launches, D2H of results.  No CPU compute path exists here by design.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <dlfcn.h>
#include <zlib.h>

#include "common.cuh"
#include "gz_kernels.cuh"
#include "match_kernel.cuh"
#include "route_kernel.cuh"
#include "scan_common.cuh"
#include "scan_ws_kernel.cuh"
#include "scan_spec_kernel.cuh"
#include "scan_verify.cuh"
#include "synth_kernel.cuh"
#include "table_kernels.cuh"

using namespace frb;

namespace {

constexpr int kHostStages = 3;
thread_local std::string g_last_error;

struct KeyList {  // device arrays of one (key,count,first) list
    unsigned long long *keys = nullptr, *counts = nullptr, *first = nullptr;
    unsigned long long* keys_hi = nullptr;  // upper key words, wide context only
    uint64_t n = 0, reads = 0;
    uint32_t ordinal = 0;
    bool sorted = true;   // in first-appearance order (a file's list is sorted when somebody first needs the order)
    int first_bits = 64;  // significant bits of `first` (passes of that sort)
};

struct ProfPair {
    cudaEvent_t a, b;
    int cls;
};

}  // namespace

struct frb_ctx {
    int device = 0, sm_count = 0;
    cudaStream_t compute = nullptr, copy = nullptr;
    uint32_t log2 = 0;
    uint64_t cap = 0;
    bool wide = false;  // keys of up to 42 symbols: WideSlot tables, (lo, hi) lists (frb_set_key_width)
    Slot *file_tab = nullptr, *total_tab = nullptr;
    DevState* st = nullptr;
    DevState* st_host = nullptr;  // pinned mirror
    unsigned long long* status = nullptr;
    unsigned int* redo = nullptr;  // tiles left to scan_redo_kernel (same capacity as status)
    size_t status_cap = 0;
    // speculative scan path: first read ordinal of every tile of the current file (composite -> ordinal)
    unsigned long long* tile_first = nullptr;
    size_t tile_first_cap = 0;
    uint64_t file_tiles = 0;            // tiles of the current file scanned so far
    int file_composite = -1;            // -1 undecided, 0 read ordinals, 1 composite positions in file_tab
    unsigned long long* block_sums = nullptr;
    size_t block_sums_cap = 0;
    // host-chunk staging
    unsigned char* stage[kHostStages] = {nullptr, nullptr, nullptr};
    cudaEvent_t stage_copied[kHostStages], stage_done[kHostStages];
    size_t stage_cap = 0;
    int stage_next = 0;
    // gz pipeline ring (pinned)
    unsigned char* ring[kHostStages] = {nullptr, nullptr, nullptr};
    // results
    std::vector<KeyList> files;
    KeyList total;
    unsigned long long* skip_slot = nullptr;  // device word: where the text begins in the buffer of a batch segment
    bool total_ready = false, in_file = false;
    size_t merged_upto = 0;        // file lists already folded into total_tab
    bool ext_merged = false;       // lists from other contexts were folded in (frb_total_merge)
    bool sharded = false;          // total holds this rank's share of a sharded merge (no table behind it)
    // exchange buffers of the sharded merge: kept (grow-only) so that NCCL sees the same addresses every step
    unsigned long long* xchg[3] = {nullptr, nullptr, nullptr};  // send parts, received parts, histograms
    size_t xchg_cap[3] = {0, 0, 0};
    bool total_tab_clean = true;   // total_tab holds no keys
    uint32_t cur_ordinal = 0;
    uint64_t cur_limit = ~0ULL;
    // sheet
    unsigned long long *sheet_fwd = nullptr, *sheet_rc = nullptr;
    unsigned long long *sheet_fwd_hi = nullptr, *sheet_rc_hi = nullptr;
    int* sheet_group = nullptr;
    unsigned char* sheet_use_rc = nullptr;
    unsigned long long *f_sum = nullptr, *rc_sum = nullptr;
    uint32_t rows = 0, l1 = 0, l2 = 0;
    // matcher outputs (device, grown on demand)
    int *m1 = nullptr, *m2 = nullptr, *srow = nullptr, *m2rc = nullptr, *srowrc = nullptr;
    unsigned char *type = nullptr, *typerc = nullptr;
    unsigned* work = nullptr;             // keys with an idx1 match (matcher work list)
    unsigned long long* work_n = nullptr;
    uint64_t match_cap = 0;
    uint64_t total_gen = 0, sheet_gen = 0;            // bumped whenever the total list / sheet changes
    uint64_t m1_total_gen = ~0ULL, m1_sheet_gen = ~0ULL;  // what c->m1 currently describes
    uint32_t m1_n_subs = ~0u;
    bool m1_from_rc = false;                              // ... and it came from an rc_mode pass
    // temp for sort
    void* cub_tmp = nullptr;
    size_t cub_tmp_bytes = 0;
    // route
    Slot* route_tab = nullptr;
    uint64_t route_cap = 0;
    uint32_t n_sinks = 0;
    struct RouteStreamHolder* route = nullptr;  // the demux stream (frb_route.inl)
    // device inflate (frb_gz.inl)
    struct GzBuffersHolder* gzbuf = nullptr;
    // synth
    SynthArgs synth{};
    unsigned *synth_i7 = nullptr, *synth_i5 = nullptr;
    unsigned long long* synth_cdf = nullptr;
    unsigned long long *synth_len = nullptr, *synth_off = nullptr;
    uint64_t synth_cap = 0;
    bool synth_ready = false;
    // nccl
    void* nccl_comm = nullptr;
    int rank = 0, n_ranks = 1;
    // measurement
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    bool prof = false;
    std::vector<ProfPair> prof_pending;
    std::vector<ProfPair> prof_free;
    double prof_ms[FRB_K_NUM] = {0};
    uint64_t prof_n[FRB_K_NUM] = {0};
    uint64_t launches = 0;
    uint64_t gz_device_files = 0;  // files inflated on the device
    std::string err;
};

namespace {

int fail(frb_ctx* c, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    if (c) c->err = buf;
    return code;
}

#define CU(c, call)                                                                         \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return fail(c, FRB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                        __LINE__);                                                          \
    } while (0)
#define TRY(expr)                   \
    do {                            \
        int rc_ = (expr);           \
        if (rc_ != FRB_OK) return rc_; \
    } while (0)

struct ProfScope {  // brackets a kernel (class) with events when profiling is on
    frb_ctx* c;
    ProfPair p{};
    bool on;
    ProfScope(frb_ctx* ctx, int cls) : c(ctx), on(ctx->prof) {
        if (!on) return;
        if (!c->prof_free.empty()) {
            p = c->prof_free.back();
            c->prof_free.pop_back();
        } else {
            cudaEventCreate(&p.a);
            cudaEventCreate(&p.b);
        }
        p.cls = cls;
        cudaEventRecord(p.a, c->compute);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(p.b, c->compute);
        c->prof_pending.push_back(p);
    }
};

void prof_collect(frb_ctx* c) {  // call after the compute stream is idle
    for (auto& p : c->prof_pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            c->prof_ms[p.cls] += ms;
            c->prof_n[p.cls] += 1;
        }
        c->prof_free.push_back(p);
    }
    c->prof_pending.clear();
}

int grid_for(uint64_t n, int threads, int sm_count, int per_sm) {
    uint64_t blocks = (n + threads - 1) / threads;
    uint64_t cap = static_cast<uint64_t>(sm_count) * per_sm;
    return static_cast<int>(std::max<uint64_t>(1, std::min(blocks, cap)));
}

int device_error_check(frb_ctx* c) {  // compute stream must be idle
    CU(c, cudaMemcpyAsync(c->st_host, c->st, sizeof(DevState), cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaStreamSynchronize(c->compute));
    prof_collect(c);
    const int code = c->st_host->err_code;
    if (code == 0) return FRB_OK;
    const unsigned long long pos = c->st_host->err_pos;
    char keytxt[48];
    frb_unpack_key2(pos, c->wide ? c->st_host->err_hi : 0ULL, keytxt);
    // clear so that the context stays usable after the caller handled the error
    CU(c, cudaMemsetAsync(&c->st->err_code, 0, sizeof(int), c->compute));
    switch (code) {
        case FRB_ERR_BAD_HEADER:
            return fail(c, code, "read %llu: header line has no second space-separated field", pos);
        case FRB_ERR_BAD_ALPHABET:
            return fail(c, code, "read %llu: index field holds a symbol outside ACGTN+", pos);
        case FRB_ERR_KEY_TOO_LONG:
            return fail(c, code, "read %llu: index field longer than %d symbols", pos, c->wide ? kMaxWideSyms : kMaxSyms);
        case FRB_ERR_TABLE_FULL:
            return fail(c, code, "unique-key table full (2^%u slots): frb_resize_tables / FRENDER_TABLE_LOG2 for a larger one",
                        c->log2);
        case FRB_ERR_BAD_LENGTH:
            return fail(c, code, "Barcode %s doesn't match the index lengths of the sample sheet (%u+%u)", keytxt,
                        c->l1, c->l2);
        case FRB_ERR_KEY_NOT_FOUND:
            return fail(c, code, "Couldn't find barcode %s in supplied frender result file!", keytxt);
        default:
            return fail(c, code, "device error %d at %llu", code, pos);
    }
}

// Stream-ordered allocations for everything sized by the number of unique keys: served from the
// device's memory pool (release threshold = never), so a steady-state step makes no driver calls
// that synchronise the device.
template <typename T>
int dmalloc(frb_ctx* c, T** p, size_t bytes) {
    CU(c, cudaMallocAsync(reinterpret_cast<void**>(p), bytes ? bytes : 8, c->compute));
    return FRB_OK;
}
int dfree(frb_ctx* c, void* p) {
    if (p) CU(c, cudaFreeAsync(p, c->compute));
    return FRB_OK;
}

int free_list(frb_ctx* c, KeyList& l) {
    TRY(dfree(c, l.keys));
    TRY(dfree(c, l.counts));
    TRY(dfree(c, l.first));
    TRY(dfree(c, l.keys_hi));
    l = KeyList{};
    return FRB_OK;
}

int clear_table(frb_ctx* c, Slot* tab) {
    ProfScope ps(c, FRB_K_OTHER);
    if (c->wide)
        clear_wide_table_kernel<<<grid_for(c->cap, 256, c->sm_count, 16), 256, 0, c->compute>>>(reinterpret_cast<WideSlot*>(tab), c->cap);
    else
        clear_table_kernel<<<grid_for(c->cap, 256, c->sm_count, 16), 256, 0, c->compute>>>(tab, c->cap);
    c->launches++;
    CU(c, cudaGetLastError());
    return FRB_OK;
}

int ensure_cub_tmp(frb_ctx* c, size_t bytes) {
    if (bytes <= c->cub_tmp_bytes) return FRB_OK;
    bytes += bytes / 2;
    if (c->cub_tmp) CU(c, cudaFree(c->cub_tmp));
    c->cub_tmp = nullptr;
    c->cub_tmp_bytes = 0;
    CU(c, cudaMalloc(&c->cub_tmp, bytes));
    c->cub_tmp_bytes = bytes;
    return FRB_OK;
}

// Dense (key,count,first) arrays in arbitrary order -> list sorted by `first` (first-appearance order,
// F:172-177 / F:199-205).  Takes over k0/c0/f0 (pool allocations) and frees them.
int unsorted_to_sorted_list(frb_ctx* c, unsigned long long* k0, unsigned long long* c0, unsigned long long* f0,
                            uint64_t n, KeyList* out, int first_bits = 64, unsigned long long* h0 = nullptr) {
    out->n = n;
    unsigned *i0 = nullptr, *i1 = nullptr;
    if (n) {
        TRY(dmalloc(c, &i0, n * 4));
        TRY(dmalloc(c, &i1, n * 4));
        TRY(dmalloc(c, &out->keys, n * 8));
        TRY(dmalloc(c, &out->counts, n * 8));
        TRY(dmalloc(c, &out->first, n * 8));
        ProfScope ps(c, FRB_K_EXPORT);
        iota_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(i0, n);
        size_t tmp = 0;
        // first_bits: significant bits of `first` (a file's read ordinals stay below 2^40: five radix passes
        // instead of eight)
        CU(c, cub::DeviceRadixSort::SortPairs(nullptr, tmp, f0, out->first, i0, i1, static_cast<int>(n), 0,
                                              first_bits, c->compute));
        TRY(ensure_cub_tmp(c, tmp));
        CU(c, cub::DeviceRadixSort::SortPairs(c->cub_tmp, tmp, f0, out->first, i0, i1, static_cast<int>(n), 0,
                                              first_bits, c->compute));
        gather2_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(i1, k0, c0, out->keys,
                                                                                       out->counts, n);
        c->launches += 9;  // iota, cub radix sort passes (approximate), gather
        if (h0) {  // a wide list: the upper key words follow the same permutation
            TRY(dmalloc(c, &out->keys_hi, n * 8));
            gather1_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(i1, h0, out->keys_hi, n);
            c->launches++;
        }
        CU(c, cudaGetLastError());
    }
    TRY(dfree(c, k0));
    TRY(dfree(c, c0));
    TRY(dfree(c, f0));
    TRY(dfree(c, h0));
    if (i0) TRY(dfree(c, i0));
    if (i1) TRY(dfree(c, i1));
    return FRB_OK;
}

// A list that came out of a table in slot order -> first-appearance order, in place.
int ensure_sorted(frb_ctx* c, KeyList& l) {
    if (l.sorted || l.n == 0) {
        l.sorted = true;
        return FRB_OK;
    }
    KeyList tmp = l;
    KeyList out = l;
    out.keys = out.counts = out.first = out.keys_hi = nullptr;
    TRY(unsorted_to_sorted_list(c, tmp.keys, tmp.counts, tmp.first, tmp.n, &out, l.first_bits, tmp.keys_hi));  // frees tmp's arrays
    out.sorted = true;
    l = out;
    return FRB_OK;
}

// Table -> list sorted by `first`.
int table_to_sorted_list(frb_ctx* c, Slot* tab, uint64_t n, KeyList* out, int first_bits = 64,
                         const unsigned long long* tile_first = nullptr) {
    out->n = n;
    if (n == 0) return FRB_OK;
    if (n >= (1ULL << 32)) return fail(c, FRB_ERR_ARG, "more than 2^32 unique keys");
    unsigned long long *k0 = nullptr, *c0 = nullptr, *f0 = nullptr, *h0 = nullptr;
    TRY(dmalloc(c, &k0, n * 8));
    TRY(dmalloc(c, &c0, n * 8));
    TRY(dmalloc(c, &f0, n * 8));
    if (c->wide) TRY(dmalloc(c, &h0, n * 8));
    {
        ProfScope ps(c, FRB_K_EXPORT);
        CU(c, cudaMemsetAsync(&c->st->scratch, 0, 8, c->compute));
        if (c->wide)
            compact_wide_table_kernel<<<grid_for(c->cap, 256, c->sm_count, 16), 256, 0, c->compute>>>(
                reinterpret_cast<const WideSlot*>(tab), c->cap, k0, h0, c0, f0, &c->st->scratch, n);
        else
            compact_table_kernel<<<grid_for(c->cap, 256, c->sm_count, 16), 256, 0, c->compute>>>(
                tab, c->cap, k0, c0, f0, &c->st->scratch, n, tile_first);
        c->launches++;
        CU(c, cudaGetLastError());
    }
    return unsorted_to_sorted_list(c, k0, c0, f0, n, out, first_bits, h0);
}

// The same when the number of occupied slots is not known: one pass over the table compacts and counts at once
// (bound = an upper limit of the occupied slots, which sizes the pool allocations).
int table_to_sorted_list_counting(frb_ctx* c, Slot* tab, uint64_t bound, KeyList* out, int first_bits,
                                  const unsigned long long* tile_first) {
    bound = std::max<uint64_t>(std::min<uint64_t>(bound, c->cap), 1);
    if (bound >= (1ULL << 32)) return fail(c, FRB_ERR_ARG, "more than 2^32 unique keys");
    unsigned long long *k0 = nullptr, *c0 = nullptr, *f0 = nullptr, *h0 = nullptr;
    TRY(dmalloc(c, &k0, bound * 8));
    TRY(dmalloc(c, &c0, bound * 8));
    TRY(dmalloc(c, &f0, bound * 8));
    if (c->wide) TRY(dmalloc(c, &h0, bound * 8));
    {
        ProfScope ps(c, FRB_K_EXPORT);
        CU(c, cudaMemsetAsync(&c->st->scratch, 0, 8, c->compute));
        if (c->wide)
            compact_wide_table_kernel<<<grid_for(c->cap, 256, c->sm_count, 16), 256, 0, c->compute>>>(
                reinterpret_cast<const WideSlot*>(tab), c->cap, k0, h0, c0, f0, &c->st->scratch, bound);
        else
            compact_table_kernel<<<grid_for(c->cap, 256, c->sm_count, 16), 256, 0, c->compute>>>(
                tab, c->cap, k0, c0, f0, &c->st->scratch, bound, tile_first);
        c->launches++;
        CU(c, cudaGetLastError());
    }
    CU(c, cudaStreamSynchronize(c->compute));
    TRY(device_error_check(c));
    const uint64_t n = c->st_host->scratch;
    if (n > bound) return fail(c, FRB_ERR_STATE, "more occupied slots (%llu) than reads scanned (%llu)", (unsigned long long)n,
                               (unsigned long long)bound);
    // left in slot order: sorted by first appearance when somebody needs the order (ensure_sorted); a sharded
    // merge does not
    out->keys = k0, out->counts = c0, out->first = f0, out->keys_hi = h0, out->n = n;
    out->sorted = false;
    out->first_bits = first_bits;
    return FRB_OK;
}

int launch_scan(frb_ctx* c, const unsigned char* dev, uint64_t nbytes, uint64_t line_base, int rule,
                unsigned long long* keys_out, unsigned long long* rec_off_out, Slot* table, uint64_t pos_base,
                uint64_t out_cap = ~0ULL, const unsigned long long* skip_ptr = nullptr) {
    if (nbytes == 0) return FRB_OK;
    if (reinterpret_cast<uintptr_t>(dev) & 15) return fail(c, FRB_ERR_ARG, "chunk pointer must be 16-byte aligned");
    // FRB_SCAN_SPEC=0: the general (look-back) kernel everywhere -- A/B switch
    static const bool lean_ok = !(getenv("FRB_SCAN_SPEC") && atoi(getenv("FRB_SCAN_SPEC")) == 0);
    const uint64_t tile = static_cast<uint64_t>(WsTile::tile);
    const uint64_t n_tiles = (nbytes + tile - 1) / tile;
    if (n_tiles >= 0xFFFFFFFFULL || nbytes >= (1ULL << 40)) return fail(c, FRB_ERR_ARG, "chunk too large");
    if (n_tiles + 1 > c->status_cap) {
        if (c->status) CU(c, cudaFree(c->status));
        c->status = nullptr;
        c->status_cap = 0;
        const size_t want = std::max<size_t>(n_tiles + 1, 1 << 16);
        CU(c, cudaMalloc(&c->status, want * 8));
        if (c->redo) CU(c, cudaFree(c->redo));
        c->redo = nullptr;
        CU(c, cudaMalloc(&c->redo, want * 4));
        c->status_cap = want;
    }
    ScanArgs a{};
    a.data = dev;
    a.nbytes = nbytes;
    a.use_carry = (line_base == FRB_CARRY);
    a.line_base = a.use_carry ? 0 : line_base;
    a.read_limit = c->cur_limit;
    a.pos_base = pos_base;
    a.table = table;
    a.table_mask = c->cap - 1;
    a.status = c->status;
    a.st = c->st;
    a.keys_out = keys_out;
    a.rec_off_out = rec_off_out;
    a.out_cap = out_cap;
    a.skip_ptr = skip_ptr;
    a.n_tiles = static_cast<unsigned>(n_tiles);
    a.rule = rule;
    static const bool no_guess = getenv("FRB_SCAN_NO_GUESS") != nullptr;
    a.no_guess = no_guess;
    a.redo = c->redo;
    a.tile_bytes = static_cast<unsigned>(tile);
    a.pat_nl = 0x0A0A0A0Au;
    a.pat_sp = 0x20202020u;
    CU(c, cudaMemsetAsync(&c->st->redo_n, 0, 8, c->compute));
    static unsigned long long* timing = nullptr;
    if (getenv("FRB_SCAN_TIMING")) {
        if (!timing) cudaMalloc(&timing, 2048);
        cudaMemsetAsync(timing, 0, 2048, c->compute);
        a.timing = timing;
    }
    // the lean (speculative) instantiation serves the tally of whole files: scan rule, no per-read outputs, no -s
    static const bool probe = getenv("FRB_SCAN_TIMING") && strcmp(getenv("FRB_SCAN_TIMING"), "spec") == 0;
    const bool lean = !c->wide && lean_ok && (!a.timing || probe) && !no_guess && rule == FRB_RULE_SCAN && !keys_out && !rec_off_out && !skip_ptr &&
                      c->cur_limit == ~0ULL && table != nullptr && table == c->file_tab && c->in_file;
    if (table == c->file_tab && c->in_file) {
        if (c->file_composite < 0) c->file_composite = lean ? 1 : 0;
        if (c->file_composite != (lean ? 1 : 0)) return fail(c, FRB_ERR_STATE, "chunks of one file must use one scan mode");
    }
    const int grid = static_cast<int>(std::min<uint64_t>(n_tiles, static_cast<uint64_t>(c->sm_count) * WsTile::ctas));
    if (!lean) {
        CU(c, cudaMemsetAsync(c->status, 0, (n_tiles + 1) * 8, c->compute));
        ProfScope ps(c, FRB_K_SCAN);
        // tiles the kernel left out (empty list unless the input is not well-formed FASTQ or has lines shorter
        // than 24 bytes on average) go to the redo kernel
        if (c->wide && rule != kRuleOffsetsOnly) {  // record offsets alone need no key of either width
            scan_ws_kernel<WsTileWide><<<grid, WsTileWide::threads, WsTileWide::smem, c->compute>>>(a);
            scan_redo_wide_kernel<<<c->sm_count, 64, 0, c->compute>>>(a);
        } else {
            scan_ws_kernel<WsTile><<<grid, WsTile::threads, WsTile::smem, c->compute>>>(a);
            scan_redo_kernel<<<c->sm_count, 64, 0, c->compute>>>(a);
        }
        c->launches += 2;
    } else {
        // room for the first read ordinal of every tile of the file
        if (c->file_tiles + n_tiles > c->tile_first_cap) {
            const size_t want = std::max<size_t>((c->file_tiles + n_tiles) * 2, 1 << 16);
            unsigned long long* grown = nullptr;
            CU(c, cudaMalloc(&grown, want * 8));
            if (c->file_tiles)
                CU(c, cudaMemcpyAsync(grown, c->tile_first, c->file_tiles * 8, cudaMemcpyDeviceToDevice, c->compute));
            CU(c, cudaStreamSynchronize(c->compute));
            if (c->tile_first) CU(c, cudaFree(c->tile_first));
            c->tile_first = grown;
            c->tile_first_cap = want;
        }
        const unsigned n_blocks = static_cast<unsigned>((n_tiles + kVerifyTiles - 1) / kVerifyTiles);
        if (n_blocks > c->block_sums_cap) {
            if (c->block_sums) CU(c, cudaFree(c->block_sums));
            c->block_sums = nullptr;
            c->block_sums_cap = 0;
            const size_t want = std::max<size_t>(n_blocks * 2, 1024);
            CU(c, cudaMalloc(&c->block_sums, want * 8));
            c->block_sums_cap = want;
        }
        a.tile_base = c->file_tiles;
        a.tile_first = c->tile_first;
        a.composite = 1;
        CU(c, cudaMemsetAsync(c->status, 0, 8, c->compute));           // the ticket counter
        CU(c, cudaMemsetAsync(&c->st->spec_err_pos, 0, 16, c->compute));  // spec_err_pos, spec_err_code, spec_bad
        {
            ProfScope ps(c, FRB_K_SCAN);
            if (probe) scan_spec_kernel<WsTile, true><<<grid, WsTile::threads, WsTile::smem, c->compute>>>(a);
            else scan_spec_kernel<WsTile><<<grid, WsTile::threads, WsTile::smem, c->compute>>>(a);
        }
        {   // the line phase of every tile by count: checks the guesses, lists the tiles without one
            ProfScope ps(c, FRB_K_VERIFY);
            unsigned long long* info = c->status + 1;
            const unsigned nt = static_cast<unsigned>(n_tiles);
            spec_sum_kernel<<<n_blocks, kVerifyTiles, 0, c->compute>>>(info, nt, c->block_sums);
            spec_scan_kernel<<<1, kVerifyTiles, 0, c->compute>>>(c->block_sums, n_blocks, info, nt, a.line_base, a.use_carry, c->st);
            spec_verify_kernel<<<n_blocks, kVerifyTiles, 0, c->compute>>>(info, nt, c->block_sums, c->st,
                                                                          c->tile_first + c->file_tiles, c->redo);
            // a wrong guess (input that is not well-formed FASTQ): take the chunk's guessed keys out of the
            // table again, forget the positions it may have set, and let scan_redo_kernel redo every tile by
            // count.  All three return at once for an ordinary chunk.
            CU(c, cudaMemsetAsync(c->status, 0, 8, c->compute));
            ScanArgs neg = a;
            neg.negate = 1;
            scan_spec_kernel<WsTile><<<grid, WsTile::threads, WsTile::smem, c->compute>>>(neg);
            spec_reset_first_kernel<<<grid_for(c->cap, 256, c->sm_count, 16), 256, 0, c->compute>>>(
                table, c->cap, c->file_tiles << kCompositeShift, c->st);
            scan_redo_kernel<<<c->sm_count, 64, 0, c->compute>>>(a);
        }
        c->file_tiles += n_tiles;
        c->launches += 7;
    }
    CU(c, cudaGetLastError());
    if (a.timing) {
        unsigned long long h[256];
        cudaStreamSynchronize(c->compute);
        cudaMemcpy(h, a.timing, 2048, cudaMemcpyDeviceToHost);
        if (probe) {
            const char* hn[4] = {"X0 wake-up lag", "X1 wake-up lag", "X2 wake-up lag", "issue->count-start"};
            for (int w = 0; w < 3; ++w)
                fprintf(stderr, "PHASES X%d per tile: loads+arrive %.0f parse %.0f finish %.0f fold+slot-load %.0f  waiting %.0f\n", w,
                        (double)h[160 + 8 * w] / (double)h[9], (double)h[161 + 8 * w] / (double)h[9],
                        (double)h[162 + 8 * w] / (double)h[9], (double)h[163 + 8 * w] / (double)h[9],
                        (double)h[164 + 8 * w] / (double)h[9]);
            for (int k = 0; k < 4; ++k) {
                fprintf(stderr, "HIST %s (500-cycle bins):", hn[k]);
                for (int b = 0; b < 32; ++b) fprintf(stderr, " %llu", h[16 + 32 * k + b]);
                fprintf(stderr, "\n");
            }
        }
        const char* names_ws[9] = {"C:wait-bytes", "C:count", "X:wait+refill", "K:lookback", "K:wait-batch", "-", "K:commit",
                                   "X:parse_header", "X:send"};
        const char* names_spec[9] = {"issue->count-start", "count", "counted->released", "released->driver", "counted->seen",
                                     "-", "-", "-", "-"};
        const char** names = probe ? names_spec : names_ws;
        double sum = 0;
        for (int i = 0; i < 9; ++i) sum += static_cast<double>(h[i]);
        const double tiles = h[9] ? static_cast<double>(h[9]) : 1.0;
        fprintf(stderr, "SCAN TIMING tiles %llu cycles/tile %.0f:", h[9], sum / tiles);
        for (int i = 0; i < 9; ++i) fprintf(stderr, " %s %.0f", names[i], (double)h[i] / tiles);
        fprintf(stderr, "\n");
    }
    return FRB_OK;
}

int ensure_stages(frb_ctx* c) {
    if (c->stage[0]) return FRB_OK;
    const char* env = getenv("FRB_STAGE_MB");
    c->stage_cap = static_cast<size_t>(env ? atoi(env) : 64) << 20;
    for (int i = 0; i < kHostStages; ++i) {
        CU(c, cudaMalloc(&c->stage[i], c->stage_cap + 64));
        CU(c, cudaEventCreateWithFlags(&c->stage_copied[i], cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&c->stage_done[i], cudaEventDisableTiming));
    }
    return FRB_OK;
}

}  // namespace

#include "frb_gz.inl"
struct GzBuffersHolder {
    GzBuffers b;
};

static void route_stream_destroy(frb_ctx* c);  // frb_route.inl

// ============================================================================================
extern "C" {

int frb_version(void) { return 200; }

int frb_device_count(int* n) {
    cudaError_t e = cudaGetDeviceCount(n);
    if (e != cudaSuccess) {
        *n = 0;
        return fail(nullptr, FRB_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    return FRB_OK;
}

const char* frb_last_error(frb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

int frb_create(int device, uint32_t table_log2, frb_ctx** out) {
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0)
        return fail(nullptr, FRB_ERR_CUDA, "no CUDA device: frender_b200 has no CPU fallback");
    if (device < 0 || device >= n) return fail(nullptr, FRB_ERR_ARG, "device %d out of range (%d present)", device, n);
    if (table_log2 < 10 || table_log2 > 32) return fail(nullptr, FRB_ERR_ARG, "table_log2 must be in [10, 32]");
    cudaDeviceProp prop;
    CU(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, FRB_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    frb_ctx* c = new frb_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->log2 = table_log2;
    c->cap = 1ULL << table_log2;
    CU(c, cudaSetDevice(device));
    {
        cudaMemPool_t pool;
        unsigned long long keep = ~0ULL;
        CU(c, cudaDeviceGetDefaultMemPool(&pool, device));
        CU(c, cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    CU(c, cudaStreamCreateWithFlags(&c->compute, cudaStreamNonBlocking));
    CU(c, cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking));
    CU(c, cudaMalloc(&c->file_tab, c->cap * sizeof(Slot)));
    CU(c, cudaMalloc(&c->total_tab, c->cap * sizeof(Slot)));
    CU(c, cudaMalloc(&c->st, sizeof(DevState)));
    CU(c, cudaMemset(c->st, 0, sizeof(DevState)));
    CU(c, cudaMallocHost(&c->st_host, sizeof(DevState)));
    CU(c, cudaEventCreate(&c->t0));
    CU(c, cudaEventCreate(&c->t1));
    CU(c, cudaFuncSetAttribute(scan_ws_kernel<WsTile>, cudaFuncAttributeMaxDynamicSharedMemorySize, WsTile::smem));
    CU(c, cudaFuncSetAttribute(scan_ws_kernel<WsTileWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, WsTileWide::smem));
    CU(c, cudaFuncSetAttribute(scan_spec_kernel<WsTile>, cudaFuncAttributeMaxDynamicSharedMemorySize, WsTile::smem));
    CU(c, cudaFuncSetAttribute(scan_spec_kernel<WsTile, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, WsTile::smem));
    CU(c, cudaFuncSetAttribute(match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CU(c, cudaFuncSetAttribute(match_cand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CU(c, cudaFuncSetAttribute(match_idx1_cand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CU(c, cudaFuncSetAttribute(match_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    TRY(clear_table(c, c->total_tab));
    CU(c, cudaStreamSynchronize(c->compute));
    *out = c;
    return FRB_OK;
}

void frb_destroy(frb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto& f : c->files) free_list(c, f);
    free_list(c, c->total);
    cudaFree(c->skip_slot);
    cudaFree(c->file_tab), cudaFree(c->total_tab), cudaFree(c->st), cudaFreeHost(c->st_host), cudaFree(c->status), cudaFree(c->redo), cudaFree(c->tile_first), cudaFree(c->block_sums);
    for (auto* p : c->xchg) cudaFree(p);
    for (int i = 0; i < kHostStages; ++i) {
        if (c->stage[i]) cudaFree(c->stage[i]), cudaEventDestroy(c->stage_copied[i]), cudaEventDestroy(c->stage_done[i]);
        if (c->ring[i]) cudaFreeHost(c->ring[i]);
    }
    cudaFree(c->sheet_fwd), cudaFree(c->sheet_rc), cudaFree(c->sheet_group), cudaFree(c->sheet_use_rc);
    cudaFree(c->sheet_fwd_hi), cudaFree(c->sheet_rc_hi);
    cudaFree(c->f_sum), cudaFree(c->rc_sum);
    cudaFree(c->m1), cudaFree(c->m2), cudaFree(c->srow), cudaFree(c->m2rc), cudaFree(c->srowrc);
    cudaFree(c->type), cudaFree(c->typerc), cudaFree(c->work), cudaFree(c->work_n), cudaFree(c->cub_tmp), cudaFree(c->route_tab);
    route_stream_destroy(c);
    if (c->gzbuf) {
        gz_free(c->gzbuf->b);
        delete c->gzbuf;
    }
    cudaFree(c->synth_i7), cudaFree(c->synth_i5), cudaFree(c->synth_cdf), cudaFree(c->synth_len), cudaFree(c->synth_off);
    for (auto& p : c->prof_pending) cudaEventDestroy(p.a), cudaEventDestroy(p.b);
    for (auto& p : c->prof_free) cudaEventDestroy(p.a), cudaEventDestroy(p.b);
    cudaEventDestroy(c->t0), cudaEventDestroy(c->t1);
    cudaStreamDestroy(c->compute), cudaStreamDestroy(c->copy);
    delete c;
}

int frb_resize_tables(frb_ctx* c, uint32_t table_log2) {
    CU(c, cudaSetDevice(c->device));
    if (table_log2 < 10 || table_log2 > 32) return fail(c, FRB_ERR_ARG, "table_log2 must be in [10, 32]");
    TRY(frb_reset(c));  // forgets every file and the total: a table cannot be re-hashed under a running tally
    CU(c, cudaStreamSynchronize(c->compute));
    CU(c, cudaFree(c->file_tab));
    CU(c, cudaFree(c->total_tab));
    c->file_tab = c->total_tab = nullptr;
    c->log2 = table_log2;
    c->cap = 1ULL << table_log2;
    CU(c, cudaMalloc(&c->file_tab, c->cap * sizeof(Slot)));
    CU(c, cudaMalloc(&c->total_tab, c->cap * sizeof(Slot)));
    TRY(clear_table(c, c->total_tab));
    c->total_tab_clean = true;
    CU(c, cudaStreamSynchronize(c->compute));
    return FRB_OK;
}

int frb_sync(frb_ctx* c) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->copy));
    CU(c, cudaStreamSynchronize(c->compute));
    return device_error_check(c);
}

// ---- memory ---------------------------------------------------------------------------------
int frb_host_alloc(void** p, size_t nbytes) {
    CU(nullptr, cudaMallocHost(p, nbytes));
    return FRB_OK;
}
int frb_host_free(void* p) {
    CU(nullptr, cudaFreeHost(p));
    return FRB_OK;
}
int frb_dev_alloc(frb_ctx* c, size_t nbytes, void** dptr) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMalloc(dptr, nbytes));
    return FRB_OK;
}
int frb_dev_free(frb_ctx* c, void* dptr) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaFree(dptr));
    return FRB_OK;
}
int frb_h2d(frb_ctx* c, void* dptr, const void* host, size_t nbytes) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMemcpyAsync(dptr, host, nbytes, cudaMemcpyHostToDevice, c->compute));
    CU(c, cudaStreamSynchronize(c->compute));
    return FRB_OK;
}
int frb_d2h(frb_ctx* c, void* host, const void* dptr, size_t nbytes) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMemcpyAsync(host, dptr, nbytes, cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaStreamSynchronize(c->compute));
    return FRB_OK;
}
int frb_mem_info(frb_ctx* c, uint64_t* free_bytes, uint64_t* total_bytes) {
    size_t f = 0, t = 0;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMemGetInfo(&f, &t));
    *free_bytes = f, *total_bytes = t;
    return FRB_OK;
}

// ---- key packing ----------------------------------------------------------------------------
int frb_pack_key(const char* s, size_t len, int sheet_mode, uint64_t* out) {
    if (len > kMaxSyms) return FRB_ERR_KEY_TOO_LONG;
    uint64_t k = 0;
    for (size_t i = 0; i < len; ++i) {
        unsigned ch = static_cast<unsigned char>(s[i]);
        if (sheet_mode && ch >= 'a' && ch <= 'z') ch -= 32;  // matching is case-insensitive, F:226
        unsigned code = enc_read(ch);
        if (code == 0) {
            if (!sheet_mode) return FRB_ERR_BAD_ALPHABET;
            code = 7;
        }
        k |= static_cast<uint64_t>(code) << (3 * i);
    }
    *out = k;
    return FRB_OK;
}
int frb_unpack_key(uint64_t key, char* out) {
    int n = 0;
    while (n < kMaxSyms) {
        const unsigned code = static_cast<unsigned>(key >> (3 * n)) & 7u;
        if (!code) break;
        out[n++] = dec_sym(code);
    }
    out[n] = 0;
    return n;
}

int frb_pack_key2(const char* s, size_t len, int sheet_mode, uint64_t* lo, uint64_t* hi) {
    if (len > static_cast<size_t>(kMaxWideSyms)) return FRB_ERR_KEY_TOO_LONG;
    const size_t n0 = std::min<size_t>(len, kMaxSyms);
    TRY(frb_pack_key(s, n0, sheet_mode, lo));
    return frb_pack_key(s + n0, len - n0, sheet_mode, hi);
}
int frb_unpack_key2(uint64_t lo, uint64_t hi, char* out) {
    const int n = frb_unpack_key(lo, out);
    return n < kMaxSyms ? n : n + frb_unpack_key(hi, out + n);
}

int frb_set_key_width(frb_ctx* c, uint32_t bits) {
    CU(c, cudaSetDevice(c->device));
    if (bits != 64 && bits != 128) return fail(c, FRB_ERR_ARG, "key width must be 64 or 128 bits");
    TRY(frb_reset(c));
    CU(c, cudaStreamSynchronize(c->compute));
    c->wide = bits == 128;
    // the tables change layout: the total table is cleared in the new one (the per-file table at every frb_scan_begin)
    TRY(clear_table(c, c->total_tab));
    c->total_tab_clean = true;
    if (c->route_tab) CU(c, cudaFree(c->route_tab));
    c->route_tab = nullptr, c->route_cap = 0, c->n_sinks = 0;
    route_stream_destroy(c);  // its key buffer is sized for one width
    // the sample sheet is packed for one width: it has to be loaded again
    cudaFree(c->sheet_fwd), cudaFree(c->sheet_rc), cudaFree(c->sheet_group), cudaFree(c->sheet_use_rc);
    cudaFree(c->f_sum), cudaFree(c->rc_sum), cudaFree(c->sheet_fwd_hi), cudaFree(c->sheet_rc_hi);
    c->sheet_fwd = c->sheet_rc = nullptr, c->sheet_group = nullptr, c->sheet_use_rc = nullptr;
    c->f_sum = c->rc_sum = nullptr, c->sheet_fwd_hi = c->sheet_rc_hi = nullptr;
    c->rows = c->l1 = c->l2 = 0;
    c->total_gen++, c->sheet_gen++;
    CU(c, cudaStreamSynchronize(c->compute));
    return FRB_OK;
}

// ---- hot path A -----------------------------------------------------------------------------
int frb_scan_begin(frb_ctx* c, uint32_t file_ordinal, uint64_t read_limit) {
    CU(c, cudaSetDevice(c->device));
    if (c->in_file) return fail(c, FRB_ERR_STATE, "frb_scan_begin: previous file not ended");
    if (c->sharded) return fail(c, FRB_ERR_STATE, "frb_scan_begin: the total is a share of a sharded merge; frb_reset first");
    if (file_ordinal >= (1u << 23)) return fail(c, FRB_ERR_ARG, "file ordinal too large");
    c->cur_ordinal = file_ordinal;
    c->cur_limit = read_limit ? read_limit : ~0ULL;
    c->file_tiles = 0;
    c->file_composite = -1;
    CU(c, cudaMemsetAsync(c->st, 0, offsetof(DevState, occupied_total), c->compute));
    TRY(clear_table(c, c->file_tab));
    c->in_file = true;
    return FRB_OK;
}

int frb_scan_chunk_dev(frb_ctx* c, const void* dev, uint64_t nbytes, uint64_t line_base, int rule,
                       uint64_t* keys_out_dev, uint64_t* rec_off_out_dev) {
    CU(c, cudaSetDevice(c->device));
    if (!c->in_file) return fail(c, FRB_ERR_STATE, "frb_scan_chunk: no file begun");
    if (c->wide && keys_out_dev)
        return fail(c, FRB_ERR_STATE, "frb_scan_chunk_dev: per-read keys are not available on a wide (128-bit key) context");
    return launch_scan(c, static_cast<const unsigned char*>(dev), nbytes, line_base, rule,
                       reinterpret_cast<unsigned long long*>(keys_out_dev),
                       reinterpret_cast<unsigned long long*>(rec_off_out_dev), c->file_tab, 0);
}

int frb_scan_chunk_host(frb_ctx* c, const void* host, uint64_t nbytes, uint64_t line_base, int rule) {
    CU(c, cudaSetDevice(c->device));
    if (!c->in_file) return fail(c, FRB_ERR_STATE, "frb_scan_chunk: no file begun");
    TRY(ensure_stages(c));
    const unsigned char* p = static_cast<const unsigned char*>(host);
    uint64_t left = nbytes;
    bool first = true;
    while (left) {
        uint64_t piece = std::min<uint64_t>(left, c->stage_cap);
        if (piece < left) {  // cut after the last newline of the piece
            const void* nl = memrchr(p, '\n', piece);
            if (!nl) return fail(c, FRB_ERR_ARG, "a single line exceeds the staging buffer (%zu bytes)", c->stage_cap);
            piece = static_cast<const unsigned char*>(nl) - p + 1;
        }
        const int s = c->stage_next;
        c->stage_next = (s + 1) % kHostStages;
        CU(c, cudaStreamWaitEvent(c->copy, c->stage_done[s], 0));  // kernel that last read this stage
        CU(c, cudaMemcpyAsync(c->stage[s], p, piece, cudaMemcpyHostToDevice, c->copy));
        CU(c, cudaEventRecord(c->stage_copied[s], c->copy));
        CU(c, cudaStreamWaitEvent(c->compute, c->stage_copied[s], 0));
        TRY(launch_scan(c, c->stage[s], piece, first ? line_base : FRB_CARRY, rule, nullptr, nullptr, c->file_tab, 0));
        CU(c, cudaEventRecord(c->stage_done[s], c->compute));
        CU(c, cudaEventSynchronize(c->stage_copied[s]));  // host bytes consumed; kernel still runs
        p += piece;
        left -= piece;
        first = false;
    }
    return FRB_OK;
}

int frb_scan_end(frb_ctx* c, uint64_t* n_reads, uint64_t* n_unique) {
    CU(c, cudaSetDevice(c->device));
    if (!c->in_file) return fail(c, FRB_ERR_STATE, "frb_scan_end: no file begun");
    c->in_file = false;
    CU(c, cudaStreamSynchronize(c->copy));
    CU(c, cudaStreamSynchronize(c->compute));
    TRY(device_error_check(c));
    KeyList fl;
    fl.reads = c->st_host->n_reads;
    fl.ordinal = c->cur_ordinal;
    // Unique keys of the file = occupied slots of its table (at most one per read): compacted and counted in one
    // pass.  Read ordinals of one file stay below 2^40; composite positions become ordinals here.
    TRY(table_to_sorted_list_counting(c, c->file_tab, fl.reads, &fl, 40, c->file_composite == 1 ? c->tile_first : nullptr));
    c->files.push_back(fl);
    c->total_ready = false;
    if (n_reads) *n_reads = fl.reads;
    if (n_unique) *n_unique = fl.n;
    return FRB_OK;
}

int frb_file_count(frb_ctx* c, uint32_t* n_files) {
    *n_files = static_cast<uint32_t>(c->files.size());
    return FRB_OK;
}
int frb_file_size(frb_ctx* c, uint32_t i, uint64_t* n_unique, uint64_t* n_reads) {
    if (i >= c->files.size()) return fail(c, FRB_ERR_ARG, "file index out of range");
    if (n_unique) *n_unique = c->files[i].n;
    if (n_reads) *n_reads = c->files[i].reads;
    return FRB_OK;
}
static int export_list(frb_ctx* c, KeyList& l, uint64_t* keys, uint64_t* counts, uint64_t* first, uint64_t cap,
                       uint64_t* keys_hi = nullptr) {
    TRY(ensure_sorted(c, l));
    if (cap < l.n) return fail(c, FRB_ERR_ARG, "export buffer too small (%llu < %llu)", (unsigned long long)cap,
                               (unsigned long long)l.n);
    if (!l.n) return FRB_OK;
    CU(c, cudaSetDevice(c->device));
    if (keys) CU(c, cudaMemcpyAsync(keys, l.keys, l.n * 8, cudaMemcpyDeviceToHost, c->compute));
    if (counts) CU(c, cudaMemcpyAsync(counts, l.counts, l.n * 8, cudaMemcpyDeviceToHost, c->compute));
    if (first) CU(c, cudaMemcpyAsync(first, l.first, l.n * 8, cudaMemcpyDeviceToHost, c->compute));
    if (keys_hi) {
        if (l.keys_hi) CU(c, cudaMemcpyAsync(keys_hi, l.keys_hi, l.n * 8, cudaMemcpyDeviceToHost, c->compute));
        else memset(keys_hi, 0, l.n * 8);  // a narrow context: every key fits the lower word
    }
    CU(c, cudaStreamSynchronize(c->compute));
    return FRB_OK;
}
int frb_file_export(frb_ctx* c, uint32_t i, uint64_t* keys, uint64_t* counts, uint64_t* first_read, uint64_t cap) {
    if (i >= c->files.size()) return fail(c, FRB_ERR_ARG, "file index out of range");
    return export_list(c, c->files[i], keys, counts, first_read, cap);
}
int frb_file_export_hi(frb_ctx* c, uint32_t i, uint64_t* keys_hi, uint64_t cap) {
    if (i >= c->files.size()) return fail(c, FRB_ERR_ARG, "file index out of range");
    return export_list(c, c->files[i], nullptr, nullptr, nullptr, cap, keys_hi);
}

static int merge_pending_files(frb_ctx* c) {  // fold file lists into total_tab (F:199-203)
    for (; c->merged_upto < c->files.size(); ++c->merged_upto) {
        const KeyList& fl = c->files[c->merged_upto];
        if (!fl.n) continue;
        ProfScope ps(c, FRB_K_EXPORT);
        if (c->wide)
            merge_wide_list_kernel<<<static_cast<unsigned>((fl.n + 255) / 256), 256, 0, c->compute>>>(
                reinterpret_cast<WideSlot*>(c->total_tab), c->cap - 1, fl.keys, fl.keys_hi, fl.counts, fl.first, fl.n,
                static_cast<unsigned long long>(fl.ordinal) << 40, &c->st->occupied_total, c->st);
        else
            merge_list_kernel<<<static_cast<unsigned>((fl.n + 255) / 256), 256, 0, c->compute>>>(
                c->total_tab, c->cap - 1, fl.keys, fl.counts, fl.first, fl.n,
                static_cast<unsigned long long>(fl.ordinal) << 40, &c->st->occupied_total, c->st);
        c->launches++;
        c->total_tab_clean = false;
        CU(c, cudaGetLastError());
    }
    return FRB_OK;
}

// need_order = false: the caller (a sharded merge) regroups the entries anyway
static int total_build(frb_ctx* c, bool need_order) {
    if (!c->total_ready) {
        TRY(free_list(c, c->total));
        if (c->files.size() == 1 && c->merged_upto == 0 && !c->ext_merged) {
            // one file: "total" is that file's list (F:199-203 degenerates to a copy); only `first`
            // gets the file ordinal in its high bits
            KeyList& fl = c->files[0];
            if (need_order) TRY(ensure_sorted(c, fl));
            c->total.sorted = fl.sorted;
            c->total.first_bits = 64;
            c->total.n = fl.n;
            if (fl.n) {
                TRY(dmalloc(c, &c->total.keys, fl.n * 8));
                TRY(dmalloc(c, &c->total.counts, fl.n * 8));
                TRY(dmalloc(c, &c->total.first, fl.n * 8));
                ProfScope ps(c, FRB_K_EXPORT);
                CU(c, cudaMemcpyAsync(c->total.keys, fl.keys, fl.n * 8, cudaMemcpyDeviceToDevice, c->compute));
                CU(c, cudaMemcpyAsync(c->total.counts, fl.counts, fl.n * 8, cudaMemcpyDeviceToDevice, c->compute));
                if (fl.keys_hi) {
                    TRY(dmalloc(c, &c->total.keys_hi, fl.n * 8));
                    CU(c, cudaMemcpyAsync(c->total.keys_hi, fl.keys_hi, fl.n * 8, cudaMemcpyDeviceToDevice, c->compute));
                }
                add_offset_kernel<<<static_cast<unsigned>((fl.n + 255) / 256), 256, 0, c->compute>>>(
                    fl.first, c->total.first, fl.n, static_cast<unsigned long long>(fl.ordinal) << 40);
                c->launches++;
                CU(c, cudaGetLastError());
            }
        } else {
            TRY(merge_pending_files(c));
            CU(c, cudaStreamSynchronize(c->compute));
            TRY(device_error_check(c));
            TRY(table_to_sorted_list(c, c->total_tab, c->st_host->occupied_total, &c->total));
        }
        c->total_ready = true;
        c->total_gen++;
    }
    if (need_order) TRY(ensure_sorted(c, c->total));
    return FRB_OK;
}

int frb_total_finish(frb_ctx* c, uint64_t* n_unique) {
    CU(c, cudaSetDevice(c->device));
    if (c->in_file) return fail(c, FRB_ERR_STATE, "frb_total_finish: a file is still open");
    TRY(total_build(c, true));
    if (n_unique) *n_unique = c->total.n;
    return FRB_OK;
}
int frb_total_export(frb_ctx* c, uint64_t* keys, uint64_t* counts, uint64_t* first_pos, uint64_t cap) {
    if (!c->total_ready) return fail(c, FRB_ERR_STATE, "frb_total_export: call frb_total_finish first");
    return export_list(c, c->total, keys, counts, first_pos, cap);
}
int frb_total_export_hi(frb_ctx* c, uint64_t* keys_hi, uint64_t cap) {
    if (!c->total_ready) return fail(c, FRB_ERR_STATE, "frb_total_export_hi: call frb_total_finish first");
    return export_list(c, c->total, nullptr, nullptr, nullptr, cap, keys_hi);
}
int frb_total_load(frb_ctx* c, const uint64_t* keys, const uint64_t* counts, uint64_t n) {
    return frb_total_load2(c, keys, nullptr, counts, n);
}
int frb_total_load2(frb_ctx* c, const uint64_t* keys, const uint64_t* keys_hi, const uint64_t* counts, uint64_t n) {
    CU(c, cudaSetDevice(c->device));
    if (keys_hi && !c->wide) return fail(c, FRB_ERR_STATE, "frb_total_load2: upper key words need a wide context (frb_set_key_width)");
    TRY(free_list(c, c->total));
    c->total.n = n;
    if (n) {
        TRY(dmalloc(c, &c->total.keys, n * 8));
        TRY(dmalloc(c, &c->total.counts, n * 8));
        TRY(dmalloc(c, &c->total.first, n * 8));
        if (c->wide) {
            TRY(dmalloc(c, &c->total.keys_hi, n * 8));
            if (keys_hi) CU(c, cudaMemcpyAsync(c->total.keys_hi, keys_hi, n * 8, cudaMemcpyHostToDevice, c->compute));
            else CU(c, cudaMemsetAsync(c->total.keys_hi, 0, n * 8, c->compute));
        }
        CU(c, cudaMemcpyAsync(c->total.keys, keys, n * 8, cudaMemcpyHostToDevice, c->compute));
        CU(c, cudaMemcpyAsync(c->total.counts, counts, n * 8, cudaMemcpyHostToDevice, c->compute));
        CU(c, cudaMemsetAsync(c->total.first, 0, n * 8, c->compute));
        CU(c, cudaStreamSynchronize(c->compute));
    }
    c->total_ready = true;
    c->total_gen++;
    return FRB_OK;
}
int frb_total_merge(frb_ctx* c, const uint64_t* keys, const uint64_t* counts, const uint64_t* first_pos, uint64_t n) {
    CU(c, cudaSetDevice(c->device));
    if (c->in_file) return fail(c, FRB_ERR_STATE, "frb_total_merge: a file is still open");
    if (c->wide) return fail(c, FRB_ERR_STATE, "frb_total_merge: not available on a wide (128-bit key) context");
    if (n) {
        unsigned long long *dk = nullptr, *dc = nullptr, *df = nullptr;
        TRY(dmalloc(c, &dk, n * 8));
        TRY(dmalloc(c, &dc, n * 8));
        TRY(dmalloc(c, &df, n * 8));
        CU(c, cudaMemcpyAsync(dk, keys, n * 8, cudaMemcpyHostToDevice, c->compute));
        CU(c, cudaMemcpyAsync(dc, counts, n * 8, cudaMemcpyHostToDevice, c->compute));
        CU(c, cudaMemcpyAsync(df, first_pos, n * 8, cudaMemcpyHostToDevice, c->compute));
        {
            ProfScope ps(c, FRB_K_EXPORT);
            merge_list_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(
                c->total_tab, c->cap - 1, dk, dc, df, n, 0ULL, &c->st->occupied_total, c->st);
            c->launches++;
        }
        CU(c, cudaGetLastError());
        CU(c, cudaStreamSynchronize(c->compute));  // the host arrays may be reused by the caller
        TRY(dfree(c, dk));
        TRY(dfree(c, dc));
        TRY(dfree(c, df));
        c->total_tab_clean = false;
    }
    c->ext_merged = true;
    c->total_ready = false;
    return FRB_OK;
}
int frb_reset(frb_ctx* c) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->compute));
    for (auto& f : c->files) TRY(free_list(c, f));
    c->files.clear();
    TRY(free_list(c, c->total));
    c->total_ready = false;
    c->in_file = false;
    CU(c, cudaMemsetAsync(c->st, 0, sizeof(DevState), c->compute));
    c->merged_upto = 0;
    c->ext_merged = false;
    c->sharded = false;
    if (!c->total_tab_clean) {
        TRY(clear_table(c, c->total_tab));
        c->total_tab_clean = true;
    }
    return FRB_OK;
}

// ---- gz pipeline ----------------------------------------------------------------------------
namespace {
// In-place universal-newline translation of buf[0, n) ("\r\n" -> "\n", lone "\r" -> "\n", as
// text-mode gzip.open does, F:159).  A "\r" as very last byte is held back (*pending) because
// the byte after it decides.  Returns the new length.
size_t normalize_cr(unsigned char* buf, size_t n, bool* pending, bool at_eof) {
    size_t w = 0;
    for (size_t r = 0; r < n; ++r) {
        if (buf[r] != '\r') {
            buf[w++] = buf[r];
            continue;
        }
        if (r + 1 < n) {
            buf[w++] = '\n';
            if (buf[r + 1] == '\n') ++r;
        } else if (at_eof) {
            buf[w++] = '\n';
        } else {
            *pending = true;
        }
    }
    return w;
}
}  // namespace

static int scan_gz_host(frb_ctx* c, const char* path, uint32_t file_ordinal, uint64_t read_limit, uint64_t* n_reads,
                        uint64_t* n_unique, uint64_t* raw_bytes) {
    CU(c, cudaSetDevice(c->device));
    TRY(ensure_stages(c));
    for (int i = 0; i < kHostStages; ++i)
        if (!c->ring[i]) CU(c, cudaMallocHost(&c->ring[i], c->stage_cap));
    gzFile gz = gzopen(path, "rb");
    if (!gz) return fail(c, FRB_ERR_IO, "cannot open %s", path);
    gzbuffer(gz, 1 << 20);
    if (gzdirect(gz)) {  // zlib would pass such a file through as it is; gzip.open raises BadGzipFile (F:159)
        gzclose(gz);
        return fail(c, FRB_ERR_IO, "%s: not a gzipped file", path);
    }
    TRY(frb_scan_begin(c, file_ordinal, read_limit));

    struct Item {
        int slot;
        size_t bytes;
        bool eof;
    };
    std::mutex mu;
    std::condition_variable cv;
    std::vector<Item> ready;
    int free_slots = kHostStages;
    bool stop = false;
    std::string io_err;
    uint64_t total_raw = 0;

    std::thread reader([&] {
        std::vector<unsigned char> tail;
        bool cr_pending = false;
        int slot = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return free_slots > 0 || stop; });
                if (stop) return;
                --free_slots;
            }
            unsigned char* buf = c->ring[slot];
            size_t have = tail.size();
            if (have) memcpy(buf, tail.data(), have);
            tail.clear();
            bool eof = false;
            while (have < c->stage_cap) {
                // a '\r' held back at the end of the last piece: it is a line end of its own unless this piece
                // begins with '\n' ("\r\n" split across two reads); one byte of room is kept for it
                const unsigned want = static_cast<unsigned>(std::min<size_t>(c->stage_cap - have - (cr_pending ? 1 : 0), 1u << 30));
                if (want == 0) break;
                const int got = gzread(gz, buf + have + (cr_pending ? 1 : 0), want);
                if (got < 0) {
                    int errnum = 0;
                    io_err = gzerror(gz, &errnum);
                    eof = true;
                    break;
                }
                if (got == 0) {
                    eof = true;
                    break;
                }
                unsigned char* piece = buf + have + (cr_pending ? 1 : 0);
                size_t n_piece = static_cast<size_t>(got);
                if (cr_pending) {  // emit the line end; a leading '\n' of this piece belongs to it
                    buf[have++] = '\n';
                    cr_pending = false;
                    if (piece[0] == '\n') ++piece, --n_piece;
                    if (piece != buf + have) memmove(buf + have, piece, n_piece);
                    piece = buf + have;
                }
                if (memchr(piece, '\r', n_piece)) {
                    // rare path: translate this piece (a trailing '\r' waits for its successor)
                    have += normalize_cr(piece, n_piece, &cr_pending, false);
                } else {
                    have += n_piece;
                }
            }
            if (eof && cr_pending) buf[have++] = '\n', cr_pending = false;
            size_t usable = have;
            if (!eof) {
                const void* nl = memrchr(buf, '\n', have);
                if (!nl) {
                    io_err = "a single line exceeds the staging buffer";
                    eof = true;
                    usable = 0;
                } else {
                    usable = static_cast<const unsigned char*>(nl) - buf + 1;
                    tail.assign(buf + usable, buf + have);
                }
            }
            total_raw += usable;
            {
                std::lock_guard<std::mutex> lk(mu);
                ready.push_back({slot, usable, eof});
            }
            cv.notify_all();
            if (eof) return;
            slot = (slot + 1) % kHostStages;
        }
    });

    int rc = FRB_OK;
    for (;;) {
        Item it;
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return !ready.empty(); });
            it = ready.front();
            ready.erase(ready.begin());
        }
        if (rc == FRB_OK && it.bytes) rc = frb_scan_chunk_host(c, c->ring[it.slot], it.bytes, FRB_CARRY, FRB_RULE_SCAN);
        bool enough = false;
        if (rc == FRB_OK && read_limit) {  // -s: stop reading once the head sample is complete
            cudaStreamSynchronize(c->compute);
            cudaMemcpy(c->st_host, c->st, sizeof(DevState), cudaMemcpyDeviceToHost);
            enough = c->st_host->n_reads >= read_limit;
        }
        {
            std::lock_guard<std::mutex> lk(mu);
            ++free_slots;
            if (rc != FRB_OK || enough) stop = true;
        }
        cv.notify_all();
        if (it.eof || rc != FRB_OK || enough) break;
    }
    {
        std::lock_guard<std::mutex> lk(mu);
        stop = true;
    }
    cv.notify_all();
    reader.join();
    {   // a stream cut short only shows here: gzread() returns 0 at the end of the bytes there are, zlib reports
        // Z_BUF_ERROR through gzerror / gzclose (gzip.open raises EOFError for such a file, F:159)
        int errnum = 0;
        const char* msg = gzerror(gz, &errnum);
        if (io_err.empty() && errnum != Z_OK && errnum != Z_STREAM_END && !(read_limit && errnum == Z_BUF_ERROR && stop))
            io_err = msg ? msg : "gzip error";
        const int closed = gzclose(gz);
        if (io_err.empty() && closed != Z_OK && !read_limit) io_err = closed == Z_BUF_ERROR ? "unexpected end of file" : "gzip error";
    }
    if (rc == FRB_OK && !io_err.empty()) rc = fail(c, FRB_ERR_IO, "%s: %s", path, io_err.c_str());
    if (rc != FRB_OK) {
        c->in_file = false;
        cudaStreamSynchronize(c->compute);
        return rc;
    }
    if (raw_bytes) *raw_bytes = total_raw;
    return frb_scan_end(c, n_reads, n_unique);
}

// Whole .gz file: inflated on the device when the stream allows it (frb_gz.inl), else by zlib on a host thread.
int frb_scan_gz(frb_ctx* c, const char* path, uint32_t file_ordinal, uint64_t read_limit, uint64_t* n_reads,
                uint64_t* n_unique, uint64_t* raw_bytes) {
    CU(c, cudaSetDevice(c->device));
    static const bool device_ok = !(getenv("FRB_GZ_DEVICE") && atoi(getenv("FRB_GZ_DEVICE")) == 0);
    if (device_ok && !read_limit) {  // -s reads a head sample only: the host path stops early
        if (!c->gzbuf) c->gzbuf = new GzBuffersHolder();
        TRY(frb_scan_begin(c, file_ordinal, 0));
        bool first = true;
        uint64_t raw = 0;
        const int rc = gz_device_inflate(
            c, c->gzbuf->b, path, &raw,
            [&](unsigned char* dev, uint64_t n, bool) {
                const int r = launch_scan(c, dev, n, first ? 0 : FRB_CARRY, FRB_RULE_SCAN, nullptr, nullptr, c->file_tab, 0);
                first = false;
                return r;
            },
            [&]() {  // start the file over (larger staging areas)
                c->in_file = false;
                first = true;
                CU(c, cudaStreamSynchronize(c->compute));
                CU(c, cudaMemsetAsync(&c->st->err_code, 0, sizeof(int), c->compute));
                return frb_scan_begin(c, file_ordinal, 0);
            });
        if (rc == FRB_OK) {
            c->gz_device_files++;
            if (raw_bytes) *raw_bytes = raw;
            return frb_scan_end(c, n_reads, n_unique);
        }
        c->in_file = false;
        CU(c, cudaStreamSynchronize(c->compute));
        if (rc != FRB_GZ_RETRY_HOST) return rc;
        CU(c, cudaMemsetAsync(&c->st->err_code, 0, sizeof(int), c->compute));  // errors of the abandoned attempt
    }
    return scan_gz_host(c, path, file_ordinal, read_limit, n_reads, n_unique, raw_bytes);
}

// A run of SMALL .gz files in one go: laid end to end they are one gzip stream of several members, which the device
// inflates with one set of launches (a small file alone leaves the GPU nine tenths idle: one warp decodes one chunk
// from end to end); the text of every file is then tallied as that file (own table, own list, own ordinals),
// exactly as frb_scan_gz would one by one.  *used_device = 0: declined, nothing has changed -- scan them one by one
// (that also is how a damaged file gets its own error message).
int frb_scan_gz_batch(frb_ctx* c, const char* const* paths, const uint32_t* ordinals, uint32_t n_files, uint64_t* n_reads,
                      uint64_t* n_unique, uint64_t* raw_bytes, int* used_device) {
    CU(c, cudaSetDevice(c->device));
    *used_device = 0;
    static const bool device_ok = !(getenv("FRB_GZ_DEVICE") && atoi(getenv("FRB_GZ_DEVICE")) == 0);
    if (!device_ok || n_files == 0) return FRB_OK;
    if (c->in_file) return fail(c, FRB_ERR_STATE, "frb_scan_gz_batch: previous file not ended");
    GzSource src;
    for (uint32_t i = 0; i < n_files; ++i) src.paths.emplace_back(paths[i]);
    TRY(src.open(c));
    for (uint32_t i = 0; i < n_files; ++i) {  // every file a gzip file of its own
        unsigned char magic[3] = {0, 0, 0};
        if (src.start[i + 1] - src.start[i] < 18 || !src.read(src.start[i], 3, magic) || magic[0] != 0x1f || magic[1] != 0x8b ||
            magic[2] != 8)
            return FRB_OK;
    }
    if (!c->gzbuf) c->gzbuf = new GzBuffersHolder();
    if (!c->skip_slot) CU(c, cudaMalloc(&c->skip_slot, 8));
    const size_t files_before = c->files.size();
    std::vector<uint64_t> text_end(n_files, ~0ULL);  // where the text of file i ends in the stream's text
    uint32_t closed = 0;      // files whose end is known
    uint32_t cur = 0;         // file being tallied
    bool open = false, first_chunk = true;
    uint64_t scanned = 0;     // text handed to the sink so far
    uint64_t file_text_start = 0;
    auto rollback = [&]() {
        c->in_file = false;
        cudaStreamSynchronize(c->compute);
        cudaMemsetAsync(&c->st->err_code, 0, sizeof(int), c->compute);
        while (c->files.size() > files_before) {
            free_list(c, c->files.back());
            c->files.pop_back();
        }
        std::fill(text_end.begin(), text_end.end(), ~0ULL);
        closed = cur = 0, open = false, first_chunk = true, scanned = 0, file_text_start = 0;
    };
    auto on_members = [&](const std::vector<GzMemberEnd>& members) {
        for (const GzMemberEnd& m : members) {
            if (closed >= n_files) return gz_decline("batch: a member behind the last file");
            // the member belongs to the first file that is not closed; that file ends where its last member does
            if (m.comp_end > src.start[closed + 1]) return gz_decline("batch: a file does not end with a member trailer");
            if (m.comp_end == src.start[closed + 1]) text_end[closed++] = m.text_end;
        }
        return FRB_OK;
    };
    auto sink = [&](unsigned char* dev, uint64_t n, bool last) {
        uint64_t pos = 0;
        for (;;) {
            if (cur >= n_files) {
                if (pos < n) return gz_decline("batch: text behind the last file");
                break;
            }
            if (!open) {
                TRY(frb_scan_begin(c, ordinals[cur], 0));
                open = true, first_chunk = true;
            }
            const bool ends_here = cur < closed && text_end[cur] <= scanned + n;
            const uint64_t seg_end = ends_here ? text_end[cur] - scanned : n;
            if (seg_end > pos) {  // text begins `skip` bytes into a 16-byte aligned buffer
                const uint64_t base = pos & ~15ULL;
                CU(c, cudaMemsetAsync(c->skip_slot, 0, 8, c->compute));
                if (pos & 15) CU(c, cudaMemsetAsync(c->skip_slot, static_cast<int>(pos & 15), 1, c->compute));
                TRY(launch_scan(c, dev + base, seg_end - base, first_chunk ? 0 : FRB_CARRY, FRB_RULE_SCAN, nullptr, nullptr,
                                c->file_tab, 0, ~0ULL, c->skip_slot));
                first_chunk = false;
            }
            pos = seg_end;
            if (!ends_here) break;
            TRY(frb_scan_end(c, &n_reads[cur], &n_unique[cur]));
            if (raw_bytes) raw_bytes[cur] = text_end[cur] - file_text_start;
            file_text_start = text_end[cur];
            open = false;
            ++cur;
        }
        scanned += n;
        if (last && (cur < n_files || open)) return gz_decline("batch: the stream ended inside a file");
        return FRB_OK;
    };
    uint64_t raw = 0;
    const int rc = gz_device_inflate_source(c, c->gzbuf->b, src, &raw, sink,
                                            [&]() {
                                                rollback();
                                                return FRB_OK;
                                            },
                                            on_members, true);
    if (rc == FRB_OK) {
        c->gz_device_files += n_files;
        *used_device = 1;
        return FRB_OK;
    }
    rollback();
    // anything about the DATA (a damaged file, a header that does not parse, ...) is reported by the one-by-one path,
    // which knows the file it belongs to
    if (rc == FRB_GZ_RETRY_HOST || rc == FRB_ERR_IO || rc == FRB_ERR_BAD_HEADER || rc == FRB_ERR_BAD_ALPHABET ||
        rc == FRB_ERR_KEY_TOO_LONG || rc == FRB_ERR_TABLE_FULL)
        return FRB_OK;
    return rc;
}

// Test / tooling entry: inflate a .gz on the device into host memory.  *used_device = 0 when the device path
// declined the stream (nothing is written then).
int frb_gz_inflate(frb_ctx* c, const char* path, void* host_out, uint64_t cap, uint64_t* nbytes, int* used_device) {
    CU(c, cudaSetDevice(c->device));
    if (!c->gzbuf) c->gzbuf = new GzBuffersHolder();
    uint64_t off = 0, raw = 0;
    *nbytes = 0, *used_device = 0;
    const int rc = gz_device_inflate(
        c, c->gzbuf->b, path, &raw,
        [&](unsigned char* dev, uint64_t n, bool) {
            if (off + n > cap) return fail(c, FRB_ERR_ARG, "frb_gz_inflate: output buffer too small");
            CU(c, cudaMemcpyAsync(static_cast<unsigned char*>(host_out) + off, dev, n, cudaMemcpyDeviceToHost, c->compute));
            CU(c, cudaStreamSynchronize(c->compute));
            off += n;
            return FRB_OK;
        },
        [&]() {
            off = 0;
            return FRB_OK;
        });
    if (rc == FRB_GZ_RETRY_HOST) return FRB_OK;
    if (rc != FRB_OK) return rc;
    *nbytes = off, *used_device = 1;
    return FRB_OK;
}

// ---- hot path B -----------------------------------------------------------------------------
int frb_sheet_load(frb_ctx* c, const uint64_t* fwd, const uint64_t* rc, const int32_t* group, uint32_t n_rows,
                   uint32_t l1, uint32_t l2) {
    return frb_sheet_load2(c, fwd, nullptr, rc, nullptr, group, n_rows, l1, l2);
}
int frb_sheet_load2(frb_ctx* c, const uint64_t* fwd, const uint64_t* fwd_hi, const uint64_t* rc, const uint64_t* rc_hi,
                    const int32_t* group, uint32_t n_rows, uint32_t l1, uint32_t l2) {
    CU(c, cudaSetDevice(c->device));
    if ((fwd_hi || rc_hi) && !c->wide) return fail(c, FRB_ERR_STATE, "frb_sheet_load2: upper key words need a wide context (frb_set_key_width)");
    if (c->wide) {
        if (l1 == 0 || l1 > kMaxSyms || l2 > kMaxSyms || l1 + (l2 ? 1 + l2 : 0) > kMaxWideSyms)
            return fail(c, FRB_ERR_ARG, "index lengths %u+%u unsupported (max 21 symbols per index, 42 incl. '+')", l1, l2);
    } else if (l1 == 0 || l1 + (l2 ? 1 + l2 : 0) > kMaxSyms) {
        return fail(c, FRB_ERR_ARG, "index lengths %u+%u unsupported (max 21 symbols incl. '+')", l1, l2);
    }
    if (n_rows > 5000) return fail(c, FRB_ERR_ARG, "sample sheet with %u rows exceeds the 5000-row limit", n_rows);
    for (uint32_t r = 0; r < n_rows; ++r)
        if (group[r] < 0 || static_cast<uint32_t>(group[r]) >= n_rows) return fail(c, FRB_ERR_ARG, "bad group id");
    CU(c, cudaStreamSynchronize(c->compute));
    cudaFree(c->sheet_fwd), cudaFree(c->sheet_rc), cudaFree(c->sheet_group), cudaFree(c->sheet_use_rc);
    cudaFree(c->f_sum), cudaFree(c->rc_sum), cudaFree(c->sheet_fwd_hi), cudaFree(c->sheet_rc_hi);
    c->sheet_fwd = c->sheet_rc = nullptr, c->sheet_group = nullptr, c->sheet_use_rc = nullptr;
    c->sheet_fwd_hi = c->sheet_rc_hi = nullptr;
    c->f_sum = c->rc_sum = nullptr;
    const size_t n = std::max<uint32_t>(n_rows, 1);
    CU(c, cudaMalloc(&c->sheet_fwd, n * 8));
    CU(c, cudaMalloc(&c->sheet_rc, n * 8));
    CU(c, cudaMalloc(&c->sheet_group, n * 4));
    CU(c, cudaMalloc(&c->sheet_use_rc, n));
    CU(c, cudaMalloc(&c->f_sum, n * 8));
    CU(c, cudaMalloc(&c->rc_sum, n * 8));
    if (c->wide) {
        CU(c, cudaMalloc(&c->sheet_fwd_hi, n * 8));
        CU(c, cudaMalloc(&c->sheet_rc_hi, n * 8));
        CU(c, cudaMemset(c->sheet_fwd_hi, 0, n * 8));
        CU(c, cudaMemset(c->sheet_rc_hi, 0, n * 8));
        if (n_rows && fwd_hi) CU(c, cudaMemcpy(c->sheet_fwd_hi, fwd_hi, n_rows * 8, cudaMemcpyHostToDevice));
        if (n_rows && rc_hi) CU(c, cudaMemcpy(c->sheet_rc_hi, rc_hi, n_rows * 8, cudaMemcpyHostToDevice));
    }
    if (n_rows) {
        CU(c, cudaMemcpy(c->sheet_fwd, fwd, n_rows * 8, cudaMemcpyHostToDevice));
        CU(c, cudaMemcpy(c->sheet_rc, rc, n_rows * 8, cudaMemcpyHostToDevice));
        CU(c, cudaMemcpy(c->sheet_group, group, n_rows * 4, cudaMemcpyHostToDevice));
    }
    c->rows = n_rows, c->l1 = l1, c->l2 = l2;
    c->sheet_gen++;
    return FRB_OK;
}

int frb_match(frb_ctx* c, uint32_t n_subs, int rc_mode, const uint8_t* use_rc_rows, int32_t* m1_row, int32_t* m2_row,
              uint8_t* type, int32_t* sample_row, int32_t* m2rc_row, uint8_t* type_rc, int32_t* sample_rc_row,
              uint64_t* f_sum, uint64_t* rc_sum) {
    CU(c, cudaSetDevice(c->device));
    if (!c->total_ready) return fail(c, FRB_ERR_STATE, "frb_match: no total list (frb_total_finish / frb_total_load)");
    if (!c->sheet_fwd) return fail(c, FRB_ERR_STATE, "frb_match: no sample sheet loaded");
    if (rc_mode && c->l2 == 0) return fail(c, FRB_ERR_ARG, "frb_match: rc_mode needs a dual-index sheet");
    const uint64_t n = c->total.n;
    if (n > c->match_cap) {
        CU(c, cudaStreamSynchronize(c->compute));
        cudaFree(c->m1), cudaFree(c->m2), cudaFree(c->srow), cudaFree(c->m2rc), cudaFree(c->srowrc);
        cudaFree(c->type), cudaFree(c->typerc), cudaFree(c->work), cudaFree(c->work_n);
        c->match_cap = 0;
        CU(c, cudaMalloc(&c->m1, n * 4));
        CU(c, cudaMalloc(&c->m2, n * 4));
        CU(c, cudaMalloc(&c->srow, n * 4));
        CU(c, cudaMalloc(&c->m2rc, n * 4));
        CU(c, cudaMalloc(&c->srowrc, n * 4));
        CU(c, cudaMalloc(&c->type, n));
        CU(c, cudaMalloc(&c->typerc, n));
        CU(c, cudaMalloc(&c->work, n * 4));
        CU(c, cudaMalloc(&c->work_n, 8));
        c->match_cap = n;
        c->m1_total_gen = ~0ULL;
    }
    const size_t rows1 = std::max<uint32_t>(c->rows, 1);
    if (use_rc_rows && c->rows)
        CU(c, cudaMemcpyAsync(c->sheet_use_rc, use_rc_rows, c->rows, cudaMemcpyHostToDevice, c->compute));
    CU(c, cudaMemsetAsync(c->f_sum, 0, rows1 * 8, c->compute));
    CU(c, cudaMemsetAsync(c->rc_sum, 0, rows1 * 8, c->compute));
    if (n) {
        MatchArgs a{};
        a.keys = c->total.keys, a.counts = c->total.counts, a.n = n;
        a.sheet_fwd = c->sheet_fwd, a.sheet_rc = c->sheet_rc, a.group = c->sheet_group;
        a.use_rc = use_rc_rows ? c->sheet_use_rc : nullptr;
        a.rows = c->rows, a.l1 = c->l1, a.l2 = c->l2, a.n_subs = n_subs, a.rc_mode = rc_mode;
        a.m1 = c->m1, a.m2 = c->m2, a.srow = c->srow, a.type = c->type;
        a.m2rc = c->m2rc, a.srowrc = c->srowrc, a.typerc = c->typerc;
        a.f_sum = c->f_sum, a.rc_sum = c->rc_sum, a.st = c->st;
        a.work = c->work, a.work_n = c->work_n;
        // An rc pass tried both orientations of every row, so its idx1 verdicts (and its work list) carry
        // over to any per-row choice of orientation over the same keys / sheet / n (F:618-630).
        const bool reuse = !rc_mode && c->m1_from_rc && c->m1_total_gen == c->total_gen &&
                           c->m1_sheet_gen == c->sheet_gen && c->m1_n_subs == n_subs;
        c->m1_total_gen = c->total_gen, c->m1_sheet_gen = c->sheet_gen, c->m1_n_subs = n_subs;
        c->m1_from_rc = rc_mode != 0;
        ProfScope ps(c, FRB_K_MATCH);
        if (c->wide) {  // sweeps over the split idx1 / idx2 words (no candidate tables for wide keys)
            WideMatchArgs w{a, c->total.keys_hi, c->sheet_fwd_hi, c->sheet_rc_hi};
            if (!reuse) {
                CU(c, cudaMemsetAsync(c->work_n, 0, 8, c->compute));
                match_idx1_wide_kernel<<<grid_for(n, kMatchThreads, c->sm_count, 8), kMatchThreads,
                                         static_cast<size_t>(c->rows) * 8 + 16, c->compute>>>(w);
                c->launches++;
            } else {
                CU(c, cudaMemsetAsync(c->m2, 0xFF, n * 4, c->compute));
                CU(c, cudaMemsetAsync(c->srow, 0xFF, n * 4, c->compute));
                CU(c, cudaMemsetAsync(c->type, 0, n, c->compute));
            }
            match_wide_kernel<<<grid_for(n, kMatchThreads, c->sm_count, 8), kMatchThreads,
                                static_cast<size_t>(c->rows) * (5 * 8 + 4) + 16, c->compute>>>(w);
            c->launches++;
            CU(c, cudaGetLastError());
        } else {
        // candidate rows from per-part tables instead of a sweep over the sheet, whenever the shape allows
        static const bool sweep_only = getenv("FRB_MATCH") && strcmp(getenv("FRB_MATCH"), "sweep") == 0;
        const unsigned parts = n_subs + 1;
        const unsigned slots = static_cast<unsigned long long>(c->rows) * parts * 2 <= 2048 ? 2048u : 4096u;
        const bool cand = !sweep_only && c->rows > 0 && c->l2 > 0 && parts_usable(c->l1, n_subs, c->rows, slots) &&
                          parts_usable(c->l2, n_subs, c->rows, slots);
        if (!reuse) {
            CU(c, cudaMemsetAsync(c->work_n, 0, 8, c->compute));
            if (cand)
                match_idx1_cand_kernel<<<grid_for(n, kMatchThreads, c->sm_count, 4), kMatchThreads,
                                         cand_bytes(c->rows, parts, slots) + 16, c->compute>>>(a, slots);
            else
                match_idx1_kernel<<<grid_for(n, kMatchThreads, c->sm_count, 8), kMatchThreads,
                                    static_cast<size_t>(c->rows) * 8 + 16, c->compute>>>(a);
            c->launches++;
        } else {
            // keys off the work list stay undetermined; m1 is already -1 for them
            CU(c, cudaMemsetAsync(c->m2, 0xFF, n * 4, c->compute));
            CU(c, cudaMemsetAsync(c->srow, 0xFF, n * 4, c->compute));
            CU(c, cudaMemsetAsync(c->type, 0, n, c->compute));
        }
        if (cand) {
            const size_t smem = static_cast<size_t>(c->rows) * 24 + 32 + (rc_mode ? 2 : 1) * cand_bytes(c->rows, parts, slots);
            match_cand_kernel<<<grid_for(n, kMatchThreads, c->sm_count, 4), kMatchThreads, smem, c->compute>>>(a, slots);
        } else {
            const size_t smem = static_cast<size_t>(c->rows) * (4 * 8 + 4) + 16;
            match_kernel<<<grid_for(n, kMatchThreads, c->sm_count, 8), kMatchThreads, smem, c->compute>>>(a);
        }
        c->launches++;
        CU(c, cudaGetLastError());
        }
    }
    if (n) {
        if (m1_row) CU(c, cudaMemcpyAsync(m1_row, c->m1, n * 4, cudaMemcpyDeviceToHost, c->compute));
        if (m2_row) CU(c, cudaMemcpyAsync(m2_row, c->m2, n * 4, cudaMemcpyDeviceToHost, c->compute));
        if (type) CU(c, cudaMemcpyAsync(type, c->type, n, cudaMemcpyDeviceToHost, c->compute));
        if (sample_row) CU(c, cudaMemcpyAsync(sample_row, c->srow, n * 4, cudaMemcpyDeviceToHost, c->compute));
        if (rc_mode) {
            if (m2rc_row) CU(c, cudaMemcpyAsync(m2rc_row, c->m2rc, n * 4, cudaMemcpyDeviceToHost, c->compute));
            if (type_rc) CU(c, cudaMemcpyAsync(type_rc, c->typerc, n, cudaMemcpyDeviceToHost, c->compute));
            if (sample_rc_row) CU(c, cudaMemcpyAsync(sample_rc_row, c->srowrc, n * 4, cudaMemcpyDeviceToHost, c->compute));
        }
    }
    if (f_sum && c->rows) CU(c, cudaMemcpyAsync(f_sum, c->f_sum, c->rows * 8, cudaMemcpyDeviceToHost, c->compute));
    if (rc_sum && c->rows) CU(c, cudaMemcpyAsync(rc_sum, c->rc_sum, c->rows * 8, cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaStreamSynchronize(c->compute));
    return device_error_check(c);
}

// demux_ok per unique key of the total list + which files hold a key they should not (F:504-564), on the device.
// match: (4 + sheet rows) x n_files bytes made by the host with the reference's regexes; file_keys == NULL: the
// per-file lists of this context (n_files == files scanned); else host arrays (file lists that live elsewhere:
// other ranks, other streams).  Needs the classification of the LAST frb_match over the current total list.
int frb_demux_ok(frb_ctx* c, const uint8_t* match, uint32_t n_files, const uint64_t* const* file_keys,
                 const uint64_t* const* file_counts, const uint64_t* file_n, uint8_t* ok_out, uint8_t* bad_files_out,
                 int32_t* err_row_out) {
    CU(c, cudaSetDevice(c->device));
    if (!c->total_ready) return fail(c, FRB_ERR_STATE, "frb_demux_ok: no total list");
    const uint64_t n = c->total.n;
    if (n > c->match_cap || c->m1_total_gen != c->total_gen)
        return fail(c, FRB_ERR_STATE, "frb_demux_ok: frb_match over the current total list first");
    if (!file_keys && n_files != c->files.size()) return fail(c, FRB_ERR_ARG, "frb_demux_ok: %u files, context holds %zu", n_files, c->files.size());
    if (file_keys && c->wide) return fail(c, FRB_ERR_STATE, "frb_demux_ok: host file lists are not available on a wide (128-bit key) context");
    if (err_row_out) *err_row_out = 0x7FFFFFFF;
    if (n_files) memset(bad_files_out, 0, n_files);
    if (!n || !n_files) return FRB_OK;
    const size_t classes = 4 + static_cast<size_t>(c->rows);
    unsigned long long *sorted_keys = nullptr, *sorted_hi = nullptr, *hi_by_lo = nullptr;
    unsigned *i0 = nullptr, *i1 = nullptr;
    unsigned char *d_match = nullptr, *d_ok = nullptr, *d_bad = nullptr;
    int* d_err = nullptr;
    TRY(dmalloc(c, &sorted_keys, n * 8));
    TRY(dmalloc(c, &i0, n * 4));
    TRY(dmalloc(c, &i1, n * 4));
    TRY(dmalloc(c, &d_match, classes * n_files));
    TRY(dmalloc(c, &d_ok, n));
    TRY(dmalloc(c, &d_bad, n_files));
    TRY(dmalloc(c, &d_err, 4));
    CU(c, cudaMemcpyAsync(d_match, match, classes * n_files, cudaMemcpyHostToDevice, c->compute));
    CU(c, cudaMemsetAsync(d_ok, 1, n, c->compute));
    CU(c, cudaMemsetAsync(d_bad, 0, n_files, c->compute));
    CU(c, cudaMemsetAsync(d_err, 0x7F, 4, c->compute));
    {
        ProfScope ps(c, FRB_K_EXPORT);
        iota_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(i0, n);
        size_t tmp = 0;
        CU(c, cub::DeviceRadixSort::SortPairs(nullptr, tmp, c->total.keys, sorted_keys, i0, i1, static_cast<int>(n), 0, 63,
                                              c->compute));
        TRY(ensure_cub_tmp(c, tmp));
        CU(c, cub::DeviceRadixSort::SortPairs(c->cub_tmp, tmp, c->total.keys, sorted_keys, i0, i1, static_cast<int>(n), 0, 63,
                                              c->compute));
        if (c->wide) {
            // second, stable pass on the upper words: sorted by (hi, lo); i1 ends as the permutation of that order
            TRY(dmalloc(c, &hi_by_lo, n * 8));
            TRY(dmalloc(c, &sorted_hi, n * 8));
            gather1_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(i1, c->total.keys_hi, hi_by_lo, n);
            CU(c, cub::DeviceRadixSort::SortPairs(nullptr, tmp, hi_by_lo, sorted_hi, i1, i0, static_cast<int>(n), 0, 63, c->compute));
            TRY(ensure_cub_tmp(c, tmp));
            CU(c, cub::DeviceRadixSort::SortPairs(c->cub_tmp, tmp, hi_by_lo, sorted_hi, i1, i0, static_cast<int>(n), 0, 63, c->compute));
            std::swap(i0, i1);
            gather1_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(i1, c->total.keys, sorted_keys, n);
            c->launches += 2;
        }
        for (uint32_t f = 0; f < n_files; ++f) {
            const unsigned long long *fk = nullptr, *fc = nullptr;
            unsigned long long *up_k = nullptr, *up_c = nullptr;
            uint64_t nf = 0;
            if (file_keys) {
                nf = file_n[f];
                if (!nf) continue;
                TRY(dmalloc(c, &up_k, nf * 8));
                CU(c, cudaMemcpyAsync(up_k, file_keys[f], nf * 8, cudaMemcpyHostToDevice, c->compute));
                if (file_counts && file_counts[f]) {
                    TRY(dmalloc(c, &up_c, nf * 8));
                    CU(c, cudaMemcpyAsync(up_c, file_counts[f], nf * 8, cudaMemcpyHostToDevice, c->compute));
                }
                fk = up_k, fc = up_c;
            } else {
                nf = c->files[f].n;
                if (!nf) continue;
                fk = c->files[f].keys, fc = c->files[f].counts;
            }
            if (c->wide)
                demux_ok_wide_kernel<<<static_cast<unsigned>((nf + 255) / 256), 256, 0, c->compute>>>(
                    fk, c->files[f].keys_hi, fc, nf, sorted_keys, sorted_hi, i1, n, c->type, c->srow, d_match, n_files, f,
                    d_ok, d_bad, d_err);
            else
                demux_ok_kernel<<<static_cast<unsigned>((nf + 255) / 256), 256, 0, c->compute>>>(
                    fk, fc, nf, sorted_keys, i1, n, c->type, c->srow, d_match, n_files, f, d_ok, d_bad, d_err);
            c->launches++;
            if (up_k) TRY(dfree(c, up_k));
            if (up_c) TRY(dfree(c, up_c));
        }
        CU(c, cudaGetLastError());
    }
    int err_row = 0x7FFFFFFF;
    CU(c, cudaMemcpyAsync(ok_out, d_ok, n, cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaMemcpyAsync(bad_files_out, d_bad, n_files, cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaMemcpyAsync(&err_row, d_err, 4, cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaStreamSynchronize(c->compute));
    if (err_row_out) *err_row_out = err_row == 0x7F7F7F7F ? 0x7FFFFFFF : err_row;
    TRY(dfree(c, sorted_keys));
    TRY(dfree(c, sorted_hi));
    TRY(dfree(c, hi_by_lo));
    TRY(dfree(c, i0));
    TRY(dfree(c, i1));
    TRY(dfree(c, d_match));
    TRY(dfree(c, d_ok));
    TRY(dfree(c, d_bad));
    TRY(dfree(c, d_err));
    return device_error_check(c);
}

// ---- synthetic input ------------------------------------------------------------------------
int frb_synth_load(frb_ctx* c, uint64_t seed, uint32_t l1, uint32_t l2, uint32_t n_samples, const uint32_t* emit_i7,
                   const uint32_t* emit_i5, const uint64_t* cdf, uint32_t lane, uint32_t read_len, uint32_t sub_t,
                   uint32_t n_t, uint64_t rand_t, uint64_t hop_t) {
    CU(c, cudaSetDevice(c->device));
    if (l1 > 12 || l2 > 12 || n_samples == 0 || lane > 9) return fail(c, FRB_ERR_ARG, "frb_synth_load: bad shape");
    cudaFree(c->synth_i7), cudaFree(c->synth_i5), cudaFree(c->synth_cdf);
    CU(c, cudaMalloc(&c->synth_i7, n_samples * 4));
    CU(c, cudaMalloc(&c->synth_i5, n_samples * 4));
    CU(c, cudaMalloc(&c->synth_cdf, n_samples * 8));
    CU(c, cudaMemcpy(c->synth_i7, emit_i7, n_samples * 4, cudaMemcpyHostToDevice));
    CU(c, cudaMemcpy(c->synth_i5, emit_i5, n_samples * 4, cudaMemcpyHostToDevice));
    CU(c, cudaMemcpy(c->synth_cdf, cdf, n_samples * 8, cudaMemcpyHostToDevice));
    SynthArgs& a = c->synth;
    a.seed = seed, a.emit_i7 = c->synth_i7, a.emit_i5 = c->synth_i5, a.cdf = c->synth_cdf;
    a.rand_t = rand_t, a.hop_t = hop_t, a.l1 = l1, a.l2 = l2, a.n_samples = n_samples, a.lane = lane;
    a.read_len = read_len, a.sub_t = sub_t, a.n_t = n_t;
    c->synth_ready = true;
    return FRB_OK;
}

int frb_synth_generate(frb_ctx* c, uint64_t g0, uint64_t g1, int read_no, void* dev_out, uint64_t cap_bytes,
                       uint64_t* nbytes) {
    CU(c, cudaSetDevice(c->device));
    if (!c->synth_ready) return fail(c, FRB_ERR_STATE, "frb_synth_generate: frb_synth_load first");
    if (g1 < g0 || g1 - g0 >= (1ULL << 31)) return fail(c, FRB_ERR_ARG, "frb_synth_generate: bad range");
    const uint64_t n = g1 - g0;
    *nbytes = 0;
    if (n == 0) return FRB_OK;
    if (n > c->synth_cap) {
        cudaFree(c->synth_len), cudaFree(c->synth_off);
        c->synth_cap = 0;
        CU(c, cudaMalloc(&c->synth_len, n * 8));
        CU(c, cudaMalloc(&c->synth_off, n * 8));
        c->synth_cap = n;
    }
    SynthArgs a = c->synth;
    a.g0 = g0, a.n = n, a.read_no = read_no;
    synth_len_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->compute>>>(a, c->synth_len);
    size_t tmp = 0;
    CU(c, cub::DeviceScan::ExclusiveSum(nullptr, tmp, c->synth_len, c->synth_off, static_cast<int>(n), c->compute));
    TRY(ensure_cub_tmp(c, tmp));
    CU(c, cub::DeviceScan::ExclusiveSum(c->cub_tmp, tmp, c->synth_len, c->synth_off, static_cast<int>(n), c->compute));
    unsigned long long last_off = 0, last_len = 0;
    CU(c, cudaMemcpyAsync(&last_off, c->synth_off + (n - 1), 8, cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaMemcpyAsync(&last_len, c->synth_len + (n - 1), 8, cudaMemcpyDeviceToHost, c->compute));
    CU(c, cudaStreamSynchronize(c->compute));
    const uint64_t total = last_off + last_len;
    if (total > cap_bytes) return fail(c, FRB_ERR_ARG, "frb_synth_generate: need %llu bytes, buffer has %llu",
                                       (unsigned long long)total, (unsigned long long)cap_bytes);
    synth_write_kernel<<<grid_for(n * 32, 256, c->sm_count, 8), 256, 0, c->compute>>>(
        a, c->synth_off, static_cast<unsigned char*>(dev_out));
    CU(c, cudaGetLastError());
    CU(c, cudaStreamSynchronize(c->compute));
    *nbytes = total;
    return FRB_OK;
}

// ---- measurement ----------------------------------------------------------------------------
int frb_timer_start(frb_ctx* c) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaEventRecord(c->t0, c->compute));
    return FRB_OK;
}
int frb_timer_stop(frb_ctx* c, float* ms) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaEventRecord(c->t1, c->compute));
    CU(c, cudaEventSynchronize(c->t1));
    CU(c, cudaEventElapsedTime(ms, c->t0, c->t1));
    return FRB_OK;
}
int frb_prof_enable(frb_ctx* c, int on) {
    c->prof = on != 0;
    return FRB_OK;
}
int frb_prof_read(frb_ctx* c, int kclass, double* ms_total, uint64_t* launches, int reset) {
    if (kclass < 0 || kclass >= FRB_K_NUM) return fail(c, FRB_ERR_ARG, "bad kernel class");
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->compute));
    prof_collect(c);
    if (ms_total) *ms_total = c->prof_ms[kclass];
    if (launches) *launches = c->prof_n[kclass];
    if (reset) c->prof_ms[kclass] = 0, c->prof_n[kclass] = 0;
    return FRB_OK;
}
uint64_t frb_launch_count(frb_ctx* c) { return c->launches; }

}  // extern "C"

#include "frb_route.inl"
#include "frb_nccl.inl"
#include "frb_csv.inl"
