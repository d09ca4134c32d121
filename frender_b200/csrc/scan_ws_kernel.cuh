// Hot path A, general form: read-name parse + 3-bit key packing (+ unique-combination count) with the exact read
// ordinal of every header known BEFORE anything is written.  Serves what the speculative tally kernel
// (scan_spec_kernel.cuh) does not: per-read outputs for the demux router (keys under the demux rule F:778, record
// offsets), the -s head sample (F:163-165) and the clock instrumentation.
//
// Every tile's line phase comes from a decoupled look-back over the newline counts the counters publish:
//
//   warps 0-3  COUNTERS    count_tile (scan_count.cuh): newline mask, scan, newline list, guess; publish the tile's
//                          newline count at once, signal `counted[stage]`.
//   warps 4-6  EXTRACTORS  one thread per header line: key extraction, fold inside the warp, key batch into a
//                          shared-memory ring for the committer; thread 0 then refills the stage (ticket + bulk
//                          copy).  With a guess they do not wait for the look-back, without one (always the case
//                          when per-read outputs or -s are on) they ask the committer for the count first.
//   warp  7    COMMITTER   per tile: look-back over the published counts (the only wait on other CTAs), check of
//                          a guess against it, bookkeeping; per batch: deferred table updates.  Tiles whose guess
//                          was wrong go to scan_redo_kernel.
//
// With 3 CTAs per SM the launch register budget is re-split between the two warpgroups (setmaxnreg): counters 48,
// extractors + committer 112.
#pragma once
#include "scan_count.cuh"

namespace frb {

template <class G>
__global__ void __launch_bounds__(G::threads) __maxnreg__(G::maxreg) scan_ws_kernel(const ScanArgs a_in) {
    ScanArgs a = a_in;
    a.skip = a.skip_ptr ? *a.skip_ptr : 0ULL;
    constexpr int kRule = kRuleRuntime;
    constexpr int kStages = G::stages;
    constexpr int kWsTile = G::tile, kWsBuf = G::buf, kWsNlCap = G::nl_cap, kWsPerThread = G::per_thread;
    constexpr int kExt = G::xgroup, kXWarps = G::xwarps;
    constexpr int kBatches = 3;  // key batches in flight between the extractors and the committer
    extern __shared__ __align__(128) unsigned char smem[];
    uint16_t* const s_nl = reinterpret_cast<uint16_t*>(smem + kStages * kWsBuf);
    __shared__ __align__(8) unsigned long long s_full[kStages], s_counted[kStages];
    __shared__ unsigned s_tile[kStages], s_total[kStages], s_valid[kStages], s_vnl[kStages], s_guess[kStages];
    __shared__ unsigned s_cwarp[kWsGroup / 32];
    __shared__ unsigned s_halo[kStages];
    // prefix of local tile i for the extractors that asked for it: ((i + 1) & 0xFFFFFF) << 40 | newlines before
    // the tile (< 2^40), one word so that no fence is needed between value and flag (a fence in the committer
    // waits for its outstanding table atomics)
    __shared__ volatile unsigned long long s_prefix[4];
    __shared__ __align__(8) unsigned long long s_bfull[kBatches], s_bfree[kBatches];
    __shared__ unsigned long long s_keys[kBatches][kExt];  // kEmpty except on the first lane of every run of equal keys
    __shared__ unsigned char s_kcnt[kBatches][kExt];      // reads folded into that entry
    __shared__ unsigned long long s_keys_hi[kBatches][G::wide ? kExt : 1];  // wide context: upper words
    __shared__ unsigned s_bmeta[kBatches][8];  // see BM_* below
    __shared__ unsigned s_berr[kBatches][kXWarps];
    __shared__ unsigned char s_lut[256];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long L0 =
        a.use_carry ? *reinterpret_cast<volatile unsigned long long*>(&a.st->line_carry) : a.line_base;
    const unsigned long long chunk_first_read = (L0 + 3) >> 2;
    volatile unsigned long long* status = a.status + 1;
    const bool timing = a.timing != nullptr;

    for (int i = tid; i < 256; i += G::threads) s_lut[i] = lut_entry(i, a.rule);
    if (tid == 0) {
        s_prefix[0] = 0, s_prefix[1] = 0, s_prefix[2] = 0, s_prefix[3] = 0;
        if (blockIdx.x == 0) a.st->chunk_l0 = L0;
#pragma unroll
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&s_full[i], 1);
            mbar_init(&s_counted[i], 1);
        }
#pragma unroll
        for (int i = 0; i < kBatches; ++i) {
            mbar_init(&s_bfull[i], kXWarps);
            mbar_init(&s_bfree[i], 1);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp < kWsGroup / 32) {
        if constexpr (G::split_regs) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(48));
        // =============================== COUNTERS ================================================
        const int ct = tid;
        unsigned full_parity = 0;  // bit s
        long long tm = (timing && ct == 0) ? clock64() : 0;
        unsigned long long t_wait = 0, t_work = 0;
        // may the line phase be guessed from the text at all?  (per-read outputs and -s need the exact
        // read ordinal before extraction)
        const bool may_guess = !a.no_guess && !a.keys_out && !a.rec_off_out && a.read_limit == ~0ULL;
        for (unsigned i = 0;; ++i) {
            const int s = i % kStages;
            mbar_wait(&s_full[s], (full_parity >> s) & 1u);
            full_parity ^= 1u << s;
            if (timing && ct == 0) { const long long now = clock64(); t_wait += now - tm; tm = now; }
            const unsigned t = s_tile[s];
            if (t == kNoTile) {
                if (ct == 0) mbar_arrive(&s_counted[s]);
                break;
            }
            // the tile's newline count goes out the moment it is known (inside count_tile): every later tile's
            // look-back waits for it
            const TileMeta m = count_tile<G, true>(a, smem + s * kWsBuf, s_nl + s * kWsNlCap, s_cwarp, t, may_guess, status);
            if (ct == 0) {
                const unsigned long long left = a.nbytes - static_cast<unsigned long long>(t) * kWsTile;
                s_halo[s] = m.halo, s_total[s] = m.total, s_vnl[s] = m.vnl, s_guess[s] = m.guess;
                s_valid[s] = static_cast<unsigned>(left < kWsTile ? left : kWsTile);
                mbar_arrive(&s_counted[s]);
            }
            if (timing && ct == 0) { const long long now = clock64(); t_work += now - tm; tm = now; }
        }
        if (timing && ct == 0) atomicAdd(&a.timing[0], t_wait), atomicAdd(&a.timing[1], t_work);
    } else {
        if constexpr (G::split_regs) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(112));
        // =============================== EXTRACTORS + COMMITTER ====================================
        // Batch descriptor words (s_bmeta): local tile index, global tile, first header index of the
        // batch, entries, newlines in the tile, lines (newlines + unterminated last line), guessed j0,
        // flags.
        enum { BM_I, BM_T, BM_H0, BM_N, BM_TOTAL, BM_LINES, BM_J0, BM_FLAGS };
        enum { BF_FIRST = 1, BF_GUESSED = 2, BF_NEED_PREFIX = 4, BF_DENSE = 8, BF_END = 16 };
        const int pt = tid - kWsGroup;
        const int pwarp = warp - kWsGroup / 32;
        unsigned counted_parity = 0;
        if (pwarp < kXWarps) {
            // ------------------------- extractor warps -------------------------------------------------
            // Key extraction needs to know WHICH lines of the tile are header lines (line number mod 4) and
            // nothing else from the look-back.  The counters' guess gives that without waiting for other
            // CTAs; keys go to the committer, which checks the guess against the newline count before
            // anything reaches the table.  A wrong guess (input that is not well-formed FASTQ) sends the
            // tile to scan_redo_kernel; without a guess the extractors ask the committer for the count
            // first.  Either way every tile is tallied by line COUNT, exactly as F:161-169 does.
            // The extractors issue no global atomics, so none of their barrier arrivals waits for one.
            // a wide context's keys_out holds out_cap lower words, then out_cap upper words
            unsigned long long key_hi = 0;  // wide context: upper word of this thread's key
            auto emit = [&](unsigned long long o, unsigned long long key, unsigned long long start_g) {
                const unsigned long long slot = o - chunk_first_read;
                if (slot < a.out_cap) {
                    if (a.keys_out) a.keys_out[slot] = key;
                    if constexpr (G::wide) {
                        if (a.keys_out) a.keys_out[a.out_cap + slot] = key < kBadKeyBase ? key_hi : 0ULL;
                    }
                    if (a.rec_off_out) a.rec_off_out[slot] = start_g;
                }
            };
            auto issue = [&](int s, unsigned ticket) {  // ticket -> stage s, start its bulk copy
                const unsigned t = ticket < a.n_tiles ? ticket : kNoTile;
                s_tile[s] = t;
                if (t == kNoTile) {
                    mbar_arrive(&s_full[s]);
                    return;
                }
                const unsigned long long off = static_cast<unsigned long long>(t) * kWsTile;
                const unsigned halo = t ? kHalo : 0;
                const unsigned long long left = a.nbytes - off;
                const unsigned avail = static_cast<unsigned>(left < kWsTile ? left : kWsTile) + halo;
                const unsigned bulk = avail & ~15u;
                if (bulk) {
                    mbar_expect_tx(&s_full[s], bulk);
                    bulk_g2s(smem + s * kWsBuf + (kHalo - halo), a.data + off - halo, bulk, &s_full[s]);
                } else {
                    mbar_arrive(&s_full[s]);
                }
            };
            const unsigned long long read_limit = a.read_limit;
            unsigned nb = 0;  // batches sent
            // hand one batch to the committer: keys (kEmpty = none), first parse error, descriptor
            auto send = [&](unsigned long long key, int rc, unsigned i, unsigned t, unsigned h0, unsigned n,
                            unsigned total, unsigned lines, unsigned j0, unsigned flags) {
                const unsigned b = nb % kBatches;
                // fold equal keys of the warp: the lowest lane (lowest read ordinal) carries the count
                unsigned cnt = 0;
                if (n) {
                    const unsigned grp = __ballot_sync(0xFFFFFFFFu, key != kEmpty);
                    if (key != kEmpty) {
                        unsigned same = __match_any_sync(grp, key);
                        if constexpr (G::wide) same &= __match_any_sync(grp, key_hi);
                        if (lane == __ffs(same) - 1) cnt = __popc(same);
                        else key = kEmpty;
                    }
                }
                mbar_wait(&s_bfree[b], ((nb / kBatches) & 1u) ^ 1u);
                if (n) s_keys[b][pt] = key, s_kcnt[b][pt] = static_cast<unsigned char>(cnt);
                if constexpr (G::wide) {
                    if (n) s_keys_hi[b][pt] = key_hi;
                }
                const unsigned e = __reduce_min_sync(0xFFFFFFFFu, rc ? ((static_cast<unsigned>(pt) << 8) | static_cast<unsigned>(-rc)) : 0xFFFFFFFFu);
                if (lane == 0) s_berr[b][pwarp] = e;
                if (pt == 0) {
                    unsigned* m = s_bmeta[b];
                    m[BM_I] = i, m[BM_T] = t, m[BM_H0] = h0, m[BM_N] = n, m[BM_TOTAL] = total, m[BM_LINES] = lines;
                    m[BM_J0] = j0, m[BM_FLAGS] = flags;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&s_bfull[b]);
                ++nb;
            };
            auto wait_prefix = [&](unsigned i) -> unsigned long long {
                unsigned long long word;
                do {
                    word = s_prefix[i & 3];
                } while ((word >> 40) != ((i + 1) & 0xFFFFFFu));
                return L0 + (word & ((1ULL << 40) - 1));
            };
            unsigned long long next_ticket = 0;
            if (pt == 0) {
                for (int s = 0; s < kStages; ++s) issue(s, static_cast<unsigned>(atomicAdd(&a.status[0], 1ULL)));
            }
            long long tm = (timing && pt == 0) ? clock64() : 0;
            unsigned long long tp[4] = {0, 0, 0, 0};
            auto tick = [&](int k) {
                if (timing && pt == 0) { const long long now = clock64(); tp[k] += now - tm; tm = now; }
            };
            for (unsigned i = 0;; ++i) {
                const int s = i % kStages;
                mbar_wait(&s_counted[s], (counted_parity >> s) & 1u);
                counted_parity ^= 1u << s;
                tick(0);
                const unsigned t = s_tile[s];
                if (t == kNoTile) {
                    send(0, 0, i, t, 0, 0, 0, 0, 0, BF_END);
                    break;
                }
                if (pt == 0) {  // ticket for the refill at the end of this tile; its round trip hides here
                    asm volatile("atom.global.add.u64 %0, [%1], 1;" : "=l"(next_ticket) : "l"(a.status) : "memory");
                }
                unsigned char* const buf = smem + s * kWsBuf;
                const unsigned total = s_total[s], vnl = s_vnl[s], guess = s_guess[s];
                const unsigned lines = total + vnl;
                const unsigned halo_start = s_halo[s];
                const unsigned long long tile_off = static_cast<unsigned long long>(t) * kWsTile;
                const uint16_t* const nl = s_nl + s * kWsNlCap;
                if (lines > static_cast<unsigned>(kWsNlCap)) {
                    // more newlines than the list holds (lines < 20 bytes on average): scan_redo_kernel
                    send(0, 0, i, t, 0, 0, total, lines, 0, BF_FIRST | BF_DENSE);
                } else {
                    const bool guessed = guess != kNoGuess;
                    unsigned j0 = guess;
                    unsigned long long of = 0;  // first read ordinal owned by the tile (known if !guessed)
                    unsigned flags = BF_FIRST | (guessed ? BF_GUESSED : 0u);
                    if (!guessed) {
                        send(0, 0, i, t, 0, 0, total, lines, 0, BF_FIRST | BF_NEED_PREFIX);
                        const unsigned long long K0 = wait_prefix(i);
                        j0 = static_cast<unsigned>((4 - (K0 & 3)) & 3);
                        of = (K0 + 3) >> 2;
                        flags = 0;
                    }
                    const unsigned n_owned = lines > j0 ? (lines - j0 + 3) / 4 : 0;
#pragma unroll 1
                    for (unsigned h0 = 0; h0 < n_owned; h0 += kExt) {
                        const unsigned h = h0 + pt;
                        bool have = h < n_owned && (guessed || of + h < read_limit);
                        unsigned long long key = kEmpty, start_g = 0;
                        int rc = 0;
                        if (have) {
                            const unsigned j = j0 + 4 * h;
                            const unsigned sb = j ? nl[j - 1] + 1u : halo_start;
                            if constexpr (G::wide) {
                                rc = parse_header_wide<true>(buf, s_lut, sb, nl[j], a, tile_off, &key, &key_hi, &start_g);
                            } else {
                                rc = parse_header<kRule, true>(buf, s_lut, sb, nl[j], a, tile_off, &key, &start_g);
                            }
                            if (rc && a.rule == FRB_RULE_DEMUX && a.keys_out && !a.table) {  // the router decides whether it matters
                                emit(of + h, kBadKeyBase + static_cast<unsigned long long>(-rc), start_g);
                                key = kEmpty, rc = 0;
                            } else if (rc) {
                                key = kEmpty;
                            } else if (!guessed) {
                                emit(of + h, key, start_g);
                            }
                        }
                        tick(1);
                        const unsigned n = n_owned - h0 < static_cast<unsigned>(kExt) ? n_owned - h0 : kExt;
                        send(key, rc, i, t, h0, n, total, lines, j0, flags);
                        flags &= ~static_cast<unsigned>(BF_FIRST);
                        tick(2);
                    }
                }
                group_sync<kExt>(3);  // every extractor is done reading stage s
                if (pt == 0) {
                    issue(s, static_cast<unsigned>(next_ticket));
                    tp[3] += 1;
                }
                tick(0);
            }
            if (timing && pt == 0) {
                atomicAdd(&a.timing[2], tp[0]), atomicAdd(&a.timing[7], tp[1]), atomicAdd(&a.timing[8], tp[2]);
                atomicAdd(&a.timing[9], tp[3]);
            }
        } else {
            // ------------------------- committer warp --------------------------------------------------
            // Per tile: look-back over the published counts (the only place a CTA waits on other CTAs),
            // check of the guess, bookkeeping; per batch: update the table.
            // Table updates are deferred in three steps -- slot load, then RED or CAS one batch later,
            // then the RED after a CAS one batch after that -- so no L2 round trip is waited for in line.
            constexpr int kRounds = kExt / 32;
            const unsigned long long read_limit = a.read_limit;
            unsigned long long p_key[kRounds], p_pos[kRounds], p_slot[kRounds], p_seen[kRounds];
            unsigned long long q_key[kRounds], q_pos[kRounds], q_slot[kRounds], q_old[kRounds];
            unsigned p_cnt[kRounds], q_cnt[kRounds];
#pragma unroll
            for (int r = 0; r < kRounds; ++r) {
                p_cnt[r] = 0, q_cnt[r] = 0, q_slot[r] = 0, q_key[r] = 0, q_old[r] = 0, q_pos[r] = 0;
                p_key[r] = 0, p_pos[r] = 0, p_slot[r] = 0, p_seen[r] = 0;
            }
            auto bump = [&](unsigned long long slot, unsigned cnt, unsigned long long pos) {
                atomicAdd(&a.table[slot].count, static_cast<unsigned long long>(cnt));
                atomicMin(&a.table[slot].first, pos);
            };
            // Step 2/3 of a set: its home slot did not hold the key.  Slot free: compare-and-swap, result
            // dropped (the instruction returns it in its compare register, the copy out of there would wait
            // for the L2 round trip on the spot), then a load of the same slot -- same thread, same address,
            // so it sees the slot after the swap.  Slot taken by another key: load of the next slot.  One
            // batch later the loaded key decides: ours -> count/first update; anything else (lost race, two
            // other keys in a row) -> the in-line probe loop, whose loads are L2 round trips.  Nobody knows
            // who won a slot, so the number of occupied slots is counted when the file ends.
            auto finish = [&](int r) {
                if (q_cnt[r]) {
                    if (q_old[r] == q_key[r]) {
                        bump(q_slot[r], q_cnt[r], q_pos[r]);
                    } else {
                        table_add(a.table, a.table_mask, q_key[r], q_cnt[r], q_pos[r], &a.st->occupied, a.st);
                    }
                    q_cnt[r] = 0;
                }
                const bool claim = p_cnt[r] && p_seen[r] == kEmpty;
                const bool look = p_cnt[r] && p_seen[r] != p_key[r];  // claim or re-probe: a q set is born
                if (p_cnt[r]) {
                    if (p_seen[r] == p_key[r]) {
                        bump(p_slot[r], p_cnt[r], p_pos[r]);
                    } else {
                        q_key[r] = p_key[r], q_pos[r] = p_pos[r], q_cnt[r] = p_cnt[r];
                        q_slot[r] = claim ? p_slot[r] : ((p_slot[r] + 1) & a.table_mask);
                    }
                    p_cnt[r] = 0;
                }
                asm volatile(
                    "{\n\t.reg .pred p, q;\n\t.reg .b64 t;\n\t"
                    "setp.ne.u32 p, %4, 0;\n\t"
                    "setp.ne.u32 q, %5, 0;\n\t"
                    "@p atom.global.cas.b64 t, [%1], %2, %3;\n\t"
                    "@q ld.volatile.global.u64 %0, [%1];\n\t}"
                    : "+l"(q_old[r])
                    : "l"(&a.table[q_slot[r] & a.table_mask].key), "l"(kEmpty), "l"(q_key[r]), "r"(claim ? 1u : 0u),
                      "r"(look ? 1u : 0u)
                    : "memory");
            };
            unsigned long long my_reads = 0, of = 0;
            bool tile_ok = false;
            long long tm = (timing && lane == 0) ? clock64() : 0;
            unsigned long long k_wait = 0, k_look = 0, k_commit = 0;
            auto ktick = [&](unsigned long long& acc) {
                if (timing && lane == 0) { const long long now = clock64(); acc += now - tm; tm = now; }
            };
            for (unsigned nb = 0;; ++nb) {
                const unsigned b = nb % kBatches;
                mbar_wait(&s_bfull[b], (nb / kBatches) & 1u);
                ktick(k_wait);
                const unsigned* m = s_bmeta[b];
                const unsigned flags = m[BM_FLAGS];
                if (flags & BF_END) break;
                const unsigned i = m[BM_I], t = m[BM_T], h0 = m[BM_H0], n = m[BM_N];
                if (flags & BF_FIRST) {
                    unsigned long long excl;
                    tile_prefix<true>(status, t, m[BM_TOTAL], lane, &excl);
                    const unsigned long long K0 = L0 + excl;
                    of = (K0 + 3) >> 2;
                    tile_ok = !(flags & BF_DENSE) &&
                              (!(flags & BF_GUESSED) || static_cast<unsigned>((4 - (K0 & 3)) & 3) == m[BM_J0]);
                    if (lane == 0) {
                        s_prefix[i & 3] = (static_cast<unsigned long long>((i + 1) & 0xFFFFFFu) << 40) | excl;
                        if (tile_ok) {
                            const unsigned long long o_end = (K0 + m[BM_LINES] + 3) >> 2;
                            const unsigned long long c_hi = o_end < read_limit ? o_end : read_limit;
                            if (c_hi > of) my_reads += c_hi - of;
                            if (t == a.n_tiles - 1) a.st->line_carry = K0 + m[BM_LINES];
                        } else {
                            a.redo[atomicAdd(&a.st->redo_n, 1ULL)] = t;
                        }
                    }
                    ktick(k_look);
                }
                unsigned long long key[kRounds], key_hi[kRounds];
                unsigned cnt[kRounds];
#pragma unroll
                for (int r = 0; r < kRounds; ++r) {
                    const unsigned idx = r * 32 + lane;
                    key[r] = (tile_ok && idx < n) ? s_keys[b][idx] : kEmpty;
                    cnt[r] = s_kcnt[b][idx];
                    if constexpr (G::wide) key_hi[r] = s_keys_hi[b][idx];
                }
                unsigned err = 0xFFFFFFFFu;
#pragma unroll
                for (int w = 0; w < kXWarps; ++w) err = min(err, s_berr[b][w]);
                __syncwarp();
                if (lane == 0) mbar_arrive(&s_bfree[b]);  // the batch is in registers
                if (tile_ok && n && err != 0xFFFFFFFFu && lane == 0) {
                    raise_error(a.st, -static_cast<int>(err & 0xFFu), of + h0 + (err >> 8));
                }
                if constexpr (G::wide) {
                    if (!a.table) continue;
                    // one probe loop per key (a 16-byte load, then the count / first updates or the claim)
#pragma unroll
                    for (int r = 0; r < kRounds; ++r) {
                        if (key[r] != kEmpty) {
                            table_add(reinterpret_cast<WideSlot*>(a.table), a.table_mask, Key128{key[r], key_hi[r]}, cnt[r],
                                      a.pos_base + of + h0 + r * 32 + lane, &a.st->occupied, a.st);
                        }
                    }
                } else if (a.table) {
#pragma unroll
                    for (int r = 0; r < kRounds; ++r) {
                        finish(r);  // the sets of the previous batch (their slot loads are long back)
                        if (key[r] != kEmpty) {
                            p_key[r] = key[r], p_pos[r] = a.pos_base + of + h0 + r * 32 + lane, p_cnt[r] = cnt[r];
                            p_slot[r] = hash64(key[r]) & a.table_mask;
                            p_seen[r] = *reinterpret_cast<volatile unsigned long long*>(&a.table[p_slot[r]].key);
                        }
                    }
                }
                ktick(k_commit);
            }
            if constexpr (!G::wide) {
#pragma unroll 1
                for (int k = 0; k < 2; ++k) {  // the second pass retires a CAS issued by the first
#pragma unroll
                    for (int r = 0; r < kRounds; ++r) finish(r);
                }
            }
            if (lane == 0 && my_reads) atomicAdd(&a.st->n_reads, my_reads);
            if (timing && lane == 0) {
                atomicAdd(&a.timing[3], k_look), atomicAdd(&a.timing[4], k_wait), atomicAdd(&a.timing[6], k_commit);
            }
        }
    }
}

// Tiles the warp-specialised kernel left out -- a guessed line phase that turned out wrong (input that is
// not well-formed FASTQ), or more newlines than a tile's position list holds -- tallied strictly by line
// count, one thread per tile, from the bytes in global memory.  status[] holds every tile's inclusive
// newline prefix by now.  Slow and exact; the list is empty for ordinary input.  A wide context (G::wide) never
// runs the speculative scan; its keys_out holds out_cap lower words, then out_cap upper words.
template <class G>
__global__ void __launch_bounds__(64) scan_redo_kernel(const ScanArgs a_in) {
    using K = KeyWidth<G::wide>;
    ScanArgs a = a_in;
    a.skip = a.skip_ptr ? *a.skip_ptr : 0ULL;
    // speculative path: a wrong guess somewhere in the chunk -> every tile is redone (the negate pass took the
    // guessed keys out again); a parse error of a guessed tile stands once all guesses are confirmed
    bool all = false;
    if constexpr (!G::wide) {
        all = a.composite && a.st->spec_bad;
        if (a.composite && !all && blockIdx.x == 0 && threadIdx.x == 0 && a.st->spec_err_code) {
            const unsigned long long p = a.st->spec_err_pos;
            raise_error(a.st, a.st->spec_err_code, a.tile_first[p >> kCompositeShift] + (p & ((1ULL << kCompositeShift) - 1)));
        }
    }
    const unsigned long long n = all ? a.n_tiles : a.st->redo_n;
    const unsigned long long L0 = a.st->chunk_l0;
    const unsigned long long chunk_first_read = (L0 + 3) >> 2;
    for (unsigned long long idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += static_cast<unsigned long long>(gridDim.x) * blockDim.x) {
        const unsigned t = all ? static_cast<unsigned>(idx) : a.redo[idx];
        const unsigned long long off = static_cast<unsigned long long>(t) * a.tile_bytes;
        const unsigned long long end = off + a.tile_bytes < a.nbytes ? off + a.tile_bytes : a.nbytes;
        unsigned long long k = L0 + (t ? (a.status[t] & kValMask) : 0ULL);  // a.status[1 + (t - 1)]
        unsigned long long prev = off > a.skip ? off : a.skip;
        while (prev > a.skip && a.data[prev - 1] != '\n') --prev;
        const bool vnl = t == a.n_tiles - 1 && end > off && end > a.skip && a.data[end - 1] != '\n';
        unsigned long long reads = 0;
        for (unsigned long long p = off > a.skip ? off : a.skip; p <= end; ++p) {
            const bool is_end = p < end ? a.data[p] == '\n' : vnl;
            if (!is_end) continue;
            if ((k & 3) == 0 && (k >> 2) < a.read_limit) {
                typename K::Key key{};
                int rc;
                if constexpr (G::wide) rc = parse_serial_wide(a.data + prev, p - prev, a.rule, &key.lo, &key.hi);
                else rc = a.rule == kRuleOffsetsOnly ? 0 : parse_serial(a.data + prev, p - prev, a.rule, &key);
                const unsigned long long pos =
                    !G::wide && a.composite ? (((a.tile_base + t) << kCompositeShift) | reads) : a.pos_base + (k >> 2);
                ++reads;
                // per-read key: the lower word, and for a wide context the upper word out_cap entries further on
                auto emit = [&](unsigned long long slot, typename K::Key out) {
                    if constexpr (G::wide) a.keys_out[slot] = out.lo, a.keys_out[a.out_cap + slot] = out.hi;
                    else a.keys_out[slot] = out;
                };
                if (rc && a.rule == FRB_RULE_DEMUX && a.keys_out && !a.table) {
                    const unsigned long long slot = (k >> 2) - chunk_first_read;
                    if (slot < a.out_cap) {
                        if (a.keys_out) emit(slot, typename K::Key{kBadKeyBase + static_cast<unsigned long long>(-rc)});
                        if (a.rec_off_out) a.rec_off_out[slot] = prev;
                    }
                } else if (rc) {
                    raise_error(a.st, rc, k >> 2);
                } else {
                    if (a.table)
                        table_add(reinterpret_cast<typename K::Slot*>(a.table), a.table_mask, key, 1, pos, &a.st->occupied, a.st);
                    const unsigned long long slot = (k >> 2) - chunk_first_read;
                    if (slot < a.out_cap) {
                        if (a.keys_out) emit(slot, key);
                        if (a.rec_off_out) a.rec_off_out[slot] = prev;
                    }
                }
            }
            prev = p + 1;
            ++k;
        }
        if (G::wide || !a.composite) {  // the speculative path takes both from the summed counts (spec_scan_kernel)
            if (reads) atomicAdd(&a.st->n_reads, reads);
            if (t == a.n_tiles - 1) a.st->line_carry = k;
        }
    }
}

}  // namespace frb
