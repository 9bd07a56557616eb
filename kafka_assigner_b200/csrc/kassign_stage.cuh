// kassign_stage.cuh — kernel A: sticky fill + orphan spread + conflict levels, one topic per warp, persistent CTAs.
// Reference: KTA:49-69, KAS:65-200, KAS:205-214 (see kassign_common.cuh for the map).
#pragma once
#include "kassign_common.cuh"

struct KaSolveParams {
    // problem
    int T;
    int topic_base;             // index of this block's first topic in the whole run (status reporting)
    const int32_t* topic_hash;  // [T]
    const int64_t* part_off;    // [T+1] or nullptr (dense: P partitions per topic)
    int P;
    const int64_t* rep_off;     // [Q+1] or nullptr (dense: RF replicas per row)
    int RF;
    const int32_t* cur;         // current replica lists (broker IDs)
    int desired_rf;
    int S;                      // row stride of the slab / output rows
    int Pmax;                   // max partitions of any topic (smem sizing)
    // broker table
    int N;
    const uint16_t* blob;       // global: rack16[Npad] | lut16[range_pad] (16B aligned, multiple of 16B)
    int blob_bytes;             // bytes staged into smem (rack, plus lut when lut_mode == SMEM)
    int lut_off;                // element offset (uint16) of lut16 inside blob
    int R;                      // number of distinct racks (compact ids 0..R-1 in rack16)
    int rackptr;                // 1: spread phase uses per-rack first-free pointers (R small); 0: window scan
    int roff_off;               // element offset of rack_off16[R+1] inside blob
    int memb_off;               // element offset of members16[N] (sorted indices grouped by rack, ascending) inside blob
    int rp_bytes;               // per-warp bytes of each of the three rack-pointer arrays
    int lut_mode;
    int min_id;
    uint32_t range;
    const uint16_t* glut;       // global lut16 (lut_mode == GLOBAL)
    const int32_t* broker_id;   // [N] ascending (global)
    // outputs (block-relative rows)
    int rec_kind;               // 3: 16 B records (S <= 3), else 32 B records (see kassign_common.cuh)
    void* rec;                  // [Q] partition records in schedule order
    uint16_t* perm;             // [Q] LEVELS && rec_kind == 3: partition ordinal (inside its topic) of each schedule position
    int chunk_w;                // LEVELS: a chunk = at most chunk_w records of one level (the order kernel's consumer threads)
    int32_t* ntl;               // [T] LEVELS: number of chunks of each topic
    uint32_t* lend;             // [Q] LEVELS: lend[g0 + i] = topic-relative end of the topic's i-th chunk (first ntl[t] entries)
    int4* tstatus;              // [T] per-topic error record (written only on error)
    unsigned* err_topic;        // unsigned atomicMin of the failing topic index (init = 0xFFFFFFFF)
};

// ------------------------------------------------------------------------------------------------
// Kernel A: sticky fill + orphan spread, one topic per warp, persistent CTAs.
// ------------------------------------------------------------------------------------------------
struct KaTab {               // CTA-shared views into the staged broker table
    const uint16_t* rack;    // [N] compact rack id of each broker (sorted-index order)
    const uint16_t* lut;     // [range] (lut_mode == SMEM)
    const uint16_t* roff;    // [R+1] member ranges per rack
    const uint16_t* memb;    // [N] sorted indices grouped by rack, ascending inside a rack
};

__device__ __forceinline__ uint32_t ka_lookup(int id, const KaTab& tab, const KaSolveParams& p) {
    return ka_id_index(id, tab.lut, p);
}

// Per-warp scratch of the conflict-level pass (LEVELS only).
struct KaLevelScratch {
    uint32_t* owner;   // [N] lane bitmask of the window's partitions holding each broker
    uint16_t* last;    // [N] level of the latest partition of this topic holding each broker
    uint16_t* lvl;     // [P] level of each partition
    uint16_t* lcur;    // [P+2] per-level cursor of the stable counting sort
};

// SM = compile-time bound on the row stride S (3 for every BASELINE config): sizes the per-partition rack lists of the spread
// phase, so that RF = 3 runs 3-wide compares instead of 8-wide ones.
template <typename LoadT, bool LEVELS, int SM>
__device__ void ka_solve_topic(const KaSolveParams& p, const KaTab& tab, int t, LoadT* load, uint16_t* slab, uint8_t* cnt,
                               uint16_t* rpos, uint16_t* rst, uint16_t* rkk, const KaLevelScratch& ls) {
    const int lane = threadIdx.x & 31;
    const uint32_t lt = ka_lanemask_lt();
    const int S = p.S;
    const int N = p.N;

    int64_t g0;
    int P;
    if (p.part_off) {
        g0 = p.part_off[t];
        P = (int)(p.part_off[t + 1] - g0);
    } else {
        P = p.P;
        g0 = (int64_t)t * P;
    }

    int err = 0, errp = -1, erra = 0, errb = 0;

    // ---- KTA:49-61 replication-factor inference / validation ------------------------------------
    int rf = p.desired_rf;
    int maxlen = 0;
    if (!p.rep_off) {
        maxlen = P > 0 ? p.RF : 0;
        if (rf < 0 && P > 0) rf = p.RF;
    } else {
        const int64_t* ro = p.rep_off + g0;
        int first = P > 0 ? (int)(ro[1] - ro[0]) : -1;
        int mism = 0x7FFFFFFF;
        for (int pp = lane; pp < P; pp += 32) {
            int sz = (int)(ro[pp + 1] - ro[pp]);
            maxlen = max(maxlen, sz);
            if (sz != first) mism = min(mism, pp);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            maxlen = max(maxlen, __shfl_xor_sync(KA_FULL, maxlen, o));
            mism = min(mism, __shfl_xor_sync(KA_FULL, mism, o));
        }
        if (rf < 0 && P > 0) {
            rf = first;
            if (mism != 0x7FFFFFFF) {  // first entry (ascending) whose size differs (KTA:57-60)
                err = KA_E_RF_MISMATCH;
                errp = mism;
                erra = (int)(ro[mism + 1] - ro[mism]);
            }
        }
    }
    if (!err && !(rf > 0)) err = KA_E_RF_NOT_POSITIVE;          // KTA:65-66
    if (!err && !(rf <= N)) { err = KA_E_RF_GT_BROKERS; erra = rf; }  // KTA:67-69

    const int32_t h = p.topic_hash[t];
    const bool hmin = (h == (int32_t)0x80000000);
    const uint32_t habs = hmin ? 0x80000000u : (uint32_t)(h < 0 ? -h : h);

    if (!err) {
        // ---- KAS:65-71 capacity: (int)ceil((double)(P*rf) / N) == integer ceil-div for int32 operands
        const int64_t tot = (int64_t)(int32_t)((uint32_t)P * (uint32_t)rf);
        const int cap = tot > 0 ? (int)((tot + N - 1) / N) : 0;

        // ---- KAS:73-99 node table: loads start empty -------------------------------------------
        {
            uint32_t* lw = reinterpret_cast<uint32_t*>(load);
            const int words = (N * (int)sizeof(LoadT) + 3) >> 2;
            for (int i = lane; i < words; i += 32) lw[i] = 0u;
            uint32_t* cw = reinterpret_cast<uint32_t*>(cnt);
            for (int i = lane; i < ((P + 3) >> 2); i += 32) cw[i] = 0u;
        }

        // ---- stage the topic's current assignment as 16-bit broker indices ----------------------
        if (!p.rep_off) {
            const int RF = p.RF;
            const int32_t* src = p.cur + g0 * RF;
            const int n = P * RF;
            if (RF == S) {
                // coalesced, 128-bit vectorised when the slab is 16B aligned
                const bool al = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((n & 3) == 0);
                if (al) {
                    const int4* s4 = reinterpret_cast<const int4*>(src);
                    for (int e = lane; e < (n >> 2); e += 32) {
                        int4 v = ka_ldg_stream_v4(s4 + e);
                        uint32_t a = ka_lookup(v.x, tab, p), b = ka_lookup(v.y, tab, p);
                        uint32_t c = ka_lookup(v.z, tab, p), d = ka_lookup(v.w, tab, p);
                        uint2 pk = make_uint2(a | (b << 16), c | (d << 16));
                        *reinterpret_cast<uint2*>(slab + 4 * e) = pk;
                    }
                } else {
                    for (int e = lane; e < n; e += 32) slab[e] = (uint16_t)ka_lookup(__ldg(src + e), tab, p);
                }
            } else {
                for (int e = lane; e < n; e += 32) {
                    int pp = e / RF, r = e - pp * RF;
                    slab[pp * S + r] = (uint16_t)ka_lookup(__ldg(src + e), tab, p);
                }
                for (int e = lane; e < P * (S - RF); e += 32) {
                    int pp = e / (S - RF), r = RF + (e - pp * (S - RF));
                    slab[pp * S + r] = (uint16_t)KA_DEAD;
                }
            }
        } else {
            const int64_t* ro = p.rep_off + g0;
            for (int pp = lane; pp < P; pp += 32) {
                int64_t off = ro[pp];
                int sz = (int)(ro[pp + 1] - off);
                for (int r = 0; r < S; ++r)
                    slab[pp * S + r] = r < sz ? (uint16_t)ka_lookup(__ldg(p.cur + off + r), tab, p) : (uint16_t)KA_DEAD;
            }
        }
        __syncwarp();

        // ---- KAS:101-131 sticky fill: visit order (slot r, partition ascending) ------------------
        for (int r = 0; r < maxlen; ++r) {
            for (int c0 = 0; c0 < P; c0 += 32) {
                const int pp = c0 + lane;
                const bool valid = pp < P;
                uint32_t idx = valid ? (uint32_t)slab[pp * S + r] : KA_DEAD;
                const int k = valid ? (int)cnt[pp] : 0;
                bool feas = idx != KA_DEAD;
                if (feas) {
                    const uint32_t rk = tab.rack[idx];
                    for (int i = 0; i < k; ++i)  // rack exclusivity (also covers "node already has p")
                        if (tab.rack[slab[pp * S + i]] == rk) feas = false;
                }
                const uint32_t fm = __ballot_sync(KA_FULL, feas);
                int rank = 0, gsz = 0, l = 0;
                if (feas) {
                    // rank among this pass's candidates of the same broker, ascending partition
                    const uint32_t m = __match_any_sync(fm, idx);
                    rank = __popc(m & lt);
                    gsz = __popc(m);
                    l = (int)load[idx];
                }
                __syncwarp();  // every candidate has read the broker's load before anyone updates it
                if (feas) {
                    if (l + rank < cap) {
                        slab[pp * S + k] = (uint16_t)idx;  // in-place compaction: k <= r
                        cnt[pp] = (uint8_t)(k + 1);
                    }
                    if (rank == 0) load[idx] = (LoadT)(l + min(gsz, max(cap - l, 0)));
                }
                __syncwarp();
            }
        }

        // ---- KAS:188-200 rotated processing order ------------------------------------------------
        uint32_t start = 0;
        if (!hmin) {
            start = habs % (uint32_t)N;
        } else {
            uint32_t rmd = 0x80000000u % (uint32_t)N;  // Math.abs(MIN_VALUE) % N == -(2^31 % N)
            if (rmd != 0) { err = KA_E_HASH_INDEX; erra = -(int)rmd; errb = N; }
        }
        const int i0 = (int)(((uint32_t)N - start) % (uint32_t)N);  // sorted index at order position 0

        // ---- KAS:133-186 orphans, ascending partition; first-fit from position 0 each time -------
        if (p.rackptr) {
            // Exact reformulation of the walk: a position is acceptable iff its node is not full and its rack does
            // not hold the partition yet, and loads / used racks only grow — so "first acceptable position from
            // j = 0" == min over the racks not yet used of that rack's first non-full member (in rotated order).
            // Each rack keeps a monotone pointer into its member list; placing a replica is one warp min-reduction.
            const int R = p.R;
            for (int r = lane; r < R; r += 32) {
                const int o = tab.roff[r], sz = (int)tab.roff[r + 1] - o;
                int lo = 0, hi = sz;
                while (lo < hi) {  // first member with sorted index >= i0 starts the rack's rotated order
                    const int mid = (lo + hi) >> 1;
                    if ((int)tab.memb[o + mid] < i0) lo = mid + 1; else hi = mid;
                }
                const int st = (lo == sz) ? 0 : lo;
                int kk = 0, pos = 0xFFFF;
                while (kk < sz) {
                    const int m = tab.memb[o + (st + kk >= sz ? st + kk - sz : st + kk)];
                    if ((int)load[m] < cap) { pos = m - i0; if (pos < 0) pos += N; break; }
                    ++kk;
                }
                rst[r] = (uint16_t)st; rkk[r] = (uint16_t)kk; rpos[r] = (uint16_t)pos;
            }
            __syncwarp();
            for (int c0 = 0; c0 < P && !err; c0 += 32) {
                const int pp0 = c0 + lane;
                const int need = pp0 < P ? rf - (int)cnt[pp0] : 0;
                uint32_t ob = __ballot_sync(KA_FULL, need > 0);
                while (ob && !err) {
                    const int src = __ffs(ob) - 1;
                    ob &= ob - 1;
                    const int pp = c0 + src;
                    int rem = __shfl_sync(KA_FULL, need, src);
                    int k = (int)cnt[pp];
                    uint32_t ur[SM];  // racks already holding this partition (warp-uniform)
#pragma unroll
                    for (int i = 0; i < SM; ++i) ur[i] = i < k ? (uint32_t)tab.rack[slab[pp * S + i]] : 0xFFFFFFFFu;
                    while (rem > 0) {
                        uint32_t best = 0xFFFFFFFFu;
                        for (int r = lane; r < R; r += 32) {
                            bool used = false;
#pragma unroll
                            for (int i = 0; i < SM; ++i) used = used || (ur[i] == (uint32_t)r);
                            const uint32_t cnd = used ? 0xFFFFFFFFu : (((uint32_t)rpos[r] << 16) | (uint32_t)r);
                            best = min(best, cnd);
                        }
                        best = __reduce_min_sync(KA_FULL, best);
                        if ((best >> 16) == 0xFFFFu) break;  // no rack can take it: stranded (KAS:183-184)
                        const int pos = (int)(best >> 16), r = (int)(best & 0xFFFFu);
                        int idx = i0 + pos;
                        if (idx >= N) idx -= N;
                        const int nl = (int)load[idx] + 1;
                        __syncwarp();
                        if (lane == 0) {
                            load[idx] = (LoadT)nl;
                            slab[pp * S + k] = (uint16_t)idx;
                        }
#pragma unroll
                        for (int i = 0; i < SM; ++i)
                            if (i == k) ur[i] = (uint32_t)r;
                        ++k;
                        --rem;
                        if (nl >= cap) {  // the rack's first-free member just filled up: advance its pointer
                            const int o = tab.roff[r], sz = (int)tab.roff[r + 1] - o, st = rst[r];
                            int kk = (int)rkk[r] + 1, np = 0xFFFF;
                            while (kk < sz) {
                                const int m = tab.memb[o + (st + kk >= sz ? st + kk - sz : st + kk)];
                                if ((int)load[m] < cap) { np = m - i0; if (np < 0) np += N; break; }
                                ++kk;
                            }
                            if (lane == 0) { rkk[r] = (uint16_t)kk; rpos[r] = (uint16_t)np; }
                        }
                        __syncwarp();
                    }
                    if (lane == 0) cnt[pp] = (uint8_t)k;
                    __syncwarp();
                    if (rem > 0 && !err) { err = KA_E_UNASSIGNABLE; errp = pp; }  // KAS:183-184
                }
            }
        } else {
        int head = 0;  // all order positions < head hold full nodes (loads never decrease)
        for (int c0 = 0; c0 < P && !err; c0 += 32) {
            const int pp0 = c0 + lane;
            const int need = pp0 < P ? rf - (int)cnt[pp0] : 0;
            uint32_t ob = __ballot_sync(KA_FULL, need > 0);
            while (ob && !err) {
                const int src = __ffs(ob) - 1;
                ob &= ob - 1;
                const int pp = c0 + src;
                int rem = __shfl_sync(KA_FULL, need, src);
                int k = (int)cnt[pp];
                uint32_t ur[SM];  // racks already holding this partition (warp-uniform)
#pragma unroll
                for (int i = 0; i < SM; ++i) ur[i] = i < k ? (uint32_t)tab.rack[slab[pp * S + i]] : 0xFFFFFFFFu;
                bool adv = true;
                for (int j = head; j < N && rem > 0; j += 32) {
                    const int pos = j + lane;
                    int idx = i0 + pos;
                    if (idx >= N) idx -= N;
                    bool nonfull = false;
                    uint32_t rk = 0xFFFFFFFEu;
                    if (pos < N) {
                        nonfull = (int)load[idx] < cap;
                        rk = tab.rack[idx];
                    }
                    if (adv) {
                        const uint32_t nb = __ballot_sync(KA_FULL, nonfull);
                        if (nb == 0) head = min(j + 32, N);
                        else { head = j + __ffs(nb) - 1; adv = false; }
                    }
                    bool feas = nonfull;
#pragma unroll
                    for (int i = 0; i < SM; ++i) feas = feas && (ur[i] != rk);
                    uint32_t fb = __ballot_sync(KA_FULL, feas);
                    while (fb && rem > 0) {
                        const int f = __ffs(fb) - 1;
                        const int cidx = __shfl_sync(KA_FULL, idx, f);
                        const uint32_t crk = __shfl_sync(KA_FULL, rk, f);
                        if (lane == f) {
                            load[idx] = (LoadT)((int)load[idx] + 1);
                            slab[pp * S + k] = (uint16_t)cidx;
                        }
#pragma unroll
                        for (int i = 0; i < SM; ++i)
                            if (i == k) ur[i] = crk;
                        ++k;
                        --rem;
                        fb &= ~((2u << f) - 1u);                          // only later positions
                        fb &= ~__ballot_sync(KA_FULL, rk == crk);        // that rack is now taken
                    }
                    __syncwarp();
                }
                if (lane == 0) cnt[pp] = (uint8_t)k;
                __syncwarp();
                if (rem > 0 && !err) { err = KA_E_UNASSIGNABLE; errp = pp; }  // KAS:183-184
            }
        }

        }

        // ---- per-partition finalisation: ascending broker order (KAS:205-214) --------------------
        if (!err) {
            int firstbad = 0x7FFFFFFF, badk = 0;
            for (int pp = lane; pp < P; pp += 32) {
                const int k = (int)cnt[pp];
                uint16_t* row = slab + pp * S;
                for (int i = 1; i < k; ++i) {  // insertion sort, k <= 8
                    uint16_t v = row[i];
                    int j = i - 1;
                    while (j >= 0 && row[j] > v) { row[j + 1] = row[j]; --j; }
                    row[j + 1] = v;
                }
                if (hmin && k >= 3 && pp < firstbad) { firstbad = pp; badk = k; }
            }
            if (hmin) {  // KAS:267 with Math.abs(MIN_VALUE): first remaining-set size that does not divide 2^31
                int fb2 = firstbad;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) fb2 = min(fb2, __shfl_xor_sync(KA_FULL, fb2, o));
                if (fb2 != 0x7FFFFFFF) {
                    const uint32_t bm = __ballot_sync(KA_FULL, firstbad == fb2);
                    const int kk = __shfl_sync(KA_FULL, badk, __ffs(bm) - 1);
                    const int kfail = (kk & (kk - 1)) ? kk : kk - 1;
                    err = KA_E_HASH_INDEX;
                    errp = -1;
                    erra = -(int)(0x80000000u % (uint32_t)kfail);
                    errb = kfail;
                }
            }
            __syncwarp();
        }
    }

    // ---- conflict levels (no reference counterpart) ------------------------------------------------------
    // The leader-ordering chain (KAS:217-237) reads and bumps Context.counter[broker][slot] partition after partition;
    // two partitions commute iff they share no broker. Level of a partition = 1 + the highest level among the earlier
    // partitions OF THIS TOPIC that share a broker with it; partitions of one level are mutually independent, so the
    // order kernel may process a level in parallel and only needs a barrier between levels. Topics are chained one
    // after the other (level numbering restarts per topic). With capacity 1 every broker holds at most one partition
    // of the topic, i.e. the whole topic is one level and this pass is compiled out (LEVELS == false).
    const bool live = !err;
    int D = P > 0 ? 1 : 0;
    if (LEVELS && live && P > 0) {
        for (int i = lane; i < N; i += 32) { ls.owner[i] = 0u; ls.last[i] = 0; }
        __syncwarp();
        int dmax = 0;
        for (int c0 = 0; c0 < P; c0 += 32) {
            const int pp = c0 + lane;
            const bool valid = pp < P;
            const int k = valid ? (int)cnt[pp] : 0;
            const uint16_t* row = slab + (size_t)(valid ? pp : 0) * S;
            for (int i = 0; i < k; ++i) atomicOr(&ls.owner[row[i]], 1u << lane);
            __syncwarp();
            uint32_t preds = 0u;
            for (int i = 0; i < k; ++i) preds |= ls.owner[row[i]];
            preds &= lt;  // earlier partitions of this window sharing a broker with mine
            bool mine = valid && k > 0;
            uint32_t done = ~__ballot_sync(KA_FULL, mine);
            int lv = valid ? 1 : 0;
            while (done != KA_FULL) {  // the lowest pending lane is always ready: terminates
                const bool ready = mine && ((preds & ~done) == 0u);
                if (ready) {
                    int m = 0;
                    for (int i = 0; i < k; ++i) m = max(m, (int)ls.last[row[i]]);
                    lv = m + 1;
                    for (int i = 0; i < k; ++i) ls.last[row[i]] = (uint16_t)lv;  // ready lanes hold disjoint brokers
                    mine = false;
                }
                __syncwarp();
                done |= __ballot_sync(KA_FULL, ready);
            }
            for (int i = 0; i < k; ++i) ls.owner[row[i]] = 0u;
            if (valid) ls.lvl[pp] = (uint16_t)lv;
            dmax = max(dmax, lv);
            __syncwarp();
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dmax = max(dmax, __shfl_xor_sync(KA_FULL, dmax, o));
        D = dmax;
        // stable counting sort by level: sizes -> cumulative ends (exported) -> per-level cursors
        for (int l = lane; l <= D + 1; l += 32) ls.lcur[l] = 0;
        __syncwarp();
        for (int c0 = 0; c0 < P; c0 += 32) {
            const int pp = c0 + lane;
            const bool valid = pp < P;
            const uint32_t vm = __ballot_sync(KA_FULL, valid);
            if (valid) {
                const int lv = ls.lvl[pp];
                const uint32_t m = __match_any_sync(vm, lv);
                if ((m & lt) == 0u) ls.lcur[lv] = (uint16_t)(ls.lcur[lv] + __popc(m));
            }
            __syncwarp();
        }
        int run = 0, crun = 0;
        const int W = p.chunk_w;
        for (int l0 = 1; l0 <= D; l0 += 32) {
            const int l = l0 + lane;
            const int v = l <= D ? (int)ls.lcur[l] : 0;
            const int nc = (v + W - 1) / W;  // a level wider than the order kernel's CTA is cut into chunks
            int x = v, y = nc;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int xo = __shfl_up_sync(KA_FULL, x, o), yo = __shfl_up_sync(KA_FULL, y, o);
                if (lane >= o) { x += xo; y += yo; }
            }
            if (l <= D) {
                const int lstart = run + x - v, cstart = crun + y - nc;
                for (int i = 0; i < nc; ++i) p.lend[g0 + cstart + i] = (uint32_t)(lstart + min((i + 1) * W, v));
                ls.lcur[l] = (uint16_t)lstart;  // first schedule position of level l
            }
            run += __shfl_sync(KA_FULL, x, 31);
            crun += __shfl_sync(KA_FULL, y, 31);
        }
        D = crun;
        __syncwarp();
    } else if (LEVELS && P > 0) {
        const int W = p.chunk_w;  // failed topic: one level of empty records
        D = (P + W - 1) / W;
        for (int i = lane; i < D; i += 32) p.lend[g0 + i] = (uint32_t)min((i + 1) * W, P);
    }
    if (LEVELS && lane == 0) p.ntl[t] = D;

    // ---- emit the partition records in schedule order ----------------------------------------------------
    const uint32_t rot = (err || hmin) ? 0u : ka_rot_bits(habs);
    for (int c0 = 0; c0 < P; c0 += 32) {
        const int pp = c0 + lane;
        const bool valid = pp < P;
        int pos = pp;
        bool first = pp == 0;   // first record of its conflict level (capacity 1 / failed topic: the topic is one level)
        if (LEVELS && live) {
            const uint32_t vm = __ballot_sync(KA_FULL, valid);
            if (valid) {
                const int lv = ls.lvl[pp];
                const uint32_t m = __match_any_sync(vm, lv);
                const uint32_t cur = ls.lcur[lv];   // cursor of the level; bit 15 = the level has been opened (P < 32768)
                pos = (int)(cur & 0x7FFFu) + __popc(m & lt);
                first = (m & lt) == 0u && !(cur & 0x8000u);
                __syncwarp(vm);
                if ((m & lt) == 0u) ls.lcur[lv] = (uint16_t)(((cur & 0x7FFFu) + __popc(m)) | 0x8000u);
            }
            __syncwarp();
        }
        if (valid) {
            const int k = live ? (int)cnt[pp] : 0;
            const uint16_t* row = slab + (size_t)pp * S;
            uint32_t ix[SM];
#pragma unroll
            for (int i = 0; i < SM; ++i) ix[i] = (i < S && i < k) ? (uint32_t)row[i] : 0u;
            if (p.rec_kind == 3) {
                // Brokers are stored in the order getNodeProcessingOrder (KAS:188-200, called at KAS:267 with the k remaining
                // brokers) scans them for slot 0: ascending list position i sits at scan position (i + |hash| % k) % k.
                const int s2 = (int)((rot >> 4) & 1u), s3 = (int)((rot >> 5) & 3u);
                const uint32_t dummy = (uint32_t)N << 2;  // broker N: "infinite" counters, pads rows shorter than 3
                uint32_t a0 = dummy, a1 = dummy, a2 = dummy, f = (uint32_t)k | (first ? 0x80u : 0u);
                if (k == 1) {
                    a0 = ix[0] << 2;
                } else if (k == 2) {
                    a0 = (s2 ? ix[1] : ix[0]) << 2;   // s2 == 1: the higher id is scanned first
                    a1 = (s2 ? ix[0] : ix[1]) << 2;
                } else if (k >= 3) {
                    const int i0 = (3 - s3) % 3, i1 = (4 - s3) % 3, i2 = (5 - s3) % 3;  // list position at scan position 0, 1, 2
                    auto pick = [&](int i) { return i == 0 ? ix[0] : (i == 1 ? ix[1] : ix[2]); };   // no dynamic indexing (stays in registers)
                    a0 = pick(i0) << 2; a1 = pick(i1) << 2; a2 = pick(i2) << 2;
                    // slot 1 scans the remaining pair in ascending id order rotated by s2; for scan positions p < q:
                    // q wins iff c_q < c_p + e_pq, e_pq = s2 when p has the lower id, 1 - s2 otherwise
                    const uint32_t e01 = (uint32_t)(i0 < i1 ? s2 : 1 - s2), e02 = (uint32_t)(i0 < i2 ? s2 : 1 - s2),
                                   e12 = (uint32_t)(i1 < i2 ? s2 : 1 - s2);
                    f |= (e01 << 2) | (e02 << 3) | (e12 << 4);
                }
                reinterpret_cast<uint4*>(p.rec)[g0 + pos] = make_uint4(a0, a1, a2, f);
                if (LEVELS) p.perm[g0 + pos] = (uint16_t)pp;
            } else {
                uint4* r8 = reinterpret_cast<uint4*>(p.rec) + 2 * (g0 + pos);
                r8[0] = make_uint4(ix[0] | (ix[1 % SM] << 16), ix[2 % SM] | (ix[3 % SM] << 16), ix[4 % SM] | (ix[5 % SM] << 16),
                                   ix[6 % SM] | (ix[7 % SM] << 16));   // SM == 8 on this path (S > 3)
                r8[1] = make_uint4((uint32_t)k | rot, (uint32_t)(g0 + pp), 0u, 0u);
            }
        }
    }
    if (err && lane == 0) {
        p.tstatus[p.topic_base + t] = make_int4(err, errp, erra, errb);
        atomicMin(p.err_topic, (unsigned)(p.topic_base + t));
    }
    __syncwarp();
}

template <typename LoadT, bool LEVELS, int SM>
__global__ void __launch_bounds__(512) ka_sticky_spread_kernel(const KaSolveParams p, int load_bytes, int slab_bytes, int cnt_bytes,
                                                               int lv_owner_bytes, int lv_last_bytes, int lv_p_bytes) {
    extern __shared__ __align__(16) unsigned char ka_smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(ka_smem);
    unsigned char* blob = ka_smem + 16;
    unsigned char* warp_base = blob + p.blob_bytes;

    // TMA bulk-stage the broker table (rack indices + id->index LUT) once per CTA.
    if (threadIdx.x == 0) {
        ka_mbar_init(bar, 1);
        ka_fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0 && p.blob_bytes > 0) {
        ka_mbar_expect_tx(bar, (uint32_t)p.blob_bytes);
        ka_tma_bulk_g2s(blob, p.blob, (uint32_t)p.blob_bytes, bar);
    }
    if (p.blob_bytes > 0) ka_mbar_wait(bar, 0);

    KaTab tab;
    tab.rack = reinterpret_cast<const uint16_t*>(blob);
    tab.lut = reinterpret_cast<const uint16_t*>(blob) + p.lut_off;
    tab.roff = reinterpret_cast<const uint16_t*>(blob) + p.roff_off;
    tab.memb = reinterpret_cast<const uint16_t*>(blob) + p.memb_off;

    const int warp = threadIdx.x >> 5;
    const int nwarp = blockDim.x >> 5;
    const int lv_bytes = LEVELS ? lv_owner_bytes + lv_last_bytes + 2 * lv_p_bytes : 0;
    const int per_warp = load_bytes + slab_bytes + cnt_bytes + 3 * p.rp_bytes + lv_bytes;
    unsigned char* mine = warp_base + (size_t)warp * per_warp;
    LoadT* load = reinterpret_cast<LoadT*>(mine);
    uint16_t* slab = reinterpret_cast<uint16_t*>(mine + load_bytes);
    uint8_t* cnt = reinterpret_cast<uint8_t*>(mine + load_bytes + slab_bytes);
    uint16_t* rpos = reinterpret_cast<uint16_t*>(mine + load_bytes + slab_bytes + cnt_bytes);
    uint16_t* rst = reinterpret_cast<uint16_t*>(mine + load_bytes + slab_bytes + cnt_bytes + p.rp_bytes);
    uint16_t* rkk = reinterpret_cast<uint16_t*>(mine + load_bytes + slab_bytes + cnt_bytes + 2 * p.rp_bytes);
    KaLevelScratch ls{};
    if (LEVELS) {
        unsigned char* lvb = mine + load_bytes + slab_bytes + cnt_bytes + 3 * p.rp_bytes;
        ls.owner = reinterpret_cast<uint32_t*>(lvb);
        ls.last = reinterpret_cast<uint16_t*>(lvb + lv_owner_bytes);
        ls.lvl = reinterpret_cast<uint16_t*>(lvb + lv_owner_bytes + lv_last_bytes);
        ls.lcur = reinterpret_cast<uint16_t*>(lvb + lv_owner_bytes + lv_last_bytes + lv_p_bytes);
    }

    const int total_warps = gridDim.x * nwarp;
    for (int t = blockIdx.x * nwarp + warp; t < p.T; t += total_warps)
        ka_solve_topic<LoadT, LEVELS, SM>(p, tab, t, load, slab, cnt, rpos, rst, rkk, ls);
}
