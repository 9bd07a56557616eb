// kassign_plan.cuh — the movement plan of a finished solve: what applying the new assignment moves, compared with the
// current one. No reference counterpart (the reference prints the new lists only); see DESIGN.md "Movement plan".
//
//   ka_row_diff              the ONE definition of a row's change class (UNCHANGED / REORDERED / MOVED), replicas added and
//                            dropped, and leader change; every kernel below calls it
//   ka_plan_kernel           per-row class, totals, and per-broker replica / leader columns keyed by a report-id table
//   ka_changed_*_kernel      stable compaction of the changed rows of one chain sub-block (ballot / popc per warp, block
//                            counts, one scan, scatter) for the changed-rows-only JSON text (kassign_json.cuh, IDX = true)
#pragma once
#include "kassign_common.cuh"

enum { KA_ROW_UNCHANGED = 0, KA_ROW_REORDERED = 1, KA_ROW_MOVED = 2 };

#define KA_PLAN_COLS 8     // replicas before/after/in/out, leaders before/after/in/out (include/kassign.h)
#define KA_PLAN_TOTALS 6   // rows, reordered, moved, replicas added, replicas dropped, leaders changed

// The rows of a finished solve, addressed by their row index g in the whole run.
struct KaRows {
    const int32_t* cur;       // current lists: dense cur[g * RF ..] (rep_off == nullptr) or ragged cur[rep_off[g] .. rep_off[g + 1])
    const int64_t* rep_off;
    int RF;
    const int32_t* out;       // [Q][S] new lists, leader first
    const int32_t* out_len;   // [Q], or nullptr: every new list is rf_t long
    int S, rf_t;
};

// Current list C and new list O of row g in registers (SM = compile-time bound on both lengths: 3 or 8).
template <int SM>
__device__ __forceinline__ void ka_load_row(const KaRows& r, int64_t g, int32_t (&C)[SM], int& lc, int32_t (&O)[SM], int& lo) {
    const int32_t* cp;
    if (r.rep_off) {
        const int64_t a = r.rep_off[g];
        lc = (int)(r.rep_off[g + 1] - a);
        cp = r.cur + a;
    } else {
        lc = r.RF;
        cp = r.cur + g * r.RF;
    }
    lo = r.out_len ? r.out_len[g] : r.rf_t;
    lc = min(max(lc, 0), SM);
    lo = min(max(lo, 0), SM);
    const int32_t* op = r.out + g * r.S;
#pragma unroll
    for (int i = 0; i < SM; ++i) {
        C[i] = i < lc ? __ldg(cp + i) : 0;
        O[i] = i < lo ? __ldg(op + i) : 0;
    }
}

struct KaRowDiff {
    uint32_t c_first;   // bit i: C[i] is the first occurrence of its broker in C (a current list may repeat a broker)
    uint32_t c_in_o;    // bit i: C[i] is in O
    uint32_t o_in_c;    // bit i: O[i] is in C
    int cls;            // KA_ROW_*
    int added, dropped; // |O \ C|, |C \ O| (as sets)
    bool lead;          // O[0] != C[0]; an empty C with a non-empty O counts as a change
};

// UNCHANGED: O == C as sequences. REORDERED: same broker set and length, different order. MOVED: the sets or lengths differ.
template <int SM>
__device__ __forceinline__ KaRowDiff ka_row_diff(const int32_t (&C)[SM], int lc, const int32_t (&O)[SM], int lo) {
    KaRowDiff d;
    d.c_first = d.c_in_o = d.o_in_c = 0u;
    bool same = lc == lo;
#pragma unroll
    for (int i = 0; i < SM; ++i) {
        const bool ci = i < lc, oi = i < lo;
        if (ci && oi && C[i] != O[i]) same = false;
        bool first = ci, cin = false, oin = false;
#pragma unroll
        for (int j = 0; j < SM; ++j) {
            if (j < i && C[j] == C[i]) first = false;
            if (j < lo && O[j] == C[i]) cin = true;
            if (j < lc && C[j] == O[i]) oin = true;
        }
        if (first) d.c_first |= 1u << i;
        if (ci && cin) d.c_in_o |= 1u << i;
        if (oi && oin) d.o_in_c |= 1u << i;
    }
    d.added = __popc(((1u << lo) - 1u) & ~d.o_in_c);
    d.dropped = __popc(d.c_first & ~d.c_in_o);
    d.cls = same ? KA_ROW_UNCHANGED : ((d.added | d.dropped) != 0 || lc != lo ? KA_ROW_MOVED : KA_ROW_REORDERED);
    d.lead = lo > 0 && (lc == 0 || O[0] != C[0]);
    return d;
}

struct KaPlanParams {
    KaRows rows;
    int64_t Q;
    // report-id table (ka_id_index): bucket of a broker id = its index in broker_id[0 .. N), or N ("other") when absent
    int lut_mode, min_id;
    uint32_t range;
    const uint16_t* glut;     // [range] LUT (KA_LUT_SMEM: staged into shared memory; KA_LUT_GLOBAL: read from L2)
    const int32_t* broker_id; // [N] the report ids, ascending
    int N;                    // report ids (M of ka_plan_last)
    int lut_bytes;            // bytes of the shared-memory copy of glut (KA_LUT_SMEM), a multiple of 16
    uint8_t* row_class;       // [Q] or nullptr
    uint32_t* stats;          // [(M + 1) * KA_PLAN_COLS]
    unsigned long long* totals;  // [KA_PLAN_TOTALS]
};

__device__ __forceinline__ uint32_t ka_plan_bucket(const KaPlanParams& p, const uint16_t* slut, int id) {
    const uint32_t b = ka_id_index(id, slut, p);
    return b == KA_DEAD ? (uint32_t)p.N : b;
}

// One pass over the rows, grid-stride. SHIST: the per-broker columns are privatised in shared memory and added to `stats`
// at the end (the host chooses it when (M + 1) x 8 counters fit); otherwise every update is a global atomic (L2-resident).
template <int SM, bool SHIST>
__global__ void __launch_bounds__(512) ka_plan_kernel(const KaPlanParams p) {
    extern __shared__ __align__(16) unsigned char ka_psmem[];
    __shared__ unsigned long long tsum[KA_PLAN_TOTALS];
    uint16_t* slut = reinterpret_cast<uint16_t*>(ka_psmem);
    uint32_t* col = SHIST ? reinterpret_cast<uint32_t*>(ka_psmem + p.lut_bytes) : p.stats;
    const int ncol = (p.N + 1) * KA_PLAN_COLS;
    {
        const uint4* src = reinterpret_cast<const uint4*>(p.glut);
        uint4* dst = reinterpret_cast<uint4*>(slut);
        for (int i = threadIdx.x; i < (p.lut_bytes >> 4); i += blockDim.x) dst[i] = __ldg(src + i);
    }
    if (SHIST)
        for (int i = threadIdx.x; i < ncol; i += blockDim.x) col[i] = 0u;
    if (threadIdx.x < KA_PLAN_TOTALS) tsum[threadIdx.x] = 0ull;
    __syncthreads();

    uint32_t n_rows = 0, n_re = 0, n_mv = 0, n_add = 0, n_drop = 0, n_lead = 0;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < p.Q; g += (int64_t)gridDim.x * blockDim.x) {
        int32_t C[SM], O[SM];
        int lc, lo;
        ka_load_row<SM>(p.rows, g, C, lc, O, lo);
        const KaRowDiff d = ka_row_diff<SM>(C, lc, O, lo);
        if (p.row_class) p.row_class[g] = (uint8_t)d.cls;
        n_rows++;
        n_re += d.cls == KA_ROW_REORDERED;
        n_mv += d.cls == KA_ROW_MOVED;
        n_add += d.added;
        n_drop += d.dropped;
        n_lead += d.lead;
#pragma unroll
        for (int i = 0; i < SM; ++i) {
            if ((d.c_first >> i) & 1u) {
                const uint32_t b = ka_plan_bucket(p, slut, C[i]) * KA_PLAN_COLS;
                atomicAdd(&col[b + 0], 1u);                                   // replicas_before
                if (!((d.c_in_o >> i) & 1u)) atomicAdd(&col[b + 3], 1u);      // replicas_out
                if (i == 0) {
                    atomicAdd(&col[b + 4], 1u);                               // leaders_before
                    if (d.lead) atomicAdd(&col[b + 7], 1u);                   // leaders_out
                }
            }
            if (i < lo) {
                const uint32_t b = ka_plan_bucket(p, slut, O[i]) * KA_PLAN_COLS;
                atomicAdd(&col[b + 1], 1u);                                   // replicas_after
                if (!((d.o_in_c >> i) & 1u)) atomicAdd(&col[b + 2], 1u);      // replicas_in
                if (i == 0) {
                    atomicAdd(&col[b + 5], 1u);                               // leaders_after
                    if (d.lead) atomicAdd(&col[b + 6], 1u);                   // leaders_in
                }
            }
        }
    }
    const uint32_t v[KA_PLAN_TOTALS] = {n_rows, n_re, n_mv, n_add, n_drop, n_lead};
#pragma unroll
    for (int k = 0; k < KA_PLAN_TOTALS; ++k) {
        const uint32_t w = __reduce_add_sync(KA_FULL, v[k]);
        if ((threadIdx.x & 31) == 0 && w) atomicAdd(&tsum[k], (unsigned long long)w);
    }
    __syncthreads();
    if (threadIdx.x < KA_PLAN_TOTALS && tsum[threadIdx.x]) atomicAdd(&p.totals[threadIdx.x], tsum[threadIdx.x]);
    if (SHIST)
        for (int i = threadIdx.x; i < ncol; i += blockDim.x)
            if (col[i]) atomicAdd(&p.stats[i], col[i]);
}

// ---- changed-row compaction of one fragment: rows row0 .. row0 + n - 1 of the run -> sel[0 .. count), fragment-relative,
// ascending. Three launches on the JSON stream, no host synchronisation: the count stays on the device.
//
// 1. class of every row (ka_row_diff), ballot per warp -> mask[warp], popc per block -> blockcnt[block]
template <int SM>
__global__ void __launch_bounds__(256) ka_changed_flag_kernel(const KaRows r, int64_t row0, uint32_t n, uint32_t* mask, uint32_t* blockcnt) {
    __shared__ uint32_t wc[8];
    const uint32_t q = blockIdx.x * 256u + threadIdx.x;
    bool changed = false;
    if (q < n) {
        int32_t C[SM], O[SM];
        int lc, lo;
        ka_load_row<SM>(r, row0 + q, C, lc, O, lo);
        changed = ka_row_diff<SM>(C, lc, O, lo).cls != KA_ROW_UNCHANGED;
    }
    const uint32_t m = __ballot_sync(KA_FULL, changed);
    if ((threadIdx.x & 31) == 0) {
        mask[q >> 5] = m;
        wc[threadIdx.x >> 5] = __popc(m);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (int i = 0; i < 8; ++i) s += wc[i];
        blockcnt[blockIdx.x] = s;
    }
}

// 2. (one CTA) exclusive scan of the block counts in place; state = {rows kept by earlier fragments, running total}:
//    frag = {rows kept before this fragment, rows kept in it}, then the running total advances
__global__ void __launch_bounds__(1024) ka_changed_scan_kernel(uint32_t* blockcnt, int nblocks, uint32_t* kept, uint32_t* frag) {
    __shared__ uint32_t wtot[32];
    __shared__ uint32_t carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0u;
    __syncthreads();
    for (int b0 = 0; b0 < nblocks; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const uint32_t v = b < nblocks ? blockcnt[b] : 0u;
        uint32_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(KA_FULL, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wtot[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = wtot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(KA_FULL, w, o);
                if (lane >= o) w += y;
            }
            wtot[lane] = w;
        }
        __syncthreads();
        const uint32_t base = carry + (warp > 0 ? wtot[warp - 1] : 0u);
        if (b < nblocks) blockcnt[b] = base + x - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = base + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        frag[0] = *kept;
        frag[1] = carry;
        *kept += carry;
    }
}

// 3. every changed row writes its fragment-relative index at its stable position
__global__ void __launch_bounds__(256) ka_changed_scatter_kernel(const uint32_t* mask, const uint32_t* blockoff, uint32_t n, uint32_t* sel) {
    const uint32_t q = blockIdx.x * 256u + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t* bm = mask + blockIdx.x * 8u;
    uint32_t before = blockoff[blockIdx.x];
    for (int i = 0; i < warp; ++i) before += __popc(bm[i]);
    const uint32_t m = bm[warp];
    if (q < n && ((m >> lane) & 1u)) sel[before + __popc(m & ka_lanemask_lt())] = q;
}
