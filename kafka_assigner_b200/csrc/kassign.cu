// kassign.cu — C ABI (include/kassign.h) over the sm_100a kernels in kassign_stage.cuh / kassign_order.cuh / kassign_json.cuh /
// kassign_plan.cuh.
//
// Reference boundary: KafkaTopicAssigner.generateAssignment (KafkaTopicAssigner.java:42-72) batched over
// the topic loop of KafkaAssignmentGenerator.java:172-184. No CPU fallback exists in this library.
#include "kassign_stage.cuh"
#include "kassign_order.cuh"
#include "kassign_json.cuh"
#include "kassign_plan.cuh"

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/kassign.h"

namespace {

constexpr int KA_SM_COUNT_FALLBACK = 148;
constexpr size_t KA_SMEM_BUDGET = 200 * 1024;   // per-CTA dynamic smem we allow ourselves (of 227 KB)
constexpr uint32_t KA_LUT_SMEM_MAX_RANGE = 32768;
constexpr uint32_t KA_LUT_GLOBAL_MAX_RANGE = 1u << 25;
constexpr size_t KA_PLAN_SMEM_BUDGET = 112 * 1024;  // plan kernel: id LUT + private per-broker columns, two CTAs per SM

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr int KA_MAX_CHAIN_BLOCKS = 8;    // slot-chain sub-blocks per staged block
constexpr int KA_MAX_CHAIN_EVENTS = 64;   // per solve: 8 staged blocks x 8 sub-blocks

struct HostPinned {
    int err_topic;
    int spin_flag;
    int4 tstatus;
};

}  // namespace

struct ka_ctx {
    int device = 0;
    int sm_count = KA_SM_COUNT_FALLBACK;
    cudaStream_t stream = nullptr;  // used by the host-buffer entry points
    // broker table
    int N = 0;
    std::vector<int32_t> broker_id;
    std::vector<int32_t> broker_rack;
    int lut_mode = KA_LUT_SMEM;
    int min_id = 0;
    uint32_t range = 0;
    int blob_bytes = 16;
    int lut_off = 0;
    int R = 0, roff_off = 0, memb_off = 0;
    DevBuf d_blob, d_glut, d_broker_id, d_ctr8;
    // counters of brokers not in the current table (Context.counter is keyed by broker id)
    std::unordered_map<int32_t, std::vector<int32_t>> parked;
    // scratch
    DevBuf d_hash, d_part_off, d_rep_off, d_cur, d_out, d_out_len, d_tstatus, d_flags;
    DevBuf d_rec, d_perm, d_ntl, d_loff, d_lend, d_lvl_end;  // records, chosen positions, schedule permutation, level tables
    HostPinned* h_pin = nullptr;
    // bookkeeping
    bool timing = false;
    cudaEvent_t ev[10] = {};
    float last_ms[8] = {};
    bool ev_valid = false;
    cudaEvent_t ev_mark = nullptr;  // where enq_sticky_hist records 'kernel A done' (timing only)
    int64_t launches = 0;
    int topic_base = 0;       // ka_ctx_set_topic_base: index of the staged block's first topic in the whole (multi-GPU) run
    bool last_was_staged = false;
    int order_threads = 0;  // leader-order CTA size override (0 = heuristic from N); env KA_ORDER_THREADS wins
    // second stream + events for the pipelined (super-chunk) solve
    cudaStream_t aux = nullptr;
    cudaStream_t sb1 = nullptr;             // slot-0 chain stream (the slot-1 chain + emit run on the caller's stream)
    cudaEvent_t ev_chain_in = nullptr, ev_b1[KA_MAX_CHAIN_EVENTS] = {}, ev_chain[KA_MAX_CHAIN_EVENTS][4] = {};
    int chain_ev_next = 0, chain_used = 0;
    // device-side JSON emission (ka_solve_dense_json)
    cudaStream_t sj = nullptr;
    cudaEvent_t ev_json_in[KA_MAX_CHAIN_EVENTS] = {}, ev_json_scan[KA_MAX_CHAIN_EVENTS] = {};
    DevBuf d_json, d_names, d_name_off, d_json_rowlen, d_json_blocksum, d_json_state;
    unsigned long long* h_frag = nullptr;  // pinned [KA_MAX_CHAIN_EVENTS][2]: {first byte, bytes} of every fragment
    struct JsonJob* json_job = nullptr;
    // host destination of a pipelined host-buffer solve: every chain sub-block is copied out on c->sj as soon as its emit is
    // done, so that no D2H sits between two slot-1 chains on the caller's stream
    int32_t* host_out = nullptr; int32_t* host_out_len = nullptr; int32_t* dev_out = nullptr; int32_t* dev_out_len = nullptr;
    int out_copies = 0;
    cudaEvent_t ev_out_done = nullptr;    // non-null while run_dense serves ka_solve_dense_json
    bool slot_timed[2] = {false, false};   // ka_order_slot_device recorded ev_chain[slot][0..1]
    cudaEvent_t ev_in = nullptr, ev_stage[8] = {};
    cudaEvent_t ev_pipe[8][5] = {};
    int last_stages = 1;
    // staged problem (between the context-free stage and the leader-order stage)
    bool staged = false;
    struct StagedBlock* staged_block = nullptr;  // StageDesc of ka_stage_dense_device, consumed by ka_order_device
    // async status
    cudaStream_t last_stream = nullptr;
    bool pending_status = false;
    const int32_t* last_part_id = nullptr;  // host pointer (ragged API) for status translation
    const int64_t* last_part_off = nullptr;
    ka_status last{};
    // movement plan (ka_plan_last): rows of the last solve, still resident; report-id table (rep_M == 0: the live table)
    bool plan_valid = false;
    KaRows plan_rows{};
    int64_t plan_Q = 0;
    int rep_M = 0, rep_mode = KA_LUT_SMEM, rep_min_id = 0;
    uint32_t rep_range = 0;
    DevBuf d_rep_lut, d_rep_ids, d_plan_tot, d_plan_stats, d_plan_class;
    DevBuf d_sel, d_sel_mask, d_sel_blockcnt, d_sel_state;  // changed-row compaction of ka_solve_dense_json_changed
};

namespace {

#define KA_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            std::fprintf(stderr, "[kassign] CUDA error %s at %s:%d: %s\n", cudaGetErrorName(_e), __FILE__, __LINE__, \
                         cudaGetErrorString(_e));                                                  \
            return KA_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

int set_status(ka_status* st, int code, int topic = -1, int part = -1, int a = 0, int b = 0) {
    if (st) {
        st->code = code;
        st->topic_index = topic;
        st->partition = part;
        st->a = a;
        st->b = b;
    }
    return code;
}

inline size_t align16(size_t v) { return (v + 15) & ~size_t(15); }

// Id -> index table of n strictly ascending ids (ka_id_index): a 16-bit LUT over the id range, staged into shared memory up
// to KA_LUT_SMEM_MAX_RANGE ids and read from global memory (L2) up to KA_LUT_GLOBAL_MAX_RANGE; beyond that a binary search
// over the ids. Used by the live broker table and by the report-id table of the movement plan.
struct IdLut {
    int mode = KA_LUT_SMEM;
    int min_id = 0;
    uint32_t range = 0;
    std::vector<uint16_t> lut;  // [range rounded up to 16 bytes], KA_DEAD where no id; empty for KA_LUT_BSEARCH
};

IdLut make_id_lut(int n, const int32_t* ids) {
    IdLut t;
    t.min_id = n > 0 ? ids[0] : 0;
    const uint64_t range64 = n > 0 ? (uint64_t)((int64_t)ids[n - 1] - (int64_t)ids[0]) + 1 : 0;
    if (range64 > KA_LUT_GLOBAL_MAX_RANGE) {
        t.mode = KA_LUT_BSEARCH;
        return t;
    }
    t.mode = range64 <= KA_LUT_SMEM_MAX_RANGE ? KA_LUT_SMEM : KA_LUT_GLOBAL;
    t.range = (uint32_t)range64;
    t.lut.assign(align16((size_t)std::max<uint64_t>(range64, 1) * 2) / 2, (uint16_t)KA_DEAD);
    for (int i = 0; i < n; ++i) t.lut[(size_t)((int64_t)ids[i] - t.min_id)] = (uint16_t)i;
    return t;
}

// download current device counters into ctx->parked keyed by id
int park_counters(ka_ctx* c) {
    if (c->N == 0 || !c->d_ctr8.p) return KA_OK;
    std::vector<int32_t> h((size_t)c->N * KA_MAX_SLOTS);
    KA_CUDA(cudaMemcpy(h.data(), c->d_ctr8.p, h.size() * 4, cudaMemcpyDeviceToHost));
    for (int i = 0; i < c->N; ++i) {
        const int32_t* row = h.data() + (size_t)i * KA_MAX_SLOTS;
        bool nz = false;
        for (int r = 0; r < KA_MAX_SLOTS; ++r) nz |= row[r] != 0;
        if (nz) c->parked[c->broker_id[i]] = std::vector<int32_t>(row, row + KA_MAX_SLOTS);
        else c->parked.erase(c->broker_id[i]);
    }
    return KA_OK;
}

struct Plan {
    // kernel A
    int a_warps, a_load_bytes, a_slab_bytes, a_cnt_bytes, a_load_kind;  // kind 0=u8 1=u16 2=u32
    int a_rackptr, a_rp_bytes, a_blob_bytes;
    int a_levels;                                   // 1: some topic may hold a broker twice -> conflict levels + tables
    int lv_owner_bytes, lv_last_bytes, lv_p_bytes;  // per-warp scratch of the level pass
    size_t a_smem;
    // leader order
    int rec_kind, rec_bytes;  // 3: 16 B records (rows <= 3), 4 / 8: 32 B records (rows of 4 / 5..8)
    int b_gctr;               // counters stay in global memory (table too large for shared memory)
    int b_ring_log2;          // log2(records per TMA ring stage)
    int b_threads;
    size_t b_smem;
};

constexpr size_t KA_ORDER_SMEM_BUDGET = 226 * 1024;

int make_plan(ka_ctx* c, int64_t Q, int S, int Pmax, int64_t capmax, bool ragged, Plan& pl, ka_status* st) {
    const int N = c->N;
    if (Q >= (int64_t)1 << 31) return set_status(st, KA_ERR_LIMIT, -1, -1, INT_MAX, 0);
    // ---- kernel A
    pl.a_load_kind = capmax <= 255 ? 0 : (capmax <= 65535 ? 1 : 2);
    const int lsz = pl.a_load_kind == 0 ? 1 : (pl.a_load_kind == 1 ? 2 : 4);
    pl.a_load_bytes = (int)align16((size_t)std::max(N, 1) * lsz);
    pl.a_slab_bytes = (int)align16((size_t)std::max(Pmax, 1) * S * 2);
    pl.a_cnt_bytes = (int)align16((size_t)std::max(Pmax, 1));
    // spread phase: window scan over the rotated order by default (measured faster on every BASELINE config: the
    // monotone head finds a slot within ~1 window); KA_SPREAD_RACKPTR=1 selects the per-rack first-free-pointer
    // variant (exact too; pays off only when walks are long: many full nodes AND tight rack constraints).
    pl.a_rackptr = 0;
    if (const char* e = std::getenv("KA_SPREAD_RACKPTR")) pl.a_rackptr = std::atoi(e) && c->R > 0 && c->R <= 4096;
    pl.a_rp_bytes = pl.a_rackptr ? (int)align16((size_t)c->R * 2) : 0;
    // capacity 1 == every broker holds at most one partition of a topic == the topic is a single conflict level
    pl.a_levels = (capmax > 1 || ragged) ? 1 : 0;
    if (const char* e = std::getenv("KA_FORCE_LEVELS")) pl.a_levels = pl.a_levels || std::atoi(e);
    if (pl.a_levels && Pmax > 32767) return set_status(st, KA_ERR_LIMIT, -1, -1, Pmax, N);  // level cursors are 15-bit
    pl.lv_owner_bytes = pl.a_levels ? (int)align16((size_t)std::max(N, 1) * 4) : 0;
    pl.lv_last_bytes = pl.a_levels ? (int)align16((size_t)std::max(N, 1) * 2) : 0;
    pl.lv_p_bytes = pl.a_levels ? (int)align16((size_t)(std::max(Pmax, 1) + 2) * 2) : 0;
    const size_t per_warp = (size_t)pl.a_load_bytes + pl.a_slab_bytes + pl.a_cnt_bytes + 3 * (size_t)pl.a_rp_bytes +
                            pl.lv_owner_bytes + pl.lv_last_bytes + 2 * (size_t)pl.lv_p_bytes;
    // the rack member lists (last part of the blob) are only read by the opt-in rack-pointer spread: not staged otherwise
    pl.a_blob_bytes = pl.a_rackptr ? c->blob_bytes : c->roff_off * 2;
    const size_t shared = 16 + (size_t)pl.a_blob_bytes;
    if (shared + per_warp > KA_SMEM_BUDGET) return set_status(st, KA_ERR_LIMIT, -1, -1, Pmax, N);
    pl.a_warps = (int)std::min<size_t>(16, (KA_SMEM_BUDGET - shared) / per_warp);
    pl.a_smem = shared + per_warp * pl.a_warps;
    // ---- leader order
    pl.rec_kind = S <= 3 ? 3 : (S == 4 ? 4 : 8);
    pl.rec_bytes = pl.rec_kind == 3 ? 16 : 32;
    const int cw = pl.rec_kind == 8 ? 8 : 4;
    const int max_nt = pl.rec_kind == 3 ? 1024 : (pl.rec_kind == 4 ? 512 : 256);
    // rows <= 3: each slot chain keeps ONE counter column (+ the dummy broker that pads short rows) in shared memory
    const size_t ctr_bytes = pl.rec_kind == 3 ? (size_t)(std::max(N, 1) + 1) * 4 : (size_t)std::max(N, 1) * cw * 4;
    // record ring: KA_RING_STAGES stages of 2^lg records, as large as fits next to the counter table (<= 128 KB)
    const int lg_max = pl.rec_kind == 3 ? 10 : 9, lg_min = 7;
    auto ring_bytes = [&](int l) { return ((size_t)KA_RING_STAGES << l) * pl.rec_bytes + 256; };
    int lg = lg_max;
    pl.b_gctr = 0;
    while (lg > lg_min && ctr_bytes + ring_bytes(lg) > KA_ORDER_SMEM_BUDGET) --lg;
    if (ctr_bytes + ring_bytes(lg) > KA_ORDER_SMEM_BUDGET) {
        pl.b_gctr = 1;  // counter table beyond shared memory: rows stay in global memory (L2)
        lg = lg_max;
    }
    if (const char* e = std::getenv("KA_ORDER_GLOBAL_CTR")) pl.b_gctr = pl.b_gctr || std::atoi(e);
    pl.b_ring_log2 = lg;
    pl.b_smem = ring_bytes(lg) + (pl.b_gctr ? 0 : ctr_bytes);
    // CTA size ~ level width: a level is one pass of the CTA. Capacity 1: level = topic (P wide). Otherwise a level
    // holds each broker at most once, i.e. at most N / S partitions; measured widths are about half of that.
    int64_t width = pl.a_levels ? std::min<int64_t>(Pmax, std::max<int64_t>(1, N / std::max(S, 1) / 2)) : Pmax;
    // a level wider than the CTA is cut into equal chunks (the kernel is issue-bound there: equal halves cost nothing)
    const int64_t cuts = (std::max<int64_t>(width, 1) + max_nt - 1) / max_nt;
    width = (std::max<int64_t>(width, 1) + cuts - 1) / cuts;
    int nt = (int)std::min<int64_t>(max_nt, ((width + 31) / 32) * 32);
    if (c->order_threads > 0) nt = c->order_threads;
    if (const char* e = std::getenv("KA_ORDER_THREADS")) nt = std::atoi(e);
    nt = std::max(32, std::min(max_nt, (nt / 32) * 32));
    nt = std::min(nt, (KA_RING_STAGES - 1) << lg);
    pl.b_threads = nt;
    return KA_OK;
}

template <typename K>
cudaError_t allow_smem(K kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

template <int SM, bool SHIST>
cudaError_t launch_plan(ka_ctx* c, cudaStream_t s, const KaPlanParams& p, size_t smem) {
    auto kern = ka_plan_kernel<SM, SHIST>;
    cudaError_t e = allow_smem(kern, smem);
    if (e != cudaSuccess) return e;
    int occ = 1;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 512, smem)) != cudaSuccess) return e;
    const int64_t grid = std::min<int64_t>((p.Q + 511) / 512, (int64_t)std::max(occ, 1) * c->sm_count);
    kern<<<(unsigned)grid, 512, smem, s>>>(p);
    return cudaGetLastError();
}

// One contiguous block of topics of a dense or ragged problem, with every device pointer already offset to the block.
struct StageDesc {
    int topic_base = 0, T = 0;
    int64_t Q = 0;                  // partitions in the block
    const int32_t* d_hash = nullptr;
    const int64_t* d_part_off = nullptr;  // ragged only (block == whole problem)
    const int64_t* d_rep_off = nullptr;
    int P = 0, RF = 0;
    const int32_t* d_cur = nullptr;
    int desired_rf = -1, S = 1, Pmax = 0;
    int64_t capmax = 0;
    int64_t q0 = 0;                 // first partition row of the block inside the ctx scratch arrays
    int blk = 0;                    // ordinal of the block inside a pipelined solve (its level tables: loff at topic_base + blk)
    Plan pl;
};

}  // namespace
struct StagedBlock { StageDesc d; };
namespace {

int reserve_scratch(ka_ctx* c, int64_t Qtot, int rec_bytes, int Ttot, int blocks, bool levels) {
    const size_t q = (size_t)std::max<int64_t>(Qtot, 1);
    KA_CUDA(c->d_rec.reserve(q * rec_bytes + 256));
    if (levels) {
        KA_CUDA(c->d_perm.reserve(q * 2));
        KA_CUDA(c->d_lend.reserve(q * 4));
        KA_CUDA(c->d_lvl_end.reserve(q * 4));
        KA_CUDA(c->d_ntl.reserve((size_t)std::max(Ttot, 1) * 4));
        KA_CUDA(c->d_loff.reserve((size_t)(std::max(Ttot, 1) + blocks + 1) * 4));
    }
    KA_CUDA(c->d_tstatus.reserve((size_t)std::max(Ttot, 1) * sizeof(int4)));
    KA_CUDA(c->d_flags.reserve(64));
    return KA_OK;
}

// flags: [0] lowest failing topic (unsigned atomicMin, 0xFFFFFFFF = none)
int reset_flags(ka_ctx* c, cudaStream_t s) {
    c->h_pin->err_topic = -1;
    c->h_pin->spin_flag = -1;
    c->chain_ev_next = 0;
    c->chain_used = 0;
    c->slot_timed[0] = c->slot_timed[1] = false;
    KA_CUDA(cudaMemsetAsync(c->d_flags.p, 0xFF, 2 * sizeof(int), s));
    return KA_OK;
}

template <typename LoadT, bool LEVELS, int SM>
cudaError_t launch_stage_t(ka_ctx* c, cudaStream_t s, const KaSolveParams& p, const Plan& pl, int T) {
    auto kern = ka_sticky_spread_kernel<LoadT, LEVELS, SM>;
    const int threads = pl.a_warps * 32;
    cudaError_t e = allow_smem(kern, pl.a_smem);
    if (e != cudaSuccess) return e;
    int occ = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, pl.a_smem);
    if (e != cudaSuccess) return e;
    int grid = (T + pl.a_warps - 1) / pl.a_warps;
    grid = std::min(grid, std::max(1, occ) * c->sm_count);
    kern<<<grid, threads, pl.a_smem, s>>>(p, pl.a_load_bytes, pl.a_slab_bytes, pl.a_cnt_bytes, pl.lv_owner_bytes, pl.lv_last_bytes, pl.lv_p_bytes);
    return cudaGetLastError();
}

template <typename LoadT, bool LEVELS>
cudaError_t launch_stage(ka_ctx* c, cudaStream_t s, const KaSolveParams& p, const Plan& pl, int T) {
    return p.S <= 3 ? launch_stage_t<LoadT, LEVELS, 3>(c, s, p, pl, T) : launch_stage_t<LoadT, LEVELS, 8>(c, s, p, pl, T);
}

// Context-free part of a block (shards across GPUs): kernel A (records in schedule order) + the level tables.
int enq_stage(ka_ctx* c, cudaStream_t s, const StageDesc& d) {
    const int N = c->N, S = d.S;
    const Plan& pl = d.pl;
    if (d.T > 0) {
        KaSolveParams p{};
        p.T = d.T;
        p.topic_base = d.topic_base;
        p.topic_hash = d.d_hash;
        p.part_off = d.d_part_off;
        p.P = d.P;
        p.rep_off = d.d_rep_off;
        p.RF = d.RF;
        p.cur = d.d_cur;
        p.desired_rf = d.desired_rf;
        p.S = S;
        p.Pmax = d.Pmax;
        p.N = N;
        p.blob = c->d_blob.as<uint16_t>();
        p.blob_bytes = pl.a_blob_bytes;
        p.lut_off = c->lut_off;
        p.R = c->R;
        p.rackptr = pl.a_rackptr;
        p.roff_off = c->roff_off;
        p.memb_off = c->memb_off;
        p.rp_bytes = pl.a_rp_bytes;
        p.lut_mode = c->lut_mode;
        p.min_id = c->min_id;
        p.range = c->range;
        p.glut = c->d_glut.as<uint16_t>();
        p.broker_id = c->d_broker_id.as<int32_t>();
        p.rec_kind = pl.rec_kind;
        p.rec = c->d_rec.as<unsigned char>() + (size_t)d.q0 * pl.rec_bytes;
        p.perm = pl.a_levels ? c->d_perm.as<uint16_t>() + d.q0 : nullptr;
        p.chunk_w = pl.b_threads;
        p.ntl = pl.a_levels ? c->d_ntl.as<int32_t>() + d.topic_base : nullptr;
        p.lend = pl.a_levels ? c->d_lend.as<uint32_t>() + d.q0 : nullptr;
        p.tstatus = c->d_tstatus.as<int4>();
        p.err_topic = c->d_flags.as<unsigned>();
        cudaError_t e;
        if (pl.a_levels) {
            if (pl.a_load_kind == 0) e = launch_stage<uint8_t, true>(c, s, p, pl, d.T);
            else if (pl.a_load_kind == 1) e = launch_stage<uint16_t, true>(c, s, p, pl, d.T);
            else e = launch_stage<uint32_t, true>(c, s, p, pl, d.T);
        } else {
            if (pl.a_load_kind == 0) e = launch_stage<uint8_t, false>(c, s, p, pl, d.T);
            else if (pl.a_load_kind == 1) e = launch_stage<uint16_t, false>(c, s, p, pl, d.T);
            else e = launch_stage<uint32_t, false>(c, s, p, pl, d.T);
        }
        KA_CUDA(e);
        c->launches++;
    }
    if (c->timing && c->ev_mark) KA_CUDA(cudaEventRecord(c->ev_mark, s));  // end of kernel A
    if (pl.a_levels && d.T > 0) {
        int32_t* ntl = c->d_ntl.as<int32_t>() + d.topic_base;
        int32_t* loff = c->d_loff.as<int32_t>() + d.topic_base + d.blk;  // every block keeps T_k + 1 entries
        ka_level_scan_kernel<<<1, 1024, 0, s>>>(ntl, d.T, loff);
        KA_CUDA(cudaGetLastError());
        ka_level_fill_kernel<<<(d.T + 7) / 8, 256, 0, s>>>(ntl, loff, c->d_lend.as<uint32_t>() + d.q0, d.d_part_off, d.P, d.T,
                                                            c->d_lvl_end.as<uint32_t>() + d.q0);
        KA_CUDA(cudaGetLastError());
        c->launches += 2;
    }
    return KA_OK;
}

template <int KIND, int MAXNT, bool GCTR, bool SINGLE, bool WARP1, bool FULL>
cudaError_t launch_order_t(cudaStream_t s, const KaOrderParams& o, const Plan& pl) {
    auto kern = ka_order_levels_kernel<KIND, GCTR, MAXNT, SINGLE, WARP1, FULL>;
    cudaError_t e = allow_smem(kern, pl.b_smem);
    if (e != cudaSuccess) return e;
    kern<<<1, pl.b_threads, pl.b_smem, s>>>(o);
    return cudaGetLastError();
}

// KIND 0 / 1: slot chains of rows <= 3 (chunk arithmetic, barrier flavour, full chunks are compile-time); 4 / 8: rows of 4 / 5..8
template <int KIND, int MAXNT>
cudaError_t launch_order(cudaStream_t s, const KaOrderParams& o, const Plan& pl) {
    if constexpr (KIND > 1) {
        return pl.b_gctr ? launch_order_t<KIND, MAXNT, true, false, false, false>(s, o, pl) : launch_order_t<KIND, MAXNT, false, false, false, false>(s, o, pl);
    } else {
        const bool warp1 = pl.b_threads == 32;                                                          // window mode
        const bool single = !warp1 && o.uniform_width != 0 && o.uniform_width <= (uint32_t)pl.b_threads;   // chunk = topic
        const bool full = single && o.uniform_width == (uint32_t)pl.b_threads;                          // no idle lane
        const int sel = (pl.b_gctr ? 4 : 0) | (warp1 ? 1 : (full ? 3 : (single ? 2 : 0)));
        switch (sel) {
            case 0: return launch_order_t<KIND, MAXNT, false, false, false, false>(s, o, pl);
            case 1: return launch_order_t<KIND, MAXNT, false, false, true, false>(s, o, pl);
            case 2: return launch_order_t<KIND, MAXNT, false, true, false, false>(s, o, pl);
            case 3: return launch_order_t<KIND, MAXNT, false, true, false, true>(s, o, pl);
            case 4: return launch_order_t<KIND, MAXNT, true, false, false, false>(s, o, pl);
            case 5: return launch_order_t<KIND, MAXNT, true, false, true, false>(s, o, pl);
            case 6: return launch_order_t<KIND, MAXNT, true, true, false, false>(s, o, pl);
            default: return launch_order_t<KIND, MAXNT, true, true, false, true>(s, o, pl);
        }
    }
}

// How many topic sub-blocks the slot chains of one staged block are cut into: the slot-0 chain of sub-block j+1 runs (on
// its own SM) while the slot-1 chain + emit of sub-block j run. A chain launch is one CTA, so sub-blocks are cheap; each
// should still hold a few hundred levels to amortise the launch + ring fill.
int chain_subblocks(const StageDesc& d, int blocks_in_solve) {
    if (d.d_part_off || d.pl.rec_kind != 3 || d.T < 2) return 1;
    int n = std::max(1, 8 / std::max(1, blocks_in_solve));
    n = std::min(n, std::max(1, d.T / 128));
    if (const char* e = std::getenv("KA_CHAIN_SUBBLOCKS")) n = std::max(1, std::min(std::atoi(e), d.T));
    return std::min(n, KA_MAX_CHAIN_BLOCKS);
}

}  // namespace
struct JsonJob {
    int32_t* d_out;        // the solve's rows (device)
    int32_t* d_out_len;
    int S;
    int blocks = 0;
    bool changed_only = false;  // ka_solve_dense_json_changed: text of the rows whose class is not UNCHANGED only
    KaRows rows{};              // changed_only: current + new lists of the run (ka_row_diff)
};
namespace {

// KAG:169-186 for a finished range of rows (a chain sub-block): rows -> JSON text at the running offset of d_json, on c->sj.
int enq_json_rows(ka_ctx* c, cudaStream_t s_done, int64_t row0, int64_t rows, int topic0, int P, bool first, bool last) {
    JsonJob* jj = c->json_job;
    const int k = jj->blocks;
    if (k >= KA_MAX_CHAIN_EVENTS) return KA_ERR_LIMIT;
    KA_CUDA(cudaEventRecord(c->ev_json_in[k], s_done));
    KA_CUDA(cudaStreamWaitEvent(c->sj, c->ev_json_in[k], 0));
    KaJsonParams p{};
    p.Q = (uint32_t)rows;
    p.row0 = (uint32_t)row0;
    p.P = std::max(P, 1);
    p.topic0 = topic0;
    p.name_off = c->d_name_off.as<int64_t>();
    p.names = c->d_names.as<char>();
    p.out = jj->d_out + row0 * jj->S;
    p.out_len = jj->d_out_len + row0;
    p.S = jj->S;
    p.rowlen = c->d_json_rowlen.as<uint32_t>() + row0;
    p.blocksum = c->d_json_blocksum.as<uint32_t>() + (row0 / 256) + k;
    p.total = c->d_json_state.as<unsigned long long>();
    p.frag = c->d_json_state.as<unsigned long long>() + 2 + 2 * k;
    p.json = c->d_json.as<char>();
    p.cap = (unsigned long long)c->d_json.cap;
    p.first = first;
    p.last = last;
    const int nblocks = (int)((rows + 255) / 256);
    if (jj->changed_only) {
        // compact the fragment's changed rows (fragment-relative, row order) into sel; the count stays on the device, so the
        // text kernels below cover every row of the fragment and their blocks beyond the count write nothing
        uint32_t* mask = c->d_sel_mask.as<uint32_t>() + (size_t)(row0 / 256 + k) * 8;
        uint32_t* blockcnt = c->d_sel_blockcnt.as<uint32_t>() + row0 / 256 + k;
        uint32_t* state = c->d_sel_state.as<uint32_t>();   // [0] rows kept so far, then {before, count} per fragment
        uint32_t* sel = c->d_sel.as<uint32_t>() + row0;
        if (nblocks > 0) {
            if (jj->S <= 3) ka_changed_flag_kernel<3><<<nblocks, 256, 0, c->sj>>>(jj->rows, row0, (uint32_t)rows, mask, blockcnt);
            else ka_changed_flag_kernel<8><<<nblocks, 256, 0, c->sj>>>(jj->rows, row0, (uint32_t)rows, mask, blockcnt);
        }
        ka_changed_scan_kernel<<<1, 1024, 0, c->sj>>>(blockcnt, nblocks, state, state + 1 + 2 * k);
        if (nblocks > 0) ka_changed_scatter_kernel<<<nblocks, 256, 0, c->sj>>>(mask, blockcnt, (uint32_t)rows, sel);
        KA_CUDA(cudaGetLastError());
        c->launches += nblocks > 0 ? 3 : 1;
        p.sel = sel;
        p.sel_state = state + 1 + 2 * k;
        if (nblocks > 0) ka_json_len_kernel<true><<<nblocks, 256, 0, c->sj>>>(p);
        ka_json_scan_kernel<<<1, 1024, 0, c->sj>>>(p, nblocks);
        KA_CUDA(allow_smem(ka_json_write_kernel<true>, KA_JSON_SMEM_BYTES + 16));
        ka_json_write_kernel<true><<<std::max(nblocks, 1), 256, KA_JSON_SMEM_BYTES + 16, c->sj>>>(p);
    } else {
        if (nblocks > 0) ka_json_len_kernel<false><<<nblocks, 256, 0, c->sj>>>(p);
        ka_json_scan_kernel<<<1, 1024, 0, c->sj>>>(p, nblocks);
        KA_CUDA(allow_smem(ka_json_write_kernel<false>, KA_JSON_SMEM_BYTES + 16));
        ka_json_write_kernel<false><<<std::max(nblocks, 1), 256, KA_JSON_SMEM_BYTES + 16, c->sj>>>(p);
    }
    KA_CUDA(cudaGetLastError());
    KA_CUDA(cudaMemcpyAsync(c->h_frag + 2 * k, p.frag, 16, cudaMemcpyDeviceToHost, c->sj));
    KA_CUDA(cudaEventRecord(c->ev_json_scan[k], c->sj));
    c->launches += 3;
    jj->blocks = k + 1;
    return KA_OK;
}

struct SubBlock { int t0, t1; int64_t r0, rq; };

SubBlock sub_block(const StageDesc& d, int j, int nsub) {
    SubBlock b;
    b.t0 = (int)((int64_t)d.T * j / nsub);
    b.t1 = (int)((int64_t)d.T * (j + 1) / nsub);
    // ragged blocks are never cut (nsub == 1): sub-block rows follow from the dense shape
    b.r0 = d.d_part_off ? 0 : (int64_t)b.t0 * d.P;
    b.rq = d.d_part_off ? d.Q : (int64_t)(b.t1 - b.t0) * d.P;
    return b;
}

// One slot chain (rows <= 3) over sub-block j of a staged block.
int enq_slot_chain(ka_ctx* c, cudaStream_t s, const StageDesc& d, int slot, int j, int nsub) {
    const Plan& pl = d.pl;
    const SubBlock b = sub_block(d, j, nsub);
    if (b.rq <= 0 || c->N <= 0) return KA_OK;
    KaOrderParams o{};
    o.N = c->N;
    o.S = d.S;
    o.uniform_width = pl.a_levels ? 0u : (uint32_t)d.P;
    o.chunk_end = pl.a_levels ? c->d_lvl_end.as<uint32_t>() + d.q0 : nullptr;
    o.ctr8 = c->d_ctr8.as<int32_t>();
    o.ring_log2 = pl.b_ring_log2;
    const int32_t* loff = pl.a_levels ? c->d_loff.as<int32_t>() + d.topic_base + d.blk : nullptr;
    o.Q = (uint32_t)b.rq;
    o.rec = c->d_rec.as<unsigned char>() + (size_t)(d.q0 + b.r0) * pl.rec_bytes;
    o.pos_base = (uint32_t)b.r0;
    o.chunk_lo_ptr = loff ? loff + b.t0 : nullptr;
    o.chunk_hi_ptr = loff ? loff + b.t1 : nullptr;
    KA_CUDA((slot == 0 ? launch_order<0, 1024>(s, o, pl) : launch_order<1, 1024>(s, o, pl)));
    c->launches++;
    return KA_OK;
}

// Emit of sub-block j (rows <= 3): ordered records -> broker ids, list lengths, slot-2 counters.
int enq_emit_block(ka_ctx* c, cudaStream_t s, const StageDesc& d, int j, int nsub, int32_t* d_out, int32_t* d_out_len) {
    const Plan& pl = d.pl;
    const SubBlock b = sub_block(d, j, nsub);
    if (b.rq <= 0 || c->N <= 0) return KA_OK;
    ka_emit3_kernel<<<(unsigned)((b.rq + 255) / 256), 256, 0, s>>>(
        reinterpret_cast<const uint4*>(c->d_rec.as<unsigned char>() + (size_t)(d.q0 + b.r0) * pl.rec_bytes),
        pl.a_levels ? c->d_perm.as<uint16_t>() + d.q0 + b.r0 : nullptr, d.d_part_off, b.t1 - b.t0, d.P, c->d_broker_id.as<int32_t>(),
        (uint32_t)b.rq, d.S, d_out + (size_t)b.r0 * d.S, d_out_len ? d_out_len + b.r0 : nullptr, c->d_ctr8.as<int32_t>());
    KA_CUDA(cudaGetLastError());
    c->launches++;
    return KA_OK;
}

// The serial chains through Context.counter (KAS:202-239) for a staged block + the parallel emit. d_out/d_out_len: the
// block's rows. Rows <= 3: slot-0 chain on c->sb1, slot-1 chain + emit on `s`; the caller has made c->sb1 wait for the
// stage (c->ev_chain_in recorded after kernel A / the counter import). Everything is joined back into `s`.
int enq_order_emit(ka_ctx* c, cudaStream_t s, const StageDesc& d, int32_t* d_out, int32_t* d_out_len, int blocks_in_solve) {
    const int N = c->N, S = d.S;
    const Plan& pl = d.pl;
    if (d.Q <= 0 || N <= 0) return KA_OK;
    KaOrderParams o{};
    o.N = N;
    o.S = S;
    o.uniform_width = pl.a_levels ? 0u : (uint32_t)d.P;
    o.chunk_end = pl.a_levels ? c->d_lvl_end.as<uint32_t>() + d.q0 : nullptr;
    o.ctr8 = c->d_ctr8.as<int32_t>();
    o.broker_id = c->d_broker_id.as<int32_t>();
    o.ring_log2 = pl.b_ring_log2;
    const int32_t* loff = pl.a_levels ? c->d_loff.as<int32_t>() + d.topic_base + d.blk : nullptr;
    unsigned char* rec = c->d_rec.as<unsigned char>() + (size_t)d.q0 * pl.rec_bytes;
    if (pl.rec_kind != 3) {  // rows of 4..8: one fused chain over all slots, rows written by the kernel
        o.Q = (uint32_t)d.Q;
        o.rec = rec;
        o.chunk_lo_ptr = loff;
        o.chunk_hi_ptr = loff ? loff + d.T : nullptr;
        o.out = d_out;
        o.out_len = d_out_len;
        KA_CUDA((pl.rec_kind == 4 ? launch_order<4, 512>(s, o, pl) : launch_order<8, 256>(s, o, pl)));
        c->launches++;
        if (c->json_job) return enq_json_rows(c, s, d.q0, d.Q, d.topic_base, d.P, d.blk == 0, d.blk == blocks_in_solve - 1);
        return KA_OK;
    }
    const int nsub = chain_subblocks(d, blocks_in_solve);
    cudaStream_t s1 = c->sb1;
    for (int j = 0; j < nsub; ++j) {
        const int e = c->chain_ev_next++ % KA_MAX_CHAIN_EVENTS;
        if (c->timing) KA_CUDA(cudaEventRecord(c->ev_chain[e][0], s1));
        int rc = enq_slot_chain(c, s1, d, 0, j, nsub);                    // slot-0 chain
        if (rc != KA_OK) return rc;
        if (c->timing) KA_CUDA(cudaEventRecord(c->ev_chain[e][1], s1));
        KA_CUDA(cudaEventRecord(c->ev_b1[e], s1));
        KA_CUDA(cudaStreamWaitEvent(s, c->ev_b1[e], 0));
        if (c->timing) KA_CUDA(cudaEventRecord(c->ev_chain[e][2], s));
        if ((rc = enq_slot_chain(c, s, d, 1, j, nsub)) != KA_OK) return rc;   // slot-1 chain
        if ((rc = enq_emit_block(c, s, d, j, nsub, d_out, d_out_len)) != KA_OK) return rc;
        if (c->timing) KA_CUDA(cudaEventRecord(c->ev_chain[e][3], s));
        if (c->host_out) {   // rows of this sub-block are final: copy them out on c->sj (on `s` itself once the events run out)
            const SubBlock b = sub_block(d, j, nsub);
            const int64_t r = d.q0 + b.r0;
            cudaStream_t so = s;
            if (c->out_copies < KA_MAX_CHAIN_EVENTS) {
                KA_CUDA(cudaEventRecord(c->ev_json_in[c->out_copies], s));
                KA_CUDA(cudaStreamWaitEvent(c->sj, c->ev_json_in[c->out_copies], 0));
                c->out_copies++;
                so = c->sj;
            }
            KA_CUDA(cudaMemcpyAsync(c->host_out + r * S, c->dev_out + r * S, (size_t)b.rq * S * 4, cudaMemcpyDeviceToHost, so));
            if (c->host_out_len) KA_CUDA(cudaMemcpyAsync(c->host_out_len + r, c->dev_out_len + r, (size_t)b.rq * 4, cudaMemcpyDeviceToHost, so));
        }
        if (c->json_job) {   // the sub-block's rows are final: their JSON text can be built and streamed out now
            const SubBlock b = sub_block(d, j, nsub);
            if ((rc = enq_json_rows(c, s, d.q0 + b.r0, b.rq, d.topic_base + b.t0, d.P, d.blk == 0 && j == 0,
                                    d.blk == blocks_in_solve - 1 && j == nsub - 1)) != KA_OK) return rc;
        }
        c->chain_used = std::min(c->chain_used + 1, KA_MAX_CHAIN_EVENTS);
    }
    return KA_OK;
}

// c->sb1 (slot-0 chain stream) must see everything enqueued on `s` so far: the staged records / imported counters
int chain_fork(ka_ctx* c, cudaStream_t s) {
    KA_CUDA(cudaEventRecord(c->ev_chain_in, s));
    KA_CUDA(cudaStreamWaitEvent(c->sb1, c->ev_chain_in, 0));
    return KA_OK;
}

// status words back to pinned host memory (async)
int enq_flags_readback(ka_ctx* c, cudaStream_t s) {
    KA_CUDA(cudaMemcpyAsync(&c->h_pin->err_topic, c->d_flags.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
    return KA_OK;
}

// How many topic super-chunks a dense solve is pipelined in (1 = no pipelining).
int pipeline_stages(int T, int64_t Q) {
    // worthwhile only when every chunk still has enough topics to keep kernel A throughput-bound (a topic is one warp:
    // with few topics per chunk A is latency-bound and K chunks cost K times as much — measured on config 5)
    int k = Q >= 262144 ? std::min(4, T / 2048) : 1;
    if (const char* e = std::getenv("KA_PIPELINE_STAGES")) k = std::atoi(e);
    return std::max(1, std::min(k, std::min(8, std::max(T, 1))));
}

// Whole dense solve on `s_main`, pipelined in K topic super-chunks: the aux stream runs (H2D,) kernel A and the level
// tables of chunk k+1 while s_main runs the leader-order chain of chunk k (and the D2H of its output); s_main orders the
// chunks strictly one after the other through the counters in ctr8.
// h_* non-null = host-buffer form (copies inside); d_* always valid device buffers of the full problem.
int run_dense(ka_ctx* c, cudaStream_t s_main, int T, int P, int RF, int desired_rf, int S, const int32_t* h_hash, const int32_t* h_cur,
              int32_t* d_hash, int32_t* d_cur, int32_t* d_out, int32_t* d_out_len, int32_t* h_out, int32_t* h_out_len, ka_status* st) {
    const int64_t Q = (int64_t)T * P;
    const int rf_t = desired_rf >= 0 ? desired_rf : RF;
    const int64_t capmax = c->N > 0 ? ((int64_t)P * std::max(rf_t, 0) + c->N - 1) / c->N : 0;
    const int K = pipeline_stages(T, Q);
    c->host_out = nullptr;
    StageDesc ds[8];
    // Block boundaries: the first block's H2D and the last block's D2H are the only copies that nothing overlaps, so with
    // host buffers the end blocks get half the weight of the inner ones (1:2:..:2:1).
    const bool host_io = (h_cur != nullptr || h_out != nullptr) && K >= 3;
    const int wsum = host_io ? 2 * (K - 1) : K;
    auto bound = [&](int k) { return k <= 0 ? 0 : (k >= K ? T : (int)((int64_t)T * (host_io ? 2 * k - 1 : k) / wsum)); };
    for (int k = 0; k < K; ++k) {
        const int t0 = bound(k), t1 = bound(k + 1);
        StageDesc& d = ds[k];
        d.topic_base = t0;
        d.T = t1 - t0;
        d.q0 = (int64_t)t0 * P;
        d.Q = (int64_t)d.T * P;
        d.d_hash = d_hash + t0;
        d.P = P;
        d.RF = RF;
        d.d_cur = d_cur + d.q0 * RF;
        d.desired_rf = desired_rf;
        d.S = S;
        d.Pmax = P;
        d.capmax = capmax;
        d.blk = k;
        int rc = make_plan(c, d.Q, S, P, capmax, false, d.pl, st);
        if (rc != KA_OK) return rc;
    }
    int rc = reserve_scratch(c, Q, ds[0].pl.rec_bytes, T, K, ds[0].pl.a_levels != 0);
    if (rc != KA_OK) return set_status(st, rc);
    c->last_stages = K;
    if (c->timing) KA_CUDA(cudaEventRecord(c->ev[0], s_main));
    if (K == 1) {
        cudaStream_t s = s_main;
        StageDesc& d = ds[0];
        if (h_hash && T > 0) KA_CUDA(cudaMemcpyAsync(d_hash, h_hash, (size_t)T * 4, cudaMemcpyHostToDevice, s));
        if (h_cur && Q * RF > 0) KA_CUDA(cudaMemcpyAsync(d_cur, h_cur, (size_t)Q * RF * 4, cudaMemcpyHostToDevice, s));
        if ((rc = reset_flags(c, s)) != KA_OK) return rc;
        if (c->timing) KA_CUDA(cudaEventRecord(c->ev[1], s));
        c->ev_mark = c->ev[2];
        if ((rc = enq_stage(c, s, d)) != KA_OK) return rc;
        c->ev_mark = nullptr;
        if (c->timing) KA_CUDA(cudaEventRecord(c->ev[3], s));
        if ((rc = chain_fork(c, s)) != KA_OK) return rc;
        if ((rc = enq_order_emit(c, s, d, d_out, d_out_len, 1)) != KA_OK) return rc;
        if (c->timing) KA_CUDA(cudaEventRecord(c->ev[4], s));

        if (h_out && Q > 0 && c->N > 0) {
            KA_CUDA(cudaMemcpyAsync(h_out, d_out, (size_t)Q * S * 4, cudaMemcpyDeviceToHost, s));
            if (h_out_len) KA_CUDA(cudaMemcpyAsync(h_out_len, d_out_len, (size_t)Q * 4, cudaMemcpyDeviceToHost, s));
        }
    } else {
        cudaStream_t aux = c->aux;
        const bool stream_out = h_out && ds[0].pl.rec_kind == 3 && !c->json_job;
        c->host_out = stream_out ? h_out : nullptr;
        c->host_out_len = stream_out ? h_out_len : nullptr;
        c->dev_out = d_out;
        c->dev_out_len = d_out_len;
        c->out_copies = 0;
        KA_CUDA(cudaEventRecord(c->ev_in, s_main));           // inputs ready / earlier work on s_main done
        if (stream_out) KA_CUDA(cudaStreamWaitEvent(c->sj, c->ev_in, 0));
        KA_CUDA(cudaStreamWaitEvent(aux, c->ev_in, 0));
        if ((rc = reset_flags(c, aux)) != KA_OK) return rc;
        for (int k = 0; k < K; ++k) {
            StageDesc& d = ds[k];
            if (h_hash && d.T > 0) KA_CUDA(cudaMemcpyAsync(d_hash + d.topic_base, h_hash + d.topic_base, (size_t)d.T * 4, cudaMemcpyHostToDevice, aux));
            if (h_cur && d.Q * RF > 0)
                KA_CUDA(cudaMemcpyAsync(d_cur + d.q0 * RF, h_cur + d.q0 * RF, (size_t)d.Q * RF * 4, cudaMemcpyHostToDevice, aux));
            if (c->timing) KA_CUDA(cudaEventRecord(c->ev_pipe[k][0], aux));
            c->ev_mark = c->timing ? c->ev_pipe[k][1] : nullptr;
            if ((rc = enq_stage(c, aux, d)) != KA_OK) return rc;
            c->ev_mark = nullptr;
            if (c->timing) KA_CUDA(cudaEventRecord(c->ev_pipe[k][2], aux));
            KA_CUDA(cudaEventRecord(c->ev_stage[k], aux));
            KA_CUDA(cudaStreamWaitEvent(s_main, c->ev_stage[k], 0));
            KA_CUDA(cudaStreamWaitEvent(c->sb1, c->ev_stage[k], 0));
            if (k == 0) KA_CUDA(cudaStreamWaitEvent(c->sb1, c->ev_in, 0));
            if (c->timing) KA_CUDA(cudaEventRecord(c->ev_pipe[k][3], s_main));
            if ((rc = enq_order_emit(c, s_main, d, d_out + d.q0 * S, d_out_len ? d_out_len + d.q0 : nullptr, K)) != KA_OK) return rc;
            if (c->timing) KA_CUDA(cudaEventRecord(c->ev_pipe[k][4], s_main));

            if (h_out && d.Q > 0 && c->N > 0 && !c->host_out) {   // rows of 4..8: one copy per block on the caller's stream
                KA_CUDA(cudaMemcpyAsync(h_out + d.q0 * S, d_out + d.q0 * S, (size_t)d.Q * S * 4, cudaMemcpyDeviceToHost, s_main));
                if (h_out_len) KA_CUDA(cudaMemcpyAsync(h_out_len + d.q0, d_out_len + d.q0, (size_t)d.Q * 4, cudaMemcpyDeviceToHost, s_main));
            }
        }
    }
    if (c->host_out) {   // join the copy-out stream back into the caller's stream
        KA_CUDA(cudaEventRecord(c->ev_out_done, c->sj));
        KA_CUDA(cudaStreamWaitEvent(s_main, c->ev_out_done, 0));
        c->host_out = nullptr;
    }
    if ((rc = enq_flags_readback(c, s_main)) != KA_OK) return rc;
    if (c->timing) { KA_CUDA(cudaEventRecord(c->ev[5], s_main)); c->ev_valid = true; }
    return KA_OK;
}

// Wait for the stream, translate device flags into a ka_status.
int finish_status(ka_ctx* c, cudaStream_t s, ka_status* st) {
    KA_CUDA(cudaStreamSynchronize(s));
    c->pending_status = false;
    ka_status r{};
    r.code = KA_OK;
    r.topic_index = -1;
    r.partition = -1;
    if (c->h_pin->err_topic != -1) {
        const int t = c->h_pin->err_topic;
        KA_CUDA(cudaMemcpy(&c->h_pin->tstatus, c->d_tstatus.as<int4>() + t, sizeof(int4), cudaMemcpyDeviceToHost));
        r.code = c->h_pin->tstatus.x;
        r.topic_index = t + (c->last_was_staged ? c->topic_base : 0);
        int ord = c->h_pin->tstatus.y;
        r.partition = ord;
        if (ord >= 0 && c->last_part_id && c->last_part_off) r.partition = c->last_part_id[c->last_part_off[t] + ord];
        r.a = c->h_pin->tstatus.z;
        r.b = c->h_pin->tstatus.w;
    }
    if (c->timing && c->ev_valid) {
        for (int i = 0; i < 8; ++i) c->last_ms[i] = 0.f;
        cudaEventElapsedTime(&c->last_ms[5], c->ev[0], c->ev[5]);  // total on the stream
        if (c->last_stages <= 1) {
            cudaEventElapsedTime(&c->last_ms[3], c->ev[0], c->ev[1]);  // H2D
            cudaEventElapsedTime(&c->last_ms[0], c->ev[1], c->ev[2]);  // kernel A
            cudaEventElapsedTime(&c->last_ms[1], c->ev[2], c->ev[3]);  // level tables (scan + fill; absent when capacity is 1)
            cudaEventElapsedTime(&c->last_ms[7], c->ev[3], c->ev[4]);  // all chains + emit, wall time on the stream
            cudaEventElapsedTime(&c->last_ms[4], c->ev[4], c->ev[5]);  // D2H
        } else {  // pipelined: phases of different chunks overlap; report the per-phase sums
            for (int k = 0; k < c->last_stages; ++k) {
                float a = 0.f, t = 0.f, b = 0.f;
                cudaEventElapsedTime(&a, c->ev_pipe[k][0], c->ev_pipe[k][1]);
                cudaEventElapsedTime(&t, c->ev_pipe[k][1], c->ev_pipe[k][2]);
                cudaEventElapsedTime(&b, c->ev_pipe[k][3], c->ev_pipe[k][4]);
                c->last_ms[0] += a;
                c->last_ms[1] += t;
                c->last_ms[7] += b;
            }
        }
        if (c->chain_used > 0) {  // rows <= 3: per-slot chains (sums over the sub-blocks; the two chains overlap in time)
            for (int e = 0; e < c->chain_used; ++e) {
                float b1 = 0.f, b2 = 0.f;
                cudaEventElapsedTime(&b1, c->ev_chain[e][0], c->ev_chain[e][1]);
                cudaEventElapsedTime(&b2, c->ev_chain[e][2], c->ev_chain[e][3]);
                c->last_ms[2] += b1;
                c->last_ms[6] += b2;
            }
        } else if (c->slot_timed[0] || c->slot_timed[1]) {  // per-slot entry points (topic-sharded runs)
            if (c->slot_timed[0]) cudaEventElapsedTime(&c->last_ms[2], c->ev_chain[0][0], c->ev_chain[0][1]);
            if (c->slot_timed[1]) cudaEventElapsedTime(&c->last_ms[6], c->ev_chain[1][0], c->ev_chain[1][1]);
        } else {
            c->last_ms[2] = c->last_ms[7];  // rows of 4..8: one fused chain
        }
    }
    c->last = r;
    if (st) *st = r;
    return r.code;
}

}  // namespace

// =================================================================================================
extern "C" {

const char* ka_version(void) { return "kassign-b200 0.1 (sm_100a)"; }

int32_t ka_java_string_hash(const char* s) {
    // java.lang.String.hashCode over UTF-16 code units (KAS:190)
    uint32_t h = 0;
    const unsigned char* u = reinterpret_cast<const unsigned char*>(s);
    while (*u) {
        uint32_t cp;
        int extra;
        unsigned char b = *u++;
        if (b < 0x80) { cp = b; extra = 0; }
        else if ((b & 0xE0) == 0xC0) { cp = b & 0x1F; extra = 1; }
        else if ((b & 0xF0) == 0xE0) { cp = b & 0x0F; extra = 2; }
        else if ((b & 0xF8) == 0xF0) { cp = b & 0x07; extra = 3; }
        else { cp = 0xFFFD; extra = 0; }
        while (extra-- > 0 && *u) cp = (cp << 6) | (*u++ & 0x3F);
        if (cp >= 0x10000) {
            cp -= 0x10000;
            h = h * 31u + (0xD800u + (cp >> 10));
            h = h * 31u + (0xDC00u + (cp & 0x3FFu));
        } else {
            h = h * 31u + cp;
        }
    }
    return (int32_t)h;
}

int32_t ka_rack_indices(int32_t N, const int32_t* broker_id, const char* const* rack_name, int32_t* broker_rack) {
    if (N < 0 || (N > 0 && (!broker_id || !broker_rack))) return KA_ERR_BAD_ARG;
    // rack key = the rack string, or Integer.toString(id) when no rack is defined (KAS:81-86); brokers
    // share a Rack object iff their keys are equal strings (KAS:90-94).
    std::map<std::string, int32_t> key2idx;
    for (int i = 0; i < N; ++i) {
        std::string key = (rack_name && rack_name[i]) ? std::string(rack_name[i]) : std::to_string(broker_id[i]);
        auto it = key2idx.find(key);
        if (it == key2idx.end()) it = key2idx.emplace(key, (int32_t)key2idx.size()).first;
        broker_rack[i] = it->second;
    }
    return KA_OK;
}

ka_ctx* ka_ctx_create(int32_t device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
        cudaGetLastError();
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    ka_ctx* c = new (std::nothrow) ka_ctx();
    if (!c) return nullptr;
    c->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return nullptr; }
    if (cudaHostAlloc(reinterpret_cast<void**>(&c->h_pin), sizeof(HostPinned), cudaHostAllocDefault) != cudaSuccess) { delete c; return nullptr; }
    for (auto& e : c->ev) cudaEventCreate(&e);
    if (cudaStreamCreateWithFlags(&c->aux, cudaStreamNonBlocking) != cudaSuccess) { delete c; return nullptr; }
    if (cudaStreamCreateWithFlags(&c->sb1, cudaStreamNonBlocking) != cudaSuccess) { delete c; return nullptr; }
    if (cudaStreamCreateWithFlags(&c->sj, cudaStreamNonBlocking) != cudaSuccess) { delete c; return nullptr; }
    if (cudaHostAlloc(reinterpret_cast<void**>(&c->h_frag), 2 * KA_MAX_CHAIN_EVENTS * sizeof(unsigned long long), cudaHostAllocDefault) != cudaSuccess) { delete c; return nullptr; }
    for (auto& e : c->ev_json_in) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    for (auto& e : c->ev_json_scan) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_chain_in, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_out_done, cudaEventDisableTiming);
    for (auto& e : c->ev_b1) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    for (auto& row : c->ev_chain)
        for (auto& e : row) cudaEventCreate(&e);
    cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming);
    for (auto& e : c->ev_stage) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    for (auto& row : c->ev_pipe)
        for (auto& e : row) cudaEventCreate(&e);
    return c;
}

void ka_ctx_destroy(ka_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (DevBuf* b : {&c->d_blob, &c->d_glut, &c->d_broker_id, &c->d_ctr8, &c->d_hash, &c->d_part_off, &c->d_rep_off, &c->d_cur, &c->d_rec,
                      &c->d_perm, &c->d_ntl, &c->d_loff, &c->d_lend, &c->d_lvl_end, &c->d_out, &c->d_out_len, &c->d_tstatus, &c->d_flags})
        b->release();
    for (auto& e : c->ev)
        if (e) cudaEventDestroy(e);
    if (c->aux) { cudaStreamSynchronize(c->aux); cudaStreamDestroy(c->aux); }
    if (c->sb1) { cudaStreamSynchronize(c->sb1); cudaStreamDestroy(c->sb1); }
    if (c->sj) { cudaStreamSynchronize(c->sj); cudaStreamDestroy(c->sj); }
    if (c->h_frag) cudaFreeHost(c->h_frag);
    for (auto& e : c->ev_json_in) if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_json_scan) if (e) cudaEventDestroy(e);
    for (DevBuf* b : {&c->d_json, &c->d_names, &c->d_name_off, &c->d_json_rowlen, &c->d_json_blocksum, &c->d_json_state}) b->release();
    for (DevBuf* b : {&c->d_rep_lut, &c->d_rep_ids, &c->d_plan_tot, &c->d_plan_stats, &c->d_plan_class, &c->d_sel, &c->d_sel_mask,
                      &c->d_sel_blockcnt, &c->d_sel_state})
        b->release();
    if (c->ev_chain_in) cudaEventDestroy(c->ev_chain_in);
    if (c->ev_out_done) cudaEventDestroy(c->ev_out_done);
    for (auto& e : c->ev_b1) if (e) cudaEventDestroy(e);
    for (auto& row : c->ev_chain)
        for (auto& e : row) if (e) cudaEventDestroy(e);
    if (c->ev_in) cudaEventDestroy(c->ev_in);
    for (auto& e : c->ev_stage) if (e) cudaEventDestroy(e);
    for (auto& row : c->ev_pipe)
        for (auto& e : row) if (e) cudaEventDestroy(e);
    if (c->h_pin) cudaFreeHost(c->h_pin);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c->staged_block;
    delete c;
}

int32_t ka_ctx_reset(ka_ctx* c) {
    if (!c) return KA_ERR_NO_DEVICE;
    KA_CUDA(cudaSetDevice(c->device));
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);  // do not race an in-flight asynchronous solve
    c->parked.clear();
    if (c->N > 0 && c->d_ctr8.p) KA_CUDA(cudaMemset(c->d_ctr8.p, 0, (size_t)c->N * KA_MAX_SLOTS * 4));
    return KA_OK;
}

int32_t ka_ctx_set_brokers(ka_ctx* c, int32_t N, const int32_t* broker_id, const int32_t* broker_rack) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (N < 0 || (N > 0 && (!broker_id || !broker_rack))) return KA_ERR_BAD_ARG;
    if (N > 65535) return KA_ERR_LIMIT;
    for (int i = 0; i < N; ++i) {
        if (i > 0 && broker_id[i] <= broker_id[i - 1]) return KA_ERR_BAD_ARG;  // strictly ascending
        if (broker_rack[i] < 0 || broker_rack[i] >= 65535) return KA_ERR_BAD_ARG;
    }
    KA_CUDA(cudaSetDevice(c->device));
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    int rc = park_counters(c);
    if (rc != KA_OK) return rc;

    c->N = N;
    c->broker_id.assign(broker_id, broker_id + N);
    c->broker_rack.assign(broker_rack, broker_rack + N);
    const size_t npad = align16((size_t)std::max(N, 1) * 2) / 2;  // uint16 elements, 16B multiple
    // compact rack ids in order of first appearance (rack identity is all that matters, KAS:90-94)
    std::vector<uint16_t> rackc(std::max(N, 1), 0);
    {
        std::unordered_map<int32_t, int> seen;
        for (int i = 0; i < N; ++i) {
            auto it = seen.find(broker_rack[i]);
            if (it == seen.end()) it = seen.emplace(broker_rack[i], (int)seen.size()).first;
            rackc[i] = (uint16_t)it->second;
        }
        c->R = (int)seen.size();
    }
    std::vector<uint16_t> blob;
    const IdLut lut = make_id_lut(N, broker_id);
    c->lut_mode = lut.mode;
    c->min_id = lut.min_id;
    c->range = lut.range;
    const size_t lut_elems = lut.mode == KA_LUT_SMEM ? lut.lut.size() : 0;  // the shared-memory LUT travels in the blob
    if (lut.mode == KA_LUT_GLOBAL) {
        KA_CUDA(c->d_glut.reserve(lut.lut.size() * 2));
        KA_CUDA(cudaMemcpy(c->d_glut.p, lut.lut.data(), lut.lut.size() * 2, cudaMemcpyHostToDevice));
    }
    const size_t roff_elems = align16((size_t)(c->R + 1) * 2) / 2;
    c->lut_off = (int)npad;
    c->roff_off = (int)(npad + lut_elems);
    c->memb_off = (int)(npad + lut_elems + roff_elems);
    blob.assign(npad + lut_elems + roff_elems + npad, (uint16_t)KA_DEAD);
    for (int i = 0; i < N; ++i) blob[i] = rackc[i];
    std::copy(lut.lut.begin(), lut.lut.begin() + lut_elems, blob.begin() + npad);
    {   // rack member lists (CSR): sorted indices ascending inside each rack
        std::vector<int> cntr(c->R + 1, 0);
        for (int i = 0; i < N; ++i) cntr[rackc[i] + 1]++;
        for (int r = 0; r < c->R; ++r) cntr[r + 1] += cntr[r];
        for (int r = 0; r <= c->R; ++r) blob[c->roff_off + r] = (uint16_t)cntr[r];
        std::vector<int> fill(cntr.begin(), cntr.end() - 1);
        for (int i = 0; i < N; ++i) blob[c->memb_off + fill[rackc[i]]++] = (uint16_t)i;
    }
    c->blob_bytes = (int)(blob.size() * 2);
    KA_CUDA(c->d_blob.reserve(blob.size() * 2));
    KA_CUDA(cudaMemcpy(c->d_blob.p, blob.data(), blob.size() * 2, cudaMemcpyHostToDevice));
    KA_CUDA(c->d_broker_id.reserve((size_t)std::max(N, 1) * 4));
    if (N > 0) KA_CUDA(cudaMemcpy(c->d_broker_id.p, broker_id, (size_t)N * 4, cudaMemcpyHostToDevice));
    // counters for the new table
    std::vector<int32_t> h((size_t)(std::max(N, 1) + 1) * KA_MAX_SLOTS, 0);  // + the order kernel's dummy row (index N)
    for (int i = 0; i < N; ++i) {
        auto it = c->parked.find(broker_id[i]);
        if (it != c->parked.end()) std::copy(it->second.begin(), it->second.end(), h.begin() + (size_t)i * KA_MAX_SLOTS);
    }
    KA_CUDA(c->d_ctr8.reserve(h.size() * 4));
    KA_CUDA(cudaMemcpy(c->d_ctr8.p, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    return KA_OK;
}

int32_t ka_ctx_counter_slots(ka_ctx*) { return KA_MAX_SLOTS; }

int32_t ka_ctx_get_counters(ka_ctx* c, int32_t* counter) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (!counter) return KA_ERR_BAD_ARG;
    KA_CUDA(cudaSetDevice(c->device));
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    if (c->N > 0) KA_CUDA(cudaMemcpy(counter, c->d_ctr8.p, (size_t)c->N * KA_MAX_SLOTS * 4, cudaMemcpyDeviceToHost));
    return KA_OK;
}

int32_t ka_ctx_set_counters(ka_ctx* c, const int32_t* counter) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (!counter) return KA_ERR_BAD_ARG;
    KA_CUDA(cudaSetDevice(c->device));
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    if (c->N > 0) KA_CUDA(cudaMemcpy(c->d_ctr8.p, counter, (size_t)c->N * KA_MAX_SLOTS * 4, cudaMemcpyHostToDevice));
    return KA_OK;
}

int32_t ka_ctx_export_counters_device(ka_ctx* c, int32_t* d_counter, void* stream) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (!d_counter) return KA_ERR_BAD_ARG;
    KA_CUDA(cudaSetDevice(c->device));
    if (c->N > 0)
        KA_CUDA(cudaMemcpyAsync(d_counter, c->d_ctr8.p, (size_t)c->N * KA_MAX_SLOTS * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return KA_OK;
}

int32_t ka_ctx_import_counters_device(ka_ctx* c, const int32_t* d_counter, void* stream) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (!d_counter) return KA_ERR_BAD_ARG;
    KA_CUDA(cudaSetDevice(c->device));
    if (c->N > 0)
        KA_CUDA(cudaMemcpyAsync(c->d_ctr8.p, d_counter, (size_t)c->N * KA_MAX_SLOTS * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return KA_OK;
}

int32_t ka_ctx_set_timing(ka_ctx* c, int32_t enabled) {
    if (!c) return KA_ERR_NO_DEVICE;
    c->timing = enabled != 0;
    return KA_OK;
}

int32_t ka_ctx_last_timing(ka_ctx* c, float* ms) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (!ms) return KA_ERR_BAD_ARG;
    for (int i = 0; i < 8; ++i) ms[i] = c->last_ms[i];
    return KA_OK;
}

int64_t ka_ctx_launch_count(ka_ctx* c) { return c ? c->launches : 0; }

int32_t ka_last_status(ka_ctx* c, ka_status* st) {
    if (!c) return set_status(st, KA_ERR_NO_DEVICE);
    if (cudaSetDevice(c->device) != cudaSuccess) return set_status(st, KA_ERR_CUDA);
    if (c->pending_status) return finish_status(c, c->last_stream, st);
    if (st) *st = c->last;
    return c->last.code;
}

static int validate_dense(ka_ctx* c, int32_t T, int32_t P, int32_t RF, int32_t desired_rf, int32_t S, ka_status* st) {
    set_status(st, KA_OK);
    if (!c) return set_status(st, KA_ERR_NO_DEVICE);
    if (T < 0 || P < 0 || RF < 0) return set_status(st, KA_ERR_BAD_ARG);
    if (S < 1 || S > KA_MAX_SLOTS) return set_status(st, KA_ERR_LIMIT, -1, -1, S);
    const int rf_t = desired_rf >= 0 ? desired_rf : RF;
    if (S < RF || (rf_t <= c->N && S < rf_t)) return set_status(st, KA_ERR_BAD_ARG, -1, -1, S);
    return KA_OK;
}

// Rows of a dense solve as the movement plan reads them; recorded when the solve is enqueued (ka_plan_last runs on them).
static void keep_dense_rows(ka_ctx* c, int64_t Q, const int32_t* d_cur, int RF, int32_t* d_out, int32_t* d_out_len, int S, int desired_rf) {
    c->plan_rows = KaRows{d_cur, nullptr, RF, d_out, d_out_len, S, desired_rf >= 0 ? desired_rf : RF};
    c->plan_Q = Q;
    c->plan_valid = true;
}

int32_t ka_solve_dense_device(ka_ctx* c, int32_t T, const int32_t* d_topic_hash, int32_t P, int32_t RF,
                              const int32_t* d_cur_broker, int32_t desired_rf, int32_t out_stride,
                              int32_t* d_out_len, int32_t* d_out_broker, void* stream, ka_status* st) {
    if (c) c->plan_valid = false;
    int rc = validate_dense(c, T, P, RF, desired_rf, out_stride, st);
    if (rc != KA_OK) return rc;
    if (cudaSetDevice(c->device) != cudaSuccess) return set_status(st, KA_ERR_CUDA);
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    cudaStream_t s = (cudaStream_t)stream;
    c->last_part_id = nullptr;
    c->last_part_off = nullptr;
    c->staged = false;
    c->last_was_staged = false;
    rc = run_dense(c, s, T, P, RF, desired_rf, out_stride, nullptr, nullptr, const_cast<int32_t*>(d_topic_hash),
                   const_cast<int32_t*>(d_cur_broker), d_out_broker, d_out_len, nullptr, nullptr, st);
    if (rc != KA_OK) { if (st && st->code != rc) set_status(st, rc); return rc; }
    keep_dense_rows(c, (int64_t)T * P, d_cur_broker, RF, d_out_broker, d_out_len, out_stride, desired_rf);
    c->last_stream = s;
    c->pending_status = true;
    if (st) return finish_status(c, s, st);
    return KA_OK;
}

int32_t ka_stage_dense_device(ka_ctx* c, int32_t T, const int32_t* d_topic_hash, int32_t P, int32_t RF,
                              const int32_t* d_cur_broker, int32_t desired_rf, int32_t out_stride, void* stream) {
    if (c) c->plan_valid = false;   // the split stage / order / emit solve has no movement plan
    ka_status lst;
    int rc = validate_dense(c, T, P, RF, desired_rf, out_stride, &lst);
    if (rc != KA_OK) return rc;
    if (cudaSetDevice(c->device) != cudaSuccess) return KA_ERR_CUDA;
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    cudaStream_t s = (cudaStream_t)stream;
    c->host_out = nullptr;
    if (!c->staged_block) c->staged_block = new StagedBlock();
    StageDesc& d = c->staged_block->d;
    d = StageDesc();
    d.T = T;
    d.Q = (int64_t)T * P;
    d.d_hash = d_topic_hash;
    d.P = P;
    d.RF = RF;
    d.d_cur = d_cur_broker;
    d.desired_rf = desired_rf;
    d.S = out_stride;
    d.Pmax = P;
    const int rf_t = desired_rf >= 0 ? desired_rf : RF;
    d.capmax = c->N > 0 ? ((int64_t)P * std::max(rf_t, 0) + c->N - 1) / c->N : 0;
    c->staged = false;
    rc = make_plan(c, d.Q, d.S, d.Pmax, d.capmax, false, d.pl, &lst);
    if (rc != KA_OK) return rc;
    if ((rc = reserve_scratch(c, d.Q, d.pl.rec_bytes, T, 1, d.pl.a_levels != 0)) != KA_OK) return rc;
    c->last_part_id = nullptr;
    c->last_part_off = nullptr;
    c->last_stages = 1;
    if (c->timing) { cudaEventRecord(c->ev[0], s); cudaEventRecord(c->ev[1], s); }
    if ((rc = reset_flags(c, s)) != KA_OK) return rc;
    c->ev_mark = c->timing ? c->ev[2] : nullptr;
    rc = enq_stage(c, s, d);
    c->ev_mark = nullptr;
    if (rc != KA_OK) return rc;
    if (c->timing) cudaEventRecord(c->ev[3], s);   // end of the stage (the chains may wait for another rank after this)
    c->staged = true;
    return KA_OK;
}

int32_t ka_order_device(ka_ctx* c, int32_t* d_out_len, int32_t* d_out_broker, void* stream, ka_status* st) {
    if (!c) return set_status(st, KA_ERR_NO_DEVICE);
    if (cudaSetDevice(c->device) != cudaSuccess) return set_status(st, KA_ERR_CUDA);
    if (!c->staged || !c->staged_block) return set_status(st, KA_ERR_BAD_ARG);
    cudaStream_t s = (cudaStream_t)stream;
    const StageDesc& d = c->staged_block->d;
    int rc;
    if ((rc = chain_fork(c, s)) != KA_OK) return set_status(st, rc);
    if ((rc = enq_order_emit(c, s, d, d_out_broker, d_out_len, 1)) != KA_OK) return set_status(st, rc);
    if (c->timing) cudaEventRecord(c->ev[4], s);
    if ((rc = enq_flags_readback(c, s)) != KA_OK) return set_status(st, rc);
    if (c->timing) { cudaEventRecord(c->ev[5], s); c->ev_valid = true; }
    c->staged = false;
    c->last_was_staged = true;
    c->last_stream = s;
    c->pending_status = true;
    if (st) return finish_status(c, s, st);
    return KA_OK;
}

int32_t ka_staged_slot_chains(ka_ctx* c) {
    if (!c || !c->staged || !c->staged_block) return 0;
    return c->staged_block->d.pl.rec_kind == 3 ? 2 : 0;
}

int32_t ka_order_slot_device(ka_ctx* c, int32_t slot, void* stream) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (cudaSetDevice(c->device) != cudaSuccess) return KA_ERR_CUDA;
    if (!c->staged || !c->staged_block || c->staged_block->d.pl.rec_kind != 3 || slot < 0 || slot > 1) return KA_ERR_BAD_ARG;
    const StageDesc& d = c->staged_block->d;
    cudaStream_t s = (cudaStream_t)stream;
    const int nsub = chain_subblocks(d, 1);
    cudaEvent_t e0 = c->ev_chain[slot][0], e1 = c->ev_chain[slot][1];
    if (c->timing) cudaEventRecord(e0, s);
    for (int j = 0; j < nsub; ++j) {
        int rc = enq_slot_chain(c, s, d, slot, j, nsub);
        if (rc != KA_OK) return rc;
    }
    if (c->timing) cudaEventRecord(e1, s);
    c->slot_timed[slot] = c->timing;
    return KA_OK;
}

int32_t ka_emit_device(ka_ctx* c, int32_t* d_out_len, int32_t* d_out_broker, void* stream, ka_status* st) {
    if (!c) return set_status(st, KA_ERR_NO_DEVICE);
    if (cudaSetDevice(c->device) != cudaSuccess) return set_status(st, KA_ERR_CUDA);
    if (!c->staged || !c->staged_block || c->staged_block->d.pl.rec_kind != 3 || !d_out_broker) return set_status(st, KA_ERR_BAD_ARG);
    const StageDesc& d = c->staged_block->d;
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    if ((rc = enq_emit_block(c, s, d, 0, 1, d_out_broker, d_out_len)) != KA_OK) return set_status(st, rc);
    if (c->timing) cudaEventRecord(c->ev[4], s);
    if ((rc = enq_flags_readback(c, s)) != KA_OK) return set_status(st, rc);
    if (c->timing) { cudaEventRecord(c->ev[5], s); c->ev_valid = true; }
    c->staged = false;
    c->last_was_staged = true;
    c->last_stream = s;
    c->pending_status = true;
    if (st) return finish_status(c, s, st);
    return KA_OK;
}

static int copy_counter_column(ka_ctx* c, int slot, int32_t* d_col, const int32_t* d_src, cudaStream_t s) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (slot < 0 || slot >= KA_MAX_SLOTS || (!d_col && !d_src)) return KA_ERR_BAD_ARG;
    KA_CUDA(cudaSetDevice(c->device));
    if (c->N <= 0) return KA_OK;
    int32_t* col = c->d_ctr8.as<int32_t>() + slot;
    if (d_col) KA_CUDA(cudaMemcpy2DAsync(d_col, 4, col, KA_MAX_SLOTS * 4, 4, (size_t)c->N, cudaMemcpyDeviceToDevice, s));
    else KA_CUDA(cudaMemcpy2DAsync(col, KA_MAX_SLOTS * 4, d_src, 4, 4, (size_t)c->N, cudaMemcpyDeviceToDevice, s));
    return KA_OK;
}

int32_t ka_ctx_export_counter_slot_device(ka_ctx* c, int32_t slot, int32_t* d_column, void* stream) {
    return copy_counter_column(c, slot, d_column, nullptr, (cudaStream_t)stream);
}

int32_t ka_ctx_import_counter_slot_device(ka_ctx* c, int32_t slot, const int32_t* d_column, void* stream) {
    return copy_counter_column(c, slot, nullptr, d_column, (cudaStream_t)stream);
}

int32_t ka_ctx_set_topic_base(ka_ctx* c, int32_t topic_base) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (topic_base < 0) return KA_ERR_BAD_ARG;
    c->topic_base = topic_base;
    return KA_OK;
}

int32_t ka_solve_dense(ka_ctx* c, int32_t T, const int32_t* topic_hash, int32_t P, int32_t RF,
                       const int32_t* cur_broker, int32_t desired_rf, int32_t out_stride,
                       int32_t* out_len, int32_t* out_broker, ka_status* st) {
    if (c) c->plan_valid = false;
    int rc = validate_dense(c, T, P, RF, desired_rf, out_stride, st);
    if (rc != KA_OK) return rc;
    if (cudaSetDevice(c->device) != cudaSuccess) return set_status(st, KA_ERR_CUDA);
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    cudaStream_t s = c->stream;
    const int64_t Q = (int64_t)T * P, R = Q * RF;
    if ((T > 0 && !topic_hash) || (R > 0 && !cur_broker) || (Q > 0 && !out_broker)) return set_status(st, KA_ERR_BAD_ARG);
    KA_CUDA(c->d_hash.reserve((size_t)std::max(T, 1) * 4));
    KA_CUDA(c->d_cur.reserve((size_t)std::max<int64_t>(R, 1) * 4));
    KA_CUDA(c->d_out.reserve((size_t)std::max<int64_t>(Q, 1) * out_stride * 4));
    KA_CUDA(c->d_out_len.reserve((size_t)std::max<int64_t>(Q, 1) * 4));
    c->last_part_id = nullptr;
    c->last_part_off = nullptr;
    c->staged = false;
    c->last_was_staged = false;
    rc = run_dense(c, s, T, P, RF, desired_rf, out_stride, topic_hash, cur_broker, c->d_hash.as<int32_t>(), c->d_cur.as<int32_t>(),
                   c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), out_broker, out_len, st);
    if (rc != KA_OK) { if (st && st->code != rc) set_status(st, rc); return rc; }
    keep_dense_rows(c, Q, c->d_cur.as<int32_t>(), RF, c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), out_stride, desired_rf);
    c->last_stream = s;
    c->pending_status = true;
    ka_status local;
    return finish_status(c, s, st ? st : &local);
}

}  // extern "C"

static int32_t solve_dense_json(ka_ctx* c, int32_t T, const int32_t* topic_hash, int32_t P, int32_t RF, const int32_t* cur_broker,
                                int32_t desired_rf, const char* names, const int64_t* name_off, char* json, int64_t json_cap,
                                int64_t* json_bytes, ka_status* st, bool changed_only) {
    const int S = std::max(std::max(RF, desired_rf), 1);
    if (json_bytes) *json_bytes = 0;
    if (c) c->plan_valid = false;
    int rc = validate_dense(c, T, P, RF, desired_rf, S, st);
    if (rc != KA_OK) return rc;
    const int64_t Q = (int64_t)T * P, R = Q * RF;
    if ((T > 0 && (!topic_hash || !names || !name_off)) || (R > 0 && !cur_broker) || !json || json_cap < KA_JSON_HEAD_LEN + KA_JSON_TAIL_LEN)
        return set_status(st, KA_ERR_BAD_ARG);
    const int64_t name_bytes = T > 0 ? name_off[T] : 0;
    for (int64_t i = 0; i < name_bytes; ++i) {  // org.json quote() would escape these: such names take the host emitter
        const unsigned char ch = (unsigned char)names[i];
        if (ch < 0x20 || ch == '"' || ch == '\\' || ch == '/') return set_status(st, KA_ERR_BAD_ARG, -1, -1, (int)ch);
    }
    if (cudaSetDevice(c->device) != cudaSuccess) return set_status(st, KA_ERR_CUDA);
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    cudaStream_t s = c->stream;
    KA_CUDA(c->d_hash.reserve((size_t)std::max(T, 1) * 4));
    KA_CUDA(c->d_cur.reserve((size_t)std::max<int64_t>(R, 1) * 4));
    KA_CUDA(c->d_out.reserve((size_t)std::max<int64_t>(Q, 1) * S * 4));
    KA_CUDA(c->d_out_len.reserve((size_t)std::max<int64_t>(Q, 1) * 4));
    KA_CUDA(c->d_json.reserve((size_t)json_cap));
    KA_CUDA(c->d_names.reserve((size_t)std::max<int64_t>(name_bytes, 1)));
    KA_CUDA(c->d_name_off.reserve((size_t)(T + 1) * 8));
    KA_CUDA(c->d_json_rowlen.reserve((size_t)std::max<int64_t>(Q, 1) * 4));
    KA_CUDA(c->d_json_blocksum.reserve((size_t)(Q / 256 + 2 * KA_MAX_CHAIN_EVENTS) * 4));
    KA_CUDA(c->d_json_state.reserve((2 + 2 * KA_MAX_CHAIN_EVENTS) * 8));
    KA_CUDA(cudaMemsetAsync(c->d_json_state.p, 0, (2 + 2 * KA_MAX_CHAIN_EVENTS) * 8, c->sj));
    if (name_bytes > 0) KA_CUDA(cudaMemcpyAsync(c->d_names.p, names, (size_t)name_bytes, cudaMemcpyHostToDevice, c->sj));
    if (T > 0) KA_CUDA(cudaMemcpyAsync(c->d_name_off.p, name_off, (size_t)(T + 1) * 8, cudaMemcpyHostToDevice, c->sj));
    JsonJob job{c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), S, 0};
    if (changed_only) {
        const size_t frag_blocks = (size_t)(Q / 256 + 2 * KA_MAX_CHAIN_EVENTS);
        KA_CUDA(c->d_sel.reserve((size_t)std::max<int64_t>(Q, 1) * 4));
        KA_CUDA(c->d_sel_mask.reserve(frag_blocks * 8 * 4));
        KA_CUDA(c->d_sel_blockcnt.reserve(frag_blocks * 4));
        KA_CUDA(c->d_sel_state.reserve((1 + 2 * KA_MAX_CHAIN_EVENTS) * 4));
        KA_CUDA(cudaMemsetAsync(c->d_sel_state.p, 0, (1 + 2 * KA_MAX_CHAIN_EVENTS) * 4, c->sj));
        job.changed_only = true;
        job.rows = KaRows{c->d_cur.as<int32_t>(), nullptr, RF, c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), S,
                          desired_rf >= 0 ? desired_rf : RF};
    }
    c->json_job = &job;
    c->last_part_id = nullptr;
    c->last_part_off = nullptr;
    c->staged = false;
    c->last_was_staged = false;
    rc = T > 0 && c->N > 0 ? run_dense(c, s, T, P, RF, desired_rf, S, topic_hash, cur_broker, c->d_hash.as<int32_t>(), c->d_cur.as<int32_t>(),
                                      c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), nullptr, nullptr, st)
                            : KA_ERR_BAD_ARG;
    c->json_job = nullptr;
    if (rc != KA_OK) { if (st && st->code != rc) set_status(st, rc); cudaStreamSynchronize(c->sj); return rc; }
    keep_dense_rows(c, Q, c->d_cur.as<int32_t>(), RF, c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), S, desired_rf);
    c->last_stream = s;
    c->pending_status = true;
    // every block is enqueued; stream the fragments out as their sizes become known (later blocks are still in the chains)
    int64_t total = 0;
    bool overflow = false;
    for (int k = 0; k < job.blocks; ++k) {
        KA_CUDA(cudaEventSynchronize(c->ev_json_scan[k]));
        const int64_t base = (int64_t)c->h_frag[2 * k], size = (int64_t)c->h_frag[2 * k + 1];
        if (base + size > json_cap) { overflow = true; break; }
        if (size > 0) KA_CUDA(cudaMemcpyAsync(json + base, c->d_json.as<char>() + base, (size_t)size, cudaMemcpyDeviceToHost, c->sj));
        total = base + size;
    }
    KA_CUDA(cudaStreamSynchronize(c->sj));
    ka_status local;
    rc = finish_status(c, s, st ? st : &local);
    if (rc == KA_OK && overflow) {
        c->plan_valid = false;
        return set_status(st, KA_ERR_LIMIT, -1, -1, (int)std::min<int64_t>(json_cap, INT_MAX));
    }
    if (json_bytes) *json_bytes = rc == KA_OK ? total : 0;
    return rc;
}

extern "C" {

int32_t ka_solve_dense_json(ka_ctx* c, int32_t T, const int32_t* topic_hash, int32_t P, int32_t RF, const int32_t* cur_broker,
                            int32_t desired_rf, const char* names, const int64_t* name_off, char* json, int64_t json_cap,
                            int64_t* json_bytes, ka_status* st) {
    return solve_dense_json(c, T, topic_hash, P, RF, cur_broker, desired_rf, names, name_off, json, json_cap, json_bytes, st, false);
}

int32_t ka_solve_dense_json_changed(ka_ctx* c, int32_t T, const int32_t* topic_hash, int32_t P, int32_t RF, const int32_t* cur_broker,
                                    int32_t desired_rf, const char* names, const int64_t* name_off, char* json, int64_t json_cap,
                                    int64_t* json_bytes, ka_status* st) {
    return solve_dense_json(c, T, topic_hash, P, RF, cur_broker, desired_rf, names, name_off, json, json_cap, json_bytes, st, true);
}

int32_t ka_solve(ka_ctx* c, int32_t T, const int32_t* topic_hash, const int64_t* part_off,
                 const int32_t* part_id, const int64_t* rep_off, const int32_t* cur_broker,
                 int32_t desired_rf, int32_t out_stride, int32_t* out_len, int32_t* out_broker,
                 ka_status* st) {
    set_status(st, KA_OK);
    if (!c) return set_status(st, KA_ERR_NO_DEVICE);
    c->plan_valid = false;
    if (T < 0 || (T > 0 && (!topic_hash || !part_off))) return set_status(st, KA_ERR_BAD_ARG);
    const int S = out_stride;
    if (S < 1 || S > KA_MAX_SLOTS) return set_status(st, KA_ERR_LIMIT, -1, -1, S);
    if (cudaSetDevice(c->device) != cudaSuccess) return set_status(st, KA_ERR_CUDA);
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    const int64_t Q = T > 0 ? part_off[T] : 0;
    if (Q < 0 || (T > 0 && part_off[0] != 0) || (Q > 0 && (!rep_off || !out_broker))) return set_status(st, KA_ERR_BAD_ARG);
    const int64_t R = Q > 0 ? rep_off[Q] : 0;
    if (R < 0 || (Q > 0 && rep_off[0] != 0) || (R > 0 && !cur_broker)) return set_status(st, KA_ERR_BAD_ARG);
    // host-side sizing scan: largest topic, largest current list, largest capacity (KAS:65-71)
    int Pmax = 0;
    int64_t capmax = 0, maxsz = 0;
    for (int t = 0; t < T; ++t) {
        const int64_t a = part_off[t], b = part_off[t + 1];
        if (b < a) return set_status(st, KA_ERR_BAD_ARG, t);
        const int64_t Pn = b - a;
        if (Pn > INT_MAX / 16) return set_status(st, KA_ERR_LIMIT, t, -1, (int)std::min<int64_t>(Pn, INT_MAX));
        Pmax = std::max<int>(Pmax, (int)Pn);
        int64_t rf_t = desired_rf;
        if (rf_t < 0 && Pn > 0) rf_t = rep_off[a + 1] - rep_off[a];
        if (rf_t > 0 && c->N > 0 && rf_t <= c->N) {
            capmax = std::max<int64_t>(capmax, (Pn * rf_t + c->N - 1) / c->N);
            if (rf_t > S) return set_status(st, KA_ERR_BAD_ARG, t, -1, S);
        }
    }
    for (int64_t g = 0; g < Q; ++g) {
        const int64_t sz = rep_off[g + 1] - rep_off[g];
        if (sz < 0) return set_status(st, KA_ERR_BAD_ARG);
        maxsz = std::max(maxsz, sz);
    }
    if (maxsz > S) return set_status(st, KA_ERR_BAD_ARG, -1, -1, S);

    cudaStream_t s = c->stream;
    KA_CUDA(c->d_hash.reserve((size_t)std::max(T, 1) * 4));
    KA_CUDA(c->d_part_off.reserve((size_t)(T + 1) * 8));
    KA_CUDA(c->d_rep_off.reserve((size_t)(Q + 1) * 8));
    KA_CUDA(c->d_cur.reserve((size_t)std::max<int64_t>(R, 1) * 4));
    KA_CUDA(c->d_out.reserve((size_t)std::max<int64_t>(Q, 1) * S * 4));
    KA_CUDA(c->d_out_len.reserve((size_t)std::max<int64_t>(Q, 1) * 4));
    c->host_out = nullptr;
    StageDesc d;
    d.T = T;
    d.Q = Q;
    d.d_hash = c->d_hash.as<int32_t>();
    d.d_part_off = c->d_part_off.as<int64_t>();
    d.d_rep_off = c->d_rep_off.as<int64_t>();
    d.d_cur = c->d_cur.as<int32_t>();
    d.desired_rf = desired_rf;
    d.S = S;
    d.Pmax = Pmax;
    d.capmax = capmax;
    c->staged = false;
    int rc = make_plan(c, Q, S, Pmax, capmax, true, d.pl, st);
    if (rc != KA_OK) return rc;
    if ((rc = reserve_scratch(c, Q, d.pl.rec_bytes, T, 1, true)) != KA_OK) return set_status(st, rc);
    c->last_stages = 1;
    if (c->timing) KA_CUDA(cudaEventRecord(c->ev[0], s));
    if (T > 0) {
        KA_CUDA(cudaMemcpyAsync(c->d_hash.p, topic_hash, (size_t)T * 4, cudaMemcpyHostToDevice, s));
        KA_CUDA(cudaMemcpyAsync(c->d_part_off.p, part_off, (size_t)(T + 1) * 8, cudaMemcpyHostToDevice, s));
    }
    if (Q > 0) KA_CUDA(cudaMemcpyAsync(c->d_rep_off.p, rep_off, (size_t)(Q + 1) * 8, cudaMemcpyHostToDevice, s));
    if (R > 0) KA_CUDA(cudaMemcpyAsync(c->d_cur.p, cur_broker, (size_t)R * 4, cudaMemcpyHostToDevice, s));
    if ((rc = reset_flags(c, s)) != KA_OK) return set_status(st, rc);
    if (c->timing) KA_CUDA(cudaEventRecord(c->ev[1], s));
    c->last_part_id = part_id;
    c->last_part_off = part_off;
    c->last_was_staged = false;
    c->ev_mark = c->timing ? c->ev[2] : nullptr;
    rc = enq_stage(c, s, d);
    c->ev_mark = nullptr;
    if (rc != KA_OK) return set_status(st, rc);
    if (c->timing) KA_CUDA(cudaEventRecord(c->ev[3], s));
    if ((rc = chain_fork(c, s)) != KA_OK) return set_status(st, rc);
    if ((rc = enq_order_emit(c, s, d, c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), 1)) != KA_OK) return set_status(st, rc);
    if (c->timing) KA_CUDA(cudaEventRecord(c->ev[4], s));
    if (Q > 0 && c->N > 0) {
        KA_CUDA(cudaMemcpyAsync(out_broker, c->d_out.p, (size_t)Q * S * 4, cudaMemcpyDeviceToHost, s));
        if (out_len) KA_CUDA(cudaMemcpyAsync(out_len, c->d_out_len.p, (size_t)Q * 4, cudaMemcpyDeviceToHost, s));
    }
    if ((rc = enq_flags_readback(c, s)) != KA_OK) return set_status(st, rc);
    if (c->timing) { KA_CUDA(cudaEventRecord(c->ev[5], s)); c->ev_valid = true; }
    c->plan_rows = KaRows{c->d_cur.as<int32_t>(), c->d_rep_off.as<int64_t>(), 0, c->d_out.as<int32_t>(), c->d_out_len.as<int32_t>(), S,
                          desired_rf};
    c->plan_Q = Q;
    c->plan_valid = true;
    c->last_stream = s;
    c->pending_status = true;
    ka_status local;
    rc = finish_status(c, s, st ? st : &local);
    c->last_part_id = nullptr;
    c->last_part_off = nullptr;
    return rc;
}

int32_t ka_ctx_set_report_brokers(ka_ctx* c, int32_t M, const int32_t* ids) {
    if (!c) return KA_ERR_NO_DEVICE;
    if (M < 0 || M > 65534 || (M > 0 && !ids)) return KA_ERR_BAD_ARG;   // bucket M ("other") must stay below KA_DEAD
    for (int i = 1; i < M; ++i)
        if (ids[i] <= ids[i - 1]) return KA_ERR_BAD_ARG;   // ascending, distinct
    KA_CUDA(cudaSetDevice(c->device));
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    c->rep_M = 0;
    if (M == 0) return KA_OK;
    const IdLut lut = make_id_lut(M, ids);
    if (!lut.lut.empty()) {
        KA_CUDA(c->d_rep_lut.reserve(lut.lut.size() * 2));
        KA_CUDA(cudaMemcpy(c->d_rep_lut.p, lut.lut.data(), lut.lut.size() * 2, cudaMemcpyHostToDevice));
    }
    KA_CUDA(c->d_rep_ids.reserve((size_t)M * 4));
    KA_CUDA(cudaMemcpy(c->d_rep_ids.p, ids, (size_t)M * 4, cudaMemcpyHostToDevice));
    c->rep_mode = lut.mode;
    c->rep_min_id = lut.min_id;
    c->rep_range = lut.range;
    c->rep_M = M;
    return KA_OK;
}

int32_t ka_plan_last(ka_ctx* c, uint8_t* row_class, uint32_t* broker_stats, ka_plan_totals* totals) {
    if (!c) return KA_ERR_NO_DEVICE;
    KA_CUDA(cudaSetDevice(c->device));
    if (c->pending_status) finish_status(c, c->last_stream, nullptr);
    if (!c->plan_valid || c->last.code != KA_OK) return KA_ERR_BAD_ARG;
    KaPlanParams p{};
    p.rows = c->plan_rows;
    p.Q = c->plan_Q;
    if (c->rep_M > 0) {
        p.lut_mode = c->rep_mode;
        p.min_id = c->rep_min_id;
        p.range = c->rep_range;
        p.glut = c->d_rep_lut.as<uint16_t>();
        p.broker_id = c->d_rep_ids.as<int32_t>();
        p.N = c->rep_M;
    } else {   // the live broker table, through the lookup kernel A uses
        p.lut_mode = c->lut_mode;
        p.min_id = c->min_id;
        p.range = c->range;
        p.glut = c->lut_mode == KA_LUT_SMEM ? c->d_blob.as<uint16_t>() + c->lut_off : c->d_glut.as<uint16_t>();
        p.broker_id = c->d_broker_id.as<int32_t>();
        p.N = c->N;
    }
    p.lut_bytes = p.lut_mode == KA_LUT_SMEM ? (int)align16((size_t)p.range * 2) : 0;
    const size_t ncol = (size_t)(p.N + 1) * KA_PLAN_COLS;
    const bool shist = p.lut_bytes + ncol * 4 <= KA_PLAN_SMEM_BUDGET;
    const size_t smem = p.lut_bytes + (shist ? ncol * 4 : 0);
    cudaStream_t s = c->stream;
    KA_CUDA(c->d_plan_tot.reserve(KA_PLAN_TOTALS * 8));
    KA_CUDA(c->d_plan_stats.reserve(ncol * 4));
    KA_CUDA(cudaMemsetAsync(c->d_plan_tot.p, 0, KA_PLAN_TOTALS * 8, s));
    KA_CUDA(cudaMemsetAsync(c->d_plan_stats.p, 0, ncol * 4, s));
    if (row_class && p.Q > 0) {
        KA_CUDA(c->d_plan_class.reserve((size_t)p.Q));
        p.row_class = c->d_plan_class.as<uint8_t>();
    }
    p.stats = c->d_plan_stats.as<uint32_t>();
    p.totals = c->d_plan_tot.as<unsigned long long>();
    if (p.Q > 0) {
        const bool wide = p.rows.S > 3;
        KA_CUDA(wide ? (shist ? launch_plan<8, true>(c, s, p, smem) : launch_plan<8, false>(c, s, p, smem))
                     : (shist ? launch_plan<3, true>(c, s, p, smem) : launch_plan<3, false>(c, s, p, smem)));
        c->launches++;
    }
    int64_t tot[KA_PLAN_TOTALS];
    KA_CUDA(cudaMemcpyAsync(tot, c->d_plan_tot.p, sizeof(tot), cudaMemcpyDeviceToHost, s));
    if (broker_stats) KA_CUDA(cudaMemcpyAsync(broker_stats, c->d_plan_stats.p, ncol * 4, cudaMemcpyDeviceToHost, s));
    if (p.row_class) KA_CUDA(cudaMemcpyAsync(row_class, p.row_class, (size_t)p.Q, cudaMemcpyDeviceToHost, s));
    KA_CUDA(cudaStreamSynchronize(s));
    if (totals) *totals = ka_plan_totals{tot[0], tot[1], tot[2], tot[3], tot[4], tot[5]};
    return KA_OK;
}

}  // extern "C"
