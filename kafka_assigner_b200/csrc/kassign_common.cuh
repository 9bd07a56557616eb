// kassign_common.cuh — shared definitions of the sm_100a kernels of the kafka-assigner hot path.
//
// Reference being replaced (SURVEY.md §8a; KAS = KafkaAssignmentStrategy.java, KTA = KafkaTopicAssigner.java):
//   kassign_stage.cuh  ka_sticky_spread_kernel  KTA:49-69 (RF inference/validation), KAS:65-71 (capacity), KAS:73-99
//                                               (node/rack table), KAS:101-131 (sticky fill), KAS:133-160 (orphans),
//                                               KAS:162-200 (rotated first-fit spread), KAS:205-214 (ascending lists)
//                                               + the conflict levels the leader-order kernel is scheduled by
//   kassign_order.cuh  ka_order_levels_kernel   KAS:202-239 + PreferenceListOrderTracker KAS:244-302 against the
//                                               cross-topic Context.counter (KAS:360-369, KTA:19-23)
//                      ka_emit3_kernel          list positions -> ordered broker ids (KAS:229-235 output lists)
//
// Everything is integer indexing: no tensor cores. Tables and record streams are staged into shared memory with TMA
// bulk copies (cp.async.bulk + mbarrier); decisions that depend on the reference's visit order are taken with warp
// ballots / match / shuffles or under a barrier-separated schedule — never by an atomics race.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define KA_MAX_SLOTS 8      // max replicas per partition row (out_stride) on the fast paths
#define KA_DEAD 0xFFFFu     // "broker not in the live set" marker in 16-bit index space
#define KA_FULL 0xFFFFFFFFu

// Error codes (mirror include/kassign.h)
#define KA_E_RF_MISMATCH 1
#define KA_E_RF_NOT_POSITIVE 2
#define KA_E_RF_GT_BROKERS 3
#define KA_E_UNASSIGNABLE 4
#define KA_E_HASH_INDEX 5

enum { KA_LUT_SMEM = 0, KA_LUT_GLOBAL = 1, KA_LUT_BSEARCH = 2 };

// ------------------------------------------------------------------------------------------------
// Partition records: what kernel A hands to the leader-order kernel, in SCHEDULE order (topic by topic; inside a
// topic by conflict level, then partition ascending). Broker indices are positions in the ascending live-id table.
//   rows of <= 3 replicas  uint4 {a0, a1, a2, f}: a_j = (index of the broker at position j of the slot-0 scan order of
//                          KAS:267, i.e. ascending list position i sits at j = (i + |hash| % len) % len) << 2 = byte offset
//                          of that broker's counter in a 4-byte column; unused slots = the dummy broker N;
//                          f = len[0:2) | e01[2] | e02[3] | e12[4] | first-of-level[7], e_pq = tie-break of the slot-1 scan over the pair
//                          (p, q) left when the third position took slot 0 (see kassign_stage.cuh / kassign_order.cuh).
//                          The slot-0 chain rewrites it as {op, oq, len | e << 2, o0} (remaining pair in scan order, its
//                          tie-break, the slot-0 broker); the slot-1 chain as the ordered list {o0, o1, o2, len | e << 2}.
//   rows of 4..8           2 x uint4 : {idx0|idx1<<16, idx2|idx3<<16, idx4|idx5<<16, idx6|idx7<<16}, {meta32, row, 0, 0}
//                          meta32 = len[0:4) | rotations for k = 2..8 (ka_rot_bits), row = block-relative output row
// ------------------------------------------------------------------------------------------------


// ------------------------------------------------------------------------------------------------
// small PTX helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ka_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void ka_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ka_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void ka_fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void ka_fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void ka_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ka_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ka_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(ka_smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// TMA bulk copy global -> shared (non-tensor form). bytes % 16 == 0, both addresses 16B aligned.
__device__ __forceinline__ void ka_tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     ka_smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(ka_smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ int4 ka_ldg_stream_v4(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// Broker id -> index in an ascending id table, KA_DEAD when absent. The host picks the mode from the id range when it builds
// the table (make_id_lut in kassign.cu): a 16-bit LUT in shared memory (`lut`), the same LUT in global memory (t.glut), or a
// binary search over the ids themselves (t.broker_id[0 .. t.N)). T = any parameter block with those fields.
template <typename T>
__device__ __forceinline__ uint32_t ka_id_index(int id, const uint16_t* lut, const T& t) {
    if (t.lut_mode == KA_LUT_SMEM) {
        uint32_t off = (uint32_t)id - (uint32_t)t.min_id;
        return off < t.range ? (uint32_t)lut[off] : KA_DEAD;
    } else if (t.lut_mode == KA_LUT_GLOBAL) {
        uint32_t off = (uint32_t)id - (uint32_t)t.min_id;
        return off < t.range ? (uint32_t)__ldg(&t.glut[off]) : KA_DEAD;
    } else {
        int lo = 0, hi = t.N - 1;
        while (lo <= hi) {
            int mid = (lo + hi) >> 1;
            int v = __ldg(&t.broker_id[mid]);
            if (v == id) return (uint32_t)mid;
            if (v < id) lo = mid + 1; else hi = mid - 1;
        }
        return KA_DEAD;
    }
}

__device__ __forceinline__ uint32_t ka_lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Rotation bits of one topic: (|hash| % k) for k = 2..8 packed above the 4-bit length (KAS:190 applied
// to the remaining-set sizes of KAS:267). Layout: len[0:4) k2[4] k3[5:7) k4[7:9) k5[9:12) k6[12:15) k7[15:18) k8[18:21)
__device__ __forceinline__ uint32_t ka_rot_bits(uint32_t habs) {
    return ((habs % 2u) << 4) | ((habs % 3u) << 5) | ((habs % 4u) << 7) | ((habs % 5u) << 9) | ((habs % 6u) << 12) |
           ((habs % 7u) << 15) | ((habs % 8u) << 18);
}
template <int RS>
__device__ __forceinline__ int ka_rot_of(uint32_t meta, int k) {
    // k in [1,RS]; select chain instead of a table so nothing lands in local memory
    int s = 0;
    if (k == 2) s = (meta >> 4) & 1u;
    if (k == 3) s = (meta >> 5) & 3u;
    if (k == 4) s = (meta >> 7) & 3u;
    if (RS > 4) {
        if (k == 5) s = (meta >> 9) & 7u;
        if (k == 6) s = (meta >> 12) & 7u;
        if (k == 7) s = (meta >> 15) & 7u;
        if (k == 8) s = (meta >> 18) & 7u;
    }
    return s;
}
