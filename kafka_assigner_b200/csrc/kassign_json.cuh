// kassign_json.cuh — the reassignment JSON of KafkaAssignmentGenerator.printLeastDisruptiveReassignment (KAG:169-186) built
// on the device from the solved rows, so that only TEXT crosses PCIe and it can stream out block by block while later topic
// blocks are still in the leader-order chains.
//
//   {"partitions":[{"partition":P,"replicas":[a,b,c],"topic":"name"},...],"version":1}
//
// org.json 20131018 prints object keys in java.util.HashMap iteration order (SURVEY.md §3.4): "partitions" before "version",
// "partition" / "replicas" / "topic" inside a record — predicted, unverified without a JVM; the order lives only in
// ka_json_row_len / ka_json_row_put below (and in kassign_host.hpp::newAssignmentJson for the host emitter).
// Topic names must not need JSON escaping (Kafka topic names are [a-zA-Z0-9._-]); the host checks before choosing this path.
#pragma once
#include "kassign_common.cuh"

struct KaJsonParams {
    uint32_t Q;                 // rows of this fragment
    uint32_t row0;              // index of the fragment's first row in the whole run (row 0 has no leading comma)
    int P;                      // dense shape: partition id = row % P, topic = topic0 + row / P
    int topic0;
    const int64_t* name_off;    // [T+1] byte offsets into names
    const char* names;          // concatenated topic names (UTF-8, no escapes needed)
    const int32_t* out;         // [Q][S] broker ids, leader first
    const int32_t* out_len;     // [Q]
    int S;
    uint32_t* rowlen;           // [Q] scratch
    uint32_t* blocksum;         // [ceil(Q / 256)] scratch
    unsigned long long* total;  // device scalar: bytes written so far (header included); advanced by this fragment
    unsigned long long* frag;   // [2] out: {first byte, byte count} of this fragment (the header / trailer included)
    char* json;
    unsigned long long cap;     // bytes of `json`: a fragment that would end beyond it is measured but NOT written
    int first, last;            // write the header before / the trailer after this fragment
    // changed-rows-only text (IDX kernels): the fragment's rows are sel[0 .. sel_state[1]) (fragment-relative, ascending);
    // sel_state[0] = rows emitted by earlier fragments, which decides the leading comma
    const uint32_t* sel;
    const uint32_t* sel_state;
};

#define KA_JSON_HEAD "{\"partitions\":["
#define KA_JSON_TAIL "],\"version\":1}"
#define KA_JSON_HEAD_LEN 15
#define KA_JSON_TAIL_LEN 14

__device__ __forceinline__ uint32_t ka_ndigits(int32_t v) {  // characters of Integer.toString(v)
    uint32_t u = v < 0 ? 0u - (uint32_t)v : (uint32_t)v, n = v < 0 ? 2u : 1u;
    while (u >= 10u) { u /= 10u; ++n; }
    return n;
}
__device__ __forceinline__ char* ka_put_int(char* p, int32_t v) {
    char tmp[11];
    uint32_t u = v < 0 ? 0u - (uint32_t)v : (uint32_t)v;
    int n = 0;
    do { tmp[n++] = (char)('0' + u % 10u); u /= 10u; } while (u);
    if (v < 0) *p++ = '-';
    while (n) *p++ = tmp[--n];
    return p;
}
__device__ __forceinline__ char* ka_put_str(char* p, const char* s, int n) {
    for (int i = 0; i < n; ++i) p[i] = s[i];
    return p + n;
}

// rows this fragment writes, and whether its q-th one is preceded by a comma (it is not the first row of the whole text)
template <bool IDX> __device__ __forceinline__ uint32_t ka_json_rows(const KaJsonParams& p) { return IDX ? p.sel_state[1] : p.Q; }
template <bool IDX> __device__ __forceinline__ bool ka_json_comma(const KaJsonParams& p, uint32_t q) {
    return IDX ? p.sel_state[0] + q > 0 : p.row0 + q > 0;
}

template <bool IDX>
__device__ __forceinline__ uint32_t ka_json_row_len(const KaJsonParams& p, uint32_t i) {
    const uint32_t q = IDX ? p.sel[i] : i;
    const int t = p.topic0 + (int)(q / (uint32_t)p.P), part = (int)(q % (uint32_t)p.P);
    const int len = p.out_len[q];
    uint32_t n = (ka_json_comma<IDX>(p, i) ? 1u : 0u) + 13u + ka_ndigits(part) + 13u + 11u + (uint32_t)(p.name_off[t + 1] - p.name_off[t]) + 2u;
    for (int i = 0; i < len; ++i) n += ka_ndigits(p.out[(size_t)q * p.S + i]) + (i ? 1u : 0u);
    return n;
}
template <bool IDX>
__device__ __forceinline__ void ka_json_row_put(const KaJsonParams& p, uint32_t i, char* w) {
    const uint32_t q = IDX ? p.sel[i] : i;
    const int t = p.topic0 + (int)(q / (uint32_t)p.P), part = (int)(q % (uint32_t)p.P);
    const int len = p.out_len[q];
    if (ka_json_comma<IDX>(p, i)) *w++ = ',';
    w = ka_put_str(w, "{\"partition\":", 13);
    w = ka_put_int(w, part);
    w = ka_put_str(w, ",\"replicas\":[", 13);
    for (int i = 0; i < len; ++i) {
        if (i) *w++ = ',';
        w = ka_put_int(w, p.out[(size_t)q * p.S + i]);
    }
    w = ka_put_str(w, "],\"topic\":\"", 11);
    w = ka_put_str(w, p.names + p.name_off[t], (int)(p.name_off[t + 1] - p.name_off[t]));
    ka_put_str(w, "\"}", 2);
}

// pass 1: text length of every row + per-block sums. IDX: the grid covers every row of the fragment, the blocks beyond the
// selected rows (known only on the device) write zero sums.
template <bool IDX>
__global__ void __launch_bounds__(256) ka_json_len_kernel(const KaJsonParams p) {
    __shared__ uint32_t wsum[8];
    const uint32_t q = blockIdx.x * 256u + threadIdx.x;
    const uint32_t nq = ka_json_rows<IDX>(p);
    uint32_t n = q < nq ? ka_json_row_len<IDX>(p, q) : 0u;
    if (q < nq) p.rowlen[q] = n;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(KA_FULL, n, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (int i = 0; i < 8; ++i) s += wsum[i];
        p.blocksum[blockIdx.x] = s;
    }
}

// pass 2 (one CTA): exclusive scan of the block sums, placed after the bytes written so far; reserves header / trailer
__global__ void __launch_bounds__(1024) ka_json_scan_kernel(const KaJsonParams p, int nblocks) {
    __shared__ unsigned long long wtot[32];
    __shared__ unsigned long long carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = *p.total + (p.first ? KA_JSON_HEAD_LEN : 0);
    __syncthreads();
    const unsigned long long base0 = *p.total;
    for (int b0 = 0; b0 < nblocks; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const unsigned long long v = b < nblocks ? p.blocksum[b] : 0ull;
        unsigned long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(KA_FULL, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wtot[warp] = x;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = wtot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long y = __shfl_up_sync(KA_FULL, w, o);
                if (lane >= o) w += y;
            }
            wtot[lane] = w;
        }
        __syncthreads();
        const unsigned long long base = carry + (warp > 0 ? wtot[warp - 1] : 0ull);
        if (b < nblocks) p.blocksum[b] = (uint32_t)(base + x - v - base0);   // relative to the fragment start (a fragment is < 4 GiB)
        __syncthreads();
        if (threadIdx.x == 1023) carry = base + x;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const unsigned long long end = carry + (p.last ? KA_JSON_TAIL_LEN : 0);
        p.frag[0] = base0;
        p.frag[1] = end - base0;
        *p.total = end;
    }
}

// pass 3: every row writes its text at its final position. The 256 rows of a block are assembled in shared memory (at the
// same 16-byte phase as their destination) and copied out with coalesced 16-byte stores; blocks whose text does not fit
// (very long topic names) write straight to global memory.
#define KA_JSON_SMEM_BYTES (64 * 1024)
template <bool IDX>
__global__ void __launch_bounds__(256) ka_json_write_kernel(const KaJsonParams p) {
    extern __shared__ __align__(16) unsigned char ka_jsmem[];
    __shared__ uint32_t wsum[8];
    if (p.frag[0] + p.frag[1] > p.cap) return;   // caller's buffer too small (uniform: the host reports KA_ERR_LIMIT)
    const uint32_t q = blockIdx.x * 256u + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t nq = ka_json_rows<IDX>(p);
    const uint32_t n = q < nq ? p.rowlen[q] : 0u;
    uint32_t x = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(KA_FULL, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    uint32_t woff = 0, bt = 0;
    for (int i = 0; i < 8; ++i) { if (i < warp) woff += wsum[i]; bt += wsum[i]; }
    char* frag = p.json + p.frag[0];
    char* dst = frag + p.blocksum[blockIdx.x];                 // this block's text
    const uint32_t loc = woff + x - n;                           // my row inside it
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u);
    if (mis + bt <= KA_JSON_SMEM_BYTES) {
        char* stage = reinterpret_cast<char*>(ka_jsmem) + mis;
        if (q < nq) ka_json_row_put<IDX>(p, q, stage + loc);
        __syncthreads();
        const uint32_t head = min(bt, (16u - mis) & 15u);       // bytes up to the first 16-byte boundary of dst
        for (uint32_t i = threadIdx.x; i < head; i += 256) dst[i] = stage[i];
        const uint32_t body = (bt - head) >> 4;
        const uint4* s4 = reinterpret_cast<const uint4*>(stage + head);
        uint4* d4 = reinterpret_cast<uint4*>(dst + head);
        for (uint32_t i = threadIdx.x; i < body; i += 256) d4[i] = s4[i];
        for (uint32_t i = head + (body << 4) + threadIdx.x; i < bt; i += 256) dst[i] = stage[i];
    } else if (q < nq) {
        ka_json_row_put<IDX>(p, q, dst + loc);
    }
    if (q == 0 && p.first) ka_put_str(frag, KA_JSON_HEAD, KA_JSON_HEAD_LEN);
    if (q == 0 && p.last) ka_put_str(frag + p.frag[1] - KA_JSON_TAIL_LEN, KA_JSON_TAIL, KA_JSON_TAIL_LEN);
}
