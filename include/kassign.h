/* kassign.h — C ABI of libkassign.so, the B200-native drop-in for ONE path of SiftScience/kafka-assigner:
 *
 *   KafkaTopicAssigner.generateAssignment            (reference: KafkaTopicAssigner.java:42-72,  "KTA")
 *     -> KafkaAssignmentStrategy.getRackAwareAssignment (KafkaAssignmentStrategy.java:40-63,      "KAS")
 *   as driven by the per-topic loop of KafkaAssignmentGenerator.printLeastDisruptiveReassignment
 *   (KafkaAssignmentGenerator.java:172-184, "KAG").
 *
 * Plain pointers and sizes only; no torch / C++ types. A Java maintainer binds these through JNI
 * (see INTEGRATION.md for the stub), a C++ host through kassign_host.hpp, Python through ctypes.
 *
 * The reference's per-topic method becomes a BATCH call: one ka_solve() == the whole KAG:173-184 loop
 * (T topics in order through ONE Context); a batch of 1 == one generateAssignment() call.
 *
 * All compute runs in hand-written sm_100a CUDA kernels. There is NO CPU fallback: without a usable
 * CUDA device ka_ctx_create() returns NULL and every entry point fails with KA_ERR_NO_DEVICE.
 */
#ifndef KASSIGN_H
#define KASSIGN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* One ka_ctx == one `KafkaTopicAssigner` instance == one `KafkaAssignmentStrategy.Context`
 * (KTA:19-23, KAS:360-369): it owns the cross-topic leader-preference counters counter[broker][slot],
 * keyed by BROKER ID (so successive calls may use different broker sets, as the reference's tests do),
 * plus the device scratch. One in-flight call per ctx (the reference is single-threaded, KAS:361-368). */
typedef struct ka_ctx ka_ctx;

/* Error report. `code` > 0 are the reference's exceptions; `topic_index` is the LOWEST failing topic in
 * loop order (KAG:173 aborts at the first throw) and, inside it, the first failure in the reference's own
 * evaluation order. After code != 0 the ctx counters are undefined (the reference process would be dead). */
typedef struct ka_status {
    int32_t code;
    int32_t topic_index; /* -1 when not topic-specific */
    int32_t partition;   /* partition id (from part_id, or the ordinal when part_id == NULL); -1 if n/a */
    int32_t a;           /* operand 1 of the message (see codes) */
    int32_t b;           /* operand 2 */
} ka_status;

enum {
    KA_OK = 0,
    /* IllegalStateException "Topic T has partition P with unexpected replication factor K"  KTA:58-60; a=K */
    KA_ERR_RF_MISMATCH = 1,
    /* IllegalStateException "Topic T does not have a positive replication factor!"           KTA:65-66 */
    KA_ERR_RF_NOT_POSITIVE = 2,
    /* IllegalStateException "Topic T has a higher replication factor (RF) than available brokers!" KTA:67-69; a=RF */
    KA_ERR_RF_GT_BROKERS = 3,
    /* IllegalStateException "Partition P could not be fully assigned!"                        KAS:183-184 */
    KA_ERR_UNASSIGNABLE = 4,
    /* ArrayIndexOutOfBoundsException from getNodeProcessingOrder when topic.hashCode()==Integer.MIN_VALUE
     * (Math.abs stays negative)                                                               KAS:190-192; a=index, b=length */
    KA_ERR_HASH_INDEX = 5,
    /* library-side failures (no reference counterpart) */
    KA_ERR_BAD_ARG = -1,
    KA_ERR_CUDA = -2,
    KA_ERR_NO_DEVICE = -3,
    KA_ERR_LIMIT = -4 /* a size beyond what the kernels' shared-memory layout supports; a=offending value */
};

/* ---- lifetime ---------------------------------------------------------------------------------- */

/* `new KafkaTopicAssigner()` (KTA:21-23). device = CUDA ordinal. NULL if no CUDA device/driver. */
ka_ctx* ka_ctx_create(int32_t device);
void ka_ctx_destroy(ka_ctx* ctx);
/* Drop all counters: a fresh Context (KAS:365-368). */
int32_t ka_ctx_reset(ka_ctx* ctx);

/* ---- the broker table ---------------------------------------------------------------------------
 * `brokers` + `rackAssignment` of generateAssignment (KTA:43-44) — the same for every topic of a run
 * (KAG:150-151,175-176) — uploaded once per run.
 *   broker_id[N]   strictly ascending live broker ids (the TreeMap order of KAS:78)
 *   broker_rack[N] dense rack index per broker, 0 <= idx < N. Brokers without a rack get an index no
 *                  other broker uses unless their decimal id equals a real rack's NAME (the string-key
 *                  quirk of KAS:82-94) — ka_rack_indices() below does that mapping from strings.
 * Counters of brokers that leave the set are retained (keyed by id) and come back if the id returns. */
int32_t ka_ctx_set_brokers(ka_ctx* ctx, int32_t N, const int32_t* broker_id, const int32_t* broker_rack);

/* Helper for the string side of KAS:81-94: rack_name[i] (NUL-terminated UTF-8, or NULL = "no rack
 * defined for this broker") -> dense indices with the id.toString() fallback and its collision quirk. */
int32_t ka_rack_indices(int32_t N, const int32_t* broker_id, const char* const* rack_name, int32_t* broker_rack);

/* java.lang.String.hashCode of a UTF-8 encoded topic name (UTF-16 code units, int32 wrap) — KAS:190. */
int32_t ka_java_string_hash(const char* utf8);

/* ---- the solve ----------------------------------------------------------------------------------
 * General (ragged) form, HOST buffers; copies in, runs the kernels, copies out, synchronises.
 *   T                topics, solved in index order through this ctx (KAG:173)
 *   topic_hash[T]    String.hashCode of each topic name
 *   part_off[T+1]    partitions of topic t are rows part_off[t] .. part_off[t+1]-1
 *   part_id[ΣP]      partition ids, ascending within a topic (TreeMap order, KAS:107-110); NULL = 0..P-1.
 *                    Only used to report ka_status.partition; the solver works on ordinals.
 *   rep_off[ΣP+1]    current replica list of row g is cur_broker[rep_off[g] .. rep_off[g+1]-1] (leader first)
 *   desired_rf       --desired_replication_factor; -1 = keep (KTA:49,55-61)
 *   out_stride       slots per output row; must be >= max(list length, target RF) over all rows
 *   out_len[ΣP]      length of each new replica list (may be NULL)
 *   out_broker[ΣP*out_stride]  new replica lists, leader first, in row order; unused slots = -1
 * Returns st->code. */
int32_t ka_solve(ka_ctx* ctx, int32_t T, const int32_t* topic_hash, const int64_t* part_off,
                 const int32_t* part_id, const int64_t* rep_off, const int32_t* cur_broker,
                 int32_t desired_rf, int32_t out_stride, int32_t* out_len, int32_t* out_broker,
                 ka_status* st);

/* Dense form (every topic P partitions 0..P-1, every list RF long): cur[T][P][RF] -> out[T][P][out_stride]. */
int32_t ka_solve_dense(ka_ctx* ctx, int32_t T, const int32_t* topic_hash, int32_t P, int32_t RF,
                       const int32_t* cur_broker, int32_t desired_rf, int32_t out_stride,
                       int32_t* out_len, int32_t* out_broker, ka_status* st);

/* Dense solve + the reference's JSON emitter (KAG:169-186) in one call: the rows never leave the device, only the TEXT
 *   {"partitions":[{"partition":p,"replicas":[..],"topic":"name"},...],"version":1}
 * crosses PCIe, streamed block by block while later topic blocks are still being ordered. names = the T topic names
 * concatenated (UTF-8, none needing JSON escapes — else KA_ERR_BAD_ARG: use the host emitter), name_off[T+1] their offsets;
 * json = host buffer of json_cap bytes (pinned for full PCIe speed; KA_ERR_LIMIT if too small: 64 + sum over rows of
 * (50 + 12*out_stride + name length) always suffices); *json_bytes = length of the text (not NUL-terminated). */
int32_t ka_solve_dense_json(ka_ctx* ctx, int32_t T, const int32_t* topic_hash, int32_t P, int32_t RF,
                            const int32_t* cur_broker, int32_t desired_rf, const char* names, const int64_t* name_off,
                            char* json, int64_t json_cap, int64_t* json_bytes, ka_status* st);

/* Same as ka_solve_dense_json, but the text lists only the rows the solve changes (movement class != UNCHANGED, see
 * ka_plan_last below), in the same order and format: {"partitions":[],"version":1} when nothing changes.
 * kafka-reassign-partitions accepts any subset of the partitions, so this is the reassignment to apply. Every finished
 * block of rows is classified and compacted on the device; only the changed rows' text crosses PCIe. The json_cap rules
 * and KA_ERR_LIMIT are those of ka_solve_dense_json. */
int32_t ka_solve_dense_json_changed(ka_ctx* ctx, int32_t T, const int32_t* topic_hash, int32_t P, int32_t RF,
                                    const int32_t* cur_broker, int32_t desired_rf, const char* names, const int64_t* name_off,
                                    char* json, int64_t json_cap, int64_t* json_bytes, ka_status* st);

/* Dense form on DEVICE buffers (d_* are device pointers on the ctx's device; d_out_len may be NULL),
 * enqueued on `stream` (a cudaStream_t, NULL = the legacy default stream) — inputs already resident in
 * HBM, outputs left in HBM. If st != NULL the call synchronises the stream and fills *st; with
 * st == NULL it is fully asynchronous and the status is fetched later with ka_last_status(). */
int32_t ka_solve_dense_device(ka_ctx* ctx, int32_t T, const int32_t* d_topic_hash, int32_t P, int32_t RF,
                              const int32_t* d_cur_broker, int32_t desired_rf, int32_t out_stride,
                              int32_t* d_out_len, int32_t* d_out_broker, void* stream, ka_status* st);

/* The same solve split at the only point where topics stop being independent, for topic-sharded
 * multi-GPU runs (SURVEY.md §8e):
 *   ka_stage_dense_device  capacity, sticky fill, orphan spread (KAS:65-200) + per-broker histograms —
 *                          touches no Context state, so every GPU stages its own topic block concurrently;
 *   ka_order_device        leader-preference ordering (KAS:202-239) of the staged block against THIS ctx's
 *                          counters — a serial chain over all topics of the run, so rank g calls it after
 *                          importing the counters rank g-1 exported (ka_ctx_*_counters_device).
 * ka_solve_dense_device == stage + order. */
int32_t ka_stage_dense_device(ka_ctx* ctx, int32_t T, const int32_t* d_topic_hash, int32_t P, int32_t RF,
                              const int32_t* d_cur_broker, int32_t desired_rf, int32_t out_stride, void* stream);
int32_t ka_order_device(ka_ctx* ctx, int32_t* d_out_len, int32_t* d_out_broker, void* stream, ka_status* st);
/* Rows of <= 3 replicas are ordered by TWO independent chains: slot r reads and bumps only counter[.][r] (KAS:263-278 with
 * replicaId = r), slot 1 needs the slot-0 winners but slot 0 never waits for slot 1, and counter[.][2] is write-only
 * (a commutative sum added by the emit). A topic-sharded run therefore hands counter[.][0] to the next rank as soon as its
 * slot-0 chain is done, then counter[.][1]:
 *   ka_staged_slot_chains()   2 if the staged block is ordered by per-slot chains (all rows <= 3), else 0 (use ka_order_device)
 *   ka_order_slot_device()    the slot-0 (slot = 0) or slot-1 (slot = 1) chain of the staged block; slot 1 after slot 0
 *   ka_emit_device()          ordered records -> d_out_broker / d_out_len, adds counter[.][2]; ends the staged solve
 *   ka_ctx_{export,import}_counter_slot_device()  one counter column, d_column = N int32 on the device
 * ka_order_device == slot 0 (internal stream) overlapped with slot 1 + emit, sub-block by sub-block. */
int32_t ka_staged_slot_chains(ka_ctx* ctx);
int32_t ka_order_slot_device(ka_ctx* ctx, int32_t slot, void* stream);
int32_t ka_emit_device(ka_ctx* ctx, int32_t* d_out_len, int32_t* d_out_broker, void* stream, ka_status* st);
int32_t ka_ctx_export_counter_slot_device(ka_ctx* ctx, int32_t slot, int32_t* d_column, void* stream);
int32_t ka_ctx_import_counter_slot_device(ka_ctx* ctx, int32_t slot, const int32_t* d_column, void* stream);

/* Index of the staged block's first topic in the whole run: ka_status.topic_index of stage/order solves is reported
 * relative to the run (rank g of a topic-sharded job passes the number of topics owned by ranks < g), so that the ranks
 * can agree on the LOWEST failing topic of the run (KAG:173 aborts at the first throw). Default 0. */
int32_t ka_ctx_set_topic_base(ka_ctx* ctx, int32_t topic_base);

/* Synchronise the last asynchronous solve and return its status. */
int32_t ka_last_status(ka_ctx* ctx, ka_status* st);

/* ---- movement plan ------------------------------------------------------------------------------
 * What applying the last solve's assignment moves. Row g has current list C (leader first; dense cur[g*RF ..] or ragged
 * cur_broker[rep_off[g] ..]) and new list O (out_len[g] long, or the target RF when the solve had no out_len). Its class:
 *   0 UNCHANGED  O == C as sequences
 *   1 REORDERED  same broker set and length, other order: only the preferred leader / fallback order changes, no data copied
 *   2 MOVED      the broker sets or the lengths differ (an empty C is MOVED)
 * added = |O \ C|, dropped = |C \ O| (as sets; a broker repeated in C counts once); leader changed = O[0] != C[0] (with an
 * empty C, O[0] is a leader gain). */
typedef struct ka_plan_totals {
    int64_t rows, rows_reordered, rows_moved, replicas_added, replicas_dropped, leaders_changed;
} ka_plan_totals;

/* Report-id list of ka_plan_last's per-broker columns: ids[M] strictly ascending, M <= 65534. M = 0 (the default): the live
 * broker table of the moment ka_plan_last runs. Brokers being decommissioned are not live: list them here to see them one
 * by one. */
int32_t ka_ctx_set_report_brokers(ka_ctx* ctx, int32_t M, const int32_t* ids);

/* Movement plan of the ctx's last successful solve (ka_solve, ka_solve_dense, ka_solve_dense_json[_changed],
 * ka_solve_dense_device), computed on the device from the rows still resident: no second upload. After
 * ka_solve_dense_device the caller's d_cur_broker / d_out_broker / d_out_len must still hold what that solve read and wrote.
 * Synchronises the last solve first, like ka_last_status. KA_ERR_BAD_ARG before any solve, after a failed solve and after the
 * split stage / order / emit solve.
 *   row_class[Q]          class of every row (NULL: not wanted)
 *   broker_stats[(M+1)*8] per report bucket (row i < M: ids[i]; row M: every other id), uint32 columns
 *                         replicas_before, replicas_after, replicas_in, replicas_out,
 *                         leaders_before, leaders_after, leaders_in, leaders_out   (NULL: not wanted)
 *   totals                (NULL: not wanted)
 * Per bucket after = before + in - out (replicas and leaders); sum(replicas_in) = replicas_added, sum(replicas_out) =
 * replicas_dropped, sum(leaders_in) = leaders_changed, sum(leaders_out) = leaders_changed - (rows with an empty C that got a
 * leader). */
int32_t ka_plan_last(ka_ctx* ctx, uint8_t* row_class, uint32_t* broker_stats, ka_plan_totals* totals);

/* ---- counters (Context.counter) -----------------------------------------------------------------
 * counter[i*slots + r] = Context.counter[broker_id[i]][r] for the CURRENT broker table (KAS:289-301:
 * absent == 0). slots = ka_ctx_counter_slots(). Used by tests and by the multi-GPU ring hand-off
 * (rank g imports what rank g-1 exported before ordering its own topics — S5 is a serial chain). */
int32_t ka_ctx_counter_slots(ka_ctx* ctx);
int32_t ka_ctx_get_counters(ka_ctx* ctx, int32_t* counter /* [N*slots] host */);
int32_t ka_ctx_set_counters(ka_ctx* ctx, const int32_t* counter /* [N*slots] host */);
/* device-to-device variants for NCCL plumbing: d_counter is a device buffer of N*slots int32. Stream contract: the copy
 * is enqueued on `stream`; pass the SAME stream as the stage/order calls (or order the streams yourself) — an import
 * must precede, and an export must follow, the ka_order_device it belongs to in stream order. */
int32_t ka_ctx_export_counters_device(ka_ctx* ctx, int32_t* d_counter, void* stream);
int32_t ka_ctx_import_counters_device(ka_ctx* ctx, const int32_t* d_counter, void* stream);

/* ---- instrumentation ----------------------------------------------------------------------------
 * Per-phase device times of the LAST solve, measured with CUDA events on the solve's stream.
 * ms[0]=sticky+spread kernel (S0-S4)  ms[1]=chunk tables of the level schedule (scan + fill; 0 when capacity is 1)
 * ms[2]=slot-0 leader-order chain (S5; sum over sub-blocks)   ms[3]=H2D   ms[4]=D2H   ms[5]=total on stream
 * ms[6]=slot-1 chain + emit (sum over sub-blocks; overlaps ms[2] in time)   ms[7]=wall time of all chains + emit
 * Enabled with ka_ctx_set_timing(ctx, 1); costs a few event records per solve. */
int32_t ka_ctx_set_timing(ka_ctx* ctx, int32_t enabled);
int32_t ka_ctx_last_timing(ka_ctx* ctx, float* ms /* [8] */);
/* Number of kernel launches issued by this ctx since creation (for bench.py's gpu_launches). */
int64_t ka_ctx_launch_count(ka_ctx* ctx);

const char* ka_version(void);

#ifdef __cplusplus
}
#endif
#endif /* KASSIGN_H */
