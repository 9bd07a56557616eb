"""Host-side mirror of the reference's interface for the hot path, over the C ABI (include/kassign.h).

  KafkaTopicAssigner.generate_assignment(...)  <->  KafkaTopicAssigner.generateAssignment
                                                    (reference KafkaTopicAssigner.java:42-72)
  Solver.solve_cluster(...)                    <->  the per-topic loop with ONE shared assigner
                                                    (reference KafkaAssignmentGenerator.java:172-184)

Same names, argument meaning and error behaviour (message texts of KTA:58-60, 65-66, 67-69 and
KAS:183-184). All compute happens in libkassign.so's CUDA kernels; nothing here falls back to a CPU
solver — if the library or a GPU is missing, construction raises.
"""
import ctypes

import numpy as np

from . import _native
from ._native import KaPlanTotals, KaStatus

# movement plan (ka_plan_last): row classes and the columns of Solver.last_plan()'s per-broker table
ROW_UNCHANGED, ROW_REORDERED, ROW_MOVED = 0, 1, 2
PLAN_COLUMNS = ("replicas_before", "replicas_after", "replicas_in", "replicas_out",
                "leaders_before", "leaders_after", "leaders_in", "leaders_out")


class IllegalStateException(Exception):
    """java.lang.IllegalStateException as thrown by Preconditions.checkState on the reference path."""


class ArrayIndexOutOfBoundsException(Exception):
    """java.lang.ArrayIndexOutOfBoundsException (topic.hashCode() == Integer.MIN_VALUE, KAS:190-192)."""


class KassignError(RuntimeError):
    """Library-side failure with no reference counterpart (bad argument, CUDA error, size limit)."""

    def __init__(self, code, msg=""):
        super().__init__("kassign error %d %s" % (code, msg))
        self.code = code


def java_string_hash(s: str) -> int:
    return _native.load().ka_java_string_hash(s.encode("utf-8"))


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def raise_for_status(st: KaStatus, topic_names=None):
    """Re-throw a ka_status as the reference's exception with the identical message."""
    if st.code == 0:
        return
    topic = topic_names[st.topic_index] if (topic_names is not None and 0 <= st.topic_index < len(topic_names)) else "?"
    if st.code == _native.KA_ERR_RF_MISMATCH:
        raise IllegalStateException("Topic %s has partition %d with unexpected replication factor %d" % (topic, st.partition, st.a))
    if st.code == _native.KA_ERR_RF_NOT_POSITIVE:
        raise IllegalStateException("Topic %s does not have a positive replication factor!" % topic)
    if st.code == _native.KA_ERR_RF_GT_BROKERS:
        raise IllegalStateException("Topic %s has a higher replication factor (%d) than available brokers!" % (topic, st.a))
    if st.code == _native.KA_ERR_UNASSIGNABLE:
        raise IllegalStateException("Partition %d could not be fully assigned!" % st.partition)
    if st.code == _native.KA_ERR_HASH_INDEX:
        raise ArrayIndexOutOfBoundsException(str(st.a))
    raise KassignError(st.code, "(topic_index=%d partition=%d a=%d b=%d)" % (st.topic_index, st.partition, st.a, st.b))


class Solver:
    """One ka_ctx: one Context (KAS:360-369) plus device scratch. Batch-level API on flat arrays."""

    def __init__(self, device=0):
        self._L = _native.load()
        h = self._L.ka_ctx_create(int(device))
        if not h:
            raise KassignError(_native.KA_ERR_NO_DEVICE, "no usable CUDA device: kassign has no CPU fallback")
        self._h = ctypes.c_void_p(h)
        self.device = device
        self.N = 0
        self.broker_id = None
        self.report_ids = None   # set_report_brokers(); None = the live broker table
        self._last_rows = None   # rows of the last solve issued through this object (None: no solve, or the split API)

    def close(self):
        if getattr(self, "_h", None):
            self._L.ka_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- Context -------------------------------------------------------------------------------
    def reset(self):
        rc = self._L.ka_ctx_reset(self._h)
        if rc:
            raise KassignError(rc)

    def set_brokers(self, broker_id, rack_index):
        b = np.ascontiguousarray(broker_id, dtype=np.int32)
        r = np.ascontiguousarray(rack_index, dtype=np.int32)
        rc = self._L.ka_ctx_set_brokers(self._h, len(b), _ptr(b), _ptr(r))
        if rc:
            raise KassignError(rc, "ka_ctx_set_brokers")
        self.N = len(b)
        self.broker_id = b

    def set_brokers_with_racks(self, brokers, rack_assignment):
        """brokers: iterable of ids (any order); rack_assignment: {id: rack string} (may lack entries)."""
        b = np.array(sorted(set(int(x) for x in brokers)), dtype=np.int32)
        names = [rack_assignment.get(int(x)) for x in b]
        arr = (ctypes.c_char_p * len(b))(*[(n.encode("utf-8") if n is not None else None) for n in names])
        racks = np.zeros(len(b), dtype=np.int32)
        rc = self._L.ka_rack_indices(len(b), _ptr(b), ctypes.cast(arr, ctypes.c_void_p), _ptr(racks))
        if rc:
            raise KassignError(rc, "ka_rack_indices")
        self.set_brokers(b, racks)
        return b

    def counters(self):
        slots = self._L.ka_ctx_counter_slots(self._h)
        out = np.zeros((self.N, slots), dtype=np.int32)
        rc = self._L.ka_ctx_get_counters(self._h, _ptr(out))
        if rc:
            raise KassignError(rc)
        return out

    def set_counters(self, ctr):
        c = np.ascontiguousarray(ctr, dtype=np.int32)
        assert c.shape == (self.N, self._L.ka_ctx_counter_slots(self._h))
        rc = self._L.ka_ctx_set_counters(self._h, _ptr(c))
        if rc:
            raise KassignError(rc)

    def set_timing(self, on=True):
        self._L.ka_ctx_set_timing(self._h, 1 if on else 0)

    def last_timing(self):
        ms = np.zeros(8, dtype=np.float32)
        self._L.ka_ctx_last_timing(self._h, _ptr(ms))
        return dict(sticky_spread_ms=float(ms[0]), level_tables_ms=float(ms[1]), leader_order_ms=float(ms[2]),
                    h2d_ms=float(ms[3]), d2h_ms=float(ms[4]), total_ms=float(ms[5]), slot1_emit_ms=float(ms[6]), chains_wall_ms=float(ms[7]))

    def set_topic_base(self, topic_base):
        """Topic-sharded runs: index of this rank's first topic in the whole run (status reporting)."""
        rc = self._L.ka_ctx_set_topic_base(self._h, int(topic_base))
        if rc:
            raise KassignError(rc)

    def launch_count(self):
        return int(self._L.ka_ctx_launch_count(self._h))

    # -- solves --------------------------------------------------------------------------------
    def solve_dense(self, topic_hash, cur, desired_rf=-1, out_stride=None, out=None, out_len=None, check=True,
                    topic_names=None):
        """cur: int32 [T, P, RF] host array -> (out [T, P, out_stride], out_len [T, P], status)."""
        cur = np.ascontiguousarray(cur, dtype=np.int32)
        T, P, RF = cur.shape
        th = np.ascontiguousarray(topic_hash, dtype=np.int32)
        assert th.shape == (T,)
        if out_stride is None:
            out_stride = max(RF, desired_rf if desired_rf >= 0 else RF, 1)
        if out is None:
            out = np.full((T, P, out_stride), -1, dtype=np.int32)
        if out_len is None:
            out_len = np.zeros((T, P), dtype=np.int32)
        st = KaStatus()
        self._last_rows = T * P
        self._L.ka_solve_dense(self._h, T, _ptr(th), P, RF, _ptr(cur), int(desired_rf), int(out_stride), _ptr(out_len),
                               _ptr(out), ctypes.byref(st))
        if check:
            raise_for_status(st, topic_names)
        return out, out_len, st

    @staticmethod
    def marshal_names(topic_names):
        """(concatenated UTF-8 bytes, offsets[T+1]) — the name slab ka_solve_dense_json takes."""
        enc = [n.encode("utf-8") for n in topic_names]
        name_off = np.zeros(len(enc) + 1, dtype=np.int64)
        name_off[1:] = np.cumsum([len(e) for e in enc])
        return np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8), name_off

    def solve_dense_json(self, topic_names, topic_hash, cur, desired_rf=-1, json_buf=None, check=True, names_slab=None,
                         changed_only=False):
        """Solve + emit the reassignment JSON on the device (KAG:169-186); returns (bytes-like view of the text, status).
        json_buf: optional writable uint8 numpy array (pinned memory for full PCIe speed); names_slab: marshal_names() result.
        changed_only: list only the partitions whose replica list changes (ka_solve_dense_json_changed); same format, and
        '{"partitions":[],"version":1}' when nothing changes."""
        cur = np.ascontiguousarray(cur, dtype=np.int32)
        T, P, RF = cur.shape
        th = np.ascontiguousarray(topic_hash, dtype=np.int32)
        names, name_off = names_slab if names_slab is not None else self.marshal_names(topic_names)
        S = max(RF, desired_rf, 1)
        cap = 64 + T * P * (50 + 12 * S) + int(P * name_off[-1])
        if json_buf is None:
            json_buf = np.empty(cap, dtype=np.uint8)
        nbytes = ctypes.c_int64(0)
        st = KaStatus()
        self._last_rows = T * P
        fn = self._L.ka_solve_dense_json_changed if changed_only else self._L.ka_solve_dense_json
        fn(self._h, T, _ptr(th), P, RF, _ptr(cur), int(desired_rf), _ptr(names), _ptr(name_off), _ptr(json_buf),
           int(json_buf.size), ctypes.byref(nbytes), ctypes.byref(st))
        if check:
            raise_for_status(st, topic_names)
        return json_buf[:nbytes.value], st

    def solve_ragged(self, topic_hash, part_off, part_id, rep_off, cur_broker, desired_rf, out_stride, check=True,
                     topic_names=None):
        th = np.ascontiguousarray(topic_hash, dtype=np.int32)
        part_off = np.ascontiguousarray(part_off, dtype=np.int64)
        part_id = None if part_id is None else np.ascontiguousarray(part_id, dtype=np.int32)
        rep_off = np.ascontiguousarray(rep_off, dtype=np.int64)
        cur_broker = np.ascontiguousarray(cur_broker, dtype=np.int32)
        Q = int(part_off[-1]) if len(part_off) else 0
        out = np.full((Q, out_stride), -1, dtype=np.int32)
        out_len = np.zeros(Q, dtype=np.int32)
        st = KaStatus()
        self._last_rows = Q
        self._L.ka_solve(self._h, len(th), _ptr(th), _ptr(part_off), _ptr(part_id), _ptr(rep_off), _ptr(cur_broker),
                         int(desired_rf), int(out_stride), _ptr(out_len), _ptr(out), ctypes.byref(st))
        if check:
            raise_for_status(st, topic_names)
        return out, out_len, st

    def solve_dense_device(self, T, d_topic_hash, P, RF, d_cur, desired_rf, out_stride, d_out_len, d_out, stream=0,
                           sync=True):
        """Device-pointer form (ints from tensor.data_ptr()); returns KaStatus when sync else None. last_plan() after this
        reads the caller's d_cur / d_out / d_out_len: keep them alive and unchanged until then."""
        st = KaStatus()
        self._last_rows = int(T) * int(P)
        rc = self._L.ka_solve_dense_device(self._h, int(T), ctypes.c_void_p(d_topic_hash), int(P), int(RF),
                                           ctypes.c_void_p(d_cur), int(desired_rf), int(out_stride),
                                           ctypes.c_void_p(d_out_len) if d_out_len else None, ctypes.c_void_p(d_out),
                                           ctypes.c_void_p(stream) if stream else None,
                                           ctypes.byref(st) if sync else None)
        if not sync:
            if rc:
                raise KassignError(rc, "ka_solve_dense_device")
            return None
        return st

    def stage_dense_device(self, T, d_topic_hash, P, RF, d_cur, desired_rf, out_stride, stream=0):
        """Context-free stage (KAS:65-200) of a topic block — shards across GPUs."""
        self._last_rows = None
        rc = self._L.ka_stage_dense_device(self._h, int(T), ctypes.c_void_p(d_topic_hash), int(P), int(RF),
                                           ctypes.c_void_p(d_cur), int(desired_rf), int(out_stride),
                                           ctypes.c_void_p(stream) if stream else None)
        if rc:
            raise KassignError(rc, "ka_stage_dense_device")

    def order_device(self, d_out_len, d_out, stream=0, sync=True):
        """Leader-order stage (KAS:202-239) of the staged block against this Context's counters."""
        st = KaStatus()
        rc = self._L.ka_order_device(self._h, ctypes.c_void_p(d_out_len) if d_out_len else None, ctypes.c_void_p(d_out),
                                     ctypes.c_void_p(stream) if stream else None, ctypes.byref(st) if sync else None)
        if not sync:
            if rc:
                raise KassignError(rc, "ka_order_device")
            return None
        return st

    def staged_slot_chains(self):
        """2 when the staged block is ordered by per-slot chains (rows <= 3), else 0."""
        return int(self._L.ka_staged_slot_chains(self._h))

    def order_slot_device(self, slot, stream=0):
        """Slot-0 / slot-1 leader-order chain of the staged block (reads and bumps only counter[.][slot])."""
        rc = self._L.ka_order_slot_device(self._h, int(slot), ctypes.c_void_p(stream) if stream else None)
        if rc:
            raise KassignError(rc, "ka_order_slot_device")

    def emit_device(self, d_out_len, d_out, stream=0, sync=True):
        st = KaStatus()
        rc = self._L.ka_emit_device(self._h, ctypes.c_void_p(d_out_len) if d_out_len else None, ctypes.c_void_p(d_out),
                                    ctypes.c_void_p(stream) if stream else None, ctypes.byref(st) if sync else None)
        if not sync:
            if rc:
                raise KassignError(rc, "ka_emit_device")
            return None
        return st

    def export_counter_slot_device(self, slot, d_ptr, stream=0):
        rc = self._L.ka_ctx_export_counter_slot_device(self._h, int(slot), ctypes.c_void_p(d_ptr), ctypes.c_void_p(stream) if stream else None)
        if rc:
            raise KassignError(rc)

    def import_counter_slot_device(self, slot, d_ptr, stream=0):
        rc = self._L.ka_ctx_import_counter_slot_device(self._h, int(slot), ctypes.c_void_p(d_ptr), ctypes.c_void_p(stream) if stream else None)
        if rc:
            raise KassignError(rc)

    def last_status(self):
        st = KaStatus()
        self._L.ka_last_status(self._h, ctypes.byref(st))
        return st

    def export_counters_device(self, d_ptr, stream=0):
        rc = self._L.ka_ctx_export_counters_device(self._h, ctypes.c_void_p(d_ptr), ctypes.c_void_p(stream) if stream else None)
        if rc:
            raise KassignError(rc)

    def import_counters_device(self, d_ptr, stream=0):
        rc = self._L.ka_ctx_import_counters_device(self._h, ctypes.c_void_p(d_ptr), ctypes.c_void_p(stream) if stream else None)
        if rc:
            raise KassignError(rc)

    # -- movement plan ---------------------------------------------------------------------------
    def set_report_brokers(self, ids=None):
        """Broker ids that last_plan() reports one by one (strictly ascending after sorting, at most 65534); every other id
        falls into the extra 'other' row. None or empty: the live broker table (decommissioned brokers land in 'other')."""
        b = np.zeros(0, dtype=np.int32) if ids is None else np.ascontiguousarray(np.sort(np.asarray(ids, dtype=np.int32)))
        rc = self._L.ka_ctx_set_report_brokers(self._h, len(b), _ptr(b) if len(b) else None)
        if rc:
            raise KassignError(rc, "ka_ctx_set_report_brokers")
        self.report_ids = b if len(b) else None

    def last_plan(self, row_class=False):
        """Movement plan of the last successful solve, computed on the device (ka_plan_last).

        Returns (totals, broker_ids, broker_stats, row_class):
          totals        dict rows, rows_reordered, rows_moved, replicas_added, replicas_dropped, leaders_changed
          broker_ids    int32 [M]: the report ids (set_report_brokers, default the live broker table)
          broker_stats  uint32 [M + 1, 8]: row i for broker_ids[i], row M for every other id; columns PLAN_COLUMNS =
                        replicas_before, replicas_after, replicas_in (copied to the broker), replicas_out (removed from it),
                        leaders_before, leaders_after, leaders_in (leadership gained), leaders_out (leadership lost)
          row_class     uint8 [rows] ROW_UNCHANGED / ROW_REORDERED (same brokers, new order) / ROW_MOVED (brokers differ), or
                        None unless row_class=True
        """
        ids = self.report_ids if self.report_ids is not None else (self.broker_id if self.broker_id is not None
                                                                   else np.zeros(0, dtype=np.int32))
        stats = np.zeros((len(ids) + 1, len(PLAN_COLUMNS)), dtype=np.uint32)
        cls = np.zeros(self._last_rows or 0, dtype=np.uint8) if row_class else None
        tot = KaPlanTotals()
        rc = self._L.ka_plan_last(self._h, _ptr(cls) if row_class and self._last_rows else None, _ptr(stats), ctypes.byref(tot))
        if rc:
            raise KassignError(rc, "ka_plan_last: no successful solve to plan")
        totals = {name: int(getattr(tot, name)) for name, _ in KaPlanTotals._fields_}
        return totals, ids.copy(), stats, cls

    def solve_cluster(self, cluster, check=True):
        """The KAG:172-184 loop for a synth.Cluster: all topics in order through this Context."""
        self.set_brokers(cluster.broker_id, cluster.rack_index)
        return self.solve_dense(cluster.topic_hash, cluster.cur, cluster.desired_rf, check=check,
                                topic_names=cluster.topic_names)


class KafkaTopicAssigner:
    """Mirror of siftscience.kafka.tools.KafkaTopicAssigner (KafkaTopicAssigner.java:18-72).

    One instance owns one Context, exactly like the reference (KTA:19-23): leader-preference counters
    persist across generate_assignment calls on the same instance.
    """

    def __init__(self, device=0):
        self._solver = Solver(device)
        self._brokers_key = None

    def generate_assignment(self, topic, current_assignment, brokers, rack_assignment, desired_replication_factor):
        """generateAssignment(topic, currentAssignment, brokers, rackAssignment, desiredReplicationFactor).

        current_assignment: {partition: [broker ids, leader first]}; brokers: set of ids;
        rack_assignment: {broker id: rack string}; returns {partition: [broker ids, leader first]}
        (ascending partition order, like the reference's TreeMap).
        """
        if current_assignment is None:
            raise TypeError("currentAssignment is null")  # NullPointerException at KTA:51
        key = (tuple(sorted(set(int(b) for b in brokers))), tuple(sorted((int(k), v) for k, v in rack_assignment.items())))
        if key != self._brokers_key:
            self._solver.set_brokers_with_racks(brokers, rack_assignment)
            self._brokers_key = key
        parts = sorted(int(p) for p in current_assignment)
        lists = [list(current_assignment[p]) for p in parts]
        part_off = np.array([0, len(parts)], dtype=np.int64)
        rep_off = np.zeros(len(parts) + 1, dtype=np.int64)
        if parts:
            np.cumsum([len(l) for l in lists], out=rep_off[1:])
        cur = np.array([b for l in lists for b in l], dtype=np.int32)
        maxlen = max([len(l) for l in lists], default=0)
        stride = max(1, maxlen, desired_replication_factor if desired_replication_factor >= 0 else 0)
        th = np.array([java_string_hash(topic)], dtype=np.int32)
        out, out_len, _ = self._solver.solve_ragged(th, part_off, np.array(parts, dtype=np.int32), rep_off, cur,
                                                    desired_replication_factor, stride, check=True, topic_names=[topic])
        return {p: [int(x) for x in out[i, :out_len[i]]] for i, p in enumerate(parts)}
