"""ctypes binding of oracle/kafka_oracle.cpp (TEST INFRASTRUCTURE — see that file's header).

Importers allowed: tests/, __graft_entry__.smoke(), bench.py (cpu_baseline / --impl reference).
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "kafka_oracle.cpp")
_LIB = os.path.join(_HERE, "liboracle.so")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class OracleStatus(ctypes.Structure):
    _fields_ = [("code", ctypes.c_int32), ("topic_index", ctypes.c_int32), ("partition", ctypes.c_int32),
                ("a", ctypes.c_int32), ("b", ctypes.c_int32), ("message", ctypes.c_char * 256)]


def _compile(src, lib):
    """g++ `src` into `lib`; when oracle/ is read-only (a shared checkout), into a fresh temporary directory instead.
    Returns the path written."""
    if not os.access(os.path.dirname(lib), os.W_OK):
        lib = os.path.join(tempfile.mkdtemp(prefix="kassign-oracle-"), os.path.basename(lib))
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", lib, src])
    return lib


def build(force=False):
    """g++ the restatements into oracle/liboracle.so + libfastoracle.so (gcc only; no reference sources are copied)."""
    global _LIB
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(_SRC):
        _LIB = _compile(_SRC, _LIB)
    fast_lib()
    return _LIB


_FSRC = os.path.join(_HERE, "fast_oracle.cpp")
_FLIB = os.path.join(_HERE, "libfastoracle.so")


class FastStatus(ctypes.Structure):
    _fields_ = [("code", ctypes.c_int32), ("topic_index", ctypes.c_int32), ("partition", ctypes.c_int32),
                ("a", ctypes.c_int32), ("b", ctypes.c_int32)]


_lib = None
_flib = None


def fast_lib():
    """The optimised flat-array CPU solver (fast_oracle.cpp) — BASELINE.md 'B1' and a third restatement."""
    global _flib, _FLIB
    if _flib is None:
        if not os.path.exists(_FLIB) or os.path.getmtime(_FLIB) < os.path.getmtime(_FSRC):
            _FLIB = _compile(_FSRC, _FLIB)
        L = ctypes.CDLL(_FLIB)
        L.fast_ctx_create.restype = ctypes.c_void_p
        L.fast_ctx_destroy.argtypes = [ctypes.c_void_p]
        L.fast_ctx_reset.argtypes = [ctypes.c_void_p]
        L.fast_solve_dense.restype = ctypes.c_int
        _flib = L
    return _flib


class FastContext:
    def __init__(self):
        self._h = ctypes.c_void_p(fast_lib().fast_ctx_create())

    def reset(self):
        fast_lib().fast_ctx_reset(self._h)

    def __del__(self):
        try:
            fast_lib().fast_ctx_destroy(self._h)
        except Exception:
            pass


def fast_run_dense(ctx, topic_hash, cur, broker_id, rack_index, desired_rf=-1, out_stride=None):
    """cur int32 [T,P,RF] -> (out [T*P, S], out_len [T*P], FastStatus). Single thread."""
    cur = np.ascontiguousarray(cur, dtype=np.int32)
    T, P, RF = cur.shape
    S = out_stride or max(RF, desired_rf, 1)
    th = np.ascontiguousarray(topic_hash, dtype=np.int32)
    b = np.ascontiguousarray(broker_id, dtype=np.int32)
    r = np.ascontiguousarray(rack_index, dtype=np.int32)
    out = np.full((T * P, S), -1, dtype=np.int32)
    out_len = np.zeros(T * P, dtype=np.int32)
    st = FastStatus()
    fast_lib().fast_solve_dense(ctx._h, ctypes.c_int32(T), _p(th), ctypes.c_int32(P), ctypes.c_int32(RF), _p(cur),
                                ctypes.c_int32(len(b)), _p(b), _p(r), ctypes.c_int32(desired_rf), ctypes.c_int32(S),
                                _p(out_len), _p(out), ctypes.byref(st))
    return out, out_len, st


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            build()
        L = ctypes.CDLL(_LIB)
        L.oracle_ctx_create.restype = ctypes.c_void_p
        L.oracle_ctx_destroy.argtypes = [ctypes.c_void_p]
        L.oracle_ctx_reset.argtypes = [ctypes.c_void_p]
        L.oracle_java_string_hash.argtypes = [ctypes.c_char_p]
        L.oracle_java_string_hash.restype = ctypes.c_int32
        L.oracle_ctx_get_counter.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32]
        L.oracle_ctx_get_counter.restype = ctypes.c_int32
        L.oracle_ctx_set_counter.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]
        L.oracle_ctx_set_counter.restype = None
        L.oracle_run.restype = ctypes.c_int
        _lib = L
    return _lib




class OracleError(Exception):
    def __init__(self, st):
        super().__init__(st.message.decode())
        self.code, self.topic_index, self.partition, self.a, self.b = st.code, st.topic_index, st.partition, st.a, st.b
        self.message = st.message.decode()


class OracleContext:
    """One KafkaTopicAssigner instance == one Context (KTA:19-23)."""

    def __init__(self):
        self._h = ctypes.c_void_p(lib().oracle_ctx_create())

    def reset(self):
        lib().oracle_ctx_reset(self._h)

    def counter(self, broker_id, slot):
        return lib().oracle_ctx_get_counter(self._h, int(broker_id), int(slot))

    def __del__(self):
        try:
            lib().oracle_ctx_destroy(self._h)
        except Exception:
            pass


def java_string_hash(s: str) -> int:
    return lib().oracle_java_string_hash(s.encode("utf-8"))


def run(ctx, topic_names, part_off, part_id, rep_off, cur_broker, broker_id, rack_names, desired_rf, out_stride,
        raise_on_error=True):
    """KAG:172-184 loop over topics through ONE context. Returns (out_len, out_part_id, out_broker, status).

    rack_names: list of str|None per broker. Arrays are numpy (int64 offsets, int32 ids)."""
    T = len(topic_names)
    names_b = [n.encode("utf-8") + b"\0" for n in topic_names]
    name_off = np.zeros(T + 1, dtype=np.int64)
    np.cumsum([len(b) for b in names_b], out=name_off[1:])
    blob = b"".join(names_b)
    rb = [(r.encode("utf-8") if r is not None else b"") for r in rack_names]
    rack_off = np.zeros(len(rb) + 1, dtype=np.int64)
    np.cumsum([len(b) for b in rb], out=rack_off[1:])
    rack_blob = b"".join(rb)
    part_off = np.ascontiguousarray(part_off, dtype=np.int64)
    part_id = np.ascontiguousarray(part_id, dtype=np.int32)
    rep_off = np.ascontiguousarray(rep_off, dtype=np.int64)
    cur_broker = np.ascontiguousarray(cur_broker, dtype=np.int32)
    broker_id = np.ascontiguousarray(broker_id, dtype=np.int32)
    nP = int(part_off[-1])
    out_len = np.zeros(nP, dtype=np.int32)
    out_pid = np.full(nP, -1, dtype=np.int32)
    out_broker = np.full(nP * out_stride, -1, dtype=np.int32)
    st = OracleStatus()
    rc = lib().oracle_run(ctx._h, ctypes.c_int32(T), ctypes.c_char_p(blob), _p(name_off), _p(part_off), _p(part_id),
                          _p(rep_off), _p(cur_broker), ctypes.c_int32(len(broker_id)), _p(broker_id),
                          ctypes.c_char_p(rack_blob), _p(rack_off), ctypes.c_int32(desired_rf),
                          ctypes.c_int32(out_stride), _p(out_len), _p(out_pid), _p(out_broker), ctypes.byref(st))
    if rc != 0 and raise_on_error:
        raise OracleError(st)
    return out_len, out_pid, out_broker.reshape(nP, out_stride), st
