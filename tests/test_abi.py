"""CPU tests: the C-ABI shared library loads and exports every symbol include/kassign.h declares; host-only
helpers behave; and without a GPU the product path FAILS LOUDLY (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

import kafka_assigner_b200 as kab

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "kassign.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ka_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(native_lib):
    names = _declared_symbols()
    assert len(names) >= 18
    raw = ctypes.CDLL(kab.lib_path())
    for n in names:
        assert hasattr(raw, n), "libkassign.so does not export %s" % n
    assert set(names) == set(kab._native.SYMBOLS), "ctypes table and header disagree"
    assert b"sm_100a" in native_lib.ka_version()


def test_library_is_sm100a_cuda_not_a_cpu_build():
    import subprocess
    out = subprocess.run([kab.build_mod.cuda_tool("cuobjdump"), "--list-elf", kab.lib_path()], capture_output=True,
                         text=True).stdout
    assert "sm_100a" in out


def test_java_string_hash_host_helper(native_lib):
    from oracle import py_oracle as po
    for s in ["test", "", "a", "polygenelubricants", "topic-000123", "héllo-日本", "\U0001F600x"]:
        assert kab.java_string_hash(s) == po.java_string_hash(s)


def test_rack_indices_string_semantics(native_lib):
    ids = np.array([13, 14, 15, 16], dtype=np.int32)
    names = [None, b"13", None, b"z"]  # broker 14's rack is literally "13" == str(13): shared (KAS:82-94)
    arr = (ctypes.c_char_p * 4)(*names)
    out = np.zeros(4, dtype=np.int32)
    assert native_lib.ka_rack_indices(4, ids.ctypes.data_as(ctypes.c_void_p), ctypes.cast(arr, ctypes.c_void_p),
                                      out.ctypes.data_as(ctypes.c_void_p)) == 0
    assert out[0] == out[1] and len({out[0], out[2], out[3]}) == 3
    assert np.array_equal(out, kab.synth.rack_indices(ids, [None, "13", None, "z"]))


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a box without a GPU")
def test_no_gpu_fails_loudly(native_lib):
    assert not native_lib.ka_ctx_create(0)
    with pytest.raises(kab.KassignError):
        kab.Solver(0)
    with pytest.raises(kab.KassignError):
        kab.KafkaTopicAssigner()
    st = kab.KaStatus()
    assert native_lib.ka_solve_dense(None, 0, None, 0, 0, None, -1, 1, None, None, ctypes.byref(st)) == kab._native.KA_ERR_NO_DEVICE
