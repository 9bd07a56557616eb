"""kafka-assigner_b200 — B200-native drop-in for kafka-assigner's generateAssignment hot path.

Holds only what the path needs: csrc/ (sm_100a CUDA kernels + the C ABI of include/kassign.h),
the host-side mirror of the reference interface (assigner.py) and the synthetic-cluster generator
used by the parity tests and bench (synth.py). Import as `kafka_assigner_b200` (see the shim module
at the repo root — the directory name carries a hyphen).
"""
from . import build as build_mod  # noqa: F401
from . import synth  # noqa: F401
from ._native import KaStatus, load as load_native, lib_path  # noqa: F401
from .assigner import (ArrayIndexOutOfBoundsException, IllegalStateException, KafkaTopicAssigner,  # noqa: F401
                       KassignError, Solver, java_string_hash, raise_for_status)
from .assigner import PLAN_COLUMNS, ROW_MOVED, ROW_REORDERED, ROW_UNCHANGED  # noqa: F401

__all__ = ["KafkaTopicAssigner", "Solver", "IllegalStateException", "ArrayIndexOutOfBoundsException",
           "KassignError", "java_string_hash", "synth", "load_native", "lib_path", "KaStatus", "raise_for_status"]
