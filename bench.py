#!/usr/bin/env python
"""bench.py — partition-replica assignments/sec of the B200-native kafka-assigner hot path.

  python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU
  torchrun ... bench.py --gpus N ...                       # one rank per GPU, topic-sharded (weak scaling)
  python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/*.npy (diff two builds)

A "step" is one pass of the hot path (KafkaTopicAssigner.generateAssignment for every topic of the
workload, in order, through ONE Context — the loop of KafkaAssignmentGenerator.java:172-184) over one
batch of synthetic input. `value` times the device-resident solve (inputs already in HBM, outputs left
in HBM) with CUDA events on the launching stream; `e2e` times the same solve through the host-buffer C-ABI
call with the H2D and D2H copies inside the timed region. Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "partition-replica assignments/sec"
UNIT = "assignments/s"
ALGO_BYTES_PER_UNIT = 8  # SURVEY.md §8(d): 4 B current broker read + 4 B new broker written per partition-replica
L2_FLUSH_BYTES = 256 << 20
DUMP_BYTES = 64 << 20
DUMP_SEED = 0x5EED0D


def dump_outputs(path, arrays, budget=DUMP_BYTES, suffix=""):
    """Write {name: array [T, ...]} as path/<name><suffix>.npy in float64 (exact for every int32), at most `budget` bytes
    in all. Above the budget a fixed seeded sample of rows of axis 0 (the same rows for every array) is written, and the
    sampled row indices go to path/rows<suffix>.npy, so two builds run with the same arguments can be diffed file by file."""
    os.makedirs(path, exist_ok=True)
    T = len(next(iter(arrays.values())))
    row_bytes = 8 * sum(a[0].size for a in arrays.values()) if T else 0
    if row_bytes * T > budget:
        k = (budget - 4096) // (row_bytes + 8)   # 4 KiB left for the .npy headers
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(T, k, replace=False))
        arrays = dict({n: a[rows] for n, a in arrays.items()}, rows=rows)
    for n, a in arrays.items():
        np.save(os.path.join(path, n + suffix + ".npy"), np.asarray(a, dtype=np.float64))
    return sorted(arrays)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons while the timed region runs (NVML; nvidia-smi equivalent)."""

    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def oracle_time(cl, ol, repeats=1):
    """Seconds for the oracle (single-threaded, like the reference) to solve cluster `cl` `repeats` times."""
    part_off, part_id, rep_off, cur = cl.ragged()
    best = []
    for _ in range(repeats):
        ctx = ol.OracleContext()
        t0 = time.perf_counter()
        ol.run(ctx, cl.topic_names, part_off, part_id, rep_off, cur, cl.broker_id, cl.rack_name, cl.desired_rf, cl.RF)
        best.append(time.perf_counter() - t0)
    return best


def cpu_sample(cl, ol, budget_s):
    """Pick a topic prefix of the workload that costs about budget_s of oracle time (pilot on 16 topics)."""
    n0 = min(cl.T, 16)
    t = min(oracle_time(cl.subset(0, n0), ol, 2))
    per_topic = max(t / n0, 1e-7)
    n = int(max(1, min(cl.T, budget_s / per_topic)))
    return cl.subset(0, n) if n < cl.T else cl


def config_desc(args, cl, world, extra):
    """The `config` object of the JSON line — the same for both arms (the driver compares them), so every value says which arm
    it is about; the bounded sample of the reference arm is in its `sample` / `cpu_baseline.sample` keys."""
    return {"workload": workload_desc(args.workload, args.kind, cl) + ("; x%d topic blocks, one per GPU" % world if world > 1 else ""),
            "l2": "GPU arm: 256 MiB buffer written between timed iterations (L2 flush); both arms: fresh Context per step",
            "parallelism": ("GPU arm: topic-sharded stage, per-slot leader-order chains handed rank to rank (counter[.][0], then "
                            "counter[.][1]); reference arm: rank 0, one host thread, one topic block") if world > 1
                           else "GPU arm: single GPU; reference arm: one host thread",
            "extra": extra}


def run_reference(args):
    """Reference arm: the reference's algorithm (oracle port; no JVM exists in this image) on host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import kafka_assigner_b200 as kab
    from oracle import oracle_lib as ol
    ol.build()
    cl = kab.synth.make_config(args.workload, args.kind)
    total = max(1, args.steps + args.warmup)
    sample = cpu_sample(cl, ol, budget_s=min(20.0, 150.0 / total))
    for _ in range(args.warmup):
        oracle_time(sample, ol, 1)
    ts = []
    for _ in range(args.steps):
        ts += oracle_time(sample, ol, 1)
    sec = float(np.sum(ts))
    val = sample.replicas * args.steps / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sec / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": config_desc(args, cl, args.gpus, None),
        "sample": "first %d of %d topics per step" % (sample.T, cl.T),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": "first %d of %d topics (%d assignments) per step; single thread like the reference "
                                   "(KafkaAssignmentGenerator.java:173); host has %d cores" % (sample.T, cl.T, sample.replicas, os.cpu_count())},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "no JVM/javac/jars in this image: the reference Java cannot run; this is oracle/kafka_oracle.cpp, the "
                "structure-faithful C++ restatement (std::map/std::set for TreeMap/TreeSet)",
    }
    print(json.dumps(line))


def chain_depth(broker_id, out):
    """Depth (levels) of the leader-order dependency DAG of a solved run: partition q depends on the previous
    partition (global order) of each of its brokers (Context.counter rows, KAS:202-239). out: [Q, S] broker ids."""
    idx = np.searchsorted(broker_id, out).tolist()
    last = [0] * (len(broker_id) + 1)
    depth = 0
    for row in idx:
        l = 0
        for b in row:
            if last[b] > l:
                l = last[b]
        l += 1
        for b in row:
            last[b] = l
        if l > depth:
            depth = l
    return depth


def workload_desc(key, kind, cl):
    return "%s: %d topics x %d partitions RF=%d, %d brokers / %d racks, %s current assignment (expansion scenario, seed %#x)" % (
        key, cl.T, cl.P, cl.RF, cl.N, cl.meta.get("R", 0), kind, cl.meta.get("seed", 0))


def jvm_probe():
    """BASELINE.md B2: is there a JVM on this box that could run the real KafkaAssignmentStrategy? (never true in this
    image; recorded so that a JDK-equipped box does not go unnoticed)."""
    import shutil
    java, javac = shutil.which("java"), shutil.which("javac")
    return {"java": java, "javac": javac, "usable": bool(java and javac),
            "note": "no JVM: the reference Java cannot be timed or diffed here; parity is pinned on the oracle" if not (java and javac)
                    else "JDK found; the reference Java is not part of this repository, so parity stays pinned on the oracle"}


class Workload:
    """One rank's topic block of a weak-scaled run, resident on the device, plus the solve closures."""

    def __init__(self, key, kind, rank, world, local, torch, kab, dist, stream):
        self.key, self.kind, self.rank, self.world, self.torch, self.dist = key, kind, rank, world, torch, dist
        T = kab.synth.CONFIGS[key]["T"]
        self.cl = cl = kab.synth.make_config(key, kind, t_offset=rank * T)
        self.S = S = cl.RF
        self.units_rank = cl.replicas
        self.units_total = cl.replicas * world
        self.solver = kab.Solver(local)
        self.solver.set_brokers(cl.broker_id, cl.rack_index)
        self.solver.set_timing(True)
        self.solver.set_topic_base(rank * T)
        self.stream, self.sptr = stream, stream.cuda_stream
        self.h_hash = torch.from_numpy(cl.topic_hash).pin_memory()
        self.h_cur = torch.from_numpy(cl.cur).pin_memory()
        self.h_out = torch.empty((cl.T, cl.P, S), dtype=torch.int32).pin_memory()
        self.h_len = torch.empty((cl.T, cl.P), dtype=torch.int32).pin_memory()
        self.d_hash = self.h_hash.cuda()
        self.d_cur = self.h_cur.cuda()
        self.d_out = torch.empty((cl.T, cl.P, S), dtype=torch.int32, device="cuda")
        self.d_len = torch.empty((cl.T, cl.P), dtype=torch.int32, device="cuda")
        self.ctr_buf = torch.zeros(cl.N * 8, dtype=torch.int32, device="cuda")
        self.col_buf = [torch.zeros(cl.N, dtype=torch.int32, device="cuda") for _ in range(2)]
        self.ring_group = dist.new_group() if world > 1 else None   # the ring's own communicator
        self.kab = kab

    def device_step(self):
        cl, s, S = self.cl, self.solver, self.S
        if self.world == 1:
            s.solve_dense_device(cl.T, self.d_hash.data_ptr(), cl.P, cl.RF, self.d_cur.data_ptr(), -1, S, self.d_len.data_ptr(),
                                 self.d_out.data_ptr(), stream=self.sptr, sync=False)
        else:
            from kafka_assigner_b200 import multi
            sp, dl, do = self.sptr, self.d_len.data_ptr(), self.d_out.data_ptr()

            def phases():  # after stage(): rows <= 3 -> two slot chains handed on separately; else one fused chain
                if s.staged_slot_chains() == 2:
                    return [(lambda r=r: s.order_slot_device(r, sp), lambda t, r=r: s.export_counter_slot_device(r, t.data_ptr(), sp),
                             lambda t, r=r: s.import_counter_slot_device(r, t.data_ptr(), sp), self.col_buf[r]) for r in (0, 1)]
                return [(lambda: s.order_device(dl, do, stream=sp, sync=False), lambda t: s.export_counters_device(t.data_ptr(), sp),
                         lambda t: s.import_counters_device(t.data_ptr(), sp), self.ctr_buf)]

            def finish():
                if s.staged_slot_chains() == 2:
                    s.emit_device(dl, do, stream=sp, sync=False)

            multi.ring_solve_phases(self.rank, self.world,
                                    lambda: s.stage_dense_device(cl.T, self.d_hash.data_ptr(), cl.P, cl.RF, self.d_cur.data_ptr(), -1, S, stream=sp),
                                    phases, self.dist, finish=finish, final_broadcast=False, group=self.ring_group)

    def check_status(self, what):
        """Synchronise; the lowest failing topic of the WHOLE run wins on every rank (KAG:173 aborts at the first throw)."""
        st = self.solver.last_status()
        bad = st.topic_index if st.code != 0 else 2**31 - 1
        if self.world > 1:
            t = self.torch.tensor([bad], dtype=self.torch.int64, device="cuda")
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
            bad = int(t.item())
        if bad != 2**31 - 1:
            raise SystemExit("%s failed: first failing topic %d (local code %d)" % (what, bad, st.code))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed_device(self, n, flush, phase=None):
        torch, tot = self.torch, 0.0
        for i in range(n):
            self.solver.reset()                 # fresh Context per run (untimed)
            flush.fill_(i & 0xFF)               # evict L2 between iterations (untimed)
            if self.world > 1:
                self.dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            self.device_step()
            e1.record(self.stream)
            self.check_status("solve")
            e1.synchronize()
            tot += e0.elapsed_time(e1)
            if phase is not None:
                tm = self.solver.last_timing()
                for k in phase:
                    phase[k].append(tm[k])
        return tot

    def e2e_step(self):
        """Pinned host buffers -> H2D -> solve -> D2H through the public C-ABI entry, all inside the caller's timer."""
        cl, S = self.cl, self.S
        if self.world == 1:
            _, _, st = self.solver.solve_dense(self.h_hash.numpy(), self.h_cur.numpy(), -1, S, out=self.h_out.numpy(),
                                               out_len=self.h_len.numpy(), check=False)
            if st.code != 0:
                raise SystemExit("e2e solve failed: %d" % st.code)
        else:
            self.d_hash.copy_(self.h_hash, non_blocking=True)
            self.d_cur.copy_(self.h_cur, non_blocking=True)
            self.device_step()
            self.h_out.copy_(self.d_out, non_blocking=True)
            self.h_len.copy_(self.d_len, non_blocking=True)
            self.check_status("e2e solve")
            self.torch.cuda.synchronize()

    def timed_e2e(self, n, flush):
        tot = 0.0
        for i in range(n):
            self.solver.reset()
            flush.fill_(i & 0xFF)
            self.barrier()
            t0 = time.perf_counter()
            self.e2e_step()
            tot += time.perf_counter() - t0
        return tot

    def timed_e2e_json(self, n, flush):
        """Same solve, but the result leaves the GPU as the reference's reassignment JSON (KAG:169-186) built on the device."""
        torch, cl = self.torch, self.cl
        S = self.S
        cap = 64 + cl.T * cl.P * (50 + 12 * S + max(len(x) for x in cl.topic_names))
        if not hasattr(self, "h_json"):
            self.h_json = torch.empty(cap, dtype=torch.uint8).pin_memory()
            self.names_slab = self.solver.marshal_names(cl.topic_names)   # flat name slab, like the hashes and the replica slab
        tot, nbytes = 0.0, 0
        for i in range(n):
            self.solver.reset()
            flush.fill_(i & 0xFF)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            text, st = self.solver.solve_dense_json(cl.topic_names, self.h_hash.numpy(), self.h_cur.numpy(), -1, json_buf=self.h_json.numpy(), check=False,
                                                    names_slab=self.names_slab)
            tot += time.perf_counter() - t0
            if st.code != 0:
                raise SystemExit("e2e json solve failed: %d" % st.code)
            nbytes = len(text)
        return tot, nbytes

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def verify_full(self, ol):
        """EVERY output row of this rank's block against the flat-array CPU solver (itself pinned to the structure-faithful
        oracle in tests/test_oracle.py): the solver replays blocks 0..rank through one Context, like the reference's loop."""
        kab, T = self.kab, self.cl.T
        fctx = ol.FastContext()
        exp = exp_len = None
        for r in range(self.rank + 1):
            blk = self.cl if r == self.rank else kab.synth.make_config(self.key, self.kind, t_offset=r * T)
            exp, exp_len, fst = ol.fast_run_dense(fctx, blk.topic_hash, blk.cur, blk.broker_id, blk.rack_index)
            if fst.code != 0:
                raise SystemExit("oracle failed on block %d: %d" % (r, fst.code))
        ok = bool(np.array_equal(self.h_out.numpy().reshape(-1, self.S), exp) and np.array_equal(self.h_len.numpy().reshape(-1), exp_len))
        if self.world > 1:
            t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int32, device="cuda")
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
            ok = bool(t.item())
        return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # c3 = the largest BASELINE.json configuration quoted "on 1 B200"; every --gpus N weak-scales c3 blocks
    ap.add_argument("--workload", default="c3", choices=["c1", "c2", "c3", "c4shard", "c4", "c5"])
    ap.add_argument("--kind", default="mixed", choices=["mixed", "structured", "random"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config-4 (c4shard per rank) extra measurement at --gpus 8")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (out [T,P,RF] broker ids, out_len [T,P]) as DIR/<name>.npy, "
                         "float64, <= 64 MB in all (a seeded sample of topics beyond that); ranks > 0 add a _rank<r> suffix")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm times a topic prefix and keeps none")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import kafka_assigner_b200 as kab

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: kassign has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    json_fd = os.dup(1)
    if world > 1:
        # NCCL writes its version banner to fd 1: park everything but the final JSON line on stderr (rank 0 prints ONE line)
        sys.stdout.flush()
        os.dup2(2, 1)
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    stream = torch.cuda.current_stream()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    # ---- workload: rank r owns topics [r*T, (r+1)*T) of a world*T-topic run (weak scaling) ----------
    wl = Workload(args.workload, args.kind, rank, world, local, torch, kab, dist, stream)
    cl, S, solver = wl.cl, wl.S, wl.solver
    phase = {"sticky_spread_ms": [], "level_tables_ms": [], "leader_order_ms": [], "slot1_emit_ms": []}

    # ---- device-resident timing ----------------------------------------------------------------------
    wl.timed_device(args.warmup, flush)
    wl.barrier()
    launches0 = solver.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    ms_total = wl.timed_device(args.steps, flush, phase)
    clocks = sampler.stop()
    launches = solver.launch_count() - launches0
    # what the last timed step handed its caller, fetched before the e2e steps reuse the device (untimed)
    last_outputs = {"out": wl.d_out.cpu().numpy(), "out_len": wl.d_len.cpu().numpy()} if args.dump_outputs else None
    wl.barrier()
    ms_total = wl.max_over_ranks(ms_total)
    value = wl.units_total * args.steps / (ms_total * 1e-3)

    # ---- end-to-end: pinned host buffers -> H2D -> solve -> D2H, every step ---------------------------
    for _ in range(args.warmup):
        solver.reset()
        wl.e2e_step()
    e2e_s = wl.max_over_ranks(wl.timed_e2e(args.steps, flush))
    e2e_stream_ms = solver.last_timing()["total_ms"]   # device-side span of the last e2e step (first copy in .. last copy out)
    e2e_val = wl.units_total * args.steps / e2e_s
    h2d = (wl.h_hash.numel() + wl.h_cur.numel()) * 4
    d2h = (wl.h_out.numel() + wl.h_len.numel()) * 4

    e2e_json = None
    if world == 1:
        nj = args.steps
        wl.timed_e2e_json(2, flush)
        js, jbytes = wl.timed_e2e_json(nj, flush)
        e2e_json = {"value": wl.units_total * nj / js, "unit": UNIT, "ms_per_step": 1e3 * js / nj, "json_bytes_per_step": jbytes,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": jbytes,
                    "note": "ka_solve_dense_json: rows stay on the device, the reassignment JSON text (KAG:169-186) is built there and "
                            "streamed out per pipeline block; inputs are the flat slabs (hashes, replicas, names)"}

    # ---- roofline of the dominant kernel (CUDA events recorded around each phase by the library) ------
    peak, peak_src = load_peaks()
    avg = {k: float(np.mean(v)) for k, v in phase.items()}
    dom = max((k for k in avg if k != "level_tables_ms"), key=avg.get)
    kname = {"sticky_spread_ms": "ka_sticky_spread_kernel", "leader_order_ms": "ka_order_levels_kernel<0,...> (slot-0 chain)",
             "slot1_emit_ms": "ka_order_levels_kernel<1,...> (slot-1 chain) + ka_emit3_kernel"}[dom]
    algo_bytes = ALGO_BYTES_PER_UNIT * wl.units_rank
    achieved = algo_bytes / (avg[dom] * 1e-3) / 1e9
    traffic = None   # dram__bytes_read+write of the dominant kernel's launches of ONE step (ncu --cache-control none), like kernel_ms
    tpath = os.path.join(ROOT, "profiles", "traffic_%s.json" % args.workload)
    if os.path.exists(tpath):
        try:
            per = json.load(open(tpath))["per_kernel_dram_bytes_per_step"]
            sym = {"sticky_spread_ms": "ka_sticky_spread_kernel", "leader_order_ms": "ka_order_levels_kernel<0", "slot1_emit_ms": "ka_order_levels_kernel<1"}[dom]
            traffic = sum(v for k, v in per.items() if k.startswith(sym)) or None
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes,
                "kernel_ms": avg[dom], "launches_of_kernel_per_step": "sub-blocks of the pipelined solve; kernel_ms, traffic and algorithmic bytes are per STEP (sums over them)", "phase_ms": avg,
                "per_phase_frac": {k: (algo_bytes / (v * 1e-3) / 1e9) / peak for k, v in avg.items() if v > 0},
                "note": "leader ordering is a serial dependency chain per replica slot through Context.counter (KAS:202-239); phase_ms are "
                        "sums over the pipelined sub-blocks (the slot-0 and slot-1 chains overlap in time); the bound is chain "
                        "latency, not HBM bandwidth — see DESIGN.md"}

    # ---- verification + CPU baseline ------------------------------------------------------------------
    from oracle import oracle_lib as ol
    if rank == 0:
        ol.build()
    wl.barrier()
    verified, cpu_baseline = None, None
    if not args.no_verify:
        if not wl.verify_full(ol):     # h_out / h_len hold the last e2e step's result
            raise SystemExit("bench output differs from the CPU solver (full compare)")
        verified = "full"
    if rank == 0:
        if not args.no_verify:
            sample = cpu_sample(cl, ol, 6.0)
            part_off, part_id, rep_off, cur = sample.ragged()
            o_len, _, o_out, _ = ol.run(ol.OracleContext(), sample.topic_names, part_off, part_id, rep_off, cur, sample.broker_id,
                                        sample.rack_name, -1, S)
            if not np.array_equal(wl.h_out.numpy()[:sample.T].reshape(-1, S), o_out):
                raise SystemExit("bench output differs from the structure-faithful oracle on the first %d topics" % sample.T)
            verified = "full (every row vs oracle/fast_oracle.cpp on every rank) + first %d topics vs oracle/kafka_oracle.cpp" % sample.T
        # the bound that actually applies to the leader-order kernel: barrier-separated levels
        if world == 1 and wl.units_rank <= 12_000_000:
            levels = chain_depth(cl.broker_id, wl.h_out.numpy().reshape(-1, S))
            # measured floor of ONE barrier-separated shared-memory level (tests/tools/micro/level_floor.cu on this B200:
            # 3 x LDS -> compare -> STS -> barrier): 120 cycles with one warp (__syncwarp), 135 with 4 warps, 190 with 8
            warps = max(1, min(32, -(-min(cl.P, 1024) // 32))) if (cl.P * cl.RF <= cl.N) else 1
            floor_cyc = {1: 120, 2: 125, 4: 135, 8: 190}.get(warps)
            ns_level = avg["leader_order_ms"] * 1e6 / levels
            roofline["chain"] = {"dag_depth": levels, "mean_width": wl.units_rank / S / levels,
                                 "ns_per_dag_level_slot0_chain": ns_level,
                                 "measured_floor_ns_per_level": (floor_cyc / 1.965) if floor_cyc else None,
                                 "frac_of_latency_floor": ((floor_cyc / 1.965) / ns_level) if floor_cyc else None,
                                 "note": "exact semantics force one read-decide-bump round trip through the counters per dependency "
                                         "level; the kernel schedules per-topic conflict levels (>= the DAG depth) with one barrier each; "
                                         "floor = micro-benchmark of a bare level at this CTA size (null: not measured for it)"}
        if world == 1 and not args.no_cpu_baseline:
            sample = cpu_sample(cl, ol, 12.0)
            reps = 3 if sample.T == cl.T else 1
            ts = oracle_time(sample, ol, reps)
            cpu_val = sample.replicas / float(np.median(ts))
            # the optimised flat-array CPU solver (oracle/fast_oracle.cpp, BASELINE.md "B1"): the fair CPU yardstick
            fts = []
            for _ in range(3):
                fctx = ol.FastContext()
                t0 = time.perf_counter()
                ol.fast_run_dense(fctx, cl.topic_hash, cl.cur, cl.broker_id, cl.rack_index)
                fts.append(time.perf_counter() - t0)
            cpu_optimized = {"value": cl.replicas / float(np.median(fts)), "unit": UNIT, "cores": 1, "kind": "optimized flat-array port",
                             "sample": "full workload, median of 3, %.4f s each" % float(np.median(fts))}
            cpu_baseline = {"value": cpu_val, "unit": UNIT, "cores": 1, "kind": "port", "optimized": cpu_optimized,
                            "sample": "first %d of %d topics (%d assignments), median of %d run(s), %.2f s each; single thread "
                                      "like the reference (KafkaAssignmentGenerator.java:173); host has %d cores"
                                      % (sample.T, cl.T, sample.replicas, reps, float(np.median(ts)), os.cpu_count())}

    # ---- at 8 GPUs: BASELINE.json config 4 exactly (100k topics x 256, 5k brokers, topic-sharded) ------
    extra = None
    if world == 8 and not args.no_extra and args.workload != "c4shard":
        del wl.d_cur, wl.d_out
        w4 = Workload("c4shard", args.kind, rank, world, local, torch, kab, dist, stream)
        n4 = args.steps
        w4.timed_device(3, flush)
        w4.barrier()
        ms4 = w4.max_over_ranks(w4.timed_device(n4, flush))
        for _ in range(2):
            w4.solver.reset()
            w4.e2e_step()
        e4 = w4.max_over_ranks(w4.timed_e2e(n4, flush))
        ok4 = True if args.no_verify else w4.verify_full(ol)
        if not ok4:
            raise SystemExit("config-4 output differs from the CPU solver (full compare)")
        extra = {"config4_topic_sharded_8gpu": {"workload": workload_desc("c4shard", args.kind, w4.cl) + "; x8 topic blocks = BASELINE config 4",
                                                 "value": w4.units_total * n4 / (ms4 * 1e-3), "ms_per_step": ms4 / n4,
                                                 "e2e_value": w4.units_total * n4 / e4, "e2e_ms_per_step": 1e3 * e4 / n4, "unit": UNIT,
                                                 "steps": n4, "verified_vs_oracle": "full" if not args.no_verify else None}}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": config_desc(args, cl, world, extra),
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s / args.steps, "timer": "host wall clock around the blocking call, max over ranks",
                    "stream_ms_last_step": e2e_stream_ms},
            "e2e_json": e2e_json,
            "gpu_launches": launches,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "verified_vs_oracle": verified,
            "jvm_probe": jvm_probe(),
        }
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if last_outputs is not None:
        dump_outputs(args.dump_outputs, last_outputs, DUMP_BYTES // world, "_rank%d" % rank if rank > 0 else "")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
