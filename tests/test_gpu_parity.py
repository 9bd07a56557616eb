"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle — bit-exact
(all arithmetic on this path is integer). Mirrors the reference's own tests
(KafkaTopicAssignerTest.java:18-157) through the host-side KafkaTopicAssigner mirror, then the golden
fixtures, seeded random clusters, the BASELINE configs and size-independent properties at full size."""
import os
import random

import numpy as np
import pytest

import kafka_assigner_b200 as kab
from tests import util

pytestmark = pytest.mark.gpu

CUR_A = {0: [10, 11], 1: [11, 12], 2: [12, 10], 3: [10, 12]}


def _verify_and_count(cur, new, k=1):  # TEST:159-187
    counts = {}
    for p, reps in new.items():
        assert len(reps) == len(set(reps))
        for b in reps:
            counts[b] = counts.get(b, 0) + 1
        assert len(set(reps) & set(cur[p])) >= k
    return counts


# ---- the reference's four JUnit tests, verbatim shape ---------------------------------------------
def test_rack_aware_expansion(native_lib):
    new = kab.KafkaTopicAssigner().generate_assignment("test", CUR_A, {10, 11, 12, 13, 14},
                                                       {10: "a", 11: "b", 12: "c", 13: "a", 14: "b"}, -1)
    c = _verify_and_count(CUR_A, new)
    assert list(c.values()).count(1) == 2 and list(c.values()).count(2) == 3
    assert new == {0: [10, 11], 1: [11, 12], 2: [12, 13], 3: [14, 10]}


def test_cluster_expansion(native_lib):
    new = kab.KafkaTopicAssigner().generate_assignment("test", CUR_A, {10, 11, 12, 13}, {}, -1)
    assert all(v == 2 for v in _verify_and_count(CUR_A, new).values())


def test_decommission(native_lib):
    cur = {0: [10, 11], 1: [11, 12], 2: [12, 13], 3: [13, 10]}
    new = kab.KafkaTopicAssigner().generate_assignment("test", cur, {10, 11, 13}, {}, -1)
    c = _verify_and_count(cur, new)
    assert 12 not in c and sorted(c.values()) == [2, 3, 3]


def test_replacement(native_lib):
    new = kab.KafkaTopicAssigner().generate_assignment("test", CUR_A, {10, 11, 13}, {}, -1)
    c = _verify_and_count(CUR_A, new)
    assert 12 not in c
    assert new[0] == CUR_A[0]  # TEST:143-144, the reference's only exact pin
    assert 11 in new[1] and (10 in new[1] or 13 in new[1])
    assert 10 in new[2] and (11 in new[2] or 13 in new[2])
    assert 10 in new[3] and (11 in new[3] or 13 in new[3])


def test_assigner_instance_keeps_context_across_calls(native_lib):
    """ONE assigner == ONE Context (KTA:19-23): leadership depends on topic order (SURVEY §3.2)."""
    A = {0: [3, 1], 1: [4, 3], 2: [1, 4]}
    B = {0: [1, 2], 1: [1, 3], 2: [2, 1]}
    asg = kab.KafkaTopicAssigner()
    a1 = asg.generate_assignment("a", A, {1, 2, 3, 4}, {}, -1)
    b1 = asg.generate_assignment("b", B, {1, 2, 3, 4}, {}, -1)
    assert a1 == {0: [3, 1], 1: [4, 3], 2: [1, 4]} and b1 == {0: [2, 1], 1: [1, 3], 2: [2, 3]}
    asg2 = kab.KafkaTopicAssigner()
    b2 = asg2.generate_assignment("b", B, {1, 2, 3, 4}, {}, -1)
    a2 = asg2.generate_assignment("a", A, {1, 2, 3, 4}, {}, -1)
    assert b2 == {0: [1, 2], 1: [3, 1], 2: [2, 3]} and a2[2] == [4, 1]


def test_error_messages_match_reference(native_lib):
    asg = kab.KafkaTopicAssigner()
    with pytest.raises(kab.IllegalStateException, match=r"^Topic t has partition 1 with unexpected replication factor 1$"):
        asg.generate_assignment("t", {0: [1, 2], 1: [1]}, {1, 2, 3}, {}, -1)
    with pytest.raises(kab.IllegalStateException, match=r"^Topic t does not have a positive replication factor!$"):
        asg.generate_assignment("t", {}, {1, 2, 3}, {}, -1)
    with pytest.raises(kab.IllegalStateException, match=r"^Topic t has a higher replication factor \(3\) than available brokers!$"):
        asg.generate_assignment("t", {0: [1, 2, 3]}, {1, 2}, {}, -1)
    with pytest.raises(kab.IllegalStateException, match=r"^Partition 0 could not be fully assigned!$"):
        asg.generate_assignment("t", {0: [1, 2], 1: [2, 1]}, {1, 2, 3}, {1: "x", 2: "x", 3: "y"}, 3)
    with pytest.raises(kab.ArrayIndexOutOfBoundsException, match=r"^-2$"):
        asg.generate_assignment("polygenelubricants", {0: [1, 2, 3]}, {1, 2, 3}, {}, -1)


# ---- committed golden fixtures + the oracle on the same inputs -------------------------------------
def test_golden_fixtures(native_lib, oracle):
    for c in util.load_golden():
        got = util.run_gpu_case(kab, c)
        exp = c["expected"]
        if "error" in exp:
            assert "error" in got, c["name"]
            assert got["error"] == exp["error"], c["name"]
        else:
            assert got.get("records") == exp["records"], c["name"]
        assert {k: v for k, v in util.run_oracle_case(oracle, c).items() if k != "topic_index"} == \
               {k: v for k, v in got.items() if k != "topic_index"}, c["name"]


def test_random_ragged_cases_vs_oracle(native_lib, oracle):
    rng = random.Random(11)
    solver = kab.Solver(0)
    n_ok = n_err = 0
    for it in range(300):
        solver.reset()
        nb = rng.randint(1, 40)
        brokers = sorted(rng.sample(range(-5, 200), nb))
        racks = {b: "k%d" % rng.randrange(max(2, nb // 3)) for b in brokers if rng.random() < 0.7}
        universe = brokers + [1000, 1001, -77]
        topics = []
        for ti in range(rng.randint(1, 6)):
            rf = rng.randint(1, min(5, nb))
            ragged = rng.random() < 0.25
            cur = {}
            for p in sorted(rng.sample(range(0, 80), rng.randint(0 if rng.random() < 0.05 else 1, 70))):
                k = rng.randint(0, 5) if ragged else rf
                cur[p] = rng.sample(universe, min(k, len(universe)))
            topics.append(("rt%d_%d" % (it, ti), cur))
        desired = rng.choice([-1, -1, -1, -1, 1, 2, 3, 4, 0])
        case = dict(topics=topics, brokers=brokers, racks=racks, desired_rf=desired)
        exp = util.run_oracle_case(oracle, case)
        got = util.run_gpu_case(kab, case, solver)
        assert got == exp, (it, case)
        n_ok += "records" in exp
        n_err += "error" in exp
    assert n_ok > 40 and n_err > 20


@pytest.mark.parametrize("kind", ["structured", "random", "mixed"])
@pytest.mark.parametrize("shape", [dict(T=7, P=5, RF=2, N=9, R=3), dict(T=40, P=33, RF=3, N=64, R=8),
                                   dict(T=16, P=100, RF=3, N=30, R=6), dict(T=5, P=300, RF=4, N=1200, R=12),
                                   dict(T=64, P=17, RF=1, N=11, R=11), dict(T=12, P=96, RF=5, N=35, R=7)])
def test_dense_clusters_vs_oracle(native_lib, oracle, shape, kind):
    cl = kab.synth.make_cluster(seed=0xABC + shape["T"], kind=kind, **shape)
    exp_out, exp_len, est = util.oracle_dense(oracle, cl)
    s = kab.Solver(0)
    out, out_len, st = s.solve_cluster(cl, check=False)
    assert st.code == est.code and st.topic_index == est.topic_index
    if est.code == 0:
        assert np.array_equal(out.reshape(-1, cl.RF), exp_out)
        assert np.array_equal(out_len.reshape(-1), exp_len)


def test_rack_awareness_disabled_and_decommission(native_lib, oracle):
    for P, expect_ok in ((44, True), (48, False)):  # P=48: zero slack -> the reference itself throws (KAS:183-184)
        cl = kab.synth.make_cluster(T=30, P=P, RF=3, N=60, R=6, seed=5, kind="mixed", rack_aware=False, remove_frac=0.2, n_old=60)
        exp_out, exp_len, est = util.oracle_dense(oracle, cl)
        out, out_len, st = kab.Solver(0).solve_cluster(cl, check=False)
        assert (est.code == 0) == expect_ok
        assert (st.code, st.topic_index, st.partition) == (est.code, est.topic_index, est.partition)
        if expect_ok:
            assert np.array_equal(out.reshape(-1, 3), exp_out)
            assert not np.isin(out, np.setdiff1d(1000 + np.arange(60), cl.broker_id)).any()  # removed brokers are gone


def test_context_persists_across_batches_and_broker_changes(native_lib, oracle):
    """Counters are keyed by broker id: split a run into batches, change the broker set in between."""
    cl = kab.synth.make_cluster(T=20, P=24, RF=3, N=40, R=5, seed=9, kind="mixed")
    octx = oracle.OracleContext()
    s = kab.Solver(0)
    a, b = cl.subset(0, 8), cl.subset(8, 20)
    ea, _, _ = util.oracle_dense(oracle, a, octx)
    ga, _, _ = s.solve_cluster(a)
    assert np.array_equal(ga.reshape(-1, 3), ea)
    # second batch on a smaller live set (decommission 1 per rack): counters must carry over by id
    b2 = kab.synth.make_cluster(T=20, P=24, RF=3, N=40, R=5, seed=9, kind="mixed", remove_frac=1 / 8.0).subset(8, 20)
    eb, _, est = util.oracle_dense(oracle, b2, octx)
    gb, _, st = s.solve_cluster(b2, check=False)
    assert st.code == est.code == 0
    assert np.array_equal(gb.reshape(-1, 3), eb)
    ctr = s.counters()
    for i, bid in enumerate(b2.broker_id):
        for slot in range(3):
            assert ctr[i, slot] == octx.counter(int(bid), slot)


def test_baseline_config1_and_config2_bit_exact(native_lib, oracle):
    for key in ("c1", "c2"):
        for kind in ("structured", "random", "mixed"):
            cl = kab.synth.make_config(key, kind)
            exp_out, exp_len, est = util.oracle_dense(oracle, cl)
            out, out_len, st = kab.Solver(0).solve_cluster(cl, check=False)
            assert st.code == est.code == 0, (key, kind)
            assert np.array_equal(out.reshape(-1, 3), exp_out), (key, kind)


def _full_compare(oracle, cl, prefix_topics=200, solver=None):
    """EVERY output row of `cl` against the flat-array CPU solver (pinned to the structure-faithful oracle on these shapes
    in tests/test_oracle.py::test_fast_solver_pinned_on_baseline_shapes), plus a topic prefix against kafka_oracle.cpp."""
    s = solver or kab.Solver(0)
    out, out_len, st = s.solve_cluster(cl, check=False)
    exp, exp_len, est = oracle.fast_run_dense(oracle.FastContext(), cl.topic_hash, cl.cur, cl.broker_id, cl.rack_index)
    assert st.code == est.code == 0, (cl.name, st.code, est.code)
    assert np.array_equal(out.reshape(-1, cl.RF), exp), cl.name
    assert np.array_equal(out_len.reshape(-1), exp_len), cl.name
    n = min(cl.T, prefix_topics)
    pre, _, pst = util.oracle_dense(oracle, cl.subset(0, n))
    assert pst.code == 0 and np.array_equal(out[:n].reshape(-1, cl.RF), pre), cl.name
    return s, out, out_len


@pytest.mark.parametrize("kind", ["structured", "random", "mixed"])
def test_baseline_config3_full_bit_exact(native_lib, oracle, kind):
    """BASELINE config 3 (10k topics x 128, 1k brokers / 20 racks) in full: all 1.28 M rows."""
    _full_compare(oracle, kab.synth.make_config("c3", kind))


def test_baseline_config4_shard_full_bit_exact(native_lib, oracle):
    """One GPU's eighth of BASELINE config 4 (12.5k topics x 256, 5k brokers / 50 racks) in full."""
    _full_compare(oracle, kab.synth.make_config("c4shard", "mixed"))


def test_baseline_config4_full_bit_exact_on_one_gpu(native_lib, oracle):
    """BASELINE config 4 itself (100k topics x 256 = 76.8 M assignments, 25.6 M rows) through one Context on one GPU."""
    cl = kab.synth.make_config("c4", "mixed")
    _full_compare(oracle, cl, prefix_topics=100)


@pytest.mark.parametrize("frac", [0.01, 0.2, 0.5])
def test_baseline_config5_full_bit_exact(native_lib, oracle, frac):
    """BASELINE config 5 (decommission sweep: 1 M partitions on 10k brokers / 50 racks, a fraction of every rack removed)."""
    cl = kab.synth.make_config("c5", "mixed", remove_frac=frac)
    s, out, _ = _full_compare(oracle, cl, prefix_topics=12)
    assert not np.isin(out, np.setdiff1d(1000 + np.arange(10000), cl.broker_id)).any()


def _check_properties(cl, out, out_len):
    """Size-independent invariants of the reference algorithm (usable at full BASELINE sizes)."""
    T, P, RF, N = cl.T, cl.P, cl.RF, cl.N
    assert (out_len == RF).all()
    idx = np.searchsorted(cl.broker_id, out)
    assert (cl.broker_id[np.clip(idx, 0, N - 1)] == out).all()            # only live brokers
    racks = cl.rack_index[idx]
    srt = np.sort(racks, axis=2)
    assert (srt[:, :, 1:] != srt[:, :, :-1]).all()                        # one replica per rack (KAS:346-348)
    cap = -(-P * RF // N)
    flat = (idx.reshape(T, -1) + (np.arange(T)[:, None] * N)).reshape(-1)
    loads = np.bincount(flat, minlength=T * N).reshape(T, N)
    assert loads.max() <= cap                                            # per-topic capacity (KAS:65-71)
    # stickiness: a current replica on a live broker is kept unless capacity/rack forced it out; at least
    # every partition whose current brokers are all live & under cap keeps >= 1 (TEST:181-184 analogue)
    kept = (out[:, :, :, None] == cl.cur[:, :, None, :]).any(axis=3).sum(axis=2)
    assert kept.mean() > 0.5
    # leader counters: per (broker, slot) totals equal the final Context.counter
    return np.stack([np.bincount(idx[:, :, r].reshape(-1), minlength=N) for r in range(RF)], axis=1)


def test_baseline_config3_full_properties_and_idempotent_counters(native_lib):
    cl = kab.synth.make_config("c3", "mixed")
    s = kab.Solver(0)
    out, out_len, st = s.solve_cluster(cl)
    slot_counts = _check_properties(cl, out, out_len)
    assert np.array_equal(s.counters()[:, :3], slot_counts)
    assert slot_counts.sum() == cl.replicas
    # determinism: same input, fresh context -> identical bytes
    out2, _, _ = kab.Solver(0).solve_cluster(cl)
    assert np.array_equal(out, out2)


def test_device_resident_entry_matches_host_entry(native_lib):
    import torch
    cl = kab.synth.make_config("c2", "mixed")
    host_out, _, _ = kab.Solver(0).solve_cluster(cl)
    s = kab.Solver(0)
    s.set_brokers(cl.broker_id, cl.rack_index)
    d_hash = torch.from_numpy(cl.topic_hash).cuda()
    d_cur = torch.from_numpy(cl.cur).cuda()
    d_out = torch.empty((cl.T, cl.P, cl.RF), dtype=torch.int32, device="cuda")
    d_len = torch.empty((cl.T, cl.P), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    st = s.solve_dense_device(cl.T, d_hash.data_ptr(), cl.P, cl.RF, d_cur.data_ptr(), -1, cl.RF, d_len.data_ptr(),
                              d_out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    assert st.code == 0
    assert np.array_equal(d_out.cpu().numpy(), host_out)
    assert (d_len.cpu().numpy() == 3).all()


def test_stage_order_split_and_counter_ring_on_one_gpu(native_lib, oracle):
    """The multi-GPU protocol with two contexts on one device: block 0 and block 1 staged independently,
    leader ordering chained through exported/imported counters == one run over all topics."""
    import torch
    from kafka_assigner_b200 import multi
    full = kab.synth.make_cluster(T=60, P=40, RF=3, N=50, R=5, seed=31, kind="mixed")
    exp, _, est = util.oracle_dense(oracle, full)
    assert est.code == 0
    world = 2
    solvers, blocks, outs = [], [], []
    for r in range(world):
        t0, t1 = multi.shard_range(full.T, world, r)
        cl = kab.synth.make_cluster(T=t1 - t0, P=40, RF=3, N=50, R=5, seed=31, kind="mixed", t_offset=t0)
        s = kab.Solver(0)
        s.set_brokers(cl.broker_id, cl.rack_index)
        blocks.append((cl, torch.from_numpy(cl.topic_hash).cuda(), torch.from_numpy(cl.cur).cuda(),
                       torch.empty((cl.T, cl.P, 3), dtype=torch.int32, device="cuda")))
        solvers.append(s)
    buf = torch.zeros(50 * 8, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    for r in range(world):  # stage everything first (no Context involved) ...
        cl, dh, dc, do = blocks[r]
        solvers[r].stage_dense_device(cl.T, dh.data_ptr(), cl.P, cl.RF, dc.data_ptr(), -1, 3)
    for r in range(world):  # ... then the serial chain
        cl, dh, dc, do = blocks[r]
        if r > 0:
            solvers[r].import_counters_device(buf.data_ptr())
        st = solvers[r].order_device(0, do.data_ptr())
        assert st.code == 0
        solvers[r].export_counters_device(buf.data_ptr())
        torch.cuda.synchronize()
        outs.append(do.cpu().numpy().reshape(-1, 3))
    assert np.array_equal(np.concatenate(outs), exp)


def test_per_slot_ring_on_one_gpu(native_lib, oracle):
    """The topic-sharded protocol of multi.ring_solve_phases with three contexts on one device: every block staged
    independently, then the slot-0 chain block after block (handing on counter[.][0] only), then the slot-1 chain the same
    way, then the emits; counter[.][2] is the sum over the blocks. Output and final Context == one run over all topics."""
    import torch
    from kafka_assigner_b200 import multi
    for shape in (dict(T=90, P=40, RF=3, N=50, R=5), dict(T=64, P=16, RF=3, N=120, R=6)):   # capacity 3 (levels) / capacity 1
        full = kab.synth.make_cluster(seed=47, kind="mixed", **shape)
        octx = oracle.OracleContext()
        exp, _, est = util.oracle_dense(oracle, full, octx)
        assert est.code == 0
        world, N = 3, full.N
        solvers, blocks = [], []
        for r in range(world):
            t0, t1 = multi.shard_range(full.T, world, r)
            cl = kab.synth.make_cluster(seed=47, kind="mixed", t_offset=t0, **dict(shape, T=t1 - t0))
            s = kab.Solver(0)
            s.set_brokers(cl.broker_id, cl.rack_index)
            s.set_topic_base(t0)
            blocks.append((cl, torch.from_numpy(cl.topic_hash).cuda(), torch.from_numpy(cl.cur).cuda(),
                           torch.empty((cl.T, cl.P, 3), dtype=torch.int32, device="cuda"), torch.empty((cl.T, cl.P), dtype=torch.int32, device="cuda")))
            solvers.append(s)
        col = torch.zeros(N, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        for r in range(world):
            cl, dh, dc, do, dl = blocks[r]
            solvers[r].stage_dense_device(cl.T, dh.data_ptr(), cl.P, cl.RF, dc.data_ptr(), -1, 3)
            assert solvers[r].staged_slot_chains() == 2
        for slot in (0, 1):
            for r in range(world):
                if r > 0:
                    solvers[r].import_counter_slot_device(slot, col.data_ptr())
                solvers[r].order_slot_device(slot)
                solvers[r].export_counter_slot_device(slot, col.data_ptr())
        outs = []
        for r in range(world):
            cl, dh, dc, do, dl = blocks[r]
            st = solvers[r].emit_device(dl.data_ptr(), do.data_ptr())
            assert st.code == 0
            outs.append(do.cpu().numpy().reshape(-1, 3))
            assert (dl.cpu().numpy() == 3).all()
        assert np.array_equal(np.concatenate(outs), exp), shape
        ctrs = [s.counters() for s in solvers]
        final = ctrs[-1].copy()
        final[:, 2] = sum(c[:, 2] for c in ctrs)
        for i, bid in enumerate(full.broker_id):
            for slot in range(3):
                assert final[i, slot] == octx.counter(int(bid), slot), (shape, int(bid), slot)


def _expected_json(cl, out, out_len):
    """KafkaAssignmentGenerator.java:169-186 in the predicted org.json key order (SURVEY §3.4), built on the host."""
    rows = out.reshape(cl.T, cl.P, -1)
    lens = out_len.reshape(cl.T, cl.P)
    parts = []
    for t, name in enumerate(cl.topic_names):
        for p in range(cl.P):
            parts.append('{"partition":%d,"replicas":[%s],"topic":"%s"}' % (p, ",".join(str(int(b)) for b in rows[t, p, :lens[t, p]]), name))
    return '{"partitions":[' + ",".join(parts) + '],"version":1}'


def test_device_json_emitter_byte_for_byte(native_lib, oracle):
    """ka_solve_dense_json: solve + JSON text on the device, streamed per pipeline block — byte-for-byte against the text built
    from the oracle's rows, on BASELINE config 2 in full, a pipelined run (3 blocks), odd shapes, and the empty run."""
    for cl, env in ((kab.synth.make_config("c2", "mixed"), None), (kab.synth.make_cluster(T=7, P=5, RF=2, N=9, R=3, seed=5, kind="random"), None),
                    (kab.synth.make_cluster(T=1, P=1, RF=1, N=3, R=3, seed=6, kind="random"), None)):
        exp_out, exp_len, est = util.oracle_dense(oracle, cl)
        assert est.code == 0
        s = kab.Solver(0)
        s.set_brokers(cl.broker_id, cl.rack_index)
        text, st = s.solve_dense_json(cl.topic_names, cl.topic_hash, cl.cur)
        assert st.code == 0
        assert bytes(text).decode() == _expected_json(cl, exp_out, exp_len), cl.name
    # a failing topic: the reference prints no NEW ASSIGNMENT at all (KAG:186 is never reached)
    bad = kab.synth.make_cluster(T=6, P=4, RF=3, N=9, R=3, seed=8, kind="random")
    s = kab.Solver(0)
    s.set_brokers(bad.broker_id[:2], bad.rack_index[:2])
    text, st = s.solve_dense_json(bad.topic_names, bad.topic_hash, bad.cur, check=False)
    assert st.code == 3 and len(text) == 0  # KA_ERR_RF_GT_BROKERS


def test_device_json_emitter_pipelined_blocks(native_lib, oracle):
    import subprocess, sys
    code = ("import numpy as np, kafka_assigner_b200 as kab\n"
            "from oracle import oracle_lib as ol\n"
            "from tests import util\n"
            "from tests.test_gpu_parity import _expected_json\n"
            "cl = kab.synth.make_cluster(T=300, P=24, RF=3, N=40, R=5, seed=77, kind='mixed')\n"
            "exp, ln, st = util.oracle_dense(ol, cl)\n"
            "s = kab.Solver(0); s.set_brokers(cl.broker_id, cl.rack_index)\n"
            "text, st = s.solve_dense_json(cl.topic_names, cl.topic_hash, cl.cur)\n"
            "assert bytes(text).decode() == _expected_json(cl, exp, ln)\n"
            "print('OK')\n")
    env = dict(os.environ, KA_PIPELINE_STAGES="3", PYTHONPATH=util.os.path.dirname(util.HERE))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


# ---- less-travelled code paths ----------------------------------------------------------------------------------------
def _random_case(rng, broker_ids, n_topics, max_rf, max_parts=40, rack_groups=None, desired=-1):
    racks = {}
    if rack_groups:
        for b in broker_ids:
            if rng.random() < 0.85:
                racks[b] = "g%d" % rng.randrange(rack_groups)
    topics = []
    universe = list(broker_ids) + [broker_ids[0] - 7, broker_ids[-1] + 11]
    for ti in range(n_topics):
        rf = rng.randint(1, min(max_rf, len(broker_ids)))
        cur = {p: rng.sample(universe, min(rf, len(universe))) for p in sorted(rng.sample(range(0, 200), rng.randint(1, max_parts)))}
        topics.append(("lt%d" % ti, cur))
    return dict(topics=topics, brokers=list(broker_ids), racks=racks, desired_rf=desired)


def test_broker_id_lookup_modes(native_lib, oracle):
    """id -> index lookup: smem LUT (dense ids), global LUT (range > 32768), binary search (range > 2^25)."""
    rng = random.Random(5)
    dense = sorted(rng.sample(range(100, 400), 60))
    wide = sorted(rng.sample(range(-40000, 40000), 60))                 # range ~80k  -> global LUT
    huge = sorted(rng.sample(range(-2**31 + 5, 2**31 - 5), 60))        # range ~4e9  -> binary search
    for ids in (dense, wide, huge):
        for it in range(6):
            case = _random_case(rng, ids, n_topics=4, max_rf=4, rack_groups=rng.choice([None, 7, 20]))
            exp = util.run_oracle_case(oracle, case)
            got = util.run_gpu_case(kab, case)
            assert got == exp, (ids[:3], it)


def test_wide_rows_five_to_eight_replicas(native_lib, oracle):
    """Lists of 5..8 replicas use the generic 8-slot leader-order kernel."""
    rng = random.Random(8)
    ids = list(range(1, 41))
    n_ok = 0
    for it in range(12):
        case = _random_case(rng, ids, n_topics=3, max_rf=8, max_parts=25, rack_groups=rng.choice([None, 12, 40]))
        exp = util.run_oracle_case(oracle, case)
        got = util.run_gpu_case(kab, case)
        assert got == exp, it
        n_ok += "records" in exp
    assert n_ok >= 3
    # replication-factor growth to 6 via --desired_replication_factor
    case = _random_case(rng, ids, n_topics=3, max_rf=3, max_parts=20, rack_groups=None, desired=6)
    assert util.run_gpu_case(kab, case) == util.run_oracle_case(oracle, case)


def test_degenerate_shapes(native_lib, oracle):
    s = kab.Solver(0)
    # zero topics
    s.set_brokers(np.array([1, 2, 3], dtype=np.int32), np.array([0, 1, 2], dtype=np.int32))
    out, out_len, st = s.solve_dense(np.zeros(0, dtype=np.int32), np.zeros((0, 4, 2), dtype=np.int32))
    assert st.code == 0 and out.shape == (0, 4, 2)
    # single broker, RF 1
    case = dict(topics=[("solo", {0: [9], 1: [9], 5: [4]})], brokers=[9], racks={}, desired_rf=-1)
    assert util.run_gpu_case(kab, case) == util.run_oracle_case(oracle, case)
    # topic with an empty partition map between two good topics: fails at that topic (KTA:65-66)
    case = dict(topics=[("a", {0: [1, 2]}), ("empty", {}), ("b", {0: [2, 3]})], brokers=[1, 2, 3], racks={}, desired_rf=-1)
    got, exp = util.run_gpu_case(kab, case), util.run_oracle_case(oracle, case)
    assert got == exp and exp["topic_index"] == 1
    # ... but with a desired RF an empty topic is fine and yields no rows
    case["desired_rf"] = 2
    assert util.run_gpu_case(kab, case) == util.run_oracle_case(oracle, case)
    # every current broker dead: everything is an orphan
    case = dict(topics=[("dead", {p: [100 + p, 200 + p] for p in range(6)})], brokers=[1, 2, 3, 4], racks={1: "x", 2: "y"}, desired_rf=-1)
    assert util.run_gpu_case(kab, case) == util.run_oracle_case(oracle, case)
    # duplicate broker inside a current list (second copy is dropped, KAS:320-324)
    case = dict(topics=[("dup", {0: [1, 1], 1: [2, 2], 2: [1, 2]})], brokers=[1, 2, 3], racks={}, desired_rf=-1)
    assert util.run_gpu_case(kab, case) == util.run_oracle_case(oracle, case)
    # limits are reported, not silently mishandled
    with pytest.raises(kab.KassignError):
        kab.KafkaTopicAssigner().generate_assignment("big", {0: list(range(1, 10))}, set(range(1, 12)), {}, -1)  # 9 replicas > 8 slots


def test_rack_pointer_spread_variant_is_exact(native_lib, oracle, tmp_path):
    """The opt-in per-rack-pointer spread (KA_SPREAD_RACKPTR=1) must give the same bytes as the default window scan."""
    import subprocess
    import sys
    code = ("import os, sys, numpy as np, kafka_assigner_b200 as kab\n"
            "for key, kind in (('c1','random'), ('c2','mixed')):\n"
            "    cl = kab.synth.make_config(key, kind)\n"
            "    out, _, st = kab.Solver(0).solve_cluster(cl)\n"
            "    np.save(os.path.join(sys.argv[1], '_rp_%s.npy' % key), out)\n")
    env = dict(os.environ, KA_SPREAD_RACKPTR="1", PYTHONPATH=util.os.path.dirname(util.HERE))
    subprocess.run([sys.executable, "-c", code, str(tmp_path)], check=True, env=env, timeout=300)
    for key, kind in (("c1", "random"), ("c2", "mixed")):
        cl = kab.synth.make_config(key, kind)
        exp, _, _ = util.oracle_dense(oracle, cl)
        assert np.array_equal(np.load(tmp_path / ("_rp_%s.npy" % key)).reshape(-1, 3), exp)


def test_pipelined_super_chunks_are_exact(native_lib, oracle, tmp_path):
    """KA_PIPELINE_STAGES=3 forces the two-stream super-chunk pipeline on small problems: same bytes, same counters,
    and a failure in a later chunk is reported with its GLOBAL topic index."""
    import subprocess
    import sys
    code = ("import os, sys, numpy as np, kafka_assigner_b200 as kab\n"
            "d = sys.argv[1]\n"
            "for key, kind in (('c1','mixed'), ('c2','mixed'), ('c2','random')):\n"
            "    cl = kab.synth.make_config(key, kind)\n"
            "    s = kab.Solver(0)\n"
            "    out, out_len, st = s.solve_cluster(cl)\n"
            "    np.save(os.path.join(d, '_pl_%s_%s.npy' % (key, kind)), out)\n"
            "    np.save(os.path.join(d, '_plc_%s_%s.npy' % (key, kind)), s.counters())\n"
            "bad = kab.synth.make_cluster(T=30, P=48, RF=3, N=60, R=6, seed=21, kind='mixed', rack_aware=False, remove_frac=0.2, n_old=60)\n"
            "_, _, st = kab.Solver(0).solve_cluster(bad, check=False)\n"
            "np.save(os.path.join(d, '_pl_bad.npy'), np.array([st.code, st.topic_index, st.partition]))\n")
    env = dict(os.environ, KA_PIPELINE_STAGES="3", PYTHONPATH=util.os.path.dirname(util.HERE))
    subprocess.run([sys.executable, "-c", code, str(tmp_path)], check=True, env=env, timeout=300)
    for key, kind in (("c1", "mixed"), ("c2", "mixed"), ("c2", "random")):
        cl = kab.synth.make_config(key, kind)
        octx = oracle.OracleContext()
        exp, _, _ = util.oracle_dense(oracle, cl, octx)
        assert np.array_equal(np.load(tmp_path / ("_pl_%s_%s.npy" % (key, kind))).reshape(-1, 3), exp), (key, kind)
        ctr = np.load(tmp_path / ("_plc_%s_%s.npy" % (key, kind)))
        for i in range(0, cl.N, 7):
            for slot in range(3):
                assert ctr[i, slot] == octx.counter(int(cl.broker_id[i]), slot)
    bad = kab.synth.make_cluster(T=30, P=48, RF=3, N=60, R=6, seed=21, kind="mixed", rack_aware=False, remove_frac=0.2, n_old=60)
    _, _, est = util.oracle_dense(oracle, bad)
    assert est.code == 4 and est.topic_index >= 10      # fails in the 2nd or 3rd chunk of 3
    assert np.load(tmp_path / "_pl_bad.npy").tolist() == [est.code, est.topic_index, est.partition]


def test_broker_tables_beyond_shared_memory(native_lib, oracle):
    """VERDICT r1 #8: N = 20 000 (counter columns still in shared memory) and N = 60 000 (global id->index LUT in kernel A,
    counter columns in global memory for the chains — the GCTR path) must give the reference's answer, not KA_ERR_LIMIT."""
    for N, R, T, P in ((20000, 50, 24, 300), (60000, 60, 6, 700)):
        cl = kab.synth.make_cluster(T=T, P=P, RF=3, N=N, R=R, seed=0xB16 + N, kind="mixed")
        exp, exp_len, est = oracle.fast_run_dense(oracle.FastContext(), cl.topic_hash, cl.cur, cl.broker_id, cl.rack_index)
        assert est.code == 0
        out, out_len, st = kab.Solver(0).solve_cluster(cl, check=False)
        assert st.code == 0, (N, st.code, st.a, st.b)
        assert np.array_equal(out.reshape(-1, 3), exp) and np.array_equal(out_len.reshape(-1), exp_len), N
    # conflict levels (capacity 3) + chunk tables + window / general chunking, all with the counters forced into global memory
    import subprocess, sys
    code = ("import numpy as np, kafka_assigner_b200 as kab\n"
            "from oracle import oracle_lib as ol\n"
            "for T, P, N, R in ((40, 500, 600, 6), (200, 21, 40, 5), (12, 2500, 3000, 10)):\n"
            "    cl = kab.synth.make_cluster(T=T, P=P, RF=3, N=N, R=R, seed=0xB17, kind='mixed')\n"
            "    exp, ln, est = ol.fast_run_dense(ol.FastContext(), cl.topic_hash, cl.cur, cl.broker_id, cl.rack_index)\n"
            "    out, out_len, st = kab.Solver(0).solve_cluster(cl, check=False)\n"
            "    assert st.code == est.code == 0, (st.code, est.code)\n"
            "    assert np.array_equal(out.reshape(-1, 3), exp), (T, P, N)\n"
            "print('OK')\n")
    env = dict(os.environ, KA_ORDER_GLOBAL_CTR="1", PYTHONPATH=util.os.path.dirname(util.HERE))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


def test_large_capacity_load_counters_and_size_limit(native_lib, oracle):
    """cap = ceil(P*RF/N) > 255 switches kernel A's per-broker load counters to 16-bit; absurd sizes are refused."""
    cl = kab.synth.make_cluster(T=3, P=700, RF=2, N=4, R=2, seed=12, kind="random", n_old=4)   # cap = 350
    exp, exp_len, est = util.oracle_dense(oracle, cl)
    out, out_len, st = kab.Solver(0).solve_cluster(cl, check=False)
    assert (st.code, st.topic_index, st.partition) == (est.code, est.topic_index, est.partition)
    if est.code == 0:
        assert np.array_equal(out.reshape(-1, 2), exp)
    # one topic with 200k partitions does not fit a warp's shared-memory slab: a clean KA_ERR_LIMIT, not a crash
    s = kab.Solver(0)
    s.set_brokers(np.arange(1, 9, dtype=np.int32), np.arange(8, dtype=np.int32) % 4)
    cur = np.tile(np.array([[1, 2]], dtype=np.int32), (1, 200000, 1))
    _, _, st = s.solve_dense(np.array([7], dtype=np.int32), cur, check=False)
    assert st.code == kab._native.KA_ERR_LIMIT
