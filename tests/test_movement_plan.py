"""Movement plan of a solve (ka_plan_last) and the changed-rows-only reassignment JSON (ka_solve_dense_json_changed).

A numpy model of the definitions in include/kassign.h lives here and is pinned on hand cases (CPU). The GPU tests compare
the device plan, exactly, with the model applied to the oracle's rows, and the changed-only text with the full text minus
its unchanged rows."""
import dataclasses
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import kafka_assigner_b200 as kab
from tests import util

_PAD_C, _PAD_O = 1 << 40, 1 << 41   # never equal to each other or to an int32 broker id


def plan_model(C, lc, O, lo, report_ids):
    """The movement plan of rows with current lists C[q, :lc[q]] and new lists O[q, :lo[q]] (leader first).
    Returns (totals dict, stats [M + 1, 8] int64, row_class [Q], number of rows with an empty current list)."""
    lc = np.asarray(lc, dtype=np.int64)
    lo = np.asarray(lo, dtype=np.int64)
    Q = len(lc)
    C = np.asarray(C, dtype=np.int64).reshape(Q, -1)
    O = np.asarray(O, dtype=np.int64).reshape(Q, -1)
    L = max(C.shape[1], O.shape[1], 1)
    pos = np.arange(L)[None, :]
    cv, ov = pos < lc[:, None], pos < lo[:, None]
    Cp = np.full((Q, L), _PAD_C, dtype=np.int64)
    Op = np.full((Q, L), _PAD_O, dtype=np.int64)
    Cp[:, :C.shape[1]] = C
    Op[:, :O.shape[1]] = O
    Cp[~cv] = _PAD_C
    Op[~ov] = _PAD_O
    eq = Cp[:, :, None] == Op[:, None, :]
    c_in_o = eq.any(axis=2) & cv
    o_in_c = eq.any(axis=1) & ov
    earlier = np.tril(np.ones((L, L), dtype=bool), -1)[None]
    c_first = cv & ~((Cp[:, :, None] == Cp[:, None, :]) & earlier).any(axis=2)
    same = (lc == lo) & ((Cp == Op) | ~cv).all(axis=1)
    added = (ov & ~o_in_c).sum(axis=1)
    dropped = (c_first & ~c_in_o).sum(axis=1)
    cls = np.where(same, 0, np.where((added > 0) | (dropped > 0) | (lc != lo), 2, 1)).astype(np.uint8)
    lead = (lo > 0) & ((lc == 0) | (Cp[:, 0] != Op[:, 0]))
    ids = np.asarray(report_ids, dtype=np.int64)
    M = len(ids)

    def count(vals):
        i = np.searchsorted(ids, vals)
        ok = i < M
        ok[ok] = ids[i[ok]] == vals[ok]
        return np.bincount(np.where(ok, i, M), minlength=M + 1)

    stats = np.stack([count(Cp[c_first]), count(Op[ov]), count(Op[ov & ~o_in_c]), count(Cp[c_first & ~c_in_o]),
                      count(Cp[lc > 0, 0]), count(Op[lo > 0, 0]), count(Op[lead, 0]), count(Cp[lead & (lc > 0), 0])], axis=1)
    totals = dict(rows=Q, rows_reordered=int((cls == 1).sum()), rows_moved=int((cls == 2).sum()),
                  replicas_added=int(added.sum()), replicas_dropped=int(dropped.sum()), leaders_changed=int(lead.sum()))
    return totals, stats, cls, int(((lc == 0) & (lo > 0)).sum())


def check_invariants(totals, stats, empty_rows=0):
    s = np.asarray(stats, dtype=np.int64)
    assert (s[:, 1] == s[:, 0] + s[:, 2] - s[:, 3]).all()
    assert (s[:, 5] == s[:, 4] + s[:, 6] - s[:, 7]).all()
    assert s[:, 2].sum() == totals["replicas_added"] and s[:, 3].sum() == totals["replicas_dropped"]
    assert s[:, 6].sum() == totals["leaders_changed"]
    assert s[:, 7].sum() == totals["leaders_changed"] - empty_rows


def _lists(d):
    """{partition: list} -> (C [Q, L], lengths) in ascending partition order."""
    rows = [d[p] for p in sorted(d)]
    L = max([len(r) for r in rows] + [1])
    a = np.zeros((len(rows), L), dtype=np.int64)
    for i, r in enumerate(rows):
        a[i, :len(r)] = r
    return a, np.array([len(r) for r in rows])


# ---- CPU: the model on hand cases ------------------------------------------------------------------------------------
README_CUR = {0: [10, 11], 1: [11, 12], 2: [12, 10], 3: [10, 12]}
README_NEW = {0: [10, 11], 1: [11, 13], 2: [13, 10], 3: [10, 13]}   # brokers {10, 11, 13}: the README's decommission example


def test_model_on_readme_decommission_example():
    C, lc = _lists(README_CUR)
    O, lo = _lists(README_NEW)
    ids = [10, 11, 12, 13]
    totals, stats, cls, empty = plan_model(C, lc, O, lo, ids)
    assert cls.tolist() == [0, 2, 2, 2]
    assert totals == dict(rows=4, rows_reordered=0, rows_moved=3, replicas_added=3, replicas_dropped=3, leaders_changed=1)
    col = dict(zip(kab.PLAN_COLUMNS, range(8)))
    b10, b12, b13 = stats[0], stats[2], stats[3]
    assert (b12[col["replicas_before"]], b12[col["replicas_after"]], b12[col["replicas_out"]]) == (3, 0, 3)
    assert (b12[col["leaders_before"]], b12[col["leaders_out"]]) == (1, 1)
    assert (b13[col["replicas_after"]], b13[col["replicas_in"]], b13[col["leaders_in"]]) == (3, 3, 1)
    assert (b10[col["replicas_before"]], b10[col["replicas_after"]], b10[col["leaders_before"]], b10[col["leaders_after"]]) == (3, 3, 2, 2)
    assert stats[4].sum() == 0
    check_invariants(totals, stats, empty)
    # the default report list is the live table {10, 11, 13}: the decommissioned broker 12 lands in "other"
    _, live, _, _ = plan_model(C, lc, O, lo, [10, 11, 13])
    assert live[3].tolist() == b12.tolist()
    assert live[2].tolist() == b13.tolist()


def test_model_hand_cases():
    col = dict(zip(kab.PLAN_COLUMNS, range(8)))
    # same brokers, new order: REORDERED, nothing copied, the leader changes
    t, s, cls, e = plan_model([[1, 2, 3]], [3], [[2, 3, 1]], [3], [1, 2, 3])
    assert cls.tolist() == [1] and t["replicas_added"] == t["replicas_dropped"] == 0 and t["leaders_changed"] == 1
    assert s[1, col["leaders_in"]] == 1 and s[0, col["leaders_out"]] == 1 and s[:, col["replicas_in"]].sum() == 0
    check_invariants(t, s, e)
    # replication factor 2 -> 3 (--desired_replication_factor): MOVED, one replica added, leader kept
    t, s, cls, e = plan_model([[1, 2]], [2], [[1, 2, 3]], [3], [1, 2, 3])
    assert cls.tolist() == [2] and (t["replicas_added"], t["replicas_dropped"], t["leaders_changed"]) == (1, 0, 0)
    assert s[2, col["replicas_in"]] == 1 and s[2, col["replicas_after"]] == 1
    check_invariants(t, s, e)
    # shrinking to the same leader: still MOVED (the length changes)
    t, s, cls, e = plan_model([[1, 2]], [2], [[1]], [1], [1, 2])
    assert cls.tolist() == [2] and t["replicas_dropped"] == 1
    # an empty current list: MOVED, every new replica added, its leader is a leadership gain with no matching loss
    t, s, cls, e = plan_model(np.zeros((1, 0)), [0], [[4, 5]], [2], [4, 5])
    assert cls.tolist() == [2] and (t["replicas_added"], t["leaders_changed"]) == (2, 1) and e == 1
    assert s[0, col["leaders_in"]] == 1 and s[:, col["leaders_out"]].sum() == 0
    check_invariants(t, s, e)
    # a broker repeated in the current list counts once
    t, s, cls, e = plan_model([[1, 1]], [2], [[1, 2]], [2], [1, 2])
    assert cls.tolist() == [2] and (t["replicas_added"], t["replicas_dropped"]) == (1, 0) and s[0, col["replicas_before"]] == 1
    check_invariants(t, s, e)
    # unchanged
    t, s, cls, e = plan_model([[7, 8]], [2], [[7, 8]], [2], [7, 8])
    assert cls.tolist() == [0] and t["rows_moved"] == t["rows_reordered"] == t["leaders_changed"] == 0


def test_plan_symbols_exported(native_lib):
    for name in ("ka_plan_last", "ka_ctx_set_report_brokers", "ka_solve_dense_json_changed"):
        assert hasattr(native_lib, name)


# ---- GPU --------------------------------------------------------------------------------------------------------------
def _device_plan(s, report_ids=None):
    """last_plan() of solver s with row classes, as (totals, stats, cls)."""
    s.set_report_brokers(report_ids)
    totals, ids, stats, cls = s.last_plan(row_class=True)
    if report_ids is not None:
        assert np.array_equal(ids, np.sort(np.asarray(report_ids)))
    return totals, stats.astype(np.int64), cls


def _assert_plan(s, C, lc, O, lo, report_ids):
    """Device plan == model on (C, O) for the given report list (None = the live table of s)."""
    exp_t, exp_s, exp_c, empty = plan_model(C, lc, O, lo, s.broker_id if report_ids is None else np.sort(report_ids))
    t, st, cls = _device_plan(s, report_ids)
    assert t == exp_t
    assert np.array_equal(st, exp_s)
    assert np.array_equal(cls, exp_c)
    check_invariants(t, st, empty)
    return t


def _ragged_lists(rep_off, cur):
    lc = np.diff(rep_off)
    C = np.zeros((len(lc), max(int(lc.max(initial=0)), 1)), dtype=np.int64)
    for g in range(len(lc)):
        C[g, :lc[g]] = cur[rep_off[g]:rep_off[g + 1]]
    return C, lc


def _ragged_case_plan(oracle, s, case, extra_ids):
    """Solve a ragged case on the GPU (ka_solve); when it succeeds, compare the plan with the model on the oracle's rows."""
    names, part_off, part_id, rep_off, cur = util.flatten(case["topics"])
    s.reset()   # a fresh Context, like the oracle's
    s.set_brokers_with_racks(case["brokers"], case["racks"])
    stride = util.stride_for(case["topics"], case["desired_rf"])
    th = np.array([kab.java_string_hash(n) for n in names], dtype=np.int32)
    out, out_len, st = s.solve_ragged(th, part_off, part_id, rep_off, cur, case["desired_rf"], stride, check=False)
    brokers = sorted(case["brokers"])
    ln, _, eout, est = oracle.run(oracle.OracleContext(), names, part_off, part_id, rep_off, cur, brokers,
                                  [case["racks"].get(b) for b in brokers], case["desired_rf"], stride, raise_on_error=False)
    assert st.code == est.code
    if st.code != 0:
        with pytest.raises(kab.KassignError):
            s.last_plan()
        return False
    assert np.array_equal(out_len, ln)
    used = np.arange(out.shape[1])[None, :] < ln[:, None]
    assert np.array_equal(np.where(used, out, 0), np.where(used, eout, 0))
    C, lc = _ragged_lists(rep_off, cur)
    _assert_plan(s, C, lc, eout, ln, None)
    _assert_plan(s, C, lc, eout, ln, np.unique(np.concatenate([np.asarray(brokers), extra_ids])))
    return True


@pytest.mark.gpu
def test_plan_after_ragged_solve_goldens_and_random(native_lib, oracle):
    s = kab.Solver(0)
    n_ok = 0
    for c in util.load_golden():
        n_ok += _ragged_case_plan(oracle, s, c, np.zeros(0, dtype=np.int64))
    rng = random.Random(23)
    for it in range(60):
        s.reset()
        nb = rng.randint(2, 30)
        brokers = sorted(rng.sample(range(-5, 200), nb))
        racks = {} if it % 3 == 0 else {b: "k%d" % rng.randrange(max(2, nb // 3)) for b in brokers if rng.random() < 0.8}
        gone = [1000, 1001, -77]   # decommissioned: in current lists, not live
        topics = []
        for ti in range(rng.randint(1, 5)):
            rf = rng.randint(1, min(5, nb))
            ragged = rng.random() < 0.3
            cur = {}
            for p in sorted(rng.sample(range(0, 60), rng.randint(1, 40))):
                k = rng.randint(0, 5) if ragged else rf
                cur[p] = rng.sample(brokers + gone, min(k, nb + 3))
            topics.append(("pt%d_%d" % (it, ti), cur))
        desired = rng.choice([-1, -1, 1, 2, 3, 4])
        case = dict(topics=topics, brokers=brokers, racks=racks, desired_rf=desired)
        n_ok += _ragged_case_plan(oracle, s, case, np.array(gone))
    assert n_ok > 30


def _dense_expect(oracle, cl):
    exp, exp_len, est = oracle.fast_run_dense(oracle.FastContext(), cl.topic_hash, cl.cur, cl.broker_id, cl.rack_index)
    assert est.code == 0
    return exp, exp_len


def _balanced(cl_base, frac):
    """Current = the GPU's solve of the base config; live set = the base brokers minus `frac` of every rack."""
    out, _, _ = kab.Solver(0).solve_cluster(cl_base)
    cl = kab.synth.make_config(cl_base.name.split("_")[0], cl_base.meta["kind"], remove_frac=frac) if frac else cl_base
    return dataclasses.replace(cl, cur=np.ascontiguousarray(out))


@pytest.mark.gpu
def test_plan_after_dense_solves_c3_and_balanced_c5(native_lib, oracle):
    cases = [kab.synth.make_config("c3", "mixed")]
    base = kab.synth.make_config("c5", "mixed")
    cases += [_balanced(base, 0.0), _balanced(base, 0.01), _balanced(base, 0.2)]
    for i, cl in enumerate(cases):
        s = kab.Solver(0)
        out, out_len, st = s.solve_cluster(cl)
        exp, exp_len = _dense_expect(oracle, cl)
        assert np.array_equal(out.reshape(-1, cl.RF), exp)
        Q = cl.T * cl.P
        t = _assert_plan(s, cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, None)
        if i == 1:   # the balanced re-run changes nothing
            assert t["rows_moved"] == t["rows_reordered"] == t["leaders_changed"] == t["replicas_added"] == 0
        else:
            assert t["rows_moved"] > 0 and t["leaders_changed"] > 0
        if i >= 2:   # decommissioned brokers listed one by one: they lose everything
            gone = np.setdiff1d(base.broker_id, cl.broker_id)
            rep = np.union1d(cl.broker_id, gone)
            _assert_plan(s, cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, rep)
            _, ids, stats, _ = s.last_plan()
            g = np.isin(ids, gone)
            assert (stats[:-1][g, 1] == 0).all() and (stats[:-1][g, 3] == stats[:-1][g, 0]).all()


@pytest.mark.gpu
def test_plan_after_device_solve(native_lib, oracle):
    import torch
    cl = kab.synth.make_config("c2", "mixed", remove_frac=0.1)
    exp, exp_len = _dense_expect(oracle, cl)
    s = kab.Solver(0)
    s.set_brokers(cl.broker_id, cl.rack_index)
    d_hash = torch.from_numpy(cl.topic_hash).cuda()
    d_cur = torch.from_numpy(cl.cur).cuda()
    d_out = torch.empty((cl.T, cl.P, cl.RF), dtype=torch.int32, device="cuda")
    Q = cl.T * cl.P
    for d_len in (torch.empty((cl.T, cl.P), dtype=torch.int32, device="cuda"), None):
        s.reset()
        torch.cuda.synchronize()
        s.solve_dense_device(cl.T, d_hash.data_ptr(), cl.P, cl.RF, d_cur.data_ptr(), -1, cl.RF,
                             d_len.data_ptr() if d_len is not None else 0, d_out.data_ptr(),
                             stream=torch.cuda.current_stream().cuda_stream, sync=False)
        _assert_plan(s, cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, None)   # synchronises the solve first
        assert np.array_equal(d_out.cpu().numpy().reshape(-1, cl.RF), exp)


@pytest.mark.gpu
def test_plan_report_list_lookup_and_histogram_paths(native_lib, oracle):
    cl = kab.synth.make_config("c2", "mixed", remove_frac=0.1)     # ids 1000..1099, 10 removed
    exp, exp_len = _dense_expect(oracle, cl)
    s = kab.Solver(0)
    s.solve_cluster(cl)
    Q = cl.T * cl.P
    C, lc = cl.cur.reshape(Q, -1), np.full(Q, cl.RF)
    rng = np.random.default_rng(3)
    all_ids = 1000 + np.arange(100)
    lists = [
        all_ids,                                                              # shared-memory LUT, private columns
        all_ids[::3],                                                         # omits live brokers: "other" is used
        np.union1d(all_ids, [-20000, 20000]),                                 # range > 32768: global LUT
        np.union1d(all_ids, [-2 ** 31 + 1, 2 ** 31 - 2]),                    # range > 2^25: binary search
        np.union1d(all_ids, 2000 + np.arange(65534 - 100)),                   # M = 65534: global-atomic columns, global LUT
        np.union1d(all_ids, rng.choice(np.arange(-2 ** 31 + 1, 2 ** 31 - 1, 65537), 60000, replace=False)),  # large M, bsearch
        np.array([1005]),                                                     # M = 1
    ]
    for ids in lists:
        ids = np.unique(ids).astype(np.int32)
        assert len(ids) <= 65534
        _assert_plan(s, C, lc, exp, exp_len, ids)
    t, st, _ = _device_plan(s, lists[1])
    assert st[-1, 0] > 0                                                      # the "other" bucket holds the omitted brokers
    with pytest.raises(kab.KassignError):
        s.set_report_brokers(np.arange(65535))                                # beyond 65534 ids


def _wide_cluster():
    return kab.synth.make_cluster(T=40, P=30, RF=5, N=80, R=10, seed=71, kind="mixed", remove_frac=0.1)


@pytest.mark.gpu
def test_plan_and_changed_json_rows_of_four_to_eight(native_lib, oracle):
    """Rows of 4..8 replicas are ordered by the fused chain (one launch per block, no sub-blocks)."""
    for cl, desired in ((_wide_cluster(), -1), (kab.synth.make_cluster(T=30, P=20, RF=4, N=50, R=8, seed=72, kind="random"), 6),
                        (kab.synth.make_cluster(T=30, P=20, RF=3, N=50, R=8, seed=73, kind="random"), 2)):
        cl.desired_rf = desired
        exp, exp_len, est = util.oracle_dense(oracle, cl)
        assert est.code == 0
        S = max(cl.RF, desired)
        Q = cl.T * cl.P
        s = kab.Solver(0)
        s.set_brokers(cl.broker_id, cl.rack_index)
        s.solve_dense(cl.topic_hash, cl.cur, desired)
        _, _, cls, _ = plan_model(cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, cl.broker_id)
        _assert_plan(s, cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, None)
        s.reset()
        text, st = s.solve_dense_json(cl.topic_names, cl.topic_hash, cl.cur, desired, changed_only=True)
        assert bytes(text).decode() == expected_changed_json(cl, exp.reshape(-1, S), exp_len, cls)
        _assert_plan(s, cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, None)


def expected_changed_json(cl, out, out_len, cls):
    """The NEW ASSIGNMENT text (KAG:169-186) of the rows whose class is not UNCHANGED, built on the host."""
    rows = out.reshape(cl.T * cl.P, -1)
    lens = out_len.reshape(-1)
    parts = []
    for g in np.flatnonzero(cls != 0):
        t, p = divmod(int(g), cl.P)
        parts.append('{"partition":%d,"replicas":[%s],"topic":"%s"}' % (p, ",".join(str(int(b)) for b in rows[g, :lens[g]]),
                                                                       cl.topic_names[t]))
    return '{"partitions":[' + ",".join(parts) + '],"version":1}'


def _changed_json_check(oracle, cl):
    exp, exp_len = _dense_expect(oracle, cl)
    Q = cl.T * cl.P
    _, _, cls, _ = plan_model(cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, cl.broker_id)
    s = kab.Solver(0)
    s.set_brokers(cl.broker_id, cl.rack_index)
    text, st = s.solve_dense_json(cl.topic_names, cl.topic_hash, cl.cur, changed_only=True)
    assert st.code == 0
    assert bytes(text).decode() == expected_changed_json(cl, exp, exp_len, cls), cl.name
    _assert_plan(s, cl.cur.reshape(Q, -1), np.full(Q, cl.RF), exp, exp_len, None)
    full, _ = s.solve_dense_json(cl.topic_names, cl.topic_hash, cl.cur)          # the full text is unchanged by the feature
    assert len(full) >= len(text)
    return cls


def _later_changes(cl, t_from):
    """A balanced cl (current = its own solve) whose lists are rotated from topic t_from on: the first changed row sits there."""
    cur = cl.cur.copy()
    cur[t_from:] = np.roll(cur[t_from:], 1, axis=2)
    return dataclasses.replace(cl, cur=cur)


@pytest.mark.gpu
def test_changed_json_c2_balanced_and_later_first_change(native_lib, oracle):
    base = kab.synth.make_config("c2", "mixed")
    cls = _changed_json_check(oracle, base)
    assert 0 < (cls != 0).sum() < len(cls)
    bal = _balanced(base, 0.0)
    s = kab.Solver(0)
    s.set_brokers(bal.broker_id, bal.rack_index)
    text, st = s.solve_dense_json(bal.topic_names, bal.topic_hash, bal.cur, changed_only=True)
    assert bytes(text).decode() == '{"partitions":[],"version":1}'
    t, _, _, _ = s.last_plan()
    assert t["rows_moved"] == t["rows_reordered"] == 0 and t["rows"] == bal.T * bal.P
    cls = _changed_json_check(oracle, _later_changes(bal, 700))
    assert np.flatnonzero(cls)[0] >= 700 * bal.P
    # too small a buffer: KA_ERR_LIMIT, and no plan
    with pytest.raises(kab.KassignError) as e:
        s.solve_dense_json(base.topic_names, base.topic_hash, base.cur, json_buf=np.empty(100, dtype=np.uint8), changed_only=True)
    assert e.value.code == kab._native.KA_ERR_LIMIT
    with pytest.raises(kab.KassignError):
        s.last_plan()
    # a failing topic: the usual exception, no text, no plan
    bad = kab.synth.make_cluster(T=6, P=4, RF=3, N=9, R=3, seed=8, kind="random")
    s.set_brokers(bad.broker_id[:2], bad.rack_index[:2])
    with pytest.raises(kab.IllegalStateException):
        s.solve_dense_json(bad.topic_names, bad.topic_hash, bad.cur, changed_only=True)
    text, st = s.solve_dense_json(bad.topic_names, bad.topic_hash, bad.cur, changed_only=True, check=False)
    assert st.code == 3 and len(text) == 0
    with pytest.raises(kab.KassignError):
        s.last_plan()


@pytest.mark.gpu
def test_changed_json_pipelined_c3_many_sub_blocks(native_lib, oracle):
    """c3 runs in K = 4 pipeline blocks; KA_CHAIN_SUBBLOCKS = 8 cuts each into 8 chain sub-blocks (32 text fragments)."""
    code = ("import numpy as np, kafka_assigner_b200 as kab\n"
            "from oracle import oracle_lib as ol\n"
            "from tests.test_movement_plan import _changed_json_check, _balanced, _later_changes\n"
            "cls = _changed_json_check(ol, kab.synth.make_config('c3', 'mixed'))\n"
            "assert 0 < (cls != 0).sum() < len(cls)\n"
            "cl = kab.synth.make_cluster(T=300, P=24, RF=3, N=40, R=5, seed=77, kind='mixed')\n"
            "cls = _changed_json_check(ol, _later_changes(_balanced(cl, 0.0), 250))\n"
            "assert np.flatnonzero(cls)[0] >= 250 * 24\n"
            "print('OK')\n")
    for env_over in (dict(KA_CHAIN_SUBBLOCKS="8"), dict(KA_PIPELINE_STAGES="3", KA_CHAIN_SUBBLOCKS="8")):
        env = dict(os.environ, PYTHONPATH=os.path.dirname(util.HERE), **env_over)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, env=env)
        assert r.returncode == 0 and "OK" in r.stdout, (env_over, r.stdout[-1500:] + r.stderr[-1500:])


@pytest.mark.gpu
def test_plan_refused_before_any_solve_and_after_split_api(native_lib):
    import torch
    s = kab.Solver(0)
    with pytest.raises(kab.KassignError) as e:
        s.last_plan()
    assert e.value.code == kab._native.KA_ERR_BAD_ARG
    cl = kab.synth.make_cluster(T=8, P=10, RF=3, N=20, R=4, seed=3, kind="mixed")
    s.solve_cluster(cl)
    s.last_plan()
    d_hash = torch.from_numpy(cl.topic_hash).cuda()
    d_cur = torch.from_numpy(cl.cur).cuda()
    d_out = torch.empty((cl.T, cl.P, 3), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    s.stage_dense_device(cl.T, d_hash.data_ptr(), cl.P, cl.RF, d_cur.data_ptr(), -1, 3)
    assert s.order_device(0, d_out.data_ptr()).code == 0
    with pytest.raises(kab.KassignError) as e:
        s.last_plan()
    assert e.value.code == kab._native.KA_ERR_BAD_ARG
