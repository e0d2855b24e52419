"""Host-side logic that needs no GPU: synthetic networks, the sampler's CPU restatement,
the VE planner (dry run), sharding, and the world_size-2 count allreduce over gloo."""
import os
import subprocess
import sys

import numpy as np
import pytest

from continuousbayesiannetwork_b200 import sharding, synth
from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, VECompiler

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import row_oracle as RO  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_networks_have_the_published_shapes():
    a = synth.asia()
    assert a.n == 8 and sum(len(p) for p in a.parents) == 8
    for c in a.cpts:
        np.testing.assert_allclose(c.sum(axis=-1), 1.0)
    al = synth.alarm()           # asserts 37 / 46 / 509 inside
    assert max(len(p) for p in al.parents) == 4 and max(al.cards) == 4
    assert max(int(np.prod(c.shape)) for c in al.cpts) == 108
    r = synth.random_ktree_dag()
    assert r.n == 200 and max(len(p) for p in r.parents) <= 4 and set(r.cards) == {4}
    L = synth.layered_dag()
    assert L.n == 1000 and 2 <= min(L.cards) and max(L.cards) <= 8
    for spec in (a, al, r, L):
        order = spec.topological_order()
        pos = {v: i for i, v in enumerate(order)}
        assert all(pos[p] < pos[i] for i in range(spec.n) for p in spec.parents[i])
        # parents are in sorted-name order (the reference's CPT axis order)
        assert all([spec.names[p] for p in ps] == sorted(spec.names[p] for p in ps) for ps in spec.parents)


def test_sampler_restatement_is_shard_invariant_and_matches_the_cpts():
    spec = synth.asia()
    full = synth.sample_forward_numpy(spec, 11, 0, 40000)
    parts = np.concatenate([synth.sample_forward_numpy(spec, 11, 0, 15001),
                            synth.sample_forward_numpy(spec, 11, 15001, 24999)], axis=1)
    assert np.array_equal(full, parts)
    assert abs(full[spec.names.index("smoke")].mean() - 0.5) < 0.01
    either = full[spec.names.index("either")]
    assert np.array_equal(either, full[spec.names.index("lung")] | full[spec.names.index("tub")])


def _dry(spec, target, ev, **kw):
    return VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()), **kw).compile(target, ev, dry=True)


def test_planner_asia_and_alarm():
    a = synth.asia()
    for t in ("lung", "tub", "bronc"):
        s = _dry(a, t, ["asia", "smoke", "xray", "dysp"])
        scope = tuple(a.names.index(e) for e in ["asia", "smoke", "xray", "dysp"]) + (a.names.index(t),)
        assert s.final_tables == [(scope, 32)]
        assert len(s.relevant_evidence) == 4 and s.n_hidden == 3
    al = synth.alarm()
    for t in synth.ALARM_TARGETS:
        s = _dry(al, t, synth.ALARM_EVIDENCE)
        assert s.n_hidden == 24 and len(s.final_tables) == 1
        assert s.final_tables[0][1] == 839808 * al.cards[al.names.index(t)]


def test_planner_prunes_barren_and_d_separated_parts():
    a = synth.asia()
    # evidence on smoke only: xray/dysp/either are barren, asia/tub irrelevant
    s = _dry(a, "lung", ["smoke"])
    assert s.n_relevant == 2 and s.n_hidden == 0 and s.final_tables == [((2, 3), 4)]
    # target with no evidence: prior marginal
    s = _dry(a, "either", [])
    assert s.relevant_evidence == [] and s.final_tables == [((5,), 2)]
    # intervention on lung cuts smoke -> lung
    s = _dry(a, "smoke", ["lung"])
    assert len(s.relevant_evidence) == 1
    c = VECompiler(DryTables(a.names, a.cards, a.parents_by_name()))
    s = c.compile("smoke", ["lung"], do=["lung"], dry=True)
    assert s.relevant_evidence == []
    with pytest.raises(ValueError):
        c.compile("smoke", [], do=["lung"], dry=True)


def test_planner_budget_and_layered_stress():
    r = synth.random_ktree_dag()
    rng = np.random.default_rng(5)
    vs = rng.choice(200, size=11, replace=False)
    s = _dry(r, r.names[vs[0]], [r.names[v] for v in vs[1:]])
    assert s.max_table_cells <= 1 << 28
    with pytest.raises(PlanTooLarge):
        _dry(r, r.names[vs[0]], [r.names[v] for v in vs[1:]], table_budget_cells=1 << 10)
    L = synth.layered_dag()
    with pytest.raises(PlanTooLarge):   # treewidth of the 20x50 layered DAG is far beyond exact inference
        _dry(L, "l16_15", ["l03_10", "l10_20", "l19_01", "l12_40", "l15_15"])


def test_shard_ranges_cover_exactly():
    for n in (0, 1, 7, 1000, 16_777_216 + 5):
        for w in (1, 2, 3, 8):
            rs = [sharding.shard_range(n, r, w) for r in range(w)]
            assert rs[0][0] == 0 and rs[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
            assert max(e - s for s, e in rs) <= (n + w - 1) // w + 15
            assert all(s % 16 == 0 for s, e in rs if e > s)


@pytest.mark.timeout(120)
def test_count_allreduce_gloo_world2(tmp_path):
    """Two CPU ranks count disjoint sample shards with the oracle and combine the int64 tables through
    sharding.allreduce_counts (gloo here, NCCL on the GPUs): the sum equals the single-process tables."""
    script = os.path.join(ROOT, "tests", "_gloo_worker.py")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29531", script, str(tmp_path)],
                         capture_output=True, text=True, timeout=110, cwd=ROOT)
    assert out.returncode == 0, out.stdout + out.stderr
    assert (tmp_path / "ok_0").exists() and (tmp_path / "ok_1").exists()


def test_incremental_greedy_matches_full_rescan():
    """The planner's incremental bookkeeping (cached elimination scopes, updated only around the eliminated variable)
    must pick exactly what a full rescan of every hidden variable picks at every step."""
    from continuousbayesiannetwork_b200.ve import _Greedy

    rng = np.random.default_rng(7)
    for trial in range(30):
        n = int(rng.integers(8, 40))
        cards = [int(c) for c in rng.integers(2, 6, size=n)]
        scopes = {}
        for k in range(n):                                  # family-like factors: a node and up to 3 earlier nodes
            ps = rng.choice(k, size=min(k, int(rng.integers(0, 4))), replace=False) if k else []
            scopes[k] = [int(p) for p in ps] + [k]
        hidden = [int(v) for v in rng.choice(n, size=int(rng.integers(1, n)), replace=False)]
        g = _Greedy(cards, scopes, hidden)
        ref = {k: list(v) for k, v in scopes.items()}
        left = set(hidden)
        nk = n
        while left:
            best = None
            for v in sorted(left):
                sc = set()
                for s in ref.values():
                    if v in s:
                        sc |= set(s)
                sc.discard(v)
                c = int(np.prod([cards[u] for u in sc])) if sc else 1
                if best is None or (c, v) < (best[0], best[1]):
                    best = (c, v, sc)
            v, c, sc = g.best()
            assert (c, v, set(sc)) == (best[0], best[1], best[2]), trial
            ref = {k: s for k, s in ref.items() if v not in s}
            ref[nk] = sorted(sc)
            g.eliminate(v, nk, sorted(sc))
            left.discard(v)
            nk += 1
        assert not g.hidden


def _cpt_statics(sch, spec):
    """The static tables of a per-row schedule compiled with a table budget of one cell: the CPTs themselves, permuted to
    the layout the schedule reads."""
    statics = []
    for scope, source in zip(sch["static_scopes"], sch["static_source_scopes"]):
        node = source[-1]
        assert source == spec.parents[node] + [node] and sorted(scope) == sorted(source)
        cpt = np.asarray(spec.cpts[node], dtype=np.float64).reshape([spec.cards[v] for v in source])
        statics.append(np.ascontiguousarray(cpt.transpose([source.index(v) for v in scope])).reshape(-1))
    return statics


def test_row_schedule_interpreted_on_the_cpu_matches_the_oracle():
    """The per-row elimination SCHEDULE (steps, offset tables, sum strides, the layout of every factor) is host logic: a numpy
    interpreter of it, fed with the ground-truth CPTs, must reproduce the oracle's posteriors.  A table budget of one cell
    leaves every hidden variable to the per-row schedule.  Checked in both layouts: every factor laid out for the step that
    consumes it (summed variable innermost, stride 1: the contract of the executor's unrolled step bodies) and the tables' own
    axis order (the strided bodies)."""
    import torch

    from oracle import cbn_oracle as O

    small_layers = synth.layered_dag(layers=4, width=6, seed=21)          # cards 2..8: odd and even run lengths
    cases = ((synth.asia(), "lung", ["asia", "xray", "dysp"]),
             (synth.random_ktree_dag(n=24, card=3, k=3, max_parents=2, seed=5), "x020", ["x003", "x011", "x017", "x023"]),
             (small_layers, "l01_02", ["l03_00", "l03_03", "l03_05", "l02_01", "l00_04"]),
             (small_layers, "l03_04", ["l00_00", "l00_03", "l01_05", "l02_02"]))
    for spec, target, ev_names in cases:
        for unit in (True, False):
            c = VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()), table_budget_cells=1, row_temp_floats=1 << 22,
                           check_support=False, row_unit_layout=unit)
            stats = c.compile(target, ev_names, dry=True)
            assert stats.per_row_hidden > 0
            sch = c.last_row_schedule
            ev_ids = sch["evidence"]
            assert ev_ids == [spec.names.index(e) for e in ev_names]
            sums = [st for st in sch["steps"] if st["sum_card"] > 1]
            n_permuted = sum(a != b for a, b in zip(sch["static_scopes"], sch["static_source_scopes"]))
            if unit:
                assert all(s == 1 for st in sums for s in st["sum_stride"]) and n_permuted > 0
                for scope in sch["static_scopes"]:         # evidence axes first, so a row's slice stays contiguous
                    is_ev = [v in ev_ids for v in scope]
                    assert is_ev == sorted(is_ev, reverse=True)
            else:
                assert n_permuted == 0 and any(s != 1 for st in sums for s in st["sum_stride"])
            # every factor is consumed exactly once, and never before it exists
            used = [i for st in sch["steps"] for i in st["in_id"]]
            assert sorted(used) == list(range(len(sch["static_scopes"]) + len(sch["steps"]) - 1))
            assert all(i < len(sch["static_scopes"]) + j for j, st in enumerate(sch["steps"]) for i in st["in_id"])
            codes = synth.sample_forward_numpy(spec, 9, 0, 40)
            rows = codes[ev_ids].T
            got = RO.posterior(RO.interpret(sch, _cpt_statics(sch, spec), spec.cards, rows))
            want = O.ve_posterior(O.DiscreteNet(spec.cards, spec.parents, spec.cpts), sch["target"], ev_ids, rows, dtype=torch.float64)
            np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-15)
