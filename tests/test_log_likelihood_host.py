"""log P(e) without a GPU: the fp64 oracles against each other, and the evidence-mode split of the VE planner (dry run)."""
import itertools
import os
import sys

import numpy as np
import pytest
import torch

from continuousbayesiannetwork_b200 import synth
from continuousbayesiannetwork_b200.ve import DryTables, VECompiler
from oracle import cbn_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import loglik_oracle as LO  # noqa: E402


def _net(spec):
    return O.DiscreteNet(spec.cards, spec.parents, spec.cpts)


def _configs(cards):
    return np.ascontiguousarray(np.indices(cards).reshape(len(cards), -1).T) if cards else np.zeros((1, 0), np.int64)


def _subsets(n):
    for k in range(n + 1):
        yield from itertools.combinations(range(n), k)


def test_ve_log_evidence_equals_enumeration_on_asia():
    spec = synth.asia()
    net = _net(spec)
    n_pairs = 0
    for sub in _subsets(spec.n):
        ev = _configs([spec.cards[v] for v in sub])
        want = LO.enumerate_log_evidence(net, sub, ev)
        got = LO.ve_log_evidence(net, sub, ev)
        fin = np.isfinite(want)
        assert np.array_equal(fin, np.isfinite(got)) and np.all(np.isneginf(got[~fin]))
        np.testing.assert_allclose(got[fin], want[fin], rtol=1e-12, atol=1e-12)
        # a distribution over the subset's configurations
        assert abs(float(torch.logsumexp(torch.as_tensor(want), 0))) < 1e-12
        assert abs(float(torch.logsumexp(torch.as_tensor(got), 0))) < 1e-12
        n_pairs += ev.shape[0]
    assert n_pairs == 3 ** 8


def test_oracles_flag_out_of_domain_codes():
    spec = synth.asia()
    net = _net(spec)
    ev = np.array([[0, 1], [2, 0], [1, 255]])
    for fn in (LO.enumerate_log_evidence, LO.ve_log_evidence):
        got = fn(net, [0, 3], ev)
        assert np.isfinite(got[0]) and np.isneginf(got[1]) and np.isneginf(got[2])


def _dry(spec, names):
    return VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name())).compile_evidence(names, dry=True)


def test_evidence_split_complete_rows_go_to_the_observed_families_kernel():
    for spec in (synth.asia(), synth.alarm()):
        split = _dry(spec, list(spec.names))
        assert split.ve_stats is None
        assert sorted(split.observed_families) == list(range(spec.n))
        # reversed column order: same split, slots follow the order given
        split = _dry(spec, list(reversed(spec.names)))
        assert split.ve_stats is None and split.evidence == list(reversed(range(spec.n)))


def test_evidence_split_alarm_headline_set():
    spec = synth.alarm()
    split = _dry(spec, synth.ALARM_EVIDENCE)
    E = {spec.names.index(e) for e in synth.ALARM_EVIDENCE}
    relevant = _net(spec).ancestors(E)
    inside = sorted(v for v in relevant if set(spec.parents[v] + [v]) <= E)
    assert sorted(split.observed_families) == inside
    st = split.ve_stats
    assert st is not None and not split.per_row and st.per_row_hidden == 0
    # every hidden ancestor is eliminated: the tables left are over evidence variables only
    assert st.n_hidden == len(relevant - E)
    for scope, _ in st.final_tables:
        assert set(scope) <= E
    # the posterior plans gather one table over the 12 evidence variables; so does log P(e)
    assert [c for _, c in st.final_tables] == [839808]


def test_evidence_per_row_schedule_when_the_budget_is_small():
    spec = synth.alarm()
    comp = VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()), table_budget_cells=1 << 10)
    split = comp.compile_evidence(synth.ALARM_EVIDENCE, dry=True)
    assert split.per_row and split.ve_stats.per_row_hidden > 0
    # the per-row schedule ends in one cell (no target)
    sched = comp.last_row_schedule
    assert sched["target"] is None and sched["steps"][-1]["out_size"] == 1


def test_evidence_split_no_evidence_and_unknown_names():
    spec = synth.asia()
    split = _dry(spec, [])
    assert split.observed_families == [] and split.ve_stats is None
    with pytest.raises(ValueError):
        _dry(spec, ["xray", "not_a_node"])
    with pytest.raises(ValueError):
        _dry(spec, ["xray", "xray"])


def test_log_likelihood_rejects_columns_that_are_not_nodes():
    import networkx as nx

    from continuousbayesiannetwork_b200.base.bayesian_network import BayesianNetwork

    bn = object.__new__(BayesianNetwork)          # column handling only: no fit, no device
    bn.device = "cpu"
    bn.nodes_obj = {"a": None, "b": None}
    bn.initial_dag = nx.DiGraph([("a", "b")])
    with pytest.raises(ValueError, match="not nodes"):
        bn._observed_columns({"a": np.zeros(3), "c": np.zeros(3)})
    with pytest.raises(ValueError, match="same number of rows"):
        bn._observed_columns({"a": np.zeros(3), "b": np.zeros(4)})
    cols, n = bn._observed_columns({"b": np.arange(5)})
    assert list(cols) == ["b"] and n == 5
    pd = pytest.importorskip("pandas")
    with pytest.raises(ValueError, match="not nodes"):
        bn._observed_columns(pd.DataFrame({"a": [0.0], "typo": [1.0]}))
    cols, n = bn._observed_columns(pd.DataFrame(index=range(7)))
    assert cols == {} and n == 7
