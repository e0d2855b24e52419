"""Most probable explanation without a GPU: the fp64 oracles against each other, the structure of the max-sum
elimination (dry run), its limits, the C layout of the decode steps, and a numpy interpreter of the decode schedule."""
import ctypes as C
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

from continuousbayesiannetwork_b200 import synth
from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, VECompiler
from oracle import cbn_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mpe_oracle as MO  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _net(spec):
    return O.DiscreteNet(spec.cards, spec.parents, spec.cpts)


def _compiler(spec, **kw):
    return VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()), **kw)


def _configs(cards):
    return np.ascontiguousarray(np.indices(cards).reshape(len(cards), -1).T) if cards else np.zeros((1, 0), np.int64)


def _check_decode_order(split, n):
    """Every context of a step is evidence or decoded by an earlier step; every hidden variable is decoded once."""
    E = set(split.evidence)
    done = set()
    for v, scope in split.decode:
        assert v not in E and v not in done and v not in scope
        assert all(u in E or u in done for u in scope), (v, scope)
        done.add(v)
    assert done == set(split.hidden) == set(range(n)) - E


def test_alarm_headline_structure():
    spec = synth.alarm()
    split = _compiler(spec).compile_mpe(synth.ALARM_EVIDENCE, dry=True)
    _check_decode_order(split, spec.n)
    assert len(split.decode) == len(split.hidden) == 25
    assert [c for _, c in split.stats.final_tables] == [839808]
    assert all(set(sc) <= set(split.evidence) for sc, _ in split.stats.final_tables)
    # the last-eliminated variable's table has the shape of the final one; the other 24 are small
    assert 839808 <= split.argmax_bytes < 1 << 20
    E = set(split.evidence)
    assert sorted(split.observed_families) == sorted(v for v in range(spec.n) if set(spec.parents[v] + [v]) <= E)


def test_decode_order_ktree_bench_patterns_and_random_dags():
    spec = synth.random_ktree_dag()
    rng = np.random.default_rng(1240)
    for _ in range(8):
        vs = [int(v) for v in rng.choice(spec.n, size=11, replace=False)]
        split = _compiler(spec).compile_mpe([spec.names[v] for v in vs[1:]], dry=True)
        _check_decode_order(split, spec.n)
        assert len(split.decode) == 190
    split = _compiler(spec).compile_mpe([], dry=True)
    _check_decode_order(split, spec.n)
    assert split.stats.final_tables == [((), 1)]
    rng = np.random.default_rng(7)
    for _ in range(30):
        cards, parents, cpts = MO.random_small_net(rng, 5, 16)
        names = [f"v{i}" for i in range(len(cards))]
        spec = synth.NetSpec(names, cards, parents, cpts)
        k = int(rng.integers(0, len(cards) + 1))
        ev = [names[int(v)] for v in rng.choice(len(cards), size=k, replace=False)]
        _check_decode_order(_compiler(spec).compile_mpe(ev, dry=True), len(cards))


def test_limits_raise_in_the_dry_pass():
    spec = synth.layered_dag()
    with pytest.raises(PlanTooLarge, match="no per-row executor"):
        _compiler(spec).compile_mpe([], dry=True)
    with pytest.raises(PlanTooLarge, match="no per-row executor"):
        _compiler(spec).compile_mpe(spec.names[:10], dry=True)
    alarm = synth.alarm()
    with pytest.raises(PlanTooLarge, match="argmax"):
        _compiler(alarm, mpe_argmax_budget_bytes=1 << 16).compile_mpe(synth.ALARM_EVIDENCE, dry=True)
    # the same budget is enough without evidence (the argmax tables are small)
    split = _compiler(alarm, mpe_argmax_budget_bytes=1 << 16).compile_mpe([], dry=True)
    assert split.argmax_bytes <= 1 << 16
    with pytest.raises(ValueError):
        _compiler(alarm).compile_mpe(["HRBP", "not_a_node"], dry=True)
    with pytest.raises(ValueError):
        _compiler(alarm).compile_mpe(["HRBP", "HRBP"], dry=True)


def test_complete_evidence_has_nothing_to_decode():
    spec = synth.asia()
    split = _compiler(spec).compile_mpe(spec.names, dry=True)
    assert split.hidden == [] and split.decode == [] and split.argmax_bytes == 0
    assert sorted(split.observed_families) == list(range(spec.n))


def test_ve_mpe_equals_enumeration_on_asia_and_random_dags():
    spec = synth.asia()
    nets = [(_net(spec), None)]
    rng = np.random.default_rng(11)
    for _ in range(12):
        cards, parents, cpts = MO.random_small_net(rng)
        nets.append((O.DiscreteNet(cards, parents, cpts), rng))
    n_rows = 0
    for net, r in nets:
        subsets = itertools.chain.from_iterable(itertools.combinations(range(net.n), k) for k in range(net.n + 1))
        if r is not None:
            subsets = [tuple(sorted(int(v) for v in r.choice(net.n, size=int(r.integers(0, net.n + 1)), replace=False)))
                       for _ in range(6)]
        for sub in subsets:
            ev = _configs([net.cards[v] for v in sub])
            best, second, assign = MO.enumerate_mpe(net, sub, ev)
            val, got = MO.ve_mpe(net, sub, ev)
            fin = np.isfinite(best)
            assert np.array_equal(fin, np.isfinite(val))
            np.testing.assert_allclose(val[fin], best[fin], rtol=1e-12, atol=1e-12)
            full = np.zeros((ev.shape[0], net.n), np.int64)
            for i, v in enumerate(sub):
                full[:, v] = ev[:, i]
            for v, c in got.items():
                full[:, v] = c
            # the traceback's assignment is optimal, and it is the oracle's wherever the best is unique
            np.testing.assert_allclose(MO.log_joint(net, full)[fin], best[fin], rtol=1e-12, atol=1e-12)
            clear = fin & ~(second >= best - 1e-4)
            assert np.array_equal(full[clear], assign[clear])
            n_rows += ev.shape[0]
    assert n_rows >= 3 ** 8


def test_mpe_step_layout_matches_the_header(tmp_path):
    from continuousbayesiannetwork_b200 import _native as N

    prog = tmp_path / "sz.c"
    prog.write_text('#include <stdio.h>\n#include "cbn_b200.h"\nint main(){printf("%zu %d\\n", sizeof(cbn_mpe_step), '
                    'CBN_MPE_MAX_SLOTS);return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    size, slots = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert size == C.sizeof(N.MpeStep) and slots == N.MPE_MAX_SLOTS


def _interpret(spec, split, ev_codes):
    """The decode schedule of ``split`` run by numpy: max-product tables built in the split's elimination order with the
    recorded scopes, each row's value from the finals plus the observed families, then the traceback step by step."""
    cards = spec.cards
    E = split.evidence
    Eset = set(E)
    factors = []
    for v in range(spec.n):
        if v in split.observed_families:
            continue
        with np.errstate(divide="ignore"):
            factors.append((spec.parents[v] + [v], np.log(np.asarray(spec.cpts[v], np.float64))))

    def expand(sc, t, full):
        perm = [sc.index(a) for a in full if a in sc]
        return t.transpose(perm).reshape([cards[a] if a in sc else 1 for a in full])

    tables = {}
    for v, scope in reversed(split.decode):                  # elimination order
        touching = [f for f in factors if v in f[0]]
        factors = [f for f in factors if v not in f[0]]
        assert sorted({a for sc, _ in touching for a in sc if a != v}) == sorted(scope)
        full = list(scope) + [v]
        acc = sum(expand(sc, t, full) for sc, t in touching)
        acc = np.broadcast_to(acc, [cards[a] for a in full])
        tables[v] = acc.argmax(axis=-1)                       # first maximum, as the device kernel
        factors.append((list(scope), acc.max(axis=-1)))
    pos = {v: i for i, v in enumerate(E)}
    n_rows = ev_codes.shape[0]
    value = np.zeros(n_rows)
    for sc, t in factors:
        assert set(sc) <= Eset
        value += t[tuple(ev_codes[:, pos[a]] for a in sc)] if sc else float(t)
    for v in split.observed_families:
        with np.errstate(divide="ignore"):
            value += np.log(spec.cpts[v][tuple(ev_codes[:, pos[a]] for a in spec.parents[v] + [v])])
    code = {v: ev_codes[:, i] for i, v in enumerate(E)}
    for v, scope in split.decode:
        code[v] = tables[v][tuple(code[a] for a in scope)] if scope else np.full(n_rows, int(tables[v]))
    return value, code


def test_decode_schedule_interpreter_on_asia():
    spec = synth.asia()
    net = _net(spec)
    for k in range(spec.n + 1):
        for sub in itertools.combinations(range(spec.n), k):
            split = _compiler(spec).compile_mpe([spec.names[v] for v in sub], dry=True)
            ev = _configs([spec.cards[v] for v in sub])
            value, code = _interpret(spec, split, ev)
            best, second, assign = MO.enumerate_mpe(net, sub, ev)
            fin = np.isfinite(best)
            assert np.array_equal(fin, np.isfinite(value))
            np.testing.assert_allclose(value[fin], best[fin], rtol=1e-12, atol=1e-12)
            full = np.stack([code[v] for v in range(spec.n)], axis=1)
            np.testing.assert_allclose(MO.log_joint(net, full)[fin], best[fin], rtol=1e-12, atol=1e-12)
            clear = fin & ~(second >= best - 1e-4)
            assert np.array_equal(full[clear], assign[clear])
