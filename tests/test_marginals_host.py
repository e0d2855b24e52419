"""Junction-tree calibration without a GPU: structure invariants, budgets, the plan's own tables interpreted in fp64
against enumeration with random per-row masks, argument errors and the C ABI of cbn_jt_*."""
import ctypes as C
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import em_oracle as EO  # noqa: E402
import jt_oracle as JO  # noqa: E402
import mpe_oracle as MO  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fams(parents):
    return [list(p) + [v] for v, p in enumerate(parents)]


def _nets():
    from continuousbayesiannetwork_b200 import synth

    out = []
    for spec in (synth.asia(), synth.alarm()):
        out.append((spec.name if hasattr(spec, "name") else spec.names[0], spec.cards, spec.parents))
    _, c, p, _ = EO.latent_class()
    out.append(("latent_class", c, p))
    _, c, p, _ = EO.hmm(steps=8)
    out.append(("hmm", c, p))
    rng = np.random.default_rng(0)
    for k in range(25):
        c, p, _ = MO.random_small_net(rng, 3, 14)
        out.append((f"random{k}", c, p))
    return out


@pytest.mark.parametrize("name,cards,parents", _nets())
def test_structure_invariants(name, cards, parents):
    from continuousbayesiannetwork_b200 import jt

    st = jt.build_structure(cards, _fams(parents))
    n_cl = len(st.cliques)
    sets = [set(c) for c in st.cliques]
    assert sorted(st.collect) == list(range(n_cl)) and st.collect[-1] == st.root
    assert [i for i in range(n_cl) if st.parent[i] < 0] == [st.root]
    seen = set()
    for i in st.collect:                                          # children come before their parent
        assert all(c in seen for c in st.children[i])
        seen.add(i)
    for i in range(n_cl):                                         # every clique is maximal
        assert not any(i != j and sets[i] <= sets[j] for j in range(n_cl))
    for v in range(len(cards)):                                   # running intersection: v's cliques form a subtree
        holders = [i for i in range(n_cl) if v in sets[i]]
        assert holders
        tops = [i for i in holders if st.parent[i] < 0 or v not in sets[st.parent[i]]]
        assert len(tops) == 1, (name, v)
        assert v in sets[st.home[v]] and st.cells(st.home[v]) == min(st.cells(i) for i in holders)
    for v, fv in enumerate(_fams(parents)):                       # every family inside its home clique
        assert set(fv) <= sets[st.assign[v]]
    sch = jt.build_schedule(st, range(len(cards)))
    for o in sch.ops:                                             # separators are the intersection with the parent
        if o["kind"] == jt.UP:
            i = o["clique"]
            assert o["out_vars"] == sorted(sets[i] & sets[st.parent[i]])
        if o["kind"] == jt.DOWN:
            child = next(c for c in st.children[o["clique"]] if st.separator(c) == o["out_vars"])
            assert st.parent[child] == o["clique"]
    assert sum(o["kind"] == jt.ROOT for o in sch.ops) == 1


def test_alarm_and_asia_sizes():
    from continuousbayesiannetwork_b200 import jt, synth

    for spec, want in ((synth.asia(), (6, 8, 40, 16)), (synth.alarm(), (27, 144, 1038, 238))):
        st = jt.build_structure(spec.cards, _fams(spec.parents))
        cells = [st.cells(i) for i in range(len(st.cliques))]
        per_direction = sum(int(np.prod([spec.cards[v] for v in st.separator(i)])) for i in range(len(cells))
                            if st.parent[i] >= 0)
        assert (len(cells), max(cells), sum(cells), per_direction) == want


def test_ktree_dag_is_refused_without_device_work():
    from continuousbayesiannetwork_b200 import jt, synth
    from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, VECompiler

    spec = synth.random_ktree_dag()
    dt = DryTables(spec.names, spec.cards, spec.parents_by_name())
    with pytest.raises(PlanTooLarge, match="clique"):
        jt.compile_tree(VECompiler(dt), dry=True)


def test_budgets_and_cardinality_255_are_refused():
    from continuousbayesiannetwork_b200 import jt
    from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, VECompiler

    dt = DryTables(["a", "b"], [255, 2], {"b": ["a"]})
    with pytest.raises(PlanTooLarge, match="cardinality 255"):
        jt.compile_tree(VECompiler(dt), dry=True)
    ok = DryTables(["a", "b"], [254, 2], {"b": ["a"]})
    assert jt.compile_tree(VECompiler(ok), dry=True).marg_floats == 256
    with pytest.raises(PlanTooLarge, match="floats of messages"):
        jt.compile_tree(VECompiler(DryTables(["a", "b", "c"], [60, 60, 2], {"b": ["a"], "c": ["b"]}), row_temp_floats=50),
                        dry=True)


@pytest.mark.parametrize("seed", range(12))
def test_plan_tables_interpreted_against_enumeration(seed):
    """The schedule jt.py hands to cbn_jt_plan_create, run in fp64, equals enumeration for every node and family, with
    per-row masks from 0 to 100 % missing, dead rows and rows of probability zero."""
    from continuousbayesiannetwork_b200 import jt

    rng = np.random.default_rng(seed)
    cards, parents, cpts = MO.random_small_net(rng, 3, 10)
    st = jt.build_structure(cards, _fams(parents))
    sch = jt.build_schedule(st, range(len(cards)))
    n = 400
    rows = np.stack([rng.integers(0, c, size=n) for c in cards], 1)
    rows = JO.random_masks(rng, rows, cards, rates=(0.0, 0.3, 0.7, 1.0))
    rows[:3] = JO.MISSING
    rows[3:6] = np.asarray(cards)[None, :] - 1
    rows[6:9, 0] = cards[0]
    rows[9:12, -1] = 255
    want_lp, want_m, want_f = JO.enumerate_rows(cards, parents, cpts, rows)
    lp, run, fams = JO.interpret(sch, cpts, rows)
    assert np.array_equal(np.isneginf(lp), np.isneginf(want_lp)) and np.isneginf(lp[6:12]).all()
    live = np.isfinite(want_lp)
    np.testing.assert_allclose(lp[live], want_lp[live], rtol=1e-10, atol=1e-12)
    assert np.abs(lp[:3]).max() < 1e-12
    for v in range(len(cards)):
        o = sch.node_out[v]
        np.testing.assert_allclose(run[live, o: o + cards[v]], want_m[v][live], atol=1e-10)
        np.testing.assert_allclose(fams[v][live], want_f[v][live], atol=1e-10)
        assert np.isnan(run[~live, o: o + cards[v]]).all()


def test_subset_of_nodes_runs_only_the_needed_messages():
    from continuousbayesiannetwork_b200 import jt, synth

    spec = synth.alarm()
    st = jt.build_structure(spec.cards, _fams(spec.parents))
    full = jt.build_schedule(st, range(spec.n))
    tv = [spec.names.index(n) for n in synth.ALARM_TARGETS]
    part = jt.build_schedule(st, tv)
    assert part.marg_floats == sum(spec.cards[v] for v in tv)
    downs = lambda s, bit: sum(1 for o in s.ops if o["kind"] == jt.DOWN and o["needed"] & bit)
    assert downs(part, jt.NEED_NODES) < downs(full, jt.NEED_NODES)
    assert downs(part, jt.NEED_FAMILIES) == downs(full, jt.NEED_FAMILIES)


# ------------------------------------------------------------------------------------------------ argument errors
def _fake_network(columns):
    from continuousbayesiannetwork_b200.base.bayesian_network import BayesianNetwork

    net = types.SimpleNamespace(inference_obj=types.SimpleNamespace(evidence_plan=lambda *a: None), inference_obj_name="exact",
                                device="cpu", nodes_obj={n: None for n in columns}, _latent_domains={})
    net._observed_columns = lambda data: BayesianNetwork._observed_columns(net, data)
    return net


def test_unknown_missing_setting_is_refused():
    from continuousbayesiannetwork_b200.base.bayesian_network import BayesianNetwork

    net = _fake_network(["a"])
    with pytest.raises(ValueError, match="missing must be"):
        BayesianNetwork.fit_em(net, {"a": np.zeros(4)}, missing="drop")


def test_all_nan_column_is_refused():
    from continuousbayesiannetwork_b200.base.bayesian_network import BayesianNetwork

    net = _fake_network(["a", "b"])
    with pytest.raises(ValueError, match="only NaN"):
        BayesianNetwork.fit_em(net, {"a": np.zeros(4), "b": np.full(4, np.nan)}, missing="marginalize")


# ------------------------------------------------------------------------------------------------ C ABI
@pytest.fixture(scope="module")
def native():
    from continuousbayesiannetwork_b200.build import build_native

    build_native()
    from continuousbayesiannetwork_b200 import _native

    return _native


def test_jt_symbols_are_exported_and_bound(native):
    lib = native.lib()
    for name in ("cbn_jt_plan_create", "cbn_jt_plan_destroy", "cbn_jt_run", "cbn_jt_plan_stats"):
        assert hasattr(lib, name) and name in native.SIGNATURES
    assert native.MISSING == 254 and native.UNSEEN == 255
    assert lib.cbn_jt_run(None, None, None, 0, 0, None, None, None, None) == native.ERR_INVALID
    assert b"ctx is NULL" in lib.cbn_last_error(None)
    assert lib.cbn_jt_plan_create(None, 0, None, 0, None, None, 0, 0, None, None, 0, None, 0, 0, 0, 0, None, None) == \
        native.ERR_INVALID
    lib.cbn_jt_plan_destroy(None)


def test_jt_struct_layouts_match_the_header(native, tmp_path):
    prog = tmp_path / "sz.c"
    prog.write_text('#include <stdio.h>\n#include "cbn_b200.h"\nint main(){printf("%zu %zu %d %d\\n", sizeof(cbn_jt_clique), '
                    'sizeof(cbn_jt_op), CBN_MISSING, CBN_JT_MAX_MEMBERS);return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out == [C.sizeof(native.JtClique), C.sizeof(native.JtOp), native.MISSING, native.JT_MAX_MEMBERS]


def test_shared_memory_budget_is_checked_in_the_dry_pass():
    """The dry pass restates the kernel's shared-memory layout (Schedule.shared_bytes; the GPU tests compare it with
    cbn_jt_plan_stats): a tree over the budget is refused before any device work, one under it is accepted."""
    from continuousbayesiannetwork_b200 import jt
    from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, VECompiler

    def dry(steps):
        names, cards, parents, _ = EO.hmm(steps=steps, k=3, card=8)
        return DryTables(names, cards, {names[v]: [names[p] for p in ps] for v, ps in enumerate(parents)})

    sch = jt.compile_tree(VECompiler(dry(100)), dry=True)
    assert 0.75 * jt.SMEM_BUDGET_BYTES < sch.shared_bytes(1) <= jt.SMEM_BUDGET_BYTES
    with pytest.raises(PlanTooLarge, match="shared memory"):
        jt.compile_tree(VECompiler(dry(130)), dry=True)


def test_structure_and_schedules_survive_a_cpt_change():
    """After an M-step only the clique tables are rebuilt: the schedules are kept by the compiler, per output set."""
    from continuousbayesiannetwork_b200 import jt, synth
    from continuousbayesiannetwork_b200.ve import DryTables, VECompiler

    spec = synth.alarm()
    dt = DryTables(spec.names, spec.cards, spec.parents_by_name())
    c = VECompiler(dt)
    full, part = jt.schedule_for(c), jt.schedule_for(c, [3, 5])
    dt.cond_version = 7
    assert jt.schedule_for(c) is full and jt.schedule_for(c, [3, 5]) is part and jt.compile_tree(c, dry=True) is full
    assert part.structure is full.structure and part.nodes == [3, 5]
