"""Junction-tree decoding without a GPU: the collect-only schedule, the decode rules interpreted in fp64 against
enumeration with random per-row masks, argument errors and the C ABI of cbn_jt_decode."""
import os
import sys
import types

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import impute_oracle as IO  # noqa: E402
import jt_oracle as JO  # noqa: E402
import mpe_oracle as MO  # noqa: E402

MISSING = 254


def _fams(parents):
    return [list(p) + [v] for v, p in enumerate(parents)]


def _rows(rng, cards, n):
    rows = np.stack([rng.integers(0, c, size=n) for c in cards], 1)
    rows = JO.random_masks(rng, rows, cards, rates=(0.0, 0.3, 0.7, 1.0))
    rows[:3] = MISSING
    rows[3:6, 0] = cards[0]
    rows[6:9, -1] = 255
    return rows


@pytest.mark.parametrize("seed", range(10))
def test_max_decode_interpreted_against_enumeration(seed):
    """The collect-only plan's tables, max-product collect and top-down argmax in fp64: the value and (where the best
    completion is unique by a margin) the completion of enumeration; observed cells kept; dead rows the same."""
    from continuousbayesiannetwork_b200 import jt

    rng = np.random.default_rng(seed)
    cards, parents, cpts = MO.random_small_net(rng, 3, 10)
    sch = jt.build_schedule(jt.build_structure(cards, _fams(parents)), [], collect_only=True)
    rows = _rows(rng, cards, 400)
    best, second, arg = IO.enumerate_mpe_rows(cards, parents, cpts, rows)
    got = IO.interpret_decode(sch, cpts, rows, 0)
    dead = ~np.isfinite(best)
    assert dead[3:9].all() and (~dead).sum() > 100
    assert np.array_equal(np.isneginf(got["log"]), dead)
    np.testing.assert_allclose(got["log"][~dead], best[~dead], rtol=1e-9, atol=1e-9)
    comp = got["codes"][0]
    assert (comp[dead] == IO.UNSEEN).all()
    live = ~dead
    np.testing.assert_allclose(IO.log_joint(cards, parents, cpts, comp[live]), best[live], rtol=1e-9, atol=1e-9)
    obs = (rows != MISSING) & live[:, None]
    assert np.array_equal(comp[obs], rows[obs])
    with np.errstate(invalid="ignore"):
        clear = live & (best - second > 1e-9)
    assert clear.sum() > 50 and np.array_equal(comp[clear], arg[clear])


@pytest.mark.parametrize("seed", range(10))
def test_sample_decode_probability_is_the_posterior_of_the_draw(seed):
    """Each draw's product of clique conditionals equals the enumerated P(completion | observed): the decode draws from
    the right conditionals, and every draw is a completion of positive probability consistent with the row."""
    from continuousbayesiannetwork_b200 import jt

    rng = np.random.default_rng(50 + seed)
    cards, parents, cpts = MO.random_small_net(rng, 3, 10)
    sch = jt.build_schedule(jt.build_structure(cards, _fams(parents)), [], collect_only=True)
    rows = _rows(rng, cards, 300)
    want_lp, _, _ = JO.enumerate_rows(cards, parents, cpts, rows)
    got = IO.interpret_decode(sch, cpts, rows, 1, seed=seed, first_row=1000, n_draws=3)
    dead = ~np.isfinite(want_lp)
    assert np.array_equal(np.isneginf(got["log"]), dead)
    np.testing.assert_allclose(got["log"][~dead], want_lp[~dead], rtol=1e-9, atol=1e-9)
    for d in range(3):
        comp = got["codes"][d]
        assert (comp[dead] == IO.UNSEEN).all()
        lj = IO.log_joint(cards, parents, cpts, comp[~dead])
        assert np.isfinite(lj).all()
        np.testing.assert_allclose(got["prob"][d][~dead], np.exp(lj - want_lp[~dead]), rtol=1e-9)
        obs = (rows != MISSING) & ~dead[:, None]
        assert np.array_equal(comp[obs], rows[obs])
    assert not np.array_equal(got["codes"][0], got["codes"][1])


def test_collect_only_schedule_has_up_messages_only():
    from continuousbayesiannetwork_b200 import jt, synth
    from continuousbayesiannetwork_b200.ve import DryTables, VECompiler

    spec = synth.alarm()
    dt = DryTables(spec.names, spec.cards, spec.parents_by_name())
    c = VECompiler(dt)
    full = jt.schedule_for(c)
    col = jt.collect_schedule(c)
    assert col is jt.collect_schedule(c) and col.structure is full.structure
    assert {o["kind"] for o in col.ops} == {jt.UP, jt.ROOT} and col.ops[-1]["kind"] == jt.ROOT
    assert col.msg_floats == 238 and full.msg_floats > col.msg_floats and col.marg_floats == 0
    # the same collect ops as the full schedule: same cliques, outputs, message offsets and inputs' messages
    head = full.ops[: len(col.ops)]
    for a, b in zip(col.ops, head):
        assert (a["kind"], a["clique"], a["out_vars"], a["out"]) == (b["kind"], b["clique"], b["out_vars"], b["out"])
        assert [m for m, _ in a["inputs"]] == [m for m, _ in b["inputs"]]
    assert col.shared_bytes(1) < full.shared_bytes(1)
    # existing schedules are unchanged by the new key
    assert jt.schedule_for(c) is full and ("jt", tuple(spec.cards), "collect") in c.structures


def test_collect_only_schedule_is_refused_in_the_dry_pass():
    from continuousbayesiannetwork_b200 import jt, synth
    from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, VECompiler

    spec = synth.random_ktree_dag()
    with pytest.raises(PlanTooLarge, match="clique"):
        jt.collect_schedule(VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name())))
    with pytest.raises(PlanTooLarge, match="cardinality 255"):
        jt.collect_schedule(VECompiler(DryTables(["a", "b"], [255, 2], {"b": ["a"]})))


# ------------------------------------------------------------------------------------------------ argument errors
def test_impute_arguments_are_checked_before_device_work():
    from continuousbayesiannetwork_b200.inference.exact import ExactInference

    def boom(*a, **k):
        raise AssertionError("device work")

    fake = types.SimpleNamespace(missing_codes=boom, junction_tree=boom, tables=None)
    for kw in ({"method": "map"}, {"method": "mpe", "n_draws": 2}, {"method": "sample", "n_draws": 0},
               {"method": "mpe", "n_draws": 0}, {"method": "sample", "first_row": -1}):
        with pytest.raises(ValueError):
            ExactInference.impute(fake, {}, **kw)


def test_network_impute_without_an_engine_method_is_refused():
    from continuousbayesiannetwork_b200.base.bayesian_network import BayesianNetwork

    net = types.SimpleNamespace(inference_obj=types.SimpleNamespace(), inference_obj_name="other", device="cpu",
                                nodes_obj={"a": None}, _latent_domains={})
    net._observed_columns = lambda data: BayesianNetwork._observed_columns(net, data)
    with pytest.raises(NotImplementedError):
        BayesianNetwork.impute(net, {"a": np.zeros(4)})
    with pytest.raises(ValueError):
        BayesianNetwork.impute(net, {"zz": np.zeros(4)})


# ------------------------------------------------------------------------------------------------ C ABI
@pytest.fixture(scope="module")
def native():
    from continuousbayesiannetwork_b200.build import build_native

    build_native()
    from continuousbayesiannetwork_b200 import _native

    return _native


def test_decode_symbol_is_exported_and_bound(native):
    import re

    lib = native.lib()
    assert hasattr(lib, "cbn_jt_decode") and "cbn_jt_decode" in native.SIGNATURES
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "cbn_b200.h")).read()
    defs = dict(re.findall(r"#define (CBN_JT_DECODE_\w+) (\d+)", hdr))
    assert defs == {"CBN_JT_DECODE_MAX": str(native.JT_DECODE_MAX), "CBN_JT_DECODE_SAMPLE": str(native.JT_DECODE_SAMPLE)}
    assert lib.cbn_jt_decode(None, None, None, 0, 0, 0, 0, 0, 1, None, 0, None, None) == native.ERR_INVALID
    assert b"ctx is NULL" in lib.cbn_last_error(None)
