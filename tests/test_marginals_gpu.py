"""GPU checks of junction-tree calibration per row (cbn_jt_run): marginals, log P(observed cells) and expected counts with
per-row missing values against fp64 enumeration and against the existing engine, range, row counts around the tile and
grid sizes, bit-identical batch splits, and EM with missing cells through the network API."""
import os
import sys

import networkx as nx
import numpy as np
import pandas as pd
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import em_oracle as EO  # noqa: E402
import jt_oracle as JO  # noqa: E402
import mpe_oracle as MO  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ONE = float(1 << 32)
MISSING = 254


def _spec(cards, parents, cpts, names=None):
    """A NetSpec with fp32-rounded CPTs (as the device holds them); parents in name order."""
    from continuousbayesiannetwork_b200 import synth

    names = names or [f"v{i:02d}" for i in range(len(cards))]
    return synth.NetSpec(list(names), list(cards), [list(p) for p in parents],
                         [np.asarray(c, np.float64).astype(np.float32).astype(np.float64) for c in cpts])


def _install(spec):
    from continuousbayesiannetwork_b200.engine import install_cpts

    return install_cpts(spec, DEV)


def _codes(t, rows):
    """int [n, n_vars] -> device uint8 [n_vars, ld]."""
    n = rows.shape[0]
    c = t.new_code_matrix(n)
    c[:, :n] = torch.from_numpy(np.ascontiguousarray(rows.T.astype(np.uint8))).to(DEV)
    return c


def _run(infer, codes, n, nodes=None, marg=True, log=True, acc=None):
    plan = infer.junction_tree().plan(nodes)
    m = torch.empty((n, plan.schedule.marg_floats), dtype=torch.float32, device=DEV) if marg else None
    lp = torch.empty(n, dtype=torch.float32, device=DEV) if log else None
    plan.run(codes, n, marg_out=m, log_out=lp, acc=acc)
    return plan, m, lp


def _sample(spec, n, seed):
    from continuousbayesiannetwork_b200.engine import sample_network

    return sample_network(spec, seed, 0, n, device=DEV)[:, :n].T.cpu().numpy().astype(np.int64)


# ------------------------------------------------------------------------------------------------ fp64 enumeration
@pytest.mark.parametrize("seed", range(8))
def test_marginals_and_log_evidence_against_enumeration(seed):
    rng = np.random.default_rng(100 + seed)
    cards, parents, cpts = MO.random_small_net(rng, 5, 9)
    spec = _spec(cards, parents, cpts)
    t, infer = _install(spec)
    n = 700
    rows = JO.random_masks(rng, _sample(spec, n, seed), cards, rates=(0.0, 0.2, 0.5, 0.8, 1.0))
    rows[:4] = MISSING                                            # fully missing rows: log P = 0, prior marginals
    rows[4:8, 0] = cards[0]                                       # out of domain
    rows[8:12, -1] = 255                                          # CBN_UNSEEN
    # rows of probability zero: observe every node at a random value (deterministic CPT rows make many impossible)
    rows[12:60] = np.stack([rng.integers(0, c, size=48) for c in cards], 1)
    plan, m, lp = _run(infer, _codes(t, rows), n)
    want_lp, want_m, _ = JO.enumerate_rows(spec.cards, spec.parents, spec.cpts, rows)
    got_lp = lp.cpu().numpy().astype(np.float64)
    dead = ~np.isfinite(want_lp)
    assert dead[4:12].all() and dead.any() and (~dead).sum() > 500
    assert np.array_equal(np.isneginf(got_lp), dead)
    np.testing.assert_allclose(got_lp[~dead], want_lp[~dead], rtol=1e-5, atol=1e-6)
    assert np.abs(got_lp[:4]).max() < 1e-5
    run = m.cpu().numpy().astype(np.float64)
    assert np.isnan(run[dead]).all()
    for v in range(len(cards)):
        o = plan.schedule.node_out[v]
        np.testing.assert_allclose(run[~dead, o: o + cards[v]], want_m[v][~dead], atol=1e-5)


def test_expected_counts_against_enumeration():
    """JT's own contribution (the rows in which a family has a missing member) on latent_class, hmm and Asia."""
    from continuousbayesiannetwork_b200 import synth

    cases = [(EO.latent_class(n_children=6, k=3, card=3, seed=1), [0]),
             (EO.hmm(steps=5, k=3, card=3, seed=2), list(range(5))),
             ((synth.asia().names, synth.asia().cards, synth.asia().parents, synth.asia().cpts), [])]
    rng = np.random.default_rng(7)
    for (names, cards, parents, cpts), hidden in cases:
        spec = _spec(cards, parents, cpts, names)
        t, infer = _install(spec)
        n = 3000
        rows = _sample(spec, n, 11)
        rows[rng.random(rows.shape) < 0.15] = MISSING
        rows[:, hidden] = MISSING
        acc = torch.zeros(t.total_cells, dtype=torch.int64, device=DEV)
        _run(infer, _codes(t, rows), n, marg=False, log=False, acc=acc)
        want = JO.expected_counts(spec.cards, spec.parents, spec.cpts, rows)
        got = acc.double().cpu().numpy() / ONE
        for v, name in enumerate(spec.names):
            g = got[t.offsets[v]: t.offsets[v] + t.n_cells[v]].reshape(want[v].shape)
            np.testing.assert_allclose(g, want[v], atol=2e-6 * n, rtol=1e-5, err_msg=name)


def test_complete_data_adds_nothing():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n = 50_000
    rows = _sample(spec, n, 3)
    acc = torch.zeros(t.total_cells, dtype=torch.int64, device=DEV)
    _, m, lp = _run(infer, _codes(t, rows), n, acc=acc)
    assert int(acc.abs().sum().item()) == 0
    # fully observed: one-hot marginals, log P = the log-likelihood of the rows
    ll = infer.evidence_plan(spec.names).run_codes(_codes(t, rows)[: spec.n], n)
    np.testing.assert_allclose(lp.cpu().numpy(), ll.cpu().numpy(), rtol=1e-5)
    want = np.concatenate([np.eye(c)[rows[:, v]] for v, c in enumerate(spec.cards)], 1)
    assert np.array_equal(m.cpu().numpy(), want.astype(np.float32))


# ------------------------------------------------------------------------------------------------ the existing engine
@pytest.mark.parametrize("rate", [0.05, 0.30])
def test_alarm_agrees_with_the_engine_per_pattern(rate):
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n = 1 << 20
    rng = np.random.default_rng(int(rate * 100))
    rows = _sample(spec, n, 5)
    rows[rng.random(rows.shape) < rate] = MISSING
    codes = _codes(t, rows)
    plan, m, lp = _run(infer, codes, n)
    run = m.cpu().numpy()
    got_lp = lp.cpu().numpy()
    assert np.isfinite(got_lp).all()
    sums = np.stack([run[:, o: o + spec.cards[v]].sum(1) for v, o in plan.schedule.node_out.items()], 1)
    assert np.abs(sums - 1).max() < 1e-5
    for v, o in plan.schedule.node_out.items():                       # observed nodes are one-hot
        obs = rows[:, v] != MISSING
        assert np.array_equal(run[obs, o: o + spec.cards[v]], np.eye(spec.cards[v], dtype=np.float32)[rows[obs, v]])
    patterns, inverse, counts = np.unique(rows == MISSING, axis=0, return_inverse=True, return_counts=True)
    inverse = inverse.reshape(-1)
    checked = 0
    for p in np.argsort(-counts)[:6]:
        sel = np.nonzero(inverse == p)[0]
        ev = [v for v in range(spec.n) if not patterns[p][v]]
        ev_names = [spec.names[v] for v in ev]
        evc = t.new_code_matrix(len(sel), max(len(ev), 1))
        evc[: len(ev), : len(sel)] = torch.from_numpy(np.ascontiguousarray(rows[sel][:, ev].T.astype(np.uint8))).to(DEV)
        want_lp = infer.evidence_plan(ev_names).run_codes(evc, len(sel)).cpu().numpy()
        np.testing.assert_allclose(got_lp[sel], want_lp, rtol=1e-5)
        for v in [u for u in range(spec.n) if patterns[p][u]][:6]:
            want = infer.plan(spec.names[v], ev_names).run_codes(evc, len(sel)).cpu().numpy()
            o = plan.schedule.node_out[v]
            np.testing.assert_allclose(run[sel, o: o + spec.cards[v]], want, atol=1e-5)
            checked += 1
    assert checked >= 4


def test_log_evidence_below_minus_200():
    """A long hidden chain with many observed emissions: log P(e) far below the fp32 range of P(e) itself."""
    steps, card = 100, 8
    names, cards, parents, cpts = EO.hmm(steps=steps, k=3, card=card, seed=5)
    spec = _spec(cards, parents, cpts, names)
    t, infer = _install(spec)
    n = 2000
    rng = np.random.default_rng(3)
    rows = np.full((n, len(cards)), MISSING, np.int64)
    # every emission at its least likely value (summed over states), 10 % of them missing
    rows[:, steps:] = [int(np.argmin(np.asarray(spec.cpts[steps + tt]).sum(0))) for tt in range(steps)]
    rows[:, steps:][rng.random((n, steps)) < 0.1] = MISSING
    _, m, lp = _run(infer, _codes(t, rows), n, nodes=[0, steps - 1])
    # exact: the forward recursion in log space
    def emit(tt):
        o = rows[:, steps + tt]
        e = np.log(np.asarray(spec.cpts[steps + tt]))[:, np.minimum(o, card - 1)].T
        return np.where((o == MISSING)[:, None], 0.0, e)
    la = np.log(np.asarray(spec.cpts[0]))[None, :] + emit(0)
    for tt in range(1, steps):
        la = np.logaddexp.reduce(la[:, :, None] + np.log(np.asarray(spec.cpts[tt]))[None], axis=1) + emit(tt)
    want = np.logaddexp.reduce(la, axis=1)
    got = lp.cpu().numpy().astype(np.float64)
    assert want.max() < -200
    np.testing.assert_allclose(got, want, rtol=1e-5)
    np.testing.assert_allclose(m.cpu().numpy()[:, 3:], np.exp(la - want[:, None]), atol=1e-5)     # filtering = smoothing at the end
    assert np.abs(m.cpu().numpy().reshape(n, 2, 3).sum(2) - 1).max() < 1e-5


# ------------------------------------------------------------------------------------------------ batches and bits
def test_row_counts_and_batch_splits_are_bit_identical():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    rng = np.random.default_rng(1)
    n = 148 * 8 * 32 * 2 + 77                                    # more than one grid round
    rows = _sample(spec, n, 21)
    rows[rng.random(rows.shape) < 0.2] = MISSING
    rows[rng.integers(0, n, 100), 3] = 255                       # dead rows
    codes = _codes(t, rows)
    acc = torch.zeros(t.total_cells, dtype=torch.int64, device=DEV)
    _, m, lp = _run(infer, codes, n, acc=acc)
    assert torch.isneginf(lp).sum().item() >= 90
    for k in (1, 31, 32, 33, 255, 256, 257, 4097):
        acc_k = torch.zeros_like(acc)
        _, mk, lk = _run(infer, codes, k, acc=acc_k)
        assert torch.equal(mk, m[:k]) or torch.equal(torch.nan_to_num(mk, 7.0), torch.nan_to_num(m[:k], 7.0))
        assert torch.equal(lk, lp[:k])
    # a split at 16-row boundaries: the same marginals, log P and counts
    acc_s = torch.zeros_like(acc)
    parts_m, parts_l = [], []
    bounds = [0, 4096, 4096 + 48, 70_000, n]
    for a, b in zip(bounds[:-1], bounds[1:]):
        _, mk, lk = _run(infer, codes[:, a:], b - a, acc=acc_s)
        parts_m.append(mk)
        parts_l.append(lk)
    assert torch.equal(torch.nan_to_num(torch.cat(parts_m), 7.0), torch.nan_to_num(m, 7.0))
    assert torch.equal(torch.cat(parts_l), lp)
    assert torch.equal(acc_s, acc)
    assert int(acc.sum().item()) > 0


# ------------------------------------------------------------------------------------------------ EM with missing cells
def _oracle_em(spec, rows, cpts, iters):
    """fp64 EM with per-row missing cells: every live row adds its family posteriors (one-hot where observed)."""
    hist = []
    for _ in range(iters):
        lp, _, fam = JO.enumerate_rows(spec.cards, spec.parents, cpts, rows)
        live = np.isfinite(lp)
        hist.append(float(lp[live].sum()))
        counts = [fam[v][live].sum(0).reshape([spec.cards[u] for u in list(spec.parents[v]) + [v]]) for v in range(spec.n)]
        cpts = EO.m_step(counts)
    return cpts, hist


def test_em_with_missing_cells_matches_fp64_em():
    from continuousbayesiannetwork_b200 import em as EMM

    names, cards, parents, cpts = EO.latent_class(n_children=5, k=3, card=3, seed=4, sharp=1.0)
    spec = _spec(cards, parents, cpts, names)
    t, infer = _install(spec)
    n = 20_000
    rng = np.random.default_rng(5)
    rows = _sample(spec, n, 13)
    rows[rng.random(rows.shape) < 0.10] = MISSING
    rows[:, 0] = MISSING                                          # the latent class
    codes = _codes(t, rows)
    t.count(codes, n)
    t.hidden = {0}
    em = EMM.JTEM(t, infer, codes, n, [0])
    init = [np.asarray(c, np.float64) for c in EO.latent_class(n_children=5, k=3, card=3, seed=9)[3]]
    cur = torch.zeros(t.total_cells, dtype=torch.float32, device=DEV)
    for v in range(spec.n):
        cur[t.offsets[v]: t.offsets[v] + t.n_cells[v]] = torch.from_numpy(init[v].reshape(-1).astype(np.float32)).to(DEV)
    em.initialise("current", 0, cur)
    start = [t.table_view(t.cond, nm).double().cpu().numpy() for nm in spec.names]
    res = em.fit(max_iter=6, tol=float("-inf"))
    want, hist = _oracle_em(spec, rows, start, 6)
    for v, nm in enumerate(spec.names):
        np.testing.assert_allclose(t.table_view(t.cond, nm).double().cpu().numpy(), want[v], atol=1e-4, err_msg=nm)
    np.testing.assert_allclose(res.log_likelihood[:6], hist, rtol=1e-5)
    ll = np.asarray(res.log_likelihood)
    assert np.all(np.diff(ll) > -1e-6 * np.abs(ll[:-1]))


def _frame(spec, rows):
    return pd.DataFrame({nm: np.where(rows[:, v] == MISSING, np.nan, rows[:, v].astype(np.float64))
                         for v, nm in enumerate(spec.names)})


def _dag(spec):
    g = nx.DiGraph()
    g.add_nodes_from(spec.names)
    for v, ps in enumerate(spec.parents):
        for p in ps:
            g.add_edge(spec.names[p], spec.names[v])
    return g


def test_network_api_missing_values_and_update_knowledge():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.base.bayesian_network import BayesianNetwork

    spec = synth.asia()
    rows = _sample(spec, 30_000, 2)
    df_full = _frame(spec, rows)
    plc = {"estimator_name": "brute_force"}
    bn = BayesianNetwork(_dag(spec), df_full, plc, {"inference_obj": "exact"}, device=DEV)
    ordinary = bn.tables.cond.clone()
    # complete data: the ordinary fit's CPTs, bit for bit
    res = bn.fit_em(df_full, missing="marginalize")
    assert res.n_iter == 1 and torch.equal(bn.tables.cond, ordinary)
    # NaN cells: marginals of the network API agree with the plan and observed nodes are one-hot
    rng = np.random.default_rng(4)
    holed = rows.copy()
    holed[rng.random(rows.shape) < 0.2] = MISSING
    df = _frame(spec, holed)
    with pytest.raises(ValueError):
        bn.fit_em(df)
    marg, lp = bn.posterior_marginals(df, nodes=["lung", "tub", "smoke"])
    assert set(marg) == {"lung", "tub", "smoke"} and marg["lung"].shape == (30_000, 2)
    full, lp2 = bn.posterior_marginals(df)
    assert torch.equal(lp, lp2) and torch.equal(full["lung"], marg["lung"])
    obs = holed[:, spec.names.index("smoke")] != MISSING
    np.testing.assert_array_equal(full["smoke"].cpu().numpy()[obs], np.eye(2, dtype=np.float32)[holed[obs, 2]])
    res = bn.fit_em(df, missing="marginalize", max_iter=30, tol=1e-9)
    assert res.n_iter >= 2 and np.all(np.diff(res.log_likelihood) > -1e-5 * np.abs(res.log_likelihood[:-1]))
    assert bn._em_settings["missing"] == "marginalize"
    # update_knowledge re-runs with the stored setting (the default would refuse NaN)
    holed2 = _sample(spec, 20_000, 3)
    holed2[rng.random(holed2.shape) < 0.1] = MISSING
    bn.update_knowledge(_frame(spec, holed2))
    assert bn.em_result.n_iter >= 2 and bn._em_settings["missing"] == "marginalize"
    # latent= with em_missing from the config
    plc2 = dict(plc, em_missing="marginalize", em_max_iter=5)
    df_lat = _frame(spec, holed).drop(columns=["either"])
    bn2 = BayesianNetwork(_dag(spec), df_lat, plc2, {"inference_obj": "exact"}, device=DEV, latent={"either": 2})
    assert 2 <= bn2.em_result.n_iter <= 5 and np.isfinite(bn2.em_result.log_likelihood).all()


def _plan_smem(plan):
    import ctypes as C

    from continuousbayesiannetwork_b200 import _native as N

    smem, warps = C.c_int64(), C.c_int32()
    assert N.lib().cbn_jt_plan_stats(plan.handle, C.byref(smem), C.byref(warps)) == 0
    return smem.value, warps.value


def test_cached_plans_run_after_a_smaller_plan_is_created():
    """The kernel's shared-memory limit belongs to the kernel, not to a plan: a plan with a larger footprint created
    first must still launch after a smaller plan was created, on the same network and across networks."""
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n = 5000
    rng = np.random.default_rng(12)
    rows = _sample(spec, n, 8)
    rows[rng.random(rows.shape) < 0.2] = MISSING
    codes = _codes(t, rows)
    big, m1, l1 = _run(infer, codes, n)                                  # every node: the largest footprint
    small, _, _ = _run(infer, codes, n, nodes=[spec.names.index("HR")])
    em_plan, _, _ = _run(infer, codes, n, nodes=[], marg=False)
    assert _plan_smem(big)[0] > _plan_smem(small)[0] > _plan_smem(em_plan)[0]
    for p in (big, small, em_plan):                                      # the dry pass restates the kernel's layout
        smem, warps = _plan_smem(p)
        assert smem == p.schedule.shared_bytes(warps)
    _, m2, l2 = _run(infer, codes, n)                                    # the cached large plan, after the small ones
    assert torch.equal(torch.nan_to_num(m2, 7.0), torch.nan_to_num(m1, 7.0)) and torch.equal(l2, l1)
    # across networks: Asia (a small plan) between two runs of Alarm's
    asia = synth.asia()
    ta, ia = _install(asia)
    arows = _sample(asia, 100, 1)
    _run(ia, _codes(ta, arows), 100)
    _, m3, l3 = _run(infer, codes, n)
    assert torch.equal(torch.nan_to_num(m3, 7.0), torch.nan_to_num(m1, 7.0)) and torch.equal(l3, l1)
