"""GPU checks of junction-tree decoding per row (cbn_jt_decode): the most probable completion against fp64 enumeration,
the log-likelihood of the completions and the fixed-set MPE path on Alarm, draws against the fp64 interpretation of the
plan and their frequencies against enumeration and posterior_marginals, log P(e) < -200, row counts, batch splits and
draw prefixes that give the same bits, and plans that launch after smaller ones."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import em_oracle as EO  # noqa: E402
import impute_oracle as IO  # noqa: E402
import jt_oracle as JO  # noqa: E402
import mpe_oracle as MO  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MISSING = 254
MAX, SAMPLE = 0, 1


def _spec(cards, parents, cpts, names=None):
    from continuousbayesiannetwork_b200 import synth

    names = names or [f"v{i:02d}" for i in range(len(cards))]
    return synth.NetSpec(list(names), list(cards), [list(p) for p in parents],
                         [np.asarray(c, np.float64).astype(np.float32).astype(np.float64) for c in cpts])


def _install(spec):
    from continuousbayesiannetwork_b200.engine import install_cpts

    return install_cpts(spec, DEV)


def _codes(t, rows):
    n = rows.shape[0]
    c = t.new_code_matrix(n)
    c[:, :n] = torch.from_numpy(np.ascontiguousarray(rows.T.astype(np.uint8))).to(DEV)
    return c


def _sample(spec, n, seed):
    from continuousbayesiannetwork_b200.engine import sample_network

    return sample_network(spec, seed, 0, n, device=DEV)[:, :n].T.cpu().numpy().astype(np.int64)


def _decode(infer, codes, n, mode, n_draws=1, seed=0, first_row=0):
    """(out uint8 [n_draws * n_vars, ld] on the device, log float32 [n] on the device)."""
    t = infer.tables
    plan = infer.junction_tree().collect_plan()
    out = t.new_code_matrix(n, n_draws * len(t.names))
    lp = torch.empty(n, dtype=torch.float32, device=DEV)
    plan.decode(codes, n, mode, n_draws, seed, first_row, out, lp)
    return out, lp


def _rows_of(out, n, nv, n_draws=1):
    """int [n_draws, n, n_vars]."""
    return out[: n_draws * nv, :n].cpu().numpy().astype(np.int64).reshape(n_draws, nv, n).transpose(0, 2, 1)


def _loglik(infer, spec, comp):
    """log P of complete rows int [n, n_vars] through the fixed-set log P(e) path."""
    t = infer.tables
    n = comp.shape[0]
    return infer.evidence_plan(spec.names).run_codes(_codes(t, comp)[: spec.n], n).cpu().numpy().astype(np.float64)


# ------------------------------------------------------------------------------------------------ fp64 enumeration
@pytest.mark.parametrize("seed", range(8))
def test_mpe_against_enumeration(seed):
    rng = np.random.default_rng(300 + seed)
    cards, parents, cpts = MO.random_small_net(rng, 5, 9)
    spec = _spec(cards, parents, cpts)
    t, infer = _install(spec)
    n = 700
    rows = JO.random_masks(rng, _sample(spec, n, seed), cards, rates=(0.0, 0.2, 0.5, 0.8, 1.0))
    rows[:4] = MISSING
    rows[4:8, 0] = cards[0]
    rows[8:12, -1] = 255
    rows[12:60] = np.stack([rng.integers(0, c, size=48) for c in cards], 1)
    rows[60:70] = _sample(spec, 80, seed + 1)[70:80]                  # fully observed rows of positive probability
    out, lp = _decode(infer, _codes(t, rows), n, MAX)
    comp = _rows_of(out, n, spec.n)[0]
    got = lp.cpu().numpy().astype(np.float64)
    best, second, arg = IO.enumerate_mpe_rows(spec.cards, spec.parents, spec.cpts, rows)
    dead = ~np.isfinite(best)
    assert dead[4:12].all() and dead.any() and (~dead).sum() > 500
    assert np.array_equal(np.isneginf(got), dead)
    assert (comp[dead] == 255).all()
    np.testing.assert_allclose(got[~dead], best[~dead], rtol=1e-5, atol=1e-6)
    obs = (rows != MISSING) & ~dead[:, None]
    assert np.array_equal(comp[obs], rows[obs])
    clear = ~dead & (best - np.where(np.isfinite(second), second, -1e30) > 1e-5)
    assert clear.sum() > 400
    assert np.array_equal(comp[clear], arg[clear])


# ------------------------------------------------------------------------------------------------ Alarm
@pytest.mark.parametrize("rate", [0.05, 0.30])
def test_alarm_completions_have_log_prob_as_log_likelihood(rate):
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n = 1 << 20
    rng = np.random.default_rng(int(rate * 100))
    rows = _sample(spec, n, 5)
    rows[rng.random(rows.shape) < rate] = MISSING
    out, lp = _decode(infer, _codes(t, rows), n, MAX)
    comp = _rows_of(out, n, spec.n)[0]
    got = lp.cpu().numpy().astype(np.float64)
    assert np.isfinite(got).all()
    obs = rows != MISSING
    assert np.array_equal(comp[obs], rows[obs])
    ll = _loglik(infer, spec, comp)
    assert np.all(np.abs(ll - got) <= 1e-5 * np.abs(got) + 1e-5)


def test_alarm_without_missing_cells_agrees_with_the_fixed_set_mpe():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n = 20_000
    rows = _sample(spec, n, 9)
    rng = np.random.default_rng(2)
    subsets = [sorted(rng.choice(spec.n, size=k, replace=False).tolist()) for k in (1, 3, 5, 8, 12, 18, 25, 33)]
    for sub in subsets:
        ev = {spec.names[v]: torch.from_numpy(rows[:, v].astype(np.float32)) for v in sub}
        completed, lp = infer.impute(ev, method="mpe")
        assign, want = infer.most_probable_explanation(ev)
        np.testing.assert_allclose(lp.cpu().numpy(), want.cpu().numpy(), rtol=1e-5, atol=1e-5)
        for v in sub:
            assert torch.equal(completed[spec.names[v]].cpu(), ev[spec.names[v]])
    c0, l0 = infer.impute({}, method="mpe")
    a0, w0 = infer.most_probable_explanation({})
    assert l0.shape == (1,) and set(c0) == set(spec.names)
    np.testing.assert_allclose(l0.cpu().numpy(), w0.cpu().numpy(), rtol=1e-5)
    # fully observed rows: log_prob is the log-likelihood and the completion is the input
    full = {nm: torch.from_numpy(rows[:, v].astype(np.float32)) for v, nm in enumerate(spec.names)}
    completed, lp = infer.impute(full, method="mpe")
    np.testing.assert_allclose(lp.cpu().numpy(), _loglik(infer, spec, rows), rtol=1e-5)
    for nm in spec.names:
        assert torch.equal(completed[nm].cpu(), full[nm])


# ------------------------------------------------------------------------------------------------ sampling
def test_draws_equal_the_interpreted_plan():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n, draws = 4096, 4
    rng = np.random.default_rng(31)
    rows = _sample(spec, n, 12)
    rows[rng.random(rows.shape) < 0.3] = MISSING
    out, lp = _decode(infer, _codes(t, rows), n, SAMPLE, n_draws=draws, seed=77, first_row=123)
    got = _rows_of(out, n, spec.n, draws)
    sch = infer.junction_tree().collect_plan().schedule
    want = IO.interpret_decode(sch, [np.asarray(c, np.float32).astype(np.float64) for c in spec.cpts], rows, SAMPLE, seed=77,
                               first_row=123,
                               n_draws=draws)
    np.testing.assert_allclose(lp.cpu().numpy(), want["log"], rtol=1e-5)
    keep = want["margin"] > 1e-5
    assert (~keep).mean() < 0.01
    for d in range(draws):
        assert np.array_equal(got[d][keep[d]], want["codes"][d][keep[d]])


def _posterior(spec, row):
    """fp64 P(completion | row) over every completion: (grid int [n_vars, configs], p [configs])."""
    grid = np.indices(spec.cards).reshape(spec.n, -1)
    ok = np.ones(grid.shape[1], bool)
    for v in range(spec.n):
        if row[v] != MISSING:
            ok &= grid[v] == row[v]
    lj = np.where(ok, IO.log_joint(spec.cards, spec.parents, spec.cpts, grid.T), -np.inf)
    p = np.exp(lj - lj.max())
    return grid, p / p.sum()


def test_joint_draw_frequencies_on_a_small_network():
    rng = np.random.default_rng(8)
    cards, parents, cpts = MO.random_small_net(rng, 7, 8)
    spec = _spec(cards, parents, [np.where(c > 0, c + 0.05, c) / np.where(c > 0, c + 0.05, c).sum(-1, keepdims=True)
                                  for c in cpts])
    t, infer = _install(spec)
    rows = _sample(spec, 4, 3)
    for r in range(4):
        rows[r, rng.random(spec.n) < 0.6] = MISSING
    rows[0] = MISSING
    draws = 1 << 16
    out, lp = _decode(infer, _codes(t, rows), 4, SAMPLE, n_draws=draws, seed=5)
    got = _rows_of(out, 4, spec.n, draws)
    for r in range(4):
        grid, p = _posterior(spec, rows[r])
        idx = np.ravel_multi_index(tuple(got[:, r, v] for v in range(spec.n)), spec.cards)
        freq = np.bincount(idx, minlength=grid.shape[1]) / draws
        assert np.all(np.abs(freq - p) <= 5 * np.sqrt(p * (1 - p) / draws) + 1e-3)
        assert freq[p == 0].sum() == 0


def test_alarm_draw_frequencies_match_posterior_marginals():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    rng = np.random.default_rng(4)
    rows = _sample(spec, 16, 6)
    rows[rng.random(rows.shape) < 0.3] = MISSING
    ev = {nm: torch.from_numpy(np.where(rows[:, v] == MISSING, np.nan, rows[:, v]).astype(np.float32))
          for v, nm in enumerate(spec.names)}
    draws_n = 1 << 14
    draws, le = infer.impute(ev, method="sample", n_draws=draws_n, seed=3)
    marg, le2 = infer.posterior_marginals(ev)
    assert torch.equal(le, le2)
    for nm in spec.names:
        d = draws[nm].cpu().numpy().astype(np.int64)
        assert d.shape == (draws_n, 16)
        p = marg[nm].cpu().numpy().astype(np.float64)
        freq = np.stack([np.bincount(d[:, r], minlength=p.shape[1]) for r in range(16)]) / draws_n
        assert np.all(np.abs(freq - p) <= 5 * np.sqrt(p * (1 - p) / draws_n) + 1e-3), nm


def test_sample_log_evidence_is_bit_identical_to_posterior_marginals():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n = 50_000
    rng = np.random.default_rng(9)
    rows = _sample(spec, n, 14)
    rows[rng.random(rows.shape) < 0.2] = MISSING
    rows[rng.integers(0, n, 50), 2] = 255
    codes = _codes(t, rows)
    _, lp = _decode(infer, codes, n, SAMPLE, n_draws=2, seed=1)
    ref = torch.empty(n, dtype=torch.float32, device=DEV)
    infer.junction_tree().plan(None).run(codes, n, log_out=ref)
    assert torch.equal(lp, ref)
    ref2 = torch.empty(n, dtype=torch.float32, device=DEV)
    infer.junction_tree().collect_plan().run(codes, n, log_out=ref2)
    assert torch.equal(lp, ref2)
    ev = {nm: torch.from_numpy(np.where(rows[:, v] >= MISSING, np.nan, rows[:, v]).astype(np.float32))
          for v, nm in enumerate(spec.names)}
    _, le = infer.impute(ev, method="sample", n_draws=3, seed=4)
    _, le2 = infer.posterior_marginals(ev)
    assert torch.equal(le, le2)


def test_chain_with_log_evidence_below_minus_200():
    steps, card = 100, 8
    names, cards, parents, cpts = EO.hmm(steps=steps, k=3, card=card, seed=5)
    spec = _spec(cards, parents, cpts, names)
    t, infer = _install(spec)
    n = 1000
    rng = np.random.default_rng(3)
    rows = np.full((n, len(cards)), MISSING, np.int64)
    rows[:, steps:] = [int(np.argmin(np.asarray(spec.cpts[steps + tt]).sum(0))) for tt in range(steps)]
    rows[:, steps:][rng.random((n, steps)) < 0.1] = MISSING
    codes = _codes(t, rows)
    logA = [np.log(np.asarray(spec.cpts[tt])) for tt in range(steps)]

    def emit(tt, missing):
        o = rows[:, steps + tt]
        logb = np.log(np.asarray(spec.cpts[steps + tt]))
        return np.where((o == MISSING)[:, None], missing(logb)[None, :], logb[:, np.minimum(o, card - 1)].T)

    summed, maxed = (lambda b: np.zeros(b.shape[0])), (lambda b: b.max(1))     # a missing emission: summed out / maximised
    la = logA[0][None, :] + emit(0, summed)
    lv = logA[0][None, :] + emit(0, maxed)
    for tt in range(1, steps):
        la = np.logaddexp.reduce(la[:, :, None] + logA[tt][None], axis=1) + emit(tt, summed)
        lv = (lv[:, :, None] + logA[tt][None]).max(1) + emit(tt, maxed)
    fwd, vit = np.logaddexp.reduce(la, axis=1), lv.max(1)
    assert fwd.max() < -200
    out, lp = _decode(infer, codes, n, MAX)
    got = lp.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(got, vit, rtol=1e-5)
    comp = _rows_of(out, n, spec.n)[0]
    assert (comp < 254).all()
    np.testing.assert_allclose(IO.log_joint(spec.cards, spec.parents, spec.cpts, comp), vit, rtol=1e-5)
    out, lp = _decode(infer, codes, n, SAMPLE, n_draws=2, seed=8)
    np.testing.assert_allclose(lp.cpu().numpy().astype(np.float64), fwd, rtol=1e-5)
    assert (_rows_of(out, n, spec.n, 2) < 254).all()


# ------------------------------------------------------------------------------------------------ batches and bits
def test_row_counts_batch_splits_and_draw_prefixes_are_bit_identical():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    rng = np.random.default_rng(1)
    n = 148 * 8 * 32 * 2 + 77
    rows = _sample(spec, n, 21)
    rows[rng.random(rows.shape) < 0.2] = MISSING
    rows[rng.integers(0, n, 100), 3] = 255
    codes = _codes(t, rows)
    nv = spec.n
    for mode, draws in ((MAX, 1), (SAMPLE, 3)):
        out, lp = _decode(infer, codes, n, mode, n_draws=draws, seed=11, first_row=5)
        assert torch.isneginf(lp).sum().item() >= 90
        dead = torch.isneginf(lp).cpu().numpy()
        assert (_rows_of(out, n, nv, draws)[:, dead] == 255).all()
        again, lp2 = _decode(infer, codes, n, mode, n_draws=draws, seed=11, first_row=5)
        assert torch.equal(again[: draws * nv, :n], out[: draws * nv, :n]) and torch.equal(lp2, lp)    # deterministic
        for k in (0, 1, 31, 32, 33, 255, 4097):
            ok, lk = _decode(infer, codes, k, mode, n_draws=draws, seed=11, first_row=5)
            assert torch.equal(ok[: draws * nv, :k], out[: draws * nv, :k]) and torch.equal(lk, lp[:k])
        bounds = [0, 4096, 4096 + 48, 70_000, n]
        for a, b in zip(bounds[:-1], bounds[1:]):
            ok, lk = _decode(infer, codes[:, a:], b - a, mode, n_draws=draws, seed=11, first_row=5 + a)
            assert torch.equal(ok[: draws * nv, : b - a], out[: draws * nv, a:b]) and torch.equal(lk, lp[a:b])
        if mode == SAMPLE:
            one, _ = _decode(infer, codes, n, mode, n_draws=1, seed=11, first_row=5)
            assert torch.equal(one[:nv, :n], out[:nv, :n])
            other, _ = _decode(infer, codes, n, mode, n_draws=1, seed=12, first_row=5)
            assert not torch.equal(other[:nv, :n], out[:nv, :n])


def test_decode_plan_launches_after_a_smaller_plan_was_created():
    from continuousbayesiannetwork_b200 import synth

    spec = synth.alarm()
    t, infer = _install(spec)
    n = 5000
    rng = np.random.default_rng(12)
    rows = _sample(spec, n, 8)
    rows[rng.random(rows.shape) < 0.2] = MISSING
    codes = _codes(t, rows)
    o1, l1 = _decode(infer, codes, n, SAMPLE, n_draws=2)
    asia = synth.asia()
    ta, ia = _install(asia)
    arows = _sample(asia, 100, 1)
    ia.junction_tree().plan([0]).run(_codes(ta, arows), 100, log_out=torch.empty(100, device=DEV))
    _decode(ia, _codes(ta, arows), 100, MAX)
    o2, l2 = _decode(infer, codes, n, SAMPLE, n_draws=2)
    assert torch.equal(o2[: 2 * spec.n, :n], o1[: 2 * spec.n, :n]) and torch.equal(l2, l1)


def test_network_api_impute():
    import networkx as nx
    import pandas as pd

    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.base.bayesian_network import BayesianNetwork

    spec = synth.asia()
    rows = _sample(spec, 20_000, 2)
    g = nx.DiGraph()
    g.add_nodes_from(spec.names)
    for v, ps in enumerate(spec.parents):
        for p in ps:
            g.add_edge(spec.names[p], spec.names[v])
    df = pd.DataFrame({nm: rows[:, v].astype(np.float64) for v, nm in enumerate(spec.names)})
    bn = BayesianNetwork(g, df, {"estimator_name": "brute_force"}, {"inference_obj": "exact"}, device=DEV)
    rng = np.random.default_rng(3)
    holed = df.mask(rng.random(df.shape) < 0.3)
    completed, lp = bn.impute(holed)
    assert set(completed) == set(spec.names) and completed["lung"].shape == (20_000,)
    np.testing.assert_allclose(bn.log_likelihood(completed).cpu().numpy(), lp.cpu().numpy(), rtol=1e-5, atol=1e-5)
    for nm in spec.names:
        obs = ~holed[nm].isna().to_numpy()
        assert np.array_equal(completed[nm].cpu().numpy()[obs], holed[nm].to_numpy()[obs].astype(np.float32))
    draws, le = bn.impute(holed, method="sample", n_draws=4, seed=2)
    assert draws["lung"].shape == (4, 20_000) and torch.equal(le, bn.posterior_marginals(holed)[1])
    with pytest.raises(ValueError):
        bn.impute(holed, method="sample", n_draws=0)
