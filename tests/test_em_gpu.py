"""GPU checks of EM: the accumulation kernel (cbn_ess_run) bit for bit against numpy, joint posteriors by the chain rule
and whole E-steps against fp64 enumeration, full EM against a numpy fp64 EM, complete data against the ordinary fit,
recovery of a latent-class model, determinism over chunkings, and the network API."""
import ctypes as C
import itertools
import os
import sys
import types

import networkx as nx
import numpy as np
import pandas as pd
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import em_oracle as EO  # noqa: E402
import mpe_oracle as MO  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PL = {"estimator_name": "brute_force"}
INF = {"inference_obj": "exact"}
ONE = float(1 << 32)


def _spec(names, cards, parents, cpts):
    """A NetSpec with fp32-rounded CPTs (as the device holds them); parents must already be in name order."""
    from continuousbayesiannetwork_b200 import synth

    return synth.NetSpec(list(names), list(cards), [list(p) for p in parents],
                         [np.asarray(c, np.float64).astype(np.float32).astype(np.float64) for c in cpts])


def _names(n):
    return [f"v{i:02d}" for i in range(n)]


def _em(spec, codes_np, hidden, chunk_rows=None, init=True, **cfg):
    """EM over tables holding ``spec``'s CPTs, with the observed columns of ``codes_np`` (int [n_rows, n_vars]).  With
    ``init`` the fully observed families get their MLE from the rows and the hidden ones keep ``spec``'s CPTs
    (init="current"); without it every CPT stays ``spec``'s."""
    from continuousbayesiannetwork_b200 import _native as N
    from continuousbayesiannetwork_b200 import em as EMM
    from continuousbayesiannetwork_b200.engine import install_cpts

    t, infer = install_cpts(spec, DEV, **cfg)
    n = codes_np.shape[0]
    codes = t.new_code_matrix(n)
    codes.fill_(N.UNSEEN)
    obs = [v for v in range(spec.n) if v not in set(hidden)]
    if obs:
        codes[obs, :n] = torch.from_numpy(np.ascontiguousarray(codes_np[:, obs].T.astype(np.uint8))).to(DEV)
    t.count(codes, n)
    t.hidden = set(hidden)
    em = EMM.EM(t, infer, codes, n, hidden, **({} if chunk_rows is None else {"chunk_rows": chunk_rows}))
    if init:
        em.initialise("current", 0, t.cond.clone())
    return t, infer, em


def _sample(spec, n, seed):
    from continuousbayesiannetwork_b200.engine import sample_network

    return sample_network(spec, seed, 0, n, device=DEV)[:, :n].T.cpu().numpy().astype(np.int64)


def _cpt(t, v):
    return t.table_view(t.cond, t.names[v]).double().cpu().numpy()


# ------------------------------------------------------------------------------------------------ cbn_ess_run, bit for bit
def _ess_case(rng, hcards, n, big_at=None):
    """Random chain factors and destinations: (plan args, factors, codes, expected int64 delta)."""
    from continuousbayesiannetwork_b200 import _native as N

    m = len(hcards)
    card_h = int(np.prod(hcards))
    obs_cards = [3, 5, 2, 7]
    ld = max(16, (n + 15) // 16 * 16)
    codes = rng.integers(0, np.array(obs_cards)[:, None] + 1, size=(4, ld)).astype(np.uint8)   # code == card: adds nothing
    codes[:, rng.random(ld) < 0.01] = 255
    factors = []
    for j in range(m):
        f = rng.random((int(np.prod(hcards[:j])), n, hcards[j])).astype(np.float32)
        f[f < 0.05] = 0.0
        factors.append(f)
    digits = np.stack(np.unravel_index(np.arange(card_h), hcards), axis=1)
    # destinations: (observed rows in table order, hidden axes position) -- hidden axes first, last, in the middle
    layouts = [([0], "last"), ([1, 2], "first"), ([3, 0], "middle"), ([], "first")]
    dests, maps, want_parts, off = [], [], [], 0
    for k, (obs, where) in enumerate(layouts):
        hperm = list(rng.permutation(m))
        axes = [("h", j) for j in hperm]
        ob = [("o", r) for r in obs]
        axes = axes + ob if where == "first" else ob + axes if where == "last" else ob[:1] + axes + ob[1:]
        card_of = lambda a: hcards[a[1]] if a[0] == "h" else obs_cards[a[1]]
        stride, s = {}, 1
        for a in reversed(axes):
            stride[a] = s
            s *= card_of(a)
        cells = s + (9000 if k == big_at else 3)            # slack cells are never reached
        cell = sum(digits[:, j] * stride[("h", j)] for j in range(m)).astype(np.int32)
        maps.append(np.ascontiguousarray(cell))
        d = N.EssDest()
        d.table_offset, d.n_cells, d.n_obs = off, cells, len(obs)
        for i, r in enumerate(obs):
            d.obs_row[i], d.obs_card[i], d.obs_stride[i] = r, obs_cards[r], stride[("o", r)]
        d.hidden_cell = maps[-1].ctypes.data
        dests.append(d)
        want_parts.append((off, obs, [stride[("o", r)] for r in obs], cell))
        off += cells
    want = np.zeros(off, np.int64)
    for h in range(card_h):
        w = np.ones(n, np.float32)
        for j in range(m):
            pre = int(np.ravel_multi_index(tuple(digits[h, :j]), hcards[:j])) if j else 0
            w = w * factors[j][pre, :, digits[h, j]]
        v = np.rint(w.astype(np.float64) * ONE)
        for base, obs, strides, cell in want_parts:
            ok = (w > 0).copy()
            idx = np.zeros(n, np.int64)
            for r, st in zip(obs, strides):
                c = codes[r, :n].astype(np.int64)
                ok &= c < obs_cards[r]
                idx += np.minimum(c, obs_cards[r] - 1) * st
            add = np.bincount(idx[ok] + cell[h], weights=v[ok], minlength=1)   # sums below 2^53: exact
            want[base: base + add.size] += add.astype(np.int64)
    return dests, maps, factors, codes, want


@pytest.mark.parametrize("hcards", [[3], [2, 4], [3, 2, 3], [3, 3, 3, 4]])
@pytest.mark.parametrize("n", [0, 1, 4095])
@pytest.mark.parametrize("big_at", [None, 0, 2])
def test_ess_run_matches_numpy_bit_for_bit(hcards, n, big_at):
    _ess_check(hcards, n, big_at, seed=len(hcards) * 7 + n)


@pytest.mark.parametrize("big_at", [None, 3])
def test_ess_run_many_grid_rounds(big_at):
    _ess_check([2, 4], (1 << 20) + 3, big_at, seed=5)


def _ess_check(hcards, n, big_at, seed):
    from continuousbayesiannetwork_b200 import _native as N

    ctx = N.context_for(DEV)
    rng = np.random.default_rng(seed)
    dests, maps, factors, codes, want = _ess_case(rng, hcards, n, big_at)
    arr = (N.EssDest * len(dests))(*dests)
    stream = N.stream_ptr(DEV)
    h = C.c_void_p()
    N.check(N.lib().cbn_ess_plan_create(ctx.handle, len(hcards), (C.c_int32 * len(hcards))(*hcards), arr, len(dests), stream,
                                        C.byref(h)), ctx.handle)
    try:
        smem = N.lib().cbn_ess_plan_smem_dests(h)
        assert smem == (len(dests) if big_at is None else big_at)      # both paths: privatised prefix, global rest
        dev_f = [torch.from_numpy(f).to(DEV) for f in factors]
        dev_c = torch.from_numpy(codes).to(DEV)
        start = torch.from_numpy(rng.integers(0, 1 << 40, size=want.size)).to(DEV)
        acc = start.clone()
        N.check(N.lib().cbn_ess_run(ctx.handle, h, N.ptr_array([f.data_ptr() for f in dev_f]), dev_c.data_ptr(), dev_c.stride(0),
                                    n, acc.data_ptr(), stream), ctx.handle)
        assert np.array_equal((acc - start).cpu().numpy(), want)
    finally:
        N.lib().cbn_ess_plan_destroy(h)


def test_ess_run_rejects_bad_arguments():
    from continuousbayesiannetwork_b200 import _native as N

    ctx = N.context_for(DEV)
    lib = N.lib()
    d = N.EssDest()
    cell = np.zeros(4, np.int32)
    cell[3] = 10
    d.table_offset, d.n_cells, d.n_obs, d.hidden_cell = 0, 10, 0, cell.ctypes.data
    h = C.c_void_p()
    assert lib.cbn_ess_plan_create(ctx.handle, 1, (C.c_int32 * 1)(4), (N.EssDest * 1)(d), 1, None, C.byref(h)) == N.ERR_INVALID
    cell[3] = 9
    N.check(lib.cbn_ess_plan_create(ctx.handle, 1, (C.c_int32 * 1)(4), (N.EssDest * 1)(d), 1, None, C.byref(h)), ctx.handle)
    f = torch.zeros(16, device=DEV)
    codes = torch.zeros((1, 16), dtype=torch.uint8, device=DEV)
    acc = torch.zeros(10, dtype=torch.int64, device=DEV)
    ptrs = N.ptr_array([f.data_ptr()])
    assert lib.cbn_ess_run(ctx.handle, h, ptrs, codes.data_ptr(), 16, 1 << 31, acc.data_ptr(), None) == N.ERR_INVALID
    assert lib.cbn_ess_run(ctx.handle, h, ptrs, codes.data_ptr(), 8, 4, acc.data_ptr(), None) == N.ERR_INVALID
    lib.cbn_ess_plan_destroy(h)


# ------------------------------------------------------------------------------------------------ chain-rule posteriors
def _chain_joint(em, hidden, n):
    """Joint posterior of ``hidden`` (in the order given) by the chain rule of the device factors, fp64 [n, card_H]."""
    from continuousbayesiannetwork_b200.em import ChainGroup

    cards = em.t.cards
    order = sorted(hidden, key=lambda u: (cards[u], u))
    fs = [f.double().cpu().numpy() for f in em.chain_factors(ChainGroup(order, []), 0, n)]
    cfg = list(itertools.product(*[range(cards[u]) for u in order]))
    joint = np.zeros((n,) + tuple(cards[u] for u in order))
    for c in cfg:
        p = np.ones(n)
        for j in range(len(order)):
            pre = int(np.ravel_multi_index(c[:j], [cards[u] for u in order[:j]])) if j else 0
            p = p * fs[j][pre, :, c[j]]
        joint[(slice(None),) + c] = p
    # back to the order given
    return joint.transpose([0] + [1 + order.index(u) for u in hidden]).reshape(n, -1)


def _all_rows(cards, obs):
    rows = np.zeros((int(np.prod([cards[v] for v in obs])), len(cards)), np.int64)
    rows[:, obs] = np.indices([cards[v] for v in obs]).reshape(len(obs), -1).T
    return rows


@pytest.mark.parametrize("size", [2, 3])
def test_chain_posteriors_asia_every_subset(size):
    from continuousbayesiannetwork_b200 import synth

    spec = _spec(*(lambda s: (s.names, s.cards, s.parents, s.cpts))(synth.asia()))
    for hidden in itertools.combinations(range(spec.n), size):
        obs = [v for v in range(spec.n) if v not in hidden]
        rows = _all_rows(spec.cards, obs)
        _, _, em = _em(spec, rows, list(hidden), init=False)
        got = _chain_joint(em, list(hidden), rows.shape[0])
        _, want = EO.posterior(spec.cards, spec.parents, spec.cpts, list(hidden), rows)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-5, err_msg=str(hidden))


@pytest.mark.parametrize("per_row", [False, True])
def test_chain_posteriors_random_small_nets(per_row):
    from continuousbayesiannetwork_b200.ve import RowPlan

    rng = np.random.default_rng(11 + per_row)
    row_plans = 0
    for _ in range(6):
        cards, parents, cpts = MO.random_small_net(rng)
        spec = _spec(_names(len(cards)), cards, parents, cpts)
        hidden = sorted(int(v) for v in rng.choice(spec.n, size=int(rng.integers(2, 4)), replace=False))
        rows = rng.integers(0, np.array(cards)[None, :], size=(300, spec.n))
        cfg = {"table_budget_cells": 1, "merge_budget_cells": 1} if per_row else {}
        _, infer, em = _em(spec, rows, hidden, init=False, **cfg)
        got = _chain_joint(em, hidden, rows.shape[0])
        _, want = EO.posterior(spec.cards, spec.parents, spec.cpts, hidden, rows)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-5)
        row_plans += sum(isinstance(p, RowPlan) for p in infer.compiler._plans.values())
    assert (row_plans > 0) == per_row


# ------------------------------------------------------------------------------------------------ one E-step, full EM
def _cases():
    from continuousbayesiannetwork_b200 import synth

    a = synth.asia()
    asia = _spec(a.names, a.cards, a.parents, a.cpts)
    lc = _spec(*EO.latent_class(n_children=8, seed=3))
    hm = _spec(*EO.hmm(steps=6, seed=4))
    return [("asia", asia, [asia.names.index(n) for n in ("tub", "lung", "either")]),
            ("latent_class", lc, [0]),
            ("hmm", hm, list(range(6)))]


def _start(spec, hidden, seed):
    """``spec`` with every CPT that has a hidden member replaced by Dirichlet(1) rows."""
    rng = np.random.default_rng(seed)
    cpts = []
    for v in range(spec.n):
        if any(u in hidden for u in spec.parents[v] + [v]):
            rows = rng.dirichlet(np.ones(spec.cards[v]), size=int(np.prod([spec.cards[u] for u in spec.parents[v]])))
            cpts.append(rows.reshape(np.shape(spec.cpts[v])))
        else:
            cpts.append(spec.cpts[v])
    return _spec(spec.names, spec.cards, spec.parents, cpts)


@pytest.mark.parametrize("case", range(3))
def test_one_e_step_matches_enumeration(case):
    name, spec, hidden = _cases()[case]
    rows = _sample(spec, 4096, seed=case)
    start = _start(spec, hidden, seed=case)
    t, _, em = _em(start, rows, hidden)
    cpts = [_cpt(t, v) for v in range(spec.n)]        # fully observed families start from their data MLE
    em.e_step()
    got = em.expected_counts().cpu().numpy()
    want, _, _ = EO.e_step(start.cards, start.parents, cpts, hidden, rows)
    n = rows.shape[0]
    for v in range(spec.n):
        g = got[t.offsets[v]: t.offsets[v] + t.n_cells[v]]
        w = want[v].reshape(-1)
        assert np.all(np.abs(g - w) <= 1e-6 * np.abs(w) + n * 2.0 ** -32), (name, spec.names[v], np.abs(g - w).max())


@pytest.mark.parametrize("case", range(3))
def test_ten_iterations_match_numpy_em(case):
    name, spec, hidden = _cases()[case]
    rows = _sample(spec, 4096, seed=10 + case)
    start = _start(spec, hidden, seed=20 + case)
    t, _, em = _em(start, rows, hidden)
    cpts = [_cpt(t, v) for v in range(spec.n)]
    res = em.fit(max_iter=10, tol=0.0)
    assert res.n_iter == 10 and len(res.log_likelihood) == 11
    want, hist = EO.em(start.cards, start.parents, cpts, hidden, rows, 10)
    for v in range(spec.n):
        np.testing.assert_allclose(_cpt(t, v), want[v], rtol=0, atol=1e-4, err_msg=f"{name} {spec.names[v]}")
    np.testing.assert_allclose(res.log_likelihood[:10], hist, rtol=1e-5)
    L = res.log_likelihood
    assert all(b >= a - 1e-6 * abs(a) for a, b in zip(L, L[1:])), (name, L)


# ------------------------------------------------------------------------------------------------ network API
def _dag(spec):
    g = nx.DiGraph()
    g.add_nodes_from(spec.names)
    for v, ps in enumerate(spec.parents):
        g.add_edges_from((spec.names[p], spec.names[v]) for p in ps)
    return g


def _frame(spec, rows, drop=()):
    return pd.DataFrame({n: rows[:, i].astype(np.float32) for i, n in enumerate(spec.names) if n not in drop})


def test_complete_data_is_bit_identical_to_the_ordinary_fit():
    from continuousbayesiannetwork_b200 import BayesianNetwork, synth

    spec = synth.alarm()
    df = _frame(spec, _sample(spec, 1 << 16, seed=3))
    bn = BayesianNetwork(_dag(spec), df, PL, INF, device=DEV)
    ref_cond, ref_joint, ref_counts = bn.tables.cond.clone(), bn.tables.joint.clone(), bn.tables.counts.clone()
    res = bn.fit_em(df)
    assert res.converged and res.n_iter == 1 and res.n_dead_rows == 0
    assert torch.equal(bn.tables.cond, ref_cond) and torch.equal(bn.tables.joint, ref_joint)
    assert torch.equal(bn.tables.counts, ref_counts)
    assert torch.equal(bn.tables.expected_counts, ref_counts.double())
    assert res.log_likelihood[0] == res.log_likelihood[1]
    np.testing.assert_allclose(res.log_likelihood[-1], bn.log_likelihood(df).double().sum().item(), rtol=1e-9)


def test_latent_class_recovery():
    """2^22 rows of a separated latent-class model without Z: the fitted CPTs are the truth up to a relabelling."""
    from continuousbayesiannetwork_b200 import BayesianNetwork
    from continuousbayesiannetwork_b200.engine import install_cpts

    truth = _spec(*EO.latent_class(n_children=20, k=4, card=3, seed=9, sharp=1.5))
    n = 1 << 22
    rows = _sample(truth, n, seed=1)
    df = _frame(truth, rows, drop=("Z",))
    pl = dict(PL, em_max_iter=300, em_tol=1e-9, em_seed=2)
    bn = BayesianNetwork(_dag(truth), df, pl, INF, device=DEV, latent={"Z": 4})
    res = bn.em_result
    t = bn.tables
    fitted = [_cpt(t, t.index[nm]) for nm in truth.names]
    best = min(itertools.permutations(range(4)),
               key=lambda p: sum(np.abs(fitted[v][list(p)] - truth.cpts[v]).sum() for v in range(1, truth.n)))
    assert np.abs(fitted[0][list(best)] - truth.cpts[0]).max() < 0.01
    for v in range(1, truth.n):
        assert np.abs(fitted[v][list(best)] - truth.cpts[v]).max() < 0.01, truth.names[v]
    _, infer = install_cpts(truth, DEV)
    cols = {nm: torch.from_numpy(rows[:, i].astype(np.float32)).to(DEV) for i, nm in enumerate(truth.names) if nm != "Z"}
    l_truth = infer.log_evidence(cols).double().sum().item()
    assert res.log_likelihood[-1] >= l_truth - 1e-4 * abs(l_truth)
    assert res.n_dead_rows == 0
    L = res.log_likelihood
    assert all(b >= a - 1e-6 * abs(a) for a, b in zip(L, L[1:]))


def test_determinism_and_chunking():
    spec = _spec(*EO.latent_class(n_children=8, seed=5))
    n = (1 << 20) + 37
    rows = _sample(spec, n, seed=6)
    start = _start(spec, [0], seed=7)
    out = []
    for chunk in (1 << 22, 1 << 22, n // 3):
        t, _, em = _em(start, rows, [0], chunk_rows=chunk)
        em.fit(max_iter=3, tol=0.0)
        out.append((em.acc.clone(), t.cond.clone(), em.chunk))
    assert out[2][2] < n < out[0][2]
    for acc, cond, _ in out[1:]:
        assert torch.equal(acc, out[0][0]) and torch.equal(cond, out[0][1])


def _asia_bn(n=1 << 14, **kw):
    from continuousbayesiannetwork_b200 import BayesianNetwork, synth

    spec = synth.asia()
    rows = _sample(spec, n, seed=4)
    df = _frame(spec, rows, drop=("tub", "either"))
    pl = dict(PL, em_max_iter=20, em_seed=3)
    return spec, rows, df, BayesianNetwork(_dag(spec), df, pl, INF, device=DEV, latent={"tub": 2, "either": [0.0, 1.0]}, **kw)


def test_latent_construction_save_load_and_update(tmp_path):
    spec, rows, df, bn = _asia_bn()
    t = bn.tables
    assert bn.em_result.n_iter >= 1 and len(bn.em_result.log_likelihood) == bn.em_result.n_iter + 1
    assert t.hidden == {t.index["tub"], t.index["either"]}
    assert torch.equal(t.domains[t.index["tub"]].cpu(), torch.tensor([0.0, 1.0]))
    # every family's expected counts sum to the number of rows
    for nm in spec.names:
        assert abs(t.table_view(t.expected_counts, nm).sum().item() - len(df)) < 1e-6 * len(df)
    # integer counts: fully observed families only
    assert t.table_view(t.counts, "smoke").sum().item() == len(df)
    assert t.table_view(t.counts, "xray").sum().item() == 0
    with pytest.raises(ValueError, match="expected_counts"):
        t.mle_tensor("xray")
    assert t.mle_tensor("smoke").shape[0] == 2
    with pytest.raises(ValueError, match="expected_counts"):
        bn.nodes_obj["either"].estimator.mle_tensor
    cond = t.cond.clone()
    path = str(tmp_path / "em.pt")
    bn.save_model(path)
    _, _, _, bn2 = _asia_bn(n=1 << 12)
    bn2.load_model(path)
    assert torch.equal(bn2.tables.cond, cond) and torch.equal(bn2.tables.expected_counts, t.expected_counts)
    post, _ = bn2.infer("either", {"xray": torch.ones(3, 1)})
    ref, _ = bn.infer("either", {"xray": torch.ones(3, 1)})
    assert torch.equal(post, ref)
    # update_knowledge re-runs EM with the stored settings: the same data gives the same bits
    bn2.update_knowledge(df)
    assert torch.equal(bn2.tables.cond, cond)
    with pytest.raises(ValueError, match="accumulate"):
        bn2.update_knowledge(df, accumulate=True)
    # fit_em on a network without latent=: the nodes without a column keep their fitted domains
    from continuousbayesiannetwork_b200 import BayesianNetwork

    full = BayesianNetwork(_dag(spec), _frame(spec, rows), PL, INF, device=DEV)
    res = full.fit_em(df, max_iter=20, seed=3)
    assert res.n_iter == bn.em_result.n_iter and torch.equal(full.tables.cond, cond)
    res = full.fit_em(df, max_iter=5, init="current")
    assert res.log_likelihood[0] >= bn.em_result.log_likelihood[-1] - 1e-6 * abs(bn.em_result.log_likelihood[-1])


def test_errors(monkeypatch):
    from continuousbayesiannetwork_b200 import BayesianNetwork, em

    spec, rows, df, bn = _asia_bn(n=1 << 10)
    dag = _dag(spec)
    with pytest.raises(ValueError, match="latent nodes"):
        bn.fit_em(_frame(spec, rows, drop=("either",)))                      # a column for latent "tub"
    with pytest.raises(ValueError, match="not a node"):
        BayesianNetwork(dag, df, PL, INF, device=DEV, latent={"tub": 2, "nope": 2, "either": 2})
    for bad in (0, 256, [], list(range(256))):
        with pytest.raises(ValueError):
            BayesianNetwork(dag, df, PL, INF, device=DEV, latent={"tub": bad, "either": 2})
    nan = df.copy()
    nan.iloc[5, 0] = np.nan
    with pytest.raises(ValueError, match="missing values"):
        bn.fit_em(nan)
    with pytest.raises(ValueError, match="rows"):
        bn.fit_em(df.iloc[:0])
    monkeypatch.setattr(em, "MAX_ROWS", 100)
    with pytest.raises(ValueError, match="rows"):
        bn.fit_em(df.iloc[:100])
    monkeypatch.undo()
    with pytest.raises(ValueError, match="init"):
        bn.fit_em(df, init="kmeans")
    bn.inference_obj = types.SimpleNamespace(bind=lambda tables: None)
    bn.inference_obj_name = "approximate"
    with pytest.raises(NotImplementedError):
        bn.fit_em(df)
