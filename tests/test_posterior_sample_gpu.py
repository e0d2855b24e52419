"""GPU checks of posterior sampling (cbn_factor_contract_cdf, VECompiler.compile_posterior_sampler, cbn_psample_run):
the threshold contraction against numpy, the traceback bit for bit against a numpy interpreter of the plan's own tables,
the draws' distribution against fp64 enumeration, support and log P(e) at full size, determinism, CUDA-graph replay and
the network API."""
import ctypes as C
import itertools
import os
import sys

import networkx as nx
import numpy as np
import pandas as pd
import pytest
import torch

from oracle import cbn_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import loglik_oracle as LO  # noqa: E402
import mpe_oracle as MO  # noqa: E402
import psample_oracle as PO  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5


def _f32(spec):
    """The spec with its CPTs rounded to fp32, as the device holds them."""
    from continuousbayesiannetwork_b200 import synth

    return synth.NetSpec(spec.names, spec.cards, spec.parents, [c.astype(np.float32).astype(np.float64) for c in spec.cpts])


def _net(spec):
    return O.DiscreteNet(spec.cards, spec.parents, spec.cpts)


def _codes_matrix(ev: np.ndarray) -> torch.Tensor:
    n, k = ev.shape
    ld = max((n + 15) // 16 * 16, 16)
    m = torch.zeros((max(k, 1), ld), dtype=torch.uint8, device=DEV)
    if k and n:
        m[:, :n] = torch.from_numpy(np.ascontiguousarray(ev.T.astype(np.uint8))).to(DEV)
    return m


def _install(spec, **cfg):
    from continuousbayesiannetwork_b200.engine import install_cpts

    return install_cpts(spec, DEV, **cfg)


def _configs(cards):
    return np.ascontiguousarray(np.indices(cards).reshape(len(cards), -1).T) if cards else np.zeros((1, 0), np.int64)


def _host_decode(plan, cards):
    return [(v, tuple(sc), tb.cpu().numpy()[: int(np.prod([cards[u] for u in sc])) * (cards[v] - 1)])
            for (v, sc), tb in zip(plan.split.decode, plan.tables)]


def _check_bits(infer, names, ev, n_draws, seed, first_row=0, what=""):
    """Device draws == the numpy interpreter run on the plan's own threshold tables, for every row and draw; returns
    (plan, hidden codes uint8 [n_draws, n_hidden, n_rows], log P(e) fp32 [n_rows])."""
    plan = infer.posterior_sampler(names)
    n = ev.shape[0]
    hidden, value = plan.run_codes(_codes_matrix(ev), n, n_draws=n_draws, seed=seed, first_row=first_row)
    nh = len(plan.hidden)
    got = hidden[: n_draws * nh, :n].cpu().numpy().reshape(n_draws, nh, n)
    value = value.cpu().numpy()
    dead = ~(value > -np.inf)
    want = PO.interpret(_host_decode(plan, infer.tables.cards), infer.tables.cards, plan.evidence, ev.astype(np.int64),
                        dead, seed, first_row, n_draws)
    for h, v in enumerate(plan.hidden):
        assert np.array_equal(got[:, h], want[v]), (what, v)
    return plan, got, value


# ------------------------------------------------------------------------------------------------ the cdf contraction
def _contract(inputs, in_axes, out_cards, sum_card, fn):
    from continuousbayesiannetwork_b200 import _native as N

    ctx = N.context_for(DEV)
    d = N.Contract()
    d.n_out_dims = len(out_cards)
    for a, c in enumerate(out_cards):
        d.out_card[a] = c
    d.sum_card = sum_card
    d.n_in = len(inputs)
    allc = list(out_cards) + [sum_card]
    for k, (t, axes) in enumerate(zip(inputs, in_axes)):
        st, s = {}, 1
        for a in reversed(axes):
            st[a] = s
            s *= allc[a]
        d.inp[k] = t.data_ptr()
        for a in range(len(out_cards)):
            d.in_stride[k][a] = st.get(a, 0)
        d.sum_stride[k] = st.get(len(out_cards), 0)
    n_out = int(np.prod(out_cards))
    out = torch.empty(n_out, dtype=torch.float32, device=DEV)
    d.out = out.data_ptr()
    d.log_space = 1
    cdf = None
    if fn == "cdf":
        cdf = torch.full((max(n_out * (sum_card - 1), 1),), 7.0, dtype=torch.float32, device=DEV)
        N.check(N.lib().cbn_factor_contract_cdf(ctx.handle, C.byref(d), cdf.data_ptr(), N.stream_ptr(DEV)), ctx.handle)
    else:
        N.check(N.lib().cbn_factor_contract(ctx.handle, C.byref(d), N.stream_ptr(DEV)), ctx.handle)
    torch.cuda.synchronize()
    return out.cpu().numpy(), (None if cdf is None else cdf.cpu().numpy()), d, ctx


def _check_cdf(out, cdf, acc, sum_card, what):
    """``cdf`` against the fp64 cumulative of exp(term - out) (out: the kernel's own normaliser), within 1e-6 plus the
    rounding bound of an fp32 running sum; exactly 1.0 from the last finite term on, and everywhere in an all -inf cell."""
    nt = sum_card - 1
    if nt == 0:
        assert cdf.size == 1 and cdf[0] == 7.0, what           # sum_card 1 writes nothing
        return
    terms = acc.reshape(-1, sum_card).astype(np.float64)
    c = cdf[: terms.shape[0] * nt].reshape(-1, nt)
    fin = np.isfinite(terms)
    last = np.where(fin.any(axis=1), sum_card - 1 - np.argmax(fin[:, ::-1], axis=1), -1)
    with np.errstate(invalid="ignore"):
        p = np.where(fin, np.exp(terms - out.astype(np.float64)[:, None]), 0.0)
    cum = np.cumsum(p, axis=1)[:, :nt]
    x = np.arange(nt)[None, :]
    ones = x >= last[:, None]
    assert (c[ones] == 1.0).all(), what
    bound = 1e-6 + (x + 1) * 2.0 ** -24
    assert (np.abs(c - cum) <= bound)[~ones].all(), what
    # a value of probability zero has an empty interval
    zero = ~fin[:, :nt][:, 1:]
    assert (c[:, 1:][zero] == c[:, :-1][zero]).all(), what
    assert (c[:, 0][~fin[:, 0]] == np.where(ones[:, 0], 1.0, 0.0)[~fin[:, 0]]).all(), what


def test_contract_cdf_against_numpy_on_both_kernels():
    from continuousbayesiannetwork_b200 import _native as N

    rng = np.random.default_rng(5)
    # the small shapes take the plain kernel, [64, 32, 40] and [16, 16, 16, 17] the tiled one (n_out >= 2^16, <= 4 inputs)
    cases = [([3, 4], 5), ([2, 3, 2], 7), ([64, 32, 40], 3), ([16, 16, 16, 17], 4), ([5], 255), ([7], 1), ([256, 256], 2),
             ([256, 257], 17), ([300, 256], 1)]
    cases += [([6], s) for s in (1, 2, 3, 4, 5, 8, 16, 31, 64, 127, 200, 254, 255)]
    for out_cards, sum_card in cases:
        for n_in in ((1, 2, 5) if int(np.prod(out_cards)) < 1 << 16 else (1, 3)):
            allc = list(out_cards) + [sum_card]
            nd = len(allc)
            in_axes, ts, hs = [], [], []
            for k in range(n_in):
                axes = sorted(set(int(a) for a in rng.choice(nd, size=int(rng.integers(1, nd + 1)), replace=False)) |
                              ({nd - 1} if k == 0 else set()))
                h = (rng.integers(-6, 1, size=[allc[a] for a in axes]) * 0.5).astype(np.float32)   # exact halves: ties
                h[rng.random(h.shape) < (0.3 if k == 0 else 0.05)] = -np.inf     # leading, inner, trailing zeros
                if k == 0 and sum_card > 2:
                    h.reshape(-1, sum_card)[::7] = -np.inf                       # all -inf cells
                in_axes.append(axes)
                hs.append(h)
                ts.append(torch.from_numpy(h.reshape(-1)).to(DEV))
            out, cdf, d, ctx = _contract(ts, in_axes, out_cards, sum_card, "cdf")
            ref, _, _, _ = _contract(ts, in_axes, out_cards, sum_card, "sum")
            what = (out_cards, sum_card, n_in)
            assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)), what
            acc = np.zeros(allc, dtype=np.float32)
            for h, axes in zip(hs, in_axes):                            # fp32, in input order, as the kernel adds
                acc = (acc + h.reshape([allc[a] if a in axes else 1 for a in range(nd)])).astype(np.float32)
            _check_cdf(out, cdf, acc, sum_card, what)
    # an all -inf reduction: -inf and every threshold 1
    t = torch.full((4 * 3,), float("-inf"), device=DEV)
    out, cdf, d, ctx = _contract([t], [[0, 1]], [4], 3, "cdf")
    assert np.isneginf(out).all() and (cdf == 1.0).all()
    # argument checks
    for field, val in (("log_space", 0), ("normalize_last", 1)):
        setattr(d, field, val)
        with pytest.raises(ValueError):
            N.check(N.lib().cbn_factor_contract_cdf(ctx.handle, C.byref(d), t.data_ptr(), N.stream_ptr(DEV)), ctx.handle)
        setattr(d, field, 1 - val)
    with pytest.raises(ValueError):
        N.check(N.lib().cbn_factor_contract_cdf(ctx.handle, C.byref(d), None, N.stream_ptr(DEV)), ctx.handle)


# ------------------------------------------------------------------------------------------------ bit-exact traceback
def test_traceback_bits_asia_every_subset_and_configuration():
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.asia())
    tables, infer = _install(spec)
    net = _net(spec)
    for k in range(spec.n + 1):
        for sub in itertools.combinations(range(spec.n), k):
            names = [spec.names[v] for v in sub]
            ev = np.repeat(_configs([spec.cards[v] for v in sub]), 8, axis=0)
            _, got, value = _check_bits(infer, names, ev, n_draws=4, seed=k + 1, first_row=3, what=sub)
            want = LO.enumerate_log_evidence(net, list(sub), ev) if sub else np.zeros(ev.shape[0])
            assert np.array_equal(np.isneginf(want), np.isneginf(value)) and not np.isnan(value).any(), sub
            fin = np.isfinite(want)
            assert (np.abs(value[fin] - want[fin]) <= TOL * np.maximum(1, np.abs(want[fin]))).all(), sub
            assert (got[:, :, ~fin] == PO.UNSEEN).all() and (got[:, :, fin] < PO.UNSEEN).all(), sub


def test_traceback_bits_alarm_headline_and_a_ktree_pattern():
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    E = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    codes = synth.sample_forward_numpy(spec, 61, 0, 1 << 16)
    ev = codes[E].T.astype(np.int64)
    ev[5, 0] = 255                                                  # an unseen value: a dead row
    plan, got, value = _check_bits(infer, synth.ALARM_EVIDENCE, ev, n_draws=4, seed=2024, what="alarm")
    want = LO.ve_log_evidence(_net(spec), E, ev)
    assert np.array_equal(np.isneginf(want), np.isneginf(value)) and np.isneginf(value[5])
    fin = np.isfinite(want)
    assert (np.abs(value[fin] - want[fin]) <= TOL * np.maximum(1, np.abs(want[fin]))).all()
    # the 200-node k-tree, bench.py's query pattern with the smallest threshold tables
    kspec = _f32(synth.random_ktree_dag())
    rng = np.random.default_rng(1240)
    pats = [[int(v) for v in rng.choice(kspec.n, size=11, replace=False)] for _ in range(8)]
    vs = pats[4]
    _, kinf = _install(kspec)
    kev = synth.sample_forward_numpy(kspec, 62, 0, 1 << 13)[vs[1:]].T.astype(np.int64)
    _check_bits(kinf, [kspec.names[v] for v in vs[1:]], kev, n_draws=2, seed=9, first_row=1 << 33, what="ktree")


# ------------------------------------------------------------------------------------------------ distribution
def _histogram_check(infer, spec, sub, n_draws_total=1 << 16, seed=1):
    """For every configuration of ``sub``: 2^16 draws of the hidden variables against the fp64 enumeration posterior,
    every cell within 5 sigma + 2^-20, and zero-probability completions never drawn."""
    net = _net(spec)
    names = [spec.names[v] for v in sub]
    plan = infer.posterior_sampler(names)
    hid = plan.hidden
    strides = torch.tensor([int(np.prod([spec.cards[u] for u in hid[h + 1:]])) for h in range(len(hid))],
                           dtype=torch.int64, device=DEV)
    cells = int(np.prod([spec.cards[u] for u in hid]))
    for cfg in _configs([spec.cards[v] for v in sub]):
        z, post = PO.enumerate_posterior(net, sub, cfg)
        ev = np.repeat(cfg[None, :], n_draws_total, axis=0)
        hidden, value = plan.run_codes(_codes_matrix(ev), n_draws_total, n_draws=1, seed=seed)
        codes = hidden[: len(hid), :n_draws_total].long()
        if z == 0:
            assert torch.isneginf(value).all() and (codes == PO.UNSEEN).all(), (sub, cfg)
            continue
        assert torch.isfinite(value).all() and (codes < PO.UNSEEN).all()
        idx = (codes * strides[:, None]).sum(0)
        freq = torch.bincount(idx, minlength=cells).cpu().numpy() / n_draws_total
        p = post.reshape(-1)                                     # hidden variables in network order, as plan.hidden
        # below a few expected counts the normal approximation of a cell fails: its sigma is taken at 4 / n
        sigma = np.sqrt(np.maximum(p, 4.0 / n_draws_total) * (1 - p) / n_draws_total)
        assert (np.abs(freq - p) <= 5 * sigma + 2.0 ** -20).all(), (sub, cfg)
        assert (freq[p == 0] == 0).all(), (sub, cfg)


def test_distribution_asia_and_random_dags_with_zeros():
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.asia())
    _, infer = _install(spec)
    for sub in [(), (7,), (6, 7), (0, 1, 6), (2, 5), (0, 1, 2, 3, 4)]:
        _histogram_check(infer, spec, sub)
    rng = np.random.default_rng(17)
    for i in range(4):
        cards, parents, cpts = MO.random_small_net(rng, 5, 9)
        s = _f32(synth.NetSpec([f"v{j}" for j in range(len(cards))], cards, parents, cpts))
        _, inf = _install(s)
        for _ in range(2):
            sub = tuple(sorted(int(v) for v in rng.choice(len(cards), size=int(rng.integers(1, 3)), replace=False)))
            _histogram_check(inf, s, sub, seed=i)


def test_distribution_alarm_without_evidence():
    """2^22 draws from the prior of Alarm: every node's marginal within 5 sigma of the exact marginal of the posterior
    plans."""
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    n = 1 << 22
    plan = infer.posterior_sampler([])
    hidden, value = plan.run_codes(torch.zeros((1, n), dtype=torch.uint8, device=DEV), n, n_draws=1, seed=77)
    assert (value.abs() <= 1e-5).all()                             # log P({}) = log 1
    exact = infer.infer_many(spec.names, {})
    for h, v in enumerate(plan.hidden):
        p = exact[spec.names[v]][0].double().cpu().numpy()
        freq = torch.bincount(hidden[h, :n].long(), minlength=spec.cards[v]).cpu().numpy() / n
        assert (np.abs(freq - p) <= 5 * np.sqrt(p * (1 - p) / n) + 2.0 ** -20).all(), spec.names[v]


# ------------------------------------------------------------------------------------------------ support and value
def _complete(plan, ev_codes, hidden, d, n, n_vars):
    full = torch.zeros((n_vars, ev_codes.shape[1]), dtype=torch.uint8, device=DEV)
    for i, v in enumerate(plan.evidence):
        full[v] = ev_codes[i]
    nh = len(plan.hidden)
    for h, v in enumerate(plan.hidden):
        full[v, :n] = hidden[d * nh + h, :n]
    return full


def test_support_and_value_alarm_headline_and_ktree_patterns():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    cases = []
    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    cases.append((spec, tables, infer, synth.ALARM_EVIDENCE, 1 << 20))
    kspec = _f32(synth.random_ktree_dag())
    ktables, kinf = _install(kspec, sample_table_budget_bytes=1 << 33)
    rng = np.random.default_rng(1240)
    for _ in range(8):
        vs = [int(v) for v in rng.choice(kspec.n, size=11, replace=False)]
        cases.append((kspec, ktables, kinf, [kspec.names[v] for v in vs[1:]], 1 << 16))
    for spec, tables, infer, names, n in cases:
        E = [spec.names.index(e) for e in names]
        codes = sample_network(spec, 63, 0, n, DEV, tables=tables)
        ev = codes[E].contiguous()
        ev[0, 11] = 255                                               # an unseen value
        plan = infer.posterior_sampler(names)
        hidden, value = plan.run_codes(ev, n, n_draws=2, seed=5)
        assert not torch.isnan(value).any()
        dead = ~torch.isfinite(value)
        ref = infer.evidence_plan(names).run_codes(ev, n)             # log P(e) of the evidence mode: ancestors only
        assert torch.equal(dead, ~torch.isfinite(ref))
        assert ((value - ref)[~dead].abs() <= TOL * ref[~dead].abs().clamp(min=1)).all()
        assert dead[11] and (hidden[: 2 * len(plan.hidden), :n][:, dead] == PO.UNSEEN).all()
        scorer = infer.evidence_plan(spec.names)
        for d in range(2):
            ll = scorer.run_codes(_complete(plan, ev, hidden, d, n, spec.n), n)
            assert torch.equal(torch.isfinite(ll), ~dead), names
        if spec.n <= 40:                                              # the fp64 oracle of log P(e) on a sample of rows
            rows = np.arange(0, n, 997)
            want = LO.ve_log_evidence(_net(spec), E, ev[:, rows].cpu().numpy().T.astype(np.int64))
            got = value[rows].cpu().numpy()
            assert np.array_equal(np.isneginf(want), np.isneginf(got))
            fin = np.isfinite(want)
            assert (np.abs(got[fin] - want[fin]) <= TOL * np.maximum(1, np.abs(want[fin]))).all()


# ------------------------------------------------------------------------------------------------ determinism
def test_determinism_calls_batch_splits_and_draw_prefixes():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    E = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    n = (1 << 20) + 37
    ev = sample_network(spec, 64, 0, n, DEV, tables=tables)[E].contiguous()
    plan = infer.posterior_sampler(synth.ALARM_EVIDENCE)
    nh = len(plan.hidden)
    h1, v1 = plan.run_codes(ev, n, n_draws=4, seed=11)
    h2, v2 = plan.run_codes(ev, n, n_draws=4, seed=11)
    assert torch.equal(h1[:, :n], h2[:, :n]) and torch.equal(v1, v2)
    h3, _ = plan.run_codes(ev, n, n_draws=2, seed=11)
    assert torch.equal(h3[: 2 * nh, :n], h1[: 2 * nh, :n])
    h4, _ = plan.run_codes(ev, n, n_draws=4, seed=12)
    assert not torch.equal(h4[:, :n], h1[:, :n])
    s = 1 << 19
    ha, va = plan.run_codes(ev[:, :s].contiguous(), s, n_draws=4, seed=11, first_row=0)
    hb, vb = plan.run_codes(ev[:, s:].contiguous(), n - s, n_draws=4, seed=11, first_row=s)
    assert torch.equal(torch.cat([va, vb]), v1)
    assert torch.equal(torch.cat([ha[:, :s], hb[:, :n - s]], 1), h1[:, :n])
    # n_draws = 0 draws nothing; rows are still valued
    h0, v0 = plan.run_codes(ev, n, n_draws=0, seed=11)
    assert torch.equal(v0, v1)


def test_cuda_graph_replay_of_gather_accumulate_sample():
    """The gather kernel triggers programmatic dependent launch at entry; the observed-families kernel adds into its output
    and the sampler reads that output: replayed from a CUDA graph with static evidence, every store must be seen."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    n = 1 << 20
    codes = sample_network(spec, 65, 0, n, DEV, tables=tables)
    names = synth.ALARM_EVIDENCE + ["HYPOVOLEMIA", "LVFAILURE"]
    ev = codes[[spec.names.index(e) for e in names]].contiguous()
    plan = infer.posterior_sampler(names)
    assert plan.value.ve_plan is not None and plan.value.loglik is not None
    h_eager, v_eager = plan.run_codes(ev, n, n_draws=2, seed=3)
    h_eager, v_eager = h_eager.clone(), v_eager.clone()
    plan.set_static_evidence(True)
    hid = torch.full_like(h_eager, 7)
    val = torch.full((n,), float("nan"), device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        plan.run_codes(ev, n, n_draws=2, seed=3, hidden_out=hid, value_out=val)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        plan.run_codes(ev, n, n_draws=2, seed=3, hidden_out=hid, value_out=val)
    for _ in range(3):
        val.fill_(float("nan"))
        hid.fill_(7)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(val, v_eager) and torch.equal(hid[:, :n], h_eager[:, :n])
    plan.set_static_evidence(False)


# ------------------------------------------------------------------------------------------------ network API
def _frozen_lake(golden_dir):
    from continuousbayesiannetwork_b200 import BayesianNetwork

    g = np.load(os.path.join(golden_dir, "frozen_lake.npz"), allow_pickle=False)
    df = pd.DataFrame(g["data"], columns=["obs_0", "action", "reward"])
    dag = nx.DiGraph()
    dag.add_edges_from([("obs_0", "reward"), ("action", "reward")])
    return df, BayesianNetwork(dag, df, {"estimator_name": "brute_force"}, {"inference_obj": "exact"}, device=DEV)


def test_network_sample_posterior(golden_dir):
    df, bn = _frozen_lake(golden_dir)
    t = bn.tables
    sub = df[["reward"]].iloc[:500]
    draws, le = bn.sample_posterior(sub, n_draws=3, seed=4)
    assert sorted(draws) == ["action", "obs_0"] and le.shape == (500,) and le.dtype == torch.float32
    ref = bn.log_likelihood(sub)
    assert ((le - ref).abs() <= TOL * ref.abs().clamp(min=1)).all()
    r = torch.tensor(sub["reward"].to_numpy(np.float32), device=DEV)
    for name, col in draws.items():
        assert col.shape == (3, 500) and col.dtype == torch.float32 and col.is_cuda
        assert torch.isin(col, t.domains[t.index[name]]).all()
    for d in range(3):
        ll = bn.log_likelihood({"reward": r, "obs_0": draws["obs_0"][d], "action": draws["action"][d]})
        assert torch.isfinite(ll).all()
    # a dict gives the same draws as the DataFrame
    d2, le2 = bn.sample_posterior({"reward": sub["reward"].to_numpy()}, n_draws=3, seed=4)
    assert all(torch.equal(d2[k], draws[k]) for k in draws) and torch.equal(le2, le)
    # complete rows: nothing to draw, log P(e) is the log-likelihood; no columns: one row, draws from the prior
    d3, le3 = bn.sample_posterior(df.iloc[:100])
    assert d3 == {} and torch.equal(le3, bn.log_likelihood(df.iloc[:100]))
    d4, le4 = bn.sample_posterior(df[[]], n_draws=5)
    assert le4.shape == (1,) and sorted(d4) == ["action", "obs_0", "reward"] and d4["reward"].shape == (5, 1)
    # unseen value and NaN: -inf and NaN draws, never a NaN log P(e); unknown column raises
    bad = df[["reward"]].iloc[:4].copy()
    bad.iloc[1, 0] = 12345.0
    bad.iloc[2, 0] = float("nan")
    draws, le = bn.sample_posterior(bad, n_draws=2)
    le = le.cpu().numpy()
    assert np.isneginf(le[[1, 2]]).all() and np.isfinite(le[[0, 3]]).all()
    for col in draws.values():
        c = col.cpu().numpy()
        assert np.isnan(c[:, [1, 2]]).all() and not np.isnan(c[:, [0, 3]]).any()
    with pytest.raises(ValueError):
        bn.sample_posterior({"rewrad": torch.zeros(3)})
    # more data changes the tables; the sampler follows them (cached plans are dropped)
    before = bn.sample_posterior(sub)[1]
    bn.update_knowledge(df[df["reward"] > 0].iloc[:50], accumulate=True)
    draws, after = bn.sample_posterior(sub)
    ref = bn.log_likelihood(sub)
    assert not torch.equal(before, after) and ((after - ref).abs() <= TOL * ref.abs().clamp(min=1)).all()


def test_new_cpts_reach_the_sampler():
    """New CPTs installed on bound tables (``set_cond_tables``) replace the sampler built from the old ones."""
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.asia())
    tables, infer = _install(spec)
    rng = np.random.default_rng(8)
    new = _f32(synth.NetSpec(spec.names, spec.cards, spec.parents,
                             [rng.dirichlet(np.ones(c.shape[-1]), size=c.shape[:-1]) for c in spec.cpts]))
    sub = (7,)
    old_plan = infer.posterior_sampler(["dysp"])
    tables.set_cond_tables(new.cpts)
    assert infer.posterior_sampler(["dysp"]) is not old_plan
    _histogram_check(infer, new, sub, seed=2)
