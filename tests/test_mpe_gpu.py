"""GPU parity of the most probable explanation (cbn_factor_contract_max, VECompiler.compile_mpe, cbn_mpe_run) against fp64
oracles, the log-likelihood identity at full size, local optimality on the 200-node DAG, and the edges."""
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
import mpe_oracle as MO  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5


def _f32(spec):
    """The spec with its CPTs rounded to fp32, as the device holds them: the oracle then scores the same numbers."""
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


def _tol(ref):
    return TOL * np.maximum(1.0, np.abs(ref))


def _run(infer, names, ev):
    """(plan, full code rows int [n_rows, n_vars] with the decoded hidden values, log_prob fp64 [n_rows])"""
    plan = infer.mpe_plan(names)
    n = ev.shape[0]
    hidden, value = plan.run_codes(_codes_matrix(ev), n)
    full = np.zeros((n, len(infer.tables.names)), np.int64)
    for i, v in enumerate(plan.evidence):
        full[:, v] = ev[:, i]
    hc = hidden[:, :n].cpu().numpy().astype(np.int64)
    for h, v in enumerate(plan.hidden):
        full[:, v] = hc[h]
    return plan, full, value.cpu().numpy().astype(np.float64)


def _check(net, ev_ids, ev, full, got, best, second=None, assign=None, what=""):
    """log_prob within TOL of the fp64 best, -inf exactly where it is, never NaN; dead rows decode to CBN_UNSEEN; the
    assignment is optimal (its fp64 log joint within TOL of the best) and equals the oracle's where the best is clear."""
    assert not np.isnan(got).any(), what
    dead = np.isneginf(best)
    assert np.array_equal(np.isneginf(got), dead), what
    hid = [v for v in range(net.n) if v not in ev_ids]
    assert (full[dead][:, hid] == 255).all(), what
    live = ~dead
    assert (np.abs(got[live] - best[live]) <= _tol(best[live])).all(), what
    lj = MO.log_joint(net, full[live])
    assert (np.abs(lj - best[live]) <= _tol(best[live])).all(), what
    if assign is not None:
        clear = live & ~(second >= best - 1e-4)
        assert np.array_equal(full[clear], assign[clear]), what


# ------------------------------------------------------------------------------------------------ the max contraction
def _contract_max(inputs, in_axes, out_cards, sum_card):
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
    am = torch.full((n_out,), 77, dtype=torch.uint8, device=DEV)
    d.out = out.data_ptr()
    d.log_space = 1
    N.check(N.lib().cbn_factor_contract_max(ctx.handle, C.byref(d), am.data_ptr(), N.stream_ptr(DEV)), ctx.handle)
    torch.cuda.synchronize()
    return out.cpu().numpy(), am.cpu().numpy(), d, ctx


def test_contract_max_against_numpy_ties_and_minus_inf():
    from continuousbayesiannetwork_b200 import _native as N

    rng = np.random.default_rng(3)
    shapes = [([3, 4], 5), ([2, 3, 2], 7), ([64, 32, 40], 3), ([16, 16, 16, 17], 4), ([5], 255)]
    for out_cards, sum_card in shapes:
        for n_in in range(1, 6):
            allc = list(out_cards) + [sum_card]
            nd = len(allc)
            in_axes, ts, hs = [], [], []
            for k in range(n_in):
                axes = sorted(set(int(a) for a in rng.choice(nd, size=int(rng.integers(1, nd + 1)), replace=False)) |
                              ({nd - 1} if k == 0 else set()))
                h = (rng.integers(-6, 1, size=[allc[a] for a in axes]) * 0.5).astype(np.float32)   # exact halves: real ties
                h[rng.random(h.shape) < 0.15] = -np.inf
                in_axes.append(axes)
                hs.append(h)
                ts.append(torch.from_numpy(h.reshape(-1)).to(DEV))
            got, am, d, ctx = _contract_max(ts, in_axes, out_cards, sum_card)
            acc = np.zeros(allc, dtype=np.float32)
            for h, axes in zip(hs, in_axes):                            # fp32, in input order, as the kernel adds
                acc = (acc + h.reshape([allc[a] if a in axes else 1 for a in range(nd)])).astype(np.float32)
            want = acc.max(axis=-1).reshape(-1)
            arg = acc.argmax(axis=-1).reshape(-1)                       # first maximum; 0 for an all -inf slice
            assert np.array_equal(got, want), (out_cards, n_in)
            assert np.array_equal(am, arg.astype(np.uint8)), (out_cards, n_in)
    # an all -inf reduction: -inf and index 0
    t = torch.full((4 * 3,), float("-inf"), device=DEV)
    got, am, d, ctx = _contract_max([t], [[0, 1]], [4], 3)
    assert np.isneginf(got).all() and (am == 0).all()
    # argument checks
    for field, val in (("log_space", 0), ("normalize_last", 1)):
        setattr(d, field, val)
        with pytest.raises(ValueError):
            N.check(N.lib().cbn_factor_contract_max(ctx.handle, C.byref(d), ts[0].data_ptr(), N.stream_ptr(DEV)), ctx.handle)
        setattr(d, field, 1 - val)
    with pytest.raises(ValueError):
        N.check(N.lib().cbn_factor_contract_max(ctx.handle, C.byref(d), None, N.stream_ptr(DEV)), ctx.handle)


# ------------------------------------------------------------------------------------------------ against the oracles
def test_asia_every_subset_and_configuration():
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.asia())
    _, infer = _install(spec)
    net = _net(spec)
    n_pairs = 0
    for k in range(spec.n + 1):
        for sub in itertools.combinations(range(spec.n), k):
            cards = [spec.cards[v] for v in sub]
            ev = np.ascontiguousarray(np.indices(cards).reshape(k, -1).T) if k else np.zeros((1, 0), np.int64)
            _, full, got = _run(infer, [spec.names[v] for v in sub], ev)
            best, second, assign = MO.enumerate_mpe(net, sub, ev)
            _check(net, sub, ev, full, got, best, second, assign, str(sub))
            n_pairs += ev.shape[0]
    assert n_pairs == 3 ** 8


def test_random_dags_with_zeros_against_enumeration():
    from continuousbayesiannetwork_b200 import synth

    rng = np.random.default_rng(2025)
    for trial in range(25):
        cards, parents, cpts = MO.random_small_net(rng)
        names = [f"v{i}" for i in range(len(cards))]
        spec = _f32(synth.NetSpec(names, cards, parents, cpts))
        net = _net(spec)
        _, infer = _install(spec)
        for _ in range(3):
            k = int(rng.integers(0, len(cards) + 1))
            ids = sorted(int(v) for v in rng.choice(len(cards), size=k, replace=False))
            ev = np.stack([rng.integers(0, cards[v], size=53) for v in ids], axis=1) if ids else np.zeros((1, 0), np.int64)
            _, full, got = _run(infer, [names[v] for v in ids], ev)
            best, second, assign = MO.enumerate_mpe(net, ids, ev)
            _check(net, ids, ev, full, got, best, second, assign, f"trial {trial} {ids}")


def _device_loglik(infer, full_dev, n, order):
    """log_likelihood of complete rows on the device: full_dev uint8 [n_vars, ld] with row v = network variable order[v]"""
    names = [infer.tables.names[v] for v in order]
    return infer.evidence_plan(names).run_codes(full_dev, n).double()


def _stack(plan, ev_dev, hidden, n):
    return torch.cat([ev_dev[:len(plan.evidence), :hidden.shape[1]], hidden]).contiguous() if plan.evidence else hidden


def test_alarm_headline_sampled_rows():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    net = _net(spec)
    n = 1 << 16
    codes = sample_network(spec, 51, 0, n, DEV, tables=tables)
    E = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    ev = codes[E].contiguous()
    plan = infer.mpe_plan(synth.ALARM_EVIDENCE)
    assert len(plan.hidden) == 25 and [c for _, c in plan.value.ve_plan.stats.final_tables] == [839808]
    hidden, value = plan.run_codes(ev, n)
    assert torch.isfinite(value).all()
    # identity on every row: the device log-likelihood of the completed rows is the returned value
    lj = _device_loglik(infer, _stack(plan, ev, hidden, n), n, plan.evidence + plan.hidden)
    v = value.double()
    assert ((lj - v).abs() <= TOL * v.abs().clamp(min=1)).all()
    # a sample against the fp64 max-product oracle, and fp64 optimality of the assignment
    rows = np.sort(np.random.default_rng(0).choice(n, size=4096, replace=False))
    r = torch.from_numpy(rows).to(DEV)
    evs = ev[:, r].cpu().numpy().T.astype(np.int64)
    best, _ = MO.ve_mpe(net, E, evs)
    full = np.zeros((len(rows), spec.n), np.int64)
    full[:, E] = evs
    full[:, plan.hidden] = hidden[:, r].cpu().numpy().T
    _check(net, E, evs, full, value[r].cpu().numpy().astype(np.float64), best, what="alarm headline")


def test_alarm_evidence_sets_of_every_size():
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.alarm())
    _, infer = _install(spec)
    net = _net(spec)
    codes = synth.sample_forward_numpy(spec, 52, 0, 257)
    rng = np.random.default_rng(9)
    for k in range(spec.n + 1):
        ids = [int(v) for v in rng.choice(spec.n, size=k, replace=False)]
        ev = codes[ids].T.astype(np.int64) if k else np.zeros((1, 0), np.int64)
        plan, full, got = _run(infer, [spec.names[v] for v in ids], ev)
        assert len(plan.hidden) == spec.n - k
        best, _ = MO.ve_mpe(net, ids, ev)
        _check(net, ids, ev, full, got, best, what=f"{k} evidence variables")
        if k == spec.n:
            assert plan.value.ve_plan is None
            ll = infer.evidence_plan(spec.names[v] for v in ids)
            assert np.array_equal(got, ll.run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy().astype(np.float64))


def test_ktree200_bench_patterns_identity_and_local_optimality():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.random_ktree_dag())
    tables, infer = _install(spec)
    n = 1 << 20
    full_codes = sample_network(spec, 53, 0, n, DEV, tables=tables)
    rng = np.random.default_rng(1240)
    pats = [[int(v) for v in rng.choice(spec.n, size=11, replace=False)] for _ in range(8)]
    for vs in pats:
        ids = vs[1:]
        plan = infer.mpe_plan([spec.names[v] for v in ids])
        ev = full_codes[ids].contiguous()
        hidden, value = plan.run_codes(ev, n)
        assert torch.isfinite(value).all() and len(plan.hidden) == 190
        order = plan.evidence + plan.hidden
        comp = _stack(plan, ev, hidden, n)
        lj = _device_loglik(infer, comp, n, order)
        v = value.double()
        assert ((lj - v).abs() <= TOL * v.abs().clamp(min=1)).all()
        # single flips of a sample of rows, scored on the device: no hidden variable's change raises the joint
        m = 64
        rows = torch.from_numpy(np.sort(rng.choice(n, size=m, replace=False))).to(DEV)
        base = comp[:, rows]
        flips = []
        for j in range(len(plan.evidence), len(order)):
            for dc in range(1, spec.cards[order[j]]):
                f = base.clone()
                f[j] = (f[j].int() + dc) % spec.cards[order[j]]
                flips.append(f)
        allf = torch.cat(flips, dim=1)
        k = allf.shape[1]
        ld = (k + 15) // 16 * 16
        mat = torch.zeros((len(order), ld), dtype=torch.uint8, device=DEV)
        mat[:, :k] = allf
        scores = _device_loglik(infer, mat, k, order).reshape(-1, m)
        b = v[rows]
        assert (scores <= b + TOL * b.abs().clamp(min=1)).all()


# ------------------------------------------------------------------------------------------------ edges
def test_edges_unseen_zero_probability_batches_determinism_and_budget():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network
    from continuousbayesiannetwork_b200.ve import PlanTooLarge

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    net = _net(spec)
    E = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    codes = synth.sample_forward_numpy(spec, 54, 0, 1001)
    for n in (0, 1, 15, 16, 17, 1001):
        ev = codes[E, :n].T.astype(np.int64)
        plan, full, got = _run(infer, synth.ALARM_EVIDENCE, ev)
        assert got.shape == (n,)
        if n:
            _check(net, E, ev, full, got, MO.ve_mpe(net, E, ev)[0], what=f"{n} rows")
    # unseen codes: -inf and CBN_UNSEEN in every hidden column, never NaN
    ev = codes[E, :64].T.astype(np.int64)
    ev[3, 0] = 255
    ev[7, 4] = 255
    plan, full, got = _run(infer, synth.ALARM_EVIDENCE, ev)
    assert np.isneginf(got[[3, 7]]).all() and np.isfinite(np.delete(got, [3, 7])).all()
    assert (full[[3, 7]][:, plan.hidden] == 255).all() and (np.delete(full, [3, 7], 0)[:, plan.hidden] < 255).all()
    # zero-probability evidence
    cp = [c.copy() for c in spec.cpts]
    v = spec.names.index("HISTORY")
    cp[v][..., 0] = 0.0
    cp[v][..., 1] = 1.0
    spec0 = synth.NetSpec(spec.names, spec.cards, spec.parents, cp)
    _, inf0 = _install(spec0)
    ev = codes[E, :256].T.astype(np.int64)
    plan, full, got = _run(inf0, synth.ALARM_EVIDENCE, ev)
    best, _ = MO.ve_mpe(_net(spec0), E, ev)
    assert np.isneginf(best).any() and np.isfinite(best).any()
    _check(_net(spec0), E, ev, full, got, best, what="zero probability")
    # identical bits across calls and across batch splits
    n = (1 << 20) + 37
    big = sample_network(spec, 55, 0, n, DEV, tables=tables)
    ev = big[E].contiguous()
    plan = infer.mpe_plan(synth.ALARM_EVIDENCE)
    h1, v1 = plan.run_codes(ev, n)
    h2, v2 = plan.run_codes(ev, n)
    assert torch.equal(h1[:, :n], h2[:, :n]) and torch.equal(v1, v2)
    s = 1 << 19
    ha, va = plan.run_codes(ev[:, :s].contiguous(), s)
    hb, vb = plan.run_codes(ev[:, s:].contiguous(), n - s)
    assert torch.equal(torch.cat([va, vb]), v1)
    assert torch.equal(torch.cat([ha[:, :s], hb[:, :n - s]], 1), h1[:, :n])
    # no per-row executor: the layered DAG fails in the structure-only pass
    _, linf = _install(_f32(synth.layered_dag()))
    with pytest.raises(PlanTooLarge):
        linf.mpe_plan([])


def test_cuda_graph_replay_of_gather_accumulate_traceback():
    """The gather kernel triggers programmatic dependent launch at entry; the observed-families kernel adds into its output
    and the traceback reads that output: replayed from a CUDA graph with static evidence, every store must be seen."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    n = 1 << 20
    codes = sample_network(spec, 56, 0, n, DEV, tables=tables)
    names = synth.ALARM_EVIDENCE + ["HYPOVOLEMIA", "LVFAILURE"]
    ev = codes[[spec.names.index(e) for e in names]].contiguous()
    plan = infer.mpe_plan(names)
    assert plan.value.ve_plan is not None and plan.value.loglik is not None
    h_eager, v_eager = plan.run_codes(ev, n)
    h_eager, v_eager = h_eager.clone(), v_eager.clone()
    plan.set_static_evidence(True)
    hid = torch.full_like(h_eager, 7)
    val = torch.full((n,), float("nan"), device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        plan.run_codes(ev, n, hid, val)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        plan.run_codes(ev, n, hid, val)
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


def test_network_most_probable_explanation(golden_dir):
    df, bn = _frozen_lake(golden_dir)
    t = bn.tables
    sub = df[["reward"]].iloc[:500]
    assign, lp = bn.most_probable_explanation(sub)
    assert sorted(assign) == ["action", "obs_0"] and lp.shape == (500,) and lp.dtype == torch.float32
    for name, col in assign.items():
        assert col.shape == (500,) and col.dtype == torch.float32 and col.is_cuda
        assert torch.isin(col, t.domains[t.index[name]]).all()
    done = {"reward": torch.tensor(sub["reward"].to_numpy(np.float32), device=DEV), **assign}
    ll = bn.log_likelihood(done)
    assert ((ll - lp).abs() <= TOL * lp.abs().clamp(min=1)).all()
    # brute force over the two hidden nodes
    doms = {n: t.domains[t.index[n]] for n in ("obs_0", "action")}
    grid = [(a, b) for a in doms["obs_0"].tolist() for b in doms["action"].tolist()]
    r = torch.tensor(sub["reward"].to_numpy(np.float32), device=DEV)
    scores = torch.stack([bn.log_likelihood({"obs_0": torch.full_like(r, a), "action": torch.full_like(r, b), "reward": r})
                          for a, b in grid])
    assert ((scores.max(0).values - lp).abs() <= TOL * lp.abs().clamp(min=1)).all()
    # complete rows: nothing to decode, the value is the log-likelihood; no columns: one row, the prior's explanation
    assign, lp = bn.most_probable_explanation(df.iloc[:100])
    assert assign == {} and torch.equal(lp, bn.log_likelihood(df.iloc[:100]))
    assign, lp = bn.most_probable_explanation(df[[]])
    assert lp.shape == (1,) and sorted(assign) == ["action", "obs_0", "reward"]
    # unseen value and NaN: -inf and NaN columns, never a NaN log_prob; unknown column raises
    bad = df[["reward"]].iloc[:4].copy()
    bad.iloc[1, 0] = 12345.0
    bad.iloc[2, 0] = float("nan")
    assign, lp = bn.most_probable_explanation(bad)
    lp = lp.cpu().numpy()
    assert np.isneginf(lp[[1, 2]]).all() and np.isfinite(lp[[0, 3]]).all()
    for col in assign.values():
        c = col.cpu().numpy()
        assert np.isnan(c[[1, 2]]).all() and not np.isnan(c[[0, 3]]).any()
    with pytest.raises(ValueError):
        bn.most_probable_explanation({"rewrad": torch.zeros(3)})
    # more data changes the tables; the explanation follows them (cached plans are dropped)
    before = bn.most_probable_explanation(sub)[1]
    bn.update_knowledge(df[df["reward"] > 0].iloc[:50], accumulate=True)
    assign, after = bn.most_probable_explanation(sub)
    assert not torch.equal(before, after)
    done = {"reward": torch.tensor(sub["reward"].to_numpy(np.float32), device=DEV), **assign}
    ll = bn.log_likelihood(done)
    assert ((ll - after).abs() <= TOL * after.abs().clamp(min=1)).all()


def test_network_alarm_headline():
    from continuousbayesiannetwork_b200 import BayesianNetwork, synth

    spec = synth.alarm()
    codes = synth.sample_forward_numpy(spec, 57, 0, 200_000)
    df = pd.DataFrame({n: codes[i].astype(np.float32) for i, n in enumerate(spec.names)})
    dag = nx.DiGraph()
    dag.add_nodes_from(spec.names)
    dag.add_edges_from((spec.names[p], spec.names[i]) for i in range(spec.n) for p in spec.parents[i])
    bn = BayesianNetwork(dag, df, {"estimator_name": "brute_force"}, {"inference_obj": "exact"}, device=DEV)
    ev = df[synth.ALARM_EVIDENCE].iloc[:4096]
    assign, lp = bn.most_probable_explanation(ev)
    assert len(assign) == 25 and set(assign) == set(spec.names) - set(synth.ALARM_EVIDENCE)
    done = {n: torch.tensor(ev[n].to_numpy(np.float32), device=DEV) for n in synth.ALARM_EVIDENCE}
    done.update(assign)
    ll = bn.log_likelihood(done)
    fin = torch.isfinite(lp)
    assert fin.any() and torch.equal(torch.isfinite(ll), fin)
    assert ((ll[fin] - lp[fin]).abs() <= TOL * lp[fin].abs().clamp(min=1)).all()
