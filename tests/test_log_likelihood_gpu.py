"""GPU parity of log P(e) and the complete-data log-likelihood (VECompiler.compile_evidence, cbn_loglik_run,
cbn_ve_run_codes_log_evidence) against fp64 oracles, probability identities at full size, and the edges."""
import itertools
import os
import subprocess
import sys

import networkx as nx
import numpy as np
import pandas as pd
import pytest
import torch

from oracle import cbn_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import loglik_oracle as LO  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def _close(got, ref, what=""):
    """|got - ref| <= 1e-5 max(1, |ref|), -inf exactly where the reference is -inf, never NaN."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert not np.isnan(got).any(), what
    dead = np.isneginf(ref)
    assert np.array_equal(np.isneginf(got), dead), what
    g, r = got[~dead], ref[~dead]
    err = np.abs(g - r) / np.maximum(1.0, np.abs(r))
    assert err.size == 0 or err.max() <= 1e-5, f"{what}: worst {err.max():.3g}"


def _install(spec, **cfg):
    from continuousbayesiannetwork_b200.engine import install_cpts

    return install_cpts(spec, DEV, **cfg)


def _run(infer, spec, names, ev):
    return infer.evidence_plan(names).run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()


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
            got = _run(infer, spec, [spec.names[v] for v in sub], ev)
            _close(got, LO.enumerate_log_evidence(net, sub, ev), str(sub))
            assert abs(float(torch.logsumexp(torch.from_numpy(got.astype(np.float64)), 0))) < 1e-5
            n_pairs += ev.shape[0]
    assert n_pairs == 3 ** 8


def test_alarm_evidence_sets_and_complete_data():
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    net = _net(spec)
    codes = synth.sample_forward_numpy(spec, 41, 0, 2051)
    rng = np.random.default_rng(5)
    sets = [[spec.names.index(e) for e in synth.ALARM_EVIDENCE]]
    sets += [list(rng.choice(spec.n, size=int(rng.integers(1, 12)), replace=False)) for _ in range(6)]
    for ids in sets:
        ev = codes[ids].T
        _close(_run(infer, spec, [spec.names[v] for v in ids], ev), LO.ve_log_evidence(net, ids, ev), str(ids))
    plan = infer.evidence_plan(synth.ALARM_EVIDENCE)
    assert [c for _, c in plan.ve_plan.stats.final_tables] == [839808]
    # complete data: only the observed-families kernel, against an fp64 sum of the same log tables
    got = _run(infer, spec, spec.names, codes.T)
    ref = np.zeros(codes.shape[1])
    for v in range(spec.n):
        idx = tuple(codes[p] for p in spec.parents[v]) + (codes[v],)
        ref += np.log(spec.cpts[v][idx])
    _close(got, ref, "complete")
    full = infer.evidence_plan(spec.names)
    assert full.ve_plan is None and full.loglik.lookups_per_row < spec.n


def test_ktree200_complete_data_tables_beyond_one_cta():
    from continuousbayesiannetwork_b200 import synth

    spec = _f32(synth.random_ktree_dag())
    _, infer = _install(spec)
    codes = synth.sample_forward_numpy(spec, 42, 0, 1 << 16)
    got = _run(infer, spec, spec.names, codes.T)
    ref = np.zeros(codes.shape[1])
    for v in range(spec.n):
        idx = tuple(codes[p] for p in spec.parents[v]) + (codes[v],)
        ref += np.log(spec.cpts[v][idx])
    _close(got, ref, "ktree200")
    plan = infer.evidence_plan(spec.names)
    assert plan.ve_plan is None and plan.loglik.lookups_per_row < spec.n


def _alarm_big(n=1 << 22):
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    codes = sample_network(spec, 77, 0, n, DEV, tables=tables)
    return spec, tables, infer, codes


def _sub(codes, ids, n):
    """Rows [ids] of a device code matrix as a fresh evidence matrix (column e = variable ids[e])."""
    return codes[list(ids)].contiguous()


def test_identities_at_full_size():
    from continuousbayesiannetwork_b200 import synth

    n = 1 << 22
    spec, tables, infer, codes = _alarm_big(n)
    E = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    ev = _sub(codes, E, n)
    lpe = infer.evidence_plan(synth.ALARM_EVIDENCE).run_codes(ev, n).double()
    assert not torch.isnan(lpe).any() and torch.isfinite(lpe).all()
    # chain rule: log P(e_1..e_k) = sum_i log P(e_i | e_<i), the conditionals from the posterior plans
    k = 5
    names = synth.ALARM_EVIDENCE[:k]
    chain = torch.zeros(n, dtype=torch.float64, device=DEV)
    for i in range(k):
        post = infer.plan(names[i], names[:i]).run_codes(ev[:max(i, 1)], n) if i else \
            infer.plan(names[0], []).run_codes(ev[:1], 1).expand(n, -1)
        chain += torch.log(post.double().gather(1, ev[i, :n].long().unsqueeze(1)).squeeze(1))
    direct = infer.evidence_plan(names).run_codes(ev[:k].contiguous(), n).double()
    err = ((direct - chain).abs() / direct.abs().clamp(min=1)).max().item()
    assert err <= 1e-5, err
    # Bayes: exp(log P(e, T=t) - log P(e)) is infer's posterior P(t | e)
    for tg in synth.ALARM_TARGETS:
        T = spec.names.index(tg)
        post = infer.plan(tg, synth.ALARM_EVIDENCE).run_codes(ev, n).double()
        plan = infer.evidence_plan(synth.ALARM_EVIDENCE + [tg])
        evt = torch.cat([ev, torch.zeros_like(ev[:1])])
        for t in range(spec.cards[T]):
            evt[-1].fill_(t)
            ratio = torch.exp(plan.run_codes(evt, n).double() - lpe)
            assert (ratio - post[:, t]).abs().max().item() <= 1e-4, (tg, t)
    # marginalisation of one variable: log P(x_{-v}) = logsumexp_v log P(x), from complete-data calls
    v = spec.names.index("HYPOVOLEMIA")
    allv = list(range(spec.n))
    rest = [u for u in allv if u != v]
    m = 1 << 20
    x = codes[:, :m].contiguous()
    full = infer.evidence_plan(spec.names)
    terms = []
    for c in range(spec.cards[v]):
        x[v].fill_(c)
        terms.append(full.run_codes(x, m).double())
    want = torch.logsumexp(torch.stack(terms), 0)
    got = infer.evidence_plan([spec.names[u] for u in rest]).run_codes(_sub(codes, rest, m), m).double()
    err = ((got - want).abs() / want.abs().clamp(min=1)).max().item()
    assert err <= 1e-5, err


def _per_row_check():
    """Per-row log-evidence plans (a 2^10-cell table budget) on Alarm, and a chain whose hidden variables are all left to
    the per-row executor, against the fp64 log-space oracle."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.ve import RowPlan

    spec = _f32(synth.alarm())
    _, infer = _install(spec, table_budget_cells=1 << 10)
    net = _net(spec)
    codes = synth.sample_forward_numpy(spec, 31, 0, 1031)
    for names in (synth.ALARM_EVIDENCE, synth.ALARM_EVIDENCE[:8]):
        ids = [spec.names.index(e) for e in names]
        ev = codes[ids].T.copy()
        ev[5, 1] = 255
        plan = infer.evidence_plan(names)
        assert isinstance(plan.ve_plan, RowPlan)
        got = _run(infer, spec, names, ev)
        _close(got, LO.ve_log_evidence(net, ids, ev), str(names))
        plan.set_static_evidence(True)          # accepted by a per-row plan; its kernels do not read the flag
        assert np.array_equal(_run(infer, spec, names, ev).view(np.uint32), got.view(np.uint32))
    n_e = 22
    names2 = ["T"] + [f"h{i:02d}" for i in range(n_e)] + [f"e{i:02d}" for i in range(n_e)]
    parents2 = [[]] + [[0]] * n_e + [[1 + i] for i in range(n_e)]
    rng = np.random.default_rng(8)
    cpts = [np.array([0.5, 0.5])] + [np.array([[0.9, 0.1], [0.2, 0.8]])] * n_e
    for i in range(n_e):
        a, b = 1e-3 * (1 + rng.random()), 3e-3 * (1 + rng.random())
        cpts.append(np.array([[1 - a, a], [1 - b, b]]))
    spec2 = _f32(synth.NetSpec(names2, [2] * len(names2), parents2, cpts))
    _, infer2 = _install(spec2, table_budget_cells=1)
    ev = np.concatenate([np.ones((3, n_e), dtype=np.int64), rng.integers(0, 2, size=(61, n_e))])
    plan = infer2.evidence_plan(names2[1 + n_e:])
    assert isinstance(plan.ve_plan, RowPlan)
    _close(_run(infer2, spec2, names2[1 + n_e:], ev), LO.ve_log_evidence(_net(spec2), list(range(1 + n_e, 1 + 2 * n_e)), ev), "chain")


def test_per_row_plans_thread_kernel():
    _per_row_check()


def test_per_row_plans_warp_kernel():
    env = dict(os.environ, CBN_ROWS_THREAD="0")
    code = "import runpy; runpy.run_path('tests/test_log_likelihood_gpu.py')['_per_row_check'](); print('ok')"
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and "ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


def test_range_tiny_evidence_and_a_long_chain():
    from continuousbayesiannetwork_b200 import synth

    # a binary cause with 22 observed effects: the all-ones evidence has probability ~1e-60
    n_e = 22
    names = ["T"] + [f"e{i:02d}" for i in range(n_e)]
    rng = np.random.default_rng(8)
    cpts = [np.array([0.5, 0.5])]
    for i in range(n_e):
        a, b = 1e-3 * (1 + rng.random()), 3e-3 * (1 + rng.random())
        cpts.append(np.array([[1 - a, a], [1 - b, b]]))
    spec = _f32(synth.NetSpec(names, [2] * (n_e + 1), [[]] + [[0]] * n_e, cpts))
    ev = np.concatenate([np.ones((3, n_e), dtype=np.int64), rng.integers(0, 2, size=(61, n_e))])
    for cfg in ({}, {"merge_budget_cells": 1 << 8}):
        _, infer = _install(spec, **cfg)
        got = _run(infer, spec, names[1:], ev)
        want = LO.ve_log_evidence(_net(spec), list(range(1, n_e + 1)), ev)
        assert want[0] < np.log(1e-50)
        _close(got, want, str(cfg))
    # a 300-node chain, evidence on every other node: log P(e) < -1000, beyond even fp64's linear range
    n = 300
    names = [f"c{i:03d}" for i in range(n)]
    parents = [[]] + [[i - 1] for i in range(1, n)]
    cp = [np.array([0.5, 0.5])] + [np.array([[0.9998, 0.0002], [0.0002, 0.9998]])] * (n - 1)
    spec = _f32(synth.NetSpec(names, [2] * n, parents, cp))
    _, infer = _install(spec)
    ids = list(range(0, n, 2))
    ev = np.tile(np.array([0, 1], dtype=np.int64), (5, (len(ids) + 1) // 2))[:, :len(ids)]
    ev[1] = 0
    got = _run(infer, spec, [names[i] for i in ids], ev)
    want = LO.ve_log_evidence(_net(spec), ids, ev)
    assert want[0] < -1000
    _close(got, want, "chain300")


def test_edges_row_counts_unseen_zero_probability_and_determinism():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    net = _net(spec)
    codes = synth.sample_forward_numpy(spec, 43, 0, 1001)
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    for n in (0, 1, 3, 4, 5, 1001):
        ev = codes[ids, :n].T
        got = _run(infer, spec, synth.ALARM_EVIDENCE, ev)
        assert got.shape == (n,)
        _close(got, LO.ve_log_evidence(net, ids, ev), f"{n} rows")
        for names in (spec.names, []):                       # complete rows; no evidence
            vs = [spec.names.index(x) for x in names]
            got = _run(infer, spec, names, codes[vs, :n].T)
            assert got.shape == (n,)
            _close(got, LO.ve_log_evidence(net, vs, codes[vs, :n].T), f"{n} rows, {len(names)} columns")
    # unseen values give -inf, never NaN: CBN_UNSEEN through the gather plan; CBN_UNSEEN or any code >= the cardinality
    # through the observed-families kernel
    ev = codes[ids, :64].T.copy()
    ev[3, 0] = 255
    ev[7, 4] = 255
    got = _run(infer, spec, synth.ALARM_EVIDENCE, ev)
    assert np.isneginf(got[3]) and np.isneginf(got[7]) and np.isfinite(np.delete(got, [3, 7])).all()
    full = codes[:, :64].T.copy()
    full[9, 2] = 255
    full[11, 5] = 200
    got = _run(infer, spec, spec.names, full)
    assert np.isneginf(got[9]) and np.isneginf(got[11]) and np.isfinite(np.delete(got, [9, 11])).all()
    # zero-probability evidence: a CPT row with zeros
    cp = [c.copy() for c in spec.cpts]
    v = spec.names.index("HISTORY")
    cp[v][..., 0] = 0.0
    cp[v][..., 1] = 1.0
    spec0 = synth.NetSpec(spec.names, spec.cards, spec.parents, cp)
    _, inf0 = _install(spec0)
    ev = codes[ids, :256].T
    got = _run(inf0, spec0, synth.ALARM_EVIDENCE, ev)
    want = LO.ve_log_evidence(_net(spec0), ids, ev)
    assert np.isneginf(want).any()
    _close(got, want, "zero probability")
    got = _run(inf0, spec0, spec0.names, codes[:, :256].T)
    assert np.isneginf(got).any() and not np.isnan(got).any()
    # tile-staged batches (>= 2^21 rows) equal the direct kernel on the same rows, and any split gives identical bits
    n = (1 << 21) + 37
    big = sample_network(spec, 99, 0, n, DEV, tables=tables)
    ev = big[ids].contiguous()
    plan = infer.evidence_plan(synth.ALARM_EVIDENCE)
    a = plan.run_codes(ev, n)
    b = plan.run_codes(ev, n)
    assert torch.equal(a, b)
    h = 1 << 20
    parts = torch.cat([plan.run_codes(ev[:, :h].contiguous(), h), plan.run_codes(ev[:, h:].contiguous(), n - h)])
    assert torch.equal(a, parts)
    c = infer.evidence_plan(spec.names).run_codes(big, n)
    parts = torch.cat([infer.evidence_plan(spec.names).run_codes(big[:, :h].contiguous(), h),
                       infer.evidence_plan(spec.names).run_codes(big[:, h:].contiguous(), n - h)])
    assert torch.equal(c, parts)


def _tiles_dump(path):
    """log P(e) of the headline evidence set on 2^21 + 37 seeded rows, saved to ``path`` (run under CBN_GATHER_TILES)."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import sample_network

    spec = _f32(synth.alarm())
    tables, infer = _install(spec)
    n = (1 << 21) + 37
    big = sample_network(spec, 99, 0, n, DEV, tables=tables)
    ev = big[[spec.names.index(e) for e in synth.ALARM_EVIDENCE]].contiguous()
    np.save(path, infer.evidence_plan(synth.ALARM_EVIDENCE).run_codes(ev, n).cpu().numpy())


def test_tile_staged_equals_direct_kernel(tmp_path):
    code = "import runpy, sys; runpy.run_path('tests/test_log_likelihood_gpu.py')['_tiles_dump'](sys.argv[1]); print('ok')"
    outs = []
    for mode in ("0", "1"):
        path = str(tmp_path / f"tiles{mode}.npy")
        env = dict(os.environ, CBN_GATHER_TILES=mode)
        out = subprocess.run([sys.executable, "-c", code, path], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
        assert out.returncode == 0 and "ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
        outs.append(np.load(path))
    assert np.isfinite(outs[0]).all()
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))


def test_cuda_graph_replay_of_gather_then_accumulate():
    """The gather kernel triggers programmatic dependent launch at entry; the observed-families kernel that adds into its
    output must still see every store.  Replayed from a CUDA graph with static evidence, as a resident batch is."""
    from continuousbayesiannetwork_b200 import synth

    n = 1 << 20
    spec, tables, infer, codes = _alarm_big(n)
    names = synth.ALARM_EVIDENCE + ["HYPOVOLEMIA", "LVFAILURE"]       # both kernels: VE gather + observed families
    ids = [spec.names.index(e) for e in names]
    ev = _sub(codes, ids, n)
    plan = infer.evidence_plan(names)
    assert plan.ve_plan is not None and plan.loglik is not None
    eager = plan.run_codes(ev, n).clone()
    plan.set_static_evidence(True)
    out = torch.full((n,), float("nan"), device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        plan.run_codes(ev, n, out)                         # warm-up (lazy attributes) outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        plan.run_codes(ev, n, out)
    for _ in range(3):
        out.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
    plan.set_static_evidence(False)


def _frozen_lake(golden_dir):
    from continuousbayesiannetwork_b200 import BayesianNetwork

    g = np.load(os.path.join(golden_dir, "frozen_lake.npz"), allow_pickle=False)
    df = pd.DataFrame(g["data"], columns=["obs_0", "action", "reward"])
    dag = nx.DiGraph()
    dag.add_edges_from([("obs_0", "reward"), ("action", "reward")])
    return g, df, BayesianNetwork(dag, df, {"estimator_name": "brute_force"}, {"inference_obj": "exact"}, device=DEV)


def test_network_log_likelihood(golden_dir):
    g, df, bn = _frozen_lake(golden_dir)
    t = bn.tables

    def ref_complete(frame):
        out = np.zeros(len(frame))
        for name in ("obs_0", "action", "reward"):
            pa = bn.get_parents(bn.initial_dag, name)
            pts = torch.tensor(frame[name].to_numpy(np.float32)[:, None], device=DEV)
            q = torch.tensor(np.ascontiguousarray(frame[pa].to_numpy(np.float32))[:, :, None], device=DEV) if pa else None
            if q is None:
                p = t.cond[t.offsets[t.index[name]]: t.offsets[t.index[name]] + t.n_cells[t.index[name]]].double().cpu().numpy()
                codes = np.searchsorted(t.domains[t.index[name]].cpu().numpy(), frame[name].to_numpy(np.float32))
                out += np.log(p[codes])
            else:
                out += np.log(t.get_prob(name, pts, q).double().cpu().numpy()[:, 0])
        return out

    got = bn.log_likelihood(df).cpu().numpy()
    _close(got, ref_complete(df), "frozen lake complete")
    # a subset of the columns: the others are summed out
    spec_cards = [t.cards[i] for i in range(len(t.names))]
    parents = [[t.index[p] for p in t.parents[n]] for n in t.names]
    cpts = [t.table_view(t.cond, n).double().cpu().numpy() for n in t.names]
    net = O.DiscreteNet(spec_cards, parents, cpts)
    sub = ["reward", "action"]
    got = bn.log_likelihood({k: torch.tensor(df[k].to_numpy(np.float32)) for k in sub}).cpu().numpy()
    codes = np.stack([np.searchsorted(t.domains[t.index[k]].cpu().numpy(), df[k].to_numpy(np.float32)) for k in sub], 1)
    _close(got, LO.ve_log_evidence(net, [t.index[k] for k in sub], codes), "subset")
    # a value outside the fitted domain and NaN give -inf; an unknown column raises
    bad = df.iloc[:4].copy()
    bad.iloc[1, 0] = 12345.0
    bad.iloc[2, 1] = float("nan")
    got = bn.log_likelihood(bad).cpu().numpy()
    assert np.isneginf(got[1]) and np.isneginf(got[2]) and np.isfinite(got[[0, 3]]).all()
    with pytest.raises(ValueError):
        bn.log_likelihood({"reward": torch.zeros(3), "rewrad": torch.zeros(3)})
    assert torch.equal(bn.log_likelihood(df[[]]), torch.zeros(len(df), device=DEV))
    # accumulating more data changes the tables, and the scores follow them
    before = bn.log_likelihood(df).cpu().numpy()
    extra = df[df["reward"] > 0].iloc[:50]
    bn.update_knowledge(extra, accumulate=True)
    after = bn.log_likelihood(df).cpu().numpy()
    assert not np.array_equal(before, after)
    _close(after, ref_complete(df), "after update_knowledge")
