"""GPU parity: batched Variable Elimination against the fp32 textbook-VE oracle (O2), fp64 full
enumeration (O3) and -- where the reference itself is a posterior -- the live reference's outputs."""
import os

import numpy as np
import pytest
import torch

from oracle import cbn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-5          # north_star: posteriors within 1e-5 relative in fp32


def _net(spec):
    return O.DiscreteNet(spec.cards, spec.parents, spec.cpts)


def _codes_matrix(ev: np.ndarray) -> torch.Tensor:
    """[n_rows, n_ev] numpy codes -> uint8 [n_ev, ld] device matrix (ld multiple of 16)."""
    n, k = ev.shape
    ld = (n + 15) // 16 * 16
    m = torch.zeros((max(k, 1), max(ld, 16)), dtype=torch.uint8, device=DEV)
    if k:
        m[:, :n] = torch.from_numpy(np.ascontiguousarray(ev.T.astype(np.uint8))).to(DEV)
    return m


def _check(spec, infer, target, ev_names, ev, rtol=RTOL, truth64=True):
    net = _net(spec)
    ids = [spec.names.index(e) for e in ev_names]
    plan = infer.plan(target, ev_names)
    got = plan.run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
    want = O.ve_posterior(net, spec.names.index(target), ids, ev)
    np.testing.assert_allclose(got, want, rtol=rtol, atol=1e-30)
    if truth64:
        w64 = O.ve_posterior(net, spec.names.index(target), ids, ev, dtype=torch.float64)
        np.testing.assert_allclose(got, w64, rtol=rtol, atol=1e-30)
    rs = got.sum(1)       # a distribution, or all zeros when the evidence has probability 0
    assert np.all((np.abs(rs - 1) < 1e-5) | (rs == 0))
    return plan, got


def test_asia_all_evidence_configurations():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.asia()
    _, infer = install_cpts(spec, DEV)
    ev_names = ["asia", "smoke", "xray", "dysp"]
    ev = np.array([[(i >> k) & 1 for k in range(4)] for i in range(16)] * 3)[:45]   # 45 rows: not a multiple of 4
    for target in ("lung", "tub", "bronc", "either"):
        plan, got = _check(spec, infer, target, ev_names, ev)
        truth = O.enumerate_posterior(_net(spec), spec.names.index(target), [spec.names.index(e) for e in ev_names], ev)
        np.testing.assert_allclose(got, truth, rtol=RTOL, atol=1e-30)
        assert plan.algorithmic_bytes_per_row() == 4 + 8
    # other evidence sets, including evidence below / above the target and none at all
    rng = np.random.default_rng(1)
    for target, names in (("lung", ["smoke"]), ("smoke", ["lung", "dysp"]), ("either", []), ("asia", ["xray"]),
                          ("dysp", ["asia", "tub", "smoke", "lung", "bronc", "either", "xray"])):
        ev = rng.integers(0, 2, size=(33, len(names)))
        _check(spec, infer, target, names, ev)


def test_new_cpts_reach_every_plan():
    """New CPTs installed on bound tables (``set_cond_tables``, no re-fit and no re-bind) replace every plan built from
    the old ones: posterior plans, fused posteriors, log P(e) and MPE all answer from the new tables."""
    import sys

    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import loglik_oracle as LO
    import mpe_oracle as MO

    spec = synth.asia()
    tables, infer = install_cpts(spec, DEV)
    ev_names = ["asia", "smoke", "xray", "dysp"]
    ids = [spec.names.index(e) for e in ev_names]
    ev = np.array([[(i >> k) & 1 for k in range(4)] for i in range(16)])
    cols = {n: torch.tensor(ev[:, e], dtype=torch.float32, device=DEV) for e, n in enumerate(ev_names)}
    rng = np.random.default_rng(11)
    new = synth.NetSpec(spec.names, spec.cards, spec.parents,
                        [rng.dirichlet(np.ones(c.shape[-1]), size=c.shape[:-1]).astype(np.float32).astype(np.float64)
                         for c in spec.cpts])
    for s in (spec, new):
        if s is new:
            tables.set_cond_tables(new.cpts)
        net = _net(s)
        many = infer.infer_many(["lung", "bronc"], cols)           # two targets of two values: one fused launch
        for tg in ("lung", "bronc"):
            want = O.enumerate_posterior(net, s.names.index(tg), ids, ev)
            np.testing.assert_allclose(infer.plan(tg, ev_names).run_codes(_codes_matrix(ev), 16).cpu().numpy(), want,
                                       rtol=RTOL, atol=1e-30)
            np.testing.assert_allclose(many[tg].cpu().numpy(), want, rtol=RTOL, atol=1e-30)
        np.testing.assert_allclose(infer.log_evidence(cols).cpu().numpy(), LO.enumerate_log_evidence(net, ids, ev),
                                   rtol=1e-5, atol=1e-5)
        assignment, log_prob = infer.most_probable_explanation(cols)
        best, _, _ = MO.enumerate_mpe(net, ids, ev)
        np.testing.assert_allclose(log_prob.cpu().numpy(), best, rtol=1e-5, atol=1e-5)
        full = np.zeros((16, s.n), dtype=np.int64)
        full[:, ids] = ev
        for name, vals in assignment.items():
            full[:, s.names.index(name)] = vals.cpu().numpy().astype(np.int64)
        np.testing.assert_allclose(MO.log_joint(net, full), best, rtol=1e-5, atol=1e-5)


def test_alarm_and_random_dags():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.alarm()
    _, infer = install_cpts(spec, DEV)
    codes = synth.sample_forward_numpy(spec, 21, 0, 2051)
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    for target in synth.ALARM_TARGETS:
        plan, _ = _check(spec, infer, target, synth.ALARM_EVIDENCE, codes[ids].T)
        assert plan.stats.final_tables[0][1] == 839808 * spec.cards[spec.names.index(target)]
    # random evidence patterns on the Alarm structure
    rng = np.random.default_rng(2)
    for _ in range(6):
        vs = rng.choice(spec.n, size=int(rng.integers(2, 9)), replace=False)
        names = [spec.names[v] for v in vs[1:]]
        _check(spec, infer, spec.names[vs[0]], names, codes[vs[1:]].T[:257])
    # partial k-tree, card 3, wide targets excluded
    spec = synth.random_ktree_dag(n=40, card=3, k=4, max_parents=3, seed=4)
    _, infer = install_cpts(spec, DEV)
    codes = synth.sample_forward_numpy(spec, 22, 0, 515)
    for _ in range(8):
        vs = rng.choice(spec.n, size=int(rng.integers(1, 8)), replace=False)
        _check(spec, infer, spec.names[vs[0]], [spec.names[v] for v in vs[1:]], codes[vs[1:]].T)


def _all_configurations(cards):
    """Every configuration of variables with cardinalities ``cards``, row-major (last fastest): int64 [prod, len]."""
    grids = np.indices(cards).reshape(len(cards), -1)
    return np.ascontiguousarray(grids.T)


def _oracle_chunked(net, target, ids, ev, dtype, chunk=1 << 16):
    return np.concatenate([O.ve_posterior(net, target, ids, ev[s: s + chunk], dtype=dtype) for s in range(0, ev.shape[0], chunk)])


def test_alarm_compiled_tables_over_every_evidence_configuration():
    """BASELINE.json configs[2]: the compiled table IS the answer of every row, so it is checked whole -- all 839,808
    configurations of the 12 evidence variables, for the four targets, single plans and the fused (interleaved) launch,
    against the fp64 textbook-VE oracle; plus Asia's 16 configurations against fp64 enumeration."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.alarm()
    _, infer = install_cpts(spec, DEV)
    net = _net(spec)
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    ev = _all_configurations([spec.cards[i] for i in ids])
    assert ev.shape[0] == 839808
    dev_ev = _codes_matrix(ev)
    fused = infer.fused_plan(synth.ALARM_TARGETS, synth.ALARM_EVIDENCE).run_codes(dev_ev, ev.shape[0])
    worst = 0.0
    for tg, fo in zip(synth.ALARM_TARGETS, fused):
        got = infer.plan(tg, synth.ALARM_EVIDENCE).run_codes(dev_ev, ev.shape[0])
        assert torch.equal(got, fo)
        want = _oracle_chunked(net, spec.names.index(tg), ids, ev, torch.float64)
        got = got.cpu().numpy()
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)
        worst = max(worst, float(np.max(np.abs(got - want) / np.maximum(want, 1e-30))))
    assert worst < RTOL
    spec = synth.asia()
    _, infer = install_cpts(spec, DEV)
    names = ["asia", "smoke", "xray", "dysp"]
    ev = _all_configurations([2, 2, 2, 2])
    for tg in ("lung", "tub", "bronc"):
        got = infer.plan(tg, names).run_codes(_codes_matrix(ev), 16).cpu().numpy()
        truth = O.enumerate_posterior(_net(spec), spec.names.index(tg), [spec.names.index(e) for e in names], ev)
        np.testing.assert_allclose(got, truth, rtol=RTOL, atol=1e-30)


def test_config4_ktree200_tables_on_a_stratified_sample():
    """BASELINE.json configs[3], query half: the 8 bench patterns (4^10 = 1,048,576 evidence configurations each) on
    32,768 configurations drawn UNIFORMLY from the configuration space -- not from the joint, so rare configurations are
    covered like common ones -- against the fp64 oracle (the CPU oracle eliminates ~190 hidden variables per row:
    ~15,000 rows/s, which bounds the sample), under the default planner and under an L2-sized merge budget."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import bind_inference, install_cpts

    spec = synth.random_ktree_dag()
    tables, infer = install_cpts(spec, DEV)
    small = bind_inference(tables, merge_budget_cells=1 << 16)
    net = _net(spec)
    rng = np.random.default_rng(1240)
    cfg = np.random.default_rng(99)
    n = 1 << 15
    for _ in range(8):
        vs = [int(v) for v in rng.choice(spec.n, size=11, replace=False)]
        ev = cfg.integers(0, 4, size=(n, 10))
        names = [spec.names[v] for v in vs[1:]]
        want = _oracle_chunked(net, vs[0], vs[1:], ev, torch.float64, chunk=4096)
        for eng in (infer, small):
            got = eng.plan(spec.names[vs[0]], names).run_codes(_codes_matrix(ev), n).cpu().numpy()
            np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)


def test_config4_large_table_path_matches_direct_kernel():
    """Plans whose tables live in global memory (the 16 MB tables of the 200-node patterns) switch to the tile-staged kernel
    with L2 policies from 2^18 rows on: the same rows through the direct kernel (a batch below the threshold) must give
    bit-identical posteriors, for a ragged row count."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts, sample_network

    spec = synth.random_ktree_dag()
    tables, infer = install_cpts(spec, DEV)
    rng = np.random.default_rng(1240)
    n = (1 << 18) + 37
    full = sample_network(spec, seed=5, first=0, n=n, device=DEV, tables=tables)
    for _ in range(2):
        vs = [int(v) for v in rng.choice(spec.n, size=11, replace=False)]
        plan = infer.plan(spec.names[vs[0]], [spec.names[v] for v in vs[1:]])
        ev = full[vs[1:]].contiguous()
        big = plan.run_codes(ev, n)                                  # tile-staged kernel
        m = 1 << 17
        small = plan.run_codes(ev, m)                                # direct kernel on the first 2^17 rows
        assert torch.equal(big[:m], small)
        start = (1 << 18) - 4096                                     # 16-byte aligned view of the ragged end
        tail = plan.run_codes(ev[:, start:], n - start)
        assert torch.equal(big[start:], tail)
        assert float((big.sum(1) - 1).abs().max()) < 1e-5


def test_random_dags_against_enumeration():
    """Seeded sweep over 40 random small DAGs (5-10 variables, cardinalities 2-4, up to 3 parents, a third of the CPT rows
    made deterministic so that zero-probability evidence occurs): random target / evidence / intervention sets against fp64
    full enumeration (O3), through gather plans, the per-row executor and the log-space schedule."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import bind_inference, install_cpts
    from continuousbayesiannetwork_b200.ve import PlanTooLarge

    rng = np.random.default_rng(2024)
    for trial in range(40):
        n = int(rng.integers(5, 11))
        cards = [int(c) for c in rng.integers(2, 5, size=n)]
        parents = [sorted(int(p) for p in rng.choice(i, size=min(i, int(rng.integers(0, 4))), replace=False)) if i else [] for i in range(n)]
        names = [f"v{i}" for i in range(n)]
        cpts = synth._dirichlet_cpts(rng, cards, parents, 0.7)
        for i, c in enumerate(cpts):                                  # deterministic rows: exact zeros in the CPTs
            flat = c.reshape(-1, cards[i])
            for r in range(flat.shape[0]):
                if rng.random() < 0.33:
                    flat[r] = np.eye(cards[i])[int(rng.integers(0, cards[i]))]
        spec = synth.NetSpec(names, cards, parents, cpts)
        net = _net(spec)
        tables, infer = install_cpts(spec, DEV)
        engines = [infer, bind_inference(tables, log_space=True, merge_budget_cells=8), bind_inference(tables, table_budget_cells=1)]
        for _ in range(3):
            k = int(rng.integers(0, n))
            vs = [int(v) for v in rng.choice(n, size=k + 1, replace=False)]
            target, ev_ids = vs[0], vs[1:]
            ev = np.stack([rng.integers(0, cards[v], size=53) for v in ev_ids], axis=1) if ev_ids else np.zeros((1, 0), dtype=np.int64)
            truth = O.enumerate_posterior(net, target, ev_ids, ev)
            n_checked = 0
            for eng in engines:
                try:
                    plan = eng.plan(names[target], [names[v] for v in ev_ids])
                except PlanTooLarge:                                  # the 1-cell table budget cannot merge evidence-only finals
                    continue
                got = plan.run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
                if plan.stats.support_unchecked:
                    # the 1-cell budget could not tabulate the support of a component that does not contain the target (the
                    # plan says so): rows whose evidence has probability zero are then not recognised -- compare the others
                    keep = truth.sum(1) > 0
                    got, want = got[keep], truth[keep]
                else:
                    want = truth
                np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-12, err_msg=f"trial {trial} target {target} evidence {ev_ids}")
                n_checked += 1
            assert n_checked >= 2


def test_config4_ktree200_patterns():
    """BASELINE.json configs[3], query half: 200-node card-4 partial 8-tree, random target + 10 random evidence
    variables (the 8 patterns bench.py times), against the fp32 and fp64 oracle."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.random_ktree_dag()
    _, infer = install_cpts(spec, DEV)
    codes = synth.sample_forward_numpy(spec, 1241, 0, 130)
    rng = np.random.default_rng(1240)
    for _ in range(8):
        vs = [int(v) for v in rng.choice(spec.n, size=11, replace=False)]
        plan, _ = _check(spec, infer, spec.names[vs[0]], [spec.names[v] for v in vs[1:]], codes[vs[1:]].T)
        assert plan.stats.per_row_hidden == 0 and plan.stats.max_table_cells <= 1 << 28


def test_config5_layered_dag_shallow_patterns():
    """BASELINE.json configs[4]: the 1000-node layered DAG.  Uniformly random patterns have an induced width far beyond
    exact inference (test_host_logic.py::test_planner_budget_and_layered_stress); patterns whose target and evidence
    lie in the first five layers are tractable and exercise both executors (gather plans and per-row elimination)."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts
    from continuousbayesiannetwork_b200.ve import PlanTooLarge, RowPlan

    spec = synth.layered_dag()
    _, infer = install_cpts(spec, DEV)
    codes = synth.sample_forward_numpy(spec, 1243, 0, 48)
    rng = np.random.default_rng(1242)
    kinds = set()
    done = 0
    for p in range(64):
        k = int(rng.integers(5, 51))
        vs = [int(v) for v in rng.choice(5 * 50, size=k + 1, replace=False)]
        if p % 8 not in (0, 5):           # a sample of the 64 patterns (the oracle takes seconds per pattern)
            continue
        try:
            plan, _ = _check(spec, infer, spec.names[vs[0]], [spec.names[v] for v in vs[1:]], codes[vs[1:]].T, truth64=False)
        except PlanTooLarge:
            continue
        kinds.add(isinstance(plan, RowPlan))
        done += 1
    assert done >= 12 and kinds == {True, False}


def test_contraction_and_rescale_kernels_on_large_outputs():
    """``cbn_factor_contract`` against torch.einsum on outputs of 2^28+ cells with 10 axes of mixed cardinalities: the
    index decoding (multiply + shift per axis) must stay exact where the running remainder is close to 2^31."""
    from continuousbayesiannetwork_b200.tables import DiscreteTables
    from continuousbayesiannetwork_b200.ve import Factor, VECompiler, _Pass

    cards = [7, 3, 8, 5, 2, 6, 4, 255, 9, 3, 2]                     # variables 0..10; variable 10 is summed out
    names = [f"v{i}" for i in range(len(cards))]
    t = DiscreteTables(names, {}, device=DEV)
    t.set_cards(cards)
    c = VECompiler(t)
    g = torch.Generator(device=DEV); g.manual_seed(4)
    a_scope, b_scope = [0, 2, 4, 7, 10], [1, 3, 5, 6, 8, 9, 10]
    A = torch.rand([cards[v] for v in a_scope], device=DEV, generator=g)
    B = torch.rand([cards[v] for v in b_scope], device=DEV, generator=g)
    out_scope = [7, 0, 1, 2, 3, 4, 5, 6, 8, 9]                      # 277,603,200 cells (1.1 GB of float32)
    n_out = int(np.prod([cards[v] for v in out_scope]))
    assert 1 << 28 < n_out < 1 << 31
    got = c._contract([Factor(a_scope, A.reshape(-1)), Factor(b_scope, B.reshape(-1))], out_scope, 10,   # the raw kernel
                      _Pass([], None, dry=False, log_space=False, rescale=False)).tensor
    letters = "abcdefghijk"
    expr = "".join(letters[v] for v in a_scope) + "," + "".join(letters[v] for v in b_scope) + "->" + "".join(letters[v] for v in out_scope)
    want = torch.einsum(expr, A, B).reshape(-1)
    assert got.numel() == n_out
    # range control: with variable 7 (the slowest output axis) declared an evidence axis, every one of its 255 slices is
    # divided by its own maximum (cbn_factor_rescale) -- bit-equal to the division done by torch
    scaled = c._contract([Factor(a_scope, A.reshape(-1)), Factor(b_scope, B.reshape(-1))], out_scope, 10,
                         _Pass([7], None, dry=False, log_space=False, rescale=True)).tensor
    w2 = want.view(255, -1)
    torch.testing.assert_close(scaled.view(255, -1), w2 * (1.0 / w2.max(dim=1, keepdim=True).values), rtol=1e-6, atol=0)
    del scaled, w2
    torch.testing.assert_close(got, want, rtol=1e-6, atol=0)
    del got, want
    torch.cuda.empty_cache()


def test_empty_and_tiny_batches():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.asia()
    _, infer = install_cpts(spec, DEV)
    names = ["asia", "smoke", "xray", "dysp"]
    ids = [spec.names.index(e) for e in names]
    plan = infer.plan("lung", names)
    fused = infer.fused_plan(["lung", "tub", "bronc"], names)
    empty = torch.zeros((4, 16), dtype=torch.uint8, device=DEV)
    assert tuple(plan.run_codes(empty, 0).shape) == (0, 2)
    assert all(tuple(o.shape) == (0, 2) for o in fused.run_codes(empty, 0))
    assert tuple(plan.run_codes_host(empty.cpu(), 0, torch.empty((0, 2), dtype=torch.float32)).shape) == (0, 2)
    codes = synth.sample_forward_numpy(spec, 77, 0, 7)
    for n in (1, 2, 3, 5, 7):
        ev = codes[ids][:, :n].T
        got = plan.run_codes(_codes_matrix(ev), n).cpu().numpy()
        want = O.ve_posterior(_net(spec), spec.names.index("lung"), ids, ev)
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)
        host = torch.full((n + 1, 2), -1.0, dtype=torch.float32)
        plan.run_codes_host(_codes_matrix(ev).cpu(), n, host)
        assert np.array_equal(host[:n].numpy(), got) and bool((host[n] == -1).all())     # nothing written past n rows


def test_wide_target_and_mixed_cards():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    rng = np.random.default_rng(3)
    names = ["a", "b", "c", "d", "e"]
    cards = [3, 11, 2, 5, 7]
    parents = [[], [0], [0, 1], [1, 2], [3]]
    cpts = synth._dirichlet_cpts(rng, cards, parents, 0.8)
    spec = synth.NetSpec(names, cards, parents, cpts)
    _, infer = install_cpts(spec, DEV)
    codes = synth.sample_forward_numpy(spec, 1, 0, 301)
    for target, ev in (("b", ["e", "a"]), ("b", ["d"]), ("e", ["a"]), ("d", ["e", "a", "c"]), ("a", ["b", "c", "d", "e"])):
        ids = [names.index(e) for e in ev]
        _check(spec, infer, target, ev, codes[ids].T)


def test_zero_probability_and_unseen_evidence_give_zero_rows():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.asia()
    _, infer = install_cpts(spec, DEV)
    # either = lung OR tub is deterministic: evidence either=0, lung=1 has probability 0
    names = ["either", "lung", "xray"]
    ev = np.array([[0, 1, 1], [1, 1, 0], [0, 0, 0], [255, 0, 1], [1, 255, 1], [1, 0, 255]])
    plan = infer.plan("tub", names)
    got = plan.run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
    want = O.ve_posterior(_net(spec), spec.names.index("tub"), [spec.names.index(e) for e in names], ev[:3])
    np.testing.assert_allclose(got[:3], want, rtol=RTOL, atol=1e-30)
    assert np.all(got[0] == 0) and got[1].sum() > 0.99
    assert np.all(got[3] == 0) and np.all(got[4] == 0)
    # xray is d-separated from tub given either: an unseen xray code is never read
    assert got[5].sum() > 0.99
    # zero-probability evidence in a part that is d-separated from the target still zeroes the row (oracle convention)
    names = ["either", "lung", "tub"]
    ev = np.array([[0, 1, 0], [1, 1, 0], [1, 0, 0]])
    got = infer.plan("smoke", names).run_codes(_codes_matrix(ev), 3).cpu().numpy()
    want = O.ve_posterior(_net(spec), spec.names.index("smoke"), [spec.names.index(e) for e in names], ev)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)
    assert np.all(got[0] == 0) and np.all(got[2] == 0)


def test_log_space_schedule_matches_linear_and_oracle():
    """north_star (1): the whole schedule in log space -- log CPTs, factor products as sums, sum-outs as log-sum-exp at
    compile time (cbn_factor_contract with log_space), log tables gathered and pushed through exp(x - max) per row
    (CBN_GATHER_LOG_SPACE) -- against the fp64 oracle, the oracle's own log-space mode and the linear engine, on Asia
    (deterministic OR node: exact zeros = -inf), Alarm (multi-table plans via a small merge budget) and a random DAG with
    zero-probability evidence."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import bind_inference, install_cpts

    spec = synth.asia()
    tables, lin = install_cpts(spec, DEV)
    lg = bind_inference(tables, log_space=True)
    lg_multi = bind_inference(tables, log_space=True, merge_budget_cells=4)
    net = _net(spec)
    rng = np.random.default_rng(12)
    for target, names in (("lung", ["asia", "smoke", "xray", "dysp"]), ("either", ["xray", "asia"]), ("smoke", ["lung", "dysp"]),
                          ("tub", ["either", "xray", "dysp", "smoke"]), ("bronc", [])):
        ev = rng.integers(0, 2, size=(67, len(names)))
        ids = [spec.names.index(e) for e in names]
        want = O.ve_posterior(net, spec.names.index(target), ids, ev, dtype=torch.float64)
        want_log = O.ve_posterior(net, spec.names.index(target), ids, ev, log_space=True)
        for eng in (lg, lg_multi):
            plan = eng.plan(target, names)
            got = plan.run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
            np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)
            np.testing.assert_allclose(got, want_log, rtol=2e-5, atol=1e-30)
        np.testing.assert_allclose(lin.plan(target, names).run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy(), got, rtol=RTOL, atol=1e-30)
    assert lg_multi.plan("lung", ["asia", "smoke", "xray", "dysp"]).log_space            # several log tables, LSE epilogue
    assert not lg.plan("lung", ["asia", "smoke", "xray", "dysp"]).log_space              # one table: normalised to linear at compile time
    # Alarm: fused launch of multi-table log plans, and MAP through the log epilogue
    spec = synth.alarm()
    tables, lin = install_cpts(spec, DEV)
    lg = bind_inference(tables, log_space=True, merge_budget_cells=1 << 10)
    codes = synth.sample_forward_numpy(spec, 21, 0, 1537)
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    ev = codes[ids].T
    dev_ev = _codes_matrix(ev)
    fused = lg.fused_plan(synth.ALARM_TARGETS, synth.ALARM_EVIDENCE).run_codes(dev_ev, ev.shape[0])
    for tg, fo in zip(synth.ALARM_TARGETS, fused):
        plan = lg.plan(tg, synth.ALARM_EVIDENCE)
        assert plan.log_space and len(plan.finals) > 1
        want = O.ve_posterior(_net(spec), spec.names.index(tg), ids, ev, dtype=torch.float64)
        np.testing.assert_allclose(fo.cpu().numpy(), want, rtol=RTOL, atol=1e-30)
        m = plan.run_codes_map(dev_ev, ev.shape[0]).cpu().numpy()
        assert np.array_equal(m, want.argmax(1).astype(np.float32))
    # zero-probability evidence in log space: all -inf rows become all-zero rows
    names = ["a", "b", "c"]
    cpts = [np.array([0.5, 0.5]), np.array([[1.0, 0.0], [0.3, 0.7]]), np.array([[0.2, 0.8], [0.0, 1.0]])]
    spec = synth.NetSpec(names, [2, 2, 2], [[], [0], [1]], cpts)
    tables, _ = install_cpts(spec, DEV)
    lg = bind_inference(tables, log_space=True, merge_budget_cells=2)
    ev = np.array([[0, 0], [1, 0], [1, 1], [0, 1]])                 # (b, c): c=0 given b=1 has probability 0
    want = O.ve_posterior(_net(spec), 0, [1, 2], ev, dtype=torch.float64)
    got = lg.plan("a", ["b", "c"]).run_codes(_codes_matrix(ev), 4).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)
    assert got[1].sum() == 0.0


def test_long_products_of_small_likelihoods_do_not_underflow():
    """Range control of the linear-space path (the alternative to log space): a binary cause with 22 observed binary
    effects whose observed values have likelihoods of 1e-3 / 3e-3 -- the all-ones configuration has probability ~1e-60,
    far below the fp32 range, and without rescaling the compiled table holds zeros there.  With every evidence slice
    divided by its maximum after each contraction (cbn_factor_rescale) and the gather product pulled back every fourth
    factor, posteriors stay within 1e-5 of the fp64 oracle: as one merged table, as 16 unmerged tables, through the per-row
    executor (linear and log space), and on a 300-node chain with evidence on every 7th node."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import bind_inference, install_cpts

    n_e = 22
    names = ["T"] + [f"e{i:02d}" for i in range(n_e)]
    cards = [2] * (n_e + 1)
    parents = [[]] + [[0]] * n_e
    rng = np.random.default_rng(8)
    cpts = [np.array([0.5, 0.5])]
    for i in range(n_e):
        a, b = 1e-3 * (1 + rng.random()), 3e-3 * (1 + rng.random())
        cpts.append(np.array([[1 - a, a], [1 - b, b]]))
    spec = synth.NetSpec(names, cards, parents, cpts)
    net = _net(spec)
    ev = np.concatenate([np.ones((3, n_e), dtype=np.int64), rng.integers(0, 2, size=(61, n_e)), np.zeros((1, n_e), dtype=np.int64)])
    ev[1, ::2] = 0
    want = O.ve_posterior(net, 0, list(range(1, n_e + 1)), ev, dtype=torch.float64)
    assert want[0, 0] < 1e-9 and want[0].sum() > 0.999           # the oracle itself resolves the tiny posterior
    tables, infer = install_cpts(spec, DEV)
    variants = {"merged": infer, "unmerged": bind_inference(tables, merge_budget_cells=1 << 8),
                "log_space_merged": bind_inference(tables, log_space=True),
                "log_space_unmerged": bind_inference(tables, log_space=True, merge_budget_cells=1 << 8)}
    for label, eng in variants.items():
        got = eng.plan("T", names[1:]).run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30, err_msg=label)
    # without range control the same query underflows (this is what the rescaling is for)
    raw = bind_inference(tables, rescale=False).plan("T", names[1:]).run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
    assert raw[0].sum() == 0.0
    # hidden effects in between: T -> h_i -> e_i, the h_i are eliminated at compile time
    names2 = ["T"] + [f"h{i:02d}" for i in range(n_e)] + [f"e{i:02d}" for i in range(n_e)]
    parents2 = [[]] + [[0]] * n_e + [[1 + i] for i in range(n_e)]
    cpts2 = [np.array([0.5, 0.5])] + [np.array([[0.9, 0.1], [0.2, 0.8]])] * n_e + cpts[1:]
    spec2 = synth.NetSpec(names2, [2] * len(names2), parents2, cpts2)
    tables2, infer2 = install_cpts(spec2, DEV)
    ids2 = list(range(1 + n_e, 1 + 2 * n_e))
    want2 = O.ve_posterior(_net(spec2), 0, ids2, ev, dtype=torch.float64)
    from continuousbayesiannetwork_b200.ve import RowPlan

    for label, eng in {"compile-time": infer2,
                       "per_row": bind_inference(tables2, table_budget_cells=1),            # every h_i is left to the per-row executor
                       "per_row_log": bind_inference(tables2, table_budget_cells=1, log_space=True)}.items():
        plan2 = eng.plan("T", names2[1 + n_e:])
        assert isinstance(plan2, RowPlan) == label.startswith("per_row")
        got2 = plan2.run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
        np.testing.assert_allclose(got2, want2, rtol=RTOL, atol=1e-30, err_msg=label)
    # a deep chain: 300 ternary nodes, evidence on every 7th, target in the middle
    n = 300
    names3 = [f"x{i:03d}" for i in range(n)]
    parents3 = [[]] + [[i - 1] for i in range(1, n)]
    cpts3 = synth._dirichlet_cpts(np.random.default_rng(9), [3] * n, parents3, 0.3)
    spec3 = synth.NetSpec(names3, [3] * n, parents3, cpts3)
    _, infer3 = install_cpts(spec3, DEV)
    ev_ids = [i for i in range(0, n, 7) if i != 147]
    codes3 = synth.sample_forward_numpy(spec3, 3, 0, 257)
    want3 = O.ve_posterior(_net(spec3), 147, ev_ids, codes3[ev_ids].T, dtype=torch.float64)
    got3 = infer3.plan("x147", [names3[i] for i in ev_ids]).run_codes(_codes_matrix(codes3[ev_ids].T), 257).cpu().numpy()
    np.testing.assert_allclose(got3, want3, rtol=RTOL, atol=1e-30)


def test_do_intervention_is_graph_surgery():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.asia()
    _, infer = install_cpts(spec, DEV)
    ev = np.array([[1, 1], [0, 1], [1, 0]])
    got = infer.plan("smoke", ["lung", "dysp"], do=["lung"]).run_codes(_codes_matrix(ev), 3).cpu().numpy()
    # mutilated network: lung has no parents (its CPT is irrelevant once it is clamped)
    cut = synth.asia()
    li = cut.names.index("lung")
    cut.parents[li] = []
    cut.cpts[li] = np.array([0.5, 0.5])
    want = O.ve_posterior(_net(cut), cut.names.index("smoke"), [li, cut.names.index("dysp")], ev)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)
    seen = infer.plan("smoke", ["lung", "dysp"]).run_codes(_codes_matrix(ev), 3).cpu().numpy()
    assert np.abs(seen - got).max() > 1e-2           # observing lung is not the same as setting it


def test_f32_and_host_entry_points_agree_with_codes():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.alarm()
    t, infer = install_cpts(spec, DEV)
    n = 3 * (1 << 20) + 77                           # several host chunks, ragged tail
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    rng = np.random.default_rng(5)
    ev = np.stack([rng.integers(0, spec.cards[i], size=n) for i in ids], axis=1).astype(np.uint8)
    m = _codes_matrix(ev)
    plan = infer.plan("LVFAILURE", synth.ALARM_EVIDENCE)
    a = plan.run_codes(m, n)
    cols = [m[i, :n].to(torch.float32) for i in range(len(ids))]
    b = plan.run_f32(cols, n)
    assert torch.equal(a, b)
    host_in = m.cpu()
    out = torch.empty((n, plan.card_t), dtype=torch.float32)
    plan.run_codes_host(host_in, n, out)
    assert torch.equal(a.cpu(), out)
    pin_in, pin_out = host_in.pin_memory(), torch.empty((n, plan.card_t), dtype=torch.float32).pin_memory()
    plan.run_codes_host(pin_in, n, pin_out)
    assert torch.equal(a.cpu(), pin_out)
    # full-size properties: rows are distributions; identical evidence -> identical posterior
    s = a.sum(1)
    assert float((s - 1).abs().max()) < 1e-5
    key = torch.zeros(n, dtype=torch.int64, device=DEV)
    for i in range(len(ids)):
        key = key * 4 + m[i, :n].long()
    _, inv = torch.unique(key, return_inverse=True)
    first = torch.full((int(inv.max()) + 1,), n, dtype=torch.int64, device=DEV).scatter_reduce(0, inv, torch.arange(n, device=DEV), "amin")
    assert torch.equal(a, a[first[inv]])


def test_compact_host_output_round_trips():
    """CBN_HOST_OUT_DROP_LAST: card_t - 1 values per row over PCIe, -1 flags an all-zero row; expanding restores the full
    posteriors (the last value to fp32 rounding), for binary (Asia, fused) and 4-valued targets, unseen evidence included."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts, sample_network
    from continuousbayesiannetwork_b200.ve import FusedPlan, expand_compact

    for spec, evn, tgs, n in ((synth.asia(), ["asia", "smoke", "xray", "dysp"], ["lung", "tub", "bronc"], 300_007),
                              (synth.random_ktree_dag(n=30, card=4, k=4, max_parents=3, seed=6), None, None, 70_001)):
        t, infer = install_cpts(spec, DEV)
        if evn is None:
            evn, tgs = [spec.names[i] for i in (3, 7, 11, 19)], [spec.names[25]]
        ids = [spec.names.index(e) for e in evn]
        ev = sample_network(spec, seed=41, first=0, n=n, device=DEV, tables=t)[ids].contiguous()
        ev[0, 5] = 255                                               # an unseen code: all-zero row
        fused = FusedPlan([infer.plan(tg, evn) for tg in tgs])
        full = [o.cpu() for o in fused.run_codes(ev, n)]
        ct = fused.card_t
        host = [torch.full((n, ct - 1), 7.0) for _ in tgs]
        fused.run_codes_host(ev.cpu(), n, host, compact=True)
        for f, c in zip(full, host):
            assert c[5, 0] == -1 and float(f[5].sum()) == 0.0
            assert torch.equal(c[:, : ct - 1][c[:, 0] >= 0], f[:, : ct - 1][c[:, 0] >= 0])        # the values that travel are bit-equal
            torch.testing.assert_close(expand_compact(c), f, rtol=0, atol=2e-7)


def test_fused_multi_target_launch_matches_single_plans():
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    for spec, ev_names, targets in ((synth.asia(), ["asia", "smoke", "xray", "dysp"], ["lung", "tub", "bronc"]),
                                    (synth.alarm(), synth.ALARM_EVIDENCE, synth.ALARM_TARGETS)):
        _, infer = install_cpts(spec, DEV)
        n = 100_003
        ids = [spec.names.index(e) for e in ev_names]
        rng = np.random.default_rng(8)
        ev = np.stack([rng.integers(0, spec.cards[i], size=n) for i in ids], axis=1)
        ev[7, 0] = 255                                  # an unseen code zeroes every target's row
        m = _codes_matrix(ev)
        fused = infer.fused_plan(targets, ev_names)
        outs = fused.run_codes(m, n)
        assert fused.n_out == len(targets)
        for t, o in zip(targets, outs):
            single = infer.plan(t, ev_names).run_codes(m, n)
            assert torch.equal(single, o), t
            assert bool((o[7] == 0).all())
        host = fused.run_codes_host(m.cpu(), n, [torch.empty((n, 2), dtype=torch.float32) for _ in targets])
        assert all(torch.equal(h, o.cpu()) for h, o in zip(host, outs))
    # mixed target cardinalities cannot be fused
    spec = synth.alarm()
    _, infer = install_cpts(spec, DEV)
    with pytest.raises(ValueError):
        infer.fused_plan(["HYPOVOLEMIA", "VENTLUNG"], synth.ALARM_EVIDENCE)


def test_tile_staged_kernel_matches_direct_kernel_on_large_batches():
    """Batches of >= 2^21 rows run through the tile-staged kernel (bulk async copies of the evidence tiles); the
    same rows answered in smaller calls use the direct kernel: the posteriors must be bit-identical, including the
    ragged last tile, an unseen code and a slice of the batch checked against the oracle."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts

    spec = synth.alarm()
    _, infer = install_cpts(spec, DEV)
    n = (1 << 22) + 1027
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    rng = np.random.default_rng(9)
    ev = np.stack([rng.integers(0, spec.cards[i], size=n) for i in ids], axis=1).astype(np.uint8)
    ev[n - 2, 4] = 255
    ev[12345, 0] = 255
    m = _codes_matrix(ev)
    half = 1 << 20
    for plan in (infer.fused_plan(synth.ALARM_TARGETS, synth.ALARM_EVIDENCE), infer.plan("VENTLUNG", synth.ALARM_EVIDENCE),
                 infer.plan("LVFAILURE", synth.ALARM_EVIDENCE[:5])):
        multi = hasattr(plan, "n_out")
        big = plan.run_codes(m, n)
        big = big if multi else [big]
        for o in big:
            assert bool((o[n - 2] == 0).all()) and bool((o[12345] == 0).all())
        for s0 in range(0, n, half):
            cnt = min(half, n - s0)
            part = plan.run_codes(m[:, s0:], cnt)            # s0 is a multiple of 16: alignment is preserved
            part = part if multi else [part]
            for o, q in zip(big, part):
                assert torch.equal(o[s0:s0 + cnt], q)
    net = _net(spec)
    got = infer.plan("VENTLUNG", synth.ALARM_EVIDENCE).run_codes(m, n)[-600:].cpu().numpy()
    ok = np.ones(600, bool); ok[600 - 2] = False
    want = O.ve_posterior(net, spec.names.index("VENTLUNG"), ids, ev[-600:][ok])
    np.testing.assert_allclose(got[ok], want, rtol=RTOL, atol=1e-30)
    # from ten 2048-row tiles per resident CTA on, the interleaved multi-target table runs two quads per thread and tile:
    # a ragged batch of that size (the rows above, repeated) against the same rows in 1M-row calls of the direct kernel
    reps = 3
    n2 = reps * n - 517
    m2 = _codes_matrix(np.concatenate([ev] * reps)[:n2])
    fused = infer.fused_plan(synth.ALARM_TARGETS, synth.ALARM_EVIDENCE)
    assert n2 // 2048 >= torch.cuda.get_device_properties(0).multi_processor_count * 40
    big = fused.run_codes(m2, n2)
    for s0 in range(0, n2, half):
        cnt = min(half, n2 - s0)
        for o, q in zip(big, fused.run_codes(m2[:, s0:], cnt)):
            assert torch.equal(o[s0:s0 + cnt], q)
    for o in big:
        assert bool((o[12345] == 0).all()) and bool((o[n + 12345] == 0).all()) and bool((o[n + n - 2] == 0).all())


def test_per_row_executor_matches_oracle():
    """A small table budget forces the per-row elimination schedule (linear-rescaled and log-space)."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import bind_inference, tables_from_spec
    from continuousbayesiannetwork_b200.ve import RowPlan

    spec = synth.alarm()
    codes = synth.sample_forward_numpy(spec, 31, 0, 1031)
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    ev = codes[ids].T.copy()
    ev[5, 3] = 255                                              # unseen value -> zero row
    net = _net(spec)
    # unit = the planner lays every factor out for the step that consumes it (the executor's unrolled step bodies);
    # without it the schedule keeps the tables' own axis order and runs on the strided bodies
    for log_space, unit in ((False, True), (True, True), (False, False), (True, False)):
        t = tables_from_spec(spec, DEV)
        t.set_cond_tables(spec.cpts)
        infer = bind_inference(t, table_budget_cells=1 << 10, log_space=log_space, row_unit_layout=unit)
        for target in ("HYPOVOLEMIA", "VENTLUNG", "CATECHOL"):
            plan = infer.plan(target, synth.ALARM_EVIDENCE)
            assert isinstance(plan, RowPlan) and plan.stats.per_row_hidden > 0
            sums = [st for st in infer.compiler.last_row_schedule["steps"] if st["sum_card"] > 1]
            assert all(s == 1 for st in sums for s in st["sum_stride"]) == unit
            got = plan.run_codes(_codes_matrix(ev), ev.shape[0]).cpu().numpy()
            ok = np.ones(ev.shape[0], bool); ok[5] = False
            want = O.ve_posterior(net, spec.names.index(target), ids, ev[ok], dtype=torch.float64)
            np.testing.assert_allclose(got[ok], want, rtol=2e-5 if log_space else RTOL, atol=1e-30)
            assert np.all(got[5] == 0)
            # the float-valued entry point encodes and runs the same plan
            cols = [torch.tensor(ev[:, i].astype(np.float32), device=DEV) for i in range(len(ids))]
            cols[3][5] = 1234.0
            got32 = plan.run_f32(cols, ev.shape[0]).cpu().numpy()
            assert np.array_equal(got32, got)
    # the schedule is host data that the library range-checks: an offset that leaves its factor is refused at plan creation
    sch = infer.compiler.last_row_schedule
    for bad_value in (-1, 1 << 28):
        bad = plan.offsets.copy()
        bad[len(bad) // 2] = bad_value
        with pytest.raises(ValueError, match="leaves the factor"):
            RowPlan(t, plan.target, plan.evidence, plan.card_t, plan.inputs, sch["steps"], bad, plan.stats, plan.log_space)
    # naive-Bayes shape: one hidden cause with many observed children: the boundary (3^40 / 3^24) cannot be tabulated.
    # 40 children -> warp-per-row kernel, 24 children -> a short schedule, the one-thread-per-row kernel; both arithmetic modes
    for n_child in (40, 24):
        rng = np.random.default_rng(12)
        names = ["cause", "t"] + [f"c{i:02d}" for i in range(n_child)]
        cards = [4, 3] + [3] * n_child
        parents = [[], [0]] + [[0]] * n_child
        spec = synth.NetSpec(names, cards, parents, synth._dirichlet_cpts(rng, cards, parents, 0.5))
        codes = synth.sample_forward_numpy(spec, 2, 0, 513)
        evn = names[2:]
        want = O.ve_posterior(_net(spec), 1, list(range(2, 2 + n_child)), codes[2:].T, dtype=torch.float64)
        ev = codes[2:].T.copy()
        ev[100, 7] = 255
        for log_space in (False, True):
            t = tables_from_spec(spec, DEV)
            t.set_cond_tables(spec.cpts)
            infer = bind_inference(t, table_budget_cells=1 << 16, log_space=log_space)
            plan = infer.plan("t", evn)
            assert isinstance(plan, RowPlan) and (plan.stats.per_row_madds <= 320) == (n_child == 24)
            got = plan.run_codes(_codes_matrix(ev), 513).cpu().numpy()
            ok = np.ones(513, bool); ok[100] = False
            np.testing.assert_allclose(got[ok], want[ok], rtol=2e-5 if log_space else RTOL, atol=1e-30)
            assert np.all(got[100] == 0)


def test_fit_then_infer_end_to_end_on_fitted_tables():
    """Config-2 shape end to end: sample -> count -> CPTs -> compile -> query, checked against the oracle
    run on the oracle's own tables (counts bit-exact, so the CPTs agree to the last bit of the division)."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import fit_network_from_codes, sample_network

    spec = synth.asia()
    n = 500_000
    codes = sample_network(spec, seed=3, first=0, n=n, device=DEV)
    ref = synth.sample_forward_numpy(spec, 3, 0, n)
    t, infer = fit_network_from_codes(spec, codes, n, DEV)
    fitted = [O.cpt_from_counts(O.dense_counts(ref, spec.parents[i] + [i], spec.cards), n)[1] for i in range(spec.n)]
    net = O.DiscreteNet(spec.cards, spec.parents, fitted)
    ev_names = ["asia", "smoke", "xray", "dysp"]
    ids = [spec.names.index(e) for e in ev_names]
    ev = ref[ids][:, :4096].T
    for target in ("lung", "tub", "bronc"):
        got = infer.plan(target, ev_names).run_codes(_codes_matrix(ev), 4096).cpu().numpy()
        want = O.ve_posterior(net, spec.names.index(target), ids, ev)
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=1e-30)


def test_full_size_query_properties():
    """BASELINE.json sizes (16,777,216 Alarm rows, 4 fused targets; 1,048,576 Asia rows, 3 fused targets): every posterior
    row is a distribution, rows with identical evidence have bit-identical posteriors, the fused launch equals the
    single-target plans, and a permutation of the rows permutes the posteriors."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts, sample_network

    for spec, evn, targets, n in ((synth.alarm(), synth.ALARM_EVIDENCE, synth.ALARM_TARGETS, 1 << 24),
                                  (synth.asia(), ["asia", "smoke", "xray", "dysp"], ["lung", "tub", "bronc"], 1 << 20)):
        t, infer = install_cpts(spec, DEV)
        ids = [spec.names.index(e) for e in evn]
        ev = sample_network(spec, seed=31, first=0, n=n, device=DEV, tables=t)[ids].contiguous()
        fused = infer.fused_plan(targets, evn)
        outs = fused.run_codes(ev, n)
        key = torch.zeros(n, dtype=torch.int64, device=DEV)
        for i, v in enumerate(ids):
            key = key * spec.cards[v] + ev[i, :n].long()
        _, inv = torch.unique(key, return_inverse=True)
        first = torch.full((int(inv.max()) + 1,), n, dtype=torch.int64, device=DEV).scatter_reduce(0, inv, torch.arange(n, device=DEV), "amin")
        perm = torch.randperm(n, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
        ev_p = ev[:, perm].contiguous()
        outs_p = fused.run_codes(ev_p, n)
        for tg, o, op in zip(targets, outs, outs_p):
            assert float((o.sum(1) - 1).abs().max()) < 1e-5
            assert torch.equal(o, o[first[inv]])                                   # same evidence -> same posterior
            assert torch.equal(op, o[perm])                                        # row order does not matter
            assert torch.equal(infer.plan(tg, evn).run_codes(ev, n), o)            # fused == single
        del outs, outs_p, ev, ev_p, key, inv, first, perm
        torch.cuda.empty_cache()
