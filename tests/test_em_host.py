"""EM without a GPU: family grouping and chain order, the plans and launches of the benchmark's E-steps, the chain budget,
the fp64 EM oracle's own properties, and the ABI of the accumulation kernel."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import em_oracle as EO  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fams(parents):
    return [list(ps) + [v] for v, ps in enumerate(parents)]


def test_latent_class_is_one_group_of_every_family():
    from continuousbayesiannetwork_b200 import em

    _, cards, parents, _ = EO.latent_class()
    sch = em.schedule(cards, _fams(parents), [0])
    assert [(g.hidden, g.families) for g in sch["groups"]] == [([0], list(range(21)))]
    assert (sch["compiles"], sch["gathers"], sch["ess_launches"], sch["floats_per_row"]) == (2, 1, 1, 4)


def test_chain_order_is_increasing_cardinality_then_id():
    from continuousbayesiannetwork_b200 import em

    cards = [4, 2, 3, 2]
    parents = [[], [], [], [0, 1, 2]]
    groups = em.plan_groups(cards, _fams(parents), [0, 1, 2, 3])
    assert [(g.hidden, g.families) for g in groups] == [([0], [0]), ([1], [1]), ([1, 3, 2, 0], [3]), ([2], [2])]
    g = groups[2]
    assert g.hidden == [1, 3, 2, 0]
    assert [g.prefix_configs(cards, j) for j in range(4)] == [1, 2, 4, 12]
    assert em.chain_floats(g.hidden, cards) == 2 + 4 + 12 + 48


def test_hmm_groups_share_chain_plans():
    from continuousbayesiannetwork_b200 import em

    _, cards, parents, _ = EO.hmm(steps=6)
    sch = em.schedule(cards, _fams(parents), range(6))
    hs = sorted(tuple(g.hidden) for g in sch["groups"])
    assert hs == [(0,), (0, 1), (1,), (1, 2), (2,), (2, 3), (3,), (3, 4), (4,), (4, 5), (5,)]
    # (S_t) and the first step of (S_t, S_t+1) are the same plan: 6 + 5 distinct chain steps, + log P(e)
    assert sch["compiles"] == 6 + 5 + 1
    assert sch["gathers"] == 6 + 5 * (1 + 3)


def test_bench_workload_schedules():
    """Plans and launches per E-step of the three workloads of tools/bench_em.py."""
    from continuousbayesiannetwork_b200 import em, synth

    spec = synth.alarm()
    fams = _fams(spec.parents)
    targets = [spec.names.index(n) for n in synth.ALARM_TARGETS]
    sch = em.schedule(spec.cards, fams, targets)
    # HYPOVOLEMIA (3), LVFAILURE (5), KINKEDTUBE (16), PULMEMBOLUS (22): LVEDVOLUME and STROKEVOLUME have two of them
    assert [(g.hidden, g.families) for g in sch["groups"]] == [([3], [3]), ([3, 5], [4, 6]), ([5], [0, 5]),
                                                               ([16], [16, 25, 30]), ([22], [21, 22, 23])]
    assert (sch["compiles"], sch["gathers"], sch["ess_launches"], sch["floats_per_row"]) == (6, 7, 5, 6)

    ev = {spec.names.index(n) for n in synth.ALARM_EVIDENCE}
    hidden = [v for v in range(spec.n) if v not in ev]
    assert len(hidden) == 25
    sch = em.schedule(spec.cards, fams, hidden)
    assert len(sch["groups"]) == 33 and max(len(g.hidden) for g in sch["groups"]) == 5
    assert (sch["compiles"], sch["gathers"], sch["ess_launches"], sch["floats_per_row"]) == (47, 209, 33, 162)


def test_chain_budget_raises_plan_too_large():
    from continuousbayesiannetwork_b200 import em
    from continuousbayesiannetwork_b200.ve import PlanTooLarge

    cards = [16, 16, 16, 2]
    parents = [[], [], [], [0, 1, 2]]
    assert em.chain_floats([3, 0, 1, 2], cards) == 2 + 32 + 512 + 8192
    with pytest.raises(PlanTooLarge, match="8738 floats"):
        em.plan_groups(cards, _fams(parents), [0, 1, 2, 3])
    assert len(em.plan_groups(cards, _fams(parents), [0, 1, 2, 3], budget_floats=8738)) == 4


def _sample(cards, parents, cpts, n, rng):
    codes = np.zeros((n, len(cards)), np.int64)
    for v in range(len(cards)):         # parents precede children in every test network
        p = np.broadcast_to(np.asarray(cpts[v])[tuple(codes[:, u] for u in parents[v])], (n, cards[v]))
        codes[:, v] = (rng.random((n, 1)) > np.cumsum(p, axis=1)).sum(axis=1).clip(max=cards[v] - 1)
    return codes


def test_oracle_em_never_decreases():
    rng = np.random.default_rng(1)
    for make, hidden in ((lambda: EO.latent_class(n_children=6, seed=2)[1:], [0]), (lambda: EO.hmm(steps=4)[1:], [0, 1, 2, 3])):
        cards, parents, cpts = make()
        codes = _sample(cards, parents, cpts, 2000, rng)
        start = [rng.dirichlet(np.ones(cards[v]), size=int(np.prod([cards[u] for u in parents[v]]))).reshape(np.shape(cpts[v]))
                 for v in range(len(cards))]
        _, hist = EO.em(cards, parents, start, hidden, codes, 15)
        assert all(b >= a - 1e-9 * abs(a) for a, b in zip(hist, hist[1:])), hist


def test_oracle_em_with_complete_data_is_the_mle():
    rng = np.random.default_rng(3)
    cards, parents, cpts = EO.latent_class(n_children=4, seed=4)[1:]
    codes = _sample(cards, parents, cpts, 3000, rng)
    fitted, _ = EO.em(cards, parents, cpts, [], codes, 1)
    for v in range(len(cards)):
        counts = np.zeros(np.shape(cpts[v]))
        np.add.at(counts, tuple(codes[:, u] for u in parents[v]) + (codes[:, v],), 1.0)
        np.testing.assert_allclose(fitted[v], counts / counts.sum(axis=-1, keepdims=True), rtol=0, atol=1e-15)


def test_ess_symbols_and_struct_layout(tmp_path):
    from continuousbayesiannetwork_b200.build import build_native

    build_native()
    from continuousbayesiannetwork_b200 import _native as N

    lib = N.lib()
    for name in ("cbn_ess_plan_create", "cbn_ess_plan_destroy", "cbn_ess_run", "cbn_ess_plan_smem_dests"):
        assert name in N.SIGNATURES and hasattr(lib, name)
    assert lib.cbn_abi_version() == 2
    prog = tmp_path / "ess.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cbn_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %d %d\\n", '
                    'sizeof(cbn_ess_dest), offsetof(cbn_ess_dest, n_cells), offsetof(cbn_ess_dest, n_obs), '
                    'offsetof(cbn_ess_dest, obs_stride), offsetof(cbn_ess_dest, hidden_cell), sizeof(cbn_family), '
                    'CBN_ESS_MAX_DESTS, CBN_ESS_MAX_CONFIGS);return 0;}\n')
    exe = tmp_path / "ess"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    D = N.EssDest
    assert got == [C.sizeof(D), D.n_cells.offset, D.n_obs.offset, D.obs_stride.offset, D.hidden_cell.offset,
                   C.sizeof(N.Family), N.ESS_MAX_DESTS, N.ESS_MAX_CONFIGS]
    assert lib.cbn_ess_run(None, None, None, None, 0, 0, None, None) == N.ERR_INVALID
