"""Posterior sampling without a GPU: the structure of the sum-product elimination with recorded conditionals (dry run),
its limits, the C layout of the sampling steps, the numpy restatement of the counter hash, and the fp64 oracles."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from continuousbayesiannetwork_b200 import synth
from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, VECompiler
from oracle import cbn_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mpe_oracle as MO  # noqa: E402
import psample_oracle as PO  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _compiler(spec, **kw):
    return VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()), **kw)


def _check_decode_order(split, n):
    """Every context of a step is evidence or drawn by an earlier step; every hidden variable is drawn once."""
    E = set(split.evidence)
    done = set()
    for v, scope in split.decode:
        assert v not in E and v not in done and v not in scope
        assert all(u in E or u in done for u in scope), (v, scope)
        done.add(v)
    assert done == set(split.hidden) == set(range(n)) - E


def _threshold_bytes(spec, split):
    return sum(4 * int(np.prod([spec.cards[u] for u in sc])) * (spec.cards[v] - 1) for v, sc in split.decode)


def test_alarm_headline_structure_is_that_of_mpe():
    spec = synth.alarm()
    split = _compiler(spec).compile_posterior_sampler(synth.ALARM_EVIDENCE, dry=True)
    _check_decode_order(split, spec.n)
    mpe = _compiler(spec).compile_mpe(synth.ALARM_EVIDENCE, dry=True)
    assert split.decode == mpe.decode and split.hidden == mpe.hidden and len(split.hidden) == 25
    assert split.stats.final_tables == mpe.stats.final_tables == [((tuple(split.stats.final_tables[0][0])), 839808)]
    assert sorted(split.observed_families) == sorted(mpe.observed_families)
    assert split.table_bytes == _threshold_bytes(spec, split)


def test_decode_order_ktree_bench_patterns_and_random_dags():
    spec = synth.random_ktree_dag()
    rng = np.random.default_rng(1240)
    over = 0
    for _ in range(8):
        ev = [spec.names[int(v)] for v in rng.choice(spec.n, size=11, replace=False)[1:]]
        split = _compiler(spec, sample_table_budget_bytes=1 << 36).compile_posterior_sampler(ev, dry=True)
        _check_decode_order(split, spec.n)
        assert len(split.decode) == 190 and split.table_bytes == _threshold_bytes(spec, split)
        if split.table_bytes > 1 << 30:         # 4 (card - 1) bytes per context where MPE takes 1
            over += 1
            with pytest.raises(PlanTooLarge, match="threshold tables"):
                _compiler(spec).compile_posterior_sampler(ev, dry=True)
    assert over == 3
    split = _compiler(spec).compile_posterior_sampler([], dry=True)
    _check_decode_order(split, spec.n)
    assert split.stats.final_tables == [((), 1)]
    rng = np.random.default_rng(7)
    for _ in range(30):
        cards, parents, cpts = MO.random_small_net(rng, 5, 16)
        names = [f"v{i}" for i in range(len(cards))]
        spec = synth.NetSpec(names, cards, parents, cpts)
        k = int(rng.integers(0, len(cards) + 1))
        ev = [names[int(v)] for v in rng.choice(len(cards), size=k, replace=False)]
        _check_decode_order(_compiler(spec).compile_posterior_sampler(ev, dry=True), len(cards))


def test_limits_raise_in_the_dry_pass():
    spec = synth.layered_dag()
    with pytest.raises(PlanTooLarge, match="posterior sampling has no per-row executor"):
        _compiler(spec).compile_posterior_sampler([], dry=True)
    with pytest.raises(PlanTooLarge, match="no per-row executor"):
        _compiler(spec).compile_posterior_sampler(spec.names[:10], dry=True)
    alarm = synth.alarm()
    with pytest.raises(PlanTooLarge, match="threshold tables"):
        _compiler(alarm, sample_table_budget_bytes=1 << 20).compile_posterior_sampler(synth.ALARM_EVIDENCE, dry=True)
    # the MPE budget does not bound the sampler, nor the other way round
    _compiler(alarm, mpe_argmax_budget_bytes=1 << 10).compile_posterior_sampler(synth.ALARM_EVIDENCE, dry=True)
    _compiler(alarm, sample_table_budget_bytes=1 << 10).compile_mpe(synth.ALARM_EVIDENCE, dry=True)
    split = _compiler(alarm, sample_table_budget_bytes=1 << 16).compile_posterior_sampler([], dry=True)
    assert split.table_bytes <= 1 << 16
    with pytest.raises(PlanTooLarge, match="cheapest hidden variable"):
        _compiler(alarm, table_budget_cells=1 << 10).compile_posterior_sampler(synth.ALARM_EVIDENCE, dry=True)
    with pytest.raises(ValueError):
        _compiler(alarm).compile_posterior_sampler(["HRBP", "not_a_node"], dry=True)
    with pytest.raises(ValueError):
        _compiler(alarm).compile_posterior_sampler(["HRBP", "HRBP"], dry=True)


def test_complete_evidence_has_nothing_to_draw():
    spec = synth.asia()
    split = _compiler(spec).compile_posterior_sampler(spec.names, dry=True)
    assert split.hidden == [] and split.decode == [] and split.table_bytes == 0
    assert sorted(split.observed_families) == list(range(spec.n))


def test_psample_step_layout_matches_the_header(tmp_path):
    from continuousbayesiannetwork_b200 import _native as N

    prog = tmp_path / "sz.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cbn_b200.h"\nint main(){printf("%zu %zu %zu %zu\\n", '
                    'sizeof(cbn_psample_step), offsetof(cbn_psample_step, cdf), offsetof(cbn_psample_step, n_cells), '
                    'offsetof(cbn_psample_step, var));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    S = N.PsampleStep
    assert got == [C.sizeof(S), S.cdf.offset, S.n_cells.offset, S.var.offset]


def _mix(z):
    m = (1 << 64) - 1
    z = (z + 0x9E3779B97F4A7C15) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    return z ^ (z >> 31)


def test_numpy_hash_against_python_integers():
    """The numpy restatement of the sampler's uniforms against the documented formula in arbitrary-precision integers,
    including a seed and rows that use the top bits."""
    m = (1 << 64) - 1
    for seed in (0, 1, 12345, (1 << 64) - 1):
        rows = np.array([0, 1, 2, 1 << 40, (1 << 63) - 1], dtype=np.uint64)
        for d in (0, 1, 7):
            for v in (0, 3, 36):
                got = synth.posterior_uniforms(seed, rows, d, v)
                want = []
                for r in rows.tolist():
                    b = _mix(seed ^ ((r * 0xD1B54A32D192ED03) & m))
                    b = _mix(b ^ ((d * 0x9E6C63D0676A9A99) & m))
                    h = _mix((b + v) & m)
                    want.append((h >> 40) / 16777216.0)
                assert got.dtype == np.float32 and np.array_equal(got, np.asarray(want, np.float32))
    # the first draw's row base is cbn_sample_forward's: the hash of (seed, row) is shared
    assert _mix(0) == 0xE220A8397B1DCDAF


def test_enumeration_posterior_sums_and_matches_bayes():
    spec = synth.asia()
    net = O.DiscreteNet(spec.cards, spec.parents, spec.cpts)
    p = PO.joint_table(net)
    assert abs(p.sum() - 1.0) < 1e-12
    z, post = PO.enumerate_posterior(net, [0, 7], [1, 0])
    assert abs(post.sum() - 1.0) < 1e-12 and abs(z - p[1, :, :, :, :, :, :, 0].sum()) < 1e-15


def test_interpreter_draws_follow_thresholds():
    """The numpy interpreter on a hand-built two-step schedule: the draws are where the uniforms fall between thresholds,
    values with empty intervals never appear, and dead rows are UNSEEN."""
    cards = [3, 2]
    # step 0 draws variable 1 (no context), step 1 variable 0 given variable 1
    decode = [(1, (), np.array([0.25], np.float32)),
              (0, (1,), np.array([[0.0, 1.0], [0.5, 0.5]], np.float32))]
    n = 4096
    dead = np.zeros(n, bool)
    dead[7] = True
    out = PO.interpret(decode, cards, [], np.zeros((n, 0), np.int64), dead, seed=3, first_row=5, n_draws=2)
    rows = np.arange(n, dtype=np.uint64) + np.uint64(5)
    for d in range(2):
        u1 = synth.posterior_uniforms(3, rows, d, 1)
        want1 = (u1 >= 0.25).astype(np.uint8)
        assert np.array_equal(out[1][d][~dead], want1[~dead]) and out[1][d][7] == PO.UNSEEN
        x0 = out[0][d][~dead]
        assert set(np.unique(x0[want1[~dead] == 0]).tolist()) <= {1}        # value 0 has an empty interval
        assert set(np.unique(x0[want1[~dead] == 1]).tolist()) <= {0, 2}     # value 1 has an empty interval
