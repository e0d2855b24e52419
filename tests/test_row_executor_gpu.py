"""The per-row elimination executor (csrc/ve.cu: ``ve_rows_kernel``, a warp per row, and ``ve_rows_thread_kernel``, a
thread per row; linear, log-space and log-evidence instantiations) against the fp64 interpreter of its contract
(tests/row_oracle.py) and fp64 enumeration, at every step body the kernels specialise on.

The schedules are built by the planner's own per-row scheduler (``VECompiler._row_plan``) over small factor graphs: a
target T, hidden variables H_j and evidence variables.  A "component" (sc, k) is one hidden variable of cardinality sc
and k factors that contain it: [H_j, T] and k - 1 tables [E_i, H_j] over fresh evidence variables.  Eliminating H_j is
one step with k factors (pre-multiplied pairwise beyond 16) summing over sc values; the final step multiplies the
components' temporaries (a step with one factor per component and no summed variable).  This reaches every (factors,
summed cardinality) cell, including those no Bayesian network's schedule produces (a single factor summed over 2-8
values).  Networks compiled end to end (``ExactInference.plan`` / ``evidence_plan`` with a small table budget) are
checked against ``oracle.cbn_oracle`` and ``tests/loglik_oracle.py`` as well.

Which kernel and which body ran is derived from the schedule by the selection rules of ``cbn_ve_plan_create_rows`` and
``ve_run_rows_t``.  The library reads its test knobs once per process: ``CBN_ROWS_THREAD=0`` forces the warp kernel,
large ``CBN_ROWT_MAX_TEMPS`` / ``CBN_ROWT_MAX_TERMS`` the thread kernel (where its shared memory fits) and
``CBN_ROWS_UNIT=0`` the strided bodies; the checks run in subprocesses under each setting and report what they ran."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import cbn_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import loglik_oracle as LO  # noqa: E402
import row_oracle as RO  # noqa: E402
from test_log_likelihood_gpu import _close  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = {False: 1e-5, True: 2e-5}          # posteriors: linear, log space

# selection rules of cbn_ve_plan_create_rows / ve_run_rows_t (csrc/ve.cu)
STEP_BYTES, INPUT_BYTES, ROWT_TPB = 160, 160, 128
ENV_WARP = {"CBN_ROWS_THREAD": "0"}
ENV_THREAD = {"CBN_ROWS_THREAD": "1", "CBN_ROWT_MAX_TEMPS": "100000", "CBN_ROWT_MAX_TERMS": "1000000000"}
ENV_STRIDED = {"CBN_ROWS_UNIT": "0"}


def _env_int(name, default):
    v = os.environ.get(name)
    return int(v) if v is not None else default


def _temp_floats(sch):
    return sum((st["out_size"] + 3) // 4 * 4 for st in sch["steps"])


def _thread_smem(sch):
    off_ints = sum(len(st["in_id"]) * st["out_size"] for st in sch["steps"])
    return (len(sch["steps"]) * STEP_BYTES + len(sch["static_scopes"]) * INPUT_BYTES + (off_ints + 3) // 4 * 16 +
            _temp_floats(sch) * ROWT_TPB * 4)


def _kernel(sch):
    terms = sum(len(st["in_id"]) * st["out_size"] * st["sum_card"] for st in sch["steps"])
    thread = (_temp_floats(sch) <= _env_int("CBN_ROWT_MAX_TEMPS", 96) and terms <= _env_int("CBN_ROWT_MAX_TERMS", 480)
              and _thread_smem(sch) <= 100 * 1024)
    return "thread" if thread and _env_int("CBN_ROWS_THREAD", 1) else "warp"


def _unit(plan, sch, st):
    """RowStepDev::unit as cbn_ve_plan_create_rows decides it."""
    nin, sc = len(st["in_id"]), st["sum_card"]
    if _env_int("CBN_ROWS_UNIT", 1) == 0 or nin > 4 or sc > 8:
        return False
    if sc > 1 and any(s != 1 for s in st["sum_stride"]):
        return False
    vec = 4 if sc % 4 == 0 else 2 if sc % 2 == 0 else 1
    if vec == 1:
        return True
    cards, ev = plan.owner.cards, set(sch["evidence"])
    offs = sch["offsets"][st["offsets_at"]: st["offsets_at"] + nin * st["out_size"]]
    if np.any(offs % vec):
        return False
    for i in st["in_id"]:
        if i < len(plan.inputs):
            f = plan.inputs[i]
            stride = 1
            for v in reversed(f.scope):
                if v in ev and stride % vec:
                    return False
                stride *= cards[v]
            if f.tensor.data_ptr() % (4 * vec):
                return False
    return True


def _sc_bucket(sc):
    return sc if sc <= 8 else ("9-99" if sc < 100 else "100+")


def _cells(plan, sch, arith, mode):
    """The (kernel, arithmetic, mode, body, factors, summed cardinality) cells one run of ``plan`` executes."""
    k = _kernel(sch)
    out = set()
    for st in sch["steps"]:
        nin = len(st["in_id"])
        body = "unit" if _unit(plan, sch, st) else "strided"
        out.add((k, arith, mode, body, nin if nin <= 4 else "5-16", _sc_bucket(st["sum_card"])))
        if any(i >= len(sch["static_scopes"]) for i in st["in_id"]):
            out.add((k, arith, mode, body + " reads a temporary", nin if nin <= 4 else "5-16", _sc_bucket(st["sum_card"])))
    return out


def _codes_matrix(ev):
    """int [rows, n_ev] -> uint8 [n_ev, ld] on the device, ld a multiple of 16."""
    n, k = ev.shape
    ld = max((n + 15) // 16 * 16, 16)
    m = torch.zeros((max(k, 1), ld), dtype=torch.uint8, device=DEV)
    if k and n:
        m[:, :n] = torch.from_numpy(np.ascontiguousarray(ev.T.astype(np.uint8))).to(DEV)
    return m


def _statics(plan):
    return [f.tensor.double().cpu().numpy() for f in plan.inputs]


# ------------------------------------------------------------------------------------------------ factor-graph cases
class Graph:
    """Variables 0 = T, then one hidden variable and its evidence variables per component.  ``values[i]`` is the fp64
    copy (of the fp32 numbers the device holds) of factor i over ``scopes[i]``, row-major."""

    def __init__(self, t_card, comps, ev_card=3, seed=0, small=None, wide_ev=False, zero_ev=False, layout_unit=True,
                 chains=()):
        rng = np.random.default_rng(seed)
        self.cards, self.scopes, self.values, self.hidden, self.E = [t_card], [], [], [], []

        def hidden(card, k):
            h = len(self.cards)
            self.cards.append(card)
            self.hidden.append(h)
            for i in range(k - 1):
                e = len(self.cards)
                self.cards.append(200 if wide_ev and not self.E else ev_card)
                self.E.append(e)
                self.scopes.append([e, h])
            return h

        for sc, k in comps:
            self.scopes.append([hidden(sc, k), 0])
        # a chain (a, b, k): H_a with k - 1 evidence tables, [H_a, H_b], [H_b, T] -- one of its summing steps reads the
        # temporary of the other
        for a, b, k in chains:
            ha = hidden(a, k)
            hb = hidden(b, 1)
            self.scopes += [[ha, hb], [hb, 0]]
        for j, scope in enumerate(self.scopes):
            shape = [self.cards[v] for v in scope]
            x = rng.uniform(0.05, 1.0, size=shape)
            if small is not None and scope[0] in self.E:
                x = rng.uniform(small, 3 * small, size=shape)             # observed children of small likelihood
            if zero_ev and scope[0] in self.E and scope[0] == self.E[0]:
                x[0] = 0.0                                              # evidence value 0 of E[0] has probability 0
            self.values.append(x.astype(np.float32).astype(np.float64).reshape(-1))
        self.layout_unit = layout_unit

    def plan(self, log_space):
        """A RowPlan over these factors, scheduled by the planner's per-row scheduler, and its schedule."""
        from continuousbayesiannetwork_b200.ve import Factor, VECompiler, _Pass
        from continuousbayesiannetwork_b200.engine import tables_from_spec
        from continuousbayesiannetwork_b200 import synth

        if not hasattr(Graph, "_tables") or Graph._tables_cards != self.cards:
            names = [f"v{i}" for i in range(len(self.cards))]
            Graph._tables = tables_from_spec(synth.NetSpec(names, self.cards, [[] for _ in names], [None] * len(names)), DEV)
            Graph._tables_cards = list(self.cards)
        comp = VECompiler(Graph._tables, row_unit_layout=self.layout_unit, row_temp_floats=1 << 16)
        facs = []
        for scope, x in zip(self.scopes, self.values):
            with np.errstate(divide="ignore"):
                v = np.log(x) if log_space else x
            facs.append(Factor(list(scope), torch.tensor(v, dtype=torch.float32, device=DEV)))
        plan = comp._row_plan(_Pass(list(self.E), 0, False, log_space, False), facs, list(self.hidden))
        return plan, comp.last_row_schedule

    def draw(self, n, seed):
        rng = np.random.default_rng(seed)
        return np.stack([rng.integers(0, self.cards[e], size=n) for e in self.E], axis=1) if self.E else np.zeros((n, 0), np.int64)

    def _message(self, h, codes):
        """[rows, card h]: the product of h's evidence tables (sliced by the row's codes) and of the sums over the hidden
        variables chained below it."""
        slot = {e: i for i, e in enumerate(self.E)}
        m = np.ones((codes.shape[0], self.cards[h]))
        for scope, x in zip(self.scopes, self.values):
            if scope[1] == h and scope[0] in slot:
                m = m * x.reshape(self.cards[scope[0]], self.cards[h])[codes[:, slot[scope[0]]]]
            elif scope[1] == h and scope[0] in self.hidden:
                m = m * (self._message(scope[0], codes) @ x.reshape(self.cards[scope[0]], self.cards[h]))
        return m

    def brute(self, codes):
        """fp64 sum over the hidden variables of the product of the factors, per row: [rows, card_T] (unnormalised)."""
        out = np.ones((codes.shape[0], self.cards[0]))
        for scope, x in zip(self.scopes, self.values):
            if scope[1] == 0:
                out = out * (self._message(scope[0], codes) @ x.reshape(self.cards[scope[0]], self.cards[0]))
        return out


def _matrix_graphs():
    """(label, Graph): together their schedules reach every cell ``_required`` asks for."""
    g = []
    for sc in range(2, 9):                     # factors 1-4 at every unrolled summed cardinality; the final step: 4 factors
        g.append((f"sc{sc}", Graph(2, [(sc, 1), (sc, 2), (sc, 3), (sc, 4)], seed=sc)))
        g.append((f"sc{sc}_strided", Graph(3, [(sc, 1), (sc, 2), (sc, 3), (sc, 4)], seed=20 + sc, layout_unit=False)))
    g.append(("final2", Graph(2, [(2, 2), (3, 2)], seed=31)))                     # final products of 2 and 3 factors
    g.append(("final3", Graph(5, [(2, 2), (3, 2), (4, 1)], seed=32)))
    g.append(("wide9", Graph(2, [(9, 1), (12, 2), (16, 3), (13, 4)], seed=33)))  # wider than the unrolled bodies
    g.append(("wide100", Graph(2, [(100, 1), (101, 2), (100, 3), (120, 4)], seed=34)))
    g.append(("many6", Graph(2, [(3, 6), (5, 16), (12, 7)], seed=35)))          # 5-16 factors: SC 3, 5, 12
    g.append(("final6", Graph(2, [(2, 2)] * 6, seed=36)))                        # a final product of 6 factors
    g.append(("over16", Graph(2, [(4, 20)] + [(2, 1)] * 17, seed=37)))           # pre-multiplied: 20 factors, 18 finals
    g.append(("t7", Graph(7, [(3, 2), (4, 3)], seed=38)))                        # target widths
    g.append(("t33", Graph(33, [(2, 2), (5, 3)], seed=39)))                      # 33-63 cells: two-cell loop and tail
    g.append(("t66", Graph(66, [(2, 3)], seed=40)))                              # >= 65 cells, not a multiple of 32;
    #                                                                                 a final step of one factor
    g.append(("t33_strided", Graph(33, [(2, 2), (7, 3)], seed=41, layout_unit=False)))
    g.append(("wide_evidence", Graph(3, [(4, 3), (3, 2)], seed=42, wide_ev=True)))  # a 200-valued evidence column
    for sc in range(2, 9):                     # summing steps that read a temporary (its scale enters the unit body's sum)
        g.append((f"chain{sc}", Graph(2, [], chains=[(4, sc, 2), (sc, 3, 3)], seed=50 + sc)))
    return g


def _required():
    """(kernel, arithmetic, mode, body, factors, summed cardinality); None matches anything.  A body "... reads a
    temporary" is a step with a temporary among its factors: its scale enters the step's arithmetic."""
    req = []
    for kern in ("warp", "thread"):
        for ar in ("lin", "log"):
            for nin in (1, 2, 3, 4):
                req += [(kern, ar, "post", "unit", nin, sc) for sc in range(1, 9)]
                req += [(kern, ar, "post", "strided", nin, sc) for sc in list(range(2, 9)) + ["9-99", "100+"]]
            req += [(kern, ar, "post", "strided", "5-16", sc) for sc in (1, 3, "9-99")]
        req += [(kern, "log", "le", None, None, sc) for sc in range(1, 9)]
        req.append((kern, "log", "le", None, "5-16", None))
        req += [(kern, ar, mode, "unit reads a temporary", None, sc) for ar, mode in (("lin", "post"), ("log", "le"))
                for sc in range(2, 9)]
    return req


def _missing(seen):
    return [r for r in _required() if not any(all(a is None or a == b for a, b in zip(r, c)) for c in seen)]


def _check_graph(label, g, n=777, seed=1):
    """Posterior and log-evidence of every arithmetic against the row oracle and fp64 enumeration; returns the cells."""
    ev = g.draw(n, seed)
    truth = g.brute(ev[:64])
    cells = set()
    for log_space in (False, True):
        plan, sch = g.plan(log_space)
        ar = "log" if log_space else "lin"
        m = _codes_matrix(ev)
        got = plan.run_codes(m, n).cpu().numpy()
        ref = RO.interpret(sch, _statics(plan), plan.owner.cards, ev, log_tables=log_space)
        want = RO.posterior(ref)
        np.testing.assert_allclose(got, want, rtol=RTOL[log_space], atol=1e-30, err_msg=f"{label} {ar}")
        np.testing.assert_allclose(got[:64], truth / truth.sum(1, keepdims=True), rtol=RTOL[log_space], atol=1e-30,
                                   err_msg=f"{label} {ar} enumeration")
        cells |= _cells(plan, sch, ar, "post")
        if log_space:
            le = plan.run_codes_log_evidence(m, n, torch.empty(n, dtype=torch.float32, device=DEV)).cpu().numpy()
            _close(le, RO.log_evidence(ref), f"{label} log-evidence")
            _close(le[:64], np.log(truth.sum(1)), f"{label} log-evidence enumeration")
            cells |= _cells(plan, sch, "log", "le")
    return cells


def _network_cells():
    """Networks compiled end to end with a table budget of one cell: a hidden H under an observed parent P, with the
    target and observed children below it; posteriors against the fp64 VE oracle, log P(e) (``compile_evidence``, the
    per-row plan under ``EvidencePlan.run_codes``) against the fp64 log-evidence oracle, both against the row oracle."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import bind_inference, install_cpts
    from continuousbayesiannetwork_b200.ve import RowPlan

    cells = set()
    for hc, tc, n_child, seed in ((5, 2, 2, 1), (8, 7, 2, 2), (9, 3, 3, 3), (6, 33, 1, 4), (3, 2, 6, 5)):
        rng = np.random.default_rng(seed)
        names = ["P", "H", "T"] + [f"E{i}" for i in range(n_child)]
        cards = [4, hc, tc] + [3] * n_child
        parents = [[], [0], [1]] + [[1]] * n_child
        spec = synth.NetSpec(names, cards, parents, synth._dirichlet_cpts(rng, cards, parents, 0.7))
        spec = synth.NetSpec(names, cards, parents, [c.astype(np.float32).astype(np.float64) for c in spec.cpts])
        evn = ["P"] + names[3:]
        ids = [names.index(e) for e in evn]
        ev = np.stack([rng.integers(0, cards[v], size=301) for v in ids], axis=1)
        m = _codes_matrix(ev)
        tables, _ = install_cpts(spec, DEV)
        net = O.DiscreteNet(spec.cards, spec.parents, spec.cpts)
        want = O.ve_posterior(net, 2, ids, ev, dtype=torch.float64)
        for log_space in (False, True):
            infer = bind_inference(tables, table_budget_cells=1, log_space=log_space)
            plan = infer.plan("T", evn)
            sch = infer.compiler.last_row_schedule
            assert isinstance(plan, RowPlan)
            got = plan.run_codes(m, 301).cpu().numpy()
            np.testing.assert_allclose(got, want, rtol=RTOL[log_space], atol=1e-30, err_msg=f"net {seed}")
            ref = RO.interpret(sch, _statics(plan), cards, ev, log_tables=log_space)
            np.testing.assert_allclose(got, RO.posterior(ref), rtol=RTOL[log_space], atol=1e-30)
            cells |= _cells(plan, sch, "log" if log_space else "lin", "post")
        infer = bind_inference(tables, table_budget_cells=1)
        ep = infer.evidence_plan(evn)
        sch = infer.compiler.last_row_schedule
        assert isinstance(ep.ve_plan, RowPlan) and sch["target"] is None
        le = ep.run_codes(m, 301).cpu().numpy()
        _close(le, LO.ve_log_evidence(net, ids, ev), f"net {seed} log P(e)")
        ref = RO.log_evidence(RO.interpret(sch, _statics(ep.ve_plan), cards, ev, log_tables=True))
        _close(ep.ve_plan.run_codes_log_evidence(m, 301, torch.empty(301, device=DEV)).cpu().numpy(), ref, "evidence plan")
        cells |= _cells(ep.ve_plan, sch, "log", "le")
    return cells


def _matrix():
    cells = set()
    for label, g in _matrix_graphs():
        cells |= _check_graph(label, g)
    return cells | _network_cells()


def _in_subprocess(fn, env, timeout=900):
    """Run ``fn`` of this file in a fresh process under ``env`` (the library reads its knobs once per process); returns
    the JSON it prints on its last line."""
    code = (f"import json, runpy; r = runpy.run_path('tests/test_row_executor_gpu.py')['{fn}'](); "
            "print('RESULT ' + json.dumps(r))")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=timeout, cwd=ROOT,
                         env=dict(os.environ, **env))
    assert out.returncode == 0, f"{fn} {env}\n" + out.stdout[-3000:] + out.stderr[-5000:]
    line = [x for x in out.stdout.splitlines() if x.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


def _matrix_json():
    return [list(c) for c in _matrix()]


# ------------------------------------------------------------------------------------------------------- a. and b.
def test_body_matrix_default_selection():
    cells = _matrix()
    assert any(c[0] == "thread" for c in cells) and any(c[0] == "warp" for c in cells)


def test_body_matrix_every_kernel_and_body_family():
    """{warp, thread} x {unit bodies allowed, CBN_ROWS_UNIT=0}: every run checks parity; the union of what ran must hold
    every required cell."""
    seen = set()
    for env in (ENV_WARP, ENV_THREAD, dict(ENV_WARP, **ENV_STRIDED), dict(ENV_THREAD, **ENV_STRIDED)):
        seen |= {tuple(c) for c in _in_subprocess("_matrix_json", env)}
    missing = _missing(seen)
    assert not missing, f"cells never run: {missing}"


# ---------------------------------------------------------------------------------------------------------- c. range
def _range_check():
    """Four hidden causes with four observed children of likelihood ~1e-3 each: every cause's temporary peaks near 1e-12
    (the warp kernel of a linear plan must rescale it in place: the unscaled product of the four in the final unit step
    is ~1e-48, below fp32), and log P(e) < -200 for the log-evidence path."""
    g = Graph(3, [(2, 5)] * 4, seed=50, small=1e-3)
    n = 513
    ev = g.draw(n, 7)
    truth = g.brute(ev[:64])
    for log_space in (False, True):
        plan, sch = g.plan(log_space)
        ref, temps = RO.interpret(sch, _statics(plan), plan.owner.cards, ev, log_tables=log_space, with_temps=True)
        if not log_space:
            taken = RO.warp_rescales(sch, temps)
            assert taken[:, :4].all() and sch["steps"][-1]["sum_card"] == 1 and len(sch["steps"][-1]["in_id"]) == 4
            assert _unit(plan, sch, sch["steps"][-1]) or _env_int("CBN_ROWS_UNIT", 1) == 0
        got = plan.run_codes(_codes_matrix(ev), n).cpu().numpy()
        np.testing.assert_allclose(got, RO.posterior(ref), rtol=RTOL[log_space], atol=1e-30)
        np.testing.assert_allclose(got[:64], truth / truth.sum(1, keepdims=True), rtol=RTOL[log_space], atol=1e-30)
    g = Graph(2, [(2, 16)] * 4, seed=51, small=1e-3)
    ev = g.draw(n, 8)
    plan, sch = g.plan(True)
    ref = RO.log_evidence(RO.interpret(sch, _statics(plan), plan.owner.cards, ev, log_tables=True))
    assert ref.max() < -200
    le = plan.run_codes_log_evidence(_codes_matrix(ev), n, torch.empty(n, device=DEV)).cpu().numpy()
    _close(le, ref, "log P(e) < -200")
    _close(le[:64], np.log(g.brute(ev[:64]).sum(1)), "log P(e) < -200, enumeration")
    return [_kernel(sch)]


@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_range_in_place_rescale_and_tiny_log_evidence(kernel):
    assert _in_subprocess("_range_check", ENV_WARP if kernel == "warp" else ENV_THREAD) == [kernel]


# ---------------------------------------------------------------------------------------------------------- d. edges
def _outputs(plan, m, n, le):
    if le:
        return plan.run_codes_log_evidence(m, n, torch.empty(n, dtype=torch.float32, device=DEV))
    return plan.run_codes(m, n)


def _edges_check():
    """Dead rows (a code equal to the cardinality, 255, zero-probability evidence), row counts around the warp and CTA
    sizes, a batch of at least three grid rounds of either kernel with every third row dead, and determinism."""
    g = Graph(3, [(3, 3), (4, 2)], seed=60, zero_ev=True)
    E0 = g.cards[g.E[0]]
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    big = 3 * sm * 8 * ROWT_TPB + 77               # >= 3 rounds of the thread kernel's (and the warp kernel's) grid
    kernels = set()
    for log_space in (False, True):
        plan, sch = g.plan(log_space)
        kernels.add(_kernel(sch))
        statics = _statics(plan)
        for le in ((False, True) if log_space else (False,)):
            def ref_of(ev):
                r = RO.interpret(sch, statics, plan.owner.cards, ev, log_tables=log_space)
                return RO.log_evidence(r) if le else RO.posterior(r)

            def check(got, ev, what):
                got = got.cpu().numpy()
                assert not np.isnan(got).any(), what
                if le:
                    _close(got, ref_of(ev), what)
                else:
                    np.testing.assert_allclose(got, ref_of(ev), rtol=RTOL[log_space], atol=1e-30, err_msg=what)

            ev = g.draw(129, 3)
            ev[:, 0] = np.maximum(ev[:, 0], 1)
            ev[5, 0] = 0                                   # zero-probability evidence
            ev[6, 1] = g.cards[g.E[1]]                     # a code equal to the cardinality
            ev[7, 2] = 255                                 # CBN_UNSEEN
            ev[8, 0] = E0
            for n in (0, 1, 2, 3, 31, 32, 33, 127, 128, 129):
                got = _outputs(plan, _codes_matrix(ev[:n]), n, le)
                assert tuple(got.shape) == ((n,) if le else (n, 3))
                check(got, ev[:n], f"{n} rows")
            got = _outputs(plan, _codes_matrix(ev), 129, le).cpu().numpy()
            for r in (5, 6, 7, 8):
                assert (np.isneginf(got[r]) if le else np.all(got[r] == 0)), r
            # a large batch with every third row dead: warps and threads go from dead rows to live ones and back
            evb = g.draw(big, 4)
            evb[::3, 1] = g.cards[g.E[1]]
            evb[1::6, 0] = 0
            mb = _codes_matrix(evb)
            a = _outputs(plan, mb, big, le)
            check(a, evb, "large batch")
            assert torch.equal(a, _outputs(plan, mb, big, le))
            cuts = [0, 16, 48, 4096 + 32, big // 2 // 16 * 16, big]
            parts = torch.cat([_outputs(plan, mb[:, s:], e - s, le) for s, e in zip(cuts, cuts[1:])])
            assert torch.equal(a, parts)
            # rows of identical evidence give identical bits
            key = np.zeros(big, dtype=np.int64)
            for j in range(evb.shape[1]):
                key = key * 256 + evb[:, j]
            _, first, inv = np.unique(key, return_index=True, return_inverse=True)
            ah = a.cpu().numpy()
            assert np.array_equal(ah.view(np.uint32), ah[first[inv]].view(np.uint32))
    return sorted(kernels)


@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_edges_dead_rows_row_counts_rounds_and_determinism(kernel):
    assert _in_subprocess("_edges_check", ENV_WARP if kernel == "warp" else ENV_THREAD) == [kernel]


# ------------------------------------------------------------------------------------------------------ e. full size
def _full_size_check():
    """A per-row plan of the benchmark's layered-DAG family (``synth.layered_dag()``, target and evidence in the first
    five layers, the benchmark's pattern generator) at 2^20 rows."""
    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import bind_inference, sample_network, tables_from_spec
    from continuousbayesiannetwork_b200.ve import DryTables, PlanTooLarge, RowPlan, VECompiler

    spec = synth.layered_dag()
    rng = np.random.default_rng(1242)
    best = None                                    # the per-row pattern with the most work whose thread kernel fits
    for _ in range(64):
        kk = int(rng.integers(5, 51))
        vs = [int(v) for v in rng.choice(5 * 50, size=kk + 1, replace=False)]
        comp = VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()))
        try:
            stats = comp.compile(spec.names[vs[0]], [spec.names[v] for v in vs[1:]], dry=True)
        except PlanTooLarge:
            continue
        if stats.per_row_hidden and _thread_smem(comp.last_row_schedule) <= 100 * 1024:
            if best is None or stats.per_row_madds > best[0]:
                best = (stats.per_row_madds, vs)
    assert best is not None and best[0] > 1000
    vs = best[1]
    tables = tables_from_spec(spec, DEV)
    tables.set_cond_tables(spec.cpts)
    infer = bind_inference(tables)
    plan = infer.plan(spec.names[vs[0]], [spec.names[v] for v in vs[1:]])
    sch = infer.compiler.last_row_schedule
    assert isinstance(plan, RowPlan)
    n = 1 << 20
    codes = sample_network(spec, seed=1244, first=0, n=n, device=DEV, tables=tables)
    ev = codes[vs[1:]].contiguous()
    half = n // 2                                  # the second half repeats rows of the first in a shuffled order
    perm = torch.from_numpy(np.random.default_rng(2).permutation(half)).to(DEV)
    ev[:, half:n] = ev[:, perm]
    a = plan.run_codes(ev, n)
    assert torch.equal(a, plan.run_codes(ev, n))
    h = (n // 3) // 16 * 16
    assert torch.equal(a, torch.cat([plan.run_codes(ev, h), plan.run_codes(ev[:, h:].contiguous(), n - h)]))
    evh = ev[:, :n].cpu().numpy().T.astype(np.int64)
    ah = a.cpu().numpy()
    pick = np.random.default_rng(3).choice(n, size=8192, replace=False)
    ref = RO.posterior(RO.interpret(sch, _statics(plan), spec.cards, evh[pick]))
    np.testing.assert_allclose(ah[pick], ref, rtol=RTOL[False], atol=1e-30)
    few = pick[:300]
    want = O.ve_posterior(O.DiscreteNet(spec.cards, spec.parents, spec.cpts), vs[0], vs[1:], evh[few], dtype=torch.float64)
    np.testing.assert_allclose(ah[few], want, rtol=RTOL[False], atol=1e-30)
    assert np.array_equal(ah[half:].view(np.uint32), ah[perm.cpu().numpy()].view(np.uint32))
    return [_kernel(sch)]


@pytest.mark.parametrize("kernel", ["warp", "thread"])
def test_full_size_layered_pattern(kernel):
    assert _in_subprocess("_full_size_check", ENV_WARP if kernel == "warp" else ENV_THREAD, timeout=1500) == [kernel]
