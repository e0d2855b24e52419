"""Every cell of the gather run path's dispatch against an fp64 statement of the gather contract.

The run entry points map a plan's target cardinality (and, for fused plans whose targets are stored interleaved, the
pair (cardinality, targets)) to a kernel instantiation; a wrong case runs the wrong kernel without an error.  Gather
plans are built here directly (``cbn_ve_plan_create_gather`` / ``cbn_ve_plan_fuse``) over small random tables and run
through every entry point for card_t 1..8, one wide target and the five interleaved pairs, once with the direct kernels
and once tile-staged (``CBN_GATHER_TILES=1``, ``CBN_GATHER_QPT=2``).  Each mode runs in a subprocess because the
library reads those switches once per process.

Contract: a posterior row is the product over the plan's tables of their slices (the sum, for tables that hold
logarithms), normalised when the plan says so (log space: a softmax); a row with an unseen code (255) in a column one of
its tables reads is all zeros; MAP stores the target domain value of the first maximum; log P(e) is the log-sum-exp of
the row over the target (-inf for an unseen code)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_ROWS = 4096 + 3                  # the last quad holds three rows
LD = (N_ROWS + 15) // 16 * 16
CARDS = [3, 130, 5]                # evidence cardinalities: column 1 has codes >= 128
UNSEEN = 255
WIDE = 11                          # a target wider than the register-resident kernels
INTERLEAVED = [(2, 2), (2, 3), (2, 4), (3, 2), (4, 2)]


def _evidence(rng):
    codes = np.stack([rng.integers(0, c, size=N_ROWS) for c in CARDS])
    codes[1, rng.choice(N_ROWS, 200, replace=False)] = rng.integers(128, CARDS[1], size=200)
    for col in range(len(CARDS)):
        codes[col, rng.choice(N_ROWS, 9, replace=False)] = UNSEEN
    codes[:, N_ROWS - 1] = [0, 129, 4]
    codes[1, N_ROWS - 2] = UNSEEN
    return codes


class Table:
    """A gather table: target fastest (when it has one), then the evidence slots in order."""

    def __init__(self, rng, ct, slots, has_target, log_space, ties=False):
        import torch

        self.slots, self.has_target = list(slots), has_target
        w = ct if has_target else 1
        self.strides, s = [], w
        for sl in self.slots:
            self.strides.append(s)
            s *= CARDS[sl]
        vals = rng.uniform(0.05, 1.0, size=(s // w, w))
        if ties and w > 1:      # equal largest entries in every fifth slice: MAP must take the first of them
            vals[::5, (w - 1) // 2:] = 1.5
        vals = vals.astype(np.float32).reshape(-1)
        self.host = np.log(vals) if log_space else vals
        self.dev = torch.from_numpy(self.host).to(DEV)
        self.ct = w

    def slices(self, codes):
        """[n, w] slices in fp64, and the rows with an unseen code in one of the table's columns."""
        dead = np.zeros(codes.shape[1], dtype=bool)
        idx = np.zeros(codes.shape[1], dtype=np.int64)
        for sl, st in zip(self.slots, self.strides):
            dead |= codes[sl] == UNSEEN
            idx += np.where(codes[sl] == UNSEEN, 0, codes[sl]) * st
        return self.host.astype(np.float64)[idx[:, None] + np.arange(self.ct)], dead


def _reference(tables, ct, codes, log_space):
    """Unnormalised rows (log space: their logarithms) and dead rows of one output."""
    acc = np.zeros((codes.shape[1], ct)) if log_space else np.ones((codes.shape[1], ct))
    dead = np.zeros(codes.shape[1], dtype=bool)
    for t in tables:
        v, d = t.slices(codes)
        acc = acc + v if log_space else acc * v
        dead |= d
    return acc, dead


def _posterior(acc, dead, normalize, log_space):
    p = np.exp(acc - acc.max(axis=1, keepdims=True)) if log_space else acc.copy()
    if normalize or log_space:
        p /= p.sum(axis=1, keepdims=True)
    p[dead] = 0.0
    return p


def _close(got, want, what, failures, rtol=1e-5, atol=1e-6):
    got = np.asarray(got, dtype=np.float64)
    if got.shape != want.shape or np.isnan(got).any():
        failures.append(f"{what}: shape {got.shape} vs {want.shape} or NaN")
        return
    ninf = np.isneginf(want)
    if not np.array_equal(np.isneginf(got), ninf):
        failures.append(f"{what}: -inf at {np.flatnonzero(np.isneginf(got) != ninf)[:5]}")
        return
    err = np.abs(got[~ninf] - want[~ninf]) - atol - rtol * np.abs(want[~ninf])
    if err.size and err.max() > 0:
        bad = np.unravel_index(np.argmax(err), err.shape)
        failures.append(f"{what}: worst excess {err.max():.3g} at {bad}")


def _check_map(got, lin, dead, domain, what, failures):
    """The domain value of the first maximum; an entry within 1e-5 of the maximum is accepted unless the maximum is an
    exact tie, which must resolve to its first index.  A dead row stores the first domain value."""
    got = np.asarray(got, dtype=np.float64)
    pos = np.searchsorted(domain, got)
    if (pos >= len(domain)).any() or not np.array_equal(domain[np.minimum(pos, len(domain) - 1)], got):
        failures.append(f"{what}: a MAP value is not a domain value")
        return
    m = lin.max(axis=1)
    ties = (lin == m[:, None]).sum(axis=1) > 1
    ok = np.where(ties, pos == np.argmax(lin, axis=1), lin[np.arange(len(pos)), np.minimum(pos, lin.shape[1] - 1)] >= m * (1 - 1e-5))
    ok = np.where(dead, pos == 0, ok)
    if not ok.all():
        failures.append(f"{what}: rows {np.flatnonzero(~ok)[:5]}")
    if lin.shape[1] > 1 and not ties[~dead].any():
        failures.append(f"{what}: no tie exercised")


class Runner:
    def __init__(self):
        import torch

        from continuousbayesiannetwork_b200 import _native as N

        self.torch, self.N = torch, N
        self.ctx = N.context_for(DEV)
        self.rng = np.random.default_rng(20261022)
        self.codes = _evidence(self.rng)
        dev = torch.zeros((len(CARDS), LD), dtype=torch.uint8)
        dev[:, :N_ROWS] = torch.from_numpy(self.codes.astype(np.uint8))
        self.host_codes = dev.clone()
        self.ev = dev.to(DEV)
        # float evidence: domain value of each code, a value outside the domain for an unseen code
        self.domains = [np.arange(c, dtype=np.float32) * 0.5 - 1.0 for c in CARDS]
        cols = [np.where(self.codes[e] == UNSEEN, 1000.25, self.domains[e][np.minimum(self.codes[e], CARDS[e] - 1)])
                for e in range(len(CARDS))]
        self.cols = [torch.from_numpy(c.astype(np.float32)).to(DEV) for c in cols]
        self.dom_dev = [torch.from_numpy(d).to(DEV) for d in self.domains]
        self.failures, self.cells = [], []
        self.plans, self.keep = [], []         # native plans, and the tables behind them

    def lib(self):
        return self.N.lib()

    def check(self, rc):
        self.N.check(rc, self.ctx.handle)

    def stream(self):
        return self.N.stream_ptr(DEV)

    def plan(self, ct, tables, normalize, log_space):
        N = self.N
        arr = (N.GatherTable * len(tables))()
        for k, t in enumerate(tables):
            g = arr[k]
            g.data, g.n_cells, g.n_ev, g.has_target = t.dev.data_ptr(), t.dev.numel(), len(t.slots), int(t.has_target)
            for j, (sl, st) in enumerate(zip(t.slots, t.strides)):
                g.ev_slot[j], g.ev_stride[j] = sl, st
        h = C.c_void_p()
        flags = (N.GATHER_NORMALIZE if normalize else 0) | (N.GATHER_LOG_SPACE if log_space else 0)
        self.check(self.lib().cbn_ve_plan_create_gather(self.ctx.handle, len(CARDS), (C.c_int32 * len(CARDS))(*CARDS), ct, arr,
                                                        len(tables), flags, self.stream(), C.byref(h)))
        self.plans.append(h)
        return h

    def fuse(self, plans):
        h = C.c_void_p()
        self.check(self.lib().cbn_ve_plan_fuse(self.ctx.handle, self.N.ptr_array([p.value for p in plans]), len(plans),
                                               self.stream(), C.byref(h)))
        self.plans.append(h)
        return h

    def empty(self, *shape):
        return self.torch.full(shape, float("nan"), dtype=self.torch.float32, device=DEV)

    def done(self, what, got, want):
        self.torch.cuda.synchronize()
        self.cells.append(what)
        _close(got.cpu().numpy() if hasattr(got, "cpu") else got, want, what, self.failures)

    def done_map(self, what, got, lin, dead, domain):
        self.torch.cuda.synchronize()
        self.cells.append(what)
        _check_map(got.cpu().numpy(), lin, dead, domain, what, self.failures)

    def run_multi(self, plan, n_out, ct):
        outs = [self.empty(N_ROWS, ct) for _ in range(n_out)]
        self.check(self.lib().cbn_ve_run_codes_multi(self.ctx.handle, plan, self.ev.data_ptr(), LD, N_ROWS,
                                                     self.N.ptr_array([o.data_ptr() for o in outs]), self.stream()))
        return outs

    def run_host(self, plan, n_out, ct, drop_last):
        torch = self.torch
        w = ct - 1 if drop_last else ct
        codes = self.host_codes.pin_memory() if drop_last else self.host_codes
        outs = [torch.full((N_ROWS, w), float("nan"), dtype=torch.float32) for _ in range(n_out)]
        if not drop_last:
            outs = [o.pin_memory() for o in outs]
        self.check(self.lib().cbn_ve_run_codes_host_multi_ex(self.ctx.handle, plan, codes.data_ptr(), codes.stride(0), N_ROWS,
                                                             self.N.ptr_array([o.data_ptr() for o in outs]),
                                                             self.N.HOST_OUT_DROP_LAST if drop_last else 0))
        return outs

    def host_cells(self, name, plan, wants):
        ct = wants[0].shape[1]
        for drop_last in (False, True) if ct >= 2 else (False,):
            got = self.run_host(plan, len(wants), ct, drop_last)
            for o, want in enumerate(wants):
                if drop_last:        # the last value stays behind; an all-zero row travels as -1 in its first value
                    want = want[:, :-1].copy()
                    want[wants[o].sum(axis=1) == 0, 0] = -1.0
                self.done(f"{name} host{' drop_last' if drop_last else ''} out {o}", got[o].numpy(), want)

    def target_cell(self, ct):
        """Single-target and fused plans of one target cardinality through every entry point that takes them."""
        rng, codes = self.rng, self.codes
        lib, h, s = self.lib(), self.ctx.handle, self.stream()
        dom = (np.arange(ct) * 1.5 + 0.25).astype(np.float32)
        dom_dev = self.torch.from_numpy(dom).to(DEV)
        ptrs = self.N.ptr_array
        cols, doms = ptrs([c.data_ptr() for c in self.cols]), ptrs([d.data_ptr() for d in self.dom_dev])
        for log_space in (False, True):
            space = "log" if log_space else "linear"
            # two tables with the target and identical indexing (the second reuses the first one's index), one without
            tabs = [Table(rng, ct, [0, 1], True, log_space, ties=True), Table(rng, ct, [0, 1], True, log_space, ties=True),
                    Table(rng, ct, [2], False, log_space)]
            self.keep += tabs
            acc, dead = _reference(tabs, ct, codes, log_space)
            want = _posterior(acc, dead, True, log_space)
            plan = self.plan(ct, tabs, True, log_space)
            name = f"card_t {ct} {space}"
            out = self.empty(N_ROWS, ct)
            self.check(lib.cbn_ve_run_codes(h, plan, self.ev.data_ptr(), LD, N_ROWS, out.data_ptr(), s))
            self.done(f"{name} posterior", out, want)
            self.host_cells(name, plan, [want])
            if ct <= 8:
                out = self.empty(N_ROWS, ct)
                self.check(lib.cbn_ve_run_f32(h, plan, cols, doms, N_ROWS, out.data_ptr(), s))
                self.done(f"{name} f32", out, want)
                for fn in ("codes", "f32"):
                    out = self.empty(N_ROWS)
                    if fn == "codes":
                        self.check(lib.cbn_ve_run_codes_map(h, plan, self.ev.data_ptr(), LD, N_ROWS, dom_dev.data_ptr(),
                                                            out.data_ptr(), s))
                    else:
                        self.check(lib.cbn_ve_run_f32_map(h, plan, cols, doms, N_ROWS, dom_dev.data_ptr(), out.data_ptr(), s))
                    self.done_map(f"{name} map {fn}", out, np.exp(acc) if log_space else acc, dead, dom.astype(np.float64))
                if log_space:
                    out = self.empty(N_ROWS)
                    self.check(lib.cbn_ve_run_codes_log_evidence(h, plan, self.ev.data_ptr(), LD, N_ROWS, out.data_ptr(), s))
                    m = acc.max(axis=1)
                    le = m + np.log(np.exp(acc - m[:, None]).sum(axis=1))
                    self.done(f"{name} log_evidence", out, np.where(dead, -np.inf, le))
            # a fused plan: this one and a second target with its own tables (unnormalised where the number space allows)
            tabs2 = [Table(rng, ct, [1, 2], True, log_space), Table(rng, ct, [0], False, log_space)]
            self.keep += tabs2
            plan2 = self.plan(ct, tabs2, log_space, log_space)
            acc2, dead2 = _reference(tabs2, ct, codes, log_space)
            want2 = _posterior(acc2, dead2, log_space, log_space)
            fused = self.fuse([plan, plan2])
            got = self.run_multi(fused, 2, ct)
            self.done(f"{name} fused out 0", got[0], want)
            self.done(f"{name} fused out 1", got[1], want2)
            self.host_cells(f"{name} fused", fused, [want, want2])

    def interleaved_cell(self, ct, n_out):
        """Single-table unnormalised plans with identical indexing: cbn_ve_plan_fuse stores them interleaved."""
        tabs = [Table(self.rng, ct, [0, 1], True, False) for _ in range(n_out)]
        self.keep += tabs
        plans = [self.plan(ct, [t], False, False) for t in tabs]
        fused = self.fuse(plans)
        wants = [_posterior(*_reference([t], ct, self.codes, False), False, False) for t in tabs]
        name = f"interleaved {ct} x {n_out}"
        for o, g in enumerate(self.run_multi(fused, n_out, ct)):
            self.done(f"{name} out {o}", g, wants[o])
        self.host_cells(name, fused, wants)

    def run_all(self):
        for ct in list(range(1, 9)) + [WIDE]:
            self.target_cell(ct)
        for ct, n_out in INTERLEAVED:
            self.interleaved_cell(ct, n_out)
        for h in self.plans:
            self.lib().cbn_ve_plan_destroy(h)
        self.plans, self.keep = [], []
        return self.cells, self.failures


def _run_all_json():
    cells, failures = Runner().run_all()
    print("RESULT " + json.dumps({"cells": cells, "failures": failures}))


ENV = {"direct": {"CBN_GATHER_TILES": "0"}, "tiled": {"CBN_GATHER_TILES": "1", "CBN_GATHER_QPT": "2"}}


@pytest.mark.parametrize("mode", sorted(ENV))
def test_every_dispatch_cell_against_the_fp64_contract(mode):
    env = dict(os.environ, **ENV[mode])
    code = "import runpy; runpy.run_path('tests/test_gather_dispatch_gpu.py')['_run_all_json']()"
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("RESULT ")]
    assert out.returncode == 0 and lines, out.stdout[-3000:] + out.stderr[-3000:]
    res = json.loads(lines[-1][len("RESULT "):])
    assert not res["failures"], "\n".join(res["failures"])
    cells = res["cells"]
    for ct in range(1, 9):
        for space in ("linear", "log"):
            name = f"card_t {ct} {space}"
            for what in ("posterior", "f32", "map codes", "map f32", "fused out 0", "fused out 1", "host out 0"):
                assert f"{name} {what}" in cells
        assert f"card_t {ct} log log_evidence" in cells
    for space in ("linear", "log"):
        assert f"card_t {WIDE} {space} posterior" in cells and f"card_t {WIDE} {space} host drop_last out 0" in cells
    for ct, n_out in INTERLEAVED:
        for o in range(n_out):
            assert f"interleaved {ct} x {n_out} out {o}" in cells
            assert f"interleaved {ct} x {n_out} host drop_last out {o}" in cells
