"""Expectation-maximisation for networks with hidden nodes: exact E-steps on the GPU, expected counts in fixed point.

A hidden node has no column: it is hidden in every row, and the observed set ``E`` is the same for every row.  The
families that have hidden members are grouped by their hidden set ``H_f``.  For a group with ``H = (h_1 .. h_m)``
(ordered by increasing cardinality, so that the chain's ``sum_j prod_{i<j} card_i`` gathers are fewest) the joint
posterior of a row is the chain ``P(H | e) = prod_j P(h_j | e, h_<j)``.  Factor ``j`` is an ordinary single-target
posterior plan, ``compile(h_j, E + h_<j)``, run once per assignment of ``h_<j`` with constant code rows for ``h_<j``;
every compile mode and executor of ``ve.py`` is reused as it is, and groups that share a prefix share plans through
the compiler's cache.  ``cbn_ess_run`` then multiplies the chain out per row and adds ``rint(w * 2^32)`` into the
destination families' int64 tables: integer sums, so the expected counts are the same bits for any row chunking.

Fully observed families enter the same int64 buffer as ``count << 32`` from the count kernel, and the M-step is the
CPT kernel with ``n_total = n_rows << 32``: fp32 division is invariant under the common power-of-two scale, so with
complete data the CPTs are bit for bit those of the ordinary fit.

With per-row missing values (``fit_em(missing="marginalize")`` on data with NaN cells) the observed set differs from row
to row, and ``JTEM`` replaces the chain: one junction-tree calibration per row (``jt.py``, ``cbn_jt_run``) gives every
family's posterior in each row where the family has a missing member, into the same int64 buffer, and the rows where the
family is fully observed stay with the count kernel.  The M-step is the same.

Python here loops over groups, chain steps, assignments and row chunks only: each iteration of those loops is a
launch.  No loop touches row data.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _native as N
from .ve import PlanTooLarge

CHUNK_ROWS = 1 << 22             # rows per E-step chunk: bounds the chain's factor buffers
CHAIN_BUDGET_FLOATS = 4096       # sum_j prod_{i<=j} card_i: floats of chain factors per row of one group
FIXED_ONE = 1 << 32              # the fixed-point scale of the expected counts
MAX_ROWS = 1 << 31               # the accumulation kernel's bound: n_rows * 2^32 per cell stays inside 64 bits


@dataclass
class ChainGroup:
    """Families whose hidden members are exactly ``hidden`` (network ids, in chain order)."""
    hidden: List[int]
    families: List[int]

    def prefix_configs(self, cards: Sequence[int], j: int) -> int:
        """Assignments of ``hidden[:j]``: the number of runs of chain step ``j``."""
        return math.prod(cards[u] for u in self.hidden[:j])


def chain_floats(hidden: Sequence[int], cards: Sequence[int]) -> int:
    """Floats of chain factors per row: ``sum_j prod_{i<=j} card_i``."""
    total, p = 0, 1
    for u in hidden:
        p *= cards[u]
        total += p
    return total


def plan_groups(cards: Sequence[int], family_vars: Sequence[Sequence[int]], hidden: Sequence[int],
                budget_floats: int = CHAIN_BUDGET_FLOATS) -> List[ChainGroup]:
    """Group the families with hidden members by their hidden set; chain order is increasing cardinality, then id.
    A chain of more than ``budget_floats`` floats per row raises ``PlanTooLarge``."""
    hid = set(hidden)
    by_set: Dict[tuple, List[int]] = {}
    for v, fv in enumerate(family_vars):
        H = sorted((u for u in fv if u in hid), key=lambda u: (cards[u], u))
        if H:
            by_set.setdefault(tuple(H), []).append(v)
    groups = [ChainGroup(list(H), fams) for H, fams in sorted(by_set.items())]
    for g in groups:
        need = chain_floats(g.hidden, cards)
        if need > budget_floats:
            raise PlanTooLarge(f"the hidden set {g.hidden} needs {need} floats of chain factors per row; the budget is "
                               f"{budget_floats}")
    return groups


def schedule(cards: Sequence[int], family_vars: Sequence[Sequence[int]], hidden: Sequence[int]) -> dict:
    """What one E-step costs in plans and launches: ``compiles`` (distinct chain plans + the log P(e) plan),
    ``gathers`` (posterior runs per row chunk), ``ess_launches`` (per row chunk), ``floats_per_row`` (largest chain)."""
    groups = plan_groups(cards, family_vars, hidden)
    steps = {(g.hidden[j], tuple(g.hidden[:j])) for g in groups for j in range(len(g.hidden))}
    return {"groups": groups,
            "compiles": len(steps) + 1,
            "gathers": sum(g.prefix_configs(cards, j) for g in groups for j in range(len(g.hidden))),
            "ess_launches": sum(-(-len(g.families) // N.ESS_MAX_DESTS) for g in groups),
            "floats_per_row": max([chain_floats(g.hidden, cards) for g in groups], default=0)}


class EssPlan:
    """Owner of the ``cbn_ess_plan`` handles of one group (at most ``ESS_MAX_DESTS`` destinations each)."""

    def __init__(self, tables, group: ChainGroup, stream: int):
        t = self.t = tables
        self.group = group
        cards = t.cards
        hid = group.hidden
        card_h = math.prod(cards[u] for u in hid)
        # joint configuration index (h_1 slowest) -> digits, as int64 [card_H, m]
        digits = np.stack(np.unravel_index(np.arange(card_h), [cards[u] for u in hid]), axis=1) if hid else np.zeros((1, 0))
        self.handles = []
        for at in range(0, len(group.families), N.ESS_MAX_DESTS):
            fams = group.families[at: at + N.ESS_MAX_DESTS]
            dests = (N.EssDest * len(fams))()
            keep = []                                   # the cell maps must live until cbn_ess_plan_create copies them
            for k, v in enumerate(fams):
                vs = t.family_vars(t.names[v])
                stride = {}
                s = 1
                for u in reversed(vs):
                    stride[u] = s
                    s *= cards[u]
                cell = np.zeros(card_h, dtype=np.int32)
                for j, u in enumerate(hid):
                    if u in stride:
                        cell += (digits[:, j] * stride[u]).astype(np.int32)
                cell = np.ascontiguousarray(cell)
                keep.append(cell)
                d = dests[k]
                d.table_offset = t.offsets[v]
                d.n_cells = t.n_cells[v]
                obs = [u for u in vs if u not in hid]
                d.n_obs = len(obs)
                for i, u in enumerate(obs):
                    d.obs_row[i] = u
                    d.obs_card[i] = cards[u]
                    d.obs_stride[i] = stride[u]
                d.hidden_cell = cell.ctypes.data
            h = C.c_void_p()
            N.check(N.lib().cbn_ess_plan_create(t.ctx.handle, len(hid), (C.c_int32 * len(hid))(*[cards[u] for u in hid]),
                                                dests, len(fams), stream, C.byref(h)), t.ctx.handle)
            self.handles.append(h)
        self.smem_dests = sum(N.lib().cbn_ess_plan_smem_dests(h) for h in self.handles)

    def run(self, factors: Sequence[torch.Tensor], codes: torch.Tensor, n_rows: int, acc: torch.Tensor, stream: int):
        ptrs = N.ptr_array([f.data_ptr() for f in factors])
        for h in self.handles:
            N.check(N.lib().cbn_ess_run(self.t.ctx.handle, h, ptrs, codes.data_ptr(), codes.stride(0), int(n_rows),
                                        acc.data_ptr(), stream), self.t.ctx.handle)

    def __del__(self):
        try:
            for h in self.handles:
                N.lib().cbn_ess_plan_destroy(h)
            self.handles = []
        except Exception:
            pass


@dataclass
class EMResult:
    """``log_likelihood``: float64 ``sum_rows log P(e_row)`` of the parameters that entered each iteration, then one entry
    for the returned parameters (rows of probability zero are left out of the sum and counted in ``n_dead_rows``);
    ``converged``: the relative gain fell below ``tol``."""
    log_likelihood: List[float] = field(default_factory=list)
    n_iter: int = 0
    converged: bool = False
    n_dead_rows: int = 0


class EM:
    """EM over bound ``tables`` (layout and domains set, integer counts of the fully observed families counted) and an
    exact inference engine bound to them.  ``codes``: the uint8 code matrix [n_vars, ld] of the data, ``CBN_UNSEEN`` in
    the rows of ``hidden``."""

    def __init__(self, tables, inference, codes: torch.Tensor, n_rows: int, hidden: Sequence[int],
                 chunk_rows: int = CHUNK_ROWS):
        t = self._bind(tables, inference, codes, n_rows, hidden)
        self.observed = [v for v in range(len(t.names)) if v not in set(self.hidden)]
        self.groups = plan_groups(t.cards, [t.family_vars(n) for n in t.names], self.hidden)
        self.ess = [EssPlan(t, g, self.stream) for g in self.groups]
        floats = max([chain_floats(g.hidden, t.cards) for g in self.groups], default=1)
        # chunks start on 16-row boundaries (the code matrix's alignment); the factor buffers stay below 2^30 bytes
        self.chunk = max(16, min(int(chunk_rows), (1 << 30) // (4 * floats)) // 16 * 16)
        # observed codes followed by the constant rows of a chain prefix (a chain has at most every hidden node)
        self.ev = t.new_code_matrix(self.n, len(self.observed) + max(len(self.hidden), 1))
        self.ev[: len(self.observed)] = codes[self.observed, : self.ev.shape[1]]
        self.ev_names = [t.names[v] for v in self.observed]

    def _bind(self, tables, inference, codes: torch.Tensor, n_rows: int, hidden: Sequence[int]):
        """What every E-step shares: the tables, the engine, the code matrix, the hidden (latent) nodes, the stream, and
        ``base``: the counts of the fully observed rows of every family, << 32 (the count kernel skips a row of a family
        when a member's code is not below its cardinality)."""
        t = self.t = tables
        self.infer = inference
        self.codes = codes
        self.n = int(n_rows)
        self.hidden = sorted(set(hidden))
        self.stream = N.stream_ptr(t.device)
        self.base = t.allreduce_buffer()[: t.total_cells].clone() * FIXED_ONE
        self.acc = torch.empty_like(self.base)
        return t

    # ------------------------------------------------------------------ E-step
    def e_step(self):
        """Expected counts of the current ``cond`` into ``self.acc`` (int64, ``2^32`` = one row); returns ``_new_sums``
        filled with the current parameters' log-likelihood."""
        self.acc.copy_(self.base)
        sums = self._new_sums()
        for s in range(0, self.n, self.chunk):
            c = min(self.chunk, self.n - s)
            self._log_likelihood(s, c, sums)
            for g, ess in zip(self.groups, self.ess):
                ess.run(self.chain_factors(g, s, c), self.codes[:, s:], c, self.acc, self.stream)
        return sums

    def chain_factors(self, g: ChainGroup, s: int, c: int) -> List[torch.Tensor]:
        """The chain of group ``g`` for rows ``s .. s+c``: factor j is float32 [prod_{i<j} card_i][c][card_j], row a of
        it ``P(h_j | e, h_<j = a)`` (assignment a in mixed radix, h_1 slowest)."""
        t, E = self.t, len(self.observed)
        factors = []
        for j, h in enumerate(g.hidden):
            plan = self.infer.plan(t.names[h], self.ev_names + [t.names[u] for u in g.hidden[:j]])
            P = g.prefix_configs(t.cards, j)
            buf = torch.empty((P, c, t.cards[h]), dtype=torch.float32, device=t.device)
            prefix_cards = [t.cards[u] for u in g.hidden[:j]]
            for a in range(P):
                for i, d in enumerate(np.unravel_index(a, prefix_cards) if j else ()):
                    self.ev[E + i, s: s + c].fill_(int(d))
                plan.run_codes(self.ev[: E + j, s:], c, out=buf[a])
            factors.append(buf)
        return factors

    def _new_sums(self):
        """Device accumulators: float64 sum of log P(e_row) over live rows, int64 count of dead rows."""
        return (torch.zeros((), dtype=torch.float64, device=self.t.device),
                torch.zeros((), dtype=torch.int64, device=self.t.device))

    def _log_likelihood(self, s: int, c: int, sums):
        ll = self.infer.evidence_plan(self.ev_names).run_codes(self.ev[: len(self.observed), s:], c)
        live = ll > float("-inf")
        sums[0].add_(torch.where(live, ll.double(), 0.0).sum())
        sums[1].add_((~live).sum())

    # ------------------------------------------------------------------ M-step
    def m_step(self, pseudo_count: float = 0.0):
        """``cond = (N + a) / sum_x (N + a)`` through the CPT kernel (with the kernel's 1e-10 term), ``joint = N / n``."""
        t = self.t
        joint = torch.zeros(t.total_cells, dtype=torch.float32, device=t.device)
        cond = torch.zeros(t.total_cells, dtype=torch.float32, device=t.device)
        n_fixed = self.n * FIXED_ONE
        stream = self.stream
        N.check(N.lib().cbn_cpt_from_counts(t.ctx.handle, self.acc.data_ptr(), t.fams, len(t.names), n_fixed,
                                            joint.data_ptr(), None if pseudo_count else cond.data_ptr(), stream), t.ctx.handle)
        if pseudo_count:
            prior = self.acc + int(round(float(pseudo_count) * FIXED_ONE))
            N.check(N.lib().cbn_cpt_from_counts(t.ctx.handle, prior.data_ptr(), t.fams, len(t.names), n_fixed, None,
                                                cond.data_ptr(), stream), t.ctx.handle)
        t.joint = joint
        t.set_cond(cond)

    def expected_counts(self) -> torch.Tensor:
        return self.acc.double() / FIXED_ONE

    def has_hidden(self) -> bool:
        """Whether any family has a hidden member (else the first M-step is the fit)."""
        return bool(self.groups)

    # ------------------------------------------------------------------ the loop
    def initialise(self, init: str, seed: int, current: Optional[torch.Tensor]):
        """Every family gets its complete-data MLE (exact for fully observed families, zeros for the rest); families with
        a hidden member then start from Dirichlet(1) rows drawn with ``seed`` or from ``current``."""
        t = self.t
        self.acc.copy_(self.base)
        self.m_step()
        cond = t.cond.clone()
        hid = set(self.hidden)
        rng = np.random.default_rng(seed)
        for v, name in enumerate(t.names):
            if not any(u in hid for u in t.family_vars(name)):
                continue
            seg = slice(t.offsets[v], t.offsets[v] + t.n_cells[v])
            if init == "current":
                cond[seg] = current[seg]
            else:
                rows = rng.dirichlet(np.ones(t.cards[v]), size=t.n_cells[v] // t.cards[v])
                cond[seg] = torch.from_numpy(rows.reshape(-1).astype(np.float32)).to(t.device)
        t.set_cond(cond)

    def fit(self, max_iter: int = 100, tol: float = 1e-6, pseudo_count: float = 0.0) -> EMResult:
        res = EMResult()
        for it in range(int(max_iter)):
            total, _ = self.e_step()
            res.log_likelihood.append(float(total.item()))
            self.m_step(pseudo_count)
            res.n_iter = it + 1
            if not self.has_hidden():         # complete data: the first M-step is the fit
                res.converged = True
                break
            if it > 0:
                prev, cur = res.log_likelihood[-2], res.log_likelihood[-1]
                if cur - prev < tol * max(abs(prev), 1e-300):
                    res.converged = True
                    break
        total, dead = self._new_sums()
        for s in range(0, self.n, self.chunk):
            self._log_likelihood(s, min(self.chunk, self.n - s), (total, dead))
        res.log_likelihood.append(float(total.item()))
        res.n_dead_rows = int(dead.item())
        return res


class JTEM(EM):
    """EM with per-row missing values: ``codes`` holds ``CBN_MISSING`` in every missing cell and in the rows of the
    ``hidden`` (latent) nodes.  The E-step is one ``cbn_jt_run`` per row chunk, with the log-likelihood of the observed
    part of each row from the same launch; the count kernel has already put the fully observed rows of every family into
    ``base`` (it skips codes >= the cardinality, CBN_MISSING among them)."""

    def __init__(self, tables, inference, codes: torch.Tensor, n_rows: int, hidden: Sequence[int],
                 chunk_rows: int = CHUNK_ROWS):
        t = self._bind(tables, inference, codes, n_rows, hidden)
        self.groups = []
        self.chunk = max(16, int(chunk_rows) // 16 * 16)
        self.log_p = torch.empty(min(self.chunk, self.n), dtype=torch.float32, device=t.device)

    def has_hidden(self) -> bool:
        """Always: this E-step runs for data with missing cells, so some family is hidden in some row."""
        return True

    def plan(self):
        """The junction tree of the current CPTs, with no node outputs.  After an M-step only its clique tables are
        rebuilt: the structure and the schedule are kept by the compiler."""
        from . import jt

        return jt.compile_tree(self.infer.compiler).plan([])

    def e_step(self):
        self.acc.copy_(self.base)
        sums = self._new_sums()
        plan = self.plan()
        for s in range(0, self.n, self.chunk):
            c = min(self.chunk, self.n - s)
            plan.run(self.codes[:, s:], c, log_out=self.log_p, acc=self.acc)
            self._add_log_p(c, sums)
        return sums

    def _add_log_p(self, c: int, sums):
        ll = self.log_p[:c]
        live = ll > float("-inf")
        sums[0].add_(torch.where(live, ll.double(), 0.0).sum())
        sums[1].add_((~live).sum())

    def _log_likelihood(self, s: int, c: int, sums):
        self.plan().run(self.codes[:, s:], c, log_out=self.log_p)
        self._add_log_p(c, sums)
