"""Variable-elimination compiler: (target, evidence set) -> gather plan or per-row elimination plan.

The reference has no working VE (cbn/inference/exact.py:13-14 is ``pass``; its
``BayesianNetwork.infer``, cbn/base/bayesian_network.py:208-305, is a posterior only
for star DAGs -- SURVEY.md section 3.3).  This module is the engine behind the reference's
empty inference plugin slot.

Idea (SURVEY.md section 7 "hard parts"): the evidence *pattern* is fixed for a batch, so the
hidden variables are eliminated ONCE, on the GPU, with the evidence variables kept as
free axes of the factors ("evidence-symbolic" elimination).  What is left is a handful
of tables over (evidence subset, target); each query row only gathers one slice per
table, multiplies and normalises -- an HBM-bound kernel (``cbn_ve_run_*``).

When the evidence boundary of the target's component is too large to tabulate (the cheapest
remaining elimination step exceeds the table budget), compile-time elimination stops and the rest
of the hidden variables is eliminated per row by a schedule of product / sum-out steps
(``RowPlan`` -> ``cbn_ve_plan_create_rows``; linear space with per-step rescaling or log-sum-exp).

Host work here is graph logic only (pruning, ordering with incremental bookkeeping, stride and
offset tables); every floating-point operation runs on the device (``cbn_factor_contract`` at
compile time, the gather / per-row kernels per evidence row).

The same elimination with ``max`` in place of the sum (``VECompiler.compile_mpe``) gives the most probable explanation:
every step also records its argmax table, and a per-row traceback (``cbn_mpe_run``) reads the hidden values back in
reverse elimination order.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _native as N


class PlanTooLarge(NotImplementedError):
    pass


def _prod(it) -> int:
    p = 1
    for x in it:
        p *= int(x)
    return p


@dataclass
class Factor:
    scope: List[int]                     # variable ids; tensor is row-major over this list
    tensor: Optional[torch.Tensor]       # float32 device tensor (None in dry-run)

    def size(self, cards) -> int:
        s = 1
        for v in self.scope:
            s *= cards[v]
        return s


@dataclass
class PlanStats:
    n_relevant: int = 0
    n_hidden: int = 0
    n_steps: int = 0
    max_table_cells: int = 0
    contraction_madds: int = 0
    final_tables: List[Tuple[Tuple[int, ...], int]] = field(default_factory=list)
    support_unchecked: bool = False
    per_row_hidden: int = 0                      # hidden variables left to the per-row executor (0 = gather plan)
    per_row_madds: int = 0                       # multiply-adds of the per-row schedule, per evidence row
    per_row_slice_cells: int = 0                 # cells of the static tables' slices one evidence row reads (per-row plans)
    contraction_gpu_ms: float = 0.0              # device time of the compile-time contraction kernels (CUDA events)
    relevant_evidence: List[int] = field(default_factory=list)


class QueryPlan:
    """A compiled (target, evidence-set) query.  Owns the final tables and the native plan."""

    def __init__(self, tables_owner, target: int, evidence: List[int], card_t: int, finals: List[Factor],
                 normalize: bool, stats: PlanStats, log_space: bool = False):
        self.owner = tables_owner
        self.ctx = tables_owner.ctx
        self.device = tables_owner.device
        self.target = target
        self.evidence = list(evidence)
        self.card_t = card_t
        self.finals = finals
        self.normalize = normalize
        self.log_space = bool(log_space)           # the final tables hold logarithms (several tables, LSE epilogue per row)
        self.stats = stats
        self.handle = None
        cards = tables_owner.cards
        slot = {v: i for i, v in enumerate(self.evidence)}
        arr = (N.GatherTable * len(finals))()
        for k, f in enumerate(finals):
            has_t = bool(f.scope) and f.scope[-1] == target
            ev_scope = f.scope[:-1] if has_t else f.scope
            g = arr[k]
            g.data = f.tensor.data_ptr()
            g.n_cells = f.tensor.numel()
            g.n_ev = len(ev_scope)
            g.has_target = 1 if has_t else 0
            stride = card_t if has_t else 1
            for j in range(len(ev_scope) - 1, -1, -1):
                g.ev_slot[j] = slot[ev_scope[j]]
                g.ev_stride[j] = stride
                stride *= cards[ev_scope[j]]
        ev_cards = (C.c_int32 * max(len(self.evidence), 1))(*[cards[v] for v in self.evidence])
        h = C.c_void_p()
        N.check(N.lib().cbn_ve_plan_create_gather(self.ctx.handle, len(self.evidence), ev_cards, card_t, arr, len(finals),
                                                  (N.GATHER_NORMALIZE if normalize else 0) | (N.GATHER_LOG_SPACE if log_space else 0),
                                                  N.stream_ptr(self.device), C.byref(h)), self.ctx.handle)
        self.handle = h

    def __del__(self):
        try:
            if self.handle is not None:
                N.lib().cbn_ve_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # bytes the kernel must move per row (SURVEY.md section 8d): relevant evidence codes in, posterior out
    def algorithmic_bytes_per_row(self) -> int:
        return len(self.stats.relevant_evidence) + 4 * self.card_t

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """ev_codes: uint8 [len(evidence), ld] on the device (row e = evidence variable e of the plan)."""
        assert ev_codes.dtype == torch.uint8 and ev_codes.is_cuda
        if out is None:
            out = torch.empty((n_rows, self.card_t), dtype=torch.float32, device=self.device)
        ld = ev_codes.stride(0) if ev_codes.dim() == 2 else 0
        N.check(N.lib().cbn_ve_run_codes(self.ctx.handle, self.handle, ev_codes.data_ptr(), ld, int(n_rows),
                                         out.data_ptr(), N.stream_ptr(self.device)), self.ctx.handle)
        return out

    def set_static_evidence(self, on: bool = True):
        """Declare that the evidence of this plan's runs is never written by the kernel preceding the run on the same
        stream (resident batches replayed from a CUDA graph): evidence loads may then overlap the previous launch."""
        N.check(N.lib().cbn_ve_plan_set_static_evidence(self.handle, 1 if on else 0), self.ctx.handle)

    def _encode_evidence(self, ev_cols: Sequence[torch.Tensor], n_rows: int) -> torch.Tensor:
        ld = (max(n_rows, 1) + 15) // 16 * 16
        codes = torch.empty((max(len(self.evidence), 1), ld), dtype=torch.uint8, device=self.device)
        for e, (v, col) in enumerate(zip(self.evidence, ev_cols)):
            self.owner.encode(col, v, codes[e])
        return codes

    def run_f32(self, ev_cols: Sequence[torch.Tensor], n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """ev_cols[e]: float32 device column of evidence variable e (the reference's [nq,1] tensors)."""
        if self.card_t > N.GATHER_MAX_CT or len(self.evidence) > N.MAX_EVIDENCE_PTRS:
            # wide targets / very many evidence columns: the float kernel keeps the posterior in registers and takes its
            # column pointers as kernel arguments; encode on the device and use the code kernels (any cardinality)
            return self.run_codes(self._encode_evidence(ev_cols, n_rows), n_rows, out)
        if out is None:
            out = torch.empty((n_rows, self.card_t), dtype=torch.float32, device=self.device)
        cols = N.ptr_array([c.data_ptr() for c in ev_cols])
        doms = N.ptr_array([self.owner.domains[v].data_ptr() for v in self.evidence])
        N.check(N.lib().cbn_ve_run_f32(self.ctx.handle, self.handle, cols, doms, int(n_rows), out.data_ptr(),
                                       N.stream_ptr(self.device)), self.ctx.handle)
        return out

    # MAP value per row: posterior + argmax + domain lookup fused into the query kernel (one float per row instead of a
    # posterior row that a second kernel would read again)
    def run_codes_map(self, ev_codes: torch.Tensor, n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if out is None:
            out = torch.empty(n_rows, dtype=torch.float32, device=self.device)
        ld = ev_codes.stride(0) if ev_codes.dim() == 2 else 0
        N.check(N.lib().cbn_ve_run_codes_map(self.ctx.handle, self.handle, ev_codes.data_ptr(), ld, int(n_rows),
                                             self.owner.domains[self.target].data_ptr(), out.data_ptr(), N.stream_ptr(self.device)),
                self.ctx.handle)
        return out

    def run_f32_map(self, ev_cols: Sequence[torch.Tensor], n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if out is None:
            out = torch.empty(n_rows, dtype=torch.float32, device=self.device)
        cols = N.ptr_array([c.data_ptr() for c in ev_cols])
        doms = N.ptr_array([self.owner.domains[v].data_ptr() for v in self.evidence])
        N.check(N.lib().cbn_ve_run_f32_map(self.ctx.handle, self.handle, cols, doms, int(n_rows),
                                           self.owner.domains[self.target].data_ptr(), out.data_ptr(), N.stream_ptr(self.device)),
                self.ctx.handle)
        return out

    def run_codes_host(self, ev_codes_host: torch.Tensor, n_rows: int, out_host: torch.Tensor) -> torch.Tensor:
        """Host buffers in, host buffer out (copies inside; synchronous)."""
        assert not ev_codes_host.is_cuda and not out_host.is_cuda
        N.check(N.lib().cbn_ve_run_codes_host(self.ctx.handle, self.handle, ev_codes_host.data_ptr(),
                                              ev_codes_host.stride(0), int(n_rows), out_host.data_ptr()), self.ctx.handle)
        return out_host


class FusedPlan:
    """Several targets over the same evidence list answered by ONE launch: the evidence codes are read once
    and every target's posterior is written (``cbn_ve_plan_fuse`` / ``cbn_ve_run_codes_multi``)."""

    def __init__(self, plans: Sequence[QueryPlan]):
        assert len(plans) >= 1
        self.plans = list(plans)            # keep the tables alive
        self.ctx = plans[0].ctx
        self.device = plans[0].device
        self.card_t = plans[0].card_t
        arr = N.ptr_array([p.handle.value for p in plans])
        h = C.c_void_p()
        N.check(N.lib().cbn_ve_plan_fuse(self.ctx.handle, arr, len(plans), N.stream_ptr(self.device), C.byref(h)), self.ctx.handle)
        self.handle = h
        self.n_out = N.lib().cbn_ve_plan_outputs(h)

    def __del__(self):
        try:
            if self.handle is not None:
                N.lib().cbn_ve_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def set_static_evidence(self, on: bool = True):
        N.check(N.lib().cbn_ve_plan_set_static_evidence(self.handle, 1 if on else 0), self.ctx.handle)

    def algorithmic_bytes_per_row(self) -> int:
        ev = set()
        for p in self.plans:
            ev |= set(p.stats.relevant_evidence)
        return len(ev) + 4 * self.card_t * self.n_out

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, outs: Optional[Sequence[torch.Tensor]] = None):
        if outs is None:
            outs = [torch.empty((n_rows, self.card_t), dtype=torch.float32, device=self.device) for _ in range(self.n_out)]
        assert len(outs) == self.n_out
        ptrs = N.ptr_array([o.data_ptr() for o in outs])
        ld = ev_codes.stride(0) if ev_codes.dim() == 2 else 0
        N.check(N.lib().cbn_ve_run_codes_multi(self.ctx.handle, self.handle, ev_codes.data_ptr(), ld, int(n_rows), ptrs,
                                               N.stream_ptr(self.device)), self.ctx.handle)
        return list(outs)


def _fused_run_codes_host(self, ev_codes_host: torch.Tensor, n_rows: int, outs_host: Sequence[torch.Tensor], compact: bool = False):
    """Host buffers in, host buffers out, one fused launch per chunk (copies inside; synchronous).  ``compact``: the
    outputs are float32 [n_rows, card_t - 1] (``CBN_HOST_OUT_DROP_LAST``; ``expand_compact`` restores the full rows)."""
    assert not ev_codes_host.is_cuda and len(outs_host) == self.n_out and all(not o.is_cuda for o in outs_host)
    width = self.card_t - 1 if compact else self.card_t
    assert all(o.is_contiguous() and o.shape[-1] == width and o.shape[0] >= n_rows for o in outs_host)
    ptrs = N.ptr_array([o.data_ptr() for o in outs_host])
    N.check(N.lib().cbn_ve_run_codes_host_multi_ex(self.ctx.handle, self.handle, ev_codes_host.data_ptr(), ev_codes_host.stride(0),
                                                   int(n_rows), ptrs, N.HOST_OUT_DROP_LAST if compact else 0), self.ctx.handle)
    return list(outs_host)


def expand_compact(compact: torch.Tensor) -> torch.Tensor:
    """[n, card - 1] rows of the compact host format -> full posterior rows [n, card] (last = 1 - sum; -1 flags a zero row)."""
    dead = compact[:, 0] < 0
    last = (1.0 - compact.sum(dim=1, keepdim=True)).clamp_(min=0.0)
    full = torch.cat([compact, last], dim=1)
    full[dead] = 0.0
    return full


FusedPlan.run_codes_host = _fused_run_codes_host


class RowPlan:
    """A query whose evidence boundary is too large to tabulate: static tables for what could be eliminated at
    compile time + a per-row schedule of product / sum-out steps (``cbn_ve_plan_create_rows``)."""

    def __init__(self, tables_owner, target: int, evidence: List[int], card_t: int, inputs: List[Factor],
                 steps: List[dict], offsets, stats: PlanStats, log_space: bool):
        self.owner = tables_owner
        self.ctx = tables_owner.ctx
        self.device = tables_owner.device
        self.target = target
        self.evidence = list(evidence)
        self.card_t = card_t
        self.inputs = inputs            # keep the tables alive
        self.offsets = offsets          # host int32 array (numpy): copied into the plan at creation
        self.stats = stats
        self.log_space = log_space
        self.handle = None
        cards = tables_owner.cards
        slot = {v: i for i, v in enumerate(self.evidence)}
        Eset = set(self.evidence)
        ins = (N.RowInput * len(inputs))()
        for k, f in enumerate(inputs):
            ins[k].data = f.tensor.data_ptr()
            ins[k].n_cells = f.tensor.numel()
            stride, j = 1, 0
            ev_axes = []
            for v in reversed(f.scope):
                if v in Eset:
                    ev_axes.append((slot[v], stride))
                stride *= cards[v]
            ins[k].n_ev = len(ev_axes)
            for j, (sl, st) in enumerate(ev_axes):
                ins[k].ev_slot[j] = sl
                ins[k].ev_stride[j] = st
        sts = (N.RowStep * len(steps))()
        for j, st in enumerate(steps):
            sts[j].out_size = st["out_size"]
            sts[j].sum_card = st["sum_card"]
            sts[j].n_in = len(st["in_id"])
            for k, (i, ss) in enumerate(zip(st["in_id"], st["sum_stride"])):
                sts[j].in_id[k] = i
                sts[j].sum_stride[k] = ss
            sts[j].offsets = offsets.ctypes.data + 4 * st["offsets_at"]
        ev_cards = (C.c_int32 * max(len(self.evidence), 1))(*[cards[v] for v in self.evidence])
        h = C.c_void_p()
        N.check(N.lib().cbn_ve_plan_create_rows(self.ctx.handle, len(self.evidence), ev_cards, card_t, ins, len(inputs), sts,
                                                len(steps), N.ROWS_LOG_SPACE if log_space else 0, N.stream_ptr(self.device),
                                                C.byref(h)), self.ctx.handle)
        self.handle = h

    def __del__(self):
        try:
            if self.handle is not None:
                N.lib().cbn_ve_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def algorithmic_bytes_per_row(self) -> int:
        return len(self.stats.relevant_evidence) + 4 * self.card_t

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        assert ev_codes.dtype == torch.uint8 and ev_codes.is_cuda
        if out is None:
            out = torch.empty((n_rows, self.card_t), dtype=torch.float32, device=self.device)
        ld = ev_codes.stride(0) if ev_codes.dim() == 2 else 0
        N.check(N.lib().cbn_ve_run_codes(self.ctx.handle, self.handle, ev_codes.data_ptr(), ld, int(n_rows),
                                         out.data_ptr(), N.stream_ptr(self.device)), self.ctx.handle)
        return out

    def run_f32(self, ev_cols: Sequence[torch.Tensor], n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Float evidence columns: encoded on the device first (unseen values -> CBN_UNSEEN -> zero rows)."""
        ld = (max(n_rows, 1) + 15) // 16 * 16
        codes = torch.empty((max(len(self.evidence), 1), ld), dtype=torch.uint8, device=self.device)
        for e, (v, col) in enumerate(zip(self.evidence, ev_cols)):
            self.owner.encode(col, v, codes[e])
        return self.run_codes(codes, n_rows, out)


@dataclass
class EvidenceSplit:
    """How ``VECompiler.compile_evidence`` splits ``log P(e)``: the families summed by the observed-families kernel
    (network ids of the CPT owners) and the statistics of the VE plan for the rest (None: there is no rest)."""
    evidence: List[int]
    observed_families: List[int]
    ve_stats: Optional[PlanStats]
    per_row: bool = False


class LogLikPlan:
    """Owner of a ``cbn_loglik_plan``: ``out[row] (+)= sum_f log cond_f[index_f(row)]`` over families whose variables are
    all columns of the code matrix handed to ``run`` (``columns[v]``: the column of network variable v)."""

    def __init__(self, tables_owner, families: Sequence[int], columns: Dict[int, int], n_cols: int):
        self.ctx = tables_owner.ctx
        self.device = tables_owner.device
        self.handle = None
        t = tables_owner
        fams = (N.Family * max(len(families), 1))()
        for i, v in enumerate(families):
            vs = t.family_vars(t.names[v])
            fams[i] = N.make_family([columns[u] for u in vs], [t.cards[u] for u in vs], t.offsets[v])
        h = C.c_void_p()
        # the plan derives its own (merged) tables from the log tables and does not keep a reference to them
        N.check(N.lib().cbn_loglik_plan_create(self.ctx.handle, fams, len(families), int(n_cols), t.log_cond.data_ptr(),
                                               N.stream_ptr(self.device), C.byref(h)), self.ctx.handle)
        self.handle = h
        self.lookups_per_row = N.lib().cbn_loglik_plan_tables(h)

    def __del__(self):
        try:
            if self.handle is not None:
                N.lib().cbn_loglik_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def run(self, codes: torch.Tensor, n_rows: int, out: torch.Tensor, accumulate: bool = False) -> torch.Tensor:
        assert codes.dtype == torch.uint8 and codes.is_cuda and out.dtype == torch.float32
        N.check(N.lib().cbn_loglik_run(self.ctx.handle, self.handle, codes.data_ptr(), codes.stride(0), int(n_rows),
                                       out.data_ptr(), 1 if accumulate else 0, N.stream_ptr(self.device)), self.ctx.handle)
        return out


class EvidencePlan:
    """A compiled ``log P(e)`` query (``VECompiler.compile_evidence``): the observed-families kernel over the CPTs that
    lie inside the evidence set, plus at most one VE plan (gather or per-row) for the rest."""

    def __init__(self, tables_owner, evidence: List[int], observed_families: List[int], ve_plan, split: EvidenceSplit):
        self.owner = tables_owner
        self.ctx = tables_owner.ctx
        self.device = tables_owner.device
        self.evidence = list(evidence)
        self.observed_families = list(observed_families)
        self.ve_plan = ve_plan
        self.split = split
        slot = {v: i for i, v in enumerate(self.evidence)}
        self.loglik = LogLikPlan(tables_owner, self.observed_families, slot, len(self.evidence)) if self.observed_families else None

    def algorithmic_bytes_per_row(self) -> int:
        return len(self.evidence) + 4

    def set_static_evidence(self, on: bool = True):
        if self.ve_plan is not None:
            self.ve_plan.set_static_evidence(on)

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """ev_codes: uint8 [len(evidence), ld] on the device (row e = evidence variable e of the plan).  Returns float32
        [n_rows]: log P(e_row), -inf for an unseen value or evidence of probability zero."""
        assert ev_codes.dtype == torch.uint8 and ev_codes.is_cuda
        if out is None:
            out = torch.empty(n_rows, dtype=torch.float32, device=self.device)
        if n_rows == 0:
            return out
        accumulate = False
        if self.ve_plan is not None:
            ld = ev_codes.stride(0) if ev_codes.dim() == 2 else 0
            N.check(N.lib().cbn_ve_run_codes_log_evidence(self.ctx.handle, self.ve_plan.handle, ev_codes.data_ptr(), ld,
                                                          int(n_rows), out.data_ptr(), N.stream_ptr(self.device)),
                    self.ctx.handle)
            accumulate = True
        if self.loglik is not None:
            self.loglik.run(ev_codes, n_rows, out, accumulate=accumulate)
        elif self.ve_plan is None:          # no evidence: log 1
            out.zero_()
        return out


@dataclass
class MPESplit:
    """Structure of a most-probable-explanation plan (``VECompiler.compile_mpe``)."""
    evidence: List[int]
    hidden: List[int]                                   # network ids; row h of the decoded code matrix is hidden[h]
    observed_families: List[int]                        # CPTs scored by the observed-families kernel
    decode: List[Tuple[int, Tuple[int, ...]]]           # (variable, scope of its argmax table) in decode order
    argmax_bytes: int
    stats: PlanStats


class MPEPlan:
    """A compiled most probable explanation: the argmax tables of the max-sum elimination, the native traceback plan
    (``cbn_mpe_plan_create``) and the ``EvidencePlan`` that computes each row's value ``log max_h P(h, e)``."""

    def __init__(self, tables_owner, split: MPESplit, decode, value: EvidencePlan):
        self.owner = tables_owner
        self.ctx = tables_owner.ctx
        self.device = tables_owner.device
        self.split = split
        self.evidence = list(split.evidence)
        self.hidden = list(split.hidden)
        self.value = value
        self.argmax = [am for _, _, am in decode]           # referenced by the native plan: kept alive with it
        self.handle = None
        cards = tables_owner.cards
        n_ev = len(self.evidence)
        slot = {v: i for i, v in enumerate(self.evidence)}
        slot.update({v: n_ev + h for h, v in enumerate(self.hidden)})
        if not self.hidden:
            return
        steps = (N.MpeStep * len(decode))()
        for k, (v, scope, am) in enumerate(decode):
            st = steps[k]
            st.slot = slot[v]
            st.card = cards[v]
            st.argmax = am.data_ptr()
            st.n_cells = am.numel()
            st.n_ctx = len(scope)
            stride = 1
            for j in range(len(scope) - 1, -1, -1):
                st.ctx_slot[j] = slot[scope[j]]
                st.ctx_stride[j] = stride
                stride *= cards[scope[j]]
        ev_cards = (C.c_int32 * max(n_ev, 1))(*[cards[v] for v in self.evidence])
        h = C.c_void_p()
        N.check(N.lib().cbn_mpe_plan_create(self.ctx.handle, n_ev, ev_cards, len(self.hidden), steps, len(decode),
                                            N.stream_ptr(self.device), C.byref(h)), self.ctx.handle)
        self.handle = h

    def __del__(self):
        try:
            if self.handle is not None:
                N.lib().cbn_mpe_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def set_static_evidence(self, on: bool = True):
        self.value.set_static_evidence(on)

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, hidden_out: Optional[torch.Tensor] = None,
                  value_out: Optional[torch.Tensor] = None):
        """ev_codes: uint8 [len(evidence), ld] on the device (row e = evidence variable e of the plan, ld a multiple of
        16).  Returns ``(hidden_codes, log_value)``: uint8 [len(hidden), ld'] (row h = network variable ``hidden[h]``,
        CBN_UNSEEN in every row whose value is -inf) and float32 [n_rows] ``log max_h P(h, e_row)``."""
        assert ev_codes.dtype == torch.uint8 and ev_codes.is_cuda
        value = self.value.run_codes(ev_codes, n_rows, value_out)
        if hidden_out is None:
            ld = (max(n_rows, 1) + 15) // 16 * 16
            hidden_out = torch.empty((len(self.hidden), ld), dtype=torch.uint8, device=self.device)
        if self.handle is not None and n_rows > 0:
            ld = ev_codes.stride(0) if ev_codes.dim() == 2 else 0
            N.check(N.lib().cbn_mpe_run(self.ctx.handle, self.handle, ev_codes.data_ptr(), ld, int(n_rows), value.data_ptr(),
                                        hidden_out.data_ptr(), hidden_out.stride(0), N.stream_ptr(self.device)),
                    self.ctx.handle)
        return hidden_out, value


class _Greedy:
    """Greedy min-size elimination with incremental bookkeeping: the scope a variable's elimination would create is
    cached and only recomputed for the variables that share a factor with the one just eliminated (the full rescan is
    quadratic in the number of hidden variables: minutes on the 1000-node configuration)."""

    def __init__(self, cards, scopes: Dict[int, List[int]], hidden: Sequence[int], count=None):
        self.cards = cards
        self.scopes = {k: list(v) for k, v in scopes.items()}          # factor key -> scope
        self.count = count if count is not None else (lambda v: True)   # which axes count towards the size
        self.by_var: Dict[int, set] = {}
        for k, sc in self.scopes.items():
            for v in sc:
                self.by_var.setdefault(v, set()).add(k)
        self.hidden = set(hidden)
        self.cost: Dict[int, tuple] = {v: self._cost(v) for v in self.hidden}

    def _cost(self, v):
        sc = set()
        for k in self.by_var.get(v, ()):
            sc.update(self.scopes[k])
        sc.discard(v)
        c = 1
        for u in sc:
            if self.count(u):
                c *= self.cards[u]
        return c, sc

    def best(self):
        """(variable, size of the table its elimination creates, scope of that table) with the smallest size."""
        v = min(self.hidden, key=lambda x: (self.cost[x][0], x))
        c, sc = self.cost[v]
        return v, c, sc

    def touching(self, v) -> List:
        return sorted(self.by_var.get(v, ()), key=lambda k: (str(type(k)), k))

    def eliminate(self, v, new_key, new_scope: Sequence[int]):
        """Remove ``v`` and the factors that mention it; add the factor ``new_key`` over ``new_scope``."""
        for k in list(self.by_var.get(v, ())):
            for u in self.scopes[k]:
                self.by_var[u].discard(k)
            del self.scopes[k]
        self.by_var.pop(v, None)
        self.hidden.discard(v)
        self.cost.pop(v, None)
        self.add(new_key, new_scope)

    def add(self, key, scope: Sequence[int]):
        self.scopes[key] = list(scope)
        for u in scope:
            self.by_var.setdefault(u, set()).add(key)
        for u in scope:
            if u in self.hidden:
                self.cost[u] = self._cost(u)

    def replace(self, old_keys, new_key, new_scope):
        """Pre-multiplication: several factors become one over the union scope (no variable disappears)."""
        for k in old_keys:
            for u in self.scopes[k]:
                self.by_var[u].discard(k)
            del self.scopes[k]
        self.add(new_key, new_scope)


class VECompiler:
    """Lower (target, evidence set) to a gather plan over a fitted ``DiscreteTables``."""

    def __init__(self, tables, table_budget_cells: int = 1 << 28, merge_budget_cells: int = 1 << 24,
                 check_support: bool = True, row_temp_floats: int = 5000, log_space: bool = False, rescale: bool = True,
                 profile_compile: bool = False, row_unit_layout: bool = True, mpe_argmax_budget_bytes: int = 1 << 30):
        self.t = tables
        # range control of the compile-time elimination: after every contraction each evidence slice of the result is
        # divided by its maximum (cbn_factor_rescale) -- a factor of the evidence configuration only, which cancels in the
        # final normalisation -- so products of many small likelihoods stay inside the fp32 range
        self.rescale = bool(rescale)
        self.profile_compile = bool(profile_compile)      # CUDA events around every contraction -> PlanStats.contraction_gpu_ms
        self._ev_set: set = set()
        self._events: list = []
        self.table_budget = int(table_budget_cells)
        self.merge_budget = int(merge_budget_cells)
        self.check_support = check_support
        self.row_temp_floats = int(row_temp_floats)     # per-row temporaries of the per-row executor (shared memory)
        self.row_unit_layout = bool(row_unit_layout)    # lay every per-row factor out with its consumer's summed variable innermost
        self.log_space = bool(log_space)
        self._cache: Dict[tuple, QueryPlan] = {}
        self._has_zero: Dict[int, bool] = {}
        self.last_row_schedule: Optional[dict] = None
        self._ev_child: Optional["VECompiler"] = None       # the evidence-mode compiler (log space, no range control)
        self._ev_cache: Dict[tuple, "EvidencePlan"] = {}
        self._ev_cache_version = None
        self.mpe_argmax_budget = int(mpe_argmax_budget_bytes)    # argmax tables of one MPE plan, in bytes
        self._mpe_cache: Dict[tuple, "MPEPlan"] = {}

    # ---------------------------------------------------------------- graph helpers
    def _parents(self, v: int) -> List[int]:
        return self.t.family_vars(self.t.names[v])[:-1]

    def _ancestors(self, seeds, cut=()) -> set:
        """Ancestors of ``seeds`` (inclusive); the parents of variables in ``cut`` (interventions) are not followed."""
        seen, stack = set(), list(seeds)
        while stack:
            v = stack.pop()
            if v in seen:
                continue
            seen.add(v)
            if v not in cut:
                stack.extend(self._parents(v))
        return seen

    def _cond_has_zero(self, v: int) -> bool:
        if v not in self._has_zero:
            view = self.t.table_view(self.t.cond, self.t.names[v])
            self._has_zero[v] = bool((view == 0).any().item())
        return self._has_zero[v]

    # ---------------------------------------------------------------- device contraction
    def _contract(self, inputs: List[Factor], out_scope: List[int], sum_var: Optional[int], dry: bool,
                  normalize_last: bool = False, argmax: Optional[torch.Tensor] = None) -> Factor:
        """``argmax``: uint8 device buffer of the output's size -- maximise over ``sum_var`` instead of summing
        (``cbn_factor_contract_max``, log space) and record the maximising value of every output cell there."""
        cards = self.t.cards
        if dry:
            return Factor(out_scope, None)
        if len(out_scope) > N.MAX_CONTRACT_DIMS:
            raise PlanTooLarge(f"factor with {len(out_scope)} axes exceeds {N.MAX_CONTRACT_DIMS}")
        d = N.Contract()
        d.n_out_dims = len(out_scope)
        for a, v in enumerate(out_scope):
            d.out_card[a] = cards[v]
        d.sum_card = cards[sum_var] if sum_var is not None else 1
        d.n_in = len(inputs)
        for k, f in enumerate(inputs):
            strides = {}
            s = 1
            for v in reversed(f.scope):
                strides[v] = s
                s *= cards[v]
            d.inp[k] = f.tensor.data_ptr()
            for a, v in enumerate(out_scope):
                d.in_stride[k][a] = strides.get(v, 0)
            d.sum_stride[k] = strides.get(sum_var, 0) if sum_var is not None else 0
        n_out = 1
        for v in out_scope:
            n_out *= cards[v]
        out = torch.empty(max(n_out, 1), dtype=torch.float32, device=self.t.device)
        d.out = out.data_ptr()
        d.normalize_last = 1 if normalize_last else 0
        d.log_space = 1 if self.log_space else 0
        if self.profile_compile:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if argmax is not None:
            N.check(N.lib().cbn_factor_contract_max(self.t.ctx.handle, C.byref(d), argmax.data_ptr(), N.stream_ptr(self.t.device)),
                    self.t.ctx.handle)
        else:
            N.check(N.lib().cbn_factor_contract(self.t.ctx.handle, C.byref(d), N.stream_ptr(self.t.device)), self.t.ctx.handle)
        if self.rescale and not normalize_last:
            # evidence axes are the slowest axes of every factor (sort_scope): one contiguous slice per evidence configuration
            lead = 0
            while lead < len(out_scope) and out_scope[lead] in self._ev_set:
                lead += 1
            n_slices = 1
            for v in out_scope[:lead]:
                n_slices *= cards[v]
            slice_size = max(n_out, 1) // max(n_slices, 1)
            if all(v not in self._ev_set for v in out_scope[lead:]):
                N.check(N.lib().cbn_factor_rescale(self.t.ctx.handle, out.data_ptr(), n_slices, slice_size,
                                                   1 if self.log_space else 0, N.stream_ptr(self.t.device)), self.t.ctx.handle)
        if self.profile_compile:
            e1.record()
            self._events.append((e0, e1))
        return Factor(out_scope, out)

    # ---------------------------------------------------------------- compile
    def compile(self, target: str, evidence: Sequence[str], do: Sequence[str] = (), dry: bool = False):
        """``do``: evidence variables that are set by intervention (graph surgery: their own CPT is dropped
        and their parents are cut off) -- the reference's ``infer(do=...)`` is a TODO (bayesian_network.py:229-232)."""
        t = self.t
        cards = t.cards
        T = t.index[target]
        E = [t.index[e] for e in evidence if e != target]      # evidence on the target itself is not forwarded
        D = set()                                               # (bayesian_network.py:190-196)
        for d in do or ():
            if d not in evidence:
                raise ValueError(f"do-variable {d} needs a value: pass it in the evidence dict as well")
            if d == target:
                raise ValueError("cannot intervene on the target node")
            D.add(t.index[d])
        key = (T, tuple(E), tuple(sorted(D)))
        if not dry and key in self._cache:
            return self._cache[key]
        if not dry:
            # structure-only pass first: a query that does not fit fails here, before any table is contracted
            self.compile(target, evidence, do=do, dry=True)
        Eset = set(E)
        self._ev_set = Eset
        if not dry:
            self._events = []
        order_key = {v: i for i, v in enumerate(E)}
        stats = PlanStats()

        def sort_scope(scope) -> List[int]:
            # evidence axes (plan order) first, then hidden, target last (fastest)
            return sorted(set(scope), key=lambda v: (2 if v == T else (0 if v in Eset else 1), order_key.get(v, v)))

        relevant = self._ancestors([T] + E, cut=D)
        stats.n_relevant = len(relevant)
        factors: List[Factor] = []
        for v in sorted(relevant):
            if v in D:
                continue
            scope = t.family_vars(t.names[v])
            tensor = None if dry else t.table_view(t.cond, t.names[v]).reshape(-1)
            if tensor is not None and self.log_space:
                tensor = torch.log(tensor)          # log 0 = -inf: a zero-probability entry stays one through sums and LSE
            factors.append(Factor(list(scope), tensor))
        hidden = [v for v in relevant if v not in Eset and v != T]
        stats.n_hidden = len(hidden)

        # connected components of the non-evidence variables (evidence instantiation cuts the graph)
        parent = {v: v for v in hidden + [T]}

        def find(a):
            while parent[a] != a:
                parent[a] = parent[parent[a]]
                a = parent[a]
            return a

        for f in factors:
            free = [v for v in f.scope if v not in Eset]
            for a, b in zip(free, free[1:]):
                parent[find(a)] = find(b)
        comp_t = find(T)
        in_t = lambda f: any(v not in Eset and find(v) == comp_t for v in f.scope)
        main = [f for f in factors if in_t(f)]
        rest = [f for f in factors if not in_t(f)]
        rel_ev = set()
        for f in main:
            rel_ev |= {v for v in f.scope if v in Eset}
        stats.relevant_evidence = [v for v in E if v in rel_ev]

        finals, left = self._eliminate(main, [v for v in hidden if find(v) == comp_t], sort_scope, stats, dry, T, partial=True)

        # support of the dropped part: a row whose (irrelevant) evidence has probability zero is all zeros in
        # the oracle's convention; only factors that can be zero matter
        if self.check_support and rest:
            if dry:
                stats.support_unchecked = True
            else:
                groups: Dict[int, List[Factor]] = {}
                consts: List[Factor] = []
                for f in rest:
                    free = [v for v in f.scope if v not in Eset]
                    (groups.setdefault(find(free[0]), []) if free else consts).append(f)
                # a constant (all-evidence) factor is a scalar table indexed by its own evidence axes
                for f in consts:
                    v = f.scope[-1]
                    if self._cond_has_zero(v):
                        finals.append(self._contract([f], sort_scope(f.scope), None, dry))
                for root, fs in groups.items():
                    owners = [f.scope[-1] for f in fs]
                    if not any(self._cond_has_zero(v) for v in owners):
                        continue
                    try:
                        sub = PlanStats()
                        res = self._eliminate(fs, [v for v in hidden if find(v) == root], sort_scope, sub, dry, T)
                        stats.contraction_madds += sub.contraction_madds
                        for r in res:
                            if bool((r.tensor == (float("-inf") if self.log_space else 0)).any().item()):
                                finals.append(r)
                    except PlanTooLarge:
                        stats.support_unchecked = True

        if left:
            # the boundary is too large to tabulate: the rest of the hidden variables is eliminated per row
            stats.per_row_hidden = len(left)
            stats.final_tables = [(tuple(f.scope), f.size(cards)) for f in finals]
            stats.per_row_slice_cells = sum(int(f.size(cards) // max(1, _prod(cards[v] for v in f.scope if v in Eset))) for f in finals)
            plan = self._row_plan(T, E, finals, left, stats, dry)
            if dry:
                return stats
            stats.contraction_gpu_ms = self._drain_events()
            self._cache[key] = plan
            return plan
        finals = self._merge_finals(finals, sort_scope, stats, dry, T)
        stats.final_tables = [(tuple(f.scope), f.size(cards)) for f in finals]
        if dry:
            return stats
        # a single pre-normalised target table needs no arithmetic per row
        normalize = True
        with_t = [f for f in finals if f.scope and f.scope[-1] == T]
        log_tables = self.log_space
        if len(finals) == 1 and len(with_t) == 1:
            # (in log space the normalising contraction returns the LINEAR distribution: the plan is an ordinary gather)
            finals = [self._contract(finals, finals[0].scope, None, dry, normalize_last=True)]
            normalize = False
            log_tables = False
        if not with_t:
            # target independent of everything kept (cannot happen: P(T|pa) always mentions T)
            raise RuntimeError("internal: no final factor mentions the target")
        stats.contraction_gpu_ms = self._drain_events()
        plan = QueryPlan(t, T, E, cards[T], finals, normalize, stats, log_space=log_tables)
        self._cache[key] = plan
        return plan

    # ---------------------------------------------------------------- evidence mode: log P(e)
    def compile_evidence(self, evidence_names: Sequence[str], dry: bool = False):
        """Compile ``log P(e)`` for the evidence set ``evidence_names`` (one value per row of every variable).

        Only ``ancestors(E)`` matter: barren descendants sum to 1.  A CPT whose scope lies inside ``E`` is a constant of
        the sum and goes to the observed-families kernel (``cbn_loglik_run``) with its variables remapped to evidence
        slots.  Every other CPT belongs to a component of hidden variables, and ALL components are eliminated completely
        (none is dropped as in the posterior compile): what is left are tables over evidence subsets only (card_t = 1),
        gathered by ``cbn_ve_run_codes_log_evidence``.  When the elimination exceeds the table budget the remaining
        hidden variables go to the per-row executor, as for posteriors.

        The elimination runs in log space WITHOUT range control: log-sum-exp contractions have no range problem in fp32,
        and dropping the per-slice rescaling is what keeps the normaliser.  The network's posterior plans keep their own
        configuration and cache; evidence plans are cached separately, keyed by the evidence tuple, and dropped when the
        tables are re-fitted.

        ``dry=True`` works on ``DryTables`` and returns the ``EvidenceSplit`` only (no device work)."""
        if not self.log_space or self.rescale:
            return self._evidence_child().compile_evidence(evidence_names, dry=dry)
        t = self.t
        cards = t.cards
        E = self._evidence_ids(evidence_names)
        key = tuple(E)
        if not dry:
            self._drop_stale_plans()
            if key in self._ev_cache:
                return self._ev_cache[key]
            # structure-only pass first: a query that does not fit fails here, before any table is contracted
            self.compile_evidence(evidence_names, dry=True)
            self._events = []
        Eset = set(E)
        self._ev_set = Eset
        order_key = {v: i for i, v in enumerate(E)}

        def sort_scope(scope) -> List[int]:
            # evidence axes (plan order) first, then hidden
            return sorted(set(scope), key=lambda v: (0 if v in Eset else 1, order_key.get(v, v)))

        stats = PlanStats()
        relevant = self._ancestors(E)
        stats.n_relevant = len(relevant)
        observed: List[int] = []
        factors: List[Factor] = []
        for v in sorted(relevant):
            scope = t.family_vars(t.names[v])
            if all(u in Eset for u in scope):
                observed.append(v)
                continue
            tensor = None if dry else t.table_view(t.log_cond, t.names[v]).reshape(-1)
            factors.append(Factor(list(scope), tensor))
        hidden = [v for v in sorted(relevant) if v not in Eset]
        stats.n_hidden = len(hidden)
        stats.relevant_evidence = list(E)
        ve_plan, per_row = None, False
        if factors:
            finals, left = self._eliminate(factors, hidden, sort_scope, stats, dry, None, partial=True)
            if left:
                per_row = True
                stats.per_row_hidden = len(left)
                stats.final_tables = [(tuple(f.scope), f.size(cards)) for f in finals]
                stats.per_row_slice_cells = sum(int(f.size(cards) // max(1, _prod(cards[v] for v in f.scope if v in Eset)))
                                                for f in finals)
                ve_plan = self._row_plan(None, E, finals, left, stats, dry)
            else:
                finals = self._merge_finals(finals, sort_scope, stats, dry, None)
                stats.final_tables = [(tuple(f.scope), f.size(cards)) for f in finals]
                if not dry:
                    ve_plan = QueryPlan(t, None, E, 1, finals, True, stats, log_space=True)
        split = EvidenceSplit(evidence=list(E), observed_families=observed, ve_stats=stats if factors else None,
                              per_row=per_row)
        if dry:
            return split
        stats.contraction_gpu_ms = self._drain_events()
        plan = EvidencePlan(t, E, observed, ve_plan, split)
        self._ev_cache[key] = plan
        return plan

    def _evidence_child(self) -> "VECompiler":
        """The evidence-mode compiler (log space, no range control, no support pruning) over the same tables."""
        if self._ev_child is None:
            self._ev_child = VECompiler(self.t, table_budget_cells=self.table_budget, merge_budget_cells=self.merge_budget,
                                        check_support=False, row_temp_floats=self.row_temp_floats, log_space=True,
                                        rescale=False, profile_compile=self.profile_compile,
                                        row_unit_layout=self.row_unit_layout, mpe_argmax_budget_bytes=self.mpe_argmax_budget)
        return self._ev_child

    def _evidence_ids(self, evidence_names: Sequence[str]) -> List[int]:
        t = self.t
        for e in evidence_names:
            if e not in t.index:
                raise ValueError(f"{e} is not a node of the network")
        E = [t.index[e] for e in evidence_names]
        if len(set(E)) != len(E):
            raise ValueError("an evidence variable is listed twice")
        return E

    def _drop_stale_plans(self):
        version = getattr(self.t, "cond_version", 0)
        if self._ev_cache_version != version:          # re-fitted tables: every cached plan is stale
            self._ev_cache = {}
            self._mpe_cache = {}
            self._ev_cache_version = version

    # ---------------------------------------------------------------- MPE mode: argmax_h P(h, e)
    def compile_mpe(self, evidence_names: Sequence[str], dry: bool = False):
        """Compile the most probable explanation for the evidence set ``evidence_names``: per row, the jointly most
        probable value of EVERY other node, ``argmax_h P(h, e)``, and ``log max_h P(h, e)``.

        The elimination of ``compile_evidence`` with max in place of log-sum-exp, over every CPT of the network (barren
        descendants are not summed out here: their values are part of the answer).  CPTs whose scope lies inside ``E`` go to
        the observed-families kernel.  Every hidden variable is eliminated by ``cbn_factor_contract_max``, which also
        records the argmax table of the step; what is left are tables over evidence subsets, so the value of a row is
        exactly what an ``EvidencePlan`` computes from them.  The traceback (``cbn_mpe_run``) decodes the hidden values
        in reverse elimination order.  There is no per-row executor for MPE: a step beyond the table budget, argmax tables
        beyond ``mpe_argmax_budget_bytes`` or a row of more than ``N.MPE_MAX_SLOTS`` codes raise ``PlanTooLarge`` in the
        structure-only pass, before any table is contracted.

        ``dry=True`` works on ``DryTables`` and returns the ``MPESplit`` only (no device work)."""
        if not self.log_space or self.rescale:
            return self._evidence_child().compile_mpe(evidence_names, dry=dry)
        t = self.t
        cards = t.cards
        E = self._evidence_ids(evidence_names)
        key = tuple(E)
        if not dry:
            self._drop_stale_plans()
            if key in self._mpe_cache:
                return self._mpe_cache[key]
            self.compile_mpe(evidence_names, dry=True)      # the limits fail here, before any table is contracted
            self._events = []
        Eset = set(E)
        self._ev_set = Eset
        order_key = {v: i for i, v in enumerate(E)}

        def sort_scope(scope) -> List[int]:
            return sorted(set(scope), key=lambda v: (0 if v in Eset else 1, order_key.get(v, v)))

        stats = PlanStats()
        stats.n_relevant = len(t.names)
        observed: List[int] = []
        factors: List[Factor] = []
        for v in range(len(t.names)):
            scope = t.family_vars(t.names[v])
            if all(u in Eset for u in scope):
                observed.append(v)
                continue
            tensor = None if dry else t.table_view(t.log_cond, t.names[v]).reshape(-1)
            factors.append(Factor(list(scope), tensor))
        hidden = [v for v in range(len(t.names)) if v not in Eset]
        stats.n_hidden = len(hidden)
        stats.relevant_evidence = list(E)
        elim: list = []
        finals: List[Factor] = []
        if factors:
            finals = self._eliminate(factors, hidden, sort_scope, stats, dry, None, decode=elim)
        argmax_bytes = sum(max(_prod(cards[u] for u in sc), 1) for _, sc, _ in elim)
        if dry:
            if argmax_bytes > self.mpe_argmax_budget:
                raise PlanTooLarge(f"the argmax tables of this explanation need {argmax_bytes} bytes "
                                   f"(budget {self.mpe_argmax_budget})")
            widest = max((len(sc) for _, sc, _ in elim), default=0)
            if widest > N.MAX_CONTRACT_DIMS:
                raise PlanTooLarge(f"an argmax table with {widest} axes exceeds {N.MAX_CONTRACT_DIMS}")
            ev_read = {u for _, sc, _ in elim for u in sc if u in Eset}
            if len(ev_read) + len(hidden) > N.MPE_MAX_SLOTS:
                raise PlanTooLarge(f"{len(ev_read)} evidence columns and {len(hidden)} hidden variables exceed the "
                                   f"{N.MPE_MAX_SLOTS} codes the traceback keeps per row")
        ve_plan = None
        if finals:
            finals = self._merge_finals(finals, sort_scope, stats, dry, None)
            stats.final_tables = [(tuple(f.scope), f.size(cards)) for f in finals]
            if not dry:
                ve_plan = QueryPlan(t, None, E, 1, finals, True, stats, log_space=True)
        decode = [(v, tuple(sc), am) for v, sc, am in reversed(elim)]
        split = MPESplit(evidence=list(E), hidden=hidden, observed_families=observed,
                         decode=[(v, sc) for v, sc, _ in decode], argmax_bytes=argmax_bytes, stats=stats)
        if dry:
            return split
        stats.contraction_gpu_ms = self._drain_events()
        value = EvidencePlan(t, E, observed, ve_plan,
                             EvidenceSplit(evidence=list(E), observed_families=observed, ve_stats=stats if factors else None))
        plan = MPEPlan(t, split, decode, value)
        self._mpe_cache[key] = plan
        return plan

    def _drain_events(self) -> float:
        if not self._events:
            return 0.0
        self._events[-1][1].synchronize()
        ms = sum(a.elapsed_time(b) for a, b in self._events)
        self._events = []
        return ms

    def _eliminate(self, factors: List[Factor], hidden: List[int], sort_scope, stats: PlanStats, dry: bool, T: int,
                   partial: bool = False, decode: Optional[list] = None):
        """Evidence-symbolic elimination.  With ``partial`` the loop stops when the cheapest step exceeds the table
        budget and returns ``(factors, remaining_hidden)`` for the per-row executor instead of raising.

        With a ``decode`` list the elimination is max-sum (log space): every step maximises over its variable and appends
        ``(variable, output scope, argmax table)`` to the list (the table is None in a dry run)."""
        cards = self.t.cards
        live: Dict[int, Factor] = dict(enumerate(factors))
        next_key = len(factors)
        g = _Greedy(cards, {k: f.scope for k, f in live.items()}, hidden)

        def cells(scope):
            s = 1
            for v in scope:
                s *= cards[v]
            return s

        while g.hidden:
            v, best_cost, best_scope = g.best()
            if best_cost > self.table_budget and partial:
                return list(live.values()), sorted(g.hidden)
            if best_cost > self.table_budget:
                raise PlanTooLarge(
                    f"eliminating the cheapest hidden variable needs a table of {best_cost} cells "
                    f"(budget {self.table_budget}); " +
                    ("the most probable explanation has no per-row executor" if decode is not None else
                     "this query needs the per-row executor"))
            keys = g.touching(v)
            touching = [live[k] for k in keys]
            # the kernel multiplies at most MAX_CONTRACT_INPUTS factors at once: pre-multiply the smallest ones
            while len(touching) > N.MAX_CONTRACT_INPUTS:
                order = sorted(range(len(touching)), key=lambda i: touching[i].size(cards))
                ia, ib = order[0], order[1]
                a, b = touching[ia], touching[ib]
                sc = sort_scope(a.scope + b.scope)
                if cells(sc) > self.table_budget:
                    raise PlanTooLarge("pre-multiplication exceeds the table budget")
                stats.contraction_madds += 2 * cells(sc)
                prod = self._contract([a, b], sc, None, dry)
                g.replace([keys[ia], keys[ib]], next_key, sc)
                for k in (keys[ia], keys[ib]):
                    del live[k]
                live[next_key] = prod
                keys = [k for i, k in enumerate(keys) if i not in (ia, ib)] + [next_key]
                touching = [f for i, f in enumerate(touching) if i not in (ia, ib)] + [prod]
                next_key += 1
            out_scope = sort_scope(best_scope)
            stats.n_steps += 1
            stats.max_table_cells = max(stats.max_table_cells, best_cost)
            stats.contraction_madds += best_cost * cards[v] * len(touching)
            if decode is not None:
                am = None if dry else torch.empty(max(best_cost, 1), dtype=torch.uint8, device=self.t.device)
                res = self._contract(touching, out_scope, v, dry, argmax=am)
                decode.append((v, out_scope, am))
            else:
                res = self._contract(touching, out_scope, v, dry)
            for k in keys:
                del live[k]
            live[next_key] = res
            g.eliminate(v, next_key, out_scope)
            next_key += 1
        out = list(live.values())
        return (out, []) if partial else out

    # ---------------------------------------------------------------- per-row schedule
    def _row_plan(self, T: int, E: List[int], statics: List[Factor], hidden: List[int], stats: PlanStats, dry: bool):
        """Schedule the elimination of ``hidden`` per row: evidence axes of the static tables are sliced by the
        row's codes, so only hidden axes (and the target) count towards the size of a temporary.

        Two passes.  The first fixes the elimination order and which factors meet in which step; the second chooses the
        LAYOUT of every factor.  A factor -- static table or temporary -- is consumed by exactly one step, so it is laid
        out for that step: the variable the step sums over innermost (stride 1), which is what the executor's unrolled
        step bodies need (csrc/ve.cu, ``row_step_unit``).  Static tables whose axes are in a different order are
        permuted once, here, at compile time."""
        import numpy as np

        cards = self.t.cards
        Eset = set(E)
        n_in = len(statics)
        MAXIN = N.MAX_CONTRACT_INPUTS

        def size_of(scope):
            return _prod(cards[v] for v in scope)

        # pass 1: (input keys, output key, output scope, summed variable or None)
        live = {k: [v for v in f.scope if v not in Eset] for k, f in enumerate(statics)}
        ops = []
        next_key = n_in
        g = _Greedy(cards, {k: list(sc) for k, sc in live.items()}, hidden)
        while g.hidden:
            v, _, sc = g.best()
            keys = list(g.touching(v))
            while len(keys) > MAXIN:                           # pre-multiply the two smallest
                order = sorted(range(len(keys)), key=lambda i: size_of(live[keys[i]]))
                ka, kb = keys[order[0]], keys[order[1]]
                psc = sorted(set(live[ka]) | set(live[kb]))
                ops.append(([ka, kb], next_key, psc, None))
                g.replace([ka, kb], next_key, psc)
                del live[ka], live[kb]
                live[next_key] = psc
                keys = [k for k in keys if k not in (ka, kb)] + [next_key]
                next_key += 1
            out_scope = sorted(sc)
            ops.append((keys, next_key, out_scope, v))
            for k in keys:
                del live[k]
            live[next_key] = out_scope
            g.eliminate(v, next_key, out_scope)
            next_key += 1
            stats.n_steps += 1
        rest = list(live.keys())
        # final product over what is left (free scope is empty or [T]; evidence mode has no target)
        last_scope = [T] if T is not None else []
        while len(rest) > MAXIN:
            ops.append((rest[:MAXIN], next_key, last_scope, None))
            rest = rest[MAXIN:] + [next_key]
            next_key += 1
        ops.append((rest, next_key, last_scope, None))

        # pass 2: layouts, offset tables, temporaries
        inner = {}                                             # factor key -> the variable its consumer sums over
        for keys, _, _, v in ops:
            for k in keys:
                inner[k] = v

        def lay_out(scope, key):
            v = inner.get(key) if self.row_unit_layout else None
            sc = sorted(scope, key=lambda a: (a == T, a))
            if v is not None and v in sc:
                sc.remove(v)
                sc.append(v)
            return sc

        def strides_of(scope):
            st, s = {}, 1
            for v in reversed(scope):
                st[v] = s
                s *= cards[v]
            return st

        laid = []                                              # the static tables as the executor reads them
        fac = {}                                               # key -> (input id, free scope, strides over the free axes)
        for k, f in enumerate(statics):
            free = [v for v in f.scope if v not in Eset]
            want = [v for v in f.scope if v in Eset] + lay_out(free, k) if self.row_unit_layout else list(f.scope)
            if want != list(f.scope):
                perm = [f.scope.index(v) for v in want]
                tensor = None
                if f.tensor is not None:
                    tensor = f.tensor.reshape([cards[v] for v in f.scope]).permute(perm).contiguous().reshape(-1)
                f = Factor(want, tensor)
            elif f.tensor is not None and f.tensor.data_ptr() % 16:
                f = Factor(list(f.scope), f.tensor.clone())    # a view into a packed buffer: realign for vector loads
            laid.append(f)
            st = strides_of(f.scope)
            fac[k] = (k, [v for v in f.scope if v not in Eset], {v: st[v] for v in f.scope if v not in Eset})
        steps, off_chunks, off_at, temp_total = [], [], 0, 0
        for keys, out_key, out_scope, sum_var in ops:
            inputs = [fac[k] for k in keys]
            out_scope = lay_out(out_scope, out_key)
            out_shape = [cards[v] for v in out_scope]
            out_size = _prod(out_shape)
            if temp_total + (out_size + 3) // 4 * 4 > self.row_temp_floats:
                raise PlanTooLarge(
                    f"per-row elimination needs more than {temp_total + out_size} floats of temporaries per row "
                    f"(budget {self.row_temp_floats}): the hidden part of this query has too large an induced width "
                    "for exact inference")
            offs = np.zeros((len(inputs), out_size), dtype=np.int64)
            grids = np.indices(out_shape).reshape(len(out_scope), -1) if out_scope else np.zeros((0, 1), dtype=np.int64)
            for k, (_, _, st) in enumerate(inputs):
                for d, v in enumerate(out_scope):
                    if v in st:
                        offs[k] += grids[d] * st[v]
            sum_card = cards[sum_var] if sum_var is not None else 1
            steps.append({"out_size": out_size, "sum_card": sum_card, "in_id": [i for i, _, _ in inputs],
                          "sum_stride": [st.get(sum_var, 0) if sum_var is not None else 0 for _, _, st in inputs],
                          "offsets_at": off_at})
            off_chunks.append(offs.astype(np.int32).reshape(-1))
            off_at += offs.size
            temp_total += (out_size + 3) // 4 * 4
            stats.contraction_madds += out_size * sum_card * len(inputs)
            stats.per_row_madds += out_size * sum_card * len(inputs)
            fac[out_key] = (n_in + len(steps) - 1, list(out_scope), strides_of(out_scope))
        offsets = np.ascontiguousarray(np.concatenate(off_chunks), dtype=np.int32)
        # the schedule as plain host data (what cbn_ve_plan_create_rows receives): kept for inspection and for the
        # CPU-side interpreter of tests/test_host_logic.py
        self.last_row_schedule = {"target": T, "evidence": list(E), "static_scopes": [list(f.scope) for f in laid],
                                  "static_source_scopes": [list(f.scope) for f in statics],
                                  "steps": steps, "offsets": offsets}
        if dry:
            return None
        return RowPlan(self.t, T, E, cards[T] if T is not None else 1, laid, steps, offsets, stats, self.log_space)

    def _merge_finals(self, finals: List[Factor], sort_scope, stats: PlanStats, dry: bool, T: int) -> List[Factor]:
        """Multiply final tables together while the product stays within the merge budget: fewer gathers
        per row, and a single table can be normalised at compile time."""
        cards = self.t.cards
        finals = [Factor(sort_scope(f.scope), f.tensor) if f.scope == sort_scope(f.scope) else
                  self._contract([f], sort_scope(f.scope), None, dry) for f in finals]

        def cells(scope):
            s = 1
            for v in scope:
                s *= cards[v]
            return s

        while len(finals) > 1:
            best = None
            for i in range(len(finals)):
                for j in range(i + 1, len(finals)):
                    sc = sort_scope(finals[i].scope + finals[j].scope)
                    c = cells(sc)
                    if best is None or c < best[0]:
                        best = (c, i, j, sc)
            c, i, j, sc = best
            if c > self.merge_budget and len(finals) <= N.MAX_GATHER_TABLES:
                break
            if c > self.table_budget:
                raise PlanTooLarge("cannot reduce the number of final tables within the budget")
            a, b = finals[i], finals[j]
            finals = [f for k, f in enumerate(finals) if k not in (i, j)]
            stats.contraction_madds += 2 * c
            stats.max_table_cells = max(stats.max_table_cells, c)
            finals.append(self._contract([a, b], sc, None, dry))
        return finals


class DryTables:
    """Structure-only stand-in for ``DiscreteTables`` (no device): lets the planner be
    exercised on a CPU-only machine with ``compile(..., dry=True)``."""

    def __init__(self, names, cards, parents_by_name):
        self.names = list(names)
        self.index = {n: i for i, n in enumerate(self.names)}
        self.cards = [int(c) for c in cards]
        self.parents = {n: list(parents_by_name.get(n, [])) for n in self.names}
        self.cond = None
        self.device = None
        self.ctx = None

    def family_vars(self, name):
        return [self.index[p] for p in self.parents[name]] + [self.index[name]]
