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
reverse elimination order.  With the sum kept and the conditional of every step recorded as cumulative thresholds
(``VECompiler.compile_posterior_sampler``), the same traceback with a random draw per step (``cbn_psample_run``) samples
the hidden values exactly from ``P(h | e)``.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field, replace
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _native as N


class PlanTooLarge(NotImplementedError):
    pass


def _cells(scope, cards) -> int:
    """Cells of a table over ``scope``."""
    return math.prod(cards[v] for v in scope)


def _strides(scope, cards) -> Dict[int, int]:
    """Variable -> stride of its axis in a row-major table over ``scope`` (last variable fastest)."""
    st, s = {}, 1
    for v in reversed(scope):
        st[v] = s
        s *= cards[v]
    return st


def _ld(ev_codes: torch.Tensor) -> int:
    """Leading dimension of an evidence code matrix (0 for a single row vector)."""
    return ev_codes.stride(0) if ev_codes.dim() == 2 else 0


def _int32s(values):
    return (C.c_int32 * max(len(values), 1))(*values)


@dataclass
class Factor:
    scope: List[int]                     # variable ids; tensor is row-major over this list
    tensor: Optional[torch.Tensor]       # float32 device tensor (None in dry-run)


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


class _NativePlan:
    """Owner of one native plan: ``handle`` is released by the C function ``_destroy`` when the owner is collected."""
    _destroy = "cbn_ve_plan_destroy"
    handle = None

    def __init__(self, tables_owner):
        self.owner = tables_owner
        self.ctx = tables_owner.ctx
        self.device = tables_owner.device

    def __del__(self):
        try:
            if self.handle is not None:
                getattr(N.lib(), self._destroy)(self.handle)
                self.handle = None
        except Exception:
            pass


class _VEPlan(_NativePlan):
    """What gather plans and per-row plans share: a ``cbn_ve_plan`` that answers ``target`` (None: ``log P(e)``) from the
    codes of ``evidence`` (row e of a code matrix = evidence variable e of the plan)."""

    def __init__(self, tables_owner, target: Optional[int], evidence: List[int], card_t: int, stats: PlanStats,
                 log_space: bool):
        super().__init__(tables_owner)
        self.target = target
        self.evidence = list(evidence)
        self.card_t = card_t
        self.stats = stats
        self.log_space = bool(log_space)           # the tables hold logarithms

    # bytes the kernel must move per row (SURVEY.md section 8d): relevant evidence codes in, posterior out
    def algorithmic_bytes_per_row(self) -> int:
        return len(self.stats.relevant_evidence) + 4 * self.card_t

    def set_static_evidence(self, on: bool = True):
        """Declare that the evidence of this plan's runs is never written by the kernel preceding the run on the same
        stream (resident batches replayed from a CUDA graph): evidence loads may then overlap the previous launch.  The
        per-row kernels do not use it."""
        N.check(N.lib().cbn_ve_plan_set_static_evidence(self.handle, 1 if on else 0), self.ctx.handle)

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """ev_codes: uint8 [len(evidence), ld] on the device (row e = evidence variable e of the plan)."""
        assert ev_codes.dtype == torch.uint8 and ev_codes.is_cuda
        if out is None:
            out = torch.empty((n_rows, self.card_t), dtype=torch.float32, device=self.device)
        N.check(N.lib().cbn_ve_run_codes(self.ctx.handle, self.handle, ev_codes.data_ptr(), _ld(ev_codes), int(n_rows),
                                         out.data_ptr(), N.stream_ptr(self.device)), self.ctx.handle)
        return out

    def run_codes_log_evidence(self, ev_codes: torch.Tensor, n_rows: int, out: torch.Tensor) -> torch.Tensor:
        """Float32 [n_rows]: the log of the sum over the plan's tables for each row (``log P(e_row)`` for a plan of
        ``VECompiler.compile_evidence``)."""
        N.check(N.lib().cbn_ve_run_codes_log_evidence(self.ctx.handle, self.handle, ev_codes.data_ptr(), _ld(ev_codes),
                                                      int(n_rows), out.data_ptr(), N.stream_ptr(self.device)),
                self.ctx.handle)
        return out

    def run_f32(self, ev_cols: Sequence[torch.Tensor], n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Float evidence columns: encoded on the device first (unseen values -> CBN_UNSEEN -> zero rows)."""
        return self.run_codes(self.owner.encode_evidence(self.evidence, ev_cols, n_rows), n_rows, out)


class QueryPlan(_VEPlan):
    """A compiled (target, evidence-set) query.  Owns the final tables and the native plan."""

    def __init__(self, tables_owner, target: int, evidence: List[int], card_t: int, finals: List[Factor],
                 normalize: bool, stats: PlanStats, log_space: bool = False):
        super().__init__(tables_owner, target, evidence, card_t, stats, log_space)
        self.finals = finals
        self.normalize = normalize
        cards = tables_owner.cards
        slot = {v: i for i, v in enumerate(self.evidence)}
        arr = (N.GatherTable * len(finals))()
        for k, f in enumerate(finals):
            has_t = bool(f.scope) and f.scope[-1] == target
            ev_scope = f.scope[:-1] if has_t else f.scope
            stride = _strides(f.scope, cards)
            g = arr[k]
            g.data = f.tensor.data_ptr()
            g.n_cells = f.tensor.numel()
            g.n_ev = len(ev_scope)
            g.has_target = 1 if has_t else 0
            for j, v in enumerate(ev_scope):
                g.ev_slot[j] = slot[v]
                g.ev_stride[j] = stride[v]
        h = C.c_void_p()
        N.check(N.lib().cbn_ve_plan_create_gather(self.ctx.handle, len(self.evidence), _int32s([cards[v] for v in self.evidence]),
                                                  card_t, arr, len(finals),
                                                  (N.GATHER_NORMALIZE if normalize else 0) | (N.GATHER_LOG_SPACE if log_space else 0),
                                                  N.stream_ptr(self.device), C.byref(h)), self.ctx.handle)
        self.handle = h

    def run_f32(self, ev_cols: Sequence[torch.Tensor], n_rows: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """ev_cols[e]: float32 device column of evidence variable e (the reference's [nq,1] tensors)."""
        if self.card_t > N.GATHER_MAX_CT or len(self.evidence) > N.MAX_EVIDENCE_PTRS:
            # wide targets / very many evidence columns: the float kernel keeps the posterior in registers and takes its
            # column pointers as kernel arguments; encode on the device and use the code kernels (any cardinality)
            return super().run_f32(ev_cols, n_rows, out)
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
        N.check(N.lib().cbn_ve_run_codes_map(self.ctx.handle, self.handle, ev_codes.data_ptr(), _ld(ev_codes), int(n_rows),
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


class FusedPlan(_NativePlan):
    """Several targets over the same evidence list answered by ONE launch: the evidence codes are read once
    and every target's posterior is written (``cbn_ve_plan_fuse`` / ``cbn_ve_run_codes_multi``)."""

    def __init__(self, plans: Sequence[QueryPlan]):
        assert len(plans) >= 1
        super().__init__(plans[0].owner)
        self.plans = list(plans)            # keep the tables alive
        self.card_t = plans[0].card_t
        arr = N.ptr_array([p.handle.value for p in plans])
        h = C.c_void_p()
        N.check(N.lib().cbn_ve_plan_fuse(self.ctx.handle, arr, len(plans), N.stream_ptr(self.device), C.byref(h)), self.ctx.handle)
        self.handle = h
        self.n_out = N.lib().cbn_ve_plan_outputs(h)

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
        N.check(N.lib().cbn_ve_run_codes_multi(self.ctx.handle, self.handle, ev_codes.data_ptr(), _ld(ev_codes), int(n_rows),
                                               ptrs, N.stream_ptr(self.device)), self.ctx.handle)
        return list(outs)

    def run_codes_host(self, ev_codes_host: torch.Tensor, n_rows: int, outs_host: Sequence[torch.Tensor], compact: bool = False):
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


class RowPlan(_VEPlan):
    """A query whose evidence boundary is too large to tabulate: static tables for what could be eliminated at
    compile time + a per-row schedule of product / sum-out steps (``cbn_ve_plan_create_rows``)."""

    def __init__(self, tables_owner, target: int, evidence: List[int], card_t: int, inputs: List[Factor],
                 steps: List[dict], offsets, stats: PlanStats, log_space: bool):
        super().__init__(tables_owner, target, evidence, card_t, stats, log_space)
        self.inputs = inputs            # keep the tables alive
        self.offsets = offsets          # host int32 array (numpy): copied into the plan at creation
        cards = tables_owner.cards
        slot = {v: i for i, v in enumerate(self.evidence)}
        ins = (N.RowInput * len(inputs))()
        for k, f in enumerate(inputs):
            stride = _strides(f.scope, cards)
            ev_axes = [(slot[v], stride[v]) for v in reversed(f.scope) if v in slot]
            ins[k].data = f.tensor.data_ptr()
            ins[k].n_cells = f.tensor.numel()
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
        h = C.c_void_p()
        N.check(N.lib().cbn_ve_plan_create_rows(self.ctx.handle, len(self.evidence), _int32s([cards[v] for v in self.evidence]),
                                                card_t, ins, len(inputs), sts, len(steps), N.ROWS_LOG_SPACE if log_space else 0,
                                                N.stream_ptr(self.device), C.byref(h)), self.ctx.handle)
        self.handle = h


@dataclass
class EvidenceSplit:
    """How ``VECompiler.compile_evidence`` splits ``log P(e)``: the families summed by the observed-families kernel
    (network ids of the CPT owners) and the statistics of the VE plan for the rest (None: there is no rest)."""
    evidence: List[int]
    observed_families: List[int]
    ve_stats: Optional[PlanStats]
    per_row: bool = False


class LogLikPlan(_NativePlan):
    """Owner of a ``cbn_loglik_plan``: ``out[row] (+)= sum_f log cond_f[index_f(row)]`` over families whose variables are
    all columns of the code matrix handed to ``run`` (``columns[v]``: the column of network variable v)."""
    _destroy = "cbn_loglik_plan_destroy"

    def __init__(self, tables_owner, families: Sequence[int], columns: Dict[int, int], n_cols: int):
        super().__init__(tables_owner)
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
        if self.ve_plan is not None:
            self.ve_plan.run_codes_log_evidence(ev_codes, n_rows, out)
        if self.loglik is not None:
            self.loglik.run(ev_codes, n_rows, out, accumulate=self.ve_plan is not None)
        elif self.ve_plan is None:          # no evidence: log 1
            out.zero_()
        return out


@dataclass
class DecodeSplit:
    """Structure of a traceback plan over every hidden variable: the most probable explanation
    (``VECompiler.compile_mpe``, ``MPESplit``) or posterior sampling (``VECompiler.compile_posterior_sampler``)."""
    evidence: List[int]
    hidden: List[int]                                   # network ids; row h of the decoded code matrix is hidden[h]
    observed_families: List[int]                        # CPTs scored by the observed-families kernel
    decode: List[Tuple[int, Tuple[int, ...]]]           # (variable, scope of its table) in decode order
    table_bytes: int                                    # argmax (uint8) or threshold (float) tables of every step
    stats: PlanStats


class MPESplit(DecodeSplit):
    @property
    def argmax_bytes(self) -> int:
        return self.table_bytes


class _TracebackPlan(_NativePlan):
    """What MPE and posterior-sampling plans share: the tables of the elimination (read by the native plan, so they are
    kept alive with it), the native plan with one step per hidden variable in decode order (``_create``, steps of type
    ``_step`` whose table pointer is the field ``_table``), and the ``EvidencePlan`` over the final tables, which gives
    each row's value."""
    _create = _step = _table = None

    def __init__(self, tables_owner, split: DecodeSplit, decode, value: EvidencePlan):
        super().__init__(tables_owner)
        self.split = split
        self.evidence = list(split.evidence)
        self.hidden = list(split.hidden)
        self.value = value
        self.tables = [tb for _, _, tb in decode]
        cards = tables_owner.cards
        n_ev = len(self.evidence)
        slot = {v: i for i, v in enumerate(self.evidence)}
        slot.update({v: n_ev + h for h, v in enumerate(self.hidden)})
        if not self.hidden:
            return
        steps = (self._step * len(decode))()
        for k, (v, scope, tb) in enumerate(decode):
            st = steps[k]
            st.slot = slot[v]
            st.card = cards[v]
            setattr(st, self._table, tb.data_ptr())
            st.n_cells = _cells(scope, cards)
            st.n_ctx = len(scope)
            stride = _strides(scope, cards)
            for j, u in enumerate(scope):
                st.ctx_slot[j] = slot[u]
                st.ctx_stride[j] = stride[u]
            self._step_var(st, v)
        h = C.c_void_p()
        N.check(getattr(N.lib(), self._create)(self.ctx.handle, n_ev, _int32s([cards[v] for v in self.evidence]),
                                               len(self.hidden), steps, len(decode), N.stream_ptr(self.device), C.byref(h)),
                self.ctx.handle)
        self.handle = h

    def _step_var(self, step, v: int):
        pass

    def set_static_evidence(self, on: bool = True):
        self.value.set_static_evidence(on)


class MPEPlan(_TracebackPlan):
    """A compiled most probable explanation: the argmax tables of the max-sum elimination, the native traceback plan
    (``cbn_mpe_plan_create``) and the ``EvidencePlan`` that computes each row's value ``log max_h P(h, e)``."""
    _destroy, _create, _step, _table = "cbn_mpe_plan_destroy", "cbn_mpe_plan_create", N.MpeStep, "argmax"

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, hidden_out: Optional[torch.Tensor] = None,
                  value_out: Optional[torch.Tensor] = None):
        """ev_codes: uint8 [len(evidence), ld] on the device (row e = evidence variable e of the plan, ld a multiple of
        16).  Returns ``(hidden_codes, log_value)``: uint8 [len(hidden), ld'] (row h = network variable ``hidden[h]``,
        CBN_UNSEEN in every row whose value is -inf) and float32 [n_rows] ``log max_h P(h, e_row)``."""
        assert ev_codes.dtype == torch.uint8 and ev_codes.is_cuda
        value = self.value.run_codes(ev_codes, n_rows, value_out)
        if hidden_out is None:
            hidden_out = self.owner.new_code_matrix(n_rows, len(self.hidden))
        if self.handle is not None and n_rows > 0:
            N.check(N.lib().cbn_mpe_run(self.ctx.handle, self.handle, ev_codes.data_ptr(), _ld(ev_codes), int(n_rows),
                                        value.data_ptr(), hidden_out.data_ptr(), hidden_out.stride(0), N.stream_ptr(self.device)),
                    self.ctx.handle)
        return hidden_out, value


class PosteriorSamplePlan(_TracebackPlan):
    """A compiled posterior sampler: the threshold tables of the sum-product elimination, the native backward-sampling
    plan (``cbn_psample_plan_create``) and the ``EvidencePlan`` that computes each row's ``log P(e)``."""
    _destroy, _create, _step, _table = "cbn_psample_plan_destroy", "cbn_psample_plan_create", N.PsampleStep, "cdf"

    def _step_var(self, step, v: int):
        step.var = v

    def run_codes(self, ev_codes: torch.Tensor, n_rows: int, n_draws: int = 1, seed: int = 0, first_row: int = 0,
                  hidden_out: Optional[torch.Tensor] = None, value_out: Optional[torch.Tensor] = None):
        """ev_codes: uint8 [len(evidence), ld] on the device (row e = evidence variable e of the plan, ld a multiple of
        16).  Returns ``(hidden_codes, log_evidence)``: uint8 [n_draws * len(hidden), ld'], row ``d * len(hidden) + h``
        holding draw d of network variable ``hidden[h]`` (CBN_UNSEEN in every row whose ``log P(e)`` is -inf), and float32
        [n_rows] ``log P(e_row)``.  Draw d of row i depends only on ``(seed, first_row + i, d)``."""
        assert ev_codes.dtype == torch.uint8 and ev_codes.is_cuda
        value = self.value.run_codes(ev_codes, n_rows, value_out)
        if hidden_out is None:
            hidden_out = self.owner.new_code_matrix(n_rows, max(int(n_draws) * len(self.hidden), 1))
        if self.handle is not None and n_rows > 0:
            N.check(N.lib().cbn_psample_run(self.ctx.handle, self.handle, ev_codes.data_ptr(), _ld(ev_codes), int(n_rows),
                                            value.data_ptr(), int(seed) & ((1 << 64) - 1), int(first_row), int(n_draws),
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


@dataclass
class _Pass:
    """One pass of a compile: the arithmetic of its contractions and the state that lives only as long as the pass.

    ``log_space``: the factors hold logarithms (log-sum-exp or max-sum contractions).  ``rescale``: range control of
    linear-space elimination -- after every contraction each evidence slice of the result is divided by its maximum
    (``cbn_factor_rescale``), a factor of the evidence configuration only, which cancels in the final normalisation, so
    products of many small likelihoods stay inside the fp32 range.  ``dry``: structure only, no device work.
    ``reduce``: the reduction of the elimination steps that record a table for a traceback -- ``"max"`` (max-sum, argmax
    tables: MPE) or ``"cdf"`` (log-sum-exp, cumulative conditionals: posterior sampling); ``"sum"`` records none."""
    E: List[int]                                        # evidence ids, in plan order
    T: Optional[int]                                    # the target (None: log P(e) and MPE)
    dry: bool
    log_space: bool
    rescale: bool
    reduce: str = "sum"
    stats: PlanStats = field(default_factory=PlanStats)
    events: list = field(default_factory=list)          # CUDA events around every contraction (profile_compile)

    def __post_init__(self):
        self.ev = set(self.E)
        self._order = {v: i for i, v in enumerate(self.E)}

    def sort_scope(self, scope) -> List[int]:
        # evidence axes (plan order) first, then hidden, target last (fastest)
        return sorted(set(scope), key=lambda v: (2 if v == self.T else (0 if v in self.ev else 1), self._order.get(v, v)))

    def device_ms(self) -> float:
        if not self.events:
            return 0.0
        self.events[-1][1].synchronize()
        return sum(a.elapsed_time(b) for a, b in self.events)


class VECompiler:
    """Lower (target, evidence set) to a gather plan over a fitted ``DiscreteTables``."""

    def __init__(self, tables, table_budget_cells: int = 1 << 28, merge_budget_cells: int = 1 << 24,
                 check_support: bool = True, row_temp_floats: int = 5000, log_space: bool = False, rescale: bool = True,
                 profile_compile: bool = False, row_unit_layout: bool = True, mpe_argmax_budget_bytes: int = 1 << 30,
                 sample_table_budget_bytes: int = 1 << 30):
        self.t = tables
        self.log_space = bool(log_space)                 # arithmetic of posterior compiles (see _Pass)
        self.rescale = bool(rescale)
        self.profile_compile = bool(profile_compile)      # CUDA events around every contraction -> PlanStats.contraction_gpu_ms
        self.table_budget = int(table_budget_cells)
        self.merge_budget = int(merge_budget_cells)
        self.check_support = check_support
        self.row_temp_floats = int(row_temp_floats)     # per-row temporaries of the per-row executor (shared memory)
        self.row_unit_layout = bool(row_unit_layout)    # lay every per-row factor out with its consumer's summed variable innermost
        self.mpe_argmax_budget = int(mpe_argmax_budget_bytes)    # argmax tables of one MPE plan, in bytes
        self.sample_table_budget = int(sample_table_budget_bytes)    # threshold tables of one posterior sampler, in bytes
        self._plans: Dict[tuple, object] = {}           # (mode, key) -> plan
        self.structures: Dict[tuple, object] = {}       # host schedules that depend on the graph only (kept across CPTs)
        self._plans_version = None
        self._has_zero: Dict[int, bool] = {}
        self.last_row_schedule: Optional[dict] = None

    def cached(self, key: tuple, build):
        """The plan stored under ``key``, built by ``build()`` when missing.  Every plan and the zero-entry memo derive from
        the CPTs: all are dropped together when the tables' ``cond_version`` changes."""
        version = getattr(self.t, "cond_version", 0)
        if self._plans_version != version:
            self._plans, self._has_zero, self._plans_version = {}, {}, version
        if key not in self._plans:
            self._plans[key] = build()
        return self._plans[key]

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

    def _evidence_ids(self, evidence_names: Sequence[str]) -> List[int]:
        t = self.t
        for e in evidence_names:
            if e not in t.index:
                raise ValueError(f"{e} is not a node of the network")
        E = [t.index[e] for e in evidence_names]
        if len(set(E)) != len(E):
            raise ValueError("an evidence variable is listed twice")
        return E

    # ---------------------------------------------------------------- device contraction
    def _contract(self, inputs: List[Factor], out_scope: List[int], sum_var: Optional[int], cx: _Pass,
                  normalize_last: bool = False, table: Optional[torch.Tensor] = None) -> Factor:
        """``table``: the traceback table of this step, reduced by ``cx.reduce`` (log space) -- ``"max"``: maximise over
        ``sum_var`` instead of summing and record the maximising value of every output cell (uint8 [cells],
        ``cbn_factor_contract_max``); ``"cdf"``: sum as usual and record the conditional of ``sum_var`` given every output
        cell as cumulative thresholds (float32 [cells, card - 1], ``cbn_factor_contract_cdf``)."""
        cards = self.t.cards
        if cx.dry:
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
            strides = _strides(f.scope, cards)
            d.inp[k] = f.tensor.data_ptr()
            for a, v in enumerate(out_scope):
                d.in_stride[k][a] = strides.get(v, 0)
            d.sum_stride[k] = strides.get(sum_var, 0) if sum_var is not None else 0
        n_out = _cells(out_scope, cards)
        out = torch.empty(max(n_out, 1), dtype=torch.float32, device=self.t.device)
        d.out = out.data_ptr()
        d.normalize_last = 1 if normalize_last else 0
        d.log_space = 1 if cx.log_space else 0
        if self.profile_compile:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if table is not None:
            fn = N.lib().cbn_factor_contract_max if cx.reduce == "max" else N.lib().cbn_factor_contract_cdf
            N.check(fn(self.t.ctx.handle, C.byref(d), table.data_ptr(), N.stream_ptr(self.t.device)), self.t.ctx.handle)
        else:
            N.check(N.lib().cbn_factor_contract(self.t.ctx.handle, C.byref(d), N.stream_ptr(self.t.device)), self.t.ctx.handle)
        if cx.rescale and not normalize_last:
            # evidence axes are the slowest axes of every factor (sort_scope): one contiguous slice per evidence configuration
            lead = 0
            while lead < len(out_scope) and out_scope[lead] in cx.ev:
                lead += 1
            n_slices = _cells(out_scope[:lead], cards)
            slice_size = max(n_out, 1) // max(n_slices, 1)
            if all(v not in cx.ev for v in out_scope[lead:]):
                N.check(N.lib().cbn_factor_rescale(self.t.ctx.handle, out.data_ptr(), n_slices, slice_size,
                                                   1 if cx.log_space else 0, N.stream_ptr(self.t.device)), self.t.ctx.handle)
        if self.profile_compile:
            e1.record()
            cx.events.append((e0, e1))
        return Factor(out_scope, out)

    # ---------------------------------------------------------------- compile front end
    def _compile(self, mode: str, key: tuple, E: List[int], T: Optional[int], dry: bool, build,
                 log_space: bool = True, rescale: bool = False, reduce: str = "sum"):
        """Run ``build(pass)`` -- the part of the compile that is the mode's own -- as a structure-only pass (``dry``), or
        return the cached plan of ``(mode, key)``.  A plan is compiled after a structure-only pass: a query that does not
        fit fails there, before any table is contracted.  The default arithmetic is that of ``log P(e)`` and MPE: log space
        without range control."""
        if dry:
            return build(_Pass(E, T, True, log_space, rescale, reduce))

        def compile_plan():
            build(_Pass(E, T, True, log_space, rescale, reduce))
            cx = _Pass(E, T, False, log_space, rescale, reduce)
            plan = build(cx)
            cx.stats.contraction_gpu_ms = cx.device_ms()
            return plan

        return self.cached((mode, key), compile_plan)

    def _factors(self, cx: _Pass, owners, split_observed: bool):
        """The CPTs of ``owners`` as factors (their logarithms in log space) and, with ``split_observed``, apart from them
        the owners whose whole family is evidence: constants of the row, summed by the observed-families kernel."""
        t = self.t
        src = None if cx.dry else (t.log_cond if cx.log_space else t.cond)
        factors, observed = [], []
        for v in owners:
            scope = t.family_vars(t.names[v])
            if split_observed and all(u in cx.ev for u in scope):
                observed.append(v)
            else:
                factors.append(Factor(list(scope), None if src is None else t.table_view(src, t.names[v]).reshape(-1)))
        return factors, observed

    def _tail(self, cx: _Pass, finals: List[Factor], left: List[int]):
        """The plan over what the compile-time elimination leaves: a per-row plan when hidden variables are ``left``, else a
        gather over the merged final tables.  Fills the statistics of either; returns None in a dry pass."""
        cards, stats = self.t.cards, cx.stats
        if left:
            # the boundary is too large to tabulate: the rest of the hidden variables is eliminated per row
            stats.per_row_hidden = len(left)
            stats.final_tables = [(tuple(f.scope), _cells(f.scope, cards)) for f in finals]
            stats.per_row_slice_cells = sum(_cells(f.scope, cards) // _cells([v for v in f.scope if v in cx.ev], cards)
                                            for f in finals)
            return self._row_plan(cx, finals, left)
        finals = self._merge_finals(cx, finals)
        stats.final_tables = [(tuple(f.scope), _cells(f.scope, cards)) for f in finals]
        if cx.dry:
            return None
        T, normalize, log_tables = cx.T, True, cx.log_space
        if T is not None:
            with_t = [f for f in finals if f.scope and f.scope[-1] == T]
            if not with_t:
                # target independent of everything kept (cannot happen: P(T|pa) always mentions T)
                raise RuntimeError("internal: no final factor mentions the target")
            if len(finals) == 1:
                # a single pre-normalised target table needs no arithmetic per row (in log space the normalising
                # contraction returns the LINEAR distribution: the plan is an ordinary gather)
                finals = [self._contract(finals, finals[0].scope, None, cx, normalize_last=True)]
                normalize, log_tables = False, False
        return QueryPlan(self.t, T, cx.E, cards[T] if T is not None else 1, finals, normalize, stats, log_space=log_tables)

    # ---------------------------------------------------------------- posterior: P(T | e)
    def compile(self, target: str, evidence: Sequence[str], do: Sequence[str] = (), dry: bool = False):
        """``do``: evidence variables that are set by intervention (graph surgery: their own CPT is dropped
        and their parents are cut off) -- the reference's ``infer(do=...)`` is a TODO (bayesian_network.py:229-232)."""
        t = self.t
        T = t.index[target]
        E = [t.index[e] for e in evidence if e != target]      # evidence on the target itself is not forwarded
        D = set()                                               # (bayesian_network.py:190-196)
        for d in do or ():
            if d not in evidence:
                raise ValueError(f"do-variable {d} needs a value: pass it in the evidence dict as well")
            if d == target:
                raise ValueError("cannot intervene on the target node")
            D.add(t.index[d])
        return self._compile("posterior", (T, tuple(E), tuple(sorted(D))), E, T, dry, lambda cx: self._posterior(cx, D),
                             log_space=self.log_space, rescale=self.rescale)

    def _posterior(self, cx: _Pass, D: set):
        T, Eset, stats = cx.T, cx.ev, cx.stats
        relevant = self._ancestors([T] + cx.E, cut=D)
        stats.n_relevant = len(relevant)
        factors, _ = self._factors(cx, sorted(relevant - D), split_observed=False)
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
        stats.relevant_evidence = [v for v in cx.E if v in rel_ev]

        finals, left = self._eliminate(cx, main, [v for v in hidden if find(v) == comp_t], partial=True)

        # support of the dropped part: a row whose (irrelevant) evidence has probability zero is all zeros in
        # the oracle's convention; only factors that can be zero matter
        if self.check_support and rest:
            if cx.dry:
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
                        finals.append(self._contract([f], cx.sort_scope(f.scope), None, cx))
                for root, fs in groups.items():
                    owners = [f.scope[-1] for f in fs]
                    if not any(self._cond_has_zero(v) for v in owners):
                        continue
                    try:
                        sub = replace(cx, stats=PlanStats())        # the same pass; only its multiply-adds are counted
                        res = self._eliminate(sub, fs, [v for v in hidden if find(v) == root])
                        stats.contraction_madds += sub.stats.contraction_madds
                        for r in res:
                            if bool((r.tensor == (float("-inf") if cx.log_space else 0)).any().item()):
                                finals.append(r)
                    except PlanTooLarge:
                        stats.support_unchecked = True

        plan = self._tail(cx, finals, left)
        return stats if cx.dry else plan

    # ---------------------------------------------------------------- evidence mode: log P(e)
    def compile_evidence(self, evidence_names: Sequence[str], dry: bool = False):
        """Compile ``log P(e)`` for the evidence set ``evidence_names`` (one value per row of every variable).

        Only ``ancestors(E)`` matter: barren descendants sum to 1.  A CPT whose scope lies inside ``E`` is a constant of
        the sum and goes to the observed-families kernel (``cbn_loglik_run``) with its variables remapped to evidence
        slots.  Every other CPT belongs to a component of hidden variables, and ALL components are eliminated completely
        (none is dropped as in the posterior compile): what is left are tables over evidence subsets only (card_t = 1),
        gathered by ``cbn_ve_run_codes_log_evidence``.  When the elimination exceeds the table budget the remaining
        hidden variables go to the per-row executor, as for posteriors.

        The elimination runs in log space WITHOUT range control, whatever the posterior configuration: log-sum-exp
        contractions have no range problem in fp32, and dropping the per-slice rescaling is what keeps the normaliser.
        Plans are cached, keyed by the evidence tuple, and dropped when the tables are re-fitted.

        ``dry=True`` works on ``DryTables`` and returns the ``EvidenceSplit`` only (no device work)."""
        E = self._evidence_ids(evidence_names)
        return self._compile("evidence", tuple(E), E, None, dry, self._evidence)

    def _evidence(self, cx: _Pass):
        stats = cx.stats
        relevant = sorted(self._ancestors(cx.E))
        stats.n_relevant = len(relevant)
        factors, observed = self._factors(cx, relevant, split_observed=True)
        hidden = [v for v in relevant if v not in cx.ev]
        stats.n_hidden = len(hidden)
        stats.relevant_evidence = list(cx.E)
        ve_plan, left = None, []
        if factors:
            finals, left = self._eliminate(cx, factors, hidden, partial=True)
            ve_plan = self._tail(cx, finals, left)
        split = EvidenceSplit(evidence=list(cx.E), observed_families=observed, ve_stats=stats if factors else None,
                              per_row=bool(left))
        return split if cx.dry else EvidencePlan(self.t, cx.E, observed, ve_plan, split)

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
        E = self._evidence_ids(evidence_names)
        return self._compile("mpe", tuple(E), E, None, dry, self._traceback, reduce="max")

    # ---------------------------------------------------------------- posterior sampling: h ~ P(h | e)
    def compile_posterior_sampler(self, evidence_names: Sequence[str], dry: bool = False):
        """Compile exact sampling from ``P(h | e)`` for the evidence set ``evidence_names``: per row and draw, a value of
        EVERY other node drawn jointly from its posterior, and the row's ``log P(e)``.

        Forward filtering, backward sampling over the elimination of ``compile_mpe`` (same order, every CPT of the
        network) with the sum kept: ``cbn_factor_contract_cdf`` eliminates each hidden variable ``v_k`` by log-sum-exp and
        records ``P(v_k | ctx_k)`` -- its touching factors over their log-sum-exp -- as cumulative thresholds per context.
        What is left are tables over evidence subsets, whose ``EvidencePlan`` gives ``log P(e)``.  The traceback
        (``cbn_psample_run``) draws the variables in reverse elimination order, each from the thresholds of a context that
        is evidence or was drawn before it, so the draws follow ``prod_k P(v_k | ctx_k) = P(h | e)``.  The limits are those
        of MPE, with the threshold tables bounded by ``sample_table_budget_bytes``; all raise ``PlanTooLarge`` in the
        structure-only pass.

        ``dry=True`` works on ``DryTables`` and returns the ``DecodeSplit`` only (no device work)."""
        E = self._evidence_ids(evidence_names)
        return self._compile("psample", tuple(E), E, None, dry, self._traceback, reduce="cdf")

    def _traceback(self, cx: _Pass):
        """The part of ``compile_mpe`` and ``compile_posterior_sampler`` that is theirs: every hidden variable is eliminated
        with its table recorded (``cx.reduce``), then the tables are handed to the traceback in decode order."""
        t, cards, stats = self.t, self.t.cards, cx.stats
        sampling = cx.reduce == "cdf"
        every = range(len(t.names))
        stats.n_relevant = len(t.names)
        factors, observed = self._factors(cx, every, split_observed=True)
        hidden = [v for v in every if v not in cx.ev]
        stats.n_hidden = len(hidden)
        stats.relevant_evidence = list(cx.E)
        elim: list = []
        finals = self._eliminate(cx, factors, hidden, decode=elim) if factors else []
        if sampling:
            table_bytes = sum(4 * _cells(sc, cards) * (cards[v] - 1) for v, sc, _ in elim)
            budget, what = self.sample_table_budget, "the threshold tables of this sampler"
        else:
            table_bytes = sum(max(_cells(sc, cards), 1) for _, sc, _ in elim)
            budget, what = self.mpe_argmax_budget, "the argmax tables of this explanation"
        if cx.dry:
            if table_bytes > budget:
                raise PlanTooLarge(f"{what} need {table_bytes} bytes (budget {budget})")
            widest = max((len(sc) for _, sc, _ in elim), default=0)
            if widest > N.MAX_CONTRACT_DIMS:
                raise PlanTooLarge(f"{'a threshold' if sampling else 'an argmax'} table with {widest} axes exceeds "
                                   f"{N.MAX_CONTRACT_DIMS}")
            ev_read = {u for _, sc, _ in elim for u in sc if u in cx.ev}
            if len(ev_read) + len(hidden) > N.MPE_MAX_SLOTS:
                raise PlanTooLarge(f"{len(ev_read)} evidence columns and {len(hidden)} hidden variables exceed the "
                                   f"{N.MPE_MAX_SLOTS} codes the traceback keeps per row")
        ve_plan = self._tail(cx, finals, []) if finals else None
        decode = [(v, tuple(sc), tb) for v, sc, tb in reversed(elim)]
        split = (DecodeSplit if sampling else MPESplit)(
            evidence=list(cx.E), hidden=hidden, observed_families=observed, decode=[(v, sc) for v, sc, _ in decode],
            table_bytes=table_bytes, stats=stats)
        if cx.dry:
            return split
        value = EvidencePlan(t, cx.E, observed, ve_plan,
                             EvidenceSplit(evidence=list(cx.E), observed_families=observed, ve_stats=stats if factors else None))
        return (PosteriorSamplePlan if sampling else MPEPlan)(t, split, decode, value)

    # ---------------------------------------------------------------- elimination
    def _eliminate(self, cx: _Pass, factors: List[Factor], hidden: List[int], partial: bool = False,
                   decode: Optional[list] = None):
        """Evidence-symbolic elimination.  With ``partial`` the loop stops when the cheapest step exceeds the table
        budget and returns ``(factors, remaining_hidden)`` for the per-row executor instead of raising.

        With a ``decode`` list every step records its traceback table, reduced by ``cx.reduce`` (see ``_contract``), and
        appends ``(variable, output scope, table)`` to the list (the table is None in a dry run)."""
        cards, stats = self.t.cards, cx.stats
        live: Dict[int, Factor] = dict(enumerate(factors))
        next_key = len(factors)
        g = _Greedy(cards, {k: f.scope for k, f in live.items()}, hidden)
        while g.hidden:
            v, best_cost, best_scope = g.best()
            if best_cost > self.table_budget and partial:
                return list(live.values()), sorted(g.hidden)
            if best_cost > self.table_budget:
                raise PlanTooLarge(
                    f"eliminating the cheapest hidden variable needs a table of {best_cost} cells "
                    f"(budget {self.table_budget}); " +
                    (f"{'the most probable explanation' if cx.reduce == 'max' else 'posterior sampling'} has no per-row "
                     "executor" if decode is not None else "this query needs the per-row executor"))
            keys = g.touching(v)
            touching = [live[k] for k in keys]
            # the kernel multiplies at most MAX_CONTRACT_INPUTS factors at once: pre-multiply the smallest ones
            while len(touching) > N.MAX_CONTRACT_INPUTS:
                order = sorted(range(len(touching)), key=lambda i: _cells(touching[i].scope, cards))
                ia, ib = order[0], order[1]
                a, b = touching[ia], touching[ib]
                sc = cx.sort_scope(a.scope + b.scope)
                if _cells(sc, cards) > self.table_budget:
                    raise PlanTooLarge("pre-multiplication exceeds the table budget")
                stats.contraction_madds += 2 * _cells(sc, cards)
                prod = self._contract([a, b], sc, None, cx)
                g.replace([keys[ia], keys[ib]], next_key, sc)
                for k in (keys[ia], keys[ib]):
                    del live[k]
                live[next_key] = prod
                keys = [k for i, k in enumerate(keys) if i not in (ia, ib)] + [next_key]
                touching = [f for i, f in enumerate(touching) if i not in (ia, ib)] + [prod]
                next_key += 1
            out_scope = cx.sort_scope(best_scope)
            stats.n_steps += 1
            stats.max_table_cells = max(stats.max_table_cells, best_cost)
            stats.contraction_madds += best_cost * cards[v] * len(touching)
            if decode is not None:
                tb = None
                if not cx.dry and cx.reduce == "max":
                    tb = torch.empty(max(best_cost, 1), dtype=torch.uint8, device=self.t.device)
                elif not cx.dry:
                    tb = torch.empty(max(best_cost * (cards[v] - 1), 1), dtype=torch.float32, device=self.t.device)
                res = self._contract(touching, out_scope, v, cx, table=tb)
                decode.append((v, out_scope, tb))
            else:
                res = self._contract(touching, out_scope, v, cx)
            for k in keys:
                del live[k]
            live[next_key] = res
            g.eliminate(v, next_key, out_scope)
            next_key += 1
        out = list(live.values())
        return (out, []) if partial else out

    # ---------------------------------------------------------------- per-row schedule
    def _row_plan(self, cx: _Pass, statics: List[Factor], hidden: List[int]):
        """Schedule the elimination of ``hidden`` per row: evidence axes of the static tables are sliced by the
        row's codes, so only hidden axes (and the target) count towards the size of a temporary.

        Two passes.  The first fixes the elimination order and which factors meet in which step; the second chooses the
        LAYOUT of every factor.  A factor -- static table or temporary -- is consumed by exactly one step, so it is laid
        out for that step: the variable the step sums over innermost (stride 1), which is what the executor's unrolled
        step bodies need (csrc/ve.cu, ``row_step_unit``).  Static tables whose axes are in a different order are
        permuted once, here, at compile time."""
        import numpy as np

        cards, T, E, Eset, stats = self.t.cards, cx.T, cx.E, cx.ev, cx.stats
        n_in = len(statics)
        MAXIN = N.MAX_CONTRACT_INPUTS

        # pass 1: (input keys, output key, output scope, summed variable or None)
        live = {k: [v for v in f.scope if v not in Eset] for k, f in enumerate(statics)}
        ops = []
        next_key = n_in
        g = _Greedy(cards, {k: list(sc) for k, sc in live.items()}, hidden)
        while g.hidden:
            v, _, sc = g.best()
            keys = list(g.touching(v))
            while len(keys) > MAXIN:                           # pre-multiply the two smallest
                order = sorted(range(len(keys)), key=lambda i: _cells(live[keys[i]], cards))
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
            st = _strides(f.scope, cards)
            fac[k] = (k, [v for v in f.scope if v not in Eset], {v: st[v] for v in f.scope if v not in Eset})
        steps, off_chunks, off_at, temp_total = [], [], 0, 0
        for keys, out_key, out_scope, sum_var in ops:
            inputs = [fac[k] for k in keys]
            out_scope = lay_out(out_scope, out_key)
            out_shape = [cards[v] for v in out_scope]
            out_size = math.prod(out_shape)
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
            fac[out_key] = (n_in + len(steps) - 1, list(out_scope), _strides(out_scope, cards))
        offsets = np.ascontiguousarray(np.concatenate(off_chunks), dtype=np.int32)
        # the schedule as plain host data (what cbn_ve_plan_create_rows receives): kept for inspection and for the
        # fp64 interpreter of tests/row_oracle.py
        self.last_row_schedule = {"target": T, "evidence": list(E), "static_scopes": [list(f.scope) for f in laid],
                                  "static_source_scopes": [list(f.scope) for f in statics],
                                  "steps": steps, "offsets": offsets}
        if cx.dry:
            return None
        return RowPlan(self.t, T, E, cards[T] if T is not None else 1, laid, steps, offsets, stats, cx.log_space)

    def _merge_finals(self, cx: _Pass, finals: List[Factor]) -> List[Factor]:
        """Multiply final tables together while the product stays within the merge budget: fewer gathers
        per row, and a single table can be normalised at compile time."""
        sort_scope = cx.sort_scope
        finals = [Factor(sort_scope(f.scope), f.tensor) if f.scope == sort_scope(f.scope) else
                  self._contract([f], sort_scope(f.scope), None, cx) for f in finals]
        while len(finals) > 1:
            best = None
            for i in range(len(finals)):
                for j in range(i + 1, len(finals)):
                    sc = sort_scope(finals[i].scope + finals[j].scope)
                    c = _cells(sc, self.t.cards)
                    if best is None or c < best[0]:
                        best = (c, i, j, sc)
            c, i, j, sc = best
            if c > self.merge_budget and len(finals) <= N.MAX_GATHER_TABLES:
                break
            if c > self.table_budget:
                raise PlanTooLarge("cannot reduce the number of final tables within the budget")
            a, b = finals[i], finals[j]
            finals = [f for k, f in enumerate(finals) if k not in (i, j)]
            cx.stats.contraction_madds += 2 * c
            cx.stats.max_table_cells = max(cx.stats.max_table_cells, c)
            finals.append(self._contract([a, b], sc, None, cx))
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
