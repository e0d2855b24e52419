"""Exact inference by Variable Elimination -- the first real occupant of the reference's
empty plugin slot (cbn/inference/exact.py:6-17, registered in cbn/inference/__init__.py:3
and selected by the ``inference_obj: exact`` config key, cbn/conf/inference/exact.yaml:1)."""
from typing import Dict, Optional, Sequence

import torch

from .. import _native as N
from ..base.inference import BaseInference
from ..ve import EvidencePlan, FusedPlan, MPEPlan, PosteriorSamplePlan, QueryPlan, RowPlan, VECompiler


class ExactInference(BaseInference):
    def __init__(self, config: Dict, **kwargs):
        super(ExactInference, self).__init__(config=config, **kwargs)
        self.normalization = "row"
        self.compiler: Optional[VECompiler] = None
        self._setup_model(config, **kwargs)

    def _setup_model(self, config: Dict, **kwargs):
        self.normalization = (config or {}).get("normalization", "row")
        if self.normalization not in ("row", "global_max"):
            raise ValueError(f"normalization must be 'row' or 'global_max', got {self.normalization!r}")
        self._budget = {k: int(config[k]) for k in ("table_budget_cells", "merge_budget_cells", "row_temp_floats",
                                                    "mpe_argmax_budget_bytes", "sample_table_budget_bytes")
                        if config and k in config}
        for k in ("log_space", "rescale", "profile_compile", "row_unit_layout"):
            if config and k in config:
                self._budget[k] = bool(config[k])

    def bind(self, tables):
        """Attach the fitted network tables (called by BayesianNetwork after every fit)."""
        self.tables = tables
        self.compiler = VECompiler(tables, **self._budget)

    def plan(self, target_node: str, evidence_names: Sequence[str], do: Sequence[str] = ()) -> QueryPlan:
        assert self.compiler is not None, "inference engine is not bound to a fitted network"
        return self.compiler.compile(target_node, list(evidence_names), do=do)

    def fused_plan(self, targets: Sequence[str], evidence_names: Sequence[str]) -> FusedPlan:
        """One launch for several targets that share the evidence list (same target cardinality)."""
        return FusedPlan([self.plan(t, evidence_names) for t in targets])

    def _columns(self, evidence: Dict[str, torch.Tensor], names: Sequence[str], n_empty: int = 1,
                 mismatch: str = "n_queries must be equal for all features."):
        """``evidence[n]`` for ``names`` (tensors [n_rows] or [n_rows, 1] of category VALUES) as contiguous float32 device
        columns, and their common number of rows (``n_empty`` when there is no column)."""
        t = self.tables
        for n in names:
            if n not in t.index:
                raise ValueError(f"{n} is not a node of the network")
        cols = [torch.as_tensor(evidence[n]).to(t.device, torch.float32, non_blocking=True).reshape(-1).contiguous()
                for n in names]
        nq = int(cols[0].numel()) if cols else n_empty
        if any(int(c.numel()) != nq for c in cols):
            raise ValueError(mismatch)
        return cols, nq

    def _codes(self, evidence: Dict[str, torch.Tensor], names: Sequence[str], **kw):
        """``_columns`` encoded on the device: (uint8 code matrix, row e = ``names[e]``; number of rows)."""
        cols, nq = self._columns(evidence, names, **kw)
        return self.tables.encode_evidence([self.tables.index[n] for n in names], cols, nq), nq

    def infer_many(self, targets: Sequence[str], evidence: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """Posteriors of SEVERAL targets under the same evidence: the evidence columns are uploaded and encoded once,
        and targets of equal cardinality are answered by one fused launch (``cbn_ve_plan_fuse``).  Not part of the
        reference's surface (its ``infer`` takes one target per call); row-normalised posteriors, float32
        [n_queries, card(target)] on the device, keyed by target name."""
        t = self.tables
        evidence = evidence or {}
        names = [n for n in evidence.keys() if n not in targets]
        for n in targets:
            if n not in t.index:
                raise ValueError(f"{n} is not a node of the network")
        codes, nq = self._codes(evidence, names)
        out: Dict[str, torch.Tensor] = {}
        by_card: Dict[int, list] = {}
        for tg in targets:
            by_card.setdefault(t.cards[t.index[tg]], []).append(tg)
        for _, group in by_card.items():
            plans = [self.plan(tg, names) for tg in group]
            fusable = len(group) > 1 and all(isinstance(p, QueryPlan) for p in plans)
            for i in range(0, len(group), 8 if fusable else 1):
                chunk = group[i: i + 8]
                if fusable and len(chunk) > 1:
                    fused = self.compiler.cached(("fused", tuple(chunk), tuple(names)), lambda: FusedPlan(plans[i: i + 8]))
                    for tg, o in zip(chunk, fused.run_codes(codes, nq)):
                        out[tg] = o
                else:
                    out[chunk[0]] = plans[i].run_codes(codes, nq)
        return out

    def evidence_plan(self, evidence_names: Sequence[str]) -> EvidencePlan:
        assert self.compiler is not None, "inference engine is not bound to a fitted network"
        return self.compiler.compile_evidence(list(evidence_names))

    def log_evidence(self, evidence: Dict[str, torch.Tensor]) -> torch.Tensor:
        """``log P(e)`` per row: float32 [n_rows] on the device (natural log).  ``evidence``: name -> tensor [n_rows] or
        [n_rows, 1] of category VALUES, the same observed set for every row; every other node is summed out exactly.
        -inf for a value outside the fitted domain (NaN included) or evidence of probability zero; an empty dict gives an
        empty result.  Not part of the reference's surface."""
        names = list(evidence or {})
        codes, nq = self._codes(evidence, names, n_empty=0, mismatch="all evidence columns must have the same number of rows")
        return self.evidence_plan(names).run_codes(codes, nq)

    def mpe_plan(self, evidence_names: Sequence[str]) -> MPEPlan:
        assert self.compiler is not None, "inference engine is not bound to a fitted network"
        return self.compiler.compile_mpe(list(evidence_names))

    def most_probable_explanation(self, evidence: Dict[str, torch.Tensor]):
        """Most probable explanation per row: ``(assignment, log_prob)``.  ``evidence``: name -> tensor [n_rows] or
        [n_rows, 1] of category VALUES, the same observed set for every row.  ``assignment`` maps every other node to
        float32 [n_rows] domain values of ``argmax_h P(h, e)`` (NaN where ``log_prob`` is -inf); ``log_prob`` is float32
        [n_rows] ``log max_h P(h, e)`` (natural log; -inf for a value outside the fitted domain, NaN included, or evidence
        of probability zero).  No evidence gives one row, the explanation of the prior.  Not part of the reference's
        surface."""
        t = self.tables
        names = list(evidence or {})
        codes, nq = self._codes(evidence, names, mismatch="all evidence columns must have the same number of rows")
        plan = self.mpe_plan(names)
        hidden, log_prob = plan.run_codes(codes, nq)
        return {t.names[v]: self._values(v, hidden[h, :nq]) for h, v in enumerate(plan.hidden)}, log_prob

    def _values(self, v: int, codes: torch.Tensor) -> torch.Tensor:
        """Codes of variable ``v`` as float32 domain values, NaN where the code is CBN_UNSEEN."""
        t = self.tables
        c = codes.long()
        vals = t.domains[v][c.clamp(max=t.cards[v] - 1)]
        return torch.where(c >= t.cards[v], torch.full_like(vals, float("nan")), vals)

    def posterior_sampler(self, evidence_names: Sequence[str]) -> PosteriorSamplePlan:
        assert self.compiler is not None, "inference engine is not bound to a fitted network"
        return self.compiler.compile_posterior_sampler(list(evidence_names))

    def sample_posterior(self, evidence: Dict[str, torch.Tensor], n_draws: int = 1, seed: int = 0, first_row: int = 0):
        """Exact draws from ``P(h | e)`` per row: ``(draws, log_evidence)``.  ``evidence``: name -> tensor [n_rows] or
        [n_rows, 1] of category VALUES, the same observed set for every row.  ``draws`` maps every other node to float32
        [n_draws, n_rows] domain values, each draw a joint sample of all of them (NaN where ``log_evidence`` is -inf);
        ``log_evidence`` is float32 [n_rows] ``log P(e)`` (natural log; -inf for a value outside the fitted domain, NaN
        included, or evidence of probability zero).  Draw d of row i depends only on ``(seed, first_row + i, d)``: split
        a batch over calls with ``first_row`` and the draws are the same bits.  No evidence gives one row of draws from the
        prior.  Not part of the reference's surface."""
        if n_draws < 0 or first_row < 0:
            raise ValueError("n_draws and first_row must not be negative")
        t = self.tables
        names = list(evidence or {})
        codes, nq = self._codes(evidence, names, mismatch="all evidence columns must have the same number of rows")
        plan = self.posterior_sampler(names)
        hidden, log_evidence = plan.run_codes(codes, nq, n_draws=n_draws, seed=seed, first_row=first_row)
        nh = len(plan.hidden)          # row d * nh + h of the code matrix: draw d of plan.hidden[h]
        return {t.names[v]: self._values(v, hidden[h::nh][:n_draws, :nq]) for h, v in enumerate(plan.hidden)}, log_evidence

    def infer_map(self, target_node: str, evidence: Dict[str, torch.Tensor]) -> Optional[torch.Tensor]:
        """MAP value of the target per row through the fused kernel (``cbn_ve_run_f32_map``); ``None`` when the plan is
        not a single-target gather plan with at most 8 target values (the caller then takes posterior + argmax)."""
        evidence = evidence or {}
        names = [n for n in evidence.keys() if n != target_node]
        cols, nq = self._columns(evidence, names)
        plan = self.plan(target_node, names)
        if not isinstance(plan, QueryPlan) or plan.card_t > N.GATHER_MAX_CT or len(names) > N.MAX_EVIDENCE_PTRS:
            return None
        return plan.run_f32_map(cols, nq)

    def _infer(self, target_node: str, evidence: Dict[str, torch.Tensor], do=None, **kwargs) -> torch.Tensor:
        """Posterior ``P(target | evidence)`` per row: float32 [n_queries, card(target)] on the device.

        evidence: name -> tensor [n_queries, 1] (or [n_queries]) of category VALUES (float), as the
        reference's ``infer`` takes them (bayesian_network.py:208-226)."""
        t = self.tables
        evidence = evidence or {}
        names = [n for n in evidence.keys() if n != target_node]
        cols, nq = self._columns(evidence, names)
        out = self.plan(target_node, names, do=do or ()).run_f32(cols, nq)
        norm = kwargs.get("normalization", self.normalization)
        if norm == "global_max":
            m = torch.zeros(1, dtype=torch.float32, device=t.device)
            s = N.stream_ptr(t.device)
            N.check(N.lib().cbn_batch_max(t.ctx.handle, out.data_ptr(), out.numel(), m.data_ptr(), s), t.ctx.handle)
            N.check(N.lib().cbn_scale_by_inv(t.ctx.handle, out.data_ptr(), out.numel(), m.data_ptr(), s), t.ctx.handle)
        return out
