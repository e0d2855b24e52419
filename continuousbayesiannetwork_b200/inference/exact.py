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

    def junction_tree(self):
        """The network's junction tree (``jt.JunctionTree``), compiled once per set of CPTs."""
        from .. import jt

        assert self.compiler is not None, "inference engine is not bound to a fitted network"
        return jt.compile_tree(self.compiler)

    def missing_codes(self, evidence: Dict[str, torch.Tensor]):
        """``evidence`` (name -> tensor [n_rows] or [n_rows, 1] of category VALUES, NaN: not observed in that row) as a
        uint8 code matrix with a row per network variable: ``encode``, then NaN -> CBN_MISSING; a node without a column
        is CBN_MISSING in every row.  Returns (codes, number of rows; 1 when there is no column)."""
        t = self.tables
        names = list(evidence or {})
        cols, nq = self._columns(evidence, names, mismatch="all evidence columns must have the same number of rows")
        codes = t.new_code_matrix(nq)
        codes.fill_(N.MISSING)
        for n, col in zip(names, cols):
            v = t.index[n]
            t.encode(col, v, codes[v])
            codes[v, :nq].masked_fill_(torch.isnan(col), N.MISSING)
        return codes, nq

    def posterior_marginals(self, evidence: Dict[str, torch.Tensor], nodes: Optional[Sequence[str]] = None):
        """Posterior marginal of every node (or of ``nodes``) given each row's own observed cells, and ``log P`` of those
        cells: ``(marginals, log_evidence)``.  ``evidence``: name -> tensor [n_rows] or [n_rows, 1] of category VALUES,
        NaN where the row does not observe the node; a node without a column is unobserved in every row.
        ``marginals`` maps each node to float32 [n_rows, card] (an observed node is one-hot), a column view of ONE
        float32 [n_rows, sum of the cards] buffer the kernel writes (not contiguous: ``.contiguous()`` copies a node's
        block out; writing into a view writes that buffer); ``log_evidence`` is float32
        [n_rows] (natural log).  A value outside the fitted domain, or observed cells of probability zero, give -inf and
        NaN marginals.  No columns give one row, the prior marginals.  One junction-tree calibration per row
        (``cbn_jt_run``); the value of a row depends on that row only.  Not part of the reference's surface."""
        t = self.tables
        if nodes is None:
            ids = list(range(len(t.names)))
        else:
            for n in nodes:
                if n not in t.index:
                    raise ValueError(f"{n} is not a node of the network")
            ids = [t.index[n] for n in nodes]
            if len(set(ids)) != len(ids):
                raise ValueError("a node is listed twice")
        codes, nq = self.missing_codes(evidence)
        plan = self.junction_tree().plan(ids)
        run = plan.schedule.marg_floats
        marg = torch.empty((nq, run), dtype=torch.float32, device=t.device)
        log_evidence = torch.empty(nq, dtype=torch.float32, device=t.device)
        plan.run(codes, nq, marg_out=marg if run else None, log_out=log_evidence)
        at = plan.schedule.node_out
        return {t.names[v]: marg[:, at[v]: at[v] + t.cards[v]] for v in ids}, log_evidence

    def impute(self, evidence: Dict[str, torch.Tensor], method: str = "mpe", n_draws: int = 1, seed: int = 0,
               first_row: int = 0):
        """Completions of each row's unobserved cells, jointly consistent: ``(completed, log_prob)`` for ``method="mpe"``,
        ``(draws, log_evidence)`` for ``method="sample"``.  ``evidence``: name -> tensor [n_rows] or [n_rows, 1] of
        category VALUES, NaN where the row does not observe the node; a node without a column is unobserved in every row.
        ``"mpe"``: ``completed`` maps EVERY node to float32 [n_rows] domain values, ``argmax_h P(h, e_row)`` filled in and
        the observed cells unchanged; ``log_prob`` is float32 [n_rows] ``log max_h P(h, e_row)`` (natural log).
        ``"sample"``: ``draws`` maps every node to float32 [n_draws, n_rows], each draw a joint sample of the row's
        unobserved cells from ``P(h | e_row)``; ``log_evidence`` is float32 [n_rows] ``log P(e_row)``, the bits of
        ``posterior_marginals``'.  Draw d of row i depends only on ``(seed, first_row + i, d)``.  A value outside the
        fitted domain, or observed cells of probability zero, give -inf and NaN in every column.  No columns give one row.
        One collect pass and one top-down decode of the junction tree per row (``cbn_jt_decode``).  Not part of the
        reference's surface."""
        if method not in ("mpe", "sample"):
            raise ValueError(f"method must be 'mpe' or 'sample', got {method!r}")
        if n_draws < 1 or (method == "mpe" and n_draws != 1):
            raise ValueError(f"n_draws must be 1 for 'mpe' and at least 1 for 'sample', got {n_draws}")
        if first_row < 0:
            raise ValueError("first_row must not be negative")
        t = self.tables
        codes, nq = self.missing_codes(evidence)
        plan = self.junction_tree().collect_plan()
        nv = len(t.names)
        out = t.new_code_matrix(nq, n_draws * nv)
        log_out = torch.empty(nq, dtype=torch.float32, device=t.device)
        mode = N.JT_DECODE_MAX if method == "mpe" else N.JT_DECODE_SAMPLE
        plan.decode(codes, nq, mode, n_draws, seed, first_row, out, log_out)
        if method == "mpe":
            return {t.names[v]: self._values(v, out[v, :nq]) for v in range(nv)}, log_out
        return {t.names[v]: self._values(v, out[v: n_draws * nv: nv, :nq]) for v in range(nv)}, log_out

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
