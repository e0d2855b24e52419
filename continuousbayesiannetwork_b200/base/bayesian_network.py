"""Network API -- same constructor and methods as the reference's ``BayesianNetwork``
(cbn/base/bayesian_network.py:17-373), running on the B200 engine.

Differences a reference user will notice (all on paths where the reference is broken
or undefined, SURVEY.md section 3.3):

* ``infer`` answers with true Variable Elimination for any DAG / evidence set, not the
  mean-and-product heuristic.  On the only shape where the reference is a posterior
  (star DAG, every parent of the target observed) the results agree: identical with
  ``normalization="global_max"`` (the reference divides the batch by one global max,
  :296), equal up to that scale with the default ``"row"`` (rows sum to 1).
* all nodes are fitted by ONE fused pass over an integer-coded sample matrix instead of
  a Python loop of ``torch.unique`` sorts (:138-160).
* ``evidence=None`` works (prior marginal); ``do`` performs graph surgery.
* ``log_likelihood(data)`` scores rows: ``log P(observed values of the row)`` for any subset of the nodes, the others
  summed out exactly (held-out log-likelihood, anomaly scores, probability of evidence); the reference has no such query.
* ``most_probable_explanation(data)`` gives, per row, the jointly most probable values of every node not in ``data`` and
  their log-probability ``log max_h P(h, e)`` (missing-value completion, diagnosis); the reference has no such query.
* ``latent={"Z": k}`` / ``fit_em(data)`` fit networks with hidden nodes (no column in the data) by exact EM; the reference
  can only fit complete data.  ``fit_em(data, missing="marginalize")`` also takes NaN cells (per-row missing values).
* ``posterior_marginals(data)`` gives every node's posterior given each row's own observed cells (NaN: not observed) and
  ``log P`` of those cells; the reference has no such query.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Sequence, Tuple

import networkx as nx
import numpy as np
import torch

from . import BASE_MAX_CARDINALITY, KEY_MAX_CARDINALITY_FOR_DISCRETE
from .node import Node
from ..tables import DiscreteTables
from ..utils import choose_inference_obj


class BayesianNetwork:
    def __init__(self, dag: nx.DiGraph, data, parameters_learning_config: Dict, inference_config: Dict, **kwargs):
        """``latent``: hidden nodes, which have no column in ``data``: name -> cardinality k (domain 0.0 .. k-1) or the list
        of domain values.  With it the network is fitted by ``fit_em``, with the settings read from
        ``parameters_learning_config`` keys ``em_max_iter`` (100), ``em_tol`` (1e-6), ``em_seed`` (0) and
        ``em_pseudo_count`` (0) and ``em_missing`` ("error"; "marginalize" accepts NaN cells); ``self.em_result`` holds the
        ``EMResult``."""
        if not nx.is_directed_acyclic_graph(dag):
            raise ValueError("The provided graph is not a directed acyclic graph (DAG).")

        latent = kwargs.pop("latent", None)
        self.initial_dag = dag
        self.column_mapping = {node: i for i, node in enumerate(self.initial_dag.nodes)}
        self.device = kwargs.get("device", "cuda")
        kwargs["device"] = self.device
        self.min_tolerance = kwargs.get("min_tolerance", 1e-10)
        self.uncertainty = kwargs.get("uncertainty", 1e-10)
        self.max_cardinality_for_discrete_domain = kwargs.get(KEY_MAX_CARDINALITY_FOR_DISCRETE, BASE_MAX_CARDINALITY)
        self.log = kwargs.get("log", False)
        self.nodes_obj = None
        self.tables: DiscreteTables = None
        self.inference_obj = None
        self._kwargs = kwargs
        self._latent_domains = self._parse_latent(latent)
        cfg = parameters_learning_config or {}
        self._em_settings = {"max_iter": int(cfg.get("em_max_iter", 100)), "tol": float(cfg.get("em_tol", 1e-6)),
                             "seed": int(cfg.get("em_seed", 0)), "pseudo_count": float(cfg.get("em_pseudo_count", 0.0)),
                             "missing": str(cfg.get("em_missing", "error"))}
        self.em_result = None

        self._setup_inference(inference_config)
        self._setup_parameters_learning(data, parameters_learning_config, **kwargs)

    # ------------------------------------------------------------------ setup
    def _setup_parameters_learning(self, data, config: Dict, **kwargs):
        estimator_name = config["estimator_name"]
        self.nodes_obj = {
            node: Node(node, estimator_name, config, self.get_parents(self.initial_dag, node), **kwargs)
            for node in self.initial_dag.nodes
        }
        if self._latent_domains:
            self.fit_em(data, **self._em_settings)
        else:
            self._train(data, self.initial_dag.nodes)

    def _parse_latent(self, latent) -> Dict[str, torch.Tensor]:
        """name -> sorted float32 domain of every declared latent node."""
        out = {}
        for name, spec in (latent or {}).items():
            if name not in self.initial_dag.nodes:
                raise ValueError(f"latent node {name!r} is not a node of the network")
            if isinstance(spec, (int, np.integer)):
                if not 1 <= int(spec) <= 255:
                    raise ValueError(f"latent node {name!r} has cardinality {int(spec)}; the discrete path supports 1..255")
                vals = np.arange(int(spec), dtype=np.float32)
            else:
                vals = np.unique(np.asarray(spec, dtype=np.float32).reshape(-1))
                if np.isnan(vals).any() or vals.size != len(spec) or not 1 <= vals.size <= 255:
                    raise ValueError(f"latent node {name!r}: the domain must be 1..255 distinct values, not NaN")
            out[name] = torch.from_numpy(vals)
        return out

    def _setup_inference(self, config: Dict):
        self.inference_obj_name = config["inference_obj"]
        self.inference_obj = choose_inference_obj(self.inference_obj_name, config, device=self.device)

    def save_model(self, path: str):
        """One file with every count table and domain (the reference's version calls a method that
        does not exist, bayesian_network.py:78-80).  An EM fit also stores its CPTs, expected counts, hidden nodes and
        EM settings: its CPTs are not a function of the counts."""
        t = self.tables
        sd = {"names": t.names, "parents": t.parents, "domains": [d.cpu() for d in t.domains],
              "counts": t.counts.cpu(), "n_total": t.n_total}
        if t.hidden:
            sd.update({"cond": t.cond.cpu(), "joint": t.joint.cpu(), "expected_counts": t.expected_counts.cpu(),
                       "hidden": sorted(t.names[v] for v in t.hidden), "em_settings": dict(self._em_settings),
                       "latent": {n: d.cpu() for n, d in self._latent_domains.items()}})
        torch.save(sd, path)

    def load_model(self, path: str):
        sd = torch.load(path)
        if list(sd["names"]) != list(self.tables.names):
            raise ValueError("saved model has different nodes")
        self.tables.set_domains(sd["domains"])
        self.tables.counts.copy_(sd["counts"].to(self.tables.device))
        self.tables.n_total = int(sd["n_total"])
        if "cond" in sd:                 # an EM fit: the CPTs are stored, not derived from the counts
            t = self.tables
            t.set_cond(sd["cond"].to(t.device))
            t.joint = sd["joint"].to(t.device)
            t.expected_counts = sd["expected_counts"].to(t.device)
            t.hidden = {t.index[n] for n in sd["hidden"]}
            self._em_settings = dict(sd["em_settings"])
            self._latent_domains = {n: d.clone() for n, d in sd["latent"].items()}
        else:
            self.tables.hidden, self.tables.expected_counts = set(), None
            self.tables.finalize()
        self._attach_all()

    # ------------------------------------------------------------------ graph helpers
    @staticmethod
    def get_nodes(dag: nx.DiGraph):
        return sorted(list(dag.nodes))

    def _node_name(self, node):
        if isinstance(node, str):
            return node
        if isinstance(node, int):
            return next((k for k, v in self.column_mapping.items() if v == node), None)
        raise ValueError(f"{node} type not supported.")

    def get_ancestors(self, dag: nx.DiGraph, node):
        name = self._node_name(node)
        if name is None:
            return set()
        ancestors = nx.ancestors(dag, name)
        ordered = list(nx.topological_sort(dag.subgraph(ancestors | {name})))
        ordered.remove(name)
        return ordered

    def get_parents(self, dag: nx.DiGraph, node):
        return sorted(list(dag.predecessors(self._node_name(node))))

    def get_children(self, dag: nx.DiGraph, node):
        return sorted(list(dag.successors(self._node_name(node))))

    @staticmethod
    def get_structure(dag: nx.DiGraph):
        return {node: list(dag.predecessors(node)) for node in nx.topological_sort(dag)}

    # ------------------------------------------------------------------ fit
    def _columns(self, data) -> Dict[str, torch.Tensor]:
        """float32 device column per node.  DataFrames go through ONE numpy block and one H2D copy
        (the reference does pandas -> list -> numpy -> torch per column, :144-157); dicts of tensors /
        arrays are taken as they are (GPU-resident data is not copied)."""
        names = list(self.initial_dag.nodes)
        dev = self.device
        if isinstance(data, dict):
            return {n: torch.as_tensor(data[n]).reshape(-1).to(dev, torch.float32) for n in names}
        missing = [n for n in names if n not in data.columns]
        if missing:
            raise ValueError(f"data has no column for nodes {missing}")
        # [n_vars, n]; pandas hands out read-only views (copy-on-write): torch wants a writable, C-contiguous block
        block = np.require(data[names].to_numpy(dtype=np.float32).T, requirements=["C", "W"])
        dev_block = torch.from_numpy(block).to(dev)
        return {n: dev_block[i] for i, n in enumerate(names)}

    def _train(self, data, pbar: Iterable = None):
        names = list(self.initial_dag.nodes)
        parents = {n: self.get_parents(self.initial_dag, n) for n in names}
        cols = self._columns(data)
        self.tables = DiscreteTables(names, parents, device=self.device)
        self.tables.fit_columns(cols)
        self._attach_all()

    def _attach_all(self):
        for n, node in self.nodes_obj.items():
            node.attach(self.tables, n)
        self.inference_obj.bind(self.tables)

    def update_knowledge(self, data, accumulate: bool = False):
        """Re-fit on ``data`` (the reference REPLACES the tables: brute_force.py:47).  With
        ``accumulate=True`` the new samples are added to the existing int64 count tables instead
        (values outside the fitted domains raise ValueError).  A network with latent nodes is re-fitted by ``fit_em`` with
        its stored settings; it cannot accumulate (its expected counts depend on the parameters)."""
        if self._latent_domains or (self.tables is not None and self.tables.hidden):
            if accumulate:
                raise ValueError("a network with latent nodes cannot accumulate counts: its expected counts depend on the "
                                 "parameters; update_knowledge(data) re-fits it by EM")
            self.fit_em(data, **self._em_settings)
            return
        if not accumulate:
            self._train(data)
            return
        cols = self._columns(data)
        codes = self.tables.encode_columns(cols, strict=True)
        self.tables.count(codes, int(next(iter(cols.values())).numel()))
        self.tables.finalize()
        self._attach_all()

    def fit_em(self, data, max_iter: int = 100, tol: float = 1e-6, seed: int = 0, init: str = "random",
               pseudo_count: float = 0.0, missing: str = "error"):
        """Fit by expectation-maximisation: every node without a column in ``data`` is hidden in every row.

        :param data: a DataFrame or a dict name -> values, as ``log_likelihood`` takes them; the observed domains are
                     discovered from it, as the ordinary fit does (a re-fit, like ``update_knowledge``).  A hidden node
                     keeps the domain the network has for it (from ``latent=`` or an earlier fit).  Every row observes
                     the same nodes unless ``missing="marginalize"``.
        :param missing: ``"error"``: NaN in a column raises ``ValueError``.  ``"marginalize"``: a NaN cell is hidden in its
                     row only (domains are discovered from the other cells; a column of NaN only raises ``ValueError``).
                     When NaN cells are present the E-step is a junction-tree calibration per row (``cbn_jt_run``), with
                     the rows in which a family is fully observed counted as in the ordinary fit; without NaN the E-step
                     is the one of ``"error"``.  The log-likelihood is that of each row's observed cells.  A node with a
                     NaN cell is then treated like a latent node by the fitted tables: it is in ``tables.hidden``, so
                     ``mle_tensor`` refuses its families (``tables.counts`` holds only the complete rows; the expected
                     counts are in ``tables.expected_counts``) and ``update_knowledge`` re-fits by EM with the stored
                     settings.  With ``init="random"`` only families with a latent member start from Dirichlet(1) rows;
                     a family with NaN cells but no latent member starts from the MLE of its complete rows.
        :param init: ``"random"``: every CPT with a hidden member starts from Dirichlet(1) rows drawn with ``seed``;
                     ``"current"``: from the network's current CPTs (the data's domains must be the current ones).  Fully
                     observed families always get their exact MLE.
        :param pseudo_count: ``a`` of the M-step ``cond = (N + a) / sum_x (N + a)`` (N: expected counts).  With 0 the
                     M-step is the ordinary fit's formula.
        :return: ``EMResult`` (log-likelihood per iteration plus the final one, ``n_iter``, ``converged`` when the
                 relative gain fell below ``tol``, ``n_dead_rows``).  The fitted CPTs are installed; ``tables.counts``
                 holds the integer counts of the fully observed families and ``tables.expected_counts`` (float64) the
                 expected counts of every family.
        """
        from .. import _native as N
        from ..em import EM, JTEM, MAX_ROWS

        if getattr(self.inference_obj, "evidence_plan", None) is None:
            raise NotImplementedError(f"inference engine {self.inference_obj_name!r} does not compute posteriors for EM")
        if init not in ("random", "current"):
            raise ValueError(f"init must be 'random' or 'current', got {init!r}")
        if not pseudo_count >= 0:
            raise ValueError("pseudo_count must not be negative")
        if missing not in ("error", "marginalize"):
            raise ValueError(f"missing must be 'error' or 'marginalize', got {missing!r}")
        cols, n_rows = self._observed_columns(data)
        given = [n for n in cols if n in self._latent_domains]
        if given:
            raise ValueError(f"data has columns for the latent nodes {given}")
        if not 0 < n_rows < MAX_ROWS:
            raise ValueError(f"EM needs 1 .. 2^31 - 1 rows, got {n_rows}")
        nan_cells = int(sum(torch.isnan(c).sum() for c in cols.values()).item()) if cols else 0
        if nan_cells and missing == "marginalize":
            empty = [n for n, c in cols.items() if bool(torch.isnan(c).all().item())]
            if empty:
                raise ValueError(f"columns {empty} hold only NaN: they have no observed value to take a domain from")
        if nan_cells and missing == "error":
            raise ValueError("an observed column holds NaN: per-row missing values are not supported (every row observes "
                             "the same nodes; a node without a column is hidden in every row)")
        names = list(self.initial_dag.nodes)
        old = self.tables
        hidden = [n for n in names if n not in cols]
        domains = {}
        for n in hidden:
            if n in self._latent_domains:
                domains[n] = self._latent_domains[n]
            elif old is not None and old.domains[old.index[n]] is not None:
                domains[n] = old.domains[old.index[n]]
            else:
                raise ValueError(f"node {n} has no column and no domain: declare it with latent=")
        current = None
        if init == "current":
            if old is None or old.cond is None:
                raise ValueError("init='current' needs a fitted network")
            current = old.cond.clone()
        t = DiscreteTables(names, {n: self.get_parents(self.initial_dag, n) for n in names}, device=self.device)
        observed = [n for n in names if n in cols]
        for n, d in zip(observed, t.discover_domains([cols[n] for n in observed])):
            if nan_cells and d.numel() and bool(torch.isnan(d[-1]).item()):
                d = d[:-1]                 # the domain kernel keeps a collapsed NaN last: a missing cell, not a value
            if d.numel() == 0:
                raise ValueError(f"column {n} holds only NaN: it has no observed value to take a domain from")
            domains[n] = d
        t.set_domains([domains[n] for n in names])
        if current is not None and not all(torch.equal(a, b.to(a.device)) for a, b in zip(t.domains, old.domains)):
            raise ValueError("init='current': the data's domains differ from the network's, so its CPTs do not apply")
        codes = t.new_code_matrix(n_rows)
        # hidden rows: the count kernel skips every family with a hidden member (both codes are >= every cardinality)
        codes.fill_(N.MISSING if nan_cells else N.UNSEEN)
        for n in observed:
            t.encode(cols[n], t.index[n], codes[t.index[n]])
            if nan_cells:
                codes[t.index[n], :n_rows].masked_fill_(torch.isnan(cols[n]), N.MISSING)
        t.count(codes, n_rows)
        t.hidden = {t.index[n] for n in hidden}
        self.tables = t
        self._attach_all()
        em = (JTEM if nan_cells else EM)(t, self.inference_obj, codes, n_rows, sorted(t.hidden))
        if nan_cells:
            # a node with a missing cell has no exact counts of its own (its families start from the complete rows' MLE)
            t.hidden |= {t.index[n] for n in observed if bool(torch.isnan(cols[n]).any().item())}
        em.initialise(init, seed, current)
        result = em.fit(max_iter, tol, pseudo_count)
        t.expected_counts = em.expected_counts()
        self._em_settings = {"max_iter": int(max_iter), "tol": float(tol), "seed": int(seed), "pseudo_count": float(pseudo_count),
                             "missing": missing}
        self._attach_all()
        self.em_result = result
        return result

    # ------------------------------------------------------------------ queries
    def get_pdf(self, target_node: str, evidence: Dict, N_max: int = 1024) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Factor of one node: only the evidence on its parents is used (reference :176-206)."""
        target_node_parents = self.get_parents(self.initial_dag, target_node)
        query = {f: v for f, v in (evidence or {}).items() if f in target_node_parents}
        return self.nodes_obj[target_node].get_prob(query, N_max)

    def infer(self, target_node: str, evidence: Dict[str, torch.Tensor] = None, do: List[str] = None,
              N_max: int = 16, plot_prob=False, normalization: str = None, pad_to_N_max: bool = False):
        """
        :param target_node: node whose posterior is computed
        :param evidence: name -> tensor [n_queries, 1] of observed VALUES
        :param do: names of evidence variables that are interventions
        :param N_max: number of evaluation points of the target domain (reference semantics, node.py:286-300):
                      ``N_max >= card(target)`` evaluates the whole domain, smaller values sub-sample it
        :param pad_to_N_max: reproduce the reference's output SHAPE for ``N_max > card(target)``: the domain is padded to
                      N_max points with never-observed values (``Node.sample_domain``, deterministic here) whose
                      probability is zero, so ``pdf`` and ``domains`` are ``[n_queries, N_max]`` as in the reference
                      (node.py:302-333).  Off by default: the posterior then has ``card(target)`` columns.
        :return: (pdf [n_queries, V], domains [n_queries, V])
        """
        if target_node not in self.nodes_obj:
            raise ValueError(f"{target_node} is not a node of the network")
        kw = {} if normalization is None else {"normalization": normalization}
        pdf = self.inference_obj.infer(target_node, evidence or {}, do, **kw)
        dom = self.tables.domains[self.tables.index[target_node]]
        if N_max < dom.shape[0]:
            idx = torch.linspace(0, dom.shape[0] - 1, N_max).round().long().to(dom.device)
            pdf = pdf[:, idx].contiguous()
            dom = dom[idx]
        elif pad_to_N_max and N_max > dom.shape[0]:
            padded = self.nodes_obj[target_node].sample_domain(target_node, N_max).to(dom.device)
            pos = torch.searchsorted(padded, dom)                      # where the fitted values sit in the padded domain
            wide = torch.zeros((pdf.shape[0], N_max), dtype=pdf.dtype, device=pdf.device)
            wide[:, pos] = pdf
            pdf, dom = wide, padded
        domains = dom.unsqueeze(0).expand(pdf.shape[0], -1)
        assert pdf.shape == domains.shape, "pdf and domain must have same shape."
        return pdf, domains

    def infer_many(self, target_nodes: List[str], evidence: Dict[str, torch.Tensor] = None) -> Dict[str, Tuple[torch.Tensor, torch.Tensor]]:
        """``infer`` for several targets under the same evidence in one pass (evidence uploaded and encoded once,
        equal-cardinality targets answered by one fused launch).  Returns name -> (pdf, domains) as ``infer`` does."""
        for tn in target_nodes:
            if tn not in self.nodes_obj:
                raise ValueError(f"{tn} is not a node of the network")
        pdfs = self.inference_obj.infer_many(list(target_nodes), evidence or {})
        out = {}
        for tn, pdf in pdfs.items():
            dom = self.tables.domains[self.tables.index[tn]]
            out[tn] = (pdf, dom.unsqueeze(0).expand(pdf.shape[0], -1))
        return out

    def log_likelihood(self, data) -> torch.Tensor:
        """Natural log of the probability of each row's observed values under the fitted CPTs: float32 [n_rows] on the
        device.

        :param data: a DataFrame or a dict name -> values (tensor / array) holding domain VALUES, as ``infer`` takes them.
                     The observed set is the set of columns passed, the same for every row; every other node is summed
                     out exactly, so a subset of the nodes gives ``log P(e)``.  A column that is not a node raises
                     ``ValueError`` (a typo must not silently marginalise a variable), as do columns of different lengths.
        :return: ``log P(row)``; ``-inf`` for a value outside the fitted domain (NaN included) or for values of
                 probability zero under the CPTs (a never-observed parent configuration among them); 0 for every row
                 when no column is passed.  ``log P(e, T=t) - log P(e)`` equals ``log`` of ``infer``'s posterior
                 ``P(t | e)``.  The value of a row depends on that row only (any batching gives identical bits).
        """
        cols, n_rows = self._observed_columns(data)
        if not cols:
            return torch.zeros(n_rows, dtype=torch.float32, device=self.device)
        log_evidence = getattr(self.inference_obj, "log_evidence", None)
        if log_evidence is None:
            raise NotImplementedError(f"inference engine {self.inference_obj_name!r} does not compute log P(e)")
        return log_evidence(cols)

    def most_probable_explanation(self, data) -> Tuple[Dict[str, torch.Tensor], torch.Tensor]:
        """Most probable explanation of each row: the jointly most likely values of every node NOT in ``data``,
        ``argmax_h P(h, e)``, and their log-probability.

        :param data: a DataFrame or a dict name -> values holding domain VALUES, as ``log_likelihood`` takes them; the
                     observed set is the set of columns passed, the same for every row.  A column that is not a node
                     raises ``ValueError``.
        :return: ``(assignment, log_prob)``.  ``assignment`` maps every other node to float32 [n_rows] domain values on the
                 device; ``log_prob`` is float32 [n_rows], ``log max_h P(h, e)`` (natural log).  A row with a value outside
                 the fitted domain (NaN included) or evidence of probability zero gives ``log_prob = -inf`` and NaN in every
                 assignment column (never a NaN ``log_prob``).  With no columns the result is one row, the explanation of
                 the prior; with every node observed ``assignment`` is empty and ``log_prob`` equals ``log_likelihood``.
                 The result is checkable: ``log_likelihood(data`` joined with ``assignment)`` equals ``log_prob`` within
                 fp32 rounding.  The value of a row depends on that row only (any batching gives identical bits).
        """
        cols, _ = self._observed_columns(data)
        mpe = getattr(self.inference_obj, "most_probable_explanation", None)
        if mpe is None:
            raise NotImplementedError(f"inference engine {self.inference_obj_name!r} does not compute explanations")
        return mpe(cols)

    def posterior_marginals(self, data, nodes: Sequence[str] = None) -> Tuple[Dict[str, torch.Tensor], torch.Tensor]:
        """Posterior marginal of every node given each row's own observed cells, and ``log P`` of those cells: for tabular
        data whose rows each miss different cells (imputation, per-row diagnosis, held-out scoring with gaps).

        :param data: a DataFrame or a dict name -> values holding domain VALUES; NaN means "not observed in this row", and
                     a node without a column is unobserved in every row.  A column that is not a node raises ``ValueError``.
        :param nodes: the nodes whose marginals are returned (default: every node); the others are not written.
        :return: ``(marginals, log_evidence)``.  ``marginals`` maps each node to float32 [n_rows, card] on the device (rows
                 sum to 1; an observed node is one-hot); these are column views of one [n_rows, sum of the cards] buffer,
                 not contiguous tensors (``.contiguous()`` copies one out); ``log_evidence`` is float32 [n_rows], ``log P(observed cells)``
                 (natural log).  A value outside the fitted domain or observed cells of probability zero give -inf and NaN
                 marginals.  With no columns the result is one row, the prior marginals.  The value of a row depends on
                 that row only.  Exact, by a junction-tree calibration per row; a network whose junction tree is over the
                 kernel's budgets raises ``PlanTooLarge``, and a node of cardinality 255 is refused the same way.
        """
        cols, _ = self._observed_columns(data)
        marginals = getattr(self.inference_obj, "posterior_marginals", None)
        if marginals is None:
            raise NotImplementedError(f"inference engine {self.inference_obj_name!r} does not compute posterior marginals")
        return marginals(cols, nodes)

    def sample_posterior(self, data, n_draws: int = 1, seed: int = 0,
                         first_row: int = 0) -> Tuple[Dict[str, torch.Tensor], torch.Tensor]:
        """Exact joint draws of every node NOT in ``data`` from its posterior given each row, ``h ~ P(h | e)``: for
        multiple imputation, uncertainty over hidden causes, or Monte Carlo estimates of joint queries.

        :param data: a DataFrame or a dict name -> values holding domain VALUES, as ``most_probable_explanation`` takes
                     them; the observed set is the set of columns passed, the same for every row.  A column that is not a
                     node raises ``ValueError``.
        :param n_draws: draws per row.
        :param seed, first_row: draw d of row i depends only on ``(seed, first_row + i, d)``, so a batch split over calls
                     (pass each part's offset as ``first_row``) or a smaller ``n_draws`` gives the same bits.
        :return: ``(draws, log_evidence)``.  ``draws`` maps every other node to float32 [n_draws, n_rows] domain values on
                 the device; ``log_evidence`` is float32 [n_rows], ``log P(e)`` (natural log).  A row with a value outside
                 the fitted domain (NaN included) or evidence of probability zero gives ``log_evidence = -inf`` and NaN in
                 every draw (never a NaN ``log_evidence``).  With no columns the result is one row of draws from the prior;
                 with every node observed ``draws`` is empty and ``log_evidence`` equals ``log_likelihood``.
        """
        cols, _ = self._observed_columns(data)
        sample = getattr(self.inference_obj, "sample_posterior", None)
        if sample is None:
            raise NotImplementedError(f"inference engine {self.inference_obj_name!r} does not sample posteriors")
        return sample(cols, n_draws=n_draws, seed=seed, first_row=first_row)

    def impute(self, data, method: str = "mpe", n_draws: int = 1, seed: int = 0,
               first_row: int = 0) -> Tuple[Dict[str, torch.Tensor], torch.Tensor]:
        """Complete each row's missing cells with values that are jointly consistent: the single most probable
        completion (``method="mpe"``) or joint draws from ``P(missing | observed)`` for multiple imputation
        (``method="sample"``).  Unlike per-node argmaxes or draws of ``posterior_marginals``, a completion never has
        probability zero.

        :param data: a DataFrame or a dict name -> values holding domain VALUES; NaN means "not observed in this row", and
                     a node without a column is unobserved in every row.  A column that is not a node raises ``ValueError``.
        :param method: ``"mpe"`` or ``"sample"``; anything else raises ``ValueError``.
        :param n_draws: draws per row for ``"sample"`` (at least 1); ``"mpe"`` takes 1 only.
        :param seed, first_row: draw d of row i depends only on ``(seed, first_row + i, d)``, so a batch split over calls
                     (pass each part's offset as ``first_row``) or a smaller ``n_draws`` gives the same bits.  These draws
                     are not ``sample_posterior``'s: the two factorise the posterior differently.
        :return: ``"mpe"``: ``(completed, log_prob)``.  ``completed`` maps EVERY node to float32 [n_rows] domain values on
                 the device (observed cells unchanged); ``log_prob`` is float32 [n_rows], ``log max P(completion)`` over
                 the completions of the row (natural log).  The result is checkable: ``log_likelihood(completed)`` equals
                 ``log_prob`` within fp32 rounding.  ``"sample"``: ``(draws, log_evidence)``.  ``draws`` maps every node
                 to float32 [n_draws, n_rows]; ``log_evidence`` is ``log P(observed cells)``, the bits of
                 ``posterior_marginals``'.  A value outside the fitted domain or observed cells of probability zero give
                 -inf and NaN in every column of the row (never a NaN log value).  With no columns the result is one row:
                 the explanation of the prior, or draws from it.  The value of a row depends on that row only.  Exact, by
                 a junction-tree pass per row; a network whose junction tree is over the kernel's budgets raises
                 ``PlanTooLarge`` before any device work.
        """
        cols, _ = self._observed_columns(data)
        impute = getattr(self.inference_obj, "impute", None)
        if impute is None:
            raise NotImplementedError(f"inference engine {self.inference_obj_name!r} does not impute")
        return impute(cols, method=method, n_draws=n_draws, seed=seed, first_row=first_row)

    def _observed_columns(self, data) -> Tuple[Dict[str, torch.Tensor], int]:
        """``_columns`` for a subset of the nodes: (name -> float32 device column, number of rows)."""
        dev = self.device
        names = list(data.keys()) if isinstance(data, dict) else list(data.columns)
        unknown = [n for n in names if n not in self.nodes_obj]
        if unknown:
            raise ValueError(f"columns {unknown} are not nodes of the network")
        if isinstance(data, dict):
            cols = {n: torch.as_tensor(data[n]).reshape(-1).to(dev, torch.float32) for n in names}
            lengths = {int(c.numel()) for c in cols.values()}
            if len(lengths) > 1:
                raise ValueError("all columns must have the same number of rows")
            return cols, (lengths.pop() if lengths else 0)
        n_rows = len(data)
        if not names:
            return {}, n_rows
        block = np.require(data[names].to_numpy(dtype=np.float32).T, requirements=["C", "W"])
        dev_block = torch.from_numpy(block).to(dev)
        return {n: dev_block[i] for i, n in enumerate(names)}, n_rows

    def sample(self, N: int, seed: int = 0, first_sample: int = 0) -> Dict[str, torch.Tensor]:
        """``N`` ancestral samples of the whole network from the fitted CPTs, as ``name -> float32 [N]`` device columns of
        domain VALUES (the network analogue of the estimator's ``sample``, brute_force.py:246-265).  Counter-based: sample
        ``first_sample + i`` depends only on ``(seed, first_sample + i)``, so any split of a range over calls or GPUs gives
        the same data.  A parent configuration that was never observed has no distribution to draw from; the sampler then
        returns the node's largest domain value."""
        import ctypes as C

        from .. import _native as NV

        t = self.tables
        if t.cond is None:
            raise ValueError("the network is not fitted")
        cdf = torch.empty_like(t.cond)
        for i in range(len(t.names)):
            card = t.cards[i]
            seg = slice(t.offsets[i], t.offsets[i] + t.n_cells[i])
            cdf[seg] = t.cond[seg].view(-1, card).cumsum(dim=1).reshape(-1)
        order_names = list(nx.topological_sort(self.initial_dag))
        order = (C.c_int32 * len(order_names))(*[t.index[self._node_name(n)] for n in order_names])
        codes = t.new_code_matrix(int(N))
        NV.check(NV.lib().cbn_sample_forward(t.ctx.handle, len(t.names), order, t.fams, cdf.data_ptr(), int(seed), int(first_sample),
                                             int(N), codes.data_ptr(), codes.stride(0), NV.stream_ptr(t.device)), t.ctx.handle)
        return {name: t.domains[i][codes[i, :N].long()] for i, name in enumerate(t.names)}

    def infer_map(self, target_node: str, evidence: Dict[str, torch.Tensor]) -> torch.Tensor:
        """MAP value of the target per row (what ``benchmarking_df`` extracts, :357-366)."""
        if target_node not in self.nodes_obj:
            raise ValueError(f"{target_node} is not a node of the network")
        fused = getattr(self.inference_obj, "infer_map", None)
        if fused is not None:
            res = fused(target_node, evidence or {})
            if res is not None:
                return res
        pdf, dom = self.infer(target_node, evidence, N_max=1 << 30)
        return torch.gather(dom, 1, torch.argmax(pdf, dim=1, keepdim=True)).squeeze(1)

    def benchmarking_df(self, data, target_feature: str, batch_size: int = 128, **kwargs) -> np.ndarray:
        """Batched MAP prediction with every other column as evidence (reference :329-373).  The whole
        frame is one launch per ``batch_size`` rows; pass a large batch_size to do it in one."""
        feats = [f for f in data.columns if f != target_feature and f in self.nodes_obj]
        block = torch.from_numpy(np.require(data[feats].to_numpy(dtype=np.float32).T, requirements=["C", "W"])).to(self.device)
        n = block.shape[1]
        pred = torch.empty(n, dtype=torch.float32, device=self.device)
        for s in range(0, n, batch_size):
            ev = {f: block[i, s: s + batch_size].unsqueeze(-1) for i, f in enumerate(feats)}
            pred[s: s + batch_size] = self.infer_map(target_feature, ev)
        return pred.cpu().numpy().astype(np.float64)
