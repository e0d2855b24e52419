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
        if not nx.is_directed_acyclic_graph(dag):
            raise ValueError("The provided graph is not a directed acyclic graph (DAG).")

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

        self._setup_inference(inference_config)
        self._setup_parameters_learning(data, parameters_learning_config, **kwargs)

    # ------------------------------------------------------------------ setup
    def _setup_parameters_learning(self, data, config: Dict, **kwargs):
        estimator_name = config["estimator_name"]
        self.nodes_obj = {
            node: Node(node, estimator_name, config, self.get_parents(self.initial_dag, node), **kwargs)
            for node in self.initial_dag.nodes
        }
        self._train(data, self.initial_dag.nodes)

    def _setup_inference(self, config: Dict):
        self.inference_obj_name = config["inference_obj"]
        self.inference_obj = choose_inference_obj(self.inference_obj_name, config, device=self.device)

    def save_model(self, path: str):
        """One file with every count table and domain (the reference's version calls a method that
        does not exist, bayesian_network.py:78-80)."""
        t = self.tables
        torch.save({"names": t.names, "parents": t.parents, "domains": [d.cpu() for d in t.domains],
                    "counts": t.counts.cpu(), "n_total": t.n_total}, path)

    def load_model(self, path: str):
        sd = torch.load(path)
        if list(sd["names"]) != list(self.tables.names):
            raise ValueError("saved model has different nodes")
        self.tables.set_domains(sd["domains"])
        self.tables.counts.copy_(sd["counts"].to(self.tables.device))
        self.tables.n_total = int(sd["n_total"])
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
        (values outside the fitted domains raise ValueError)."""
        if not accumulate:
            self._train(data)
            return
        cols = self._columns(data)
        codes = self.tables.encode_columns(cols, strict=True)
        self.tables.count(codes, int(next(iter(cols.values())).numel()))
        self.tables.finalize()
        self._attach_all()

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
