"""Device-resident discrete network: domains, integer codes, count tables, CPTs.

This is the host-side owner of the buffers the C ABI works on.  It replaces the
per-node ``torch.unique`` fitting of the reference with ONE pass over a code
matrix for all families (``BayesianNetwork._train`` -> ``Node.fit`` ->
``BruteForce._fit``; reference cbn/base/bayesian_network.py:138-160,
cbn/base/node.py:45-110, cbn/parameter_learning/brute_force.py:17-53).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import torch

from . import _native as N


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


class DiscreteTables:
    """Variables ``names`` with ``parents[name]`` (sorted by name, as the reference sorts
    them: bayesian_network.py:104-106).  Family of v = ``parents[v] + [v]``; its dense
    table is row-major over that list, node fastest."""

    def __init__(self, names: Sequence[str], parents: Dict[str, Sequence[str]], device="cuda"):
        self.ctx = N.context_for(device)
        self.device = torch.device("cuda", self.ctx.device_index)
        self.names: List[str] = list(names)
        self.index: Dict[str, int] = {n: i for i, n in enumerate(self.names)}
        self.parents: Dict[str, List[str]] = {n: list(parents.get(n, [])) for n in self.names}
        for n, ps in self.parents.items():
            if len(ps) + 1 > N.MAX_FAMILY_VARS:
                raise ValueError(f"node {n} has {len(ps)} parents; at most {N.MAX_FAMILY_VARS - 1} are supported")
        self.domains: List[Optional[torch.Tensor]] = [None] * len(self.names)   # float32 [card], sorted
        self.cards: List[int] = [0] * len(self.names)
        self._n_host = 0                 # samples counted so far; mirrored on the device next to the tables
        self._n_host_valid = True
        self._n_dev: Optional[torch.Tensor] = None
        self.fams = None
        self.offsets: List[int] = []
        self.n_cells: List[int] = []
        self.total_cells = 0
        self.counts: Optional[torch.Tensor] = None   # int64 [total_cells]
        self.joint: Optional[torch.Tensor] = None    # float32 [total_cells]
        self.cond: Optional[torch.Tensor] = None     # float32 [total_cells]
        self._log_cond: Optional[torch.Tensor] = None
        self.cond_version = 0                        # bumped whenever cond changes: plans derived from it are stale
        self._count_plan = None
        self._dom_matrix = None
        self._layout_cards: Optional[List[int]] = None
        self._discovered = None
        self._counts_buf: Optional[torch.Tensor] = None
        self._reduced = False            # the tables hold GLOBAL counts (summed over the ranks of a sharded fit)

    # ------------------------------------------------------------------ layout
    def set_domains(self, domains: Sequence[torch.Tensor]):
        """Fix the per-variable sorted domains (float32 tensors) and lay out the tables."""
        assert len(domains) == len(self.names)
        self.domains = [d.to(self.device, torch.float32).contiguous() for d in domains]
        self.cards = [int(d.numel()) for d in self.domains]
        self._dom_matrix = None
        for n, c in zip(self.names, self.cards):
            if not 1 <= c <= N.MAX_CARD:
                raise ValueError(f"variable {n} has {c} distinct values; the discrete path supports 1..{N.MAX_CARD}")
        self._layout()

    def set_cards(self, cards: Sequence[int]):
        """Integer-coded variables (synthetic workloads): domain of v is 0..card-1."""
        self.set_domains([torch.arange(int(c), dtype=torch.float32) for c in cards])

    def _layout(self):
        if self.fams is not None and self._layout_cards == self.cards and self._counts_buf is not None:
            # same structure and cardinalities as before (a re-fit): keep the tables' layout and the count plan
            self.reset_counts()
            self.joint = None
            self.cond = None
            self._drop_log_cond()
            return
        self._destroy_plan()
        self._layout_cards = list(self.cards)
        fams = (N.Family * len(self.names))()
        self.offsets, self.n_cells = [], []
        off = 0
        for i, n in enumerate(self.names):
            vs = [self.index[p] for p in self.parents[n]] + [i]
            cs = [self.cards[v] for v in vs]
            cells = 1
            for c in cs:
                cells *= c
            if cells > 1 << 31:
                raise ValueError(f"family table of {n} has {cells} cells (> 2^31)")
            fams[i] = N.make_family(vs, cs, off)
            self.offsets.append(off)
            self.n_cells.append(cells)
            off += _round_up(cells, 4)      # keep every table 16-byte aligned as float32
        self.fams = fams
        self.total_cells = off
        # the sample count lives right behind the tables, so a sharded fit moves both with ONE all-reduce and the
        # normalisation kernel reads it on the device (no host round trip)
        self._counts_buf = torch.zeros(off + 2, dtype=torch.int64, device=self.device)
        self.counts = self._counts_buf[:off]
        self._n_dev = self._counts_buf[off:off + 1]
        self.joint = None
        self.cond = None
        self._drop_log_cond()
        self._n_host, self._n_host_valid = 0, True
        self._reduced = False

    def _drop_log_cond(self):
        self._log_cond = None
        self.cond_version += 1

    @property
    def log_cond(self) -> torch.Tensor:
        """``log(cond)`` (natural log, -inf for zero entries), same layout as ``cond``; computed on first use and dropped
        whenever the conditional tables change (``finalize``, ``set_cond_tables``), together with the log-evidence plans
        built from it."""
        if self.cond is None:
            raise ValueError("the network is not fitted")
        if self._log_cond is None:
            self._log_cond = torch.log(self.cond)
        return self._log_cond

    def reset_counts(self):
        """Empty tables (and sample count) for a fresh fit; the layout and the count plan are kept."""
        self._counts_buf.zero_()
        self._n_host, self._n_host_valid = 0, True
        self._reduced = False

    @property
    def n_total(self) -> int:
        """Samples behind the current tables (global after a sharded fit)."""
        if not self._n_host_valid:
            self._n_host, self._n_host_valid = int(self._n_dev.item()), True
        return self._n_host

    @n_total.setter
    def n_total(self, v: int):
        self._n_host, self._n_host_valid = int(v), True
        if self._n_dev is not None:
            self._n_dev.fill_(int(v))

    def allreduce_buffer(self) -> torch.Tensor:
        """Tables + sample count as one int64 tensor; after summing it over the ranks call ``mark_reduced``."""
        return self._counts_buf

    def mark_reduced(self):
        """The buffer now holds the sum over all ranks: later sharded calls must reduce only their own delta."""
        self._n_host_valid = False
        self._reduced = True

    def is_reduced(self) -> bool:
        return self._reduced

    def count_delta(self, codes: torch.Tensor, n: int) -> torch.Tensor:
        """Counts (and sample count) of ``n`` samples in a fresh zeroed buffer laid out like ``allreduce_buffer()``;
        the tables themselves are not touched.  ``add_delta`` folds a (reduced) delta in."""
        assert codes.dtype == torch.uint8 and codes.dim() == 2 and codes.shape[0] == len(self.names) and codes.stride(1) == 1
        self._ensure_plan()
        delta = torch.zeros_like(self._counts_buf)
        N.check(N.lib().cbn_count_run(self.ctx.handle, self._count_plan, codes.data_ptr(), codes.stride(0), int(n),
                                      delta.data_ptr(), N.stream_ptr(self.device)), self.ctx.handle)
        delta[self.total_cells] = int(n)
        return delta

    def add_delta(self, delta: torch.Tensor):
        self._counts_buf.add_(delta)
        self._n_host_valid = False

    def _destroy_plan(self):
        if self._count_plan is not None:
            N.lib().cbn_count_plan_destroy(self._count_plan)
            self._count_plan = None

    def __del__(self):
        try:
            self._destroy_plan()
        except Exception:
            pass

    def family_vars(self, name: str) -> List[int]:
        return [self.index[p] for p in self.parents[name]] + [self.index[name]]

    def table_view(self, which: torch.Tensor, name: str) -> torch.Tensor:
        i = self.index[name]
        shape = [self.cards[v] for v in self.family_vars(name)]
        return which[self.offsets[i]: self.offsets[i] + self.n_cells[i]].view(*shape)

    # ------------------------------------------------------------------ ingestion
    def discover_domain(self, col: torch.Tensor) -> torch.Tensor:
        """Sorted distinct values of a float32 device column (Node.fit's torch.unique, node.py:85)."""
        col = col.to(self.device, torch.float32).contiguous()
        dom = torch.empty(256, dtype=torch.float32, device=self.device)
        card = torch.empty(1, dtype=torch.int32, device=self.device)
        N.check(N.lib().cbn_domain_f32(self.ctx.handle, col.data_ptr(), col.numel(), dom.data_ptr(), card.data_ptr(),
                                       N.stream_ptr(self.device)), self.ctx.handle)
        c = int(card.item())
        if c < 0:
            raise ValueError(
                f"column has more than {N.MAX_CARD} distinct values; it is not a discrete variable for the "
                "brute-force estimator")
        return dom[:c].clone()

    def discover_domains(self, cols: Sequence[torch.Tensor]) -> List[torch.Tensor]:
        """``discover_domain`` for many columns: one multi-column launch sequence (``cbn_domain_f32_multi``) and ONE
        host synchronisation."""
        k = len(cols)
        n = int(cols[0].numel()) if k else 0
        dom = torch.empty((max(k, 1), 256), dtype=torch.float32, device=self.device)
        card = torch.empty(max(k, 1), dtype=torch.int32, device=self.device)
        keep = [c.to(self.device, torch.float32).contiguous() for c in cols]
        for c in keep:
            if c.numel() != n:
                raise ValueError("all columns must have the same number of rows")
        if k:
            N.check(N.lib().cbn_domain_f32_multi(self.ctx.handle, N.ptr_array([c.data_ptr() for c in keep]), k, n, dom.data_ptr(),
                                                 card.data_ptr(), N.stream_ptr(self.device)), self.ctx.handle)
        cards = card.cpu().tolist()[:k]
        for i, c in enumerate(cards):
            if c < 0:
                raise ValueError(
                    f"column {i} has more than {N.MAX_CARD} distinct values; it is not a discrete variable for the "
                    "brute-force estimator")
        self._discovered = (dom, card, cards)        # fit_columns adopts the device matrix as it is (no second round trip)
        return [dom[i, :c] for i, c in enumerate(cards)]

    def encode(self, col: torch.Tensor, var: int, out: torch.Tensor, unseen: Optional[torch.Tensor] = None):
        col = col.to(self.device, torch.float32).contiguous()
        N.check(N.lib().cbn_encode_f32(self.ctx.handle, col.data_ptr(), col.numel(), self.domains[var].data_ptr(),
                                       self.cards[var], out.data_ptr(), unseen.data_ptr() if unseen is not None else None,
                                       N.stream_ptr(self.device)), self.ctx.handle)

    def new_code_matrix(self, n: int, n_vars: Optional[int] = None) -> torch.Tensor:
        """uint8 [n_vars (default: every variable), ld] for ``n`` samples; ld is a multiple of 16."""
        ld = _round_up(max(n, 1), 16)
        return torch.empty((len(self.names) if n_vars is None else n_vars, ld), dtype=torch.uint8, device=self.device)

    def encode_evidence(self, variables: Sequence[int], cols: Sequence[torch.Tensor], n: int) -> torch.Tensor:
        """Evidence columns of category VALUES -> uint8 code matrix [max(len(variables), 1), ld] whose row e holds the
        codes of ``cols[e]`` for variable ``variables[e]`` (an unseen value, NaN included, becomes CBN_UNSEEN)."""
        codes = self.new_code_matrix(n, max(len(variables), 1))
        for e, (v, col) in enumerate(zip(variables, cols)):
            self.encode(col, v, codes[e])
        return codes

    def _domain_matrix(self):
        """All domains as one device matrix [n_vars, 256] + cardinalities (built once per ``set_domains``)."""
        if self._dom_matrix is None:
            host = torch.zeros((len(self.names), 256), dtype=torch.float32)
            doms = torch.cat([d.reshape(-1) for d in self.domains]).cpu()          # one D2H copy
            at = 0
            for i, c in enumerate(self.cards):
                host[i, :c] = doms[at: at + c]
                at += c
            self._dom_matrix = (host.to(self.device), torch.tensor(self.cards, dtype=torch.int32, device=self.device))
        return self._dom_matrix

    def encode_columns(self, cols: Dict[str, torch.Tensor], strict: bool = True) -> torch.Tensor:
        """float32 columns (by node name) -> uint8 code matrix [n_vars, ld], all columns in one launch."""
        n = int(next(iter(cols.values())).numel())
        codes = self.new_code_matrix(n)
        unseen = torch.zeros(1, dtype=torch.int64, device=self.device)
        k = len(self.names)
        keep = [cols[name].reshape(-1).to(self.device, torch.float32).contiguous() for name in self.names]
        dom, card = self._domain_matrix()
        N.check(N.lib().cbn_encode_f32_multi(self.ctx.handle, N.ptr_array([c.data_ptr() for c in keep]), k, n, dom.data_ptr(),
                                             card.data_ptr(), codes.data_ptr(), codes.stride(0), unseen.data_ptr(),
                                             N.stream_ptr(self.device)), self.ctx.handle)
        if strict and int(unseen.item()) != 0:
            raise ValueError(f"{int(unseen.item())} values are not in the fitted domains")
        return codes

    # ------------------------------------------------------------------ counting
    def count(self, codes: torch.Tensor, n: int):
        """Accumulate the family counts of ``n`` samples (columns of ``codes``: uint8 [n_vars, ld])."""
        assert codes.dtype == torch.uint8 and codes.dim() == 2 and codes.shape[0] == len(self.names)
        assert codes.stride(1) == 1
        lib = N.lib()
        self._ensure_plan()
        N.check(lib.cbn_count_run(self.ctx.handle, self._count_plan, codes.data_ptr(), codes.stride(0), int(n),
                                  self.counts.data_ptr(), N.stream_ptr(self.device)), self.ctx.handle)
        self._n_dev.add_(int(n))
        if self._n_host_valid:
            self._n_host += int(n)

    def count_host(self, codes_host: torch.Tensor, n: int):
        """``count`` for a HOST code matrix (uint8 [n_vars, ld], pinned or pageable): chunked copies overlap the counting."""
        assert codes_host.dtype == torch.uint8 and codes_host.dim() == 2 and codes_host.shape[0] == len(self.names)
        assert not codes_host.is_cuda and codes_host.stride(1) == 1
        self._ensure_plan()
        N.check(N.lib().cbn_count_run_host(self.ctx.handle, self._count_plan, codes_host.data_ptr(), codes_host.stride(0), int(n),
                                           self.counts.data_ptr(), N.stream_ptr(self.device)), self.ctx.handle)
        self._n_dev.add_(int(n))
        if self._n_host_valid:
            self._n_host += int(n)

    def _ensure_plan(self):
        if self._count_plan is None:
            h = C.c_void_p()
            N.check(N.lib().cbn_count_plan_create(self.ctx.handle, self.fams, len(self.names), len(self.names), C.byref(h)),
                    self.ctx.handle)
            self._count_plan = h

    def count_updates_per_sample(self) -> int:
        self._ensure_plan()
        return N.lib().cbn_count_plan_updates_per_sample(self._count_plan)

    def count_groups(self) -> int:
        return N.lib().cbn_count_plan_groups(self._count_plan) if self._count_plan is not None else 0

    def finalize(self):
        """counts -> joint (fp32(c)/fp32(n)) and cond (joint / (parent + 1e-10))."""
        if self._n_host_valid and self._n_host < 1:
            raise ValueError("no samples counted")
        if self.joint is None or self.cond is None:
            self.joint = torch.zeros(self.total_cells, dtype=torch.float32, device=self.device)
            self.cond = torch.zeros(self.total_cells, dtype=torch.float32, device=self.device)
        self._ensure_plan()
        self._drop_log_cond()
        N.check(N.lib().cbn_cpt_from_plan_dev(self.ctx.handle, self._count_plan, self.counts.data_ptr(), self._n_dev.data_ptr(),
                                              self.joint.data_ptr(), self.cond.data_ptr(), N.stream_ptr(self.device)),
                self.ctx.handle)

    def set_cond_tables(self, cpts: Sequence):
        """Install ground-truth conditional tables (synthetic workloads; no counting)."""
        self.cond = torch.zeros(self.total_cells, dtype=torch.float32, device=self.device)
        self._drop_log_cond()
        for i, t in enumerate(cpts):
            t = torch.as_tensor(t, dtype=torch.float32).reshape(-1)
            assert t.numel() == self.n_cells[i]
            self.cond[self.offsets[i]: self.offsets[i] + self.n_cells[i]] = t.to(self.device)

    def fit_columns(self, cols: Dict[str, torch.Tensor]):
        """Full fit from float32 columns: domains, codes, counts, CPTs."""
        doms = self.discover_domains([cols[n].reshape(-1) for n in self.names])
        dom, card, _ = self._discovered
        self.set_domains(doms)
        self._dom_matrix = (dom, card)               # rows are zero-padded beyond the cardinality by the finish kernel
        codes = self.encode_columns(cols, strict=False)   # every value is in the domain that was just built from it
        n = int(next(iter(cols.values())).numel())
        self.count(codes, n)
        self.finalize()
        return codes

    # ------------------------------------------------------------------ reference views
    def mle_tensor(self, name: str) -> torch.Tensor:
        """The reference's sparse ``mle_tensor`` [M, P+2] of one family (brute_force.py:45-53)."""
        i = self.index[name]
        vs = self.family_vars(name)
        out = torch.empty((self.n_cells[i], len(vs) + 1), dtype=torch.float32, device=self.device)
        rows = torch.zeros(1, dtype=torch.int64, device=self.device)
        doms = N.ptr_array([self.domains[v].data_ptr() for v in vs])
        fam = N.make_family(list(range(len(vs))), [self.cards[v] for v in vs], 0)
        N.check(N.lib().cbn_mle_from_counts(self.ctx.handle, self.counts[self.offsets[i]:].data_ptr(), C.byref(fam), doms,
                                            self.n_total, out.data_ptr(), rows.data_ptr(), N.stream_ptr(self.device)),
                self.ctx.handle)
        return out[: int(rows.item())].clone()

    def get_prob(self, name: str, points: torch.Tensor, query: Optional[torch.Tensor]) -> torch.Tensor:
        """``P(x = points[q, v] | parents = query[q])`` (BruteForce._get_prob, brute_force.py:172-244)."""
        i = self.index[name]
        vs = self.family_vars(name)
        points = points.to(self.device, torch.float32).contiguous()
        assert points.dim() == 2
        fam = N.make_family(list(range(len(vs))), [self.cards[v] for v in vs], 0)
        doms = N.ptr_array([self.domains[v].data_ptr() for v in vs])
        if query is None:
            table = self.joint[self.offsets[i]:]
            nq = points.shape[0]
            qptr = None
        else:
            assert query.dim() == 3 and query.shape[-1] == 1, f"Query must be [n_queries, n_parents, 1]. Got {tuple(query.shape)}."
            if query.shape[1] != len(vs) - 1:
                raise ValueError(f"query has {query.shape[1]} parent columns, node {name} has {len(vs) - 1} parents")
            query = query.to(self.device, torch.float32).contiguous()
            table = self.cond[self.offsets[i]:]
            nq = query.shape[0]
            qptr = query.data_ptr()
        out = torch.empty((nq, points.shape[1]), dtype=torch.float32, device=self.device)
        N.check(N.lib().cbn_get_prob_f32(self.ctx.handle, table.data_ptr(), C.byref(fam), doms, points.data_ptr(),
                                         points.shape[0], points.shape[1], qptr, nq, out.data_ptr(),
                                         N.stream_ptr(self.device)), self.ctx.handle)
        return out
