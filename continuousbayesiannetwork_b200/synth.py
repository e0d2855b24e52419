"""Synthetic discrete networks of the benchmark configurations (BASELINE.json `configs`).

None of these networks ships with the reference (no ``.bif`` files; SURVEY.md section 8c):
Asia uses the published Lauritzen-Spiegelhalter CPTs, the other structures get seeded
Dirichlet CPTs.  A network here is a plain description (names, cards, parents, CPTs as
numpy arrays) that ``tables.DiscreteTables`` / the oracle can both consume.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Sequence

import numpy as np


@dataclass
class NetSpec:
    names: List[str]
    cards: List[int]
    parents: List[List[int]]          # parent ids of node i, sorted by NAME (the reference's CPT axis order)
    cpts: List[np.ndarray]            # [card(pa_1).., card(i)] float64, rows sum to 1

    @property
    def n(self) -> int:
        return len(self.names)

    def parents_by_name(self) -> Dict[str, List[str]]:
        return {self.names[i]: [self.names[p] for p in self.parents[i]] for i in range(self.n)}

    def topological_order(self) -> List[int]:
        indeg = [len(p) for p in self.parents]
        children = [[] for _ in range(self.n)]
        for i, ps in enumerate(self.parents):
            for p in ps:
                children[p].append(i)
        order, stack = [], [i for i in range(self.n) if indeg[i] == 0]
        while stack:
            v = stack.pop()
            order.append(v)
            for c in children[v]:
                indeg[c] -= 1
                if indeg[c] == 0:
                    stack.append(c)
        assert len(order) == self.n, "not a DAG"
        return order

    def cdfs(self) -> List[np.ndarray]:
        """float32 cumulative tables for the ancestral sampler."""
        return [np.cumsum(c.astype(np.float64), axis=-1).astype(np.float32) for c in self.cpts]


def _sort_parents(names: Sequence[str], parents: List[List[int]]) -> List[List[int]]:
    return [sorted(ps, key=lambda p: names[p]) for ps in parents]


def _dirichlet_cpts(rng, cards, parents, alpha=1.0):
    cpts = []
    for i, ps in enumerate(parents):
        shape = [cards[p] for p in ps]
        rows = int(np.prod(shape)) if shape else 1
        t = rng.dirichlet(np.full(cards[i], alpha), size=rows)
        cpts.append(t.reshape(shape + [cards[i]]))
    return cpts


def asia() -> NetSpec:
    """Asia (Lauritzen & Spiegelhalter 1988): 8 binary nodes, 8 arcs."""
    names = ["asia", "tub", "smoke", "lung", "bronc", "either", "xray", "dysp"]
    ix = {n: i for i, n in enumerate(names)}
    par = {"asia": [], "tub": ["asia"], "smoke": [], "lung": ["smoke"], "bronc": ["smoke"],
           "either": ["lung", "tub"], "xray": ["either"], "dysp": ["bronc", "either"]}
    parents = _sort_parents(names, [[ix[p] for p in par[n]] for n in names])
    T = lambda p: np.array([1.0 - p, p])
    cpts = [None] * 8
    cpts[ix["asia"]] = T(0.01)
    cpts[ix["tub"]] = np.stack([T(0.01), T(0.05)])
    cpts[ix["smoke"]] = T(0.5)
    cpts[ix["lung"]] = np.stack([T(0.01), T(0.1)])
    cpts[ix["bronc"]] = np.stack([T(0.3), T(0.6)])
    # either | lung, tub  (sorted parents: lung, tub) = OR
    cpts[ix["either"]] = np.array([[T(0.0), T(1.0)], [T(1.0), T(1.0)]])
    cpts[ix["xray"]] = np.stack([T(0.05), T(0.98)])
    # dysp | bronc, either
    cpts[ix["dysp"]] = np.array([[T(0.1), T(0.7)], [T(0.8), T(0.9)]])
    return NetSpec(names, [2] * 8, parents, cpts)


_ALARM = ("[HISTORY|LVFAILURE][CVP|LVEDVOLUME][PCWP|LVEDVOLUME][HYPOVOLEMIA][LVEDVOLUME|HYPOVOLEMIA:LVFAILURE]"
          "[LVFAILURE][STROKEVOLUME|HYPOVOLEMIA:LVFAILURE][ERRLOWOUTPUT][HRBP|ERRLOWOUTPUT:HR][HREKG|ERRCAUTER:HR]"
          "[ERRCAUTER][HRSAT|ERRCAUTER:HR][INSUFFANESTH][ANAPHYLAXIS][TPR|ANAPHYLAXIS][EXPCO2|ARTCO2:VENTLUNG]"
          "[KINKEDTUBE][MINVOL|INTUBATION:VENTLUNG][FIO2][PVSAT|FIO2:VENTALV][SAO2|PVSAT:SHUNT][PAP|PULMEMBOLUS]"
          "[PULMEMBOLUS][SHUNT|INTUBATION:PULMEMBOLUS][INTUBATION][PRESS|INTUBATION:KINKEDTUBE:VENTTUBE][DISCONNECT]"
          "[MINVOLSET][VENTMACH|MINVOLSET][VENTTUBE|DISCONNECT:VENTMACH][VENTLUNG|INTUBATION:KINKEDTUBE:VENTTUBE]"
          "[VENTALV|INTUBATION:VENTLUNG][ARTCO2|VENTALV][CATECHOL|ARTCO2:INSUFFANESTH:SAO2:TPR][HR|CATECHOL]"
          "[CO|HR:STROKEVOLUME][BP|CO:TPR]")
_ALARM_CARD2 = {"HISTORY", "HYPOVOLEMIA", "LVFAILURE", "ERRLOWOUTPUT", "ERRCAUTER", "INSUFFANESTH", "ANAPHYLAXIS",
                "KINKEDTUBE", "FIO2", "PULMEMBOLUS", "SHUNT", "DISCONNECT", "CATECHOL"}
_ALARM_CARD4 = {"EXPCO2", "MINVOL", "PRESS", "VENTMACH", "VENTTUBE", "VENTLUNG", "VENTALV"}
ALARM_EVIDENCE = ["HRBP", "HREKG", "HRSAT", "BP", "CO", "CVP", "PCWP", "EXPCO2", "MINVOL", "PRESS", "PAP", "HISTORY"]
ALARM_TARGETS = ["HYPOVOLEMIA", "LVFAILURE", "KINKEDTUBE", "PULMEMBOLUS"]


def alarm(seed: int = 1236, alpha: float = 1.0) -> NetSpec:
    """Alarm-shaped network: the published 37-node / 46-arc structure and cardinalities
    (Beinlich et al. 1989) with seeded Dirichlet CPTs (the CPT values are not available offline)."""
    names, par = [], {}
    for item in _ALARM.strip("[]").split("]["):
        if "|" in item:
            n, ps = item.split("|")
            par[n] = ps.split(":")
        else:
            n = item
            par[n] = []
        names.append(n)
    ix = {n: i for i, n in enumerate(names)}
    cards = [2 if n in _ALARM_CARD2 else 4 if n in _ALARM_CARD4 else 3 for n in names]
    parents = _sort_parents(names, [[ix[p] for p in par[n]] for n in names])
    n_arcs = sum(len(p) for p in parents)
    free = sum((cards[i] - 1) * int(np.prod([cards[p] for p in parents[i]])) for i in range(len(names)))
    assert (len(names), n_arcs, free) == (37, 46, 509), (len(names), n_arcs, free)
    rng = np.random.default_rng(seed)
    return NetSpec(names, cards, parents, _dirichlet_cpts(rng, cards, parents, alpha))


def random_ktree_dag(n: int = 200, card: int = 4, k: int = 8, max_parents: int = 4, seed: int = 1237,
                     alpha: float = 1.0) -> NetSpec:
    """Random DAG built as a partial k-tree: node i picks 1..max_parents parents inside an existing
    k-clique, so the moral graph has treewidth <= k and every family table has <= card^(max_parents+1) cells."""
    rng = np.random.default_rng(seed)
    names = [f"x{i:03d}" for i in range(n)]
    cliques = [list(range(min(k, n)))]
    parents: List[List[int]] = []
    for i in range(n):
        if i < k:
            cand = list(range(i))
            m = min(len(cand), int(rng.integers(0, max_parents + 1)))
            ps = list(rng.choice(cand, size=m, replace=False)) if m else []
        else:
            cl = cliques[int(rng.integers(0, len(cliques)))]
            m = int(rng.integers(1, max_parents + 1))
            ps = list(rng.choice(cl, size=m, replace=False))
            drop = int(rng.integers(0, len(cl)))
            cliques.append([v for j, v in enumerate(cl) if j != drop] + [i])
        parents.append([int(p) for p in ps])
    parents = _sort_parents(names, parents)
    cards = [card] * n
    return NetSpec(names, cards, parents, _dirichlet_cpts(rng, cards, parents, alpha))


def layered_dag(layers: int = 20, width: int = 50, seed: int = 1238, alpha: float = 1.0) -> NetSpec:
    """Layered DAG: `layers` x `width` nodes, cards ~ U{2..8}, each node has 1..3 parents within
    +-2 positions in the previous layer (elimination-order stress)."""
    rng = np.random.default_rng(seed)
    names, cards, parents = [], [], []
    for l in range(layers):
        for j in range(width):
            names.append(f"l{l:02d}_{j:02d}")
            cards.append(int(rng.integers(2, 9)))
            if l == 0:
                parents.append([])
            else:
                cand = [(l - 1) * width + jj for jj in range(max(0, j - 2), min(width, j + 3))]
                m = int(rng.integers(1, 4))
                parents.append([int(p) for p in rng.choice(cand, size=min(m, len(cand)), replace=False)])
    parents = _sort_parents(names, parents)
    return NetSpec(names, cards, parents, _dirichlet_cpts(rng, cards, parents, alpha))


def splitmix64(z: np.ndarray) -> np.ndarray:
    """numpy restatement of the sampler's counter hash (csrc/fit.cu: splitmix64)."""
    z = (z + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)).astype(np.uint64)
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)).astype(np.uint64)
    return z ^ (z >> np.uint64(31))


def sample_forward_numpy(spec: NetSpec, seed: int, first: int, n: int) -> np.ndarray:
    """CPU restatement of ``cbn_sample_forward`` (bit-identical codes); returns uint8 [n_vars, n]."""
    with np.errstate(over="ignore"):
        sid = (np.arange(n, dtype=np.uint64) + np.uint64(first))
        base = splitmix64(np.uint64(seed) ^ (sid * np.uint64(0xD1B54A32D192ED03)))
        codes = np.zeros((spec.n, n), dtype=np.uint8)
        cdfs = spec.cdfs()
        for v in spec.topological_order():
            h = splitmix64(base + np.uint64(v))
            u = ((h >> np.uint64(40)).astype(np.uint32)).astype(np.float32) * np.float32(1.0 / 16777216.0)
            c = cdfs[v]
            rows = c[tuple(codes[p].astype(np.int64) for p in spec.parents[v])] if spec.parents[v] else np.broadcast_to(c, (n, spec.cards[v]))
            x = (u[:, None] >= rows[:, : spec.cards[v] - 1]).sum(axis=1)
            codes[v] = x.astype(np.uint8)
    return codes


def posterior_uniforms(seed: int, rows: np.ndarray, draw: int, var: int) -> np.ndarray:
    """numpy restatement of ``cbn_psample_run``'s uniforms (bit-identical float32): the uniform of draw ``draw`` of
    network variable ``var`` in each global row index of ``rows`` (``first_row + i``).  The row base is that of
    ``sample_forward_numpy``; the draw index is mixed in before the variable."""
    with np.errstate(over="ignore"):
        rows = np.asarray(rows, dtype=np.uint64)
        base = splitmix64(np.uint64(seed) ^ (rows * np.uint64(0xD1B54A32D192ED03)))
        base = splitmix64(base ^ (np.uint64(draw) * np.uint64(0x9E6C63D0676A9A99)))
        h = splitmix64(base + np.uint64(var))
    return ((h >> np.uint64(40)).astype(np.uint32)).astype(np.float32) * np.float32(1.0 / 16777216.0)
