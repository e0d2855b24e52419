"""fp64 oracles of the most probable explanation for the MPE tests and ``tools/bench_mpe.py``.  TEST INFRASTRUCTURE ONLY.

Nothing under ``continuousbayesiannetwork_b200/`` imports this file.  Networks are ``oracle.cbn_oracle.DiscreteNet``
containers (cards, parents ordered as the CPT axes, CPTs).  Codes outside a variable's domain make a row -inf.
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from oracle.cbn_oracle import DiscreteNet


def random_small_net(rng, n_lo=5, n_hi=11):
    """A random small DAG (cardinalities 2-4, up to 3 parents) with a third of the CPT rows deterministic, so that
    zero-probability evidence occurs: (cards, parents, cpts)."""
    n = int(rng.integers(n_lo, n_hi))
    cards = [int(c) for c in rng.integers(2, 5, size=n)]
    parents = [sorted(int(p) for p in rng.choice(i, size=min(i, int(rng.integers(0, 4))), replace=False)) if i else []
               for i in range(n)]
    cpts = []
    for i in range(n):
        rows = int(np.prod([cards[p] for p in parents[i]])) if parents[i] else 1
        t = rng.dirichlet(np.full(cards[i], 0.7), size=rows)
        for r in range(rows):
            if rng.random() < 0.33:
                t[r] = np.eye(cards[i])[int(rng.integers(0, cards[i]))]
        cpts.append(t.reshape([cards[p] for p in parents[i]] + [cards[i]]))
    return cards, parents, cpts


def log_joint(net: DiscreteNet, codes: np.ndarray) -> np.ndarray:
    """fp64 log P(x) of complete rows: codes int [n_rows, n_vars]; a code outside the domain gives -inf."""
    codes = np.asarray(codes, dtype=np.int64).reshape(-1, net.n)
    bad = np.zeros(codes.shape[0], dtype=bool)
    for v in range(net.n):
        bad |= (codes[:, v] < 0) | (codes[:, v] >= net.cards[v])
    c = np.where(bad[:, None], 0, codes)
    out = np.zeros(codes.shape[0], dtype=np.float64)
    with np.errstate(divide="ignore"):
        for v in range(net.n):
            idx = tuple(c[:, p] for p in net.parents[v]) + (c[:, v],)
            out += np.log(np.asarray(net.cpts[v], dtype=np.float64)[idx])
    out[bad] = -np.inf
    return out


def enumerate_mpe(net: DiscreteNet, evidence_vars: Sequence[int], codes: np.ndarray):
    """fp64 MPE by enumerating the full joint (small networks only).  Returns ``(best, second, assignment)``: the best and
    second-best log joint over the configurations consistent with each row's evidence (second = -inf when there is no
    other configuration of positive probability) and int [n_rows, n_vars] the best configuration (the first in row-major
    order among equal values; -1 everywhere for a row whose best is -inf)."""
    evidence_vars = [int(v) for v in evidence_vars]
    ec = np.asarray(codes, dtype=np.int64).reshape(-1, len(evidence_vars)) if evidence_vars else \
        np.zeros((np.asarray(codes).shape[0], 0), np.int64)
    total = int(np.prod(net.cards))
    assert total <= 1 << 22, "enumeration oracle is for small networks"
    grid = np.indices(net.cards).reshape(net.n, -1)
    lj = log_joint(net, grid.T)
    n_rows = ec.shape[0]
    best = np.full(n_rows, -np.inf)
    second = np.full(n_rows, -np.inf)
    assign = np.full((n_rows, net.n), -1, dtype=np.int64)
    uniq, inv = np.unique(ec, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    for u, cfg in enumerate(uniq):
        if any(c < 0 or c >= net.cards[v] for v, c in zip(evidence_vars, cfg)):
            continue
        mask = np.ones(total, dtype=bool)
        for v, c in zip(evidence_vars, cfg):
            mask &= grid[v] == c
        idx = np.flatnonzero(mask)
        vals = lj[idx]
        order = np.argsort(-vals, kind="stable")
        b = vals[order[0]]
        if not np.isfinite(b):
            continue
        rows = inv == u
        best[rows] = b
        second[rows] = vals[order[1]] if len(order) > 1 else -np.inf
        assign[rows] = grid[:, idx[order[0]]]
    return best, second, assign


def ve_mpe(net: DiscreteNet, evidence_vars: Sequence[int], codes: np.ndarray, dtype=torch.float64
           ) -> Tuple[np.ndarray, Dict[int, np.ndarray]]:
    """Textbook batched max-product Variable Elimination in log space with traceback (Alarm-sized networks).

    Every CPT is a log table; those that mention evidence are sliced per row (leading row axis).  Every hidden variable
    is maximised out in min-size order, recording the argmax (first maximum) per row and context; what is left is added
    into the row's value.  The hidden values are then read back in reverse order.  Returns ``(log_value, assignment)``:
    fp64 [n_rows] ``log max_h P(h, e)`` (-inf for a code outside the domain or evidence of probability zero) and
    hidden variable -> int [n_rows] codes (meaningless where the value is -inf)."""
    ROW = -1
    evidence_vars = [int(v) for v in evidence_vars]
    ec = np.asarray(codes, dtype=np.int64).reshape(-1, len(evidence_vars)) if evidence_vars else \
        np.zeros((np.asarray(codes).shape[0], 0), np.int64)
    n_rows = int(ec.shape[0])
    invalid = np.zeros(n_rows, dtype=bool)
    ev = {}
    for i, v in enumerate(evidence_vars):
        c = ec[:, i]
        invalid |= (c < 0) | (c >= net.cards[v])
        ev[v] = torch.as_tensor(np.clip(c, 0, net.cards[v] - 1))
    factors: List[Tuple[List[int], torch.Tensor]] = []
    for v in range(net.n):
        scope = net.parents[v] + [v]
        t = torch.log(torch.as_tensor(np.asarray(net.cpts[v], dtype=np.float64)).to(dtype))
        ev_axes = [a for a in scope if a in ev]
        if ev_axes:
            perm = [scope.index(a) for a in ev_axes] + [i for i, a in enumerate(scope) if a not in ev]
            t = t.permute(perm)[tuple(ev[a] for a in ev_axes)]
            factors.append(([ROW] + [a for a in scope if a not in ev], t))
        else:
            factors.append((list(scope), t))
    hidden = [v for v in range(net.n) if v not in ev]

    def size_after(v):
        s = set()
        for sc, _ in factors:
            if v in sc:
                s |= set(sc)
        s.discard(v); s.discard(ROW)
        return (int(np.prod([net.cards[a] for a in s])) if s else 1, v)

    trace = []
    while hidden:
        v = min(hidden, key=size_after)
        hidden.remove(v)
        touching = [(sc, t) for sc, t in factors if v in sc]
        factors = [(sc, t) for sc, t in factors if v not in sc]
        out_scope = sorted({a for sc, _ in touching for a in sc if a != v}, key=lambda a: (a != ROW, a))
        full = out_scope + [v]
        acc = None
        for sc, t in touching:
            shape = [t.shape[sc.index(a)] if a in sc else 1 for a in full]
            tt = t.permute([sc.index(a) for a in full if a in sc]).reshape(shape)
            acc = tt if acc is None else acc + tt
        if ROW in out_scope and acc.shape[0] != n_rows:
            acc = acc.expand(*([n_rows] + list(acc.shape[1:])))
        res, arg = acc.max(dim=-1)
        trace.append((v, out_scope, arg))
        factors.append((out_scope, res))
    out = torch.zeros(n_rows, dtype=dtype)
    for sc, t in factors:       # scopes are [ROW] or []
        out = out + (t if sc else t.reshape(()))
    value = out.numpy().astype(np.float64)
    value[np.isnan(value)] = -np.inf
    value[invalid] = -np.inf
    assign: Dict[int, torch.Tensor] = {v: ev[v] for v in ev}
    rows = torch.arange(n_rows)
    for v, sc, arg in reversed(trace):
        idx = tuple(rows if a == ROW else assign[a] for a in sc)
        a = arg[idx] if sc else arg.reshape(()).expand(n_rows)
        if sc and ROW not in sc:
            a = a.reshape(-1)
            if a.numel() != n_rows:
                a = a.expand(n_rows)
        assign[v] = a.reshape(n_rows)
    return value, {v: assign[v].numpy().astype(np.int64) for v in range(net.n) if v not in ev}
