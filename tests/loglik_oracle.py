"""fp64 oracles of log P(e) for the log-likelihood tests and ``tools/bench_loglik.py``.  TEST INFRASTRUCTURE ONLY.

Nothing under ``continuousbayesiannetwork_b200/`` imports this file.  Networks are ``oracle.cbn_oracle.DiscreteNet``
containers (cards, parents ordered as the CPT axes, CPTs).
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np
import torch

from oracle.cbn_oracle import DiscreteNet


def enumerate_log_evidence(net: DiscreteNet, evidence_vars: Sequence[int], codes: np.ndarray) -> np.ndarray:
    """fp64 ``log P(e)`` per row by summing the full joint of the evidence's ancestors (small networks only).

    codes int[n_rows, len(evidence_vars)]; a code outside the variable's domain or evidence of probability zero gives
    -inf; no evidence gives 0."""
    evidence_vars = [int(v) for v in evidence_vars]
    ec = np.asarray(codes).reshape(-1, len(evidence_vars)) if evidence_vars else np.zeros((np.asarray(codes).shape[0], 0))
    if not evidence_vars:
        return np.zeros(ec.shape[0], dtype=np.float64)
    keep = sorted(net.ancestors(evidence_vars))
    pos = {v: i for i, v in enumerate(keep)}
    cards = [net.cards[v] for v in keep]
    total = int(np.prod(cards))
    assert total <= 1 << 24, "enumeration oracle is for small networks"
    grid = np.indices(cards).reshape(len(keep), -1)
    joint = np.ones(total, dtype=np.float64)
    for v in keep:
        idx = tuple(grid[pos[p]] for p in net.parents[v]) + (grid[pos[v]],)
        joint *= np.asarray(net.cpts[v], dtype=np.float64)[idx]
    uniq, inv = np.unique(ec, axis=0, return_inverse=True)
    res = np.full(uniq.shape[0], -np.inf, dtype=np.float64)
    for u, cfg in enumerate(uniq):
        if any(c < 0 or c >= net.cards[v] for v, c in zip(evidence_vars, cfg)):
            continue
        mask = np.ones(total, dtype=bool)
        for v, c in zip(evidence_vars, cfg):
            mask &= grid[pos[v]] == c
        z = joint[mask].sum()
        res[u] = np.log(z) if z > 0 else -np.inf
    return res[inv.reshape(-1)]


def ve_log_evidence(net: DiscreteNet, evidence_vars: Sequence[int], codes: np.ndarray, dtype=torch.float64) -> np.ndarray:
    """Textbook batched Variable Elimination in log space: ``log P(e)`` per row (Alarm-sized networks).

    Every CPT of the evidence's ancestors is taken as a log table; those that mention evidence are sliced per row
    (leading row axis), every hidden variable is summed out by logsumexp in min-size order, and what is left (per-row
    values and scalars) is added.  A code outside the variable's domain gives -inf; no evidence gives 0."""
    ROW = -1
    evidence_vars = [int(v) for v in evidence_vars]
    ec = np.asarray(codes).reshape(-1, len(evidence_vars)) if evidence_vars else np.zeros((np.asarray(codes).shape[0], 0), np.int64)
    n_rows = int(ec.shape[0])
    if not evidence_vars:
        return np.zeros(n_rows, dtype=np.float64)
    invalid = np.zeros(n_rows, dtype=bool)
    ev = {}
    for i, v in enumerate(evidence_vars):
        c = ec[:, i].astype(np.int64)
        invalid |= (c < 0) | (c >= net.cards[v])
        ev[v] = torch.as_tensor(np.clip(c, 0, net.cards[v] - 1))
    keep = net.ancestors(evidence_vars)
    factors: List[Tuple[List[int], torch.Tensor]] = []
    for v in sorted(keep):
        scope = net.parents[v] + [v]
        t = torch.log(torch.as_tensor(np.asarray(net.cpts[v])).to(dtype))
        ev_axes = [a for a in scope if a in ev]
        if ev_axes:
            perm = [scope.index(a) for a in ev_axes] + [i for i, a in enumerate(scope) if a not in ev]
            t = t.permute(perm)[tuple(ev[a] for a in ev_axes)]
            factors.append(([ROW] + [a for a in scope if a not in ev], t))
        else:
            factors.append((list(scope), t))
    hidden = [v for v in keep if v not in ev]

    def size_after(v):
        s = set()
        for sc, _ in factors:
            if v in sc:
                s |= set(sc)
        s.discard(v); s.discard(ROW)
        return (int(np.prod([net.cards[a] for a in s])) if s else 1, v)

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
        res = torch.logsumexp(acc, dim=-1)
        res = torch.where(torch.isnan(res), torch.full_like(res, -float("inf")), res)
        factors.append((out_scope, res))
    out = torch.zeros(n_rows, dtype=dtype)
    for sc, t in factors:       # scopes are [ROW] or []
        out = out + (t if sc else t.reshape(()))
    out = out.numpy().astype(np.float64)
    out[invalid] = -np.inf
    return out
