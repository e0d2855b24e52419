"""fp64 oracles of posterior sampling for the posterior-sampling tests and ``tools/bench_posterior_sample.py``.  TEST
INFRASTRUCTURE ONLY.

Nothing under ``continuousbayesiannetwork_b200/`` imports this file.  Networks are ``oracle.cbn_oracle.DiscreteNet``
containers (cards, parents ordered as the CPT axes, CPTs).
"""
from __future__ import annotations

from typing import Dict, Sequence, Tuple

import numpy as np

from continuousbayesiannetwork_b200.synth import posterior_uniforms
from oracle.cbn_oracle import DiscreteNet

UNSEEN = 255


def joint_table(net: DiscreteNet) -> np.ndarray:
    """fp64 P(x) of every configuration, shaped ``net.cards`` (small networks only)."""
    assert int(np.prod(net.cards)) <= 1 << 22, "enumeration oracle is for small networks"
    args = []
    for v in range(net.n):
        args += [np.asarray(net.cpts[v], dtype=np.float64), net.parents[v] + [v]]
    return np.einsum(*args, list(range(net.n)))


def enumerate_posterior(net: DiscreteNet, evidence_vars: Sequence[int], cfg: Sequence[int]) -> Tuple[float, np.ndarray]:
    """``(P(e), P(h | e))`` for one evidence configuration by enumeration: the second is fp64 shaped by the cards of the
    hidden variables in network order (all zeros when P(e) = 0)."""
    p = joint_table(net)
    idx = [slice(None)] * net.n
    for v, c in zip(evidence_vars, cfg):
        idx[int(v)] = int(c)
    post = p[tuple(idx)]
    z = float(post.sum())
    return z, (post / z if z > 0 else np.zeros_like(post))


def interpret(decode, cards, evidence: Sequence[int], ev_codes: np.ndarray, dead: np.ndarray, seed: int,
              first_row: int, n_draws: int) -> Dict[int, np.ndarray]:
    """The backward-sampling schedule run by numpy: ``decode`` = [(variable, scope, float32 thresholds [cells, card-1])]
    in decode order (the plan's tables copied to the host), ``ev_codes`` int [n_rows, len(evidence)], ``dead`` bool
    [n_rows] (rows whose log P(e) is -inf or NaN).  Returns variable -> uint8 [n_draws, n_rows], UNSEEN in dead rows;
    bit-identical to ``cbn_psample_run`` by construction (same uniforms, same comparison in float32)."""
    n_rows = ev_codes.shape[0]
    rows = np.arange(n_rows, dtype=np.uint64) + np.uint64(first_row)
    out = {v: np.zeros((n_draws, n_rows), np.uint8) for v, _, _ in decode}
    for d in range(n_draws):
        code = {u: np.minimum(ev_codes[:, i], cards[u] - 1).astype(np.int64) for i, u in enumerate(evidence)}
        for v, scope, cdf in decode:
            ix = np.zeros(n_rows, np.int64)
            for u in scope:
                ix = ix * cards[u] + code[u]
            u01 = posterior_uniforms(seed, rows, d, v)
            thr = np.asarray(cdf, np.float32).reshape(-1, cards[v] - 1)[ix] if cards[v] > 1 else np.zeros((n_rows, 0), np.float32)
            code[v] = (u01[:, None] >= thr).sum(axis=1).astype(np.int64)
            out[v][d] = np.where(dead, UNSEEN, code[v]).astype(np.uint8)
    return out
