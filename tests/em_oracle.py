"""fp64 EM by enumeration for the EM tests and ``tools/bench_em.py``.  TEST INFRASTRUCTURE ONLY.

Nothing under ``continuousbayesiannetwork_b200/`` imports this file.  A network is ``(cards, parents, cpts)`` with parents
ordered as the CPT axes; ``codes`` are int [n_rows, n_vars] whose hidden columns are ignored.  Enumeration over the joint
configurations of the hidden variables: small hidden sets only.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np


def _configs(cards: Sequence[int]) -> np.ndarray:
    return np.indices(cards).reshape(len(cards), -1).T if len(cards) else np.zeros((1, 0), np.int64)


def posterior(cards, parents, cpts, hidden: Sequence[int], codes: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """``(P(e_row), P(H = config | e_row))``: fp64 [n_rows] and [n_rows, card_H] over the joint configurations of
    ``hidden`` (mixed radix in the given order, first slowest); a row of probability zero has an all-zero posterior."""
    codes = np.asarray(codes, np.int64)
    n = codes.shape[0]
    cfg = _configs([cards[h] for h in hidden])
    joint = np.empty((n, cfg.shape[0]))
    full = codes.copy()
    for k, c in enumerate(cfg):
        full[:, list(hidden)] = c
        p = np.ones(n)
        for v in range(len(cards)):
            idx = tuple(full[:, u] for u in parents[v]) + (full[:, v],)
            p *= np.asarray(cpts[v], np.float64)[idx]
        joint[:, k] = p
    pe = joint.sum(axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        post = np.where(pe[:, None] > 0, joint / pe[:, None], 0.0)
    return pe, post


def e_step(cards, parents, cpts, hidden: Sequence[int], codes: np.ndarray) -> Tuple[List[np.ndarray], float, int]:
    """Expected family counts (fp64, shaped like the CPTs), ``sum log P(e_row)`` over live rows, number of dead rows."""
    codes = np.asarray(codes, np.int64)
    pe, post = posterior(cards, parents, cpts, hidden, codes)
    cfg = _configs([cards[h] for h in hidden])
    counts = [np.zeros(np.shape(c)) for c in cpts]
    full = codes.copy()
    for k, c in enumerate(cfg):
        full[:, list(hidden)] = c
        for v in range(len(cards)):
            idx = tuple(full[:, u] for u in parents[v]) + (full[:, v],)
            np.add.at(counts[v], idx, post[:, k])
    live = pe > 0
    return counts, float(np.log(pe[live]).sum()), int((~live).sum())


def m_step(counts: Sequence[np.ndarray], pseudo_count: float = 0.0) -> List[np.ndarray]:
    out = []
    for c in counts:
        c = c + pseudo_count
        s = c.sum(axis=-1, keepdims=True)
        out.append(np.where(s > 0, c / np.where(s > 0, s, 1), 0.0))
    return out


def em(cards, parents, cpts, hidden: Sequence[int], codes: np.ndarray, n_iter: int, pseudo_count: float = 0.0):
    """``n_iter`` EM iterations from ``cpts``: (final CPTs, log-likelihood of the parameters entering each iteration)."""
    history = []
    for _ in range(n_iter):
        counts, ll, _ = e_step(cards, parents, cpts, hidden, codes)
        history.append(ll)
        cpts = m_step(counts, pseudo_count)
    return cpts, history


def latent_class(n_children: int = 20, k: int = 4, card: int = 3, seed: int = 0, sharp: float = 0.0):
    """Z -> X_1 .. X_n: (names, cards, parents, cpts), Z first.  ``sharp`` > 0 makes the children's rows separated
    (each class puts that much extra mass on one value)."""
    rng = np.random.default_rng(seed)
    names = ["Z"] + [f"X{i:02d}" for i in range(n_children)]
    cards = [k] + [card] * n_children
    parents = [[]] + [[0]] * n_children
    cpts = [rng.dirichlet(np.full(k, 5.0))]
    for _ in range(n_children):
        t = rng.dirichlet(np.ones(card), size=k)
        if sharp:
            t = t + sharp * np.eye(card)[rng.integers(0, card, size=k)]
            t /= t.sum(axis=1, keepdims=True)
        cpts.append(t)
    return names, cards, parents, cpts


def hmm(steps: int = 6, k: int = 3, card: int = 4, seed: int = 0):
    """Hidden chain S0 -> S1 -> .. with one observation O_t per state: (names, cards, parents, cpts)."""
    rng = np.random.default_rng(seed)
    names = [f"S{t}" for t in range(steps)] + [f"O{t}" for t in range(steps)]
    cards = [k] * steps + [card] * steps
    parents = [[]] + [[t - 1] for t in range(1, steps)] + [[t] for t in range(steps)]
    cpts = [rng.dirichlet(np.ones(k))] + [rng.dirichlet(np.ones(k), size=k) for _ in range(1, steps)] + \
           [rng.dirichlet(np.ones(card), size=k) for _ in range(steps)]
    return names, cards, parents, cpts
