"""fp64 references of junction-tree calibration with per-row missing values.  TEST INFRASTRUCTURE ONLY.

Nothing under ``continuousbayesiannetwork_b200/`` imports this file.  A network is ``(cards, parents, cpts)`` with
parents ordered as the CPT axes.  ``codes`` are int [n_rows, n_vars]: a code below the cardinality is observed,
``MISSING`` (254) is summed out, anything else makes the row dead.

* ``enumerate_rows``: full-joint enumeration (small networks only): log P(observed cells), every node's marginal and every
  family's posterior per row;
* ``interpret``: the plan's own tables (``jt.Schedule``: ops, maps, message offsets) run op by op in fp64, vectorised over
  rows, with the kernel's rules (messages divided by their maximum, the UP log-scales plus log Z, dead rows);
* ``expected_counts``: the E-step the kernel adds to the count tables (families with a missing member in the row).
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence

import numpy as np

MISSING = 254


def _dead(cards, codes):
    codes = np.asarray(codes, np.int64)
    bad = np.zeros(codes.shape[0], bool)
    for v, c in enumerate(cards):
        bad |= ~((codes[:, v] < c) | (codes[:, v] == MISSING))
    return bad


def enumerate_rows(cards, parents, cpts, codes, chunk: int = 256):
    """``(log_p [n], marginals: list of [n, card_v], family posteriors: list of [n, cells_f] (family-table order))``;
    dead rows and rows of probability zero give -inf and NaN."""
    codes = np.asarray(codes, np.int64)
    n, nv = codes.shape
    total = int(np.prod(cards))
    assert total <= 1 << 18, "enumeration oracle is for small networks"
    grid = np.indices(cards).reshape(nv, -1)                       # [n_vars, configs]
    joint = np.ones(total)
    for v in range(nv):
        idx = tuple(grid[u] for u in parents[v]) + (grid[v],)
        joint *= np.asarray(cpts[v], np.float64)[idx]
    fam_cell = []
    for v in range(nv):
        fv = list(parents[v]) + [v]
        fam_cell.append(np.ravel_multi_index(tuple(grid[u] for u in fv), [cards[u] for u in fv]) if fv else np.zeros(total, int))
    dead = _dead(cards, codes)
    log_p = np.full(n, -np.inf)
    marg = [np.full((n, c), np.nan) for c in cards]
    fam = [np.full((n, int(np.prod([cards[u] for u in list(parents[v]) + [v]]))), np.nan) for v in range(nv)]
    for s in range(0, n, chunk):
        c = codes[s: s + chunk]
        ok = np.ones((c.shape[0], total), bool)
        for v in range(nv):
            ok &= (c[:, v: v + 1] == MISSING) | (grid[v][None, :] == c[:, v: v + 1])
        w = ok * joint[None, :]
        pe = w.sum(1)
        live = (pe > 0) & ~dead[s: s + chunk]
        with np.errstate(divide="ignore", invalid="ignore"):
            log_p[s: s + chunk] = np.where(live, np.log(pe), -np.inf)
            post = w / pe[:, None]
        for v in range(nv):
            m = np.stack([post[:, grid[v] == x].sum(1) for x in range(cards[v])], 1)
            marg[v][s: s + chunk] = np.where(live[:, None], m, np.nan)
            cells = fam[v].shape[1]
            f = np.stack([post[:, fam_cell[v] == k].sum(1) for k in range(cells)], 1)
            fam[v][s: s + chunk] = np.where(live[:, None], f, np.nan)
    return log_p, marg, fam


def expected_counts(cards, parents, cpts, codes):
    """Per family, fp64 sum over live rows in which a member is MISSING of the family's posterior (family-table shape)."""
    codes = np.asarray(codes, np.int64)
    log_p, _, fam = enumerate_rows(cards, parents, cpts, codes)
    out = []
    for v in range(len(cards)):
        fv = list(parents[v]) + [v]
        use = (log_p > -np.inf) & (codes[:, fv] == MISSING).any(1)
        out.append(fam[v][use].sum(0).reshape([cards[u] for u in fv]))
    return out


def clique_tables(structure, cpts) -> List[np.ndarray]:
    """fp64 table of every clique (row-major over its ascending members): the product of its assigned CPTs."""
    cards = structure.cards
    out = []
    for i, members in enumerate(structure.cliques):
        t = np.ones([cards[v] for v in members])
        for v, home in enumerate(structure.assign):
            if home != i:
                continue
            fv = list(structure.family_vars[v])
            cpt = np.asarray(cpts[v], np.float64).reshape([cards[u] for u in fv]).transpose([fv.index(u) for u in sorted(fv)])
            t = t * cpt.reshape([cards[u] if u in fv else 1 for u in members])
        out.append(t.reshape(-1))
    return out


def interpret(schedule, cpts, codes):
    """The plan run in fp64 over rows: ``(log_p [n], marginal run [n, marg_floats], family posteriors per op)``.  Follows
    the kernel op by op; dead rows give -inf and NaN."""
    from continuousbayesiannetwork_b200 import jt

    st = schedule.structure
    cards = st.cards
    codes = np.asarray(codes, np.int64)
    n = codes.shape[0]
    psi = clique_tables(st, cpts)
    maps = schedule.maps.astype(np.int64)
    msg = np.zeros((n, max(schedule.msg_floats, 1)))
    dead = _dead(cards, codes)
    log_p = np.zeros(n)
    digits = {}

    def ok(i):
        if i not in digits:
            members = st.cliques[i]
            digits[i] = np.indices([cards[v] for v in members]).reshape(len(members), -1)
        d = digits[i]
        m = np.ones((n, d.shape[1]), bool)
        for k, v in enumerate(st.cliques[i]):
            m &= (codes[:, v: v + 1] == MISSING) | (d[k][None, :] == codes[:, v: v + 1])
        return m

    def products(o):
        i = o["clique"]
        cells = st.cells(i)
        vals = psi[i][None, :] * ok(i)
        for m, mp in o["inputs"]:
            vals = vals * msg[:, m + maps[mp: mp + cells]]
        perm = np.arange(cells) if o["perm"] < 0 else maps[o["perm"]: o["perm"] + cells]
        return vals[:, perm].reshape(n, o["out_size"], -1).sum(2)

    marg = np.full((n, max(schedule.marg_floats, 1)), np.nan)
    fams: Dict[int, np.ndarray] = {}
    with np.errstate(divide="ignore", invalid="ignore"):
        for o in schedule.ops:
            k = o["kind"]
            out = products(o)
            if k in (jt.UP, jt.DOWN):
                mx = out.max(1)
                if k == jt.UP:
                    dead |= ~(mx > 0)
                    log_p += np.log(np.where(mx > 0, mx, 1.0))
                msg[:, o["out"]: o["out"] + o["out_size"]] = np.where(mx[:, None] > 0, out / mx[:, None], 0.0)
            elif k == jt.ROOT:
                dead |= ~(out[:, 0] > 0)
                log_p += np.log(np.where(out[:, 0] > 0, out[:, 0], 1.0))
            elif k == jt.NODE:
                marg[:, o["out"]: o["out"] + o["out_size"]] = out / out.sum(1, keepdims=True)
            else:
                fams[o["out"]] = out / out.sum(1, keepdims=True)
    log_p[dead] = -np.inf
    marg[dead] = np.nan
    for v in fams:
        fams[v][dead] = np.nan
    return log_p, marg[:, : schedule.marg_floats], fams


def random_masks(rng, codes, cards, rates=(0.0, 0.1, 0.5, 1.0)):
    """``codes`` with MISSING cells at a random per-row rate from ``rates`` (fully observed and fully missing rows
    included)."""
    codes = np.array(codes, np.int64)
    rate = np.asarray(rates)[rng.integers(0, len(rates), size=codes.shape[0])]
    mask = rng.random(codes.shape) < rate[:, None]
    codes[mask] = MISSING
    return codes
