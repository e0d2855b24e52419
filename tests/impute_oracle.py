"""fp64 references of junction-tree decoding with per-row missing values (``cbn_jt_decode``).  TEST INFRASTRUCTURE ONLY.

Nothing under ``continuousbayesiannetwork_b200/`` imports this file.  Networks and codes are those of ``jt_oracle``:
``codes`` are int [n_rows, n_vars], a code below the cardinality is observed, ``MISSING`` (254) is not, anything else
makes the row dead.

* ``enumerate_mpe_rows``: the best and second-best log joint over the completions consistent with each row, and the
  best completion, by enumeration (small networks only);
* ``interpret_decode``: the collect-only plan's own tables (``jt.Schedule``) run op by op in fp64, vectorised over rows,
  then decoded top-down with the kernel's rules; in SAMPLE mode it also returns the product of the clique conditionals
  each draw was drawn from, which equals ``P(completion | observed)`` when the decode is right.
"""
from __future__ import annotations

import numpy as np

import jt_oracle as JO

MISSING = JO.MISSING
UNSEEN = 255


def log_joint(cards, parents, cpts, rows) -> np.ndarray:
    """fp64 log P of complete rows (int [n, n_vars], every code inside its domain)."""
    rows = np.asarray(rows, np.int64)
    out = np.zeros(rows.shape[0])
    with np.errstate(divide="ignore"):
        for v in range(len(cards)):
            out += np.log(np.asarray(cpts[v], np.float64)[tuple(rows[:, p] for p in parents[v]) + (rows[:, v],)])
    return out


def enumerate_mpe_rows(cards, parents, cpts, codes, chunk: int = 256):
    """``(best [n], second [n], argmax int [n, n_vars])``: the best and second-best log joint over the completions
    consistent with each row (second = -inf when there is no other completion of positive probability) and the best
    completion (the first in row-major order among equals; -1 where best is -inf).  Dead rows give -inf."""
    codes = np.asarray(codes, np.int64)
    n, nv = codes.shape
    total = int(np.prod(cards))
    assert total <= 1 << 18, "enumeration oracle is for small networks"
    grid = np.indices(cards).reshape(nv, -1)
    lj = log_joint(cards, parents, cpts, grid.T)
    dead = JO._dead(cards, codes)
    best = np.full(n, -np.inf)
    second = np.full(n, -np.inf)
    arg = np.full((n, nv), -1, np.int64)
    for s in range(0, n, chunk):
        c = codes[s: s + chunk]
        ok = np.ones((c.shape[0], total), bool)
        for v in range(nv):
            ok &= (c[:, v: v + 1] == MISSING) | (grid[v][None, :] == c[:, v: v + 1])
        vals = np.where(ok, lj[None, :], -np.inf)
        top = vals.argmax(1)
        b = vals[np.arange(len(c)), top]
        vals[np.arange(len(c)), top] = -np.inf
        sec = vals.max(1)
        live = np.isfinite(b) & ~dead[s: s + chunk]
        best[s: s + chunk] = np.where(live, b, -np.inf)
        second[s: s + chunk] = np.where(live, sec, -np.inf)
        arg[s: s + chunk] = np.where(live[:, None], grid[:, top].T, -1)
    return best, second, arg


def interpret_decode(schedule, cpts, codes, mode, seed=0, first_row=0, n_draws=1):
    """The collect-only plan run in fp64 and decoded per ``cbn_jt_decode``'s rules (mode 0: MAX, 1: SAMPLE).  Returns a
    dict: ``codes`` int [n_draws, n, n_vars] (UNSEEN in every column of a dead row), ``log`` [n] (MAX: log max_h P(h, e);
    SAMPLE: log P(e); -inf for dead rows), ``prob`` [n_draws, n] (SAMPLE: the product of the clique conditionals the draw
    was drawn from), ``margin`` [n_draws, n] (SAMPLE: the smallest distance of u * total to a cumulative boundary of a
    decoded clique, relative to the total; +inf where nothing was drawn)."""
    from continuousbayesiannetwork_b200 import jt, synth

    st = schedule.structure
    cards = st.cards
    codes = np.asarray(codes, np.int64)
    n = codes.shape[0]
    psi = JO.clique_tables(st, cpts)
    maps = schedule.maps.astype(np.int64)
    msg = np.zeros((n, max(schedule.msg_floats, 1)))
    digits = [np.indices([cards[v] for v in m]).reshape(len(m), -1) for m in st.cliques]
    assert all(o["kind"] in (jt.UP, jt.ROOT) for o in schedule.ops) and schedule.ops[-1]["kind"] == jt.ROOT

    def weights(o, work):
        i = o["clique"]
        d = digits[i]
        ok = np.ones((n, d.shape[1]), bool)
        for k, v in enumerate(st.cliques[i]):
            ok &= (work[:, v: v + 1] == MISSING) | (d[k][None, :] == work[:, v: v + 1])
        w = psi[i][None, :] * ok
        for m, mp in o["inputs"]:
            w = w * msg[:, m + maps[mp: mp + d.shape[1]]]
        return w

    maxprod = mode == 0
    dead = JO._dead(cards, codes)
    log_v = np.zeros(n)
    with np.errstate(divide="ignore", invalid="ignore"):
        for o in schedule.ops:
            cells = st.cells(o["clique"])
            perm = np.arange(cells) if o["perm"] < 0 else maps[o["perm"]: o["perm"] + cells]
            g = weights(o, codes)[:, perm].reshape(n, o["out_size"], -1)
            out = g.max(2) if maxprod else g.sum(2)
            mx = out.max(1)
            dead |= ~(mx > 0)
            log_v += np.log(np.where(mx > 0, mx, 1.0))
            if o["kind"] == jt.UP:
                msg[:, o["out"]: o["out"] + o["out_size"]] = np.where(mx[:, None] > 0, out / mx[:, None], 0.0)
    rows = np.arange(n)
    out_codes = np.zeros((n_draws, n, len(cards)), np.int64)
    prob = np.ones((n_draws, n))
    margin = np.full((n_draws, n), np.inf)
    for d in range(n_draws):
        work = codes.copy()
        bad = dead.copy()
        for o in reversed(schedule.ops):
            i = o["clique"]
            members = st.cliques[i]
            todo = (work[:, members] == MISSING).any(1) & ~bad
            if not todo.any():
                continue
            w = weights(o, work)
            total = w.sum(1)
            if maxprod:
                x = w.argmax(1)
            else:
                u = synth.posterior_uniforms(seed, first_row + rows, d, i).astype(np.float64)
                target = u * total
                cum = np.cumsum(w, 1)
                hit = (cum > target[:, None]) & (w > 0)
                last = w.shape[1] - 1 - (w[:, ::-1] > 0).argmax(1)
                x = np.where(hit.any(1), hit.argmax(1), last)
                with np.errstate(divide="ignore", invalid="ignore"):
                    gap = np.where(w > 0, np.abs(cum - target[:, None]), np.inf).min(1) / total
                    p = w[rows, x] / total
                margin[d] = np.where(todo, np.minimum(margin[d], gap), margin[d])
                prob[d] = np.where(todo, prob[d] * p, prob[d])
            zero = ~(total > 0)
            bad |= todo & zero
            sel = todo & ~zero
            work[np.ix_(sel, members)] = digits[i][:, x[sel]].T
        work[bad] = UNSEEN
        out_codes[d] = work
        dead = dead | bad
    log_v[dead] = -np.inf
    out_codes[:, dead] = UNSEEN
    return {"codes": out_codes, "log": log_v, "prob": prob, "margin": margin}
