"""fp64 reference of the per-row elimination executor (``cbn_ve_plan_create_rows``; csrc/ve.cu ``ve_rows_kernel`` and
``ve_rows_thread_kernel``): an interpreter of a per-row schedule (``VECompiler.last_row_schedule``) over the plan's own
static tables, vectorised over evidence rows.

It works in the log domain, so it has no range limit: ``interpret`` returns, for every row, the log of the last temporary
(posterior = softmax over the target, log-evidence = log-sum-exp).  A row with a code >= its variable's cardinality in a
column that some static table reads is dead (all -inf), as in the kernels.

``warp_rescales`` restates the warp kernel's range rule of linear plans (temporaries stored as computed, each one's scale
1/max folded into its consumer, a temporary whose maximum leaves [2^-12, 2^12] rescaled in place) only to report which
steps take the in-place branch; the values are always the unscaled fp64 ones."""
import numpy as np

LOG_2_12 = 12 * np.log(2.0)


def _strides(scope, cards):
    st, s = {}, 1
    for v in reversed(scope):
        st[v] = s
        s *= cards[v]
    return st


def _log(a):
    with np.errstate(divide="ignore"):
        return np.log(np.asarray(a, dtype=np.float64))


def _slice_bases(sch, cards, codes):
    """Per static table, the offset of every row's evidence slice; and the rows with an out-of-domain code in a column
    that some static table reads."""
    codes = np.asarray(codes, dtype=np.int64)
    slot = {v: i for i, v in enumerate(sch["evidence"])}
    dead = np.zeros(codes.shape[0], dtype=bool)
    bases = []
    for scope in sch["static_scopes"]:
        st = _strides(scope, cards)
        b = np.zeros(codes.shape[0], dtype=np.int64)
        for v in scope:
            if v in slot:
                c = codes[:, slot[v]]
                dead |= c >= cards[v]
                b += c * st[v]
        bases.append(b)
    return [np.where(dead, 0, b) for b in bases], dead


def interpret(sch, statics, cards, codes, log_tables=False, with_temps=False):
    """``sch``: a per-row schedule; ``statics[i]``: the flat table of ``sch["static_scopes"][i]`` as the executor reads it
    (logarithms when ``log_tables``); ``codes``: int [rows, len(evidence)].  Returns float64 [rows, last out_size]: the log
    of the last temporary (all -inf for a dead row); with ``with_temps`` also every temporary's log values."""
    bases, dead = _slice_bases(sch, cards, codes)
    n = dead.shape[0]
    tabs = [np.asarray(t, dtype=np.float64).reshape(-1) if log_tables else _log(t).reshape(-1) for t in statics]
    n_static = len(tabs)
    temps = []
    for st in sch["steps"]:
        n_in, out_size = len(st["in_id"]), st["out_size"]
        offs = sch["offsets"][st["offsets_at"]: st["offsets_at"] + n_in * out_size].reshape(n_in, out_size).astype(np.int64)
        acc = np.full((n, out_size), -np.inf)
        for sv in range(st["sum_card"]):
            term = np.zeros((n, out_size))
            for k, i in enumerate(st["in_id"]):
                idx = offs[k] + sv * st["sum_stride"][k]
                if i < n_static:
                    term = term + tabs[i][bases[i][:, None] + idx[None, :]]
                else:
                    term = term + temps[i - n_static][:, idx]
            acc = np.logaddexp(acc, term)
        temps.append(acc)
    last = temps[-1].copy()
    last[dead] = -np.inf
    return (last, temps) if with_temps else last


def posterior(log_last):
    """Softmax over the target; an all -inf row gives all zeros."""
    m = log_last.max(axis=1, keepdims=True)
    ok = np.isfinite(m[:, 0])
    out = np.zeros_like(log_last)
    e = np.exp(log_last[ok] - m[ok])
    out[ok] = e / e.sum(axis=1, keepdims=True)
    return out


def log_evidence(log_last):
    """Log-sum-exp over the last temporary: -inf for a dead row or evidence of probability zero."""
    m = log_last.max(axis=1)
    out = np.full(log_last.shape[0], -np.inf)
    ok = np.isfinite(m)
    out[ok] = m[ok] + np.log(np.exp(log_last[ok] - m[ok, None]).sum(axis=1))
    return out


def warp_rescales(sch, temps):
    """Bool [rows, steps]: where the warp kernel of a linear plan rescales a temporary in place.  ``temps``: the log
    temporaries of ``interpret(..., with_temps=True)``.  Restates the kernel's bookkeeping in logs: a temporary is stored
    as computed, its inputs' stored values times their scales; its scale is -max (log of 1/max, 0 for an all-zero
    temporary); outside [-12 ln 2, 12 ln 2] the stored values are multiplied by it in place and the scale becomes 0."""
    n_static = len(sch["static_scopes"])
    n = temps[0].shape[0]
    stored_off, scale = [], []                 # per step: log(stored / unscaled) and the log scale its consumer applies
    taken = np.zeros((n, len(sch["steps"])), dtype=bool)
    for j, st in enumerate(sch["steps"]):
        off = np.zeros(n)
        for i in st["in_id"]:
            if i >= n_static:
                off = off + stored_off[i - n_static] + scale[i - n_static]
        mx = temps[j].max(axis=1) + off
        live = np.isfinite(mx)
        sc = np.where(live, -np.where(live, mx, 0.0), 0.0)
        big = live & (np.abs(sc) > LOG_2_12)
        taken[:, j] = big
        stored_off.append(np.where(big, off + sc, off))
        scale.append(np.where(big, 0.0, sc))
    return taken
