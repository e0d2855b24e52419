"""Junction-tree compiler: one structure per network, calibrated per row with that row's own observed set.

Every other query mode compiles a plan for ONE observed set, shared by all rows of a call.  Tabular data with missing
cells has a different observed set in almost every row, so here the structure is compiled once per network and the
evidence enters each row as indicators:

* the moral graph is triangulated by greedy min-fill (ties: the smaller clique, then the lower id); the clique of an
  eliminated variable hangs below the clique of its first later-eliminated member, which gives the running-intersection
  property by construction; cliques contained in a neighbour are merged away, and the roots of a forest are chained
  below one root with empty separators;
* every CPT is assigned to the smallest clique that contains its family (the family's home); a clique's table is the
  product of its CPTs, contracted on the device (``cbn_factor_contract`` without a summed variable), all ones if none;
* a node's home is the smallest clique that contains it.

``cbn_jt_run`` (csrc/jt.cu) calibrates the tree per row by Shafer-Shenoy message passing: a collect pass towards the
root (which yields ``log P(observed part of the row)``), a distribute pass towards the cliques that host an output, then
every requested node marginal and, for EM, every family posterior of a row in which the family has a missing member.
``cbn_jt_decode`` runs the collect pass only (sum- or max-product) and decodes the cliques top-down: the most probable
completion of the row's missing cells, or joint draws of them; its plan is the collect-only schedule (UP and ROOT ops).
Host work here is graph logic and int32 / int16 index tables only.

Evidence codes per row: below the cardinality is observed, ``MISSING`` (254) is summed out, anything else makes the row
dead (``log P = -inf``, NaN marginals, no counts).  A node of cardinality 255 would make 254 a value, so it is refused.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _native as N
from .ve import Factor, PlanTooLarge, _Pass, _strides

MISSING = 254                    # CBN_MISSING: not observed in this row
MAX_CLIQUE_CELLS = 4096          # largest clique table (the kernel's maps are int16)
MAX_CLIQUES = 512
SMEM_BUDGET_BYTES = 200 * 1024   # plan tables + one warp's per-row floats; the kernel stages both in shared memory
SMEM_FAMILY_TABLE_BYTES = 32 * 1024   # family tables the kernel privatises in shared memory (JT_SMEM_TABLE_BYTES)
UP, ROOT, DOWN, NODE, FAMILY = 0, 1, 2, 3, 4
NEED_NODES, NEED_FAMILIES = 1, 2


# ------------------------------------------------------------------------------------------------ structure
def min_fill_order(cards: Sequence[int], family_vars: Sequence[Sequence[int]], max_clique_cells: int = MAX_CLIQUE_CELLS):
    """Greedy min-fill elimination of the moral graph: (order, elimination cliques).  Ties go to the smaller clique
    (cells), then the lower id.  A clique above ``max_clique_cells`` raises ``PlanTooLarge`` as soon as it appears."""
    n = len(cards)
    adj = [set() for _ in range(n)]
    for fv in family_vars:
        for a in fv:
            for b in fv:
                if a != b:
                    adj[a].add(b)
    alive = set(range(n))
    score: Dict[int, tuple] = {}

    def evaluate(v):
        nb = list(adj[v])
        fill = sum(1 for i in range(len(nb)) for j in range(i + 1, len(nb)) if nb[j] not in adj[nb[i]])
        return fill, math.prod(cards[u] for u in nb) * cards[v], v

    for v in range(n):
        score[v] = evaluate(v)
    order, cliques = [], []
    while alive:
        v = min(alive, key=lambda u: score[u])
        clique = sorted(adj[v] | {v})
        cells = math.prod(cards[u] for u in clique)
        if cells > max_clique_cells:
            raise PlanTooLarge(f"the junction tree needs a clique of {cells} cells (budget {max_clique_cells}): the network's "
                               "treewidth is too large for per-row calibration")
        order.append(v)
        cliques.append(clique)
        nb = list(adj[v])
        for a in nb:
            adj[a].discard(v)
            adj[a].update(u for u in nb if u != a)
        alive.discard(v)
        del score[v]
        touched = set(nb)
        for a in nb:
            touched |= adj[a]
        for u in touched & alive:
            score[u] = evaluate(u)
    return order, cliques


@dataclass
class Structure:
    """A junction tree over network ids: ``cliques[i]`` ascending, ``parent[i]`` (-1: the root), ``children[i]``,
    ``collect`` (children before parents, root last), ``assign[v]`` (home clique of v's family), ``home[v]`` (smallest
    clique holding v)."""
    cards: List[int]
    family_vars: List[List[int]]
    cliques: List[List[int]]
    parent: List[int]
    root: int
    children: List[List[int]] = field(default_factory=list)
    collect: List[int] = field(default_factory=list)
    assign: List[int] = field(default_factory=list)
    home: List[int] = field(default_factory=list)

    def cells(self, i: int) -> int:
        return math.prod(self.cards[v] for v in self.cliques[i])

    def separator(self, i: int) -> List[int]:
        """Variables shared by clique ``i`` and its parent (ascending)."""
        p = self.parent[i]
        return sorted(set(self.cliques[i]) & set(self.cliques[p])) if p >= 0 else []


def build_structure(cards: Sequence[int], family_vars: Sequence[Sequence[int]],
                    max_clique_cells: int = MAX_CLIQUE_CELLS, max_cliques: int = MAX_CLIQUES) -> Structure:
    cards = [int(c) for c in cards]
    fams = [list(f) for f in family_vars]
    order, ecl = min_fill_order(cards, fams, max_clique_cells)
    pos = {v: i for i, v in enumerate(order)}
    # clique k belongs to order[k]; its parent is the clique of its first later-eliminated member
    members = [set(c) for c in ecl]
    parent = []
    for k, v in enumerate(order):
        rest = [u for u in ecl[k] if u != v]
        parent.append(pos[min(rest, key=lambda u: pos[u])] if rest else -1)
    alive = set(range(len(order)))

    def kids(k):
        return sorted(c for c in alive if parent[c] == k)

    changed = True
    while changed:                       # merge every clique contained in a neighbour into that neighbour
        changed = False
        for k in sorted(alive):
            p = parent[k]
            if p >= 0 and members[k] <= members[p]:
                for c in kids(k):
                    parent[c] = p
                alive.discard(k)
                changed = True
                break
            sub = next((c for c in kids(k) if members[k] <= members[c]), None)
            if sub is not None:
                parent[sub] = p
                for c in kids(k):
                    if c != sub:
                        parent[c] = sub
                alive.discard(k)
                changed = True
                break
    roots = sorted(k for k in alive if parent[k] < 0)          # clique k is the k-th eliminated
    for k in roots[:-1]:                 # a forest: the other roots hang below the last one (empty separators)
        parent[k] = roots[-1]
    keep = sorted(alive)
    if len(keep) > max_cliques:
        raise PlanTooLarge(f"the junction tree has {len(keep)} cliques (budget {max_cliques})")
    new = {k: i for i, k in enumerate(keep)}
    cliques = [sorted(members[k]) for k in keep]
    par = [new[parent[k]] if parent[k] >= 0 else -1 for k in keep]
    st = Structure(cards, fams, cliques, par, par.index(-1))
    st.children = [[] for _ in keep]
    for i, p in enumerate(par):
        if p >= 0:
            st.children[p].append(i)
    stack, post = [(st.root, False)], []
    while stack:
        i, done = stack.pop()
        if done:
            post.append(i)
            continue
        stack.append((i, True))
        for c in reversed(st.children[i]):
            stack.append((c, False))
    st.collect = post
    sizes = [st.cells(i) for i in range(len(cliques))]
    sets = [set(c) for c in cliques]
    st.assign = [min((i for i in range(len(cliques)) if set(fv) <= sets[i]), key=lambda i: (sizes[i], i)) for fv in fams]
    st.home = [min((i for i in range(len(cliques)) if v in sets[i]), key=lambda i: (sizes[i], i)) for v in range(len(cards))]
    return st


# ------------------------------------------------------------------------------------------------ per-row schedule
def _layout_map(st: Structure, i: int, out_vars: Sequence[int]) -> np.ndarray:
    """Canonical cell of clique ``i`` for every (output cell, fiber cell): int64 [cells], output-major.  The output is
    row-major over ``out_vars`` (in that order), the fiber row-major over the other members (ascending)."""
    cl, cards = st.cliques[i], st.cards
    rest = [v for v in cl if v not in out_vars]
    axes = list(out_vars) + rest
    canon = _strides(cl, cards)
    grid = np.indices([cards[v] for v in axes]).reshape(len(axes), -1) if axes else np.zeros((0, 1), np.int64)
    cell = np.zeros(grid.shape[1], np.int64)
    for d, v in enumerate(axes):
        cell += grid[d] * canon[v]
    return cell


def _sep_map(st: Structure, i: int, sep: Sequence[int]) -> np.ndarray:
    """Separator cell (row-major over ``sep``, ascending) of every canonical cell of clique ``i``: int64 [cells]."""
    cl, cards = st.cliques[i], st.cards
    grid = np.indices([cards[v] for v in cl]).reshape(len(cl), -1) if cl else np.zeros((0, 1), np.int64)
    sst = _strides(sep, cards)
    out = np.zeros(grid.shape[1], np.int64)
    for d, v in enumerate(cl):
        if v in sst:
            out += grid[d] * sst[v]
    return out


@dataclass
class Schedule:
    """The per-row program, as ``cbn_jt_plan_create`` receives it (also read by the fp64 interpreter of the tests).

    ``ops``: dicts with kind, clique, out_vars, out_size, perm (offset in ``maps`` of the output-major layout, -1:
    identity), inputs ([(message offset, offset in ``maps`` of the clique-cell -> separator-cell map)]), out (message
    offset, offset in the row's marginal run, or the family's node), needed (DOWN: NEED_NODES | NEED_FAMILIES).
    ``msg_floats``: messages per row; ``scratch_floats``: the largest node / family output; ``marg_floats``: the row's
    marginal run (``node_out``: node -> offset)."""
    structure: Structure
    ops: List[dict]
    maps: np.ndarray
    msg_floats: int
    scratch_floats: int
    nodes: List[int]
    node_out: Dict[int, int]
    marg_floats: int

    def row_floats(self) -> int:
        return self.msg_floats + self.scratch_floats

    def madds_per_row(self, kinds=(UP, ROOT, DOWN, NODE, FAMILY)) -> int:
        """Multiply-adds of a row whose every op runs: clique cells x (1 + incoming messages) per op."""
        st = self.structure
        return sum(st.cells(o["clique"]) * (1 + len(o["inputs"])) for o in self.ops if o["kind"] in kinds)

    def shared_bytes(self, warps: int = 1) -> int:
        """Shared memory of one CTA with ``warps`` warps: the layout of ``cbn_jt_plan_create``, restated (ops of 104 B,
        cliques of 32 B, members, cardinalities, input pairs, clique tables, int16 maps, member digits, the privatised
        family tables, the code tile of 32 rows, then one row's floats per warp; every section 16-byte aligned)."""
        st = self.structure
        a16 = lambda x: (x + 15) // 16 * 16
        cells = [st.cells(i) for i in range(len(st.cliques))]
        priv = 0
        for o in self.ops:                      # privatised first come first served, up to 32 KB, stopping at the first miss
            if o["kind"] == FAMILY:
                if (priv + o["out_size"]) * 8 > SMEM_FAMILY_TABLE_BYTES:
                    break
                priv += o["out_size"]
        sections = [104 * len(self.ops), 32 * len(st.cliques), 4 * sum(len(c) for c in st.cliques), 4 * len(st.cards),
                    8 * sum(len(o["inputs"]) for o in self.ops), 4 * sum(cells), 2 * int(self.maps.size),
                    sum(c * len(m) for c, m in zip(cells, st.cliques)), 8 * priv, 32 * len(st.cards)]
        return sum(a16(x) for x in sections) + warps * 4 * self.row_floats()


def build_schedule(st: Structure, nodes: Sequence[int], row_floats_budget: int = 5000,
                   smem_budget: int = SMEM_BUDGET_BYTES, collect_only: bool = False) -> Schedule:
    """The per-row program with ``nodes`` as outputs; ``collect_only``: the UP ops and the ROOT op alone (no down
    messages, ``nodes`` must be empty), the program ``cbn_jt_decode`` runs."""
    assert not (collect_only and len(nodes)), "a collect-only schedule has no outputs"
    cards = st.cards
    nodes = list(nodes)
    n_cl = len(st.cliques)
    maps: List[np.ndarray] = []
    at = 0

    def put(a):
        nonlocal at
        maps.append(a.astype(np.int16))
        at += a.size
        return at - a.size

    # messages: up[i] (i -> parent), down[i] (parent -> i), each row-major over the separator
    msg, up, down = 0, {}, {}
    for i in st.collect:
        if st.parent[i] >= 0:
            s = math.prod(cards[v] for v in st.separator(i))
            up[i] = msg
            msg += s
    # which down messages an output needs: every clique on the way from the root to its home
    need = [0] * n_cl
    outputs = () if collect_only else ((NEED_NODES, [st.home[v] for v in nodes]), (NEED_FAMILIES, list(st.assign)))
    for bit, homes in outputs:
        for h in homes:
            while h >= 0 and not need[h] & bit:
                need[h] |= bit
                h = st.parent[h]
    for i in range(n_cl):
        if st.parent[i] >= 0 and need[i]:
            down[i] = msg
            msg += math.prod(cards[v] for v in st.separator(i))
    # clique-cell -> separator-cell maps, one per directed edge into a clique
    in_map = {}
    for i in range(n_cl):
        p = st.parent[i]
        if p < 0:
            continue
        sep = st.separator(i)
        in_map[(i, p)] = put(_sep_map(st, p, sep))      # up[i] read by p
        if i in down:
            in_map[(p, i)] = put(_sep_map(st, i, sep))  # down[i] read by i

    def inputs(i, exclude):
        ins = [(up[c], in_map[(c, i)]) for c in st.children[i] if c != exclude]
        if st.parent[i] >= 0 and st.parent[i] != exclude and i in down:
            ins.append((down[i], in_map[(st.parent[i], i)]))
        return ins

    def op(kind, i, out_vars, exclude, out, needed=0):
        out_vars = list(out_vars)
        size = math.prod(cards[v] for v in out_vars)
        ident = out_vars == st.cliques[i][: len(out_vars)]
        return {"kind": kind, "clique": i, "out_vars": out_vars, "out_size": size,
                "perm": -1 if ident else put(_layout_map(st, i, out_vars)), "inputs": inputs(i, exclude),
                "out": out, "needed": needed}

    ops = []
    for i in st.collect:
        if st.parent[i] >= 0:
            ops.append(op(UP, i, st.separator(i), st.parent[i], up[i]))
    ops.append(op(ROOT, st.root, [], None, 0))
    for i in reversed(st.collect):                       # parents before children
        for c in st.children[i]:
            if c in down:
                ops.append(op(DOWN, i, st.separator(c), c, down[c], need[c]))
    node_out, run = {}, 0
    for v in nodes:
        node_out[v] = run
        ops.append(op(NODE, st.home[v], [v], None, run))
        run += cards[v]
    for v, fv in enumerate([] if collect_only else st.family_vars):
        ops.append(op(FAMILY, st.assign[v], fv, None, v))
    scratch = max([o["out_size"] for o in ops if o["kind"] in (NODE, FAMILY)] + [1])
    sch = Schedule(st, ops, np.concatenate(maps) if maps else np.zeros(0, np.int16), msg, scratch, nodes, node_out, run)
    if sch.row_floats() > row_floats_budget:
        raise PlanTooLarge(f"junction-tree calibration needs {sch.row_floats()} floats of messages per row (budget "
                           f"{row_floats_budget})")
    if sch.shared_bytes(1) > smem_budget:
        raise PlanTooLarge(f"the junction tree's tables and one row's messages need {sch.shared_bytes(1)} bytes of shared "
                           f"memory (budget {smem_budget})")
    return sch


def compile_structure(tables, row_floats_budget: int = 5000) -> Schedule:
    """Structure and full schedule (every node an output) of ``tables`` (``DiscreteTables`` or ``DryTables``); raises
    ``PlanTooLarge`` for a node of cardinality 255 or a tree over a budget.  No device work."""
    cards = list(tables.cards)
    for v, c in enumerate(cards):
        if c > MISSING:
            raise PlanTooLarge(f"node {tables.names[v]} has cardinality {c}: per-row missing values need codes up to "
                               f"{MISSING - 1} (code {MISSING} marks a missing cell)")
    fams = [tables.family_vars(n) for n in tables.names]
    st = build_structure(cards, fams)
    return build_schedule(st, range(len(cards)), row_floats_budget)


# ------------------------------------------------------------------------------------------------ device plans
class JTPlan:
    """Owner of one ``cbn_jt_plan`` (a schedule with its output nodes) over the clique tables of a ``JunctionTree``."""

    def __init__(self, tree: "JunctionTree", sch: Schedule):
        t = tree.t
        self.t, self.schedule, self.tree = t, sch, tree
        st = sch.structure
        cl = (N.JtClique * len(st.cliques))()
        for i, members in enumerate(st.cliques):
            cl[i].n_members = len(members)
            for k, v in enumerate(members):
                cl[i].member[k] = v
            cl[i].table_offset = tree.table_offsets[i]
        ops = (N.JtOp * len(sch.ops))()
        flat_in = []
        for k, o in enumerate(sch.ops):
            d = ops[k]
            d.kind, d.clique, d.out_size, d.perm = o["kind"], o["clique"], o["out_size"], o["perm"]
            d.n_in, d.in_at, d.out, d.needed = len(o["inputs"]), len(flat_in) // 2, o["out"], o["needed"]
            d.n_out_vars = len(o["out_vars"]) if o["kind"] in (NODE, FAMILY) else 0
            for j, v in enumerate(o["out_vars"] if d.n_out_vars else []):
                d.out_var[j] = v
            d.table_offset = t.offsets[o["out"]] if o["kind"] == FAMILY else 0
            for m, mp in o["inputs"]:
                flat_in += [m, mp]
        cards = (C.c_int32 * len(st.cards))(*st.cards)
        ins = (C.c_int32 * max(len(flat_in), 1))(*flat_in)
        maps = np.ascontiguousarray(sch.maps, dtype=np.int16)
        h = C.c_void_p()
        N.check(N.lib().cbn_jt_plan_create(t.ctx.handle, len(st.cards), cards, len(st.cliques), cl, tree.tables.data_ptr(),
                                           int(tree.tables.numel()), len(sch.ops), ops, ins, len(flat_in) // 2,
                                           maps.ctypes.data_as(C.POINTER(C.c_int16)), int(maps.size), sch.msg_floats,
                                           sch.scratch_floats, sch.marg_floats, N.stream_ptr(t.device), C.byref(h)),
                t.ctx.handle)
        self.handle = h

    def run(self, codes, n_rows: int, marg_out=None, log_out=None, acc=None):
        """``codes``: uint8 [n_vars, ld] (network ids as rows); outputs as in ``cbn_jt_run`` (each may be None)."""
        t = self.t
        ptr = lambda x: None if x is None else x.data_ptr()
        N.check(N.lib().cbn_jt_run(t.ctx.handle, self.handle, codes.data_ptr(), codes.stride(0), int(n_rows), ptr(marg_out),
                                   ptr(log_out), ptr(acc), N.stream_ptr(t.device)), t.ctx.handle)

    def decode(self, codes, n_rows: int, mode: int, n_draws: int, seed: int, first_row: int, out_codes, log_out=None):
        """``cbn_jt_decode``: ``codes`` as in ``run``; ``mode`` ``N.JT_DECODE_MAX`` or ``N.JT_DECODE_SAMPLE``;
        ``out_codes``: uint8 [n_draws * n_vars, out_ld] (row ``d * n_vars + v``: draw d of variable v); ``log_out``: float32
        [n_rows] or None."""
        t = self.t
        N.check(N.lib().cbn_jt_decode(t.ctx.handle, self.handle, codes.data_ptr(), codes.stride(0), int(n_rows), int(mode),
                                      int(seed) & ((1 << 64) - 1), int(first_row), int(n_draws), out_codes.data_ptr(),
                                      out_codes.stride(0), None if log_out is None else log_out.data_ptr(),
                                      N.stream_ptr(t.device)), t.ctx.handle)

    def __del__(self):
        try:
            if self.handle is not None:
                N.lib().cbn_jt_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class JunctionTree:
    """The compiled tree of one network: the structure, the clique tables on the device (float32, canonical layout,
    concatenated) and one native plan per requested set of output nodes."""

    def __init__(self, compiler, schedule: Schedule):
        t = self.t = compiler.t
        self.compiler = compiler
        self.schedule = schedule
        st = schedule.structure
        import torch

        cx = _Pass([], None, False, False, False)
        offs, parts, at = [], [], 0
        by_clique: Dict[int, List[int]] = {}
        for v, i in enumerate(st.assign):
            by_clique.setdefault(i, []).append(v)
        for i, members in enumerate(st.cliques):
            fams = [Factor(list(st.family_vars[v]), t.table_view(t.cond, t.names[v]).reshape(-1)) for v in by_clique.get(i, [])]
            if not fams:
                tab = torch.ones(st.cells(i), dtype=torch.float32, device=t.device)
            else:
                while len(fams) > N.MAX_CONTRACT_INPUTS:        # pre-multiply: the contraction takes 16 inputs
                    head = fams[: N.MAX_CONTRACT_INPUTS]
                    sc = sorted(set().union(*[f.scope for f in head]))
                    fams = [compiler._contract(head, sc, None, cx)] + fams[N.MAX_CONTRACT_INPUTS:]
                tab = compiler._contract(fams, list(members), None, cx).tensor[: st.cells(i)]
            offs.append(at)
            parts.append(tab)
            at += st.cells(i)
        self.tables = torch.cat(parts).contiguous()
        self.table_offsets = offs
        self._plans: Dict[tuple, JTPlan] = {}

    def plan(self, nodes: Optional[Sequence[int]] = None) -> JTPlan:
        key = tuple(range(len(self.t.cards))) if nodes is None else tuple(nodes)
        if key not in self._plans:
            self._plans[key] = JTPlan(self, schedule_for(self.compiler, key))
        return self._plans[key]

    def collect_plan(self) -> JTPlan:
        """The plan of the collect-only schedule (``cbn_jt_decode``), cached like ``plan``."""
        if "collect" not in self._plans:
            self._plans["collect"] = JTPlan(self, collect_schedule(self.compiler))
        return self._plans["collect"]


def schedule_for(compiler, nodes: Optional[Sequence[int]] = None) -> Schedule:
    """The schedule of the compiler's network with ``nodes`` as outputs (default: every node).  It depends on the structure
    only, so it is kept in ``compiler.structures`` across CPT changes (an EM iteration rebuilds the clique tables only);
    the full schedule is built first, so its budgets decide whether the network is refused."""
    t = compiler.t
    full = tuple(range(len(t.cards)))
    key = full if nodes is None else tuple(nodes)
    base = ("jt", tuple(t.cards))
    if base + (full,) not in compiler.structures:
        compiler.structures[base + (full,)] = compile_structure(t, compiler.row_temp_floats)
    if base + (key,) not in compiler.structures:
        st = compiler.structures[base + (full,)].structure
        compiler.structures[base + (key,)] = build_schedule(st, key, compiler.row_temp_floats)
    return compiler.structures[base + (key,)]


def collect_schedule(compiler) -> Schedule:
    """The collect-only schedule (UP and ROOT ops; ``msg_floats`` counts the up messages only) of the compiler's network,
    kept in ``compiler.structures`` beside the others.  The full schedule is built first, so the same budgets refuse a
    network here as in ``posterior_marginals``."""
    key = ("jt", tuple(compiler.t.cards), "collect")
    if key not in compiler.structures:
        st = schedule_for(compiler).structure
        compiler.structures[key] = build_schedule(st, [], compiler.row_temp_floats, collect_only=True)
    return compiler.structures[key]


def compile_tree(compiler, dry: bool = False):
    """The junction tree of the compiler's tables, cached under ``("jt",)`` (dropped when the CPTs change; the structure
    and schedules are kept, see ``schedule_for``).  ``dry``: the full schedule only (``DryTables`` work; no device)."""
    if dry:
        return schedule_for(compiler)
    return compiler.cached(("jt",), lambda: JunctionTree(compiler, schedule_for(compiler)))
