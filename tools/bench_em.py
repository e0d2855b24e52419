"""Cost of one EM iteration on one GPU, phase by phase; prints ONE JSON line.

Workloads (data: sample() of seeded networks, hidden rows dropped):
  * latent class: one hidden node Z (card 4) and 20 observed children (card 3), 2^24 rows -- one group, one chain step;
  * Alarm with its four ALARM_TARGETS hidden and the other 33 nodes observed, 2^24 rows -- five groups, one of two steps;
  * Alarm with every node but ALARM_EVIDENCE hidden (25 hidden, chains of up to 5 steps), 2^22 rows.
Each runs EM from Dirichlet(1) rows (seed 0) for a warm-up iteration and then --iters timed iterations.  Per iteration:
  * compile_ms: host clock around compiling every chain plan and the log P(e) plan after the M-step changed the CPTs
    (ends in a device synchronise; includes the contraction kernels);
  * gather_us: CUDA events around the chain's posterior runs (and the constant-row fills between them);
  * ess_us: CUDA events around the cbn_ess_run launches, with the kernel's model: bytes per row (chain factors read +
    observed codes read) and atomics per row (destinations x joint configurations, an upper bound: w = 0 adds nothing);
  * loglik_us: CUDA events around the log P(e) runs and their float64 sums; mstep_us likewise for the CPT kernel;
  * iteration_ms: host clock around the whole E-step + M-step, compile included (ends in a device synchronise).
The inputs are larger than the 126 MB L2 (2^24 rows x 33 observed codes = 554 MB).  In the same run the expected counts
of the families with hidden members over the first 4,096 rows under the final CPTs are checked against an fp64 numpy E-step by enumeration (tests/em_oracle.py)
on the two workloads whose hidden set enumerates (16 configurations at most); the deep Alarm workload reports instead the
largest deviation of a family's total expected count from the number of live rows.  The card name and power limit are
read in the same run.

    python tools/bench_em.py [--iters 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from continuousbayesiannetwork_b200 import _native as N  # noqa: E402
from continuousbayesiannetwork_b200 import synth  # noqa: E402
from continuousbayesiannetwork_b200.em import EM, chain_floats  # noqa: E402
from continuousbayesiannetwork_b200.engine import bind_inference, sample_network, tables_from_spec  # noqa: E402
import em_oracle as EO  # noqa: E402

DEV = "cuda:0"


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:            # the numbers are still reported, without their power limit
        out = f"unavailable ({e})"
    return name, out


def _workloads():
    names, cards, parents, cpts = EO.latent_class(n_children=20, k=4, card=3, seed=0)
    lc = synth.NetSpec(names, cards, parents, cpts)
    alarm = synth.alarm()
    ev = {alarm.names.index(n) for n in synth.ALARM_EVIDENCE}
    return [("latent_class_z4_x20", lc, [0], 1 << 24),
            ("alarm_targets_hidden", alarm, [alarm.names.index(n) for n in synth.ALARM_TARGETS], 1 << 24),
            ("alarm_all_but_evidence_hidden", alarm, [v for v in range(alarm.n) if v not in ev], 1 << 22)]


class _Events:
    def __init__(self):
        self.us = 0.0
        self.pairs = []

    def __enter__(self):
        self.e0 = torch.cuda.Event(enable_timing=True)
        self.e0.record()

    def __exit__(self, *a):
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        self.pairs.append((self.e0, e1))

    def total_us(self):
        torch.cuda.synchronize()
        return 1e3 * sum(a.elapsed_time(b) for a, b in self.pairs)


def _iteration(em):
    """One EM iteration with every phase timed: the E-step of EM.e_step, split by phase."""
    t = em.t
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    c0 = time.perf_counter()
    for g in em.groups:
        for j, h in enumerate(g.hidden):
            em.infer.plan(t.names[h], em.ev_names + [t.names[u] for u in g.hidden[:j]])
    em.infer.evidence_plan(em.ev_names)
    torch.cuda.synchronize()
    compile_ms = 1e3 * (time.perf_counter() - c0)
    gather, ess, ll, mstep = _Events(), _Events(), _Events(), _Events()
    em.acc.copy_(em.base)
    sums = em._new_sums()
    for s in range(0, em.n, em.chunk):
        c = min(em.chunk, em.n - s)
        with ll:
            em._log_likelihood(s, c, sums)
        for g, plan in zip(em.groups, em.ess):
            with gather:
                factors = em.chain_factors(g, s, c)
            with ess:
                plan.run(factors, em.codes[:, s:], c, em.acc, em.stream)
    with mstep:
        em.m_step()
    torch.cuda.synchronize()
    whole_ms = 1e3 * (time.perf_counter() - w0)
    return {"compile_ms": round(compile_ms, 3), "gather_us": round(gather.total_us(), 1), "ess_us": round(ess.total_us(), 1),
            "loglik_us": round(ll.total_us(), 1), "mstep_us": round(mstep.total_us(), 1), "iteration_ms": round(whole_ms, 3),
            "log_likelihood": float(sums[0].item())}


def _check(spec, hidden, t, infer, codes, n_check=4096):
    """Expected counts of the first n_check rows under the current CPTs: device vs fp64."""
    em = EM(t, infer, codes, n_check, hidden)
    em.e_step()
    got = em.expected_counts().cpu().numpy()
    fams = [f for g in em.groups for f in g.families]          # the observed families' counts are those of every row
    if np.prod([spec.cards[h] for h in hidden]) > 16:
        dev = max(abs(got[t.offsets[v]: t.offsets[v] + t.n_cells[v]].sum() - n_check) for v in fams)
        return {"rows": n_check, "max_family_total_minus_rows": float(dev)}
    cpts = [t.table_view(t.cond, t.names[v]).double().cpu().numpy() for v in range(spec.n)]
    rows = codes[:, :n_check].T.cpu().numpy().astype(np.int64)
    want, _, _ = EO.e_step(spec.cards, spec.parents, cpts, hidden, rows)
    err = max(float(np.max(np.abs(got[t.offsets[v]: t.offsets[v] + t.n_cells[v]] - want[v].reshape(-1))
                             / (np.abs(want[v].reshape(-1)) + n_check * 2.0 ** -32))) for v in fams)
    return {"rows": n_check, "max_rel_err_vs_fp64": err}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    name, power = _card()
    legs = []
    for label, spec, hidden, n in _workloads():
        t = tables_from_spec(spec, DEV)
        codes = sample_network(spec, 7, 0, n, device=DEV, tables=t)
        codes[hidden] = N.UNSEEN
        t.count(codes, n)
        t.hidden = set(hidden)
        infer = bind_inference(t)
        em = EM(t, infer, codes, n, hidden)
        em.initialise("random", 0, None)
        _iteration(em)                                         # warm-up: module loads, allocator, first compiles
        its = [_iteration(em) for _ in range(args.iters)]
        cards = t.cards
        model = {"bytes_per_row": sum(4 * chain_floats(g.hidden, cards)
                                      + len({u for f in g.families for u in t.family_vars(t.names[f]) if u not in hidden})
                                      for g in em.groups),
                 "atomics_per_row_max": sum(len(g.families) * int(np.prod([cards[u] for u in g.hidden])) for g in em.groups),
                 "smem_dests": sum(p.smem_dests for p in em.ess), "dests": sum(len(g.families) for g in em.groups)}
        med = {k: float(np.median([it[k] for it in its])) for k in its[0] if k != "log_likelihood"}
        ess_s = med["ess_us"] * 1e-6
        legs.append({"workload": label, "rows": n, "hidden": len(hidden), "groups": len(em.groups), "chunk_rows": em.chunk,
                     "gathers_per_chunk": sum(g.prefix_configs(cards, j) for g in em.groups for j in range(len(g.hidden))),
                     "iterations": its, "median": med, "ess_model": model,
                     "ess_rows_per_s": n / ess_s, "ess_model_gbs": model["bytes_per_row"] * n / ess_s / 1e9,
                     "check": _check(spec, hidden, t, infer, codes)})
        del em, codes
        torch.cuda.empty_cache()
    res = {"bench": "em", "gpu": name, "power_limit_and_max_sm_clock": power, "legs": legs}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
