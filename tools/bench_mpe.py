"""Throughput of the most probable explanation on one GPU; prints ONE JSON line.

Legs:
  * Alarm, headline evidence synth.ALARM_EVIDENCE, 2^24 sampled rows resident in HBM (evidence 201 MB + value 67 MB +
    hidden codes 419 MB, larger than the 126 MB L2): the whole MPE (MPEPlan.run_codes), and each of its launches alone --
    the log-evidence gather (cbn_ve_run_codes_log_evidence), the observed-families kernel accumulating into its output
    (cbn_loglik_run; no CPT of Alarm lies inside the headline set, so that launch does not occur there) and the traceback
    (cbn_mpe_run);
  * Alarm without evidence, the traceback alone on 2^24 rows: 37 dependent lookups per row, every argmax table staged in
    shared memory and no L2 gather -- set against the headline traceback, it separates the cost of the random L2 byte
    gather from the cost of the chain of lookups;
  * the 200-node k-tree, bench.py's query pattern with the smallest argmax tables (rng(1240), 10 evidence variables),
    2^20 rows: the whole MPE, the traceback alone, and the compile (host time and contraction_gpu_ms).
Each timing is warmed up, then taken with CUDA events over a window of at least 60 ms.  Reported: rows/s, us per launch,
algorithmic bytes per row (evidence codes in + 4 B value + hidden codes out) and the fraction of the HBM peak those bytes
imply (peak from MEASURED_PEAKS.json when present, as bench.py does).  Every leg checks a bounded sample of rows in the
same run: Alarm against the fp64 max-product oracle, the k-tree by the log-likelihood identity on every row and single-flip
local optimality on a sample.  The card name and power limit are read in the same run.

    python tools/bench_mpe.py [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from continuousbayesiannetwork_b200 import _native as N  # noqa: E402
from continuousbayesiannetwork_b200 import synth  # noqa: E402
from continuousbayesiannetwork_b200.engine import install_cpts, sample_network  # noqa: E402
from oracle import cbn_oracle as O  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mpe_oracle as MO  # noqa: E402
from bench_loglik import _card, _f32, _peak, _time  # noqa: E402

DEV = "cuda:0"
SAMPLE = 4096          # Alarm rows checked against the fp64 oracle
TOL = 1e-5


def _rate(name, n, ms, bpr, peak, iters, window, **extra):
    return dict({"leg": name, "rows": n, "launch_us": round(ms * 1e3, 2), "rows_per_s": n / (ms * 1e-3),
                 "bytes_per_row": bpr, "hbm_fraction": round(bpr * n / (ms * 1e-3) / (peak * 1e9), 4),
                 "timed_launches": iters, "window_ms": round(window, 1)}, **extra)


def _traceback(plan, ev, n, value, hidden):
    N.check(N.lib().cbn_mpe_run(plan.ctx.handle, plan.handle, ev.data_ptr(), ev.stride(0), n, value.data_ptr(),
                                hidden.data_ptr(), hidden.stride(0), N.stream_ptr(DEV)), plan.ctx.handle)


def _loglik_of(infer, comp, n, order):
    return infer.evidence_plan([infer.tables.names[v] for v in order]).run_codes(comp, n).double()


def alarm_legs(peak):
    spec = _f32(synth.alarm())
    tables, infer = install_cpts(spec, DEV)
    n = 1 << 24
    codes = sample_network(spec, 71, 0, n, DEV, tables=tables)
    E = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    ev = codes[E].contiguous()
    del codes
    plan = infer.mpe_plan(synth.ALARM_EVIDENCE)
    value = torch.empty(n, dtype=torch.float32, device=DEV)
    hidden = torch.empty((len(plan.hidden), ev.stride(0)), dtype=torch.uint8, device=DEV)
    bpr = len(E) + 4 + len(plan.hidden)
    legs = []
    ms, it, win = _time(lambda: plan.run_codes(ev, n, hidden, value))
    legs.append(_rate("alarm_mpe", n, ms, bpr, peak, it, win, launches=2 + (plan.value.loglik is not None)))
    vp = plan.value
    gather = lambda: N.check(N.lib().cbn_ve_run_codes_log_evidence(  # noqa: E731
        vp.ctx.handle, vp.ve_plan.handle, ev.data_ptr(), ev.stride(0), n, value.data_ptr(), N.stream_ptr(DEV)), vp.ctx.handle)
    ms, it, win = _time(gather)
    legs.append(_rate("alarm_gather_log_evidence", n, ms, len(E) + 4, peak, it, win))
    if vp.loglik is not None:          # no CPT of Alarm lies inside the headline set: there is no such launch
        obs_cols = sorted({E.index(u) for v in vp.observed_families for u in spec.parents[v] + [v]})
        ms, it, win = _time(lambda: vp.loglik.run(ev, n, value, accumulate=True))
        legs.append(_rate("alarm_loglik_accumulate", n, ms, len(obs_cols) + 8, peak, it, win,
                          table_lookups_per_row=vp.loglik.lookups_per_row))
    plan.run_codes(ev, n, hidden, value)                  # the value the traceback reads
    ms, it, win = _time(lambda: _traceback(plan, ev, n, value, hidden))
    ev_read = sorted({u for _, sc in plan.split.decode for u in sc if u in set(E)})
    legs.append(_rate("alarm_traceback", n, ms, len(ev_read) + 4 + len(plan.hidden), peak, it, win,
                      dependent_lookups_per_row=len(plan.hidden), evidence_columns_read=len(ev_read),
                      argmax_bytes=plan.split.argmax_bytes,
                      largest_argmax_table=max(int(a.numel()) for a in plan.tables)))
    # oracle: a seeded sample of rows of the last launches
    rows = np.sort(np.random.default_rng(71).choice(n, size=SAMPLE, replace=False))
    r = torch.from_numpy(rows).to(DEV)
    evs = ev[:, r].cpu().numpy().T.astype(np.int64)
    net = O.DiscreteNet(spec.cards, spec.parents, spec.cpts)
    best, _ = MO.ve_mpe(net, E, evs)
    got = value[r].cpu().numpy().astype(np.float64)
    full = np.zeros((SAMPLE, spec.n), np.int64)
    full[:, E] = evs
    full[:, plan.hidden] = hidden[:, r].cpu().numpy().T
    lj = MO.log_joint(net, full)
    fin = np.isfinite(best)
    err_v = float(np.max(np.abs(got[fin] - best[fin]) / np.maximum(1, np.abs(best[fin])))) if fin.any() else 0.0
    err_a = float(np.max(np.abs(lj[fin] - best[fin]) / np.maximum(1, np.abs(best[fin])))) if fin.any() else 0.0
    ok = bool(np.array_equal(np.isneginf(got), ~fin) and not np.isnan(got).any() and err_v <= TOL and err_a <= TOL)
    for leg in legs:
        leg["oracle"] = {"rows": SAMPLE, "ok": ok, "worst_rel_err_value": err_v, "worst_rel_err_assignment": err_a}
    del ev, hidden
    torch.cuda.empty_cache()
    # no evidence: the traceback alone with every table staged in shared memory
    prior = infer.mpe_plan([])
    zero = torch.zeros(n, dtype=torch.float32, device=DEV)
    hid = torch.empty((len(prior.hidden), (n + 15) // 16 * 16), dtype=torch.uint8, device=DEV)
    dummy = torch.zeros((1, 16), dtype=torch.uint8, device=DEV)
    ms, it, win = _time(lambda: _traceback(prior, dummy, n, zero, hid))
    h1, v1 = prior.run_codes(dummy, 1)
    same = bool((hid[:, :4096] == h1[:, :1]).all())           # every row decodes the prior's explanation
    legs.append(_rate("alarm_prior_traceback", n, ms, 4 + len(prior.hidden), peak, it, win,
                      dependent_lookups_per_row=len(prior.hidden), argmax_bytes=prior.split.argmax_bytes,
                      oracle={"rows": 4096, "ok": same, "check": "every row equals the one-row explanation of the prior"}))
    return legs


def ktree_legs(peak):
    spec = _f32(synth.random_ktree_dag())
    tables, infer = install_cpts(spec, DEV, profile_compile=True)
    from continuousbayesiannetwork_b200.ve import DryTables, VECompiler

    rng = np.random.default_rng(1240)
    pats = [[int(v) for v in rng.choice(spec.n, size=11, replace=False)] for _ in range(8)]
    dry = VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()))
    sizes = [dry.compile_mpe([spec.names[v] for v in vs[1:]], dry=True).argmax_bytes for vs in pats]
    pi = int(np.argmin(sizes))
    ids = pats[pi][1:]
    names = [spec.names[v] for v in ids]
    n = 1 << 20
    codes = sample_network(spec, 72, 0, n, DEV, tables=tables)
    ev = codes[ids].contiguous()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    plan = infer.mpe_plan(names)
    torch.cuda.synchronize()
    compile_ms = (time.perf_counter() - t0) * 1e3
    value = torch.empty(n, dtype=torch.float32, device=DEV)
    hidden = torch.empty((len(plan.hidden), ev.stride(0)), dtype=torch.uint8, device=DEV)
    bpr = len(ids) + 4 + len(plan.hidden)
    ms, it, win = _time(lambda: plan.run_codes(ev, n, hidden, value))
    legs = [_rate("ktree200_mpe", n, ms, bpr, peak, it, win, pattern=pi, launches=3 if plan.value.loglik else 2,
                  compile_host_ms=round(compile_ms, 1), contraction_gpu_ms=round(plan.split.stats.contraction_gpu_ms, 2),
                  argmax_bytes=plan.split.argmax_bytes, max_table_cells=plan.split.stats.max_table_cells,
                  note="inputs of this leg (10 MB of evidence) fit the L2")]
    plan.run_codes(ev, n, hidden, value)
    ms, it, win = _time(lambda: _traceback(plan, ev, n, value, hidden))
    legs.append(_rate("ktree200_traceback", n, ms, bpr, peak, it, win, dependent_lookups_per_row=len(plan.hidden)))
    # identity on every row; single-flip local optimality on a sample, scored on the device
    order = plan.evidence + plan.hidden
    comp = torch.cat([ev[:, :hidden.shape[1]], hidden]).contiguous()
    lj = _loglik_of(infer, comp, n, order)
    v = value.double()
    err = float(((lj - v).abs() / v.abs().clamp(min=1)).max())
    m = 32
    rows = torch.from_numpy(np.sort(np.random.default_rng(72).choice(n, size=m, replace=False))).to(DEV)
    base = comp[:, rows]
    flips = []
    for j in range(len(plan.evidence), len(order)):
        for dc in range(1, spec.cards[order[j]]):
            f = base.clone()
            f[j] = (f[j].int() + dc) % spec.cards[order[j]]
            flips.append(f)
    allf = torch.cat(flips, dim=1)
    k = allf.shape[1]
    mat = torch.zeros((len(order), (k + 15) // 16 * 16), dtype=torch.uint8, device=DEV)
    mat[:, :k] = allf
    scores = _loglik_of(infer, mat, k, order).reshape(-1, m)
    b = v[rows]
    gain = float(((scores - b) / b.abs().clamp(min=1)).max())
    ok = bool(torch.isfinite(v).all() and err <= TOL and gain <= TOL)
    for leg in legs:
        leg["oracle"] = {"rows": n, "ok": ok, "worst_rel_err_identity": err, "flip_rows": m, "flips": k,
                         "best_rel_flip_gain": gain}
    return legs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    name, power = _card()
    peak, peak_src = _peak()
    legs = alarm_legs(peak)
    torch.cuda.empty_cache()
    legs += ktree_legs(peak)
    res = {"bench": "mpe", "gpu": name, "power_limit_and_max_sm_clock": power, "hbm_peak_gbs": peak,
           "hbm_peak_source": peak_src, "timing": "CUDA events, warm-up first, >= 60 ms window, Alarm inputs resident > L2",
           "oracle_ok": all(l["oracle"]["ok"] for l in legs), "legs": legs}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if res["oracle_ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
