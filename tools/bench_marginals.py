"""Junction-tree calibration per row (cbn_jt_run) on one GPU; prints ONE JSON line.

Legs:
  * Alarm, 2^24 rows sampled from the network, cells missing completely at random at 0 %, 5 % and 30 %; the uint8 code
    matrix (37 x 2^24 = 620 MB) is larger than the 126 MB L2.  Per rate: (a) log P(observed cells) only, (b) the expected
    counts only (the E-step), (c) the marginals of the four ALARM_TARGETS with log P.  Kernel time: CUDA events around
    --iters launches after a warm-up launch; rows/s; the plan's modelled multiply-adds per row (clique cells x (1 +
    incoming messages) of every op the leg runs; an upper bound: skipped ops and inconsistent cells are counted) and
    bytes per row (codes read + outputs written), with the achieved rates;
  * one EM iteration with 5 % missing cells on Alarm (2^24 rows), phase by phase: compile_ms (host clock around the
    junction tree's compile after the M-step changed the CPTs, ending in a device synchronise), estep_us (CUDA events
    around the cbn_jt_run launches with log P), mstep_us (CUDA events around the CPT kernel), iteration_ms (host clock);
  * the junction-tree E-step beside the chain E-step of tools/bench_em.py on its workloads with hidden nodes (no missing
    cells): host clock around one E-step each, compile included, and the largest relative difference of their expected
    counts (for the record; which E-step should run there is not decided here);
  * in-run check: 4,096 Alarm rows at 30 % missing against the fp64 interpretation of the plan's tables
    (tests/jt_oracle.py), and 4,096 rows of a random small network against fp64 enumeration.
The card name and power limit are read in the same run.

    python tools/bench_marginals.py [--iters 10] [--out FILE]
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
from continuousbayesiannetwork_b200 import jt, synth  # noqa: E402
from continuousbayesiannetwork_b200.em import EM, JTEM  # noqa: E402
from continuousbayesiannetwork_b200.engine import bind_inference, install_cpts, sample_network, tables_from_spec  # noqa: E402
import em_oracle as EO  # noqa: E402
import jt_oracle as JO  # noqa: E402
import mpe_oracle as MO  # noqa: E402

DEV = "cuda:0"


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        out = f"unavailable ({e})"
    return name, out


def _mask(codes, n, rate, seed):
    if rate <= 0:
        return
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    m = torch.rand(codes.shape[0], n, generator=g, device=DEV) < rate
    codes[:, :n].masked_fill_(m, N.MISSING)


def _time(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def alarm_legs(iters, n):
    spec = synth.alarm()
    t, infer = install_cpts(spec, DEV)
    tree = infer.junction_tree()
    targets = [spec.names.index(x) for x in synth.ALARM_TARGETS]
    plan_all = tree.plan([])
    plan_t = tree.plan(targets)
    sch = plan_t.schedule
    smem = torch.zeros(1, dtype=torch.int64)
    warps = torch.zeros(1, dtype=torch.int32)
    import ctypes as C
    N.lib().cbn_jt_plan_stats(plan_t.handle, C.cast(smem.data_ptr(), C.POINTER(C.c_int64)),
                              C.cast(warps.data_ptr(), C.POINTER(C.c_int32)))
    lp = torch.empty(n, dtype=torch.float32, device=DEV)
    marg = torch.empty((n, sch.marg_floats), dtype=torch.float32, device=DEV)
    acc = torch.zeros(t.total_cells, dtype=torch.int64, device=DEV)
    up = (jt.UP, jt.ROOT)
    model = {"log": plan_all.schedule.madds_per_row(up),
             "acc": plan_all.schedule.madds_per_row(up + (jt.FAMILY,)) + sum(
                 plan_all.schedule.structure.cells(o["clique"]) * (1 + len(o["inputs"])) for o in plan_all.schedule.ops
                 if o["kind"] == jt.DOWN and o["needed"] & jt.NEED_FAMILIES),
             "marg": sch.madds_per_row(up + (jt.NODE,)) + sum(
                 sch.structure.cells(o["clique"]) * (1 + len(o["inputs"])) for o in sch.ops
                 if o["kind"] == jt.DOWN and o["needed"] & jt.NEED_NODES)}
    out_bytes = {"log": 4, "acc": 0, "marg": 4 + 4 * sch.marg_floats}
    legs = []
    for rate in (0.0, 0.05, 0.30):
        codes = sample_network(spec, 17, 0, n, device=DEV, tables=t)
        _mask(codes, n, rate, 5)
        runs = {"log": lambda: plan_all.run(codes, n, log_out=lp),
                "acc": lambda: plan_all.run(codes, n, acc=acc),
                "marg": lambda: plan_t.run(codes, n, marg_out=marg, log_out=lp)}
        for kind, fn in runs.items():
            us = _time(fn, iters)
            bpr = spec.n + out_bytes[kind]
            legs.append({"leg": f"alarm_{kind}", "missing_rate": rate, "rows": n, "kernel_us": round(us, 1),
                         "rows_per_s": n / (us * 1e-6), "madds_per_row_model": model[kind], "bytes_per_row_model": bpr,
                         "gmadds_per_s": model[kind] * n / (us * 1e-6) / 1e9, "gbytes_per_s": bpr * n / (us * 1e-6) / 1e9,
                         "hbm_share": bpr * n / (us * 1e-6) / 7.7e12})
        del codes
    return legs, {"cliques": len(sch.structure.cliques), "msg_floats_per_row": plan_all.schedule.msg_floats,
                  "smem_bytes_per_cta": int(smem.item()), "warps_per_cta": int(warps.item())}


def em_iteration(n, iters=2):
    spec = synth.alarm()
    t, infer = install_cpts(spec, DEV)
    codes = sample_network(spec, 23, 0, n, device=DEV, tables=t)
    _mask(codes, n, 0.05, 9)
    t.count(codes, n)
    em = JTEM(t, infer, codes, n, [])
    em.initialise("random", 0, None)
    em.e_step()
    em.m_step()
    torch.cuda.synchronize()
    out = []
    for _ in range(iters):
        h0 = time.perf_counter()
        em.plan()
        torch.cuda.synchronize()
        compile_ms = (time.perf_counter() - h0) * 1e3
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        em.e_step()
        e1.record()
        em.m_step()
        e2.record()
        e2.synchronize()
        out.append({"compile_ms": round(compile_ms, 2), "estep_us": round(e0.elapsed_time(e1) * 1e3, 1),
                    "mstep_us": round(e1.elapsed_time(e2) * 1e3, 1),
                    "iteration_ms": round((time.perf_counter() - h0) * 1e3, 2)})
    return {"leg": "em_iteration_alarm_5pct", "rows": n, "iterations": out}


def chain_vs_jt():
    names, cards, parents, cpts = EO.latent_class(n_children=20, k=4, card=3, seed=0)
    lc = synth.NetSpec(names, cards, parents, cpts)
    alarm = synth.alarm()
    ev = {alarm.names.index(x) for x in synth.ALARM_EVIDENCE}
    work = [("latent_class_z4_x20", lc, [0], 1 << 24),
            ("alarm_targets_hidden", alarm, [alarm.names.index(x) for x in synth.ALARM_TARGETS], 1 << 24),
            ("alarm_all_but_evidence_hidden", alarm, [v for v in range(alarm.n) if v not in ev], 1 << 22)]
    out = []
    for name, spec, hidden, n in work:
        t = tables_from_spec(spec, DEV)
        t.set_cond_tables(spec.cpts)
        infer = bind_inference(t)
        codes = sample_network(spec, 3, 0, n, device=DEV, tables=t)
        codes[hidden] = N.UNSEEN
        t.count(codes, n)
        t.hidden = set(hidden)
        res = {"workload": name, "rows": n}
        accs = {}
        for label, cls, fill in (("chain", EM, N.UNSEEN), ("jt", JTEM, N.MISSING)):
            codes[hidden] = fill
            em = cls(t, infer, codes, n, hidden)
            em.e_step()                                   # warm: plans compiled
            infer.bind(t)                                 # drop the plans: the timed E-step compiles, as after an M-step
            torch.cuda.synchronize()
            h0 = time.perf_counter()
            em.e_step()
            torch.cuda.synchronize()
            res[f"{label}_estep_ms"] = round((time.perf_counter() - h0) * 1e3, 2)
            accs[label] = em.acc.double()
        a, b = accs["chain"], accs["jt"]
        res["max_rel_diff_expected_counts"] = float(((a - b).abs() / a.abs().clamp(min=float(1 << 32))).max().item())
        out.append(res)
        del codes
    return out


def in_run_check():
    spec = synth.alarm()
    t, infer = install_cpts(spec, DEV)
    n = 4096
    codes = sample_network(spec, 31, 0, n, device=DEV, tables=t)
    _mask(codes, n, 0.30, 2)
    plan = infer.junction_tree().plan(None)
    marg = torch.empty((n, plan.schedule.marg_floats), dtype=torch.float32, device=DEV)
    lp = torch.empty(n, dtype=torch.float32, device=DEV)
    plan.run(codes, n, marg_out=marg, log_out=lp)
    rows = codes[:, :n].T.cpu().numpy().astype(np.int64)
    cpts = [np.asarray(c, np.float32).astype(np.float64) for c in spec.cpts]
    want_lp, want_run, _ = JO.interpret(plan.schedule, cpts, rows)
    rng = np.random.default_rng(8)
    cards, parents, small = MO.random_small_net(rng, 8, 9)
    sspec = synth.NetSpec([f"v{i}" for i in range(len(cards))], cards, parents,
                          [np.asarray(c, np.float32).astype(np.float64) for c in small])
    st, sinfer = install_cpts(sspec, DEV)
    sc = sample_network(sspec, 4, 0, n, device=DEV, tables=st)
    _mask(sc, n, 0.4, 3)
    splan = sinfer.junction_tree().plan(None)
    sm = torch.empty((n, splan.schedule.marg_floats), dtype=torch.float32, device=DEV)
    slp = torch.empty(n, dtype=torch.float32, device=DEV)
    splan.run(sc, n, marg_out=sm, log_out=slp)
    srows = sc[:, :n].T.cpu().numpy().astype(np.int64)
    e_lp, e_m, _ = JO.enumerate_rows(sspec.cards, sspec.parents, sspec.cpts, srows)
    live = np.isfinite(e_lp)
    e_run = np.concatenate([e_m[v] for v in range(len(cards))], 1)
    return {"alarm_rows": n, "alarm_max_abs_marginal_err": float(np.abs(marg.cpu().numpy() - want_run).max()),
            "alarm_max_abs_log_p_err": float(np.abs(lp.cpu().numpy() - want_lp).max()),
            "small_net_rows": n, "small_net_live_rows": int(live.sum()),
            "small_net_max_abs_marginal_err": float(np.abs(sm.cpu().numpy()[live] - e_run[live]).max()),
            "small_net_max_abs_log_p_err": float(np.abs(slp.cpu().numpy()[live] - e_lp[live]).max()),
            "small_net_dead_rows_agree": bool(np.array_equal(np.isneginf(slp.cpu().numpy()), ~live))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rows-log2", type=int, default=24)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = _card()
    n = 1 << a.rows_log2
    legs, plan = alarm_legs(a.iters, n)
    res = {"bench": "jt_marginals", "gpu": name, "power_limit_and_max_sm_clock": power, "alarm_plan": plan, "legs": legs,
           "em": em_iteration(n), "chain_vs_jt": chain_vs_jt(), "check": in_run_check()}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
