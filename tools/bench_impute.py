"""Junction-tree decoding per row (cbn_jt_decode) on one GPU; prints ONE JSON line.

Legs:
  * Alarm, 2^24 rows sampled from the network, cells missing completely at random at 0 %, 5 % and 30 % (the uint8 code
    matrix, 37 x 2^24 = 620 MB, and the completions written back are each larger than the 126 MB L2).  Per rate: (a) the
    most probable completion (MAX), (b) one posterior draw (SAMPLE), and the collect pass alone (cbn_jt_run with log P on
    the same collect-only plan), so the decode's own cost is the difference;
  * 2^22 rows x 8 draws at 30 % missing;
  * for the record, the fixed-set MPE path (most_probable_explanation's plan for the headline evidence set) on the same
    2^24 rows with no missing cell.
Kernel time: CUDA events around --iters launches after a warm-up launch; rows/s; the plan's modelled multiply-adds per
row (clique cells x (1 + incoming messages) of every collect op, counted once more per draw for the decode: an upper
bound, skipped cliques and inconsistent cells are counted) and bytes per row (codes read, completions and log written).
In-run check: 4,096 Alarm rows at 30 % missing against the fp64 interpretation of the plan (tests/impute_oracle.py):
the MAX value, and the draws of every (row, draw) whose u * total is not within 1e-5 of a cumulative boundary.
The card name and power limit are read in the same run.

    python tools/bench_impute.py [--iters 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from continuousbayesiannetwork_b200 import _native as N  # noqa: E402
from continuousbayesiannetwork_b200 import jt, synth  # noqa: E402
from continuousbayesiannetwork_b200.engine import install_cpts, sample_network  # noqa: E402
import impute_oracle as IO  # noqa: E402

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


def _leg(name, rate, n, us, madds, bpr, draws=1):
    return {"leg": name, "missing_rate": rate, "rows": n, "draws": draws, "kernel_us": round(us, 1),
            "rows_per_s": n / (us * 1e-6), "madds_per_row_model": madds, "bytes_per_row_model": bpr,
            "gmadds_per_s": madds * n / (us * 1e-6) / 1e9, "gbytes_per_s": bpr * n / (us * 1e-6) / 1e9}


def alarm_legs(iters, n, n_multi, draws_multi):
    spec = synth.alarm()
    t, infer = install_cpts(spec, DEV)
    plan = infer.junction_tree().collect_plan()
    sch = plan.schedule
    nv = spec.n
    import ctypes as C
    smem, warps = C.c_int64(), C.c_int32()
    N.lib().cbn_jt_plan_stats(plan.handle, C.byref(smem), C.byref(warps))
    collect = sch.madds_per_row((jt.UP, jt.ROOT))
    lp = torch.empty(n, dtype=torch.float32, device=DEV)
    out = t.new_code_matrix(n, nv)
    legs = []
    for rate in (0.0, 0.05, 0.30):
        codes = sample_network(spec, 17, 0, n, device=DEV, tables=t)
        _mask(codes, n, rate, 5)
        runs = {"collect_only": (lambda: plan.run(codes, n, log_out=lp), collect, nv + 4),
                "mpe": (lambda: plan.decode(codes, n, N.JT_DECODE_MAX, 1, 0, 0, out, lp), 2 * collect, 2 * nv + 4),
                "sample_1": (lambda: plan.decode(codes, n, N.JT_DECODE_SAMPLE, 1, 3, 0, out, lp), 2 * collect, 2 * nv + 4)}
        for kind, (fn, madds, bpr) in runs.items():
            legs.append(_leg(f"alarm_{kind}", rate, n, _time(fn, iters), madds, bpr))
        if rate == 0.0:                                     # the fixed-set MPE path on the same rows, for the record
            ev = [spec.names.index(x) for x in synth.ALARM_EVIDENCE]
            evc = t.new_code_matrix(n, len(ev))
            evc[:, :n] = codes[ev, :n]
            mplan = infer.mpe_plan(list(synth.ALARM_EVIDENCE))
            legs.append(_leg("alarm_fixed_set_mpe_headline_evidence", rate, n,
                             _time(lambda: mplan.run_codes(evc, n), iters), 0, len(ev) + (nv - len(ev)) + 4))
            del evc
        del codes
    del out
    codes = sample_network(spec, 19, 0, n_multi, device=DEV, tables=t)
    _mask(codes, n_multi, 0.30, 6)
    outm = t.new_code_matrix(n_multi, draws_multi * nv)
    lpm = torch.empty(n_multi, dtype=torch.float32, device=DEV)
    us = _time(lambda: plan.decode(codes, n_multi, N.JT_DECODE_SAMPLE, draws_multi, 3, 0, outm, lpm), iters)
    legs.append(_leg(f"alarm_sample_{draws_multi}", 0.30, n_multi, us, (1 + draws_multi) * collect,
                     nv + draws_multi * nv + 4, draws_multi))
    return legs, {"cliques": len(sch.structure.cliques), "collect_ops": len(sch.ops), "msg_floats_per_row": sch.msg_floats,
                  "smem_bytes_per_cta": int(smem.value), "warps_per_cta": int(warps.value)}


def in_run_check():
    spec = synth.alarm()
    t, infer = install_cpts(spec, DEV)
    n, draws = 4096, 4
    codes = sample_network(spec, 31, 0, n, device=DEV, tables=t)
    _mask(codes, n, 0.30, 2)
    plan = infer.junction_tree().collect_plan()
    rows = codes[:, :n].T.cpu().numpy().astype(np.int64)
    cpts = [np.asarray(c, np.float32).astype(np.float64) for c in spec.cpts]
    out = t.new_code_matrix(n, draws * spec.n)
    lp = torch.empty(n, dtype=torch.float32, device=DEV)
    plan.decode(codes, n, N.JT_DECODE_MAX, 1, 0, 0, out, lp)
    want = IO.interpret_decode(plan.schedule, cpts, rows, 0)
    comp = out[: spec.n, :n].cpu().numpy().astype(np.int64).T
    res = {"rows": n, "mpe_max_rel_log_err": float(np.abs(lp.cpu().numpy() - want["log"]).max() / np.abs(want["log"]).min()),
           "mpe_max_abs_loglik_minus_log_prob": float(np.abs(IO.log_joint(spec.cards, spec.parents, cpts, comp) -
                                                             lp.cpu().numpy()).max())}
    plan.decode(codes, n, N.JT_DECODE_SAMPLE, draws, 9, 0, out, lp)
    want = IO.interpret_decode(plan.schedule, cpts, rows, 1, seed=9, first_row=0, n_draws=draws)
    got = out[: draws * spec.n, :n].cpu().numpy().astype(np.int64).reshape(draws, spec.n, n).transpose(0, 2, 1)
    keep = want["margin"] > 1e-5
    res.update({"draws": draws, "sample_pairs_checked": int(keep.sum()), "sample_pairs_near_a_boundary": int((~keep).sum()),
                "sample_pairs_equal": int(sum((got[d][keep[d]] == want["codes"][d][keep[d]]).all(1).sum()
                                              for d in range(draws))),
                "sample_max_abs_log_evidence_err": float(np.abs(lp.cpu().numpy() - want["log"]).max())})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rows-log2", type=int, default=24)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = _card()
    n = 1 << a.rows_log2
    legs, plan = alarm_legs(a.iters, n, n >> 2, 8)
    res = {"bench": "jt_decode", "gpu": name, "power_limit_and_max_sm_clock": power, "alarm_plan": plan, "legs": legs,
           "check": in_run_check()}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
