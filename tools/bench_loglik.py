"""Throughput of the log-likelihood / log P(e) kernels on one GPU; prints ONE JSON line.

Three legs, every input resident in HBM and larger than the 126 MB L2:
  * complete-data log-likelihood on Alarm, 2^26 sampled rows (observed-families kernel only, cbn_loglik_run);
  * complete-data log-likelihood on the 200-node k-tree DAG, 2^24 rows (union tables beyond one CTA's shared memory);
  * log P(e) for the headline evidence set synth.ALARM_EVIDENCE on 2^24 rows (the evidence-mode VE gather plus the
    observed-families kernel accumulating into its output).
Each leg is warmed up, then timed with CUDA events over a window of at least 60 ms.  Reported per leg: rows/s, us per
launch, algorithmic bytes per row (codes in + one float out) and the fraction of the HBM peak those bytes imply (peak
from MEASURED_PEAKS.json when present, as bench.py does).  Every leg checks a bounded sample of its rows against an fp64
oracle in the same run; the card name and power limit are read in the same run.

    python tools/bench_loglik.py [--out FILE]
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

from continuousbayesiannetwork_b200 import synth  # noqa: E402
from continuousbayesiannetwork_b200.engine import install_cpts, sample_network  # noqa: E402
from oracle import cbn_oracle as O  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tests"))
import loglik_oracle as LO  # noqa: E402

DEV = "cuda:0"
SAMPLE = 4096          # rows per leg checked against the fp64 oracle


def _peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:            # the number is still reported, without its power limit
        out = f"unavailable ({e})"
    return name, out


def _time(fn, min_ms=60.0):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); e1.synchronize()
    one = max(e0.elapsed_time(e1), 1e-3)
    iters = max(10, int(np.ceil(1.5 * min_ms / one)))
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    assert ms >= min_ms, ms
    return ms / iters, iters, ms


def _f32(spec):
    return synth.NetSpec(spec.names, spec.cards, spec.parents, [c.astype(np.float32).astype(np.float64) for c in spec.cpts])


def _complete_ref(spec, codes):
    ref = np.zeros(codes.shape[1])
    for v in range(spec.n):
        ref += np.log(spec.cpts[v][tuple(codes[p] for p in spec.parents[v]) + (codes[v],)])
    return ref


def _check(got, ref):
    got = np.asarray(got, np.float64)
    dead = np.isneginf(ref)
    ok = not np.isnan(got).any() and np.array_equal(np.isneginf(got), dead)
    err = np.abs(got[~dead] - ref[~dead]) / np.maximum(1.0, np.abs(ref[~dead]))
    worst = float(err.max()) if err.size else 0.0
    return bool(ok and worst <= 1e-5), worst


def _leg(name, spec, names, n, seed, peak):
    tables, infer = install_cpts(spec, DEV)
    codes = sample_network(spec, seed, 0, n, DEV, tables=tables)
    ids = [spec.names.index(x) for x in names]
    ev = codes if ids == list(range(spec.n)) else codes[ids].contiguous()
    plan = infer.evidence_plan(names)
    out = torch.empty(n, dtype=torch.float32, device=DEV)
    ms, iters, window = _time(lambda: plan.run_codes(ev, n, out))
    # oracle: a seeded sample of the rows of the last timed launch
    rows = np.sort(np.random.default_rng(seed).choice(n, size=SAMPLE, replace=False))
    got = out[torch.from_numpy(rows).to(DEV)].cpu().numpy()
    sample = ev[:, torch.from_numpy(rows).to(DEV)].cpu().numpy().astype(np.int64)
    if plan.ve_plan is None:
        full = np.zeros((spec.n, SAMPLE), np.int64)
        full[ids] = sample
        ref = _complete_ref(spec, full)
    else:
        ref = LO.ve_log_evidence(O.DiscreteNet(spec.cards, spec.parents, spec.cpts), ids, sample.T)
    ok, worst = _check(got, ref)
    bpr = len(ids) + 4
    return {"leg": name, "rows": n, "launch_us": round(ms * 1e3, 2), "rows_per_s": n / (ms * 1e-3),
            "bytes_per_row": bpr, "hbm_fraction": round(bpr * n / (ms * 1e-3) / (peak * 1e9), 4),
            "table_lookups_per_row": plan.loglik.lookups_per_row if plan.loglik is not None else 0,
            "ve_tables": [c for _, c in plan.ve_plan.stats.final_tables] if plan.ve_plan is not None else [],
            "timed_launches": iters, "window_ms": round(window, 1),
            "oracle": {"rows": SAMPLE, "ok": ok, "worst_rel_err": worst}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    name, power = _card()
    peak, peak_src = _peak()
    legs = []
    alarm = _f32(synth.alarm())
    legs.append(_leg("alarm_complete", alarm, alarm.names, 1 << 26, 61, peak))
    torch.cuda.empty_cache()
    kt = _f32(synth.random_ktree_dag())
    legs.append(_leg("ktree200_complete", kt, kt.names, 1 << 24, 62, peak))
    torch.cuda.empty_cache()
    legs.append(_leg("alarm_log_evidence", alarm, synth.ALARM_EVIDENCE, 1 << 24, 63, peak))
    res = {"bench": "loglik", "gpu": name, "power_limit_and_max_sm_clock": power, "hbm_peak_gbs": peak,
           "hbm_peak_source": peak_src, "timing": "CUDA events, warm-up first, >= 60 ms window, resident inputs > L2",
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
