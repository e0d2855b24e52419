"""Throughput of exact posterior sampling on one GPU; prints ONE JSON line.

Legs:
  * Alarm, headline evidence synth.ALARM_EVIDENCE, 2^24 sampled rows x 1 draw resident in HBM (evidence 201 MB + value
    67 MB + hidden codes 419 MB, larger than the 126 MB L2): the whole query (PosteriorSamplePlan.run_codes: log P(e) gather,
    then the sampler) and the sampler alone (cbn_psample_run);
  * the same evidence, 2^22 rows x 8 draws: the whole query and the sampler alone -- the evidence is loaded once per row
    and the 25 hidden variables are drawn 8 times;
  * Alarm without evidence, the sampler alone on 2^24 rows x 1 draw: every threshold table staged in shared memory;
  * the 200-node k-tree, bench.py's query pattern with the smallest threshold tables (rng(1240), 10 evidence variables),
    2^20 rows x 1 draw: the whole query, the sampler alone, and the compile (host time and contraction_gpu_ms).
Each timing is warmed up, then taken with CUDA events over a window of at least 60 ms.  Reported: row-draws/s, us per
launch, algorithmic bytes (evidence codes the tables read + 4 B value per row, one byte per hidden variable and draw) and
the fraction of the HBM peak those bytes imply (peak from MEASURED_PEAKS.json when present, as bench.py does).  Every leg
checks a block of rows of its own last launch in the same run: the draws bit for bit against the numpy interpreter of
the plan's threshold tables (tests/psample_oracle.py) and, on Alarm, log P(e) against the fp64 oracle.  The card name and
power limit are read in the same run.

    python tools/bench_posterior_sample.py [--out FILE]
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
import loglik_oracle as LO  # noqa: E402
import psample_oracle as PO  # noqa: E402
from bench_loglik import _card, _f32, _peak, _time  # noqa: E402

DEV = "cuda:0"
BLOCK = 4096           # rows checked per leg
TOL = 1e-5
SEED = 2026


def _rate(name, n, draws, ms, nbytes, peak, iters, window, **extra):
    return dict({"leg": name, "rows": n, "draws": draws, "launch_us": round(ms * 1e3, 2),
                 "row_draws_per_s": n * draws / (ms * 1e-3), "algorithmic_bytes": nbytes,
                 "hbm_fraction": round(nbytes / (ms * 1e-3) / (peak * 1e9), 4), "timed_launches": iters,
                 "window_ms": round(window, 1)}, **extra)


def _sampler(plan, ev, n, value, hidden, draws):
    N.check(N.lib().cbn_psample_run(plan.ctx.handle, plan.handle, ev.data_ptr(), ev.stride(0), n, value.data_ptr(), SEED, 0,
                                    draws, hidden.data_ptr(), hidden.stride(0), N.stream_ptr(DEV)), plan.ctx.handle)


def _bytes(plan, n, draws):
    ev_read = {u for _, sc in plan.split.decode for u in sc if u in set(plan.evidence)}
    return n * (len(ev_read) + 4) + n * draws * len(plan.hidden)


def _check_block(spec, plan, ev, value, hidden, n, draws, with_oracle):
    """Bit-exact draws of a block of rows against the numpy interpreter; log P(e) against the fp64 oracle on Alarm."""
    off = int(np.random.default_rng(n + draws).integers(0, n - BLOCK))
    evb = ev[:, off: off + BLOCK].cpu().numpy().T.astype(np.int64) if plan.evidence else np.zeros((BLOCK, 0), np.int64)
    val = value[off: off + BLOCK].cpu().numpy()
    decode = [(v, tuple(sc), tb.cpu().numpy()) for (v, sc), tb in zip(plan.split.decode, plan.tables)]
    want = PO.interpret(decode, spec.cards, plan.evidence, evb, ~(val > -np.inf), SEED, off, draws)
    nh = len(plan.hidden)
    got = hidden[: draws * nh, off: off + BLOCK].cpu().numpy().reshape(draws, nh, BLOCK)
    bits = all(np.array_equal(got[:, h], want[v]) for h, v in enumerate(plan.hidden))
    res = {"rows": BLOCK, "first_row": off, "draws_bit_exact": bits}
    ok = bits and not np.isnan(val).any()
    if with_oracle:
        ref = LO.ve_log_evidence(O.DiscreteNet(spec.cards, spec.parents, spec.cpts), plan.evidence, evb)
        fin = np.isfinite(ref)
        err = float(np.max(np.abs(val[fin] - ref[fin]) / np.maximum(1, np.abs(ref[fin])))) if fin.any() else 0.0
        ok = ok and bool(np.array_equal(np.isneginf(val), ~fin)) and err <= TOL
        res["worst_rel_err_log_evidence"] = err
    res["ok"] = bool(ok)
    return res


def alarm_legs(peak):
    spec = _f32(synth.alarm())
    tables, infer = install_cpts(spec, DEV)
    E = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    plan = infer.posterior_sampler(synth.ALARM_EVIDENCE)
    legs = []
    for n, draws in ((1 << 24, 1), (1 << 22, 8)):
        ev = sample_network(spec, 81, 0, n, DEV, tables=tables)[E].contiguous()
        value = torch.empty(n, dtype=torch.float32, device=DEV)
        hidden = torch.empty((draws * len(plan.hidden), ev.stride(0)), dtype=torch.uint8, device=DEV)
        tag = f"alarm_{n >> 20}M_x{draws}"
        ms, it, win = _time(lambda: plan.run_codes(ev, n, draws, SEED, 0, hidden, value))
        legs.append(_rate(tag + "_whole", n, draws, ms, _bytes(plan, n, draws), peak, it, win, launches=2))
        ms, it, win = _time(lambda: _sampler(plan, ev, n, value, hidden, draws))
        legs.append(_rate(tag + "_sampler", n, draws, ms, _bytes(plan, n, draws), peak, it, win,
                          dependent_draws_per_row=len(plan.hidden) * draws, threshold_bytes=plan.split.table_bytes))
        chk = _check_block(spec, plan, ev, value, hidden, n, draws, True)
        legs[-1]["oracle"] = legs[-2]["oracle"] = chk
        del ev, hidden, value
        torch.cuda.empty_cache()
    # no evidence: every threshold table staged in shared memory
    prior = infer.posterior_sampler([])
    n = 1 << 24
    value = torch.zeros(n, dtype=torch.float32, device=DEV)
    hidden = torch.empty((len(prior.hidden), n), dtype=torch.uint8, device=DEV)
    dummy = torch.zeros((1, 16), dtype=torch.uint8, device=DEV)
    ms, it, win = _time(lambda: _sampler(prior, dummy, n, value, hidden, 1))
    legs.append(_rate("alarm_prior_sampler", n, 1, ms, _bytes(prior, n, 1), peak, it, win,
                      dependent_draws_per_row=len(prior.hidden), threshold_bytes=prior.split.table_bytes,
                      oracle=_check_block(spec, prior, dummy, value, hidden, n, 1, False)))
    return legs


def ktree_legs(peak):
    spec = _f32(synth.random_ktree_dag())
    tables, infer = install_cpts(spec, DEV, profile_compile=True)
    from continuousbayesiannetwork_b200.ve import DryTables, VECompiler

    rng = np.random.default_rng(1240)
    pats = [[int(v) for v in rng.choice(spec.n, size=11, replace=False)] for _ in range(8)]
    dry = VECompiler(DryTables(spec.names, spec.cards, spec.parents_by_name()), sample_table_budget_bytes=1 << 40)
    sizes = [dry.compile_posterior_sampler([spec.names[v] for v in vs[1:]], dry=True).table_bytes for vs in pats]
    pi = int(np.argmin(sizes))
    ids = pats[pi][1:]
    names = [spec.names[v] for v in ids]
    n = 1 << 20
    ev = sample_network(spec, 82, 0, n, DEV, tables=tables)[ids].contiguous()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    plan = infer.posterior_sampler(names)
    torch.cuda.synchronize()
    compile_ms = (time.perf_counter() - t0) * 1e3
    value = torch.empty(n, dtype=torch.float32, device=DEV)
    hidden = torch.empty((len(plan.hidden), ev.stride(0)), dtype=torch.uint8, device=DEV)
    ms, it, win = _time(lambda: plan.run_codes(ev, n, 1, SEED, 0, hidden, value))
    legs = [_rate("ktree200_whole", n, 1, ms, _bytes(plan, n, 1), peak, it, win, pattern=pi,
                  launches=3 if plan.value.loglik else 2, compile_host_ms=round(compile_ms, 1),
                  contraction_gpu_ms=round(plan.split.stats.contraction_gpu_ms, 2), threshold_bytes=plan.split.table_bytes,
                  max_table_cells=plan.split.stats.max_table_cells, note="inputs of this leg (10 MB of evidence) fit the L2")]
    ms, it, win = _time(lambda: _sampler(plan, ev, n, value, hidden, 1))
    legs.append(_rate("ktree200_sampler", n, 1, ms, _bytes(plan, n, 1), peak, it, win,
                      dependent_draws_per_row=len(plan.hidden)))
    legs[0]["oracle"] = legs[1]["oracle"] = _check_block(spec, plan, ev, value, hidden, n, 1, False)
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
    res = {"bench": "posterior_sample", "gpu": name, "power_limit_and_max_sm_clock": power, "hbm_peak_gbs": peak,
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
