"""Generate golden fixtures by running the UNMODIFIED reference on CPU.

Needs a source checkout of the reference (the directory that holds ``cbn/``) and no
GPU: ``CBN_REFERENCE=<checkout> python tests/golden/make_golden.py``.  Writes
``tests/golden/*.npz``.
The reference imports ``gpytorch`` eagerly (cbn/parameter_learning/__init__.py:2)
which is not installed; a dummy module tree in ``sys.modules`` is enough because
only ``BruteForce`` is exercised (SURVEY.md section 8c).  No reference file is edited
or copied; only the numbers it produces are stored.
"""
import os
import random
import sys
import types

import numpy as np

REF = os.environ.get("CBN_REFERENCE", "")
HERE = os.path.dirname(os.path.abspath(__file__))


def _stub_gpytorch():
    names = ["gpytorch"] + ["gpytorch." + s for s in
                            ("models", "kernels", "means", "likelihoods", "mlls", "distributions", "settings")]
    for n in names:
        sys.modules[n] = types.ModuleType(n)
    sys.modules["gpytorch.models"].ExactGP = object
    for n in names[1:]:
        setattr(sys.modules["gpytorch"], n.split(".")[1], sys.modules[n])


def main():
    if not REF or not os.path.isdir(os.path.join(REF, "cbn")):
        sys.exit("set CBN_REFERENCE to a checkout of the reference (the directory that holds cbn/)")
    _stub_gpytorch()
    sys.path.insert(0, REF)
    import networkx as nx
    import pandas as pd
    import torch
    from cbn.base.bayesian_network import BayesianNetwork
    from cbn.parameter_learning.brute_force import BruteForce

    torch.manual_seed(0)
    cfg_pl = {"estimator_name": "brute_force"}
    cfg_inf = {"inference_obj": "exact"}

    # ------------------------------------------------------------------ FrozenLake (config 1)
    df = pd.read_pickle(os.path.join(REF, "cbn/examples/frozen_lake.pkl"))
    df.columns = ["obs_0", "action", "reward"]
    data = df.values.astype(np.float32)
    dag = nx.DiGraph()
    dag.add_edges_from([("obs_0", "reward"), ("action", "reward")])
    bn = BayesianNetwork(dag, df, cfg_pl, cfg_inf, device="cpu")
    out = {"data": data}
    for name in ("obs_0", "action", "reward"):
        out["mle_" + name] = bn.nodes_obj[name].estimator.mle_tensor.numpy()
        out["domain_" + name] = bn.nodes_obj[name].info[name][3].numpy()
    # parents of reward sorted by name: action, obs_0 (cbn/base/bayesian_network.py:104-106)
    est = bn.nodes_obj["reward"].estimator
    q_rows = torch.tensor(data[:, [1, 0]]).unsqueeze(-1)                     # [n, P=2, 1] (action, obs_0)
    dom_y = torch.unique(torch.tensor(data[:, 2])).unsqueeze(0)
    out["getprob_rows"] = est.get_prob(dom_y.expand(q_rows.shape[0], -1), q_rows).numpy()
    # 100x100 linspace grid of tests/test_frozen_lake_parameter_learning.py:30-33 (obs, action order
    # of that script: train_x = [obs, action]) -- evaluated against an estimator fitted the same way
    obs = torch.tensor(data[:, 0]); act = torch.tensor(data[:, 1]); rew = torch.tensor(data[:, 2])
    est2 = BruteForce(cfg_pl, device="cpu")
    est2.fit(rew, torch.stack([obs, act], dim=0))
    out["mle_reward_obs_action"] = est2.mle_tensor.numpy()
    ot = torch.linspace(obs.min(), obs.max(), 100); at = torch.linspace(act.min(), act.max(), 100)
    AA, BB = torch.meshgrid(ot, at, indexing="ij")
    grid = torch.stack([AA.reshape(-1), BB.reshape(-1)], dim=1)
    out["grid_query"] = grid.numpy()
    out["getprob_grid"] = est2.get_prob(dom_y.expand(grid.shape[0], -1), grid.unsqueeze(-1)).numpy()
    # marginal branch (no parents)
    out["getprob_marginal_reward_pts"] = np.array([[0.0, 1.0, 0.5]], dtype=np.float32)
    est3 = BruteForce(cfg_pl, device="cpu"); est3.fit(rew, None)
    out["mle_reward_marginal"] = est3.mle_tensor.numpy()
    out["getprob_marginal_reward"] = est3.get_prob(torch.tensor(out["getprob_marginal_reward_pts"])).numpy()
    # BayesianNetwork.infer, full parent evidence, N_max = card(reward) = 2
    ev = {"obs_0": torch.tensor(data[:, 0:1]), "action": torch.tensor(data[:, 1:2])}
    pdf, dom = bn.infer("reward", ev, N_max=2)
    out["infer_rows_pdf"] = pdf.numpy(); out["infer_rows_dom"] = dom.numpy()
    # a batch with unseen configurations (obs 5, 7 never occur; action 9 never occurs)
    ev2 = {"obs_0": torch.tensor([[14.0], [5.0], [0.0], [10.0], [7.0], [14.0]]),
           "action": torch.tensor([[2.0], [1.0], [9.0], [1.0], [0.0], [1.0]])}
    pdf2, dom2 = bn.infer("reward", ev2, N_max=2)
    out["infer_unseen_obs"] = ev2["obs_0"].numpy(); out["infer_unseen_act"] = ev2["action"].numpy()
    out["infer_unseen_pdf"] = pdf2.numpy(); out["infer_unseen_dom"] = dom2.numpy()
    np.savez_compressed(os.path.join(HERE, "frozen_lake.npz"), **out)

    # ------------------------------------------------------------------ seeded synthetic families
    rng = np.random.default_rng(1234)
    fam = {}
    cases = [  # (P, cards parents..., card node, n)
        (0, [], 5, 3000), (1, [3], 2, 4000), (2, [4, 3], 3, 5000), (3, [4, 4, 4], 4, 20000),
        (4, [2, 3, 2, 5], 6, 30000), (2, [11, 7], 20, 6000),
    ]
    for ci, (P, pc, nc, n) in enumerate(cases):
        # float-valued categories, some negative / non-integer (the reference keys on float equality)
        doms = [np.sort(rng.choice(np.arange(-8, 40) * 0.25, size=c, replace=False)).astype(np.float32) for c in pc + [nc]]
        codes = [rng.integers(0, c, size=n) for c in pc]
        # node depends on parents through a random table so the CPT is not flat
        tbl = rng.dirichlet(np.ones(nc) * 0.5, size=int(np.prod(pc)) if pc else 1)
        flat = np.zeros(n, dtype=np.int64)
        for c, k in zip(codes, pc):
            flat = flat * k + c
        u = rng.random(n)
        xcode = (u[:, None] > np.cumsum(tbl[flat], axis=1)).sum(axis=1).clip(0, nc - 1)
        node = torch.tensor(doms[-1][xcode])
        parents = torch.tensor(np.stack([doms[i][codes[i]] for i in range(P)])) if P else None
        e = BruteForce(cfg_pl, device="cpu")
        e.fit(node, parents)
        fam[f"c{ci}_node"] = node.numpy()
        if P:
            fam[f"c{ci}_parents"] = parents.numpy()
        fam[f"c{ci}_mle"] = e.mle_tensor.numpy()
        # queries: 256 rows, mixture of seen values, values outside the domain, candidate points incl. unseen
        Q = 256
        V = nc + 1
        pts = np.tile(np.concatenate([doms[-1], [123.5]]).astype(np.float32), (Q, 1))
        pts = pts[:, rng.permutation(V)]
        fam[f"c{ci}_pts"] = pts
        if P:
            qv = np.stack([doms[i][rng.integers(0, pc[i], size=Q)] for i in range(P)], axis=1)
            qv[rng.random(Q) < 0.1, 0] = 777.0  # unseen parent value
            fam[f"c{ci}_query"] = qv.astype(np.float32)
            fam[f"c{ci}_getprob"] = e.get_prob(torch.tensor(pts), torch.tensor(qv.astype(np.float32)).unsqueeze(-1)).numpy()
        else:
            fam[f"c{ci}_getprob"] = e.get_prob(torch.tensor(pts[:1])).numpy()
    fam["n_cases"] = np.array(len(cases))
    np.savez_compressed(os.path.join(HERE, "synthetic_families.npz"), **fam)

    # ------------------------------------------------------------------ star DAG through BayesianNetwork.infer
    rng = np.random.default_rng(99)
    n = 20000
    pc = [3, 4, 5]; nc = 3
    names = ["p_b", "p_a", "p_c"]           # deliberately not in sorted order
    doms = {nm: np.sort(rng.choice(np.arange(0, 30) * 0.5, size=c, replace=False)).astype(np.float32) for nm, c in zip(names, pc)}
    doms["y"] = np.array([-1.0, 0.5, 2.0], dtype=np.float32)
    codes = {nm: rng.integers(0, c, size=n) for nm, c in zip(names, pc)}
    tbl = rng.dirichlet(np.ones(nc) * 0.7, size=int(np.prod(pc)))
    flat = (codes["p_b"] * 4 + codes["p_a"]) * 5 + codes["p_c"]
    ycode = (rng.random(n)[:, None] > np.cumsum(tbl[flat], axis=1)).sum(axis=1).clip(0, nc - 1)
    sdf = pd.DataFrame({nm: doms[nm][codes[nm]] for nm in names})
    sdf["y"] = doms["y"][ycode]
    sdag = nx.DiGraph(); sdag.add_edges_from([(nm, "y") for nm in names])
    sbn = BayesianNetwork(sdag, sdf, cfg_pl, cfg_inf, device="cpu")
    Q = 512
    qi = rng.integers(0, n, size=Q)
    sev = {nm: torch.tensor(sdf[nm].values[qi].astype(np.float32)).reshape(-1, 1) for nm in names}
    sev["p_a"][5, 0] = 1234.0   # one unseen parent value
    spdf, sdom = sbn.infer("y", sev, N_max=3)
    star = {"data": sdf[names + ["y"]].values.astype(np.float32), "columns": np.array(names + ["y"]),
            "mle_y": sbn.nodes_obj["y"].estimator.mle_tensor.numpy(),
            "infer_pdf": spdf.numpy(), "infer_dom": sdom.numpy()}
    for nm in names:
        star["ev_" + nm] = sev[nm].numpy()
        star["mle_" + nm] = sbn.nodes_obj[nm].estimator.mle_tensor.numpy()
    np.savez_compressed(os.path.join(HERE, "star_infer.npz"), **star)
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    random.seed(0)
    main()
