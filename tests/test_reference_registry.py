"""INTEGRATION.md section 2, executed: the engine's classes are registered in the reference's OWN registries
(cbn/parameter_learning/__init__.py:7-13, cbn/inference/__init__.py:3) and the reference's Node / factories dispatch into
them.  Needs a source checkout of the reference (Giovannibriglia/ContinuousBayesianNetwork, the directory that holds
`cbn/`) named by the CBN_REFERENCE environment variable; the repository does not ship it, so without one the test
skips.  Without a GPU the call chain is followed up to the device boundary, where the engine must fail loudly
(there is no CPU fallback); what happens behind that boundary is covered by the golden-vector tests in test_fit_gpu.py,
which make exactly the calls the reference's Node makes (estimator.fit(node_data, parents_data), get_prob(points, query))."""
import os
import sys
import types

import pytest
import torch

REF = os.environ.get("CBN_REFERENCE", "")


def _import_reference():
    if not REF or not os.path.isdir(os.path.join(REF, "cbn")):
        pytest.skip("no reference checkout (set CBN_REFERENCE to the directory that holds cbn/)")
    names = ["gpytorch"] + ["gpytorch." + s for s in ("models", "kernels", "means", "likelihoods", "mlls", "distributions", "settings")]
    for n in names:                       # the reference imports gpytorch eagerly (cbn/parameter_learning/__init__.py:2)
        sys.modules.setdefault(n, types.ModuleType(n))
    sys.modules["gpytorch.models"].ExactGP = object
    for n in names[1:]:
        setattr(sys.modules["gpytorch"], n.split(".")[1], sys.modules[n])
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import cbn.inference as ref_inf
    import cbn.parameter_learning as ref_pl
    from cbn.base.node import Node as RefNode
    from cbn.utils import choose_probability_estimator

    return ref_pl, ref_inf, RefNode, choose_probability_estimator


def test_engine_classes_register_in_the_reference_registries():
    ref_pl, ref_inf, RefNode, choose = _import_reference()
    from cbn.base.inference import BaseInference as RefBaseInference
    from cbn.base.parameter_learning import BaseParameterLearningEstimator as RefBaseEstimator

    from continuousbayesiannetwork_b200.inference import ExactInference
    from continuousbayesiannetwork_b200.parameter_learning import BruteForce

    ref_pl.ESTIMATORS["brute_force_b200"] = BruteForce
    ref_inf.INFERENCE_OBJS["exact_b200"] = ExactInference
    try:
        # same plugin surface as the reference's ABCs (names the reference's Node / BayesianNetwork call)
        for name in ("fit", "get_prob", "sample", "save_model", "load_model"):
            assert callable(getattr(BruteForce, name)) and hasattr(RefBaseEstimator, name)
        assert callable(getattr(ExactInference, "infer")) and hasattr(RefBaseInference, "infer")
        cfg = {"estimator_name": "brute_force_b200"}
        est = choose("brute_force_b200", cfg, device="cuda")                 # the reference's factory, cbn/utils.py:23-32
        assert isinstance(est, BruteForce) and est.mle_tensor is None
        node = RefNode("reward", "brute_force_b200", cfg, ["obs_0", "action"], device="cuda")   # the reference's Node
        assert isinstance(node.estimator, BruteForce)
        with pytest.raises(ValueError):                                      # unknown names still fail as in the reference
            choose("no_such_estimator", cfg)
        if not torch.cuda.is_available():
            # Node.fit validates, sorts the parents and calls estimator.fit (cbn/base/node.py:45-83): the engine is reached
            # and refuses to run without a CUDA device -- no silent CPU path
            x = torch.tensor([0.0, 1.0, 1.0, 0.0])
            pa = torch.tensor([[0.0, 1.0, 2.0, 1.0], [1.0, 0.0, 1.0, 0.0]])
            with pytest.raises(RuntimeError, match="CUDA"):
                node.fit(x, pa)
    finally:
        ref_pl.ESTIMATORS.pop("brute_force_b200", None)
        ref_inf.INFERENCE_OBJS.pop("exact_b200", None)
