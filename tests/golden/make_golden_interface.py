#!/usr/bin/env python
"""Golden interface of the reference's host-side metric classes (nnueehcs/evaluation.py:205-227,
:383-516, :700-812): names, result keys, objectives, metric lists, the factories' choices, and the
Euclidean / row-wise Jensen-Shannon values on stored seeded inputs.

The reference package is not vendored.  These values are recorded from the mirror
``nnueehcs_b200.evaluation`` as of commit 79aa993, whose tests compared every one of them with the
live reference classes and passed; the module has not changed since.  Recording them lets
``tests/test_host.py`` keep that comparison without the reference tree:

    python tests/golden/make_golden_interface.py
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from nnueehcs_b200 import evaluation as ev  # noqa: E402

RUNTIME_CLASSES = ("BaseModelRuntimeEvaluation", "UncertaintyEstimatingRuntimeEvaluation",
                   "BaseModelThroughputEvaluation", "UncertaintyEstimatingThroughputEvaluation")
EVALUATOR_CONFIG = [{"name": "uncertainty_estimating_throughput", "trials": 3, "warmup": 2},
                    {"name": "runtime", "trials": 4}, {"name": "max_memory_usage"},
                    {"name": "mean_score"}]
UNCERTAINTY_EVALUATOR_CONFIG = [{"name": "runtime", "trials": 4}, "uncertainty_estimating_runtime",
                                "euclidean_distance",
                                {"name": "uncertainty_estimating_throughput", "warmup": 1}]


class Fake(torch.nn.Module):
    def forward(self, x, return_ue=False):
        return (x, x[:, 0]) if return_ue else x


def main():
    rng = np.random.default_rng(7)
    idd, ood = (torch.rand(20, 3), None), (torch.rand(20, 3), None)
    out = {"runtime_classes": {}}
    for name in RUNTIME_CLASSES:
        cls = getattr(ev, name)
        inst = cls(num_trials=2, num_warmup=1)
        out["runtime_classes"][name] = {
            "name": cls.name, "objectives": cls.get_objectives(), "metrics": cls.get_metrics(),
            "instance_name": inst.get_name(), "result_keys": sorted(inst.evaluate(Fake(), idd, ood))}
    mm = ev.MaxMemoryUsageEvaluation
    out["max_memory_usage"] = {"name": mm.name, "objectives": mm().get_objectives()}

    ua, ub = rng.random((17, 4), dtype=np.float32), rng.random((17, 4), dtype=np.float32)
    r = ev.EuclideanEvaluation()._evaluate_uncertainties(
        ev.UncertaintyEstimate(torch.from_numpy(ua)), ev.UncertaintyEstimate(torch.from_numpy(ub)))
    out["euclidean"] = {"a": ua.tolist(), "b": ub.tolist(), "result": r}
    pa = rng.random((9, 4), dtype=np.float32) + np.float32(0.1)
    pb = rng.random((9, 4), dtype=np.float32) + np.float32(0.1)
    pa[0, 1] = 0.0
    r = ev.JensenShannonEvaluation()._evaluate_uncertainties(
        ev.UncertaintyEstimate(torch.from_numpy(pa)), ev.UncertaintyEstimate(torch.from_numpy(pb)))
    out["jensen_shannon"] = {"a": pa.tolist(), "b": pb.tolist(),
                             "result": {k: float(v) for k, v in r.items()}}

    mine = ev.get_evaluator(EVALUATOR_CONFIG)
    out["get_evaluator"] = {
        "config": EVALUATOR_CONFIG, "classes": [type(m).__name__ for m in mine.metrics],
        "trials_warmup": [[getattr(m, "num_trials", None), getattr(m, "num_warmup", None)]
                          for m in mine.metrics]}
    mine = ev.get_uncertainty_evaluator(UNCERTAINTY_EVALUATOR_CONFIG)
    out["get_uncertainty_evaluator"] = {"config": UNCERTAINTY_EVALUATOR_CONFIG,
                                        "classes": [type(m).__name__ for m in mine.metrics]}
    path = os.path.join(HERE, "host_metrics_interface.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(path)


if __name__ == "__main__":
    main()
