"""Host-side logic (CPU only): the builder/wrapper mirror, the network walk, the C-ABI library.

The builder tests follow the reference's own ``tests/test_model_builder.py`` (layer types and
shapes :152-186, Delta-UQ input doubling :189-237, ensemble ``num_models`` :240-264, MC-dropout
placement and train-mode flags :292-334).
"""
import ctypes
import io
import json
import os
import pickle
import re

import numpy as np
import pytest
import torch
import torch.nn as nn
import yaml

from nnueehcs_b200 import _lib, build as nbuild, evaluation, extract, ops
from nnueehcs_b200.model_builder import (DeltaUQMLPModelBuilder, EnsembleModelBuilder,
                                         KDEModelBuilder, MCDropoutModelBuilder, MLPModelBuilder,
                                         ModelBuilder, build_network)
from nnueehcs_b200.models import DeltaUQMLP, EnsembleModel, MCDropoutModel, MLPModel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MODEL_YAML = """
architecture_cnn:
  - Conv2d:
      args: [3, 16, 25]
      stride: 1
      padding: 2
  - ReLU:
      inplace: true
  - Conv2d:
      args: [16, 25, 5]
architecture_mlp:
  - Linear:
      args: [16, 25]
  - ReLU:
      inplace: true
  - Linear:
      args: [25, 25]
  - ReLU:
      inplace: true
  - Linear:
      args: [25, 5]
architecture_mlp4:
  - Linear:
      args: [16, 25]
  - ReLU:
      inplace: true
  - Linear:
      args: [25, 25]
  - ReLU:
      inplace: true
  - Linear:
      args: [25, 25]
  - ReLU:
      inplace: true
  - Linear:
      args: [25, 5]
delta_uq_model:
  estimator: std
  num_anchors: 5
  anchored_batch_size: 64
ensemble_model:
  num_models: 3
mc_dropout_model:
  num_samples: 7
  dropout_percent: 0.2
"""


@pytest.fixture
def descr():
    return yaml.safe_load(io.StringIO(MODEL_YAML))


def test_build_network_layer_types_and_shapes(descr):
    net = ModelBuilder(descr["architecture_mlp"]).build()
    assert isinstance(net, nn.Sequential) and len(net) == 5
    assert [type(m) for m in net] == [nn.Linear, nn.ReLU, nn.Linear, nn.ReLU, nn.Linear]
    assert (net[0].in_features, net[0].out_features) == (16, 25)
    assert (net[4].in_features, net[4].out_features) == (25, 5)
    cnn = ModelBuilder(descr["architecture_cnn"]).build()
    assert isinstance(cnn[0], nn.Conv2d) and cnn[0].stride == (1, 1) and cnn[0].padding == (2, 2)
    info = ModelBuilder(descr["architecture_cnn"]).get_info()
    assert info.is_cnn() and not info.is_mlp() and info.num_layers() == 3 and info.num_inputs() == 3
    info2 = ModelBuilder(descr["architecture_mlp"]).get_info()
    assert info2.is_mlp() and info2.num_layers() == 5 and info2.num_inputs() == 16
    assert not hasattr(info2, "get_estimator")
    # the builder must not mutate the caller's description
    assert descr["architecture_mlp"][0]["Linear"]["args"] == [16, 25]


def test_mlp_builder_and_unknown_loss(descr):
    m = MLPModelBuilder(descr["architecture_mlp"]).build()
    assert isinstance(m, MLPModel)
    assert m(torch.zeros(2, 16)).shape == (2, 5)
    with pytest.raises(ValueError, match="Unknown loss function"):
        MLPModelBuilder(descr["architecture_mlp"], train_config={"loss": "nope"}).build()
    with pytest.raises(Exception):
        build_network([{"NoSuchLayer": {"args": [1]}}])


def test_ensemble_builder(descr):
    b = EnsembleModelBuilder(descr["architecture_mlp"], descr["ensemble_model"])
    model = b.build()
    assert isinstance(model, EnsembleModel) and len(model.models) == 3
    assert b.get_info().get_num_models() == 3
    assert model.vectorize is False  # the reference builder never forwards it
    # member i is seeded torch.manual_seed(42 + i)  (model_builder.py:229)
    torch.manual_seed(43)
    ref1 = build_network(descr["architecture_mlp"])
    assert torch.equal(ref1[0].weight, model.models[1][0].weight)
    assert not torch.equal(model.models[0][0].weight, model.models[1][0].weight)


def test_mc_dropout_builder_placement_and_modes(descr):
    b = MCDropoutModelBuilder(descr["architecture_mlp4"], descr["mc_dropout_model"])
    model = b.build()
    assert isinstance(model, MCDropoutModel)
    names = [type(m).__name__ for m in model.model]
    # Dropout right before every Linear of descr[1:-1]; none before the first or the last Linear
    assert names == ["Linear", "ReLU", "Dropout", "Linear", "ReLU", "Dropout", "Linear", "ReLU",
                     "Linear"]
    assert [m.p for m in model.model if isinstance(m, nn.Dropout)] == [0.2, 0.2]
    assert model.num_samples == 7 and model.dropout_percent == 0.2
    info = b.get_info()
    assert info.get_num_samples() == 7 and info.get_dropout_percent() == 0.2
    model.eval()
    for layer in model.model:
        assert layer.training == isinstance(layer, nn.Dropout)
    model.train()
    assert all(layer.training for layer in model.model)
    # training forward = one plain pass of the net (models.py:148-149)
    x = torch.randn(4, 16)
    torch.manual_seed(0)
    a = model(x)
    torch.manual_seed(0)
    assert torch.equal(a, model.model(x))


def test_delta_uq_builder_doubles_inputs(descr):
    b = DeltaUQMLPModelBuilder(descr["architecture_mlp"], descr["delta_uq_model"])
    model = b.build()
    assert isinstance(model, DeltaUQMLP)
    assert model.net[0].in_features == 32 and model.num_anchors == 5 and model.batch_size == 64
    info = b.get_info()
    assert info.num_inputs() == 32 and info.get_estimator() == "std" and info.get_batch_size() == 64
    assert b.build().net[0].in_features == 32  # doubled once, not per build()
    with pytest.raises(KeyError):
        DeltaUQMLPModelBuilder(descr["architecture_mlp"],
                               {"estimator": "std", "num_anchors": 5}).build()
    # training-mode forward stays stock torch and keeps the batch size
    model.train()
    assert model(torch.randn(6, 16)).shape == (6, 5)
    model.anchors = torch.randn(5, 16)
    assert model.anchors.shape == (5, 16) and "_anchors" in dict(model.named_buffers())


def test_pager_builder_and_wrapper_contract(descr):
    """reference tests/test_model_builder.py:215-237 (input doubling, num_anchors) + the wrapper's
    buffers, callbacks and loud failure off the GPU."""
    from nnueehcs_b200.model_builder import PAGERModelBuilder
    from nnueehcs_b200.models import PAGERMLP
    b = PAGERModelBuilder(descr["architecture_mlp"], {"estimator": "std", "num_anchors": 4})
    model = b.build()
    assert isinstance(model, PAGERMLP) and isinstance(model, DeltaUQMLP)
    assert model.net[0].in_features == 32 and model.num_anchors == 4
    assert b.get_info().num_inputs() == 32 and b.get_info().get_estimator() == "std"
    model.anchors = torch.randn(4, 16)
    model.anchors_Y = torch.randn(4, 5)
    bufs = dict(model.named_buffers())
    assert "_anchors" in bufs and "_anchors_Y" in bufs
    cb = model.get_callbacks()[0]
    for i in range(3):
        cb.on_train_batch_end(None, model, None, (torch.full((2, 16), float(i)),
                                                  torch.full((2, 5), float(10 + i))), i)
    cb.on_validation_epoch_start(None, model)
    assert model.anchors.shape == (4, 16) and model.anchors_Y.shape == (4, 5)
    assert float(model.anchors_Y[2, 0]) == 11.0          # rows 2-3 come from the second batch
    model.train()
    assert model(torch.randn(6, 16)).shape == (6, 5)      # training forward: stock torch
    model.eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(torch.randn(6, 16), return_ue=True)


def test_out_of_scope_wrappers_say_so(descr):
    from nnueehcs_b200.model_builder import KNNKDEModelBuilder
    with pytest.raises(NotImplementedError, match="outside the hot path"):
        KNNKDEModelBuilder(descr["architecture_mlp"], {"bandwidth": "scott", "k": 10}).build()


def test_kde_builder_and_wrapper_contract(descr):
    """KDEMLPModel mirror (reference models.py:191-240): fit on a train_fit_prop share, sklearn's
    scott bandwidth, errors before the fit, the fit callback, no CPU path for the score."""
    from nnueehcs_b200.models import KDEMLPModel
    model = KDEModelBuilder(descr["architecture_mlp"],
                            {"bandwidth": "scott", "rtol": 0.1, "train_fit_prop": 0.5}).build()
    assert isinstance(model, KDEMLPModel) and isinstance(model, MLPModel)
    assert model.rtol == pytest.approx(1e-5) and model.kde is None
    x = torch.randn(6, 16)
    assert model(x).shape == (6, 5)
    with pytest.raises(ValueError, match="KDE not fitted yet"):
        model(x, return_ue=True)
    cb = model.get_callbacks()[0]
    for i in range(4):
        cb.on_train_batch_end(None, model, None, (torch.randn(25, 16), None), i)
    cb.on_train_epoch_end(None, model)
    assert model._kde_data.shape == (50, 16) and "_kde_data" in dict(model.named_buffers())
    assert model.kde["bandwidth_"] == pytest.approx(50 ** (-1 / 20))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(x, return_ue=True)
    with pytest.raises(ValueError, match="bandwidth must be"):
        KDEModelBuilder(descr["architecture_mlp"], {"bandwidth": "epanechnikov"}).build()
    sil = KDEModelBuilder(descr["architecture_mlp"], {"bandwidth": "silverman"}).build()
    sil.fit_kde(torch.randn(50, 16))        # sklearn: (n (d + 2) / 4) ** (-1 / (d + 4))
    assert sil.kde["bandwidth_"] == pytest.approx((50 * 18 / 4) ** (-1 / 20))


def test_runtime_and_throughput_metrics_protocol():
    """Reference evaluation.py:413-516: warm-ups untimed, every timed trial is one call on the
    concatenated ID + OOD inputs; runtime = mean / std of the seconds, throughput = mean / std of
    samples / seconds; the UQ variants call model(x, return_ue=True)."""
    calls = []

    class Fake(torch.nn.Module):
        def forward(self, x, return_ue=False):
            calls.append((x.shape[0], return_ue, self.training))
            return (x, x[:, 0]) if return_ue else x

    idd, ood = (torch.zeros(30, 2), None), (torch.ones(12, 2), None)
    m = Fake().train()
    r = evaluation.UncertaintyEstimatingRuntimeEvaluation(num_trials=3, num_warmup=2).evaluate(m, idd, ood)
    assert set(r) == {"runtime", "runtime_std"} and r["runtime"] > 0 and r["runtime_std"] >= 0
    assert calls == [(42, True, False)] * 5          # eval mode, 2 warm-ups + 3 trials
    calls.clear()
    r = evaluation.BaseModelThroughputEvaluation(num_trials=2, num_warmup=0).evaluate(m, idd, ood)
    assert set(r) == {"base_model_throughput", "throughput_std"} and calls == [(42, False, False)] * 2
    assert r["base_model_throughput"] > 0
    r = evaluation.UncertaintyEstimatingThroughputEvaluation.from_config({"trials": 2, "warmup": 1}) \
        .evaluate(m, idd, ood)
    assert set(r) == {"uncertainty_estimating_throughput", "throughput_std"}
    assert evaluation.UncertaintyEstimatingThroughputEvaluation.get_objectives() == [
        {"name": "uncertainty_estimating_throughput", "type": "maximize"}]
    assert evaluation.BaseModelRuntimeEvaluation.get_metrics() == ["base_model_runtime", "runtime_std"]
    with pytest.raises(NotImplementedError):
        evaluation.RuntimeEvaluation().evaluate(m, idd, ood)
    # JensenShannonEvaluation on [N, d > 1] scores: mean of jensenshannon(p[i], q[i]) over rows
    from oracle import metrics_oracle
    rng = np.random.default_rng(0)
    pa, pb = rng.random((7, 5)).astype(np.float32), rng.random((7, 5)).astype(np.float32)
    exp = np.mean([metrics_oracle.jensenshannon(pa[i], pb[i]) for i in range(7)])
    got = evaluation.JensenShannonEvaluation()._evaluate_uncertainties(
        evaluation.UncertaintyEstimate(torch.from_numpy(pa)),
        evaluation.UncertaintyEstimate(torch.from_numpy(pb)))["jensen_shannon_distance"]
    assert got == pytest.approx(exp, rel=1e-12)
    # EuclideanEvaluation: mean over rows of the L2 norm of the paired difference
    a = evaluation.UncertaintyEstimate(torch.tensor([[3.0, 4.0], [0.0, 0.0]]))
    b = evaluation.UncertaintyEstimate(torch.tensor([[0.0, 0.0], [6.0, 8.0]]))
    assert evaluation.EuclideanEvaluation()._evaluate_uncertainties(a, b) == {"euclidean_distance": 7.5}


def test_host_side_metrics_have_the_reference_interface(golden_dir):
    """The mirrored host-side metric classes expose the reference's names, result keys,
    objectives, metric lists and factory behaviour (evaluation.py:205-227, :383-516, :700-812),
    as recorded in tests/golden/host_metrics_interface.json (make_golden_interface.py)."""
    with open(os.path.join(golden_dir, "host_metrics_interface.json")) as f:
        ref = json.load(f)

    class Fake(torch.nn.Module):
        def forward(self, x, return_ue=False):
            return (x, x[:, 0]) if return_ue else x

    idd, ood = (torch.rand(20, 3), None), (torch.rand(20, 3), None)
    assert sorted(ref["runtime_classes"]) == sorted(
        ("BaseModelRuntimeEvaluation", "UncertaintyEstimatingRuntimeEvaluation",
         "BaseModelThroughputEvaluation", "UncertaintyEstimatingThroughputEvaluation"))
    for cls_name, theirs in ref["runtime_classes"].items():
        mine = getattr(evaluation, cls_name)
        assert mine.name == theirs["name"]
        assert mine.get_objectives() == theirs["objectives"]
        assert mine.get_metrics() == theirs["metrics"]
        a = mine(num_trials=2, num_warmup=1)
        assert a.get_name() == theirs["instance_name"]
        assert sorted(a.evaluate(Fake(), idd, ood)) == theirs["result_keys"]
    assert evaluation.MaxMemoryUsageEvaluation.name == ref["max_memory_usage"]["name"]
    assert (evaluation.MaxMemoryUsageEvaluation().get_objectives()
            == ref["max_memory_usage"]["objectives"])

    def scores(rows):
        return evaluation.UncertaintyEstimate(torch.tensor(rows, dtype=torch.float32))

    e = ref["euclidean"]
    got = evaluation.EuclideanEvaluation()._evaluate_uncertainties(scores(e["a"]), scores(e["b"]))
    assert got == e["result"]
    # JensenShannonEvaluation on [N, d > 1] scores: mean of scipy's jensenshannon over the rows
    j = ref["jensen_shannon"]
    got = evaluation.JensenShannonEvaluation()._evaluate_uncertainties(scores(j["a"]), scores(j["b"]))
    assert got["jensen_shannon_distance"] == pytest.approx(
        j["result"]["jensen_shannon_distance"], rel=1e-6)
    g = ref["get_evaluator"]
    mine = evaluation.get_evaluator(g["config"])
    assert [type(m).__name__ for m in mine.metrics] == g["classes"]
    assert [[getattr(m, "num_trials", None), getattr(m, "num_warmup", None)] for m in mine.metrics] \
        == g["trials_warmup"]
    g = ref["get_uncertainty_evaluator"]
    mine = evaluation.get_uncertainty_evaluator(g["config"])
    assert [type(m).__name__ for m in mine.metrics] == g["classes"]


def test_split_blocks_vocabulary(descr):
    net = MCDropoutModelBuilder(descr["architecture_mlp4"], descr["mc_dropout_model"]).build().model
    blocks = extract.split_blocks(net)
    assert [(b.linear.out_features, b.bn is not None, b.relu, b.dropout) for b in blocks] == [
        (25, False, True, True), (25, False, True, True), (25, False, True, False),
        (5, False, False, False)]
    assert extract.dropout_widths(blocks) == [25, 25]
    bn_net = build_network([{"Linear": {"args": [5, 8]}}, {"BatchNorm1d": {"args": [8]}},
                            {"ReLU": None}, {"Linear": {"args": [8, 1]}}])
    b2 = extract.split_blocks(bn_net)
    assert b2[0].bn is bn_net[1] and b2[0].relu and not b2[1].relu
    with pytest.raises(ValueError, match="Conv2d is not supported"):
        extract.split_blocks(ModelBuilder(descr["architecture_cnn"]).build())
    with pytest.raises(ValueError, match="BatchNorm1d must directly follow"):
        extract.split_blocks(nn.Sequential(nn.Linear(4, 4), nn.ReLU(), nn.BatchNorm1d(4)))
    with pytest.raises(ValueError, match="do not chain"):
        extract.split_blocks(nn.Sequential(nn.Linear(4, 4), nn.Linear(5, 1)))


def test_tensors_version_tracks_inplace_updates():
    net = nn.Sequential(nn.Linear(3, 3))
    k0 = extract.tensors_version([net])
    assert k0 == extract.tensors_version([net])
    with torch.no_grad():
        net[0].weight.add_(1.0)
    assert k0 != extract.tensors_version([net])
    # a replaced parameter and a structural edit change the key (an edit through the .data
    # alias cannot be seen by any version counter: invalidate_packed() is the explicit way)
    k2 = extract.tensors_version([net])
    net[0].bias = nn.Parameter(net[0].bias.detach().clone())
    k3 = extract.tensors_version([net])
    assert k3 != k2
    net.append(nn.ReLU())
    assert extract.tensors_version([net]) != k3


def test_invalidate_packed_and_shared_seed_without_a_shard():
    class _Handle:
        closed = False

        def close(self):
            self.closed = True

    model = EnsembleModel([nn.Sequential(nn.Linear(3, 1))])
    h = _Handle()
    model.__dict__["_uq_cache"] = ("key", h)
    model.invalidate_packed()
    assert h.closed and model.__dict__["_uq_cache"] is None
    model.invalidate_packed()                      # idempotent
    assert model._shared_seed(1234, "cpu") == 1234  # no shard: the rank's own seed


def test_eval_forward_requires_cuda_and_never_falls_back(descr):
    model = EnsembleModelBuilder(descr["architecture_mlp"], descr["ensemble_model"]).build()
    model.eval()
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        model(torch.zeros(2, 16), return_ue=True)
    mc = MCDropoutModelBuilder(descr["architecture_mlp4"], descr["mc_dropout_model"]).build()
    mc.eval()
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        mc(torch.zeros(2, 16), return_ue=True)
    # training-mode forward is the stock autograd path and works on CPU
    model.train()
    mean, std = model(torch.zeros(2, 16), return_ue=True)
    assert mean.shape == (2, 5) and std.shape == (2, 5) and mean.requires_grad


def test_wrappers_pickle_without_device_cache(descr):
    model = EnsembleModelBuilder(descr["architecture_mlp"], descr["ensemble_model"]).build()
    model.__dict__["_uq_cache"] = ("key", object())  # pretend a packed handle exists
    clone = pickle.loads(pickle.dumps(model))
    assert clone.__dict__["_uq_cache"] is None and clone.uq_precision == model.uq_precision
    assert torch.equal(clone.models[2][0].weight, model.models[2][0].weight)
    buf = io.BytesIO()
    torch.save(model, buf)  # the reference checkpoints whole modules (training.py:64-65)
    buf.seek(0)
    again = torch.load(buf, weights_only=False)
    assert isinstance(again, EnsembleModel) and again.__dict__["_uq_cache"] is None


def test_evaluator_factories():
    ev = evaluation.get_uncertainty_evaluator(["wasserstein_distance",
                                               {"name": "jensen_shannon_distance"}])
    assert [m.get_name() for m in ev.metrics] == ["wasserstein_distance", "jensen_shannon_distance"]
    assert ev.get_all_metrics() == ["wasserstein_distance", "jensen_shannon_distance"]
    assert ev.get_training_objectives()[0] == {"name": "wasserstein_distance", "type": "maximize"}
    assert isinstance(evaluation.get_evaluator({"name": "wasserstein"}).metrics[0],
                      evaluation.WassersteinEvaluation)
    # the host-side metrics the reference's configs name (evaluation.py:383-516, :205-227)
    ev = evaluation.get_uncertainty_evaluator(
        [{"name": "runtime", "trials": 3, "warmup": 1}, "uncertainty_estimating_runtime",
         {"name": "uncertainty_estimating_throughput", "trials": 4}, "euclidean_distance"])
    assert [type(m).__name__ for m in ev.metrics] == [
        "BaseModelRuntimeEvaluation", "UncertaintyEstimatingRuntimeEvaluation",
        "UncertaintyEstimatingThroughputEvaluation", "EuclideanEvaluation"]
    assert (ev.metrics[0].num_trials, ev.metrics[0].num_warmup) == (3, 1)
    assert (ev.metrics[2].num_trials, ev.metrics[2].num_warmup) == (4, 5)
    ev = evaluation.get_evaluator([{"name": "uncertainty_estimating_throughput", "trials": 2},
                                   {"name": "base_model_throughput"}, {"name": "max_memory_usage"},
                                   {"name": "runtime"}, {"name": "no_such_metric"}])
    assert [m.get_name() for m in ev.metrics] == [
        "uncertainty_estimating_throughput", "base_model_throughput", "max_memory_usage",
        "base_model_runtime"]      # unknown names are skipped by this factory, as in the reference
    ev = evaluation.get_uncertainty_evaluator(
        ["auroc", "mean_score", "max_score", {"name": "percentile_score", "percentile": 90.0},
         {"name": "tnr_at_tpr", "target_tpr": 0.95},
         {"name": "percentile_classification", "threshold": 0.95},
         {"name": "percentile_classification", "threshold": 0.95, "reversed": True}])
    assert [type(m).__name__ for m in ev.metrics] == [
        "AUROC", "MeanScoreEvaluation", "MaxScoreEvaluation", "PercentileScoreEvaluation", "TNRatTPX",
        "PercentileBasedIdOodClassifier", "ReversedPercentileBasedIdOodClassifier"]
    assert ev.metrics[3].percentile == 90.0 and ev.metrics[4].get_name() == "tnr_at_tpr95"
    ev = evaluation.get_evaluator([{"name": "percentile_classification", "threshold": 0.9,
                                    "reversed": True}, {"name": "tnr_at_tpr", "target_tpr": 0.5}])
    assert ev.metrics[0].get_name() == "percentile_classification_reversed_90"
    assert ev.get_all_metrics() == ["sensitivity", "specificity", "tnr_at_tpr"]
    with pytest.raises(ValueError, match="between 0 and 1"):
        evaluation.TNRatTPX(1.5)
    with pytest.raises(ValueError, match="between 0 and 100"):
        evaluation.PercentileScoreEvaluation(101)
    with pytest.raises(ValueError, match="Invalid metric type"):
        evaluation.get_uncertainty_evaluator("bogus")


def test_uncertainty_estimate_contract():
    with pytest.raises(ValueError, match="empty"):
        evaluation.UncertaintyEstimate(torch.zeros(0))
    with pytest.raises(ValueError, match="same first dimension"):
        evaluation.UncertaintyEstimate((torch.zeros(3), torch.zeros(4)))
    with pytest.raises(TypeError):
        evaluation.UncertaintyEstimate([1, 2, 3])
    ue = evaluation.UncertaintyEstimate(torch.arange(6.0).reshape(3, 2))
    assert ue.dimensions == 1 and ue.flatten().shape == (6,) and ue.mean() == 2.5
    assert ue.data.shape == (3, 2)
    two = evaluation.UncertaintyEstimate((torch.ones(3), torch.zeros(3)))
    assert two.dimensions == 2 and two.mean() == 0.5
    with pytest.raises(ValueError, match="flatten"):
        two.flatten()


# ---- the C-ABI shared library -------------------------------------------------------------------

def test_library_builds_loads_and_exports_every_declared_symbol():
    path = nbuild.build()
    assert os.path.exists(path)
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "nnueehcs_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(uq_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    raw = ctypes.CDLL(path)
    for name in declared:
        assert hasattr(raw, name), f"{name} not exported"
    assert lib.uq_abi_version() == _lib.ABI_VERSION == 3
    lib.uq_launch_count_reset()
    assert lib.uq_launch_count() == 0


def test_abi_struct_layouts_match_header():
    # uq_layer_desc: 2 x int32, 6 pointers, float, 2 x int32 -> 72 bytes on LP64
    assert ctypes.sizeof(_lib.LayerDesc) == 72
    assert _lib.LayerDesc.weight.offset == 8 and _lib.LayerDesc.bn_eps.offset == 56
    # uq_forward_args (ABI 2): 8 x int32, double, 2 x uint64, 4 pointers -> 88 bytes
    assert ctypes.sizeof(_lib.ForwardArgs) == 88
    assert _lib.ForwardArgs.dropout_p.offset == 32 and _lib.ForwardArgs.masks.offset == 56
    assert _lib.ForwardArgs.anchor_targets.offset == 72 and _lib.ForwardArgs.score_floor.offset == 80


def test_argument_errors_surface_as_python_exceptions_without_a_gpu():
    lib = _lib.load()
    out = ctypes.c_double()
    # NULL pointers / empty input are rejected before any CUDA call is made
    rc = lib.uq_wasserstein_1d(None, 0, None, 0, ctypes.byref(out), None, 0, None)
    assert rc == _lib.UQ_ERR_INVALID
    with pytest.raises(ValueError, match="can't be empty"):
        _lib.check(rc)
    h = ctypes.c_void_p()
    rc = lib.uq_model_create(ctypes.byref(h), 0, 0, None, None)
    assert rc == _lib.UQ_ERR_INVALID and not h.value
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.wasserstein_1d(torch.zeros(4), torch.zeros(4))


def test_metric_evaluator_shares_one_forward_per_dataset():
    """SURVEY 8f row 3: the two UQ forwards run once for all score-based metrics (the reference
    runs them once per metric); ``share_forward=False`` restores the reference's call pattern."""
    calls = []

    class Model(torch.nn.Module):
        def forward(self, x, return_ue=False):
            calls.append(int(x.shape[0]))
            return x[:, :1], x[:, :1] * 2.0

    class U(evaluation.UncertaintyEvaluationMetric):
        def __init__(self, name): self._n = name
        def _evaluate_uncertainties(self, a, b): return {self._n: a.mean() + b.mean()}
        @classmethod
        def get_objectives(cls): return []
        @classmethod
        def get_metrics(cls): return []
        def get_name(self): return self._n

    class Cm(evaluation.ClassificationMetric):
        def _evaluate_scores(self, a, b): return {"c": float(a.sum() + b.sum())}
        @classmethod
        def get_objectives(cls): return []
        @classmethod
        def get_metrics(cls): return ["c"]
        def get_name(self): return "c"

    id_d, ood_d = (torch.ones(3, 2), None), (torch.ones(5, 2), None)
    out = evaluation.MetricEvaluator([U("a"), U("b"), Cm()]).evaluate(Model(), id_d, ood_d)
    assert calls == [3, 5] and out == {"a": 4.0, "b": 4.0, "c": 16.0}
    calls.clear()
    out2 = evaluation.MetricEvaluator([U("a"), U("b"), Cm()], share_forward=False).evaluate(
        Model(), id_d, ood_d)
    assert calls == [3, 5] * 3 and out2 == out


def test_custom_ops_are_registered_for_cuda_only():
    """SURVEY 8b: the C ABI is reachable as torch.ops.nnueehcs_b200.*; the ops have a CUDA
    implementation and nothing else, so CPU tensors fail loudly at the dispatcher."""
    ns = getattr(torch.ops, ops.OP_NAMESPACE)
    for name in ops.OP_SCHEMAS:
        assert hasattr(ns, name), name
        assert torch._C._dispatch_has_kernel_for_dispatch_key(f"{ops.OP_NAMESPACE}::{name}", "CUDA")
        assert not torch._C._dispatch_has_kernel_for_dispatch_key(f"{ops.OP_NAMESPACE}::{name}",
                                                                  "CPU")
    with pytest.raises(NotImplementedError):
        ns.wasserstein_1d(torch.rand(8), torch.rand(8))
    with pytest.raises(NotImplementedError):
        ns.kde_jsd(torch.rand(8), torch.rand(8), 100)
    with pytest.raises(NotImplementedError):
        ns.moments_merge(torch.rand(2, 8), torch.rand(2, 8), [1.0, 1.0])


def test_graft_entry_build_runs_on_cpu():
    """The driver's "does it build" check: compiles (or reuses) the library, loads it through the
    C ABI, checks the ABI version against the binding, imports the package and the oracle."""
    import __graft_entry__ as entry
    entry.build()
