"""Parity of the CUDA UQ forward with the reference (B200 only: ``pytest -m gpu``).

Every comparison goes through the C ABI (``ops.PackedModel`` -> ``uq_forward``) or the wrapper
mirror on top of it.  References are (a) the golden outputs of the reference's own classes
(``tests/golden``) and (b) the CPU oracle on the same seeded inputs.

Tolerances
----------
fp32 mode : north_star's 1e-5 relative, read as ``|got-ref| <= 1e-5*|ref| + 1e-5*max|mean_ref|``
            (the absolute floor is tied to the output scale because std -> 0 in-distribution).
            ``precision='fp32'`` is the tensor-core split kernel (csrc/mlp_tcx.cu) wherever the model
            is eligible and the CUDA-core path otherwise; ``'fp32_ffma'`` forces the CUDA-core path.
            Both are held to the same 1e-5.
bf16 mode : stated tolerance (``tests.util.bf16_check``): mean and std within ``1e-2 * scale`` with
            ``scale = max|ref_mean| + max|ref_std|`` (the size of one member's output; measured worst
            case 2.3e-3 .. 4.3e-3), and the std within ``5e-2`` of its own scale (measured <= 2.2e-2).
            bf16 rounds weights and activations to 8 bits once per layer.  Measured errors are printed.
"""
import os

import numpy as np
import pytest
import torch

from nnueehcs_b200 import ops
from nnueehcs_b200.model_builder import (DeltaUQMLPModelBuilder, EnsembleModelBuilder,
                                         MCDropoutModelBuilder, build_network)
from oracle import uq_oracle
from tests.util import (assert_close_ref, bf16_check, delta_arch, golden_arch, golden_masks,
                        injected_to_masks, load_golden, masks_to_injected, mc_arch_with_dropout,
                        nets_from_golden, randomise_bn, wide_arch)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
RTOL32 = 1e-5


FP32_MODES = ["fp32", "fp32_ffma"]


# ---- ensemble -----------------------------------------------------------------------------------

@pytest.mark.parametrize("precision", FP32_MODES)
@pytest.mark.parametrize("name", ["ensemble_small.npz", "ensemble_bn.npz", "ensemble_binomial.npz"])
def test_ensemble_fp32_matches_reference_golden(name, precision):
    g = load_golden(name)
    k = int(g["k"])
    packed = ops.PackedModel(nets_from_golden(g, k), DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    mean, std = packed.forward(x, "ensemble", total_members=k, precision=precision)
    assert mean.shape == g["mean"].shape
    assert_close_ref(mean, g["mean"], RTOL32, what=f"{name} mean")
    assert_close_ref(std, g["std"], RTOL32, scale_ref=g["mean"], what=f"{name} std")


@pytest.mark.parametrize("name", ["ensemble_bn.npz", "ensemble_binomial.npz"])
def test_ensemble_bf16_within_stated_tolerance(name):
    g = load_golden(name)
    k = int(g["k"])
    packed = ops.PackedModel(nets_from_golden(g, k), DEV)
    assert packed.supports_bf16, packed.bf16_reason
    x = torch.from_numpy(g["x"]).to(DEV)
    mean, std = packed.forward(x, "ensemble", total_members=k, precision="bf16")
    bf16_check(mean, std, g["mean"], g["std"], name)


def test_bf16_rejects_unsupported_shapes_loudly():
    g = load_golden("ensemble_small.npz")  # 25-wide layers, 5 outputs
    packed = ops.PackedModel(nets_from_golden(g, int(g["k"])), DEV)
    assert not packed.supports_bf16
    x = torch.from_numpy(g["x"]).to(DEV)
    with pytest.raises(ValueError, match="bf16 path unavailable"):
        packed.forward(x, "ensemble", total_members=int(g["k"]), precision="bf16")


def test_ensemble_wrapper_drop_in():
    """Model built by the builder mirror from the YAML-style description, golden weights loaded,
    ``model(x, return_ue=True)`` as ``evaluation.py:135`` calls it."""
    g = load_golden("ensemble_binomial.npz")
    k = int(g["k"])
    model = EnsembleModelBuilder(golden_arch(g), {"num_models": k}).build()
    for net, ref in zip(model.models, nets_from_golden(g, k)):
        net.load_state_dict(ref.state_dict())
    model.to(DEV)
    model.eval()
    x = torch.from_numpy(g["x"]).to(DEV)
    with torch.no_grad():
        mean, std = model(x, return_ue=True)
        only_mean = model(x)
    assert_close_ref(mean, g["mean"], RTOL32, what="wrapper mean")
    assert_close_ref(std, g["std"], RTOL32, scale_ref=g["mean"], what="wrapper std")
    assert torch.equal(only_mean, mean)
    # packed-weight cache: reused while weights are untouched, rebuilt after an in-place update
    cache = model.__dict__["_uq_cache"][1]
    model(x)
    assert model.__dict__["_uq_cache"][1] is cache
    with torch.no_grad():
        model.models[0][-1].bias.add_(1.0)
    mean2 = model(x)
    assert model.__dict__["_uq_cache"][1] is not cache
    assert_close_ref(mean2, g["mean"] + 1.0 / k, RTOL32, what="wrapper mean after update")
    # float64 datasets (bo.py:396 casts models with .to(dset.dtype)): outputs keep x's dtype
    m64, s64 = model(x.double(), return_ue=True)
    assert m64.dtype == torch.float64 and s64.dtype == torch.float64


# ---- MC dropout -----------------------------------------------------------------------------------

@pytest.mark.parametrize("precision", FP32_MODES)
@pytest.mark.parametrize("name", ["mcdropout_small.npz", "mcdropout_binomial.npz"])
def test_mc_dropout_fp32_injected_reference_masks(name, precision):
    g = load_golden(name)
    p, passes = float(g["p"]), int(g["passes"])
    net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    packed = ops.PackedModel([net], DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    inj = masks_to_injected(golden_masks(g)).to(DEV)
    mean, std = packed.forward(x, "mc_dropout", total_members=passes, precision=precision,
                               dropout_p=p, masks=inj)
    assert_close_ref(mean, g["mean"], RTOL32, what=f"{name} mean")
    assert_close_ref(std, g["std"], RTOL32, scale_ref=g["mean"], what=f"{name} std")


@pytest.mark.parametrize("precision", FP32_MODES)
@pytest.mark.parametrize("name", ["mcdropout_small.npz", "mcdropout_binomial.npz"])
def test_mc_dropout_off_fp32(name, precision):
    g = load_golden(name)
    p, passes = float(g["p"]), int(g["passes"])
    net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    packed = ops.PackedModel([net], DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    mean, std = packed.forward(x, "mc_dropout", total_members=passes, precision=precision,
                               dropout_p=p, dropout_active=False)
    assert_close_ref(mean, g["mean_off"], RTOL32, what=f"{name} mean_off")
    assert float(std.abs().max()) <= RTOL32 * float(np.abs(g["mean_off"]).max())


def test_mc_dropout_bf16_injected_masks():
    g = load_golden("mcdropout_binomial.npz")
    p, passes = float(g["p"]), int(g["passes"])
    net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    packed = ops.PackedModel([net], DEV)
    assert packed.supports_bf16, packed.bf16_reason
    x = torch.from_numpy(g["x"]).to(DEV)
    inj = masks_to_injected(golden_masks(g)).to(DEV)
    mean, std = packed.forward(x, "mc_dropout", total_members=passes, precision="bf16",
                               dropout_p=p, masks=inj)
    bf16_check(mean, std, g["mean"], g["std"], "mcdropout_binomial injected")
    mean0, std0 = packed.forward(x, "mc_dropout", total_members=passes, precision="bf16",
                                 dropout_p=p, dropout_active=False)
    bf16_check(mean0, std0, g["mean_off"], g["std_off"], "mcdropout_binomial off")


@pytest.mark.parametrize("precision", ["fp32", "fp32_ffma", "bf16"])
def test_mc_dropout_native_philox_replays_exactly_through_oracle(precision):
    """Native masks are a pure function of (seed, pass, layer, sample, feature): export them with
    uq_philox_keep_masks, replay through the CPU oracle, compare -- exact parity for the native
    RNG path, not just statistics."""
    g = load_golden("mcdropout_binomial.npz")
    p, passes, seed = 0.2, 12, 20261018
    net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    packed = ops.PackedModel([net], DEV)
    x_cpu = torch.from_numpy(g["x"])[:150]
    x = x_cpu.to(DEV)
    mean, std = packed.forward(x, "mc_dropout", total_members=passes, precision=precision,
                               dropout_p=p, seed=seed)
    flat = ops.philox_keep_masks(x.shape[0], packed.dropout_widths, passes, p, seed, 0, DEV)
    masks = injected_to_masks(flat.cpu(), x.shape[0], packed.dropout_widths, passes)
    ref_mean, ref_std = uq_oracle.mc_dropout_forward(net, x_cpu, passes, p, masks=masks)
    if precision != "bf16":
        assert_close_ref(mean, ref_mean, RTOL32, what="philox replay mean")
        assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what="philox replay std")
    else:
        bf16_check(mean, std, ref_mean, ref_std, "philox replay")
    # and feeding the exported masks back as injected masks gives the identical result
    mean_i, std_i = packed.forward(x, "mc_dropout", total_members=passes, precision=precision,
                                   dropout_p=p, masks=flat)
    assert torch.equal(mean, mean_i) and torch.equal(std, std_i)


def test_philox_mask_statistics():
    p, n, w, passes = 0.2, 4096, 128, 16
    flat = ops.philox_keep_masks(n, [w], passes, p, 7, 0, DEV).float()
    m = flat.reshape(passes, n, w)
    total = m.numel()
    keep = float(m.mean())
    # 99.99 % two-sided binomial interval
    half = 3.9 * (p * (1 - p) / total) ** 0.5
    assert abs(keep - (1 - p)) < half + 2 ** -16
    # different passes / features are uncorrelated: pairwise agreement ~ keep^2 + (1-keep)^2
    agree = float((m[0] == m[1]).float().mean())
    assert abs(agree - (keep ** 2 + (1 - keep) ** 2)) < 5e-3
    other = ops.philox_keep_masks(n, [w], passes, p, 8, 0, DEV).float()
    assert float((other == flat).float().mean()) < 0.75
    again = ops.philox_keep_masks(n, [w], passes, p, 7, 0, DEV).float()
    assert torch.equal(again, flat)


def test_mc_dropout_wrapper_statistical_parity_with_reference_rng():
    """Native Philox vs the reference's torch-RNG run (golden): per-sample mean inside
    +-5 standard errors, pooled std ratio inside the chi-square band (stated CI)."""
    g = load_golden("mcdropout_binomial.npz")
    p = float(g["p"])
    passes = 512
    model = MCDropoutModelBuilder(golden_arch(g), {"num_samples": passes,
                                                   "dropout_percent": p}).build()
    ref_net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    model.model.load_state_dict(ref_net.state_dict())
    model.to(DEV)
    model.eval()
    x_cpu = torch.from_numpy(g["x"])[:64]
    torch.manual_seed(3)
    with torch.no_grad():
        mean, std = model(x_cpu.to(DEV), return_ue=True)
    torch.manual_seed(11)
    ref_mean, ref_std = uq_oracle.mc_dropout_forward(ref_net, x_cpu, passes, p)  # torch RNG
    se = (ref_std ** 2 / passes + std.cpu() ** 2 / passes).sqrt().clamp_min(1e-7)
    z = ((mean.cpu() - ref_mean).abs() / se).max()
    assert float(z) < 5.0, f"mean z-score {float(z)}"
    ratio = (std.cpu() / ref_std)
    assert float(ratio.min()) > 0.8 and float(ratio.max()) < 1.25, (ratio.min(), ratio.max())
    # nn.Module.eval semantics (dropout off) -> identical passes, std == 0
    torch.nn.Module.eval(model)
    with torch.no_grad():
        m_off, s_off = model(x_cpu.to(DEV), return_ue=True)
    assert float(s_off.abs().max()) <= 1e-5 * float(m_off.abs().max())


# ---- Delta-UQ (parity unpinned: oracle restatement only) -------------------------------------------

@pytest.mark.parametrize("precision", ["fp32", "fp32_ffma", "bf16"])
def test_delta_uq_matches_restatement(precision):
    g = load_golden("deltauq_small.npz")
    k = int(g["k"])
    net = nets_from_golden(g, 1, arch=delta_arch(golden_arch(g)))[0]
    packed = ops.PackedModel([net], DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    anchors = torch.from_numpy(g["anchors"]).to(DEV)
    mean, std = packed.forward(x, "delta_uq", total_members=k, precision=precision,
                               anchors=anchors)
    ref_mean, ref_std = uq_oracle.delta_uq_forward(net, torch.from_numpy(g["x"]),
                                                   torch.from_numpy(g["anchors"]), k)
    if precision != "bf16":
        assert_close_ref(mean, ref_mean, RTOL32, what="delta mean")
        assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what="delta std")
    else:
        bf16_check(mean, std, ref_mean, ref_std, "delta_uq")


def test_delta_uq_wrapper():
    g = load_golden("deltauq_small.npz")
    k = int(g["k"])
    model = DeltaUQMLPModelBuilder(golden_arch(g), {"estimator": "std", "num_anchors": k,
                                                    "anchored_batch_size": int(g["chunk"])}).build()
    ref_net = nets_from_golden(g, 1, arch=delta_arch(golden_arch(g)))[0]
    model.net.load_state_dict(ref_net.state_dict())
    model.anchors = torch.from_numpy(g["anchors"])
    model.to(DEV)
    model.eval()
    with torch.no_grad():
        mean, std = model(torch.from_numpy(g["x"]).to(DEV), return_ue=True)
    assert_close_ref(mean, g["mean"], 2e-5, what="delta wrapper mean")
    assert_close_ref(std, g["std"], 2e-5, scale_ref=g["mean"], what="delta wrapper std")


# ---- PAGER (SURVEY 8f row 2; anchoring parity-unpinned like Delta-UQ) -----------------------------------

@pytest.mark.parametrize("precision", ["fp32", "fp32_ffma", "bf16"])
def test_pager_matches_reference_class_golden(precision):
    """uq_forward(mode=UQ_MODE_PAGER) against the outputs of the reference's own PAGERMLP
    (tests/golden/make_golden_pager.py) and the oracle restatement."""
    g = load_golden("pager_small.npz")
    k = int(g["k"])
    net = nets_from_golden(g, 1, arch=delta_arch(golden_arch(g)))[0]
    packed = ops.PackedModel([net], DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    anchors = torch.from_numpy(g["anchors"]).to(DEV)
    ys = torch.from_numpy(g["anchors_y"]).to(DEV)
    mu, std = packed.forward(x, "delta_uq", total_members=k, precision=precision, anchors=anchors)
    pmean, conformal = packed.forward(x, "pager", total_members=k, precision=precision,
                                      anchors=anchors, targets=ys)
    _, score = packed.forward(x, "pager", total_members=k, precision=precision, anchors=anchors,
                              targets=ys, score_floor=std)
    assert torch.equal(score, torch.maximum(conformal, std))   # the fused floor IS torch.maximum
    ref_pred, ref_score, ref_conf = uq_oracle.pager_forward(
        net, torch.from_numpy(g["x"]), torch.from_numpy(g["anchors"]),
        torch.from_numpy(g["anchors_y"]), k)
    if precision != "bf16":
        assert_close_ref(mu, g["pred"], 2e-5, what="pager pred")
        assert_close_ref(conformal, g["conformal"], RTOL32, scale_ref=g["pred"], what="conformal")
        assert_close_ref(score, g["score"], 2e-5, scale_ref=g["pred"], what="pager score")
        assert_close_ref(conformal, ref_conf, RTOL32, scale_ref=ref_pred, what="conformal/oracle")
    else:
        scale = float(np.abs(g["pred"]).max())
        e_c = float((conformal.cpu() - ref_conf).abs().max())
        e_s = float((score.cpu() - ref_score).abs().max())
        print(f"[bf16 pager] max|conformal err| = {e_c:.3e}, max|score err| = {e_s:.3e}, "
              f"scale {scale:.3e}")
        assert e_c <= 3e-2 * scale and e_s <= 6e-2 * scale
    # the by-product mean is the mean over anchors of the swapped-role predictions
    with torch.no_grad():
        cols = [uq_oracle.sequential_forward(
            net, uq_oracle.anchored_input(torch.from_numpy(g["anchors"])[j:j + 1].expand(
                g["x"].shape[0], -1), torch.from_numpy(g["x"]))) for j in range(k)]
    ref_pmean = torch.stack(cols).mean(0)
    tol = RTOL32 if precision != "bf16" else 3e-2
    assert float((pmean.cpu() - ref_pmean).abs().max()) <= tol * float(ref_pmean.abs().max()) + 1e-7


def test_pager_wrapper_drop_in_and_errors():
    from nnueehcs_b200.model_builder import PAGERModelBuilder
    g = load_golden("pager_small.npz")
    k = int(g["k"])
    model = PAGERModelBuilder(golden_arch(g), {"estimator": "std", "num_anchors": k}).build()
    ref_net = nets_from_golden(g, 1, arch=delta_arch(golden_arch(g)))[0]
    model.net.load_state_dict(ref_net.state_dict())
    model.anchors = torch.from_numpy(g["anchors"])
    model.to(DEV)
    model.eval()
    x = torch.from_numpy(g["x"]).to(DEV)
    with torch.no_grad():
        with pytest.raises(ValueError, match="anchors_Y not set"):
            model(x, return_ue=True)
        model.anchors_Y = torch.from_numpy(g["anchors_y"]).to(DEV)
        pred, score = model(x, return_ue=True)
        only = model(x)
        conf = model._score_samples(x, model.anchors, model.anchors_Y)
    assert_close_ref(pred, g["pred"], 2e-5, what="pager wrapper pred")
    assert_close_ref(only, g["pred_only"], 2e-5, what="pager wrapper pred (no ue)")
    assert_close_ref(score, g["score"], 2e-5, scale_ref=g["pred"], what="pager wrapper score")
    assert_close_ref(conf, g["conformal"], 2e-5, scale_ref=g["pred"], what="pager wrapper conformal")
    packed = model._packed([model.net], x.device)
    with pytest.raises(ValueError, match="anchors_Y"):
        packed.forward(x, "pager", total_members=k, anchors=model.anchors)
    with pytest.raises(ValueError, match="only apply to mode='pager'"):
        packed.forward(x, "delta_uq", total_members=k, anchors=model.anchors,
                       targets=model.anchors_Y)
    with pytest.raises(ValueError, match="max over anchors"):
        packed.forward(x, "pager", total_members=k, anchors=model.anchors,
                       targets=model.anchors_Y, output="moments")


def test_pager_narrow_and_wide_kernels_bf16():
    """The same fold runs in all three fused kernels: 6x128 (four-slot kernel), 3x256 (pair
    kernel), 2x768 (wide kernel); ragged N, K = 7 anchors."""
    for width, depth, n in ((128, 6, 1000), (256, 3, 700), (768, 2, 300)):
        torch.manual_seed(width)
        net = build_network(delta_arch(wide_arch(5, width, depth, 1))).eval()
        x, anchors, ys = torch.rand(n, 5), torch.rand(7, 5), torch.rand(7, 1) * 0.2
        packed = ops.PackedModel([net], DEV)
        assert packed.supports_bf16
        _, conf = packed.forward(x.to(DEV), "pager", total_members=7, precision="bf16",
                                 anchors=anchors.to(DEV), targets=ys.to(DEV))
        _, conf32 = packed.forward(x.to(DEV), "pager", total_members=7, precision="fp32",
                                   anchors=anchors.to(DEV), targets=ys.to(DEV))
        ref_pred, _, ref_conf = uq_oracle.pager_forward(net, x, anchors, ys, 7)
        scale = float(ref_pred.abs().max()) + float(ys.abs().max())
        assert_close_ref(conf32, ref_conf, RTOL32, scale_ref=ref_pred, what=f"pager fp32 {width}")
        err = float((conf.cpu() - ref_conf).abs().max())
        print(f"[bf16 pager {depth}x{width}] max|conformal err| = {err:.3e} of scale {scale:.3e}")
        assert err <= 3e-2 * scale


# ---- K-axis shards, tails, errors ---------------------------------------------------------------------

@pytest.mark.parametrize("precision", ["fp32", "fp32_ffma", "bf16"])
def test_member_shards_merge_to_the_full_result(precision):
    g = load_golden("ensemble_binomial.npz")
    k = int(g["k"])
    packed = ops.PackedModel(nets_from_golden(g, k), DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    full_mean, full_std = packed.forward(x, "ensemble", total_members=k, precision=precision)
    means, m2s, counts = [], [], []
    for b, c in ((0, 1), (1, 2)):
        m, s = packed.forward(x, "ensemble", total_members=k, precision=precision,
                              member_begin=b, member_count=c, output="moments")
        means.append(m), m2s.append(s), counts.append(c)
    mean, std = ops.moments_merge(torch.stack(means), torch.stack(m2s), counts)
    tol = 1e-6 if precision == "fp32_ffma" else 2e-6
    assert_close_ref(mean, full_mean, tol, what="sharded mean")
    assert_close_ref(std, full_std, 10 * tol, scale_ref=full_mean, what="sharded std")


@pytest.mark.parametrize("precision", ["fp32", "fp32_ffma", "bf16"])
@pytest.mark.parametrize("n", [1, 63, 65, 127, 129, 1000])
def test_ragged_sample_counts(precision, n):
    g = load_golden("ensemble_bn.npz")
    k = int(g["k"])
    nets = nets_from_golden(g, k)
    packed = ops.PackedModel(nets, DEV)
    x_cpu = torch.rand(n, 5, generator=torch.Generator().manual_seed(n))
    mean, std = packed.forward(x_cpu.to(DEV), "ensemble", total_members=k, precision=precision)
    ref_mean, ref_std = uq_oracle.ensemble_forward(nets, x_cpu)
    if precision != "bf16":
        assert_close_ref(mean, ref_mean, RTOL32, what=f"n={n} mean")
        assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what=f"n={n} std")
    else:
        bf16_check(mean, std, ref_mean, ref_std, f"n={n}")


def test_many_passes_few_samples_uses_member_splits():
    """cfg-1 shape (few sample tiles, many passes): the bf16 kernel also splits the pass axis over
    CTAs and Chan-merges the partial moments; result must equal the fp32 path on the same masks."""
    g = load_golden("mcdropout_binomial.npz")
    p, passes, seed = 0.2, 96, 5
    net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    packed = ops.PackedModel([net], DEV)
    x = torch.rand(300, 5, generator=torch.Generator().manual_seed(1)).to(DEV)
    m32, s32 = packed.forward(x, "mc_dropout", total_members=passes, precision="fp32",
                              dropout_p=p, seed=seed)
    m16, s16 = packed.forward(x, "mc_dropout", total_members=passes, precision="bf16",
                              dropout_p=p, seed=seed)
    bf16_check(m16, s16, m32.cpu(), s32.cpu(), "member splits")


def test_single_member_std_is_nan_like_torch():
    g = load_golden("ensemble_bn.npz")
    nets = nets_from_golden(g, 1)
    packed = ops.PackedModel(nets, DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    for precision in ("fp32", "fp32_ffma", "bf16"):
        mean, std = packed.forward(x, "ensemble", total_members=1, precision=precision)
        assert torch.isnan(std).all() and torch.isfinite(mean).all()


def test_argument_errors():
    g = load_golden("ensemble_bn.npz")
    k = int(g["k"])
    packed = ops.PackedModel(nets_from_golden(g, k), DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    with pytest.raises(ValueError, match="total_members"):
        packed.forward(x, "ensemble", total_members=k + 1)
    with pytest.raises(ValueError, match="single packed network"):
        packed.forward(x, "mc_dropout", total_members=4, dropout_p=0.1)
    with pytest.raises(ValueError, match=r"x must be \[n, 5\]"):
        packed.forward(x[:, :3], "ensemble", total_members=k)
    with pytest.raises(ValueError, match="no rows"):
        packed.forward(x[:0], "ensemble", total_members=k)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        packed.forward(x.cpu(), "ensemble", total_members=k)
    with pytest.raises(ValueError, match="unknown precision"):
        packed.forward(x, "ensemble", total_members=k, precision="fp8")
    with pytest.raises(ValueError, match="different architecture"):
        ops.PackedModel([build_network([{"Linear": {"args": [5, 8]}}]),
                         build_network([{"Linear": {"args": [5, 9]}}])], DEV)


def test_host_buffer_entry_point():
    g = load_golden("ensemble_binomial.npz")
    k = int(g["k"])
    packed = ops.PackedModel(nets_from_golden(g, k), DEV)
    x = torch.from_numpy(g["x"]).contiguous().pin_memory()
    out0 = torch.empty(g["mean"].shape, dtype=torch.float32).pin_memory()
    out1 = torch.empty_like(out0).pin_memory()
    packed.forward_host(x, out0, out1, "ensemble", total_members=k, precision="fp32")
    assert_close_ref(out0, g["mean"], RTOL32, what="host mean")
    assert_close_ref(out1, g["std"], RTOL32, scale_ref=g["mean"], what="host std")


# ---- wide nets (hidden width 768 / 1024): the 64-rows-per-CTA pair kernel, mlp_tc3.cu -----------

@pytest.mark.parametrize("width,n_hidden,k,n,d_out", [(1024, 2, 3, 300, 1), (1024, 7, 2, 129, 1),
                                                      (768, 3, 2, 64, 3)])
def test_wide_ensemble_bf16(width, n_hidden, k, n, d_out):
    nets = []
    for i in range(k):
        torch.manual_seed(42 + i)
        net = build_network(wide_arch(5, width, n_hidden, d_out)).eval()
        randomise_bn(net, 1 + i)
        nets.append(net)
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(0))
    packed = ops.PackedModel(nets, DEV)
    assert packed.supports_bf16, packed.bf16_reason
    mean, std = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16")
    ref_mean, ref_std = uq_oracle.ensemble_forward(nets, x)
    bf16_check(mean, std, ref_mean, ref_std, f"wide ensemble {width}x{n_hidden}")
    # K-axis shards of the same forward merge to the same result
    m_a, s_a = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16",
                              member_begin=0, member_count=1, output="moments")
    m_b, s_b = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16",
                              member_begin=1, member_count=k - 1, output="moments")
    mm, ss = ops.moments_merge(torch.stack([m_a, m_b]), torch.stack([s_a, s_b]), [1, k - 1])
    assert float((mm - mean).abs().max()) <= 1e-5 * float(mean.abs().max())
    assert float((ss - std).abs().max()) <= 1e-4 * float(std.abs().max()) + 1e-6


def test_wide_mc_dropout_philox_replays_through_oracle():
    p, passes, seed, n = 0.2, 6, 77, 150
    torch.manual_seed(42)
    net = build_network(mc_arch_with_dropout(wide_arch(5, 1024, 3, 1), p)).eval()
    randomise_bn(net, 1)
    packed = ops.PackedModel([net], DEV)
    assert packed.supports_bf16, packed.bf16_reason
    x_cpu = torch.rand(n, 5, generator=torch.Generator().manual_seed(5))
    mean, std = packed.forward(x_cpu.to(DEV), "mc_dropout", total_members=passes, precision="bf16",
                               dropout_p=p, seed=seed)
    flat = ops.philox_keep_masks(n, packed.dropout_widths, passes, p, seed, 0, DEV)
    masks = injected_to_masks(flat.cpu(), n, packed.dropout_widths, passes)
    ref_mean, ref_std = uq_oracle.mc_dropout_forward(net, x_cpu, passes, p, masks=masks)
    bf16_check(mean, std, ref_mean, ref_std, "wide philox replay")
    mean_i, std_i = packed.forward(x_cpu.to(DEV), "mc_dropout", total_members=passes,
                                   precision="bf16", dropout_p=p, masks=flat)
    assert torch.equal(mean, mean_i) and torch.equal(std, std_i)
    # many passes over few samples: the member axis is split over CTA pairs and merged
    mean_s, std_s = packed.forward(x_cpu[:70].to(DEV), "mc_dropout", total_members=96,
                                   precision="bf16", dropout_p=p, dropout_active=False)
    # dropout off: 96 identical passes -> zero spread
    assert float(std_s.abs().max()) <= 1e-3 * float(mean_s.abs().max())


def test_wide_delta_uq_bf16():
    k, n = 4, 200
    torch.manual_seed(42)
    net = build_network(delta_arch(wide_arch(5, 768, 2, 1))).eval()
    randomise_bn(net, 1)
    packed = ops.PackedModel([net], DEV)
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(2))
    anchors = torch.rand(k, 5, generator=torch.Generator().manual_seed(3))
    mean, std = packed.forward(x.to(DEV), "delta_uq", total_members=k, precision="bf16",
                               anchors=anchors.to(DEV))
    ref_mean, ref_std = uq_oracle.delta_uq_forward(net, x, anchors, k)
    bf16_check(mean, std, ref_mean, ref_std, "wide delta_uq")


# ---- every kernel family at awkward sizes --------------------------------------------------------

@pytest.mark.parametrize("width,n_hidden,n,k", [
    (64, 2, 1, 2),        # narrow-net kernel (4 tile slots), a single row
    (64, 3, 1025, 3),     # one row into the second unit of 1024
    (128, 2, 2049, 2),
    (192, 2, 257, 2),     # pair kernel, one accumulator half, tile pair + 1 row
    (256, 3, 130, 4),
    (320, 2, 383, 2),     # two unequal accumulator halves (N = 160)
    (448, 2, 129, 2),
    (1024, 2, 1, 2),      # wide-net kernel (64 rows per CTA), a single row
    (1024, 2, 65, 3),
    (768, 2, 193, 2),
])
def test_bf16_kernels_at_ragged_sizes(width, n_hidden, n, k):
    nets = []
    for i in range(k):
        torch.manual_seed(100 + i)
        net = build_network(wide_arch(7, width, n_hidden, 1)).eval()
        randomise_bn(net, 50 + i)
        nets.append(net)
    x = torch.rand(n, 7, generator=torch.Generator().manual_seed(n))
    packed = ops.PackedModel(nets, DEV)
    assert packed.supports_bf16, packed.bf16_reason
    mean, std = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16")
    ref_mean, ref_std = uq_oracle.ensemble_forward(nets, x)
    bf16_check(mean, std, ref_mean, ref_std, f"ragged {width}x{n_hidden} n={n}")
    # the same rows inside a larger batch give bit-identical results (tiles are independent)
    xb = torch.cat([x, torch.rand(300, 7, generator=torch.Generator().manual_seed(1))])
    mean_b, std_b = packed.forward(xb.to(DEV), "ensemble", total_members=k, precision="bf16")
    assert torch.equal(mean_b[:n], mean) and torch.equal(std_b[:n], std)


def test_narrow_kernel_many_passes_member_splits():
    """MC dropout on the 6 x 128 surrogate with few samples and many passes: the member axis is
    split over CTA pairs (each pair runs 4 tile slots) and merged; dropout off -> zero spread and
    the same mean as a single pass."""
    g = load_golden("mcdropout_binomial.npz")
    p = float(g["p"])
    net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    packed = ops.PackedModel([net], DEV)
    x = torch.from_numpy(g["x"]).to(DEV)
    mean, std = packed.forward(x, "mc_dropout", total_members=256, precision="bf16", dropout_p=p,
                               dropout_active=False)
    one, _ = packed.forward(x, "mc_dropout", total_members=2, precision="bf16", dropout_p=p,
                            dropout_active=False)
    assert float((mean - one).abs().max()) <= 2e-6 * float(one.abs().max())
    assert float(std.abs().max()) <= 1e-5 * float(one.abs().max())
    # live dropout, native Philox: same seed -> same bits regardless of how passes are split
    a = packed.forward(x, "mc_dropout", total_members=64, precision="bf16", dropout_p=p, seed=5)
    lo = packed.forward(x, "mc_dropout", total_members=64, precision="bf16", dropout_p=p, seed=5,
                        member_begin=0, member_count=24, output="moments")
    hi = packed.forward(x, "mc_dropout", total_members=64, precision="bf16", dropout_p=p, seed=5,
                        member_begin=24, member_count=40, output="moments")
    mm, ss = ops.moments_merge(torch.stack([lo[0], hi[0]]), torch.stack([lo[1], hi[1]]), [24, 40])
    assert float((mm - a[0]).abs().max()) <= 1e-5 * float(a[0].abs().max())
    assert float((ss - a[1]).abs().max()) <= 1e-3 * float(a[1].abs().max())


def test_shard_objects_on_a_single_rank_nccl_group():
    """World-size-1 NCCL group: KShard and NShard degenerate to the plain forward (the N > 1 logic is
    covered by the gloo tests and by bench.py --gpus N / tools/dist_metrics_check.py on real GPUs)."""
    import socket
    import torch.distributed as dist
    from nnueehcs_b200.distributed import KShard, NShard
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=DEV)
    try:
        g = load_golden("ensemble_bn.npz")
        k = int(g["k"])
        model = EnsembleModelBuilder(golden_arch(g), {"num_models": k}).build()
        for m, ref in zip(model.models, nets_from_golden(g, k)):
            m.load_state_dict(ref.state_dict())
        model.to(DEV).eval()
        x = torch.from_numpy(g["x"]).to(DEV)
        with torch.no_grad():
            plain = model(x, return_ue=True)
            for shard in (KShard(), NShard()):
                model.uq_shard = shard
                got = model(x, return_ue=True)
                assert_close_ref(got[0], plain[0], 1e-6, what=type(shard).__name__ + " mean")
                assert_close_ref(got[1], plain[1], 1e-5, scale_ref=plain[0],
                                 what=type(shard).__name__ + " std")
        model.uq_shard = None
        assert_close_ref(plain[0], g["mean"], RTOL32, what="mean")
        # PAGER with the anchors on the K-shard path (conformal shards combine with a max)
        from nnueehcs_b200.model_builder import PAGERModelBuilder
        pg = load_golden("pager_small.npz")
        pk = int(pg["k"])
        pm = PAGERModelBuilder(golden_arch(pg), {"estimator": "std", "num_anchors": pk}).build()
        pm.net.load_state_dict(nets_from_golden(pg, 1, arch=delta_arch(golden_arch(pg)))[0].state_dict())
        pm.anchors = torch.from_numpy(pg["anchors"])
        pm.anchors_Y = torch.from_numpy(pg["anchors_y"])
        pm.to(DEV).eval()
        pm.uq_shard = KShard()
        with torch.no_grad():
            pred, score = pm(torch.from_numpy(pg["x"]).to(DEV), return_ue=True)
        assert_close_ref(pred, pg["pred"], 2e-5, what="sharded pager pred")
        assert_close_ref(score, pg["score"], 2e-5, scale_ref=pg["pred"], what="sharded pager score")
    finally:
        if created:
            dist.destroy_process_group()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_pager_multi_output_and_anchor_prefix(precision):
    """d_out = 3 (targets are indexed [anchor][output]; the multi-output epilogue of the pair
    kernel), more anchor rows stored than num_anchors uses, and a K-range call that covers only the
    last anchors (member_begin > 0: targets / per-anchor biases are indexed by the GLOBAL id)."""
    torch.manual_seed(3)
    net = build_network(delta_arch(wide_arch(4, 128, 3, 3))).eval()
    x, anchors, ys = torch.rand(500, 4), torch.rand(9, 4), torch.rand(9, 3) * 0.3
    k = 6
    packed = ops.PackedModel([net], DEV)
    _, conf = packed.forward(x.to(DEV), "pager", total_members=k, precision=precision,
                             anchors=anchors.to(DEV), targets=ys.to(DEV))
    with torch.no_grad():
        cols = [uq_oracle.sequential_forward(
            net, uq_oracle.anchored_input(anchors[j:j + 1].expand(x.shape[0], -1), x))
            for j in range(k)]
    p = torch.stack(cols)                                            # [K, N, 3]
    ref = (p - ys[:k].unsqueeze(1)).abs().max(dim=0)[0]
    tol = RTOL32 if precision == "fp32" else 3e-2
    scale = float(p.abs().max()) + float(ys.abs().max())
    assert float((conf.cpu() - ref).abs().max()) <= tol * scale
    # anchors [2, 6) only: max over the last four anchors
    _, tail = packed.forward(x.to(DEV), "pager", total_members=k, member_begin=2, member_count=4,
                             precision=precision, anchors=anchors.to(DEV), targets=ys.to(DEV))
    ref_tail = (p[2:] - ys[2:k].unsqueeze(1)).abs().max(dim=0)[0]
    assert float((tail.cpu() - ref_tail).abs().max()) <= tol * scale
    # ... so K-shards of the conformal score combine with an element-wise max
    _, head = packed.forward(x.to(DEV), "pager", total_members=k, member_begin=0, member_count=2,
                             precision=precision, anchors=anchors.to(DEV), targets=ys.to(DEV))
    assert torch.equal(torch.maximum(head, tail), conf)


# ---- fp32 parity mode on the tensor cores (csrc/mlp_tcx.cu): every width, awkward sizes ----------------

def test_fp32_runs_on_the_tensor_cores_where_eligible():
    g = load_golden("ensemble_binomial.npz")   # the reference's YAML architecture, 6 x 128
    packed = ops.PackedModel(nets_from_golden(g, int(g["k"])), DEV)
    assert packed.fp32_on_tensor_cores, packed.fp32_tc_reason
    g = load_golden("ensemble_small.npz")      # 25-wide layers: CUDA-core path, and it says why
    packed = ops.PackedModel(nets_from_golden(g, int(g["k"])), DEV)
    assert not packed.fp32_on_tensor_cores and "hidden" in packed.fp32_tc_reason
    torch.manual_seed(0)                       # 1024-wide: no room for two fp16 pieces of a tile
    packed = ops.PackedModel([build_network(wide_arch(5, 1024, 2, 1)).eval()], DEV)
    assert not packed.fp32_on_tensor_cores and "512" in packed.fp32_tc_reason
    torch.manual_seed(0)                       # 17 inputs: the layer-0 chunk holds at most 16
    packed = ops.PackedModel([build_network(wide_arch(17, 128, 2, 1)).eval()], DEV)
    assert not packed.fp32_on_tensor_cores and "16" in packed.fp32_tc_reason


@pytest.mark.parametrize("width,n_hidden,n,k,d_in,d_out", [
    (64, 2, 1, 2, 5, 1), (64, 3, 1025, 3, 7, 1), (128, 1, 300, 2, 5, 1), (128, 6, 2049, 2, 5, 1),
    (192, 2, 257, 2, 16, 1), (256, 3, 130, 4, 5, 3), (320, 2, 383, 2, 9, 1), (384, 2, 200, 2, 5, 8),
    (448, 2, 129, 2, 5, 1), (512, 3, 4097, 4, 5, 1), (512, 2, 65, 2, 12, 2),
    (128, 2, 259, 3, 16, 1),   # four-slot split kernel, layer 0 built in place (K0 = 64)
])
def test_fp32_split_kernel_all_widths(width, n_hidden, n, k, d_in, d_out):
    nets = []
    for i in range(k):
        torch.manual_seed(100 + i)
        net = build_network(wide_arch(d_in, width, n_hidden, d_out)).eval()
        randomise_bn(net, 50 + i)
        nets.append(net)
    # unnormalised inputs on purpose: the row scales must absorb them
    x = torch.rand(n, d_in, generator=torch.Generator().manual_seed(n)) * 37.0 - 11.0
    packed = ops.PackedModel(nets, DEV)
    assert packed.fp32_on_tensor_cores, packed.fp32_tc_reason
    mean, std = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="fp32")
    ref_mean, ref_std = uq_oracle.ensemble_forward(nets, x)
    assert_close_ref(mean, ref_mean, RTOL32, what=f"split {width}x{n_hidden} mean")
    assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what=f"split {width}x{n_hidden} std")
    # the same rows inside a larger batch give bit-identical results (tiles are independent)
    xb = torch.cat([x, torch.rand(300, d_in, generator=torch.Generator().manual_seed(1))])
    mean_b, std_b = packed.forward(xb.to(DEV), "ensemble", total_members=k, precision="fp32")
    assert torch.equal(mean_b[:n], mean) and torch.equal(std_b[:n], std)


@pytest.mark.parametrize("scale", [1e-6, 1.0, 3e4])
def test_fp32_split_kernel_is_scale_free(scale):
    """Activations far from 1 (tiny / huge weights and inputs): the power-of-two row and weight
    scales keep every fp16 piece in range, so the result tracks the reference at any magnitude."""
    torch.manual_seed(7)
    net = build_network(wide_arch(5, 256, 3, 1, bn=False)).eval()
    with torch.no_grad():
        net[0].weight.mul_(scale)
        net[0].bias.mul_(scale)
        net[-1].weight.mul_(1.0 / scale)
    x = torch.rand(500, 5, generator=torch.Generator().manual_seed(2))
    packed = ops.PackedModel([net, net], DEV)
    assert packed.fp32_on_tensor_cores
    mean, _ = packed.forward(x.to(DEV), "ensemble", total_members=2, precision="fp32")
    ref_mean, _ = uq_oracle.ensemble_forward([net, net], x)
    assert torch.isfinite(mean).all()
    assert_close_ref(mean, ref_mean, RTOL32, what=f"scale {scale} mean")


def test_dropout_before_the_final_linear():
    """A hand-built net with a Dropout between the last activation and the final Linear (the
    reference's builder never makes one, model_builder.py:257-262): its 1 / (1 - p) applies to the
    final dot product in every kernel."""
    p, passes, seed, n = 0.25, 10, 11, 200
    arch = mc_arch_with_dropout(wide_arch(5, 128, 3, 1), p)
    arch.insert(len(arch) - 1, {"Dropout": {"args": [p]}})
    torch.manual_seed(42)
    net = build_network(arch).eval()
    randomise_bn(net, 1)
    packed = ops.PackedModel([net], DEV)
    x_cpu = torch.rand(n, 5, generator=torch.Generator().manual_seed(5))
    flat = ops.philox_keep_masks(n, packed.dropout_widths, passes, p, seed, 0, DEV)
    masks = injected_to_masks(flat.cpu(), n, packed.dropout_widths, passes)
    ref_mean, ref_std = uq_oracle.mc_dropout_forward(net, x_cpu, passes, p, masks=masks)
    for precision in ("fp32", "fp32_ffma", "bf16"):
        mean, std = packed.forward(x_cpu.to(DEV), "mc_dropout", total_members=passes,
                                   precision=precision, dropout_p=p, seed=seed)
        if precision == "bf16":
            bf16_check(mean, std, ref_mean, ref_std, "dropout before final Linear")
        else:
            assert_close_ref(mean, ref_mean, RTOL32, what=f"{precision} mean")
            assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what=f"{precision} std")


# ---- the BASELINE.json shapes (the kernel instantiations bench.py times) --------------------------------

def _baseline_nets(d_in, width, n_hidden, k, d_out=1):
    nets = []
    for i in range(k):
        torch.manual_seed(42 + i)            # model_builder.py:229 seeds member i with 42 + i
        net = build_network(wide_arch(d_in, width, n_hidden, d_out)).eval()
        randomise_bn(net, 1 + i)
        nets.append(net)
    return nets


def test_baseline_config1_ensemble16x512():
    """BASELINE configs[1]: 16 members x (5 -> 512 -> 512 -> 512 -> 1), here on 40 960 + 37 samples:
    uq_mlp_tc2_kernel<512, 1, 2> (bf16: all 512 TMEM columns, 8 K chunks, minimum weight ring) and
    uq_mlp_tcx_kernel<512, 1> (fp32 split), through PackedModel.forward and through the wrapper."""
    k, n = 16, 40997
    nets = _baseline_nets(5, 512, 3, k)
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(0))
    ref_mean, ref_std = uq_oracle.ensemble_forward(nets, x)
    packed = ops.PackedModel(nets, DEV)
    assert packed.fp32_on_tensor_cores and packed.supports_bf16
    mean, std = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="fp32")
    assert_close_ref(mean, ref_mean, RTOL32, what="cfg1 fp32 mean")
    assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what="cfg1 fp32 std")
    mean, std = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16")
    bf16_check(mean, std, ref_mean, ref_std, "cfg1 bf16")
    model = EnsembleModelBuilder(wide_arch(5, 512, 3, 1), {"num_models": k}).build()
    for m, ref in zip(model.models, nets):
        m.load_state_dict(ref.state_dict())
    model.to(DEV).eval()
    with torch.no_grad():
        for precision in ("fp32", "bf16"):
            model.uq_precision = precision
            w_mean, w_std = model(x.to(DEV), return_ue=True)
            d_mean, d_std = packed.forward(x.to(DEV), "ensemble", total_members=k,
                                           precision=precision)
            assert torch.equal(w_mean, d_mean) and torch.equal(w_std, d_std)


def test_baseline_config2_deltauq_32_anchors_6x128():
    """BASELINE configs[2]: Delta-UQ, 32 anchors, the 6 x 128 binomial-options net: the four-slot
    kernel (bf16) and the split kernel (fp32) with per-anchor layer-0 biases.  Parity unpinned
    (oracle restatement), like every Delta-UQ check."""
    k, n = 32, 20011
    torch.manual_seed(42)
    net = build_network(delta_arch(wide_arch(5, 128, 6, 1))).eval()
    randomise_bn(net, 1)
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(0))
    anchors = torch.rand(k, 5, generator=torch.Generator().manual_seed(2))
    ref_mean, ref_std = uq_oracle.delta_uq_forward(net, x, anchors, k)
    packed = ops.PackedModel([net], DEV)
    assert packed.fp32_on_tensor_cores
    mean, std = packed.forward(x.to(DEV), "delta_uq", total_members=k, precision="fp32",
                               anchors=anchors.to(DEV))
    assert_close_ref(mean, ref_mean, RTOL32, what="cfg2 fp32 mean")
    assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what="cfg2 fp32 std")
    mean, std = packed.forward(x.to(DEV), "delta_uq", total_members=k, precision="bf16",
                               anchors=anchors.to(DEV))
    bf16_check(mean, std, ref_mean, ref_std, "cfg2 bf16")
    model = DeltaUQMLPModelBuilder(wide_arch(5, 128, 6, 1), {"estimator": "std", "num_anchors": k,
                                                              "anchored_batch_size": 4096}).build()
    model.net.load_state_dict(net.state_dict())
    model.anchors = anchors
    model.to(DEV).eval()
    with torch.no_grad():
        w_mean, w_std = model(x.to(DEV), return_ue=True)     # default precision: fp32
    assert_close_ref(w_mean, ref_mean, RTOL32, what="cfg2 wrapper mean")
    assert_close_ref(w_std, ref_std, RTOL32, scale_ref=ref_mean, what="cfg2 wrapper std")


def test_baseline_config3_mcdropout_8x1024_philox_replay():
    """BASELINE configs[3]'s net (8 Linear layers of width 1024, dropout before Linears 2..7, p = 0.2)
    with native Philox masks replayed exactly through the oracle: the wide kernel (bf16) and the
    CUDA-core path (fp32; width 1024 has no split kernel)."""
    p, passes, seed, n = 0.2, 8, 20261018, 1500
    torch.manual_seed(42)
    net = build_network(mc_arch_with_dropout(wide_arch(5, 1024, 7, 1), p)).eval()
    randomise_bn(net, 1)
    packed = ops.PackedModel([net], DEV)
    x_cpu = torch.rand(n, 5, generator=torch.Generator().manual_seed(5))
    flat = ops.philox_keep_masks(n, packed.dropout_widths, passes, p, seed, 0, DEV)
    masks = injected_to_masks(flat.cpu(), n, packed.dropout_widths, passes)
    ref_mean, ref_std = uq_oracle.mc_dropout_forward(net, x_cpu, passes, p, masks=masks)
    mean, std = packed.forward(x_cpu.to(DEV), "mc_dropout", total_members=passes, precision="fp32",
                               dropout_p=p, seed=seed)
    assert_close_ref(mean, ref_mean, RTOL32, what="cfg3 fp32 mean")
    assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what="cfg3 fp32 std")
    mean, std = packed.forward(x_cpu.to(DEV), "mc_dropout", total_members=passes, precision="bf16",
                               dropout_p=p, seed=seed)
    bf16_check(mean, std, ref_mean, ref_std, "cfg3 bf16")
    model = MCDropoutModelBuilder(wide_arch(5, 1024, 7, 1), {"num_samples": passes,
                                                              "dropout_percent": p}).build()
    model.model.load_state_dict(net.state_dict())
    model.to(DEV).eval()
    model.uq_precision = "bf16"
    torch.manual_seed(3)
    with torch.no_grad():
        w_mean, w_std = model(x_cpu.to(DEV), return_ue=True)
    assert torch.isfinite(w_mean).all() and float(w_std.min()) > 0.0


@pytest.mark.parametrize("precision", ["fp32", "fp32_ffma", "bf16"])
def test_native_masks_do_not_depend_on_sample_sharding(precision):
    """A rank that runs rows [b, e) of the batch with row_base = b draws the bits of the whole-batch
    call (Philox counters use the GLOBAL row), so an N-sharded MC-dropout run reproduces the
    single-GPU result bit for bit."""
    g = load_golden("mcdropout_binomial.npz")
    p, passes, seed = 0.2, 10, 99
    net = nets_from_golden(g, 1, arch=mc_arch_with_dropout(golden_arch(g), p))[0]
    packed = ops.PackedModel([net], DEV)
    x = torch.rand(333, 5, generator=torch.Generator().manual_seed(4)).to(DEV)
    full = packed.forward(x, "mc_dropout", total_members=passes, precision=precision, dropout_p=p,
                          seed=seed)
    for b, e in ((0, 100), (100, 333), (64, 65)):
        part = packed.forward(x[b:e], "mc_dropout", total_members=passes, precision=precision,
                              dropout_p=p, seed=seed, row_base=b)
        assert torch.equal(part[0], full[0][b:e]) and torch.equal(part[1], full[1][b:e])
    other = packed.forward(x[100:333], "mc_dropout", total_members=passes, precision=precision,
                           dropout_p=p, seed=seed)          # row_base 0: different rows' bits
    assert not torch.equal(other[1], full[1][100:333])


def test_wide_ensemble_split_major_member_groups():
    """A wide ensemble whose weights exceed the L2 (24 members x 2.1 MB) is cut into member groups
    that mlp_tc3.cu walks split-major (all clusters on the same group at a time) and Chan-merges;
    the result must equal the oracle like any other bf16 forward."""
    k, n = 24, 9600
    nets = _baseline_nets(5, 1024, 2, k)
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(0))
    packed = ops.PackedModel(nets, DEV)
    mean, std = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16")
    ref_mean, ref_std = uq_oracle.ensemble_forward(nets, x)
    bf16_check(mean, std, ref_mean, ref_std, "split-major wide ensemble")
    # the same forward as two K-shards (no member groups inside a moments call) merges to it
    a = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16", member_begin=0,
                       member_count=10, output="moments")
    b = packed.forward(x.to(DEV), "ensemble", total_members=k, precision="bf16", member_begin=10,
                       member_count=14, output="moments")
    mm, ss = ops.moments_merge(torch.stack([a[0], b[0]]), torch.stack([a[1], b[1]]), [10, 14])
    assert float((mm - mean).abs().max()) <= 1e-5 * float(mean.abs().max())
    assert float((ss - std).abs().max()) <= 1e-4 * float(std.abs().max())


# ---- bias in the MMA (default) against the epilogue-bias variant ---------------------------------

def _both_bias_variants(call):
    """Run ``call()`` with UQ_TC_BIAS_MMA=0 (the epilogue adds the bias) and =1 (the tensor core
    accumulates it from a bias stage: csrc/mlp_tc2.cu, mlp_tc3.cu, mlp_tc4.cu); the launchers read
    the variable on every call."""
    old = os.environ.get("UQ_TC_BIAS_MMA")
    out = {}
    try:
        for flag in ("0", "1"):
            os.environ["UQ_TC_BIAS_MMA"] = flag
            mean, std = call()
            torch.cuda.synchronize()
            out[flag] = (mean.clone(), std.clone())
    finally:
        if old is None:
            os.environ.pop("UQ_TC_BIAS_MMA", None)
        else:
            os.environ["UQ_TC_BIAS_MMA"] = old
    return out


def _large_bias_nets(width, n_hidden, k, d_in, bias_scale=20.0):
    nets = []
    for i in range(k):
        torch.manual_seed(7 + i)
        net = build_network(wide_arch(d_in, width, n_hidden, 1, bn=False)).eval()
        with torch.no_grad():
            for m in net:
                if isinstance(m, torch.nn.Linear):   # a dropped bias piece is an O(1) error
                    m.bias.mul_(bias_scale).add_(0.37 * bias_scale * torch.randn_like(m.bias))
        nets.append(net)
    return nets


@pytest.mark.parametrize("width,n_hidden,k,n", [
    (64, 3, 2, 1025), (128, 6, 5, 3000),        # narrow-net kernel
    (192, 2, 3, 257), (320, 2, 2, 383), (512, 3, 4, 5000),   # pair kernel (one / two unequal / two halves)
    (768, 3, 2, 193), (1024, 2, 3, 300),        # wide-net kernel
])
def test_bias_in_mma_matches_epilogue_bias_ensemble(width, n_hidden, k, n):
    nets = _large_bias_nets(width, n_hidden, k, 5)
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(n))
    packed = ops.PackedModel(nets, DEV)
    ref_mean, ref_std = uq_oracle.ensemble_forward(nets, x)
    out = _both_bias_variants(lambda: packed.forward(x.to(DEV), "ensemble", total_members=k,
                                                     precision="bf16"))
    for flag, (mean, std) in out.items():
        bf16_check(mean, std, ref_mean, ref_std, f"bias variant {flag}, {width}x{n_hidden}")
    # the two variants differ by accumulation order only
    scale = float(torch.as_tensor(ref_mean).abs().max() + torch.as_tensor(ref_std).abs().max())
    assert float((out["1"][0] - out["0"][0]).abs().max()) <= 2e-3 * scale


@pytest.mark.parametrize("width,n_hidden,k,n", [(128, 6, 32, 2011), (256, 3, 7, 1500), (1024, 3, 5, 333)])
def test_bias_in_mma_per_anchor_layer0_stages(width, n_hidden, k, n):
    """Delta-UQ: the per-anchor layer-0 bias reaches the kernel as bias stages built per call."""
    net = _large_bias_nets(width, n_hidden, 1, 10)[0]
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(n))
    anchors = torch.rand(k, 5, generator=torch.Generator().manual_seed(2)) * 3.0
    packed = ops.PackedModel([net], DEV)
    ref_mean, ref_std = uq_oracle.delta_uq_forward(net, x, anchors, k)
    out = _both_bias_variants(lambda: packed.forward(x.to(DEV), "delta_uq", total_members=k,
                                                     precision="bf16", anchors=anchors.to(DEV)))
    # the large biases put the outputs at ~10 with a spread over anchors of ~0.03: bf16 rounding of
    # the last hidden activations alone is ~10 % of that spread (either variant), so the std is held
    # to the output scale (1e-2, measured 3e-4) and to half of its own scale only
    for flag, (mean, std) in out.items():
        bf16_check(mean, std, ref_mean, ref_std, f"bias variant {flag}, delta-uq {width}x{n_hidden}",
                    tol_std=0.5)
    scale = float(torch.as_tensor(ref_mean).abs().max() + torch.as_tensor(ref_std).abs().max())
    assert float((out["1"][0] - out["0"][0]).abs().max()) <= 2e-3 * scale
    assert float((out["1"][1] - out["0"][1]).abs().max()) <= 2e-3 * scale
    # and a member shard [2, k) of the same call reads the same per-anchor stages
    os.environ.pop("UQ_TC_BIAS_MMA", None)
    m_a, q_a = packed.forward(x.to(DEV), "delta_uq", total_members=k, precision="bf16",
                              anchors=anchors.to(DEV), member_begin=2, member_count=k - 2,
                              output="moments")
    ref_a = uq_oracle.delta_uq_forward(net, x, anchors[2:], k - 2)
    bf16_check(m_a, torch.sqrt(q_a / (k - 3)), ref_a[0], ref_a[1], "anchor shard", tol_std=0.5)


@pytest.mark.parametrize("width,n_hidden,passes,n,final_drop", [
    (128, 6, 9, 700, False), (64, 3, 5, 300, True), (512, 3, 5, 400, True), (1024, 4, 5, 300, False)])
def test_bias_in_mma_with_live_dropout_philox_replay(width, n_hidden, passes, n, final_drop):
    """With the bias in the MMA the activations are stored with their dropout's 1/(1-p); native
    masks replayed through the oracle, including a Dropout right before the final Linear."""
    pdrop, seed = 0.2, 1234 + width
    torch.manual_seed(3)
    layers, fan = [], 5
    for i in range(n_hidden):
        layers += [torch.nn.Linear(fan, width), torch.nn.ReLU()]
        if 0 < i < n_hidden - 1 or (final_drop and i == n_hidden - 1):
            layers.append(torch.nn.Dropout(pdrop))
        fan = width
    layers.append(torch.nn.Linear(fan, 1))
    net = torch.nn.Sequential(*layers).eval()
    with torch.no_grad():
        for m in net:
            if isinstance(m, torch.nn.Linear):
                m.bias.mul_(5.0).add_(1.8 * torch.randn_like(m.bias))
    x = torch.rand(n, 5, generator=torch.Generator().manual_seed(n))
    packed = ops.PackedModel([net], DEV)
    flat = ops.philox_keep_masks(n, packed.dropout_widths, passes, pdrop, seed, 0, DEV)
    masks = injected_to_masks(flat.cpu(), n, packed.dropout_widths, passes)
    ref_mean, ref_std = uq_oracle.mc_dropout_forward(net, x, passes, pdrop, masks=masks)
    out = _both_bias_variants(lambda: packed.forward(x.to(DEV), "mc_dropout", total_members=passes,
                                                     precision="bf16", dropout_p=pdrop, seed=seed))
    for flag, (mean, std) in out.items():
        bf16_check(mean, std, ref_mean, ref_std, f"bias variant {flag}, mc-dropout {width}x{n_hidden}")
