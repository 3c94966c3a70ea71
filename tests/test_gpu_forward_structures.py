"""The fused forward on every layer structure ``extract.split_blocks`` accepts (B200 only:
``pytest -m gpu``).

``split_blocks`` takes any stack of blocks ``Linear [-> BatchNorm1d] [-> ReLU] [-> Dropout]`` and the
kernels branch on each layer's flags: ``TcParams::relu_mask`` / ``dropout_mask`` / ``last_relu`` in
the tensor-core families, ``Epilogue::relu`` and ``linear_small_out_kernel`` on the CUDA-core
(FFMA) path, a NULL Linear bias packed as zeros, a BatchNorm without ``weight`` / ``bias`` folded
by ``bn_fold_kernel``.  The other GPU tests only run equal-width ``Linear -> [BN] -> ReLU`` stacks
with a plain final Linear; this file runs the rest:

- hidden layers without ReLU, in every pattern over three layers, with and without BatchNorm;
- a ReLU after the final Linear, its bias centred so that about half of the outputs are clamped;
- Linears without bias, and ensemble members that differ below the structure signature;
- BatchNorm with ``affine=False``, on one layer only, with a non-default ``eps``, and with a
  spread of ~16 decades in its scale;
- Dropout without ReLU, on one middle layer, and right before the final Linear;
- 16 hidden layers (``MAX_MMA_LAYERS``), 17, and none;
- the structures only the FFMA path takes: unequal or unsupported hidden widths, d_out 9,
  BatchNorm or Dropout after the final Linear.

Each case computes ONE float64 reference per mode (``copy.deepcopy(net).double()``, float64 inputs
/ anchors / targets, ``oracle.uq_oracle``; native Philox masks exported and replayed) and checks
every precision the model supports against it: ``bf16`` (``bf16_check``), ``fp32`` and
``fp32_ffma`` (``assert_close_ref`` at 1e-5).  Where bf16 or the fp32 split kernels refuse a
structure, the refusal is asserted by name.  Every forward runs under ``torch.profiler`` and must
launch exactly the kernels ``tests.util.expected_kernels`` restates from the dispatch; the file
prints every instantiation it ran.

The hidden Linears are rescaled to unit gain (x sqrt(6) before a ReLU, x sqrt(3) otherwise), so
that every layer of a deep stack still moves the output instead of leaving only the last bias.
"""
import copy
import math

import pytest
import torch

from nnueehcs_b200 import ops
from nnueehcs_b200.model_builder import MCDropoutModelBuilder, build_network
from oracle import uq_oracle
from tests.util import (RTOL32, assert_close_ref, assert_live_spread, check, injected_to_masks,
                        pager_reference, run, tc_refusal, tcx_refusal)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
N = 259                   # two 128-row tiles + 3 rows; four 64-row tiles + 3 rows
D_IN = 5                  # network input 5, or 10 for Delta-UQ / PAGER: both fp32 kernel families
P_DROP, PASSES, ENSEMBLE_K, ANCHORS = 0.2, 5, 3, 5

# (hidden width, d_out): tc4 / tcx4; tc2 with two unequal accumulator halves and the bias in the
# MMA / tcx; tc2 / tcx with the epilogue bias (DOUT = 8); tc3 with fp32 on FFMA
FAMILIES = [(64, 1), (320, 1), (128, 3), (1024, 1)]
FAM_IDS = [f"h{h}-o{o}" for h, o in FAMILIES]


# bf16 bounds, bf16_check's ``(tol, tol_std)``: the error as a share of max|mean| + max|std|, and the
# std's error as a share of max|std|.  The bf16 error of these networks is the rounding of the
# hidden activations and folded hidden weights to bf16 (layer 0 is split into bf16 pieces and the
# final Linear runs in fp32, so they add next to nothing).  Their hidden Linears have unit gain, so
# every layer carries its rounding on to the output at full size, where the suite's other networks
# shrink it; the error grows with depth.  A float64 CPU emulation of exactly those roundings
# reproduces the kernel's worst errors to four digits: 1.12e-2 of max|output| for the 64-wide
# hidden1 network with dropout off (three hidden layers), and (1.774e-2, 5.270e-2) for the 16-layer
# 64-wide ensemble.  Measured worst on a B200 (1000 W): (1.14e-2, 1.36e-2) at <= 3 hidden layers,
# (4.41e-2, 5.57e-2) at 16.  The bounds are ~2-3x that.  The deliberate kernel bugs the file was
# checked with fail their bf16 cases by 4.5e-2 .. 0.46 of scale.  The fp32 modes are held to 1e-5
# at every depth.
BF16_TOL = {3: (3e-2, 5e-2), 16: (0.1, 0.15)}


def bf16_tol(packed):
    return BF16_TOL[3] if packed.n_layers - 1 <= 3 else BF16_TOL[16]


@pytest.fixture(scope="module")
def seen():
    """Every forward kernel instantiation this file ran, printed at the end."""
    names = set()
    yield names
    print("\n[forward structures] kernel instantiations run:\n  " + "\n  ".join(sorted(names)))


# ---- networks --------------------------------------------------------------------------------------

def _per(v, l):
    return v[l] if isinstance(v, (tuple, list)) else v


def arch_of(d_in, widths, d_out, *, bn=True, relu=True, drop=(), bias=True, bn_kw=None,
            last_relu=False, last_bn=False, last_drop=False):
    """``Linear(d_in, widths[0]) [-> BN] [-> ReLU] [-> Dropout] ... -> Linear(widths[-1], d_out)``.
    ``bn`` / ``relu`` / ``bn_kw``: one value for every hidden layer or one per hidden layer;
    ``bias``: one value or one per Linear (the final one included); ``drop``: the hidden layers
    followed by a Dropout.  ``last_*`` append those modules after the final Linear."""
    arch, prev = [], d_in
    for l, w in enumerate(widths):
        arch.append({"Linear": {"args": [prev, w], "bias": _per(bias, l)}})
        if _per(bn, l):
            arch.append({"BatchNorm1d": {"args": [w], **(_per(bn_kw, l) or {})}})
        if _per(relu, l):
            arch.append({"ReLU": {}})
        if l in drop:
            arch.append({"Dropout": {"args": [P_DROP]}})
        prev = w
    arch.append({"Linear": {"args": [prev, d_out], "bias": _per(bias, len(widths))}})
    if last_bn:
        arch.append({"BatchNorm1d": {"args": [d_out], **(bn_kw or {})}})
    if last_relu:
        arch.append({"ReLU": {}})
    if last_drop:
        arch.append({"Dropout": {"args": [P_DROP]}})
    return arch


def init_net(net, seed, bn_spread=False):
    """Unit-gain hidden Linears; eval BatchNorm statistics (and affine parameters) that matter.
    ``bn_spread``: running_var log-uniform over 1e-4 .. 1e4, gamma of random sign with magnitude
    log-uniform over 1e-2 .. 1e2."""
    gen = torch.Generator().manual_seed(seed)
    mods = list(net)
    with torch.no_grad():
        for i, m in enumerate(mods):
            if isinstance(m, torch.nn.Linear) and any(isinstance(n, torch.nn.Linear)
                                                      for n in mods[i + 1:]):
                nxt = next((n for n in mods[i + 1:] if not isinstance(n, torch.nn.BatchNorm1d)),
                           None)
                m.weight.mul_(math.sqrt(6.0 if isinstance(nxt, torch.nn.ReLU) else 3.0))
            elif isinstance(m, torch.nn.BatchNorm1d):
                f = m.num_features
                m.running_mean.copy_(torch.randn(f, generator=gen) * 0.1)
                if bn_spread:
                    m.running_var.copy_(10.0 ** (torch.rand(f, generator=gen) * 8 - 4))
                else:
                    m.running_var.copy_(torch.rand(f, generator=gen) + 0.5)
                if m.affine:
                    sign = torch.where(torch.rand(f, generator=gen) < 0.5, -1.0, 1.0)
                    if bn_spread:
                        m.weight.copy_(sign * 10.0 ** (torch.rand(f, generator=gen) * 4 - 2))
                    else:
                        m.weight.copy_(torch.rand(f, generator=gen) + 0.5)
                    m.bias.copy_(torch.randn(f, generator=gen) * 0.1)
    return net


def make_nets(arch, k, seed, bn_spread=False):
    nets = []
    for i in range(k):
        torch.manual_seed(seed + i)
        nets.append(init_net(build_network(arch).eval(), seed + 100 + i, bn_spread))
    return nets


def f64(net):
    return copy.deepcopy(net).double()


def rows(d, seed, n=N):
    """Inputs in [0, 1) (the min-max scaled range of the reference's data_utils)."""
    return torch.rand(n, d, generator=torch.Generator().manual_seed(seed))


def center_last_relu(net, inputs):
    """Shift the bias of the Linear before the final ReLU by the median of its outputs over
    ``inputs`` (one tensor per way the net is called), so that about half of them are clamped."""
    lin = [m for m in net if isinstance(m, torch.nn.Linear)][-1]
    with torch.no_grad():
        pre = torch.cat([net[:-1](x) for x in inputs])
        lin.bias.sub_(pre.median(dim=0).values)
        out = torch.cat([net(x) for x in inputs])
    clamped = float((out == 0).double().mean())
    assert 0.3 <= clamped <= 0.7, f"final ReLU clamps {clamped:.2f} of the outputs"


# ---- one mode, every precision ---------------------------------------------------------------------

def precisions_of(packed, what):
    """The precisions a model runs in; a bf16 / fp32-split refusal must give the dispatch's reason."""
    sig = packed.signature
    why, why_x = tc_refusal(sig), tcx_refusal(sig)
    assert packed.supports_bf16 == (why is None), f"{what}: {packed.bf16_reason}"
    assert packed.fp32_on_tensor_cores == (why_x is None), f"{what}: {packed.fp32_tc_reason}"
    if why is not None:
        assert why in packed.bf16_reason, f"{what}: bf16 refused with {packed.bf16_reason!r}"
    if why_x is not None:
        assert why_x in packed.fp32_tc_reason, f"{what}: {packed.fp32_tc_reason!r}"
    return (["bf16"] if why is None else []) + ["fp32", "fp32_ffma"]


def bf16_refused(packed, x, mode, **kw):
    why = tc_refusal(packed.signature)
    if why is not None:
        with pytest.raises(ValueError, match=why.split(" (")[0]):
            packed.forward(x, mode, precision="bf16", **kw)


def check_ensemble(seen, what, nets, x):
    nets64, x64 = [f64(n) for n in nets], x.double()
    ref = uq_oracle.ensemble_forward(nets64, x64)
    ref_tail = uq_oracle.ensemble_forward(nets64[1:], x64)
    assert_live_spread(*ref, what)
    packed = ops.PackedModel(nets, DEV)
    xd = x.to(DEV)
    kw = dict(total_members=len(nets))
    tol = bf16_tol(packed)
    bf16_refused(packed, xd, "ensemble", **kw)
    for precision in precisions_of(packed, what):
        mean, std = run(seen, packed, precision, what, xd, "ensemble", **kw)
        check(precision, mean, std, *ref, what, tol)
        m, m2 = run(seen, packed, precision, what, xd, "ensemble", member_begin=1,
                    output="moments", **kw)
        check(precision, m, torch.sqrt(m2.double().clamp_min(0) / (len(nets) - 2)), *ref_tail,
              what + " moments", tol)


def check_mc(seen, what, net, x, seed):
    """Live dropout on the native Philox stream and on the same masks injected, then dropout off."""
    packed = ops.PackedModel([net], DEV)
    assert packed.dropout_widths, what
    flat = ops.philox_keep_masks(N, packed.dropout_widths, PASSES, P_DROP, seed, 0, DEV)
    masks = injected_to_masks(flat.cpu(), N, packed.dropout_widths, PASSES)
    net64, x64 = f64(net), x.double()
    ref = uq_oracle.mc_dropout_forward(net64, x64, PASSES, P_DROP, masks=masks)
    ref_off = uq_oracle.mc_dropout_forward(net64, x64, PASSES, P_DROP, dropout_active=False)
    assert_live_spread(*ref, what)
    xd = x.to(DEV)
    kw = dict(total_members=PASSES, dropout_p=P_DROP, seed=seed)
    tol = bf16_tol(packed)
    bf16_refused(packed, xd, "mc_dropout", **kw)
    for precision in precisions_of(packed, what):
        mean, std = run(seen, packed, precision, what, xd, "mc_dropout", True, **kw)
        check(precision, mean, std, *ref, what + " philox", tol)
        mean, std = run(seen, packed, precision, what, xd, "mc_dropout", True, masks=flat, **kw)
        check(precision, mean, std, *ref, what + " masks", tol)
        mean, std = run(seen, packed, precision, what, xd, "mc_dropout", dropout_active=False,
                        **kw)
        check(precision, mean, std, ref_off[0], torch.zeros_like(ref_off[0]), what + " off", tol)


def check_anchored(seen, what, net, x, anchors, ys):
    """Delta-UQ and PAGER (anchor_first, the public deltauq channel order)."""
    net64, x64, a64 = f64(net), x.double(), anchors.double()
    ref = uq_oracle.delta_uq_forward(net64, x64, a64, ANCHORS, anchor_first=True)
    ref_pmean, ref_conf = pager_reference(net64, x64, a64, ys.double(), True)
    assert_live_spread(*ref, what)
    packed = ops.PackedModel([net], DEV, anchor_first=True)
    xd, ad, yd = x.to(DEV), anchors.to(DEV), ys.to(DEV)
    bf16_refused(packed, xd, "delta_uq", total_members=ANCHORS, anchors=ad)
    scale = float(ref_pmean.abs().max()) + float(ys.abs().max())
    tol = bf16_tol(packed)
    for precision in precisions_of(packed, what):
        mean, std = run(seen, packed, precision, what, xd, "delta_uq", total_members=ANCHORS,
                        anchors=ad)
        check(precision, mean, std, *ref, what + " delta", tol)
        pmean, conf = run(seen, packed, precision, what, xd, "pager", total_members=ANCHORS,
                          anchors=ad, targets=yd)
        e_p = float((pmean.double().cpu() - ref_pmean).abs().max())
        e_c = float((conf.double().cpu() - ref_conf).abs().max())
        print(f"[{precision} {what} pager] max|mean err| = {e_p:.3e}, max|conformal err| = "
              f"{e_c:.3e}, scale {scale:.3e}")
        if precision == "bf16":   # the bf16 PAGER bound of test_gpu_forward_layouts
            assert e_p <= max(3e-2, tol[0]) * scale and e_c <= max(3e-2, tol[0]) * scale, what
        else:
            assert_close_ref(pmean, ref_pmean, RTOL32, what=f"{what} pager mean")
            assert_close_ref(conf, ref_conf, RTOL32, scale_ref=ref_pmean, what=f"{what} conformal")


def check_structure(seen, what, arch, seed, *, ensemble=True, mc=None, anchored=True,
                    bn_spread=False, last_relu=False):
    """``arch`` (a network of D_IN inputs) in every mode it allows: a K = 3 ensemble, MC dropout
    when it holds a Dropout, and Delta-UQ / PAGER on the same structure with 2 * D_IN inputs."""
    x = rows(D_IN, seed)
    if ensemble:
        nets = make_nets(arch, ENSEMBLE_K, seed, bn_spread)
        if last_relu:
            for net in nets:
                center_last_relu(net, [x])
        check_ensemble(seen, f"ensemble {what}", nets, x)
    has_drop = any("Dropout" in e for e in arch)
    if has_drop if mc is None else mc:
        net = make_nets(arch, 1, seed + 10, bn_spread)[0]
        if last_relu:
            center_last_relu(net, [x])
        check_mc(seen, f"mc {what}", net, x, seed)
    if anchored:
        darch = copy.deepcopy(arch)
        darch[0]["Linear"]["args"][0] *= 2
        net = make_nets(darch, 1, seed + 20, bn_spread)[0]
        anchors = rows(D_IN, seed + 1, n=ANCHORS)
        if last_relu:
            center_last_relu(net, [uq_oracle.anchored_input(anchors[j:j + 1].expand(N, -1), x,
                                                            True) for j in range(ANCHORS)])
        d_out = arch_out(arch)
        ys = torch.rand(ANCHORS, d_out, generator=torch.Generator().manual_seed(seed + 2)) * 0.3
        check_anchored(seen, f"anchored {what}", net, x, anchors, ys)


def arch_out(arch):
    return [e for e in arch if "Linear" in e][-1]["Linear"]["args"][1]


# ---- 1. hidden layers without ReLU -------------------------------------------------------------------

RELU_PATTERNS = [(False, False, False), (True, False, True), (False, True, False)]


@pytest.mark.parametrize("bn", [True, False], ids=["bn", "nobn"])
@pytest.mark.parametrize("relu", RELU_PATTERNS, ids=["FFF", "TFT", "FTF"])
@pytest.mark.parametrize("width,d_out", FAMILIES, ids=FAM_IDS)
def test_hidden_relu_patterns(seen, width, d_out, relu, bn):
    """The RELU = false drain steps (a bf16 store without the ReLU clamp), hidden and last hidden,
    and Epilogue::relu = 0 on the FFMA path."""
    what = f"relu={''.join('TF'[not r] for r in relu)} bn={bn} {width}/{d_out}"
    arch = arch_of(D_IN, [width] * 3, d_out, bn=bn, relu=relu)
    check_structure(seen, what, arch, 11000 + width + d_out)


# ---- 2. ReLU after the final Linear ------------------------------------------------------------------

@pytest.mark.parametrize("width,d_out", FAMILIES + [(1024, 3), (320, 3)],
                         ids=FAM_IDS + ["h1024-o3", "h320-o3"])
def test_last_relu(seen, width, d_out):
    """``TcParams::last_relu`` and linear_small_out_kernel's ``relu``; the final bias is centred
    so that about half of every member's outputs are clamped (a dropped clamp changes the mean by
    a sizeable part of its scale).  MC dropout on hidden layer 0 runs the MC = true variants."""
    arch = arch_of(D_IN, [width] * 2, d_out, drop=(0,), last_relu=True)
    check_structure(seen, f"last relu {width}/{d_out}", arch, 12000 + width + d_out,
                    last_relu=True)


# ---- 3. Linear without bias --------------------------------------------------------------------------

@pytest.mark.parametrize("bn", [True, False], ids=["bn", "nobn"])
@pytest.mark.parametrize("which", ["all", "layer0"])
@pytest.mark.parametrize("width,d_out", FAMILIES, ids=FAM_IDS)
def test_linear_without_bias(seen, width, d_out, which, bn):
    """A NULL Linear bias is packed as zeros (api.cu); layer 0 without bias under Delta-UQ / PAGER
    goes through delta_bias_kernel's folded bias."""
    bias = False if which == "all" else (False, True, True)
    arch = arch_of(D_IN, [width] * 2, d_out, bn=bn, bias=bias)
    check_structure(seen, f"no bias {which} bn={bn} {width}/{d_out}", arch,
                    13000 + width + d_out)


# ---- 4. BatchNorm variants ---------------------------------------------------------------------------

BN_VARIANTS = {
    "affine_false": dict(bn_kw={"affine": False}),
    "one_layer": dict(bn=(False, True, False)),
    "eps": dict(bn_kw={"eps": 0.1}),
    "spread": dict(),
}


@pytest.mark.parametrize("variant", list(BN_VARIANTS))
@pytest.mark.parametrize("width,d_out", FAMILIES, ids=FAM_IDS)
def test_batchnorm_variants(seen, width, d_out, variant):
    """``affine=False`` (bn_fold_kernel with NULL gamma / beta), BatchNorm on the middle layer
    only, ``eps`` = 0.1, and ``spread``: running_var log-uniform over 1e-4 .. 1e4 and gamma of
    random sign over 1e-2 .. 1e2, so that the folded row scales alpha = gamma / sqrt(var + eps)
    of one layer span ~1e-4 .. 1e4.

    The spread case targets the fp32 split kernels, which scale each (member, layer) by ONE
    power of two taken from the layer's largest folded weight (layer_stats_kernel): a row ~1e8
    below the maximum keeps few bits in its fp16 pieces (the ``h2`` piece goes subnormal).  What
    the test measures is the error of the network OUTPUT against the suite's 1e-5 bound, whose
    absolute floor is 1e-5 of the output scale: a small row's lost bits count by the share of
    the output that row carries."""
    kw = dict(BN_VARIANTS[variant])
    arch = arch_of(D_IN, [width] * 3, d_out, **kw)
    check_structure(seen, f"bn {variant} {width}/{d_out}", arch, 14000 + width + d_out,
                    bn_spread=variant == "spread")


# ---- 5. Dropout off the usual positions --------------------------------------------------------------

DROPOUT_PATTERNS = {
    "linear_bn_dropout": dict(relu=False, drop=(0, 1, 2)),
    "linear_dropout": dict(relu=False, bn=False, drop=(0, 1, 2)),
    "hidden1": dict(drop=(1,)),
    "hidden0_2": dict(drop=(0, 2)),
}


@pytest.mark.parametrize("pattern", list(DROPOUT_PATTERNS))
@pytest.mark.parametrize("width,d_out", FAMILIES, ids=FAM_IDS)
def test_dropout_positions(seen, width, d_out, pattern):
    """Dropout without a ReLU before it, on the middle layer alone (the Philox layer ordinal is the
    Dropout's, not the Linear's), and right before the final Linear (final_dropout_scale).  At
    d_out 1 the bias rides in the MMA and the activations carry 1/(1-p); at d_out 3 the next
    layer's epilogue owes it."""
    arch = arch_of(D_IN, [width] * 3, d_out, **DROPOUT_PATTERNS[pattern])
    check_structure(seen, f"dropout {pattern} {width}/{d_out}", arch, 15000 + width + d_out,
                    anchored=False)


# ---- 6. depth ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("width", [64, 128, 512, 1024])
def test_depth_16_hidden_layers(seen, width):
    """MAX_MMA_LAYERS hidden layers: every bf16 family width, and fp32 on the split kernels at
    64 / 128 / 512 (1024 runs on FFMA).  MC dropout on every hidden layer walks all 16 Philox
    layer ordinals and mask blocks."""
    arch = arch_of(D_IN, [width] * 16, 1, drop=tuple(range(16)))
    check_structure(seen, f"depth 16 {width}", arch, 16000 + width)


def test_depth_17_hidden_layers(seen):
    """One layer more than MAX_MMA_LAYERS: bf16 refuses with "too many layers", fp32 runs on FFMA."""
    arch = arch_of(D_IN, [128] * 17, 1, drop=tuple(range(17)))
    assert tc_refusal(structure_of(arch)) == "too many layers"
    check_structure(seen, "depth 17 128", arch, 16500)


@pytest.mark.parametrize("d_out", [1, 3])
def test_single_linear(seen, d_out):
    """No hidden Linear: bf16 refuses with "needs at least one hidden Linear"; both fp32 modes
    run it on linear_small_out_kernel, and with a live Dropout after it on sgemm_tn_kernel."""
    check_structure(seen, f"single linear d_out={d_out}", arch_of(D_IN, [], d_out), 17000 + d_out)
    check_structure(seen, f"single linear + dropout d_out={d_out}",
                    arch_of(D_IN, [], d_out, last_drop=True), 17100 + d_out, anchored=False)


# ---- 7. structures only the FFMA path takes ----------------------------------------------------------

FFMA_ONLY = {
    "5-192-96-1": dict(widths=[192, 96], d_out=1),
    "5-100-37-3": dict(widths=[100, 37], d_out=3),
    "width96": dict(widths=[96, 96], d_out=1),
    "width1536": dict(widths=[1536, 1536], d_out=1),
    "dout9": dict(widths=[128, 128], d_out=9),
    "bn_after_last": dict(widths=[128, 128], d_out=3, last_bn=True),
    "dropout_after_last": dict(widths=[128, 128], d_out=1, last_drop=True),
}


@pytest.mark.parametrize("case", list(FFMA_ONLY))
def test_ffma_only_structures(seen, case):
    """bf16 and the fp32 split kernels refuse these by name (precisions_of); fp32 and fp32_ffma
    match the reference on sgemm_tn_kernel / linear_small_out_kernel.  A Dropout on hidden layer 0
    adds the MC modes; after the final Linear, its masks are d_out wide."""
    spec = dict(FFMA_ONLY[case])
    arch = arch_of(D_IN, spec.pop("widths"), spec.pop("d_out"), drop=(0,), **spec)
    assert tc_refusal(structure_of(arch)) is not None, case
    check_structure(seen, case, arch, 18000 + len(case))


def structure_of(arch):
    from nnueehcs_b200.extract import split_blocks, structure_signature
    return structure_signature(split_blocks(build_network(arch)))


# ---- 8. ensemble members that differ below the structure signature -----------------------------------

@pytest.mark.parametrize("width,d_out", FAMILIES, ids=FAM_IDS)
def test_members_differ_below_signature(seen, width, d_out):
    """Member 0 as built; member 1 without the layer-0 and final Linear biases; member 2 with
    ``affine=False`` BatchNorms.  The structure signature is the same, so they pack as one
    ensemble; each member's missing parameters must be packed as its own zeros / ones."""
    archs = [arch_of(D_IN, [width] * 2, d_out),
             arch_of(D_IN, [width] * 2, d_out, bias=(False, True, False)),
             arch_of(D_IN, [width] * 2, d_out, bn_kw={"affine": False})]
    nets = [make_nets(a, 1, 19000 + width + d_out + 7 * i)[0] for i, a in enumerate(archs)]
    assert len({structure_of(a) for a in archs}) == 1
    check_ensemble(seen, f"members differ {width}/{d_out}", nets, rows(D_IN, 19000 + width))


# ---- the MC-dropout wrapper and per-module Dropout state ---------------------------------------------

def test_mc_wrapper_dropout_state(seen):
    """MCDropoutModel.forward passes ONE dropout_p and ONE live flag to the fused op; the reference
    calls ``self.model(x)``, which honours every Dropout's own ``p`` and train / eval state.  The
    wrapper matches the reference when all Dropouts agree (live after ``eval()``, or all put in
    eval mode) and raises a ValueError naming the module when one differs."""
    arch = arch_of(D_IN, [128] * 3, 1, bn=False)
    model = MCDropoutModelBuilder(arch, {"num_samples": PASSES, "dropout_percent": P_DROP}).build()
    init_net(model.model, 20000)
    model.eval()
    x = rows(D_IN, 20001)
    widths = ops.PackedModel([model.model.to(DEV)], DEV).dropout_widths
    assert len(widths) == 2
    flat = ops.philox_keep_masks(N, widths, PASSES, P_DROP, 20002, 0, DEV)
    masks = injected_to_masks(flat.cpu(), N, widths, PASSES)
    net64 = f64(model.model).cpu()
    ref = uq_oracle.mc_dropout_forward(net64, x.double(), PASSES, P_DROP, masks=masks)
    model.inject_masks(flat)
    with torch.no_grad():
        mean, std = model(x.to(DEV), return_ue=True)
    check("fp32", mean, std, *ref, "wrapper mc live")

    drops = [(i, m) for i, m in enumerate(model.model) if isinstance(m, torch.nn.Dropout)]
    idx, d1 = drops[1]
    d1.eval()
    with pytest.raises(ValueError, match=f"Dropout '{idx}'"):
        model(x.to(DEV))
    d1.train()
    d1.p = 0.5
    with pytest.raises(ValueError, match=f"Dropout '{idx}'"):
        model(x.to(DEV))
    d1.p = P_DROP
    for _, m in drops:
        m.eval()
    model.inject_masks(None)
    ref_off = uq_oracle.mc_dropout_forward(net64, x.double(), PASSES, P_DROP,
                                           dropout_active=False)
    with torch.no_grad():
        mean, std = model(x.to(DEV), return_ue=True)
    check("fp32", mean, std, ref_off[0], torch.zeros_like(ref_off[0]), "wrapper mc all eval")
