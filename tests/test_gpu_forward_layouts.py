"""The fused forward at every layer-0 input layout, output count and anchor order (B200 only:
``pytest -m gpu``).

Each case builds its networks, computes ONE float64 reference (``copy.deepcopy(net).double()``,
float64 inputs / anchors / targets, the dtype-generic ``oracle.uq_oracle``; native Philox masks are
exported and replayed) and checks every precision against it in the same body.  Every forward also
runs under ``torch.profiler``: the kernel instantiations it launched must be the ones
``tests.util.expected_kernels`` restates from the dispatch code, so that no case silently stops
covering its kernel when the dispatch changes.

Layer 0 of the bf16 kernels packs ``[x_hi | x_lo | x_hi] . [w_hi | w_hi | w_lo]`` into one K <= 64
chunk.  The split factor ``s`` is 3 for d_in <= 21, 2 for 22 .. 32 (``w_hi`` only) and 1 for
33 .. 64 (inputs rounded to 8 bits); the row goes through a shared-memory stash when K0 <= 32
(d_in <= 10 at s = 3) and is built in place in chunk 0 otherwise.  The fp32 split kernels take at
most 16 network inputs; wider inputs run on the CUDA-core (FFMA) path.

Tolerances are the suite's own: ``assert_close_ref`` at 1e-5 for fp32 (absolute floor tied to the
mean's scale), ``bf16_check`` for bf16, and for the bf16-exact one-layer nets of
``test_layer0_input_bits_bf16`` a bound per ``s`` set at ~4x the measured worst case.
"""
import copy

import pytest
import torch

from nnueehcs_b200 import ops
from nnueehcs_b200.model_builder import (DeltaUQMLPModelBuilder, EnsembleModelBuilder,
                                         build_network)
from oracle import uq_oracle
from tests.util import (RTOL32, assert_close_ref, assert_live_spread, bf16_check, check,
                        delta_arch, injected_to_masks, mc_arch_with_dropout, pager_reference,
                        randomise_bn, run, wide_arch)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
N = 259                   # two 128-row tiles + 3 rows; four 64-row tiles + 3 rows
WIDTHS = [128, 320, 1024]
P_DROP, PASSES, ENSEMBLE_K, ANCHORS = 0.2, 5, 3, 5


# ---- dispatch restated -----------------------------------------------------------------------------

def split_factor(d_in):
    s = 3
    while s > 1 and s * d_in > 64:
        s -= 1
    return s


@pytest.fixture(scope="module")
def seen():
    """Every forward kernel instantiation this file ran, printed at the end."""
    names = set()
    yield names
    print("\n[forward layouts] kernel instantiations run:\n  " + "\n  ".join(sorted(names)))


def check_moments(precision, mean, m2, count, ref_mean, ref_std, what):
    """``output='moments'`` of ``count`` members against the float64 (mean, std) of that range."""
    check(precision, mean, torch.sqrt(m2.double().clamp_min(0) / (count - 1)), ref_mean, ref_std,
          what + " moments")


def make_nets(arch, k, seed, bn=True):
    nets = []
    for i in range(k):
        torch.manual_seed(seed + i)
        net = build_network(arch).eval()
        if bn:
            randomise_bn(net, seed + 100 + i)
        nets.append(net)
    return nets


def f64(nets):
    return [copy.deepcopy(n).double() for n in nets]


def rows(d, seed, n=N, offset=0.0):
    """Inputs in [0, 1) (the min-max scaled range of the reference's data_utils), plus ``offset``."""
    return torch.rand(n, d, generator=torch.Generator().manual_seed(seed)) + offset


# ---- reference computations (float64) ------------------------------------------------------------

def ensemble_case(d_in, width, d_out, seed):
    nets = make_nets(wide_arch(d_in, width, 2, d_out), ENSEMBLE_K, seed)
    x = rows(d_in, seed)
    nets64, x64 = f64(nets), x.double()
    ref = uq_oracle.ensemble_forward(nets64, x64)
    ref_tail = uq_oracle.ensemble_forward(nets64[1:], x64)
    return ops.PackedModel(nets, DEV), x, ref, ref_tail


def mc_case(d_in, width, d_out, seed):
    net = make_nets(mc_arch_with_dropout(wide_arch(d_in, width, 2, d_out), P_DROP), 1, seed)[0]
    x = rows(d_in, seed)
    packed = ops.PackedModel([net], DEV)
    flat = ops.philox_keep_masks(N, packed.dropout_widths, PASSES, P_DROP, seed, 0, DEV)
    masks = injected_to_masks(flat.cpu(), N, packed.dropout_widths, PASSES)
    net64, x64 = f64([net])[0], x.double()
    ref = uq_oracle.mc_dropout_forward(net64, x64, PASSES, P_DROP, masks=masks)
    ref_tail = uq_oracle.mc_dropout_forward(net64, x64, PASSES - 1, P_DROP, masks=masks[1:])
    ref_off = uq_oracle.mc_dropout_forward(net64, x64, PASSES, P_DROP, dropout_active=False)
    return packed, x, ref, ref_tail, ref_off


def anchored_case(dx, width, d_out, seed, anchor_first):
    net = make_nets(delta_arch(wide_arch(dx, width, 2, d_out)), 1, seed)[0]
    x = rows(dx, seed)
    anchors = rows(dx, seed + 1, n=ANCHORS)
    ys = torch.rand(ANCHORS, d_out, generator=torch.Generator().manual_seed(seed + 2)) * 0.3
    net64, x64, a64 = f64([net])[0], x.double(), anchors.double()
    ref = uq_oracle.delta_uq_forward(net64, x64, a64, ANCHORS, anchor_first=anchor_first)
    ref_tail = uq_oracle.delta_uq_forward(net64, x64, a64[1:], ANCHORS - 1,
                                          anchor_first=anchor_first)
    ref_pager = pager_reference(net64, x64, a64, ys.double(), anchor_first)
    packed = ops.PackedModel([net], DEV, anchor_first=anchor_first)
    return packed, x, anchors, ys, ref, ref_tail, ref_pager


# ---- shared case bodies ------------------------------------------------------------------------------

def run_ensemble(seen, what, packed, x, ref, ref_tail, precisions):
    assert_live_spread(*ref, what)
    xd = x.to(DEV)
    for precision in precisions:
        mean, std = run(seen, packed, precision, what, xd, "ensemble", total_members=ENSEMBLE_K)
        check(precision, mean, std, *ref, what)
        m, m2 = run(seen, packed, precision, what, xd, "ensemble", total_members=ENSEMBLE_K,
                    member_begin=1, member_count=ENSEMBLE_K - 1, output="moments")
        check_moments(precision, m, m2, ENSEMBLE_K - 1, *ref_tail, what)


def run_mc(seen, what, packed, x, ref, ref_tail, ref_off, precisions, seed, off=False):
    assert_live_spread(*ref, what)
    xd = x.to(DEV)
    kw = dict(total_members=PASSES, dropout_p=P_DROP, seed=seed)
    for precision in precisions:
        mean, std = run(seen, packed, precision, what, xd, "mc_dropout", True, **kw)
        check(precision, mean, std, *ref, what)
        m, m2 = run(seen, packed, precision, what, xd, "mc_dropout", True, member_begin=1,
                    member_count=PASSES - 1, output="moments", **kw)
        check_moments(precision, m, m2, PASSES - 1, *ref_tail, what)
        if off:
            mean, std = run(seen, packed, precision, what + " off", xd, "mc_dropout",
                            dropout_active=False, **kw)
            if precision == "bf16":
                bf16_check(mean, std, *ref_off, what + " dropout off")
            else:
                assert_close_ref(mean, ref_off[0], RTOL32, what=f"{what} dropout-off mean")
                assert float(std.abs().max()) <= RTOL32 * float(ref_off[0].abs().max())


def run_delta(seen, what, packed, x, anchors, ref, ref_tail, precisions):
    assert_live_spread(*ref, what)
    xd, ad = x.to(DEV), anchors.to(DEV)
    for precision in precisions:
        mean, std = run(seen, packed, precision, what, xd, "delta_uq", total_members=ANCHORS,
                        anchors=ad)
        check(precision, mean, std, *ref, what)
        m, m2 = run(seen, packed, precision, what, xd, "delta_uq", total_members=ANCHORS,
                    anchors=ad, member_begin=1, member_count=ANCHORS - 1, output="moments")
        check_moments(precision, m, m2, ANCHORS - 1, *ref_tail, what)


def run_pager(seen, what, packed, x, anchors, ys, ref_pager, precisions):
    ref_pmean, ref_conf = ref_pager
    scale = float(ref_pmean.abs().max()) + float(ys.abs().max())
    for precision in precisions:
        pmean, conf = run(seen, packed, precision, what, x.to(DEV), "pager", total_members=ANCHORS,
                          anchors=anchors.to(DEV), targets=ys.to(DEV))
        e_p = float((pmean.double().cpu() - ref_pmean).abs().max())
        e_c = float((conf.double().cpu() - ref_conf).abs().max())
        print(f"[{precision} {what} pager] max|mean err| = {e_p:.3e}, max|conformal err| = "
              f"{e_c:.3e}, scale {scale:.3e}")
        if precision == "bf16":
            assert e_p <= 3e-2 * scale and e_c <= 3e-2 * scale, what
        else:
            assert_close_ref(pmean, ref_pmean, RTOL32, what=f"{what} pager mean")
            assert_close_ref(conf, ref_conf, RTOL32, scale_ref=ref_pmean,
                             what=f"{what} conformal")


def fp32_is_split(width, d_in_net):
    return width <= 512 and d_in_net <= 16


# ---- T1: layer-0 layouts, ensemble and MC dropout ------------------------------------------------

D_IN = [6, 8, 10, 11, 16, 21, 22, 32, 33, 40, 64]


@pytest.mark.parametrize("width", WIDTHS)
@pytest.mark.parametrize("d_in", D_IN)
def test_layer0_layouts_ensemble(seen, d_in, width):
    """s = 3 / 2 / 1 and the stash / in-place boundary (d_in 10 / 11) in every bf16 family; the
    FFMA path at 17 .. 64 inputs with its vectorised (d_in % 4 == 0) and scalar loaders.  fp32
    split-kernel ensembles at d_in <= 16 are test_fp32_split_kernel_all_widths' cases."""
    what = f"ensemble d_in={d_in} s={split_factor(d_in)} {width}"
    packed, x, ref, ref_tail = ensemble_case(d_in, width, 1, 1000 + d_in)
    precisions = ["bf16"] + ([] if fp32_is_split(width, d_in) else ["fp32"])
    run_ensemble(seen, what, packed, x, ref, ref_tail, precisions)


@pytest.mark.parametrize("width", WIDTHS)
@pytest.mark.parametrize("d_in", D_IN)
def test_layer0_layouts_mc_dropout(seen, d_in, width):
    what = f"mc d_in={d_in} s={split_factor(d_in)} {width}"
    packed, x, ref, ref_tail, ref_off = mc_case(d_in, width, 1, 2000 + d_in)
    run_mc(seen, what, packed, x, ref, ref_tail, ref_off, ["bf16", "fp32"], 2000 + d_in)


# ---- T2: anchored layer-0 layouts, Delta-UQ and PAGER ----------------------------------------------

ANCHORED = [(dx, True) for dx in (5, 11, 16, 21, 22, 32)] + [(5, False), (22, False)]


@pytest.mark.parametrize("width", WIDTHS)
@pytest.mark.parametrize("dx,anchor_first", ANCHORED)
def test_anchored_layouts(seen, dx, anchor_first, width):
    """k0_delta layouts, per-anchor bias stages, and both channel orders in delta_bias_kernel,
    column_diff*, the image packers and delta_input_kernel."""
    what = f"anchored dx={dx} s={split_factor(dx)} anchor_first={anchor_first} {width}"
    packed, x, anchors, ys, ref, ref_tail, ref_pager = anchored_case(dx, width, 1, 3000 + dx,
                                                                     anchor_first)
    run_delta(seen, what, packed, x, anchors, ref, ref_tail, ["bf16", "fp32"])
    run_pager(seen, what, packed, x, anchors, ys, ref_pager, ["bf16", "fp32"])


# ---- T3: several outputs ---------------------------------------------------------------------------

@pytest.mark.parametrize("width", WIDTHS)
@pytest.mark.parametrize("d_out", [3, 8])
def test_several_outputs(seen, d_out, width):
    """The DOUT = 8 instantiations of every family, with live Philox dropout (MC = true) too."""
    d_in, seed = 7, 4000 + d_out
    packed, x, ref, ref_tail = ensemble_case(d_in, width, d_out, seed)
    run_ensemble(seen, f"ensemble d_out={d_out} {width}", packed, x, ref, ref_tail,
                 ["bf16", "fp32"])
    packed, x, ref, ref_tail, ref_off = mc_case(d_in, width, d_out, seed)
    run_mc(seen, f"mc d_out={d_out} {width}", packed, x, ref, ref_tail, ref_off, ["bf16", "fp32"],
           seed, off=True)
    packed, x, anchors, ys, ref, ref_tail, ref_pager = anchored_case(d_in, width, d_out, seed, True)
    run_delta(seen, f"delta d_out={d_out} {width}", packed, x, anchors, ref, ref_tail,
              ["bf16", "fp32"])
    if d_out == 3:
        run_pager(seen, f"d_out={d_out} {width}", packed, x, anchors, ys, ref_pager,
                  ["bf16", "fp32"])


# ---- T4: layer-0 exactness with bf16-exact weights -----------------------------------------------

# With weights and biases that are exact in bf16 and a single hidden layer (whose output Linear
# runs in fp32 in the epilogue), the only bf16 error left is the input's representation: ~16 bits
# (x_hi + x_lo) for s = 3 / 2, 8 bits for s = 1.  Measured worst case on a B200 (1000 W): 3.0e-6 of
# scale for s = 3, 2.9e-6 for s = 2, 1.7e-3 for s = 1; the bounds are ~4x that.  Storing 0 for the
# x_lo piece, or packing w_lo into segment 1, gives >= 7.2e-4.
INPUT_BITS_BOUND = {3: 1.2e-5, 2: 1.2e-5, 1: 7e-3}


@pytest.mark.parametrize("d_out", [1, 3])
@pytest.mark.parametrize("width", WIDTHS)
@pytest.mark.parametrize("d_in", [6, 11, 16, 21, 22, 32, 33, 40, 64])
def test_layer0_input_bits_bf16(seen, d_in, width, d_out):
    """A dropped or misplaced x_lo piece is ~2^-9 of an input: far inside bf16_check's 1e-2 bound,
    far outside this one."""
    s = split_factor(d_in)
    nets = make_nets(wide_arch(d_in, width, 1, d_out, bn=False), 2, 5000 + d_in, bn=False)
    with torch.no_grad():
        for net in nets:
            for m in net:
                if isinstance(m, torch.nn.Linear):
                    m.weight.copy_(m.weight.bfloat16().float())
                    m.bias.copy_(m.bias.bfloat16().float())
    x = rows(d_in, 5000 + d_in)
    ref_mean, ref_std = uq_oracle.ensemble_forward(f64(nets), x.double())
    packed = ops.PackedModel(nets, DEV)
    mean, std = run(seen, packed, "bf16", f"input bits d_in={d_in}", x.to(DEV), "ensemble",
                    total_members=2)
    scale = float(ref_mean.abs().max()) + float(ref_std.abs().max())
    e_mean = float((mean.double().cpu() - ref_mean).abs().max()) / scale
    e_std = float((std.double().cpu() - ref_std).abs().max()) / scale
    print(f"[bf16 input bits d_in={d_in} s={s} {width} d_out={d_out}] max|mean err| = "
          f"{e_mean:.3e} of scale, max|std err| = {e_std:.3e} of scale")
    bound = INPUT_BITS_BOUND[s]
    assert e_mean <= bound and e_std <= bound, \
        f"s={s}: error {max(e_mean, e_std):.3e} of scale > {bound:.1e}"


# ---- T5: beyond the bf16 input limit ----------------------------------------------------------------

@pytest.mark.parametrize("d_in", [65, 80])
def test_wide_inputs_run_on_ffma(seen, d_in):
    """More than 64 network inputs: bf16 refuses by name, fp32 runs on the FFMA path at 1e-5, and
    the wrapper's default precision works end to end."""
    width = 320
    packed, x, ref, ref_tail = ensemble_case(d_in, width, 1, 6000 + d_in)
    with pytest.raises(ValueError, match="input width"):
        packed.forward(x.to(DEV), "ensemble", total_members=ENSEMBLE_K, precision="bf16")
    run_ensemble(seen, f"ensemble d_in={d_in} {width}", packed, x, ref, ref_tail, ["fp32"])
    model = EnsembleModelBuilder(wide_arch(d_in, width, 2, 1), {"num_models": ENSEMBLE_K}).build()
    for m, net in zip(model.models, make_nets(wide_arch(d_in, width, 2, 1), ENSEMBLE_K,
                                              6000 + d_in)):
        m.load_state_dict(net.state_dict())
    model.to(DEV).eval()
    with torch.no_grad():
        mean, std = model(x.to(DEV), return_ue=True)
    check("fp32", mean, std, *ref, f"wrapper ensemble d_in={d_in}")

    packed, x, ref, ref_tail, ref_off = mc_case(d_in, width, 1, 6100 + d_in)
    with pytest.raises(ValueError, match="input width"):
        packed.forward(x.to(DEV), "mc_dropout", total_members=PASSES, precision="bf16",
                       dropout_p=P_DROP)
    run_mc(seen, f"mc d_in={d_in} {width}", packed, x, ref, ref_tail, ref_off, ["fp32"],
           6100 + d_in)


def test_ailerons_width_anchored_runs_on_ffma(seen):
    """Delta-UQ / PAGER on 40 sample features (network input 80, the ailerons benchmark)."""
    dx, width = 40, 320
    packed, x, anchors, ys, ref, ref_tail, ref_pager = anchored_case(dx, width, 1, 7000, True)
    for mode in ("delta_uq", "pager"):
        with pytest.raises(ValueError, match="input width"):
            packed.forward(x.to(DEV), mode, total_members=ANCHORS, precision="bf16",
                           anchors=anchors.to(DEV), targets=ys.to(DEV) if mode == "pager" else None)
    run_delta(seen, f"delta dx={dx} {width}", packed, x, anchors, ref, ref_tail, ["fp32"])
    run_pager(seen, f"dx={dx} {width}", packed, x, anchors, ys, ref_pager, ["fp32"])
    model = DeltaUQMLPModelBuilder(wide_arch(dx, width, 2, 1),
                                   {"estimator": "std", "num_anchors": ANCHORS,
                                    "anchored_batch_size": 4096}).build()
    model.net.load_state_dict(make_nets(delta_arch(wide_arch(dx, width, 2, 1)), 1, 7000)[0]
                              .state_dict())
    model.anchors = anchors
    model.to(DEV).eval()
    with torch.no_grad():
        mean, std = model(x.to(DEV), return_ue=True)
    check("fp32", mean, std, *ref, f"wrapper delta dx={dx}")


# ---- T6: float64 callers -----------------------------------------------------------------------------

def test_float64_callers_get_fp32_accuracy():
    """A model cast with ``.double()`` and float64 inputs (bo.py casts models to the dataset's
    dtype): the outputs are float64 and hold the fp32 bound (1e-5) of a float64 reference -- not
    float64 accuracy, the forward computes in fp32."""
    d_in, width = 5, 128
    model = EnsembleModelBuilder(wide_arch(d_in, width, 2, 1), {"num_models": 4}).build()
    for i, m in enumerate(model.models):
        randomise_bn(m, 8000 + i)
    model.double().to(DEV).eval()
    x = rows(d_in, 8000).double()
    ref_mean, ref_std = uq_oracle.ensemble_forward([copy.deepcopy(m).cpu() for m in model.models],
                                                   x)
    with torch.no_grad():
        mean, std = model(x.to(DEV), return_ue=True)
    assert mean.dtype == torch.float64 and std.dtype == torch.float64
    check("fp32", mean, std, ref_mean, ref_std, "float64 ensemble")

    model = DeltaUQMLPModelBuilder(wide_arch(d_in, width, 2, 1),
                                   {"estimator": "std", "num_anchors": ANCHORS,
                                    "anchored_batch_size": 4096}).build()
    randomise_bn(model.net, 8100)
    model.anchors = rows(d_in, 8101, n=ANCHORS).double()
    model.double().to(DEV).eval()
    ref_mean, ref_std = uq_oracle.delta_uq_forward(copy.deepcopy(model.net).cpu(), x,
                                                   model.anchors.cpu(), ANCHORS)
    with torch.no_grad():
        mean, std = model(x.to(DEV), return_ue=True)
    assert mean.dtype == torch.float64 and std.dtype == torch.float64
    check("fp32", mean, std, ref_mean, ref_std, "float64 delta_uq")


# ---- T7: inputs far from zero ------------------------------------------------------------------------

@pytest.mark.parametrize("d_in", [16, 22, 40])
def test_inputs_far_from_zero_bf16(seen, d_in):
    """x = 50 + U[0, 1): s = 3 / 2 keep ~16 input bits and meet the bf16 bound; s = 1 rounds the
    inputs to 8 bits and meets it too (measured 2.3e-3 of scale on a B200)."""
    width = 320
    nets = make_nets(wide_arch(d_in, width, 2, 1), ENSEMBLE_K, 9000 + d_in)
    x = rows(d_in, 9000 + d_in, offset=50.0)
    ref = uq_oracle.ensemble_forward(f64(nets), x.double())
    packed = ops.PackedModel(nets, DEV)
    mean, std = run(seen, packed, "bf16", f"far inputs d_in={d_in}", x.to(DEV), "ensemble",
                    total_members=ENSEMBLE_K)
    bf16_check(mean, std, *ref, f"far inputs d_in={d_in} s={split_factor(d_in)}")
