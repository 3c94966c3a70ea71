"""Shared helpers for the test-suite: rebuild the golden networks, pack masks, tolerances."""
import os
import re

import numpy as np
import torch
import yaml

from nnueehcs_b200.model_builder import build_network

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def golden_arch(g):
    return yaml.safe_load(str(g["arch_yaml"]))


def _state(g, prefix):
    pre = prefix + "."
    return {k[len(pre):]: torch.from_numpy(g[k]) for k in g.files if k.startswith(pre)}


def nets_from_golden(g, k=1, arch=None):
    """Rebuild the K nn.Sequential members stored in a golden file (weights + BN statistics)."""
    arch = golden_arch(g) if arch is None else arch
    nets = []
    for i in range(k):
        net = build_network(arch)
        net.load_state_dict(_state(g, f"m{i}"))
        net.eval()
        nets.append(net)
    return nets


def mc_arch_with_dropout(arch, p):
    """The architecture MCDropoutModelBuilder._add_dropout produces (model_builder.py:254-263)."""
    out = [arch[0]]
    for layer in arch[1:-1]:
        if layer.get("Linear") or layer.get("Conv2d"):
            out.append({"Dropout": {"args": [p]}})
        out.append(layer)
    out.append(arch[-1])
    return out


def delta_arch(arch):
    """DeltaUQMLPModelBuilder doubles the first Linear's in_features (model_builder.py:174-188)."""
    import copy
    arch = copy.deepcopy(arch)
    arch[0]["Linear"]["args"][0] *= 2
    return arch


def golden_masks(g):
    """masks[pass][dropout_layer] -> bool [N, width] from the bit-packed golden arrays."""
    nl = int(g["n_dropout_layers"])
    passes = int(g["passes"])
    per_layer = []
    for l in range(nl):
        w = int(g[f"mask_l{l}_width"])
        m = np.unpackbits(g[f"mask_l{l}"], axis=-1)[..., :w].astype(bool)  # [P, N, w]
        per_layer.append(torch.from_numpy(m))
    return [[per_layer[l][s] for l in range(nl)] for s in range(passes)]


def masks_to_injected(masks):
    """masks[pass][layer] -> flat uint8 tensor in the C ABI's injected layout:
    per dropout layer a [total_members][n][width] block, blocks concatenated in layer order."""
    nl = len(masks[0])
    blocks = []
    for l in range(nl):
        blocks.append(torch.stack([m[l] for m in masks]).to(torch.uint8).reshape(-1))
    return torch.cat(blocks).contiguous()


def injected_to_masks(flat, n, widths, total):
    """Inverse of masks_to_injected."""
    out = [[None] * len(widths) for _ in range(total)]
    off = 0
    for l, w in enumerate(widths):
        blk = flat[off:off + total * n * w].reshape(total, n, w).bool()
        for s in range(total):
            out[s][l] = blk[s]
        off += total * n * w
    return out


def wide_arch(d_in, width, n_hidden, d_out, bn=True):
    """``n_hidden`` x (Linear -> [BatchNorm1d] -> ReLU) of equal width, then Linear(width, d_out)."""
    arch, prev = [], d_in
    for _ in range(n_hidden):
        arch.append({"Linear": {"args": [prev, width]}})
        if bn:
            arch.append({"BatchNorm1d": {"args": [width]}})
        arch.append({"ReLU": {"inplace": True}})
        prev = width
    arch.append({"Linear": {"args": [prev, d_out]}})
    return arch


def randomise_bn(net, seed):
    """Non-trivial eval-mode BatchNorm statistics, so that folding them into the weights matters."""
    gen = torch.Generator().manual_seed(seed)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=gen) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=gen) + 0.5)


def bf16_check(mean, std, ref_mean, ref_std, what, tol=1e-2, tol_std=5e-2):
    """bf16 tolerance.  The natural unit is the magnitude of one member's output, taken as
    ``scale = max|ref_mean| + max|ref_std|``: both errors must stay within ``tol * scale`` (measured
    worst case over every bf16 test: 2.3e-3, and 4.3e-3 for identical passes whose std is 0 -- the
    bound is 2.5-5x that; a mis-addressed K chunk is an error of >= 1/8 of scale), and the std
    additionally within ``tol_std`` of its OWN scale (measured 1e-3 .. 2.2e-2; the largest values
    belong to anchored nets whose spread is 16x smaller than their mean)."""
    mean, std = mean.double().cpu(), std.double().cpu()
    ref_mean, ref_std = torch.as_tensor(ref_mean).double(), torch.as_tensor(ref_std).double()
    ms, ss = float(ref_mean.abs().max()), float(ref_std.abs().max())
    scale = ms + ss
    e_mean = float((mean - ref_mean).abs().max())
    e_std = float((std - ref_std).abs().max())
    print(f"[bf16 {what}] max|mean err| = {e_mean:.3e} ({e_mean / scale:.3e} of scale), "
          f"max|std err| = {e_std:.3e} ({e_std / scale:.3e} of scale, "
          f"{e_std / max(ss, 1e-30):.3e} of std scale)")
    assert e_mean <= tol * scale, f"{what}: bf16 mean error {e_mean / scale:.3e} of scale > {tol}"
    assert e_std <= tol * scale, f"{what}: bf16 std error {e_std / scale:.3e} of scale > {tol}"
    if ss > 1e-3 * ms:   # identical passes have std == 0: nothing relative to check
        assert e_std <= tol_std * ss, \
            f"{what}: bf16 std error {e_std / ss:.3e} of std scale > {tol_std}"


def assert_close_ref(got, ref, rtol, scale_ref=None, what=""):
    """|got - ref| <= rtol * |ref| + rtol * max|scale_ref|  (north_star's 1e-5 'relative', with the
    absolute floor tied to the output scale: std -> 0 in-distribution, SURVEY 8d)."""
    got = torch.as_tensor(got).double().cpu()
    ref = torch.as_tensor(ref).double().cpu()
    scale = ref if scale_ref is None else torch.as_tensor(scale_ref).double().cpu()
    atol = rtol * float(scale.abs().max())
    err = (got - ref).abs()
    bound = rtol * ref.abs() + atol
    worst = float((err - bound).max())
    assert worst <= 0, (f"{what}: max err {float(err.max()):.3e} exceeds rtol={rtol} "
                        f"(atol {atol:.3e}); worst excess {worst:.3e}")


# ---- forward kernel attribution ---------------------------------------------------------------------
# Every forward of the GPU forward tests runs under torch.profiler: the kernel instantiations it
# launched must be the ones expected_kernels() restates from the dispatch code, so that no case
# silently stops covering its kernel when the dispatch changes.

RTOL32 = 1e-5
MAX_MMA_LAYERS = 16       # tc_params.cuh


def tc_refusal(sig):
    """Why ``tc_plan`` (csrc/mlp_tc.cu) refuses the bf16 path for this structure signature, or
    None.  ``sig`` is ``extract.structure_signature``: one (in, out, bn, relu, dropout) per block."""
    if len(sig) < 2:
        return "needs at least one hidden Linear"
    width = sig[0][1]
    if any(blk[1] != width for blk in sig[:-1]):
        return "hidden widths differ"
    if not (width % 64 == 0 and 64 <= width <= 512) and width not in (768, 1024):
        return "hidden width must be a multiple of 64"
    if len(sig) - 1 > MAX_MMA_LAYERS:
        return "too many layers"
    if sig[-1][1] > 8:
        return "final out_features > 8"
    if sig[-1][2] or sig[-1][4]:
        return "BatchNorm/Dropout after the final Linear"
    if sig[0][0] > 64:
        return "input width > 64"
    return None


def tcx_refusal(sig):
    """Why ``tcx_plan`` (csrc/mlp_tcx.cu) refuses the fp32 split kernels, or None."""
    why = tc_refusal(sig)
    if why is not None:
        return why
    if sig[0][1] > 512:
        return f"hidden width {sig[0][1]} > 512"
    if sig[0][0] > 16:
        return "input width > 16"
    return None


def expected_kernels(precision, mode, sig, live_dropout):
    """The forward kernel instantiations one call launches, as ``family<args>`` strings.

    ``sig`` is the packed structure signature; its first ``in`` is the NETWORK input width (twice
    the sample width for Delta-UQ / PAGER).  Restates ``tc_plan`` / ``tc_forward`` (mlp_tc.cu),
    ``tc2_launch`` / ``dispatch_h3`` / ``tc4_launch`` (the bias-in-the-MMA variants are the default
    for d_out 1), ``tcx_plan`` (mlp_tcx.cu: hidden width <= 512 and at most 16 network inputs) and
    ``fp32_forward`` (mlp_fp32.cu), which runs per layer either ``linear_small_out_kernel`` (the
    last layer without BatchNorm or live Dropout and at most 8 outputs) or ``sgemm_tn_kernel``
    (its vectorised loader needs a multiple of 4 inputs).  A model the bf16 path refuses launches
    no forward kernel in bf16."""
    b = lambda v: "true" if v else "false"
    width, d_out = sig[0][1], sig[-1][1]
    dpad = 1 if d_out == 1 else 8
    mc = live_dropout and mode == "mc_dropout"
    if precision == "bf16":
        if tc_refusal(sig) is not None:
            return set()
        mc = mc and any(blk[4] for blk in sig[:-1])
        if width > 512:
            return {f"tc3<{width},1,true>" if dpad == 1 else f"tc3<{width},8,false>"}
        if width in (64, 128) and dpad == 1:
            return {f"tc4<{width},true,{b(mc)}>"}
        return {f"tc2<{width},{dpad},2,{b(mc)},{b(dpad == 1)}>"}
    if precision == "fp32" and tcx_refusal(sig) is None:
        mc = mc and any(blk[4] for blk in sig[:-1])
        if width in (64, 128) and dpad == 1:
            return {f"tcx4<{width},{b(mc)}>"}
        return {f"tcx<{width},{dpad},{b(mc)}>"}
    found = set()
    for l, (d_in, d_out_l, bn, _, drop) in enumerate(sig):
        if l == len(sig) - 1 and not bn and not (drop and mc) and d_out_l <= 8:
            found.add("linear_small_out_kernel")
        else:
            found.add(f"sgemm_tn_kernel<{b(d_in % 4 == 0)}>")
    return found


_KERNEL = re.compile(r"\b(?:uq_mlp_(tc2|tc3|tc4|tcx|tcx4)_kernel|(sgemm_tn_kernel))\s*<([^<>]*)>"
                     r"|\b(linear_small_out_kernel)\b")


def forward_kernels(call):
    """Run ``call()`` under the CUDA profiler; return its result and the forward kernels it ran."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = call()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names, "the profiler recorded no CUDA kernel at all: kernel attribution is impossible"
    found = set()
    for name in names:
        m = _KERNEL.search(name)
        if m and m.group(4):
            found.add(m.group(4))
        elif m:
            found.add(f"{m.group(1) or m.group(2)}<{re.sub(r'\s+', '', m.group(3))}>")
    return out, found


def run(seen, packed, precision, what, x, mode, live_dropout=False, **kw):
    """``packed.forward`` with kernel attribution; ``seen`` collects the instantiations run."""
    (a, b), found = forward_kernels(lambda: packed.forward(x, mode, precision=precision, **kw))
    expect = expected_kernels(precision, mode, packed.signature, live_dropout)
    assert found == expect, f"{what} [{precision}]: ran {sorted(found)}, dispatch says {sorted(expect)}"
    seen.update(found)
    return a, b


def check(precision, mean, std, ref_mean, ref_std, what, bf16_tol=(1e-2, 5e-2)):
    """bf16: ``bf16_check`` with ``(tol, tol_std) = bf16_tol``; fp32 / fp32_ffma:
    ``assert_close_ref`` at RTOL32, the std's absolute floor tied to the mean's scale."""
    if precision == "bf16":
        bf16_check(mean, std, ref_mean, ref_std, what, tol=bf16_tol[0], tol_std=bf16_tol[1])
        return
    e_mean = float((mean.double().cpu() - ref_mean).abs().max())
    e_std = float((std.double().cpu() - ref_std).abs().max())
    print(f"[{precision} {what}] max|mean err| = {e_mean:.3e}, max|std err| = {e_std:.3e} "
          f"(mean scale {float(ref_mean.abs().max()):.3e})")
    assert_close_ref(mean, ref_mean, RTOL32, what=f"{what} mean")
    assert_close_ref(std, ref_std, RTOL32, scale_ref=ref_mean, what=f"{what} std")


def assert_live_spread(ref_mean, ref_std, what):
    """A std check means nothing when the members agree: the reference must spread."""
    ms, ss = float(ref_mean.abs().max()), float(ref_std.abs().max())
    assert ss >= 1e-2 * ms, f"{what}: reference std {ss:.3e} < 1e-2 of mean scale {ms:.3e}"


def pager_reference(net64, x64, a64, ys64, anchor_first):
    """(mean over anchors of the swapped-role predictions, max_k |P[k] - Y_k|) for any d_out."""
    from oracle import uq_oracle
    with torch.no_grad():
        p = torch.stack([uq_oracle.sequential_forward(
            net64, uq_oracle.anchored_input(a64[j:j + 1].expand(x64.shape[0], -1), x64,
                                            anchor_first))
            for j in range(a64.shape[0])])                                # [K, N, d_out]
    return p.mean(0), (p - ys64.unsqueeze(1)).abs().max(dim=0)[0]
