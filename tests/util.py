"""Shared helpers for the test-suite: rebuild the golden networks, pack masks, tolerances."""
import os

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
