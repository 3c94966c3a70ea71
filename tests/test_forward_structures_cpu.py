"""The host side of the layer structures the fused forward accepts (no GPU needed):
``extract.split_blocks`` / ``structure_signature`` / ``dropout_widths``, and the MC-dropout
wrapper's check that every Dropout shares one ``p`` and one train / eval state."""
import pytest
import torch
import torch.nn as nn

from nnueehcs_b200.extract import dropout_widths, split_blocks, structure_signature
from nnueehcs_b200.model_builder import MCDropoutModelBuilder

L, BN, R, D = nn.Linear, nn.BatchNorm1d, nn.ReLU, nn.Dropout

STRUCTURES = {
    "hidden_without_relu": (
        [L(5, 8), L(8, 8), BN(8), L(8, 1)],
        ((5, 8, False, False, False), (8, 8, True, False, False), (8, 1, False, False, False)),
        []),
    "relu_pattern_TFT": (
        [L(5, 8), R(), L(8, 8), L(8, 8), R(), L(8, 3)],
        ((5, 8, False, True, False), (8, 8, False, False, False), (8, 8, False, True, False),
         (8, 3, False, False, False)),
        []),
    "relu_after_final": (
        [L(5, 8), BN(8), R(), L(8, 3), R()],
        ((5, 8, True, True, False), (8, 3, False, True, False)), []),
    "linear_bn_dropout": (
        [L(5, 8), BN(8), D(0.2), L(8, 8), D(0.2), L(8, 1)],
        ((5, 8, True, False, True), (8, 8, False, False, True), (8, 1, False, False, False)),
        [8, 8]),
    "dropout_on_middle_layer": (
        [L(5, 8), R(), L(8, 8), R(), D(0.2), L(8, 8), R(), L(8, 1)],
        ((5, 8, False, True, False), (8, 8, False, True, True), (8, 8, False, True, False),
         (8, 1, False, False, False)),
        [8]),
    "unequal_widths": (
        [L(5, 100), R(), L(100, 37), R(), D(0.2), L(37, 3)],
        ((5, 100, False, True, False), (100, 37, False, True, True), (37, 3, False, False, False)),
        [37]),
    "bn_and_dropout_after_final": (
        [L(5, 8), R(), L(8, 3), BN(3), D(0.2)],
        ((5, 8, False, True, False), (8, 3, True, False, True)), [3]),
    "single_linear": ([L(5, 3)], ((5, 3, False, False, False),), []),
    "single_linear_dropout": ([L(5, 1), D(0.2)], ((5, 1, False, False, True),), [1]),
}


@pytest.mark.parametrize("name", list(STRUCTURES))
def test_structure_signature(name):
    mods, sig, widths = STRUCTURES[name]
    blocks = split_blocks(nn.Sequential(*mods))
    assert structure_signature(blocks) == sig
    assert dropout_widths(blocks) == widths


def test_seventeen_hidden_layers_split():
    """Depth is not split_blocks' concern: 17 hidden layers (one beyond the tensor-core limit) are
    accepted and run on the FFMA path."""
    mods = []
    for _ in range(17):
        mods += [L(8, 8), BN(8), R()]
    blocks = split_blocks(nn.Sequential(*mods, L(8, 1)))
    assert len(blocks) == 18 and all(b.bn is not None and b.relu for b in blocks[:-1])


def test_bias_and_affine_do_not_change_the_signature():
    """A Linear without bias and a BatchNorm without affine parameters pack as zeros / ones, so
    members that differ in them share one signature and pack as one ensemble."""
    a = nn.Sequential(L(5, 8), BN(8), R(), L(8, 1))
    b = nn.Sequential(L(5, 8, bias=False), BN(8, affine=False), R(), L(8, 1, bias=False))
    c = nn.Sequential(L(5, 8), BN(8, eps=0.1, affine=False), R(), L(8, 1))
    sigs = {structure_signature(split_blocks(n)) for n in (a, b, c)}
    assert sigs == {((5, 8, True, True, False), (8, 1, False, False, False))}
    blk = split_blocks(b)[0]
    assert blk.linear.bias is None and blk.bn.weight is None and blk.bn.bias is None


@pytest.mark.parametrize("mods,match", [
    ([L(5, 8), D(0.2), R(), L(8, 1)], "unexpected ReLU position"),
    ([L(5, 8), R(), BN(8), L(8, 1)], "BatchNorm1d must directly follow its Linear"),
    ([L(5, 8), D(0.2), D(0.2), L(8, 1)], "two Dropouts in a row"),
    ([L(5, 8), BN(8, track_running_stats=False), L(8, 1)], "without running statistics"),
    ([R(), L(5, 1)], "precedes the first Linear"),
])
def test_structures_outside_the_block_grammar(mods, match):
    with pytest.raises(ValueError, match=match):
        split_blocks(nn.Sequential(*mods))


def _mc_model():
    arch = []
    for prev in (5, 16, 16):
        arch += [{"Linear": {"args": [prev, 16]}}, {"ReLU": {}}]
    arch.append({"Linear": {"args": [16, 1]}})
    model = MCDropoutModelBuilder(arch, {"num_samples": 4, "dropout_percent": 0.2}).build()
    model.eval()
    drops = [(i, m) for i, m in enumerate(model.model) if isinstance(m, nn.Dropout)]
    assert len(drops) == 2 and all(m.training for _, m in drops)
    return model, drops


def test_mc_wrapper_refuses_a_dropout_in_eval_mode():
    model, drops = _mc_model()
    idx, d = drops[1]
    d.eval()
    with pytest.raises(ValueError, match=f"Dropout '{idx}' is in eval mode"):
        model(torch.rand(3, 5))


def test_mc_wrapper_refuses_a_dropout_with_its_own_p():
    model, drops = _mc_model()
    idx, d = drops[0]
    d.p = 0.5
    with pytest.raises(ValueError, match=f"Dropout '{idx}' has p = 0.5"):
        model(torch.rand(3, 5))


def test_mc_wrapper_accepts_dropouts_that_agree():
    """All live (after eval()) or all in eval mode: the check passes, and a CPU tensor then meets
    the fused forward's CUDA requirement."""
    model, drops = _mc_model()
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        model(torch.rand(3, 5))
    for _, m in drops:
        m.eval()
        m.p = 0.9          # an inactive Dropout's p does not matter
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        model(torch.rand(3, 5))
