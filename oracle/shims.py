"""Import shims so the UNMODIFIED reference package can be imported in the authoring container.

TEST INFRASTRUCTURE (oracle).  Used only by the ``tests/golden/make_golden*.py`` scripts that
record the reference's outputs; the test-suite reads those recordings and never the reference.

``nnueehcs/models.py`` imports three modules that are not installed here and are not vendored
in the reference tree (``models.py:2,3,8-9``): ``deltauq``, ``kde`` and ``pytorch_lightning``.
The shims are inert for the ensemble / MC-dropout arithmetic (``LightningModule`` degenerates
to ``nn.Module``; ``Callback`` is an empty class).  ``deltauq.deltaUQ_MLP`` is bound to this
repo's *restatement* (``oracle.uq_oracle.DeltaUQMLPRestated``), so anything computed through
``nnueehcs.models.DeltaUQMLP`` is **parity-unpinned** -- it only checks that the reference's
chunk/concat wrapper logic (``models.py:313-341``) composes with the restatement.
"""
import os
import sys
import types

import torch.nn as nn

REFERENCE_ROOT = os.environ.get("NNUEEHCS_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "nnueehcs"))


def _make_lightning_stub() -> types.ModuleType:
    pl = types.ModuleType("pytorch_lightning")

    class LightningModule(nn.Module):
        def log(self, *args, **kwargs):  # Lightning logging is a no-op outside a Trainer
            return None

    class Callback:
        pass

    class Trainer:  # only needed so ``nnueehcs.training`` would import; never used here
        def __init__(self, *a, **k):
            raise RuntimeError("pytorch_lightning is not installed; Trainer is a stub")

    callbacks = types.ModuleType("pytorch_lightning.callbacks")
    callbacks.Callback = Callback
    pl.LightningModule = LightningModule
    pl.Trainer = Trainer
    pl.callbacks = callbacks
    pl.__stub__ = True
    return pl


def install() -> None:
    """Install the stub modules and put the reference tree on ``sys.path`` (idempotent)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if "pytorch_lightning" not in sys.modules:
        pl = _make_lightning_stub()
        sys.modules["pytorch_lightning"] = pl
        sys.modules["pytorch_lightning.callbacks"] = pl.callbacks
    if "deltauq" not in sys.modules:
        from .uq_oracle import DeltaUQMLPRestated

        duq = types.ModuleType("deltauq")
        duq.deltaUQ_MLP = DeltaUQMLPRestated
        duq.deltaUQ_CNN = type("deltaUQ_CNN", (nn.Module,), {})
        duq.__stub__ = True
        sys.modules["deltauq"] = duq
    if "kde" not in sys.modules:
        kde = types.ModuleType("kde")
        kde.KNNKDE = type("KNNKDE", (), {})
        kde.__stub__ = True
        sys.modules["kde"] = kde
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def import_reference():
    """Return the reference's ``(models, model_builder, evaluation)`` modules."""
    install()
    import nnueehcs.models as ref_models
    import nnueehcs.model_builder as ref_builder
    import nnueehcs.evaluation as ref_eval

    return ref_models, ref_builder, ref_eval
