"""Host-side mirror of the reference's UQ wrappers (``nnueehcs/models.py``), same names and
signatures, with the inference forward routed to the fused B200 op.

What stays stock torch: construction, ``.to()``, pickling, and the *training* forward (it needs
autograd; reference ``models.py:148-149,316-317``).  What is replaced: the eval-mode
``forward(x, return_ue)`` bodies --

* ``EnsembleModel.forward``   (models.py:99-108):  ``stack([m(x) for m in models])`` -> mean/std
* ``MCDropoutModel.forward``  (models.py:147-163): ``num_samples`` stochastic passes -> mean/std
* ``DeltaUQMLP.forward``      (models.py:313-341): anchored passes inside ``deltauq`` -> mean/std

all become one call into ``libnnueehcs_b200.so`` (``ops.PackedModel.forward``).  There is no CPU
fallback: an eval-mode forward on a non-CUDA tensor raises ``RuntimeError``.

Knobs that do not exist in the reference (all optional, attributes on the wrapper):
``uq_precision``  ``'fp32'`` (default; the 1e-5 parity mode: scaled fp16 x 2 split on tcgen05,
                  CUDA-core FFMA for shapes the split kernels do not cover) or ``'bf16'`` (tcgen05
                  tensor-core mode); default overridable with ``NNUEEHCS_B200_PRECISION``.
``uq_shard``      optional ``distributed.KShard`` -- shard members/passes/anchors over ranks.

float64 callers (a model cast with ``.double()`` and float64 inputs, as ``bo.py`` does with the
dataset's dtype) get float64 outputs, but the forward computes in fp32: with ``'fp32'`` the results
are within the fp32 bound, ``1e-5 * |ref| + 1e-5 * max|ref_mean|``, of a float64 reference -- not
float64 accuracy.
"""
from __future__ import annotations

import copy
import os
import sys
from typing import Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .extract import tensors_version

try:  # Lightning is optional: the reference trains with it, inference does not need it
    import pytorch_lightning as pl  # type: ignore
    _Base = pl.LightningModule
    _Callback = pl.callbacks.Callback
    HAVE_LIGHTNING = True
except Exception:  # pragma: no cover - depends on the environment
    HAVE_LIGHTNING = False

    class _Base(nn.Module):  # type: ignore
        def log(self, *args, **kwargs):
            return None

    class _Callback:  # type: ignore
        pass

training_defaults = {
    'learning_rate': 1e-3,
    'batch_size': 32,
    'num_workers': 1,
    'num_epochs': 10,
    'loss': 'l1_loss',
}


def _default_precision() -> str:
    return os.environ.get("NNUEEHCS_B200_PRECISION", "fp32")


class WrappedModelBase(_Base):
    """Loss / optimizer plumbing shared by every wrapper (reference models.py:22-85)."""

    def __init__(self, train_config=None, validation_config=None):
        super().__init__()
        self.train_config = copy.deepcopy(training_defaults)
        self.validation_config = copy.deepcopy(training_defaults)
        self.set_train_config(train_config)
        self.set_validation_config(validation_config)
        self.uq_precision = _default_precision()
        self.uq_shard = None
        self._uq_cache = None

    def set_train_config(self, train_config):
        if train_config is not None:
            self.train_config.update(train_config)
        self.loss = self.get_loss_fn(self.train_config['loss'])

    def set_validation_config(self, validation_config):
        # the validation config defaults to the train config, as in the reference
        self.validation_config.update(self.train_config if validation_config is None
                                      else validation_config)
        self.val_loss = self.get_loss_fn(self.validation_config['loss'])

    def get_loss_fn(self, name):
        fn = getattr(F, name, None)
        if fn is None:
            raise ValueError(f"Unknown loss function: {name}")
        return fn

    def training_step(self, batch, batch_idx):
        x, y = batch
        loss = self.loss(self(x), y)
        self.log('train_loss', loss)
        return loss

    def validation_step(self, batch, batch_idx):
        x, y = batch
        loss = self.loss(self(x), y)
        self.log('val_loss', loss)
        return loss

    def on_train_start(self):
        self.logger.log_hyperparams({'train_config': self.train_config,
                                     'validation_config': self.validation_config})

    def configure_optimizers(self):
        opt = torch.optim.AdamW(self.parameters(), lr=self.train_config['learning_rate'],
                                weight_decay=self.train_config.get('weight_decay', 0))
        sched = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, 'min')
        return {'optimizer': opt, 'lr_scheduler': sched, 'monitor': 'val_loss'}

    def get_callbacks(self):
        return []

    # ---- packed-weight cache ---------------------------------------------------------------
    # Rebuilt lazily whenever a parameter/buffer changed (in-place version counter), moved
    # (.to()), or after unpickling -- the reference checkpoints whole modules with torch.save
    # (training.py:54-65) and reloads them with torch.load (examples/bo_driven/bo.py:409).
    def _packed(self, nets: Sequence[nn.Sequential], device: torch.device) -> ops.PackedModel:
        anchor_first = bool(getattr(self, "anchor_first", True))
        key = (str(device), tensors_version(nets), anchor_first)
        cache = self.__dict__.get("_uq_cache")
        if cache is None or cache[0] != key:
            if cache is not None:
                cache[1].close()
            cache = (key, ops.PackedModel(nets, device, anchor_first=anchor_first))
            self.__dict__["_uq_cache"] = cache
        return cache[1]

    def invalidate_packed(self) -> None:
        """Drop the packed-weight cache explicitly (it is rebuilt on the next eval-mode forward).
        The cache key follows parameter identity, versions and module structure; call this after
        an edit it cannot see."""
        cache = self.__dict__.get("_uq_cache")
        if cache is not None:
            cache[1].close()
        self.__dict__["_uq_cache"] = None

    def _shared_seed(self, seed: int, device) -> int:
        """Under a shard every rank must key Philox with the SAME seed, whatever its own CPU
        generator holds (``manual_seed(base + rank)`` is a common setup): rank 0's seed is
        broadcast over the shard's group."""
        shard = self.__dict__.get("uq_shard")
        if shard is None or getattr(shard, "world", 1) <= 1:
            return seed
        import torch.distributed as dist
        t = torch.tensor([seed], dtype=torch.int64, device=device)
        dist.broadcast(t, src=dist.get_global_rank(shard.group, 0) if shard.group is not None else 0,
                       group=shard.group)
        return int(t.item())

    def __getstate__(self):
        state = dict(self.__dict__)
        state["_uq_cache"] = None  # device handles are not picklable; rebuilt on first use
        return state

    def __setstate__(self, state):
        super().__setstate__(state)
        self.__dict__.setdefault("_uq_cache", None)
        self.__dict__.setdefault("uq_precision", _default_precision())
        self.__dict__.setdefault("uq_shard", None)

    def _fused(self, packed: ops.PackedModel, x: torch.Tensor, mode: str, total: int, **kw):
        shard = self.__dict__.get("uq_shard")
        if shard is not None:
            mean, std = shard.forward(packed, x, mode, total_members=total,
                                      precision=self.uq_precision, **kw)
        else:
            mean, std = packed.forward(x, mode, total_members=total,
                                       precision=self.uq_precision, **kw)
        if x.dtype != torch.float32:  # datasets may be float64 (bo.py:396); compute is fp32
            mean, std = mean.to(x.dtype), std.to(x.dtype)
        return mean, std


class EnsembleModel(WrappedModelBase):
    def __init__(self, models, vectorize=False, **kwargs):
        super().__init__(**kwargs)
        self.models = nn.ModuleList(models)
        # `vectorize` selected the vmap path in the reference (models.py:93-101); both paths
        # compute the same thing and the fused op supersedes them in inference.
        self.vectorize = vectorize

    def forward(self, x, return_ue=False):
        if self.training:
            outputs = torch.stack([model(x) for model in self.models])
            if return_ue:
                return outputs.mean(0), outputs.std(0)
            return outputs.mean(0)
        ops._require_cuda(x, "x")
        packed = self._packed(list(self.models), x.device)
        mean, std = self._fused(packed, x, "ensemble", len(self.models))
        return (mean, std) if return_ue else mean

    def to(self, *args, **kwargs):
        super().to(*args, **kwargs)
        return self


class MCDropoutModel(WrappedModelBase):
    def __init__(self, model, num_samples=100, dropout_percent=0.5, vectorize=False, **kwargs):
        super().__init__(**kwargs)
        self.model = model
        self.num_samples = num_samples
        self.dropout_percent = dropout_percent
        self.vectorize = vectorize
        for module in self.model.modules():  # reference models.py:132-134
            if isinstance(module, nn.Dropout):
                module.p = dropout_percent
        self._injected_masks = None

    def _dropout_live(self) -> bool:
        """Whether the Dropouts are live.  The fused op applies ONE ``p`` (``dropout_percent``) and
        ONE live flag to every Dropout, where the reference's ``self.model(x)`` honours each
        module's own ``p`` and train / eval state: a Dropout that differs from the others is a
        ``ValueError`` naming it, not a silently different result."""
        drops = [(name, m) for name, m in self.model.named_modules() if isinstance(m, nn.Dropout)]
        live = any(m.training for _, m in drops)
        for name, m in drops:
            if m.training != live:
                raise ValueError(
                    f"MCDropoutModel: Dropout {name!r} is in {'train' if m.training else 'eval'} "
                    f"mode and another Dropout is not; the fused forward needs every Dropout live "
                    "(after eval()) or every one in eval mode")
            if live and m.p != self.dropout_percent:
                raise ValueError(
                    f"MCDropoutModel: Dropout {name!r} has p = {m.p}, not dropout_percent = "
                    f"{self.dropout_percent}; the fused forward applies one p to every Dropout")
        return live

    def inject_masks(self, masks: Optional[torch.Tensor]) -> None:
        """Testing hook: use these keep-masks (uint8, layout of ``uq_forward_args.masks``) instead
        of the native Philox stream on the next forwards; ``None`` restores Philox."""
        self._injected_masks = masks

    def forward(self, x, return_ue=False):
        if self.training:
            return self.model(x)
        live = self._dropout_live()
        ops._require_cuda(x, "x")
        packed = self._packed([self.model], x.device)
        # Philox stream keyed from torch's CPU generator: reproducible under torch.manual_seed
        seed = self._shared_seed(int(torch.randint(0, 2 ** 62, (1,)).item()), x.device)
        mean, std = self._fused(packed, x, "mc_dropout", int(self.num_samples),
                                dropout_p=float(self.dropout_percent),
                                dropout_active=live, seed=seed,
                                masks=self._injected_masks)
        return (mean, std) if return_ue else mean

    def eval(self):
        # reference models.py:165-169: everything in eval mode except the Dropout modules
        super().eval()
        for module in self.model.modules():
            if isinstance(module, nn.Dropout):
                module.train()
        return self


class MLPModel(WrappedModelBase):
    def __init__(self, model, **kwargs):
        super().__init__(**kwargs)
        self.model = model

    def forward(self, x):
        return self.model(x)


class DeltaUQMLP(WrappedModelBase):
    """Anchored (Delta-UQ) MLP.  The reference subclasses the third-party ``deltaUQ_MLP``
    (models.py:288); that package is absent from the reference tree, so the anchoring scheme here
    follows the published method and is PARITY-UNPINNED (see DESIGN.md).

    ``anchor_first`` (class attribute, default True): the network sees ``cat([a, x - a], dim=1)``,
    the channel order of the public ``deltauq`` package (``create_anchored_batch``:
    ``torch.cat([A, diff], axis=1)``), so a first-Linear weight trained with the reference stack
    means the same thing here.  Set it to False on an instance whose checkpoint was trained with
    the other order, ``cat([x - a, a])``."""

    anchor_first = True

    def __init__(self, base_model, estimator='std', num_anchors=5, anchored_batch_size=None,
                 **kwargs):
        super().__init__(**kwargs)
        self.net = base_model
        self.estimator = estimator
        self.num_anchors = num_anchors
        # kept for API parity; the fused kernel never materialises the K x N anchored batch, so
        # chunking by anchored_batch_size (models.py:329-341) has nothing left to bound
        self.batch_size = sys.maxsize if anchored_batch_size is None else anchored_batch_size
        self.register_buffer('_anchors', None)

    def training_step(self, batch, batch_idx):
        x, y = batch
        y_hat = self(x)
        loss = self.loss(y_hat, y)
        self.log('train_loss', loss)
        return loss

    def _anchored_torch(self, x, anchors_per_row):
        parts = ([anchors_per_row, x - anchors_per_row] if self.anchor_first
                 else [x - anchors_per_row, anchors_per_row])
        return self.net(torch.cat(parts, dim=1))

    def forward(self, x, return_ue=False):
        if self.training or self._anchors is None:
            if not self.training and return_ue:
                print("WARNING: Returning UE without anchors")
            # stochastic data centering: one random in-batch anchor per sample (training path)
            a = x[torch.randperm(x.shape[0], device=x.device)]
            return self._anchored_torch(x, a)
        ops._require_cuda(x, "x")
        packed = self._packed([self.net], x.device)
        mean, std = self._fused(packed, x, "delta_uq", int(self.num_anchors),
                                anchors=self._anchors.to(x.device))
        return (mean, std) if return_ue else mean

    @property
    def anchors(self):
        return self._anchors

    @anchors.setter
    def anchors(self, value):
        self._anchors = value.detach().clone()

    class DeltaUQGetAnchorsCallback(_Callback):
        """First ``num_anchors`` rows of the first training batches become the anchors
        (reference models.py:354-369)."""

        def __init__(self):
            super().__init__()
            self._train_data_to_fit = []
            self._epochs = 0

        def on_validation_epoch_start(self, trainer, pl_module):
            if self._epochs == 0 and len(self._train_data_to_fit) > 0:
                trn = torch.cat(self._train_data_to_fit)
                pl_module.anchors = trn[0:pl_module.num_anchors].detach().clone()
            self._epochs += 1

        def on_train_batch_end(self, trainer, pl_module, outputs, batch, batch_idx):
            bs = batch[0].shape[0]
            if self._epochs == 0 and bs * len(self._train_data_to_fit) < pl_module.num_anchors:
                self._train_data_to_fit.append(batch[0].detach())

    def get_callbacks(self):
        return [DeltaUQMLP.DeltaUQGetAnchorsCallback()]


def _out_of_scope(name):
    class _Unsupported(WrappedModelBase):
        def __init__(self, *a, **k):
            raise NotImplementedError(
                f"{name} is outside the hot path this package accelerates (SURVEY.md section 8: "
                "KNN-KDE needs the absent third-party `kde` package); use the reference class")
    _Unsupported.__name__ = name
    return _Unsupported




class KDEMLPModel(MLPModel):
    """MLP + input-density uncertainty score, reference models.py:191-240.

    ``fit_kde(data)`` keeps a random ``train_fit_prop`` share of the training inputs (on their
    device) and sklearn's 'scott' (``m ** (-1 / (d + 4))``) or 'silverman' bandwidth;
    ``forward(x, return_ue=True)``
    returns ``(pred, dens)`` with ``dens = -exp(KernelDensity.score_samples(x))`` as a float64
    ``[N]`` tensor, computed by ``uq_kde_density`` on the GPU (the reference copies ``x`` to the
    host and walks a KD-tree per call).  ``rtol`` is kept for API parity: sklearn stops refining
    at ``rtol / 10000`` relative, the kernel adds every term."""

    def __init__(self, base_model, bandwidth='scott', rtol=0.1, train_fit_prop=1.0, **kwargs):
        super().__init__(base_model, **kwargs)
        if bandwidth not in ('scott', 'silverman') and not isinstance(bandwidth, (int, float)):
            raise ValueError(f"bandwidth must be 'scott', 'silverman' or a number, got "
                             f"{bandwidth!r}")
        self.bandwidth = bandwidth
        self.rtol = rtol / 10000
        self.kde = None
        self.train_fit_prop = train_fit_prop
        self.register_buffer('_kde_data', None)

    def fit_kde(self, data):
        idx = torch.randperm(len(data))[:int(self.train_fit_prop * len(data))]
        kept = data[idx.to(data.device)].detach().to(torch.float32).contiguous()
        self._kde_data = kept
        m, d = kept.shape
        rules = {'scott': ops.kde_scott_bandwidth, 'silverman': ops.kde_silverman_bandwidth}
        h = rules[self.bandwidth](m, d) if self.bandwidth in rules else float(self.bandwidth)
        self.kde = {"bandwidth_": h, "n_fit": m}

    def forward(self, x, return_ue=False):
        if return_ue and self.kde is None:
            raise ValueError("KDE not fitted yet")
        pred = super().forward(x)
        if return_ue:
            ops._require_cuda(x, "x")
            dens = ops.kde_density(self._kde_data.to(x.device), x, self.kde["bandwidth_"])
            return pred, dens
        return pred

    class KDEFitCallback(_Callback):
        """Fits the KDE on the inputs of the first training epoch (reference models.py:224-238)."""

        def __init__(self):
            super().__init__()
            self._train_data_to_fit = []
            self._epochs = 0

        def on_train_epoch_end(self, trainer, pl_module):
            if self._epochs == 0:
                pl_module.fit_kde(torch.cat(self._train_data_to_fit))
            self._epochs += 1

        def on_train_batch_end(self, trainer, pl_module, outputs, batch, batch_idx):
            if self._epochs == 0:
                self._train_data_to_fit.append(batch[0])

    def get_callbacks(self):
        return [KDEMLPModel.KDEFitCallback()]


KNNKDEMLPModel = _out_of_scope("KNNKDEMLPModel")


class PAGERMLP(DeltaUQMLP):
    """Delta-UQ + anchor-consistency (conformal) score, reference models.py:376-468.

    ``forward(x, return_ue=True)`` returns ``(mu, max(std, score))`` where ``mu, std`` are the
    Delta-UQ mean/std over the anchors and ``score[n] = max_k |net(cat(x_n, a_k - x_n)) - Y_k|``
    (``_score_samples`` / ``_anchored_predictions``, :396-429: the roles of sample and anchor are
    swapped).  Both are one fused launch each; the second one takes the first one's ``std`` as a
    floor, so the ``[N, K]`` prediction matrix and the ``torch.maximum`` never materialise.
    PARITY-UNPINNED like ``DeltaUQMLP`` (the anchoring lives in the absent ``deltauq`` package).
    With ``uq_shard = KShard()`` the anchors of both passes are split over the ranks; the conformal
    shards combine with one element-wise max all-reduce."""

    def __init__(self, base_model, estimator='std', anchored_batch_size=None, num_anchors=5,
                 vectorize=False, **kwargs):
        super().__init__(base_model, estimator=estimator, num_anchors=num_anchors,
                         anchored_batch_size=anchored_batch_size, **kwargs)
        self.vectorize = vectorize   # loop and vectorised branches of :398-424 compute the same
        self.register_buffer('_anchors_Y', None)

    def forward(self, x, return_ue=False):
        res = super().forward(x, return_ue)
        if not return_ue or self.training or self._anchors is None:
            return res
        if self._anchors_Y is None:
            raise ValueError("PAGER anchors_Y not set yet")
        mu, std = res
        packed = self._packed([self.net], x.device)
        k = int(self.num_anchors)
        kw = dict(total_members=k, precision=self.uq_precision, anchors=self._anchors.to(x.device),
                  targets=self._anchors_Y.to(x.device), score_floor=std.to(torch.float32))
        shard = self.__dict__.get("uq_shard")
        if shard is not None and hasattr(shard, "split"):
            # anchors sharded over the ranks (KShard): the conformal score is a max over anchors,
            # so the shards combine with ONE element-wise max all-reduce
            import torch.distributed as dist
            begin, count = shard.split(k)
            if count > 0:
                _, score = packed.forward(x, "pager", member_begin=begin, member_count=count, **kw)
            else:
                score = kw["score_floor"].clone()
            dist.all_reduce(score, op=dist.ReduceOp.MAX, group=shard.group)
        else:
            _, score = packed.forward(x, "pager", **kw)
        return mu, score.to(std.dtype)

    def _score_samples(self, x, anchors_X, anchors_Y):
        """Conformal score alone (reference :426-429), shape ``[N, 1]``."""
        ops._require_cuda(x, "x")
        packed = self._packed([self.net], x.device)
        k = anchors_X.shape[0]
        _, score = packed.forward(x, "pager", total_members=int(k), precision=self.uq_precision,
                                  anchors=anchors_X.to(x.device), targets=anchors_Y.to(x.device))
        return score

    @property
    def anchors_Y(self):
        return self._anchors_Y

    @anchors_Y.setter
    def anchors_Y(self, value):
        self._anchors_Y = value.detach().clone()

    class PAGERGetAnchorsCallback(_Callback):
        """Inputs AND targets of the first ``num_anchors`` training rows (reference :451-468)."""

        def __init__(self):
            super().__init__()
            self._anchor_X, self._anchor_Y = [], []
            self._epochs = 0

        def on_validation_epoch_start(self, trainer, pl_module):
            if self._epochs == 0 and len(self._anchor_X) > 0:
                k = pl_module.num_anchors
                pl_module.anchors = torch.cat(self._anchor_X)[0:k].detach().clone()
                pl_module.anchors_Y = torch.cat(self._anchor_Y)[0:k].detach().clone()
            self._epochs += 1

        def on_train_batch_end(self, trainer, pl_module, outputs, batch, batch_idx):
            bs = batch[0].shape[0]
            if self._epochs == 0 and bs * len(self._anchor_X) < pl_module.num_anchors:
                self._anchor_X.append(batch[0].detach())
                self._anchor_Y.append(batch[1].detach())

    def get_callbacks(self):
        return [PAGERMLP.PAGERGetAnchorsCallback()]
